// runtime.cu — per-GPU contexts (frame pool, pinned staging, one stream per in-flight request),
// device-resident clips, the noise generator, and the small C-ABI utility entry points.
#include <cuda_fp16.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>

#include "common.h"

namespace vsz {

static thread_local std::string t_error;
std::atomic<uint64_t> g_launches{0};
std::atomic<uint64_t> g_transfer[2] = {{0}, {0}};

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    t_error = buf;
}

// --------------------------------------------------------------------------- formats
bool select_kind(const vszip_video_info& vi, const char* name, bool enable_u32, SampleKind* out) {
    if (vi.sample_type == VSZIP_ST_INTEGER) {
        if (vi.bytes_per_sample == 1) { *out = K_U8; return true; }
        if (vi.bytes_per_sample == 2) { *out = K_U16; return true; }
        if (vi.bytes_per_sample == 4 && enable_u32) { *out = K_U32; return true; }  // Limiter; PlaneAverage rejects it right after
        set_error("%s: not supported Int format.", name);
        return false;
    }
    if (vi.bytes_per_sample == 2) { *out = K_F16; return true; }
    if (vi.bytes_per_sample == 4) { *out = K_F32; return true; }
    set_error("%s: not supported Float format.", name);
    return false;
}

FrameLayout make_layout(const vszip_video_info& vi, SampleKind kind) {
    FrameLayout l{};
    l.nplanes = vi.num_planes;
    l.bps = vi.bytes_per_sample;
    l.kind = kind;
    l.bits = vi.bits_per_sample;
    size_t off = 0;
    for (int p = 0; p < l.nplanes; ++p) {
        const int sw = p ? vi.sub_sampling_w : 0, sh = p ? vi.sub_sampling_h : 0;
        l.pl[p].w = vi.width >> sw;
        l.pl[p].h = vi.height >> sh;
        l.pl[p].pitch = (int)(((size_t)l.pl[p].w * l.bps + 127) / 128 * 128);
        l.pl[p].offset = off;
        off += (size_t)l.pl[p].pitch * l.pl[p].h;
        off = (off + 255) / 256 * 256;
    }
    l.frame_stride = off;
    return l;
}

size_t layout_algorithmic_bytes(const FrameLayout& l) {
    size_t s = 0;
    for (int p = 0; p < l.nplanes; ++p) s += (size_t)l.pl[p].w * l.pl[p].h * l.bps;
    return s;
}

// --------------------------------------------------------------------------- contexts
static std::mutex g_init_mu;
static std::vector<DeviceCtx*> g_devs;
static constexpr int kSlotsPerDevice = 16;
// host_copy.cpp: row copies between application memory and the pinned staging buffers (streaming stores when many requests are in flight)
void copy_rows(char* dst, ptrdiff_t dpitch, const char* src, ptrdiff_t spitch, size_t row_bytes, int rows, bool streaming);
static constexpr int kStreamingBusySlots = 10;

Slot* DeviceCtx::acquire() {
    std::unique_lock<std::mutex> lk(mu);
    cv.wait(lk, [&] { return !idle.empty(); });
    Slot* s = idle.back();
    idle.pop_back();
    // how crowded the host side is right now decides how this request copies its planes (see host_copy.cpp)
    s->streaming_copies = (int)(all.size() - idle.size()) >= kStreamingBusySlots;
    return s;
}

void DeviceCtx::release(Slot* s) {
    {
        std::lock_guard<std::mutex> lk(mu);
        idle.push_back(s);
    }
    cv.notify_one();
}

int num_devices() { return (int)g_devs.size(); }
DeviceCtx* device_ctx(int index) { return (index >= 0 && index < (int)g_devs.size()) ? g_devs[index] : nullptr; }
DeviceCtx* device_for_frame(int32_t n) {
    if (g_devs.empty()) return nullptr;
    const int k = (int)g_devs.size();
    return g_devs[((n % k) + k) % k];
}

int slot_reserve(DeviceCtx* d, Slot* s, int which, size_t bytes) {
    if (s->cap[which] >= bytes) return 0;
    VSZ_CUDA(cudaSetDevice(d->ordinal));
    VSZ_CUDA(cudaStreamSynchronize(s->stream));
    if (s->pin[which]) cudaFreeHost(s->pin[which]);
    if (s->dev[which]) cudaFree(s->dev[which]);
    s->pin[which] = s->dev[which] = nullptr;
    s->cap[which] = 0;
    VSZ_CUDA(cudaHostAlloc((void**)&s->pin[which], bytes, cudaHostAllocDefault));
    VSZ_CUDA(cudaMalloc((void**)&s->dev[which], bytes));
    s->cap[which] = bytes;
    return 0;
}

int slot_reserve_extra(DeviceCtx* d, Slot* s, int which, size_t bytes) {
    if ((int)s->xdev.size() <= which) { s->xdev.resize(which + 1, nullptr); s->xcap.resize(which + 1, 0); }
    if (s->xcap[which] >= bytes) return 0;
    VSZ_CUDA(cudaSetDevice(d->ordinal));
    VSZ_CUDA(cudaStreamSynchronize(s->stream));
    if (s->xdev[which]) cudaFree(s->xdev[which]);
    s->xdev[which] = nullptr;
    s->xcap[which] = 0;
    VSZ_CUDA(cudaMalloc((void**)&s->xdev[which], bytes));
    s->xcap[which] = bytes;
    return 0;
}

// largest dynamic shared memory size a kernel may ask for (see allow_max_dynamic_smem in common.h)
int max_dynamic_smem_of(const void* kern) {
    static std::mutex mu;
    static std::map<const void*, int> known;
    std::lock_guard<std::mutex> lk(mu);
    auto it = known.find(kern);
    if (it != known.end()) return it->second;
    cudaFuncAttributes a;
    if (cudaFuncGetAttributes(&a, kern) != cudaSuccess) { cudaGetLastError(); return -1; }
    const int lim = kMaxSmemPerCta - (int)a.sharedSizeBytes;
    known[kern] = lim;
    return lim;
}

// --------------------------------------------------------------------------- host buffers: pinned or not
// VapourSynth hands getFrame pageable plane buffers that come out of the core's frame pool, i.e. the same addresses keep
// coming back (src/helper.zig:510-531 only sees pointers + strides).  A pageable buffer costs a staging memcpy into the slot's
// pinned buffer in each direction; a page-locked one is DMA'd in place.  The runtime keeps a cache keyed by buffer address:
//   * buffers the application pinned itself (cudaHostAlloc / cudaHostRegister) are recognised - the WHOLE plane must lie inside
//     one registration (CU_POINTER_ATTRIBUTE_RANGE_*), a plane that merely starts in pinned memory is staged - and remembered;
//   * opt-in (vszip_cuda_host_register_limit / VSZIP_HOST_REGISTER_MB > 0): a pageable buffer seen for the second time is
//     page-locked with cudaHostRegister (portable, so every GPU can reach it) and from then on treated like application-pinned
//     memory.  Only a registration of exactly the buffer's own pages counts: a buffer that shares a page with a neighbour that is
//     already registered (small heap allocations) stays on the staging path.  Nothing is evicted behind the application's back.
// Why opt-in: a registration describes physical pages.  If the owner frees a registered buffer without telling us (munmap) and the
// address range is mapped again later, the driver still DMAs to/from the OLD pages - silently wrong pixels.  VapourSynth's frame
// pool gives a filter no hook for "this buffer is going back to the OS", so registering the core's buffers is only safe when the
// host application guarantees the rule below (INTEGRATION.md): before memory that was passed to a get_frame call is freed or
// unmapped, call vszip_cuda_host_forget(ptr) (or with NULL for everything).
namespace {
struct HostRange {
    uintptr_t end = 0;
    bool ours = false;  // registered by this library (must be unregistered by it)
    int seen = 0;       // sightings while still pageable; -1 = known pinned; 0 = never try again
};
std::mutex g_host_mu;
std::map<uintptr_t, HostRange> g_host;  // key = first byte of the plane buffer as passed in
size_t g_host_registered = 0;

std::atomic<size_t> g_host_cap{SIZE_MAX};  // SIZE_MAX = not set yet: take VSZIP_HOST_REGISTER_MB (default 0 = off)

size_t host_register_cap() {
    size_t cap = g_host_cap.load(std::memory_order_relaxed);
    if (cap == SIZE_MAX) {
        const char* e = getenv("VSZIP_HOST_REGISTER_MB");
        cap = (size_t)(e ? strtoull(e, nullptr, 10) : 0ull) << 20;
        g_host_cap.store(cap, std::memory_order_relaxed);
    }
    return cap;
}

// cuPointerGetAttribute through the runtime's driver entry point lookup (libcuda is not linked)
using PointerAttrFn = int (*)(void*, int, unsigned long long);
PointerAttrFn pointer_attr_fn() {
    static const PointerAttrFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuPointerGetAttribute", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            p = nullptr;
        }
        return reinterpret_cast<PointerAttrFn>(p);
    }();
    return fn;
}

// true when [p, p + bytes) lies inside ONE page-locked host allocation / registration known to the driver
bool whole_range_pinned(const void* p, size_t bytes) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (a.type != cudaMemoryTypeHost) return false;
    const PointerAttrFn attr = pointer_attr_fn();
    if (!attr) return false;
    unsigned long long start = 0;
    size_t size = 0;
    // CU_POINTER_ATTRIBUTE_RANGE_START_ADDR = 11, CU_POINTER_ATTRIBUTE_RANGE_SIZE = 12 (cuda.h)
    if (attr(&start, 11, (unsigned long long)(uintptr_t)p) != 0 || attr(&size, 12, (unsigned long long)(uintptr_t)p) != 0) return false;
    return (uintptr_t)start <= (uintptr_t)p && (uintptr_t)p + bytes <= (uintptr_t)start + size;
}
}  // namespace

// true when the plane buffer [p, p + bytes) can be reached by the DMA engines directly; may page-lock it (see above)
static bool host_plane_pinned(const void* p, size_t bytes) {
    const uintptr_t a = (uintptr_t)p;
    std::lock_guard<std::mutex> lk(g_host_mu);
    auto it = g_host.find(a);
    if (it != g_host.end() && it->second.seen < 0) return it->second.end >= a + bytes;  // known pinned (seen = -1)
    const size_t cap = host_register_cap();
    if (it == g_host.end()) {
        HostRange r;
        const bool pinned = whole_range_pinned(p, bytes);
        if (pinned) { r.end = a + bytes; r.seen = -1; } else r.seen = 1;
        if (g_host.size() < 65536) g_host[a] = r;  // bounded bookkeeping; a remembered "pageable" also saves the driver query next time
        return pinned;
    }
    HostRange& r = it->second;
    if (r.seen == 0) return false;  // registration failed before: stay on the staging path
    ++r.seen;
    const uintptr_t lo = a & ~(uintptr_t)4095, hi = (a + bytes + 4095) & ~(uintptr_t)4095;
    if (cap == 0 || g_host_registered + (hi - lo) > cap) return false;
    const cudaError_t e = cudaHostRegister((void*)lo, hi - lo, cudaHostRegisterPortable);
    if (e == cudaSuccess) {
        r.end = a + bytes; r.ours = true; r.seen = -1;
        g_host_registered += hi - lo;
        return true;
    }
    cudaGetLastError();
    // e.g. cudaErrorHostMemoryAlreadyRegistered: the buffer shares a page with a registered neighbour, or the application pinned
    // a larger buffer in the meantime - the latter is fine if the driver now covers the whole plane with one range
    if (whole_range_pinned(p, bytes)) { r.end = a + bytes; r.seen = -1; return true; }
    r.seen = 0;
    return false;
}

static size_t plane_span_bytes(const FrameLayout& l, int p, ptrdiff_t stride) {
    return (size_t)(stride < 0 ? -stride : stride) * (size_t)(l.pl[p].h - 1) + (size_t)l.pl[p].w * l.bps;
}
static bool is_pinned_host(const FrameLayout& l, int p, const vszip_frame* host) {
    if (host->stride[p] <= 0) return false;
    return host_plane_pinned(host->data[p], plane_span_bytes(l, p, host->stride[p]));
}

// Pinned planes go by DMA straight from/to the application's memory.  Fewer, larger copies keep the copy engines
// busier: a plane whose host stride equals the device pitch is one linear copy, and a run of planes that sit in host
// memory exactly as they do in the device frame (same pitch, back to back - e.g. a frame carved out of one pinned
// buffer) is a single copy.  Returns the index after the last plane covered by the copy issued for plane p.
static int pinned_copy(Slot* s, int dev_buf, const FrameLayout& l, const vszip_frame* host, const bool mask[3], const bool pinned[3], int p,
                       bool to_device, cudaError_t* err) {
    const PlaneGeom& g = l.pl[p];
    const size_t row_bytes = (size_t)g.w * l.bps;
    char* hp = (char*)host->data[p];
    char* dp = s->dev[dev_buf] + g.offset;
    if (host->stride[p] != (ptrdiff_t)g.pitch) {
        *err = to_device ? cudaMemcpy2DAsync(dp, g.pitch, hp, host->stride[p], row_bytes, g.h, cudaMemcpyHostToDevice, s->stream)
                         : cudaMemcpy2DAsync(hp, host->stride[p], dp, g.pitch, row_bytes, g.h, cudaMemcpyDeviceToHost, s->stream);
        return p + 1;
    }
    int q = p;  // extend over planes laid out identically and contiguously on both sides
    while (q + 1 < l.nplanes && mask[q + 1] && pinned[q + 1] && host->stride[q + 1] == (ptrdiff_t)l.pl[q + 1].pitch &&
           (size_t)l.pl[q].pitch * l.pl[q].h == (size_t)l.pl[q].w * l.bps * l.pl[q].h &&               // no row padding
           l.pl[q].offset + (size_t)l.pl[q].pitch * l.pl[q].h == l.pl[q + 1].offset &&                 // no gap on the device
           (char*)host->data[q + 1] == (char*)host->data[q] + (size_t)l.pl[q].pitch * l.pl[q].h)        // nor on the host
        ++q;
    const PlaneGeom& e = l.pl[q];
    const size_t bytes = (e.offset - g.offset) + (size_t)e.pitch * (e.h - 1) + (size_t)e.w * l.bps;  // not past the last sample
    *err = to_device ? cudaMemcpyAsync(dp, hp, bytes, cudaMemcpyHostToDevice, s->stream)
                     : cudaMemcpyAsync(hp, dp, bytes, cudaMemcpyDeviceToHost, s->stream);
    return q + 1;
}

int stage_in(Slot* s, int which, const FrameLayout& l, const vszip_frame* host, const bool mask[3]) {
    bool pinned[3] = {false, false, false};
    for (int p = 0; p < l.nplanes; ++p) {
        pinned[p] = mask[p] && is_pinned_host(l, p, host);
        if (mask[p]) count_transfer(0, (size_t)l.pl[p].w * l.pl[p].h * l.bps);
    }
    for (int p = 0; p < l.nplanes;) {
        if (!mask[p]) { ++p; continue; }
        const PlaneGeom& g = l.pl[p];
        if (pinned[p]) {
            cudaError_t e = cudaSuccess;
            p = pinned_copy(s, which, l, host, mask, pinned, p, true, &e);
            VSZ_CUDA(e);
            continue;
        }
        // pageable VapourSynth memory -> pinned staging (same layout as the device frame)
        copy_rows(s->pin[which] + g.offset, g.pitch, (const char*)host->data[p], host->stride[p], (size_t)g.w * l.bps, g.h, s->streaming_copies);
        VSZ_CUDA(cudaMemcpyAsync(s->dev[which] + g.offset, s->pin[which] + g.offset, (size_t)g.pitch * g.h,
                                 cudaMemcpyHostToDevice, s->stream));
        ++p;
    }
    return 0;
}

// D2H of the result planes: straight into the destination when it is pinned, else into the slot's
// pinned buffer (stage_out_finish then copies it out after the stream has been synchronised).
int stage_out_begin(Slot* s, const FrameLayout& l, vszip_frame* host, const bool mask[3], bool direct[3]) {
    bool pinned[3] = {false, false, false};
    for (int p = 0; p < l.nplanes; ++p) {
        pinned[p] = mask[p] && is_pinned_host(l, p, host); direct[p] = pinned[p];
        if (mask[p]) count_transfer(1, (size_t)l.pl[p].w * l.pl[p].h * l.bps);
    }
    for (int p = 0; p < l.nplanes;) {
        if (!mask[p]) { ++p; continue; }
        const PlaneGeom& g = l.pl[p];
        if (pinned[p]) {
            cudaError_t e = cudaSuccess;
            p = pinned_copy(s, 2, l, host, mask, pinned, p, false, &e);
            VSZ_CUDA(e);
            continue;
        }
        VSZ_CUDA(cudaMemcpyAsync(s->pin[2] + g.offset, s->dev[2] + g.offset, (size_t)g.pitch * g.h,
                                 cudaMemcpyDeviceToHost, s->stream));
        ++p;
    }
    return 0;
}

void stage_out_finish(Slot* s, const FrameLayout& l, vszip_frame* host, const bool mask[3], const bool direct[3]) {
    for (int p = 0; p < l.nplanes; ++p) {
        if (!mask[p] || direct[p]) continue;
        const PlaneGeom& g = l.pl[p];
        copy_rows((char*)host->data[p], host->stride[p], s->pin[2] + g.offset, g.pitch, (size_t)g.w * l.bps, g.h, s->streaming_copies);
    }
}

// --------------------------------------------------------------------------- noise generator
__device__ __forceinline__ uint32_t mix64to32(uint64_t z) {  // splitmix64 finaliser
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (uint32_t)(z >> 32);
}

template <typename T>
__global__ void noise_kernel(char* base, size_t frame_stride, size_t plane_off, int pitch, int w, int h, int plane,
                             uint64_t seed, int first_frame_no, int frame_no_stride, int kind, int bits, int chroma_centered) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    const int f = blockIdx.z;
    if (x >= w) return;
    const uint64_t key = (seed * 0x100000001B3ull) ^ ((uint64_t)(uint32_t)(first_frame_no + f * frame_no_stride) << 40) ^
                         ((uint64_t)plane << 36) ^ ((uint64_t)y << 18) ^ (uint64_t)x;
    const uint32_t u = mix64to32(key);
    T* row = reinterpret_cast<T*>(base + (size_t)f * frame_stride + plane_off + (size_t)y * pitch);
    if constexpr (std::is_same<T, uint8_t>::value || std::is_same<T, uint16_t>::value) {
        row[x] = (T)(u >> (32 - bits));
    } else {
        float v = (float)(u >> 8) * (1.0f / 16777216.0f);  // [0,1)
        if (chroma_centered) v -= 0.5f;
        if constexpr (std::is_same<T, __half>::value) row[x] = __float2half_rn(v);
        else row[x] = v;
    }
}

}  // namespace vsz

using namespace vsz;

// =========================================================================== C ABI: runtime
extern "C" {

int vszip_cuda_abi_version(void) { return VSZIP_CUDA_ABI_VERSION; }
const char* vszip_cuda_last_error(void) { return t_error.c_str(); }
uint64_t vszip_cuda_kernel_launches(void) { return g_launches.load(); }
uint64_t vszip_cuda_transfer_bytes(int32_t direction) { return (direction == 0 || direction == 1) ? g_transfer[direction].load() : 0; }
int vszip_cuda_device_count(void) { return num_devices(); }

int vszip_cuda_init(const int32_t* device_ids, int32_t n) {
    std::lock_guard<std::mutex> lk(g_init_mu);
    if (!g_devs.empty()) return (int)g_devs.size();
    int visible = 0;
    cudaError_t e = cudaGetDeviceCount(&visible);
    if (e != cudaSuccess || visible <= 0) {
        set_error("vszip_cuda_init: no CUDA device available (%s); there is no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return -1;
    }
    std::vector<int> ids;
    if (n <= 0 || device_ids == nullptr) for (int i = 0; i < visible; ++i) ids.push_back(i);
    else for (int i = 0; i < n; ++i) ids.push_back(device_ids[i]);
    for (int id : ids) {
        if (id < 0 || id >= visible) { set_error("vszip_cuda_init: device ordinal %d out of range (0..%d)", id, visible - 1); return -1; }
        cudaDeviceProp prop;
        VSZ_CUDA(cudaGetDeviceProperties(&prop, id));
        if (prop.major < 10) {
            set_error("vszip_cuda_init: device %d (%s, sm_%d%d) is not a Blackwell sm_100 GPU; kernels are built for sm_100a only",
                      id, prop.name, prop.major, prop.minor);
            return -1;
        }
    }
    for (int id : ids) {
        VSZ_CUDA(cudaSetDevice(id));
        DeviceCtx* d = new DeviceCtx();
        d->ordinal = id;
        VSZ_CUDA(cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, id));
        VSZ_CUDA(cudaStreamCreateWithFlags(&d->batch_stream, cudaStreamNonBlocking));
        cudaMemPool_t pool;  // keep stream-ordered scratch cached between calls
        if (cudaDeviceGetDefaultMemPool(&pool, id) == cudaSuccess) {
            uint64_t thr = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
        for (int i = 0; i < kSlotsPerDevice; ++i) {
            Slot* s = new Slot();
            VSZ_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
            VSZ_CUDA(cudaHostAlloc(&s->pin_small, 4096, cudaHostAllocDefault));
            VSZ_CUDA(cudaMalloc(&s->dev_small, 1 << 16));
            d->all.push_back(s);
            d->idle.push_back(s);
        }
        g_devs.push_back(d);
    }
    return (int)g_devs.size();
}

void vszip_cuda_shutdown(void) {
    vszip_cuda_host_forget(nullptr);
    std::lock_guard<std::mutex> lk(g_init_mu);
    for (DeviceCtx* d : g_devs) {
        cudaSetDevice(d->ordinal);
        cudaDeviceSynchronize();
        for (Slot* s : d->all) {
            for (int i = 0; i < 4; ++i) { if (s->pin[i]) cudaFreeHost(s->pin[i]); if (s->dev[i]) cudaFree(s->dev[i]); }
            for (char* x : s->xdev) if (x) cudaFree(x);
            if (s->pin_small) cudaFreeHost(s->pin_small);
            if (s->dev_small) cudaFree(s->dev_small);
            cudaStreamDestroy(s->stream);
            delete s;
        }
        cudaStreamDestroy(d->batch_stream);
        delete d;
    }
    g_devs.clear();
}

void vszip_cuda_host_forget(const void* ptr) {
    std::lock_guard<std::mutex> lk(g_host_mu);
    auto drop = [](std::map<uintptr_t, HostRange>::iterator it) {
        if (it->second.ours) {
            const uintptr_t lo = it->first & ~(uintptr_t)4095, hi = (it->second.end + 4095) & ~(uintptr_t)4095;
            if (cudaHostUnregister((void*)lo) != cudaSuccess) cudaGetLastError();
            g_host_registered -= std::min(g_host_registered, (size_t)(hi - lo));
        }
    };
    if (!ptr) {
        for (auto it = g_host.begin(); it != g_host.end(); ++it) drop(it);
        g_host.clear();
        return;
    }
    auto it = g_host.find((uintptr_t)ptr);
    if (it == g_host.end()) return;
    drop(it);
    g_host.erase(it);
}

size_t vszip_cuda_host_register_limit(size_t bytes) {
    const size_t before = host_register_cap();
    g_host_cap.store(bytes == SIZE_MAX ? SIZE_MAX - 1 : bytes, std::memory_order_relaxed);
    return before;
}

// Sizes the staging buffers of every request slot of every GPU for frames of this format now, instead of on the first frames
// that come through each slot (cudaHostAlloc + cudaMalloc of a frame: a first-call latency spike of milliseconds).
int32_t vszip_cuda_reserve(const vszip_video_info* vi, int32_t buffers) {
    if (!vi || vi->width <= 0 || vi->height <= 0 || vi->bytes_per_sample <= 0) { set_error("vszip_cuda_reserve: bad video info"); return -1; }
    if (num_devices() == 0) { set_error("vszip_cuda_reserve: vszip_cuda_init has not been called"); return -1; }
    const SampleKind kind = vi->bytes_per_sample == 1 ? K_U8 : (vi->bytes_per_sample == 2 ? K_U16 : K_F32);  // only the sample size matters here
    const FrameLayout l = make_layout(*vi, kind);
    const int nb = std::max(1, std::min(buffers, 4));
    for (int i = 0; i < num_devices(); ++i) {
        DeviceCtx* d = device_ctx(i);
        size_t nslots;
        { std::lock_guard<std::mutex> lk(d->mu); nslots = d->all.size(); }
        std::vector<Slot*> held;
        int rc = 0;
        for (size_t k = 0; k < nslots; ++k) held.push_back(d->acquire());  // every slot once: none is in flight while it grows
        for (Slot* s : held)
            for (int which = 0; which < nb && rc == 0; ++which) rc = slot_reserve(d, s, which, l.frame_stride);
        for (Slot* s : held) d->release(s);
        if (rc) return -1;
    }
    return 0;
}

size_t vszip_cuda_host_registered_bytes(void) {
    std::lock_guard<std::mutex> lk(g_host_mu);
    return g_host_registered;
}

int vszip_cuda_stream_sync(int32_t device, void* stream) {
    DeviceCtx* d = device_ctx(device);
    if (!d) { set_error("vszip_cuda_stream_sync: bad device index %d", device); return -1; }
    VSZ_CUDA(cudaSetDevice(d->ordinal));
    VSZ_CUDA(cudaStreamSynchronize(stream ? (cudaStream_t)stream : d->batch_stream));
    return 0;
}

// --------------------------------------------------------------------------- device clips
vszip_dev_clip* vszip_dev_clip_alloc(const vszip_video_info* vi, int32_t num_frames, int32_t device) {
    DeviceCtx* d = device_ctx(device);
    if (!d) { set_error("vszip_dev_clip_alloc: library not initialised or bad device index %d", device); return nullptr; }
    SampleKind kind;
    if (!select_kind(*vi, "vszip_dev_clip_alloc", false, &kind)) return nullptr;
    if (num_frames <= 0 || vi->width <= 0 || vi->height <= 0 || vi->num_planes < 1 || vi->num_planes > 3) {
        set_error("vszip_dev_clip_alloc: bad geometry");
        return nullptr;
    }
    vszip_dev_clip* c = new vszip_dev_clip();
    c->device_index = device;
    c->ordinal = d->ordinal;
    c->vi = *vi;
    c->layout = make_layout(*vi, kind);
    c->num_frames = num_frames;
    if (cudaSetDevice(d->ordinal) != cudaSuccess ||
        cudaMalloc((void**)&c->base, c->layout.frame_stride * (size_t)num_frames) != cudaSuccess) {
        set_error("vszip_dev_clip_alloc: cudaMalloc of %zu bytes failed", c->layout.frame_stride * (size_t)num_frames);
        delete c;
        return nullptr;
    }
    // padding bytes are never read as pixels, but keep them defined
    cudaMemset(c->base, 0, c->layout.frame_stride * (size_t)num_frames);
    return c;
}

void vszip_dev_clip_free(vszip_dev_clip* c) {
    if (!c) return;
    cudaSetDevice(c->ordinal);
    cudaFree(c->base);
    delete c;
}

size_t vszip_dev_clip_frame_bytes(const vszip_dev_clip* c) { return layout_algorithmic_bytes(c->layout); }

void* vszip_dev_clip_plane_ptr(const vszip_dev_clip* c, int32_t frame, int32_t plane, ptrdiff_t* pitch) {
    if (frame < 0 || frame >= c->num_frames || plane < 0 || plane >= c->layout.nplanes) return nullptr;
    if (pitch) *pitch = c->layout.pl[plane].pitch;
    return c->base + (size_t)frame * c->layout.frame_stride + c->layout.pl[plane].offset;
}

int vszip_dev_clip_upload(vszip_dev_clip* c, int32_t frame, const vszip_frame* host) {
    if (frame < 0 || frame >= c->num_frames) { set_error("vszip_dev_clip_upload: frame out of range"); return -1; }
    VSZ_CUDA(cudaSetDevice(c->ordinal));
    for (int p = 0; p < c->layout.nplanes; ++p) {
        const PlaneGeom& g = c->layout.pl[p];
        VSZ_CUDA(cudaMemcpy2D(c->base + (size_t)frame * c->layout.frame_stride + g.offset, g.pitch, host->data[p],
                              host->stride[p], (size_t)g.w * c->layout.bps, g.h, cudaMemcpyHostToDevice));
        count_transfer(0, (size_t)g.w * g.h * c->layout.bps);
    }
    return 0;
}

int vszip_dev_clip_download(const vszip_dev_clip* c, int32_t frame, vszip_frame* host) {
    if (frame < 0 || frame >= c->num_frames) { set_error("vszip_dev_clip_download: frame out of range"); return -1; }
    VSZ_CUDA(cudaSetDevice(c->ordinal));
    VSZ_CUDA(cudaDeviceSynchronize());
    for (int p = 0; p < c->layout.nplanes; ++p) {
        const PlaneGeom& g = c->layout.pl[p];
        VSZ_CUDA(cudaMemcpy2D(host->data[p], host->stride[p], c->base + (size_t)frame * c->layout.frame_stride + g.offset,
                              g.pitch, (size_t)g.w * c->layout.bps, g.h, cudaMemcpyDeviceToHost));
        count_transfer(1, (size_t)g.w * g.h * c->layout.bps);
    }
    return 0;
}

int vszip_dev_clip_fill_noise(vszip_dev_clip* c, uint64_t seed, int32_t first_frame_no, int32_t frame_no_stride) {
    DeviceCtx* d = device_ctx(c->device_index);
    if (!d) { set_error("vszip_dev_clip_fill_noise: library not initialised"); return -1; }
    VSZ_CUDA(cudaSetDevice(c->ordinal));
    const FrameLayout& l = c->layout;
    for (int p = 0; p < l.nplanes; ++p) {
        const PlaneGeom& g = l.pl[p];
        const dim3 grid((g.w + 255) / 256, g.h, 1);
        const int centered = (p > 0 && c->vi.color_family == VSZIP_CF_YUV) ? 1 : 0;
        // grid.z is limited to 65535 frames per launch
        for (int f0 = 0; f0 < c->num_frames; f0 += 32768) {
            dim3 gz = grid;
            gz.z = (unsigned)std::min(32768, c->num_frames - f0);
            char* base = c->base + (size_t)f0 * l.frame_stride;
            switch (l.kind) {
                case K_U8: noise_kernel<uint8_t><<<gz, 256, 0, d->batch_stream>>>(base, l.frame_stride, g.offset, g.pitch, g.w, g.h, p, seed, first_frame_no + f0 * frame_no_stride, frame_no_stride, l.kind, l.bits, centered); break;
                case K_U16: noise_kernel<uint16_t><<<gz, 256, 0, d->batch_stream>>>(base, l.frame_stride, g.offset, g.pitch, g.w, g.h, p, seed, first_frame_no + f0 * frame_no_stride, frame_no_stride, l.kind, l.bits, centered); break;
                case K_F16: noise_kernel<__half><<<gz, 256, 0, d->batch_stream>>>(base, l.frame_stride, g.offset, g.pitch, g.w, g.h, p, seed, first_frame_no + f0 * frame_no_stride, frame_no_stride, l.kind, l.bits, centered); break;
                case K_F32: noise_kernel<float><<<gz, 256, 0, d->batch_stream>>>(base, l.frame_stride, g.offset, g.pitch, g.w, g.h, p, seed, first_frame_no + f0 * frame_no_stride, frame_no_stride, l.kind, l.bits, centered); break;
            }
            count_launch();
        }
    }
    VSZ_CUDA(cudaGetLastError());
    VSZ_CUDA(cudaStreamSynchronize(d->batch_stream));
    return 0;
}

}  // extern "C"
