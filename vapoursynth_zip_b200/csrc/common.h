// common.h — internal declarations shared by the runtime, the filter host logic and the kernels.
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <condition_variable>
#include <cstdarg>
#include <cstdint>
#include <mutex>
#include <vector>

#include "vszip_cuda.h"

namespace vsz {

// --------------------------------------------------------------------------- errors / counters
void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }
extern std::atomic<uint64_t> g_transfer[2];  // sample bytes of frames moved host -> device [0] / device -> host [1]
inline void count_transfer(int dir, size_t bytes) { g_transfer[dir].fetch_add((uint64_t)bytes, std::memory_order_relaxed); }

#define VSZ_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            ::vsz::set_error("CUDA error '%s' at %s:%d (%s)", cudaGetErrorString(e__), __FILE__,    \
                             __LINE__, #call);                                                      \
            return -1;                                                                              \
        }                                                                                           \
    } while (0)

// Opt-in to more than 48 KB of dynamic shared memory.  The attribute belongs to the function (per device), not to a launch:
// getFrame is re-entrant, so two host threads launching the same kernel with different sizes would race if each set its own size
// (thread A's small value lands between thread B's set and B's launch -> "invalid argument").  Every launch therefore sets the same
// constant, the architectural maximum; occupancy is decided by the size passed to the launch itself.
// (227 KB per CTA minus the kernel's static __shared__ variables, looked up once per kernel.)
constexpr int kMaxSmemPerCta = 227 * 1024;
int max_dynamic_smem_of(const void* kern);  // runtime.cu
template <class K>
inline cudaError_t allow_max_dynamic_smem(K kern) {
    const int lim = max_dynamic_smem_of(reinterpret_cast<const void*>(kern));
    if (lim < 0) return cudaErrorInvalidDeviceFunction;
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
}

// Stream-ordered scratch that is returned to the pool on every exit path (the error macros return early).
struct AsyncScratch {
    char* p = nullptr;
    cudaStream_t st = nullptr;
    AsyncScratch() = default;
    AsyncScratch(const AsyncScratch&) = delete;
    AsyncScratch& operator=(const AsyncScratch&) = delete;
    ~AsyncScratch() { release(); }
    cudaError_t alloc(size_t bytes, cudaStream_t s) { release(); st = s; return cudaMallocAsync((void**)&p, bytes, s); }
    void release() { if (p) { cudaFreeAsync(p, st); p = nullptr; } }
};

// --------------------------------------------------------------------------- formats / layout
// helper.zig DataType (src/helper.zig:59-97): selected by bytesPerSample, so 9..16-bit integer
// clips are all u16.
enum SampleKind { K_U8 = 0, K_U16 = 1, K_F16 = 2, K_F32 = 3, K_U32 = 4 };  // K_U32: Limiter only (src/helper.zig:14-56, BPSType.U32)

struct PlaneGeom {
    int w, h;
    int pitch;      // bytes, multiple of 128
    size_t offset;  // bytes from the frame base
};

// How one frame is laid out in HBM (and, identically, in the pinned staging buffers).
struct FrameLayout {
    int nplanes;
    PlaneGeom pl[3];
    size_t frame_stride;  // bytes, multiple of 256
    int bps;              // bytes per sample
    SampleKind kind;
    int bits;
};

// returns false (and sets the "<name>: not supported Int/Float format." error) for formats
// DataType.select rejects.
bool select_kind(const vszip_video_info& vi, const char* filter_name, bool enable_u32, SampleKind* out);
FrameLayout make_layout(const vszip_video_info& vi, SampleKind kind);
size_t layout_algorithmic_bytes(const FrameLayout& l);

// --------------------------------------------------------------------------- device runtime
struct Slot {  // one in-flight getFrame request
    cudaStream_t stream = nullptr;
    char* pin[4] = {nullptr, nullptr, nullptr, nullptr};  // pinned host: src, ref/clipb, dst, third input (LimitFilter ref)
    char* dev[4] = {nullptr, nullptr, nullptr, nullptr};  // device: same roles
    size_t cap[4] = {0, 0, 0, 0};
    void* pin_small = nullptr;  // 4 KB pinned scratch for tiny results
    void* dev_small = nullptr;  // 64 KB device scratch for reductions
    std::vector<char*> xdev;    // device-only frame buffers beyond dev[] (fused chains whose buffer plan needs more), grown on demand
    std::vector<size_t> xcap;
    bool streaming_copies = false;  // set at acquire(): the host is crowded, staging copies bypass the cache
};

struct DeviceCtx {
    int ordinal = -1;  // CUDA device ordinal
    int sm_count = 0;
    cudaStream_t batch_stream = nullptr;
    std::mutex mu;
    std::condition_variable cv;
    std::vector<Slot*> all, idle;
    Slot* acquire();
    void release(Slot* s);
};

int num_devices();
DeviceCtx* device_ctx(int index);                // index into the init list
DeviceCtx* device_for_frame(int32_t n);          // n mod k routing
int slot_reserve(DeviceCtx* d, Slot* s, int which, size_t bytes);  // grow pin[which]/dev[which]
int slot_reserve_extra(DeviceCtx* d, Slot* s, int which, size_t bytes);  // grow xdev[which] (no pinned twin)

// host <-> slot staging of the selected planes of one frame (async on s->stream)
int stage_in(Slot* s, int which, const FrameLayout& l, const vszip_frame* host, const bool mask[3]);
int stage_out_begin(Slot* s, const FrameLayout& l, vszip_frame* host, const bool mask[3], bool direct[3]);  // async D2H
void stage_out_finish(Slot* s, const FrameLayout& l, vszip_frame* host, const bool mask[3], const bool direct[3]);  // after sync

}  // namespace vsz

// --------------------------------------------------------------------------- public opaque types
struct vszip_dev_clip {
    int device_index;
    int ordinal;
    vszip_video_info vi;
    vsz::FrameLayout layout;
    int num_frames;
    char* base;
};

// --------------------------------------------------------------------------- kernel-side batch descriptors
namespace vsz {

struct PlaneJob {
    size_t src_off, dst_off, ref_off;
    int src_pitch, dst_pitch, ref_pitch;
    int w, h;
    int cta_begin;  // first blockIdx.x of this plane within a frame
    int aux;        // per-plane parameter index (bilateral)
};

struct BatchJob {
    const char* src;
    const char* ref;
    char* dst;
    size_t src_fs, ref_fs, dst_fs;  // frame strides
    int nplanes;                    // number of PROCESSED planes listed in pl[]
    int ctas_per_frame;
    PlaneJob pl[3];
};

// Builds the descriptor for the processed planes; ctas_for(plane w,h) says how many CTAs a plane needs.
template <class F>
inline BatchJob make_batch(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, const char* ref,
                           size_t ref_fs, char* dst, size_t dst_fs, F ctas_for) {
    BatchJob b{};
    b.src = src; b.ref = ref; b.dst = dst;
    b.src_fs = src_fs; b.ref_fs = ref_fs; b.dst_fs = dst_fs;
    int cta = 0, k = 0;
    for (int p = 0; p < l.nplanes; ++p) {
        if (!mask[p]) continue;
        PlaneJob& j = b.pl[k++];
        j.src_off = j.dst_off = j.ref_off = l.pl[p].offset;
        j.src_pitch = j.dst_pitch = j.ref_pitch = l.pl[p].pitch;
        j.w = l.pl[p].w; j.h = l.pl[p].h;
        j.cta_begin = cta;
        j.aux = p;
        cta += ctas_for(l.pl[p].w, l.pl[p].h);
    }
    b.nplanes = k;
    b.ctas_per_frame = cta;
    return b;
}

}  // namespace vsz
