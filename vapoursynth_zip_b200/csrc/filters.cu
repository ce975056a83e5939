// filters.cu — host side of the seven filters: argument parsing/validation with the reference's
// defaults and error strings (the twin of the create callbacks in src/vapoursynth/{boxblur,bilateral,planeminmax,
// planeaverage,limiter,limit_filter,adaptive_binarize}.zig), the synchronous getFrame-style entry points (host
// buffers, staged through the per-request slot), the batched device-resident entry points and the fused chains.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <array>
#include <limits>
#include <string>

#include "colormap_tables.h"
#include "filter.h"

using namespace vsz;

namespace {

// ZAPI getValue(u32/i32, ...) narrows the VapourSynth int64 with a saturating cast.
uint32_t sat_u32(int64_t v) { return v < 0 ? 0u : (v > 0xffffffffll ? 0xffffffffu : (uint32_t)v); }
int32_t sat_i32(int64_t v) { return v < INT32_MIN ? INT32_MIN : (v > INT32_MAX ? INT32_MAX : (int32_t)v); }

// hz.mapGetPlanes (src/helper.zig:128-158): an absent key keeps the filter's default mask.
bool parse_planes(const int64_t* planes, int n, int num_planes, const char* name, bool process[3]) {
    if (n < 0 || planes == nullptr) return true;
    process[0] = process[1] = process[2] = false;
    for (int i = 0; i < n; ++i) {
        const int64_t e = planes[i];
        if (e < 0 || e >= num_planes) { set_error("%s: plane index out of range", name); return false; }
        if (process[e]) { set_error("%s: plane specified twice.", name); return false; }
        process[e] = true;
    }
    return true;
}

// hz.compareNodes(..., .BIGGER_THAN, ...) (src/helper.zig:166-215)
bool compare_nodes(const vszip_video_info& a, const vszip_video_info& b, const char* name, bool same_len = false) {
    if (a.width != b.width || a.height != b.height) { set_error("%s: all input clips must have the same width and height.", name); return false; }
    if (a.color_family != b.color_family) { set_error("%s: all input clips must have the same color family.", name); return false; }
    if (a.sub_sampling_w != b.sub_sampling_w || a.sub_sampling_h != b.sub_sampling_h) { set_error("%s: all input clips must have the same subsampling.", name); return false; }
    if (a.bits_per_sample != b.bits_per_sample) { set_error("%s: all input clips must have the same bit depth.", name); return false; }
    if (same_len) {  // .SAME_LEN
        if (a.num_frames != b.num_frames) { set_error("%s: all input clips must have the same length.", name); return false; }
        return true;
    }
    if (a.num_frames > b.num_frames) { set_error("%s: second clip has less frames than input clip.", name); return false; }
    return true;
}

std::string fmt_num(double v) {  // Zig's {d}: shortest decimal that round-trips, never an exponent
    char buf[400];
    if (v == std::floor(v) && std::fabs(v) < 1e15) {
        snprintf(buf, sizeof buf, "%.0f", v);
        return buf;
    }
    for (int prec = 1; prec <= 17; ++prec) {
        snprintf(buf, sizeof buf, "%.*g", prec, v);
        if (strtod(buf, nullptr) == v) break;
    }
    if (strchr(buf, 'e')) snprintf(buf, sizeof buf, "%.17f", v);
    return buf;
}

std::string fmt_num_f32(float v) {  // {d} of an f32: shortest decimal that round-trips as f32
    char buf[400];
    if (v == std::floor(v) && std::fabs(v) < 1e15f) {
        snprintf(buf, sizeof buf, "%.0f", (double)v);
        return buf;
    }
    for (int prec = 1; prec <= 9; ++prec) {
        snprintf(buf, sizeof buf, "%.*g", prec, (double)v);
        if (strtof(buf, nullptr) == v) break;
    }
    if (strchr(buf, 'e')) snprintf(buf, sizeof buf, "%.9f", (double)v);
    return buf;
}

// hz.getArray(f32, ...) as LimitFilter uses it (src/helper.zig:340-404): values narrowed to f32 before the range tests
bool get_array_f32(const double* src, int n, float def, float lo, float hi, const char* key, const char* name, float out[3]) {
    if (n > 3) { set_error("%s: %s has too many elements (got %d, max 3).", name, key, n); return false; }
    for (int i = 0; i < 3; ++i) {
        if (i < n) out[i] = (float)src[i];
        else if (i == 0) out[i] = def;
        else out[i] = out[i - 1];
        if (out[i] < lo) { set_error("%s: %s value %s is below minimum %s.", name, key, fmt_num_f32(out[i]).c_str(), fmt_num_f32(lo).c_str()); return false; }
        if (out[i] > hi) { set_error("%s: %s value %s is above maximum %s.", name, key, fmt_num_f32(out[i]).c_str(), fmt_num_f32(hi).c_str()); return false; }
    }
    return true;
}

// hz.scaleValue(value, node, .{}) (src/helper.zig:312-338): an 8-bit integer-scale value brought to the clip's depth, f32
float scale_value8(float value, const vszip_video_info& vi, bool limited) {
    if (vi.bits_per_sample == 8) return value;
    const bool flt = vi.sample_type == VSZIP_ST_FLOAT;
    const int bits = vi.bits_per_sample, sh = bits - 8;
    const float full_peak = (float)((1ll << bits) - 1);
    const float in_peak = limited ? 235.0f : 255.0f, in_low = limited ? 16.0f : 0.0f;
    const float out_peak = flt ? 1.0f : (limited ? (float)(235ll << sh) : full_peak);
    const float out_low = flt ? 0.0f : (limited ? (float)(16ll << sh) : 0.0f);
    const float scale = (out_peak - out_low) / (in_peak - in_low);
    float v = value * scale;
    if (!flt) v = std::fmax(std::fmin(std::round(v), full_peak), 0.0f);
    return v;
}

// hz.getArray (src/helper.zig:340-404)
template <class T, class S>
bool get_array(const S* src, int n, T def, double lo, double hi, const char* key, const char* name, T out[3], T (*conv)(S)) {
    if (n > 3) { set_error("%s: %s has too many elements (got %d, max 3).", name, key, n); return false; }
    for (int i = 0; i < 3; ++i) {
        if (i < n) out[i] = conv(src[i]);
        else if (i == 0) out[i] = def;
        else out[i] = out[i - 1];
        if ((double)out[i] < lo) { set_error("%s: %s value %s is below minimum %s.", name, key, fmt_num((double)out[i]).c_str(), fmt_num(lo).c_str()); return false; }
        if ((double)out[i] > hi) { set_error("%s: %s value %s is above maximum %s.", name, key, fmt_num((double)out[i]).c_str(), fmt_num(hi).c_str()); return false; }
    }
    return true;
}

bool basic_vi_ok(const vszip_video_info* vi, const char* name) {
    if (!vi || vi->width <= 0 || vi->height <= 0 || vi->num_planes < 1 || vi->num_planes > 3) {
        set_error("%s: invalid video info", name);
        return false;
    }
    return true;
}

struct SlotGuard {
    DeviceCtx* d;
    Slot* s;
    explicit SlotGuard(DeviceCtx* dd) : d(dd), s(dd->acquire()) {}
    ~SlotGuard() { d->release(s); }
};

DeviceCtx* route(int32_t n, const char* name) {
    DeviceCtx* d = device_for_frame(n);
    if (!d) set_error("%s: vszip_cuda_init has not been called (no GPU context; there is no CPU fallback)", name);
    return d;
}

bool same_clip_format(const vszip_dev_clip* a, const vszip_video_info& vi, SampleKind kind, const char* name) {
    if (!a || a->vi.width != vi.width || a->vi.height != vi.height || a->layout.kind != kind || a->vi.num_planes != vi.num_planes ||
        a->vi.sub_sampling_w != vi.sub_sampling_w || a->vi.sub_sampling_h != vi.sub_sampling_h ||
        a->vi.bits_per_sample != vi.bits_per_sample || a->vi.sample_type != vi.sample_type) {
        set_error("%s: device clip does not match the format the filter was created for", name);
        return false;
    }
    return true;
}

bool same_clip_shape(const vszip_dev_clip* a, const vszip_filter* f, const char* name) { return same_clip_format(a, f->vi, f->sample, name); }

bool range_ok(const vszip_dev_clip* c, int first, int count, const char* name) {
    if (first < 0 || count < 0 || first + count > c->num_frames) { set_error("%s: frame range out of bounds", name); return false; }
    return true;
}

// The checks of a batched call: every clip it reads matches the instance's format and the clip it writes (the last one, when
// `output` is set) the format of the frames it returns (a NULL clip does not match); every clip holds frames [first, first + count),
// and all of them live on one initialised device, which becomes current.  *st: the caller's stream, or that device's batch stream.
int begin_device_call(const vszip_filter* f, const char* name, const vszip_dev_clip* const* clips, int n, int32_t first, int32_t count,
                      void* stream, cudaStream_t* st, bool output = false) {
    for (int i = 0; i < n; ++i) {
        const bool out = output && i == n - 1;
        if (!same_clip_format(clips[i], out ? f->out_vi : f->vi, out ? f->out_layout.kind : f->sample, name)) return -1;
    }
    for (int i = 0; i < n; ++i) if (!range_ok(clips[i], first, count, name)) return -1;
    for (int i = 1; i < n; ++i)
        if (clips[i]->device_index != clips[0]->device_index) { set_error("%s: clips live on different devices", name); return -1; }
    DeviceCtx* d = device_ctx(clips[0]->device_index);
    if (!d) { set_error("%s: library not initialised", name); return -1; }
    VSZ_CUDA(cudaSetDevice(d->ordinal));
    *st = stream ? (cudaStream_t)stream : d->batch_stream;
    return 0;
}

int device_index_of(DeviceCtx* d) {
    for (int i = 0; i < num_devices(); ++i) if (device_ctx(i) == d) return i;
    return 0;
}

bool same_format(const vszip_video_info& a, const vszip_video_info& b) {
    return a.width == b.width && a.height == b.height && a.color_family == b.color_family && a.sample_type == b.sample_type &&
           a.bits_per_sample == b.bits_per_sample && a.sub_sampling_w == b.sub_sampling_w && a.sub_sampling_h == b.sub_sampling_h &&
           a.num_planes == b.num_planes;
}

// The format every create function gives its instance: it reads and returns frames of vi (ColorMap then sets its output format).
void set_format(vszip_filter* f, const vszip_video_info& vi, SampleKind kind) {
    f->vi = f->out_vi = vi;
    f->sample = kind;
    f->layout = f->out_layout = make_layout(vi, kind);
}

// A filter whose output format differs from its input's: it writes every plane of its output.
bool converts(const vszip_filter* f) { return !same_format(f->vi, f->out_vi); }

// The planes of the output frame a pixel filter writes: the ones it processes, or all of them when it changes the format.
void written_planes(const vszip_filter* f, bool w[3]) {
    for (int p = 0; p < 3; ++p) w[p] = converts(f) ? p < f->out_layout.nplanes : f->process[p];
}

int processed_planes(const vszip_filter* f) {
    int k = 0;
    for (int p = 0; p < f->layout.nplanes; ++p) k += f->process[p] ? 1 : 0;
    return k;
}

// What each filter kind takes and gives, indexed by FilterKind - 1.
struct KindInfo {
    const char* name;
    bool pixel;            // has a pixel output (else it measures frame statistics)
    const char* input[2];  // the filter's names for its second and third inputs (nullptr: none)
    bool optional[2];      // an instance may be created without that input
};
constexpr KindInfo kKinds[] = {
    {"BoxBlur", true, {nullptr, nullptr}, {false, false}},
    {"Bilateral", true, {"ref", nullptr}, {true, false}},
    {"PlaneMinMax", false, {"clipb", nullptr}, {true, false}},
    {"PlaneAverage", false, {"clipb", nullptr}, {true, false}},
    {"Limiter", true, {nullptr, nullptr}, {false, false}},
    {"LimitFilter", true, {"src", "ref"}, {false, true}},
    {"AdaptiveBinarize", true, {"clip", nullptr}, {false, false}},
    {"CLAHE", true, {nullptr, nullptr}, {false, false}},
    {"ColorMap", true, {nullptr, nullptr}, {false, false}},
};
static_assert(sizeof kKinds / sizeof kKinds[0] == F_COLORMAP, "one row per FilterKind");

const KindInfo& kind_info(int kind) { return kKinds[kind - 1]; }
bool is_pixel(const vszip_filter* f) { return kind_info(f->kind).pixel; }

// An optional input must be passed exactly when the instance was created with it.  get_frame says "ref frame" / "clipb frame",
// _device "ref clip" / "clipb".
bool inputs_match(const vszip_filter* f, const void* second, const void* third, bool device) {
    const KindInfo& k = kind_info(f->kind);
    const bool given[2] = {second != nullptr, third != nullptr};
    for (int i = 0; i < 2; ++i) {
        if (!k.optional[i] || f->has_input[i] == given[i]) continue;
        const char* noun = !device ? " frame" : (strcmp(k.input[i], "clipb") ? " clip" : "");
        set_error("%s: %s%s presence does not match the filter instance", k.name, k.input[i], noun);
        return false;
    }
    return true;
}

}  // namespace

extern "C" {

void vszip_filter_free(vszip_filter* f) {
    if (!f) return;
    for (size_t d = 0; d < f->gr_dev.size(); ++d) {
        DeviceCtx* ctx = device_ctx((int)d);
        if (ctx) cudaSetDevice(ctx->ordinal);
        for (float* p : f->gr_dev[d]) if (p && cudaFree(p) != cudaSuccess) set_error("vszip_filter_free: cudaFree failed (%s)", cudaGetErrorString(cudaGetLastError()));
        for (float* p : f->gs_dev[d]) if (p && cudaFree(p) != cudaSuccess) set_error("vszip_filter_free: cudaFree failed (%s)", cudaGetErrorString(cudaGetLastError()));
    }
    for (size_t d = 0; d < f->exclude_i_dev.size(); ++d) {
        DeviceCtx* ctx = device_ctx((int)d);
        if (ctx) cudaSetDevice(ctx->ordinal);
        if (f->exclude_i_dev[d]) cudaFree(f->exclude_i_dev[d]);
        if (f->exclude_f_dev[d]) cudaFree(f->exclude_f_dev[d]);
    }
    delete f;
}

int vszip_filter_planes(const vszip_filter* f, int32_t process[3]) {
    for (int i = 0; i < 3; ++i) process[i] = (i < f->vi.num_planes && f->process[i]) ? 1 : 0;
    return 0;
}

int vszip_filter_output_info(const vszip_filter* f, vszip_video_info* out) {
    if (!f || !out) { set_error("vszip_filter_output_info: bad filter handle"); return -1; }
    *out = f->out_vi;
    return 0;
}

// =========================================================================== shared entry-point bodies
// The dispatchers, defined after the filters' own sections.  `in` holds a pixel filter's main input, then its second and third
// (the chain's numbering, whatever order the filter's own entry points take them in); consecutive frames are in_fs bytes apart in
// the inputs and out_fs bytes apart in the output (they differ only for a filter that changes the format).
static int run_pixels(const vszip_filter* f, int dev_index, const char* const in[3], size_t in_fs, char* out, size_t out_fs, int count,
                      cudaStream_t st);
static int run_stats(const vszip_filter* f, int dev_index, const char* a, const char* b, size_t fs, int count, void* scratch,
                     StatsRaw* raw, cudaStream_t st);
static void stats_finalize(const vszip_filter* f, const StatsRaw* raw, void* props, int i);  // into element i of a props array

using Frames = std::array<const vszip_frame*, 3>;
using DevClips = std::array<const vszip_dev_clip*, 3>;

// getFrame of a pixel filter: the inputs staged into slot buffers 0, 1 and 3, the output computed into dev[2] and brought back
// (the planes it writes, in the output format).
static int pixel_get_frame(const vszip_filter* f, int kind, int32_t n, const Frames& in, vszip_frame* dst) {
    const char* name = kind_info(kind).name;
    if (!f || f->kind != kind) { set_error("%s: bad filter handle", name); return -1; }
    if (!inputs_match(f, in[1], in[2], false)) return -1;
    DeviceCtx* d = route(n, name);
    if (!d) return -1;
    SlotGuard g(d);
    Slot* s = g.s;
    VSZ_CUDA(cudaSetDevice(d->ordinal));
    static const int buf[3] = {0, 1, 3};  // the slot buffer of each input
    const size_t bytes = f->layout.frame_stride;
    if (slot_reserve(d, s, 2, f->out_layout.frame_stride)) return -1;
    for (int k = 0; k < 3; ++k)  // the main input always, the others when given
        if ((k == 0 || in[k]) && slot_reserve(d, s, buf[k], bytes)) return -1;
    const char* dev_in[3] = {nullptr, nullptr, nullptr};
    for (int k = 0; k < 3; ++k) {
        if (k > 0 && !in[k]) continue;
        if (stage_in(s, buf[k], f->layout, in[k], f->process)) return -1;
        dev_in[k] = s->dev[buf[k]];
    }
    const int rc = run_pixels(f, device_index_of(d), dev_in, 0, s->dev[2], 0, 1, s->stream);
    if (rc) return rc;
    bool written[3], direct[3];
    written_planes(f, written);
    if (stage_out_begin(s, f->out_layout, dst, written, direct)) return -1;
    VSZ_CUDA(cudaStreamSynchronize(s->stream));
    stage_out_finish(s, f->out_layout, dst, written, direct);
    return 0;
}

// getFrame of PlaneMinMax / PlaneAverage: a (and clipb b) staged into slot buffers 0 (and 1), the sums back through the slot's
// small buffers.
static int stats_get_frame(const vszip_filter* f, int kind, int32_t n, const vszip_frame* a, const vszip_frame* b, void* out) {
    const char* name = kind_info(kind).name;
    if (!f || f->kind != kind) { set_error("%s: bad filter handle", name); return -1; }
    if (!inputs_match(f, b, nullptr, false)) return -1;
    DeviceCtx* d = route(n, name);
    if (!d) return -1;
    SlotGuard g(d);
    Slot* s = g.s;
    VSZ_CUDA(cudaSetDevice(d->ordinal));
    const size_t bytes = f->layout.frame_stride;
    const int np = processed_planes(f);
    const size_t scratch = stats_scratch_bytes(1, np) + 256;
    if (slot_reserve(d, s, 0, bytes) || (b && slot_reserve(d, s, 1, bytes)) || slot_reserve(d, s, 2, scratch)) return -1;
    if (stage_in(s, 0, f->layout, a, f->process)) return -1;
    if (b && stage_in(s, 1, f->layout, b, f->process)) return -1;
    StatsRaw* raw_dev = (StatsRaw*)s->dev_small;
    const int rc = run_stats(f, device_index_of(d), s->dev[0], b ? s->dev[1] : nullptr, 0, 1, s->dev[2], raw_dev, s->stream);
    if (rc) return rc;
    VSZ_CUDA(cudaMemcpyAsync(s->pin_small, raw_dev, sizeof(StatsRaw) * np, cudaMemcpyDeviceToHost, s->stream));
    VSZ_CUDA(cudaStreamSynchronize(s->stream));
    stats_finalize(f, (const StatsRaw*)s->pin_small, out, 0);
    return 0;
}

// The batched entry points' checks, in one order: the handle, the optional inputs, then every clip the call reads or writes (a
// required input that is NULL fails as a clip of the wrong format).  dst: the pixel output, unused for statistics.
static int device_call(const vszip_filter* f, int kind, const DevClips& in, const vszip_dev_clip* dst, int32_t first, int32_t count,
                       void* stream, cudaStream_t* st) {
    const KindInfo& k = kind_info(kind);
    if (!f || f->kind != kind) { set_error("%s: bad filter handle", k.name); return -1; }
    if (!inputs_match(f, in[1], in[2], true)) return -1;
    const vszip_dev_clip* clips[4] = {in[0]};
    int n = 1;
    for (int i = 0; i < 2; ++i) if (f->has_input[i]) clips[n++] = in[i + 1];
    if (k.pixel) clips[n++] = dst;
    return begin_device_call(f, k.name, clips, n, first, count, stream, st, k.pixel);
}

static int pixel_device(const vszip_filter* f, int kind, const DevClips& in, vszip_dev_clip* dst, int32_t first, int32_t count, void* stream) {
    cudaStream_t st;
    if (device_call(f, kind, in, dst, first, count, stream, &st)) return -1;
    const char* p[3];
    for (int k = 0; k < 3; ++k) p[k] = in[k] ? in[k]->base + (size_t)first * in[k]->layout.frame_stride : nullptr;
    const size_t out_fs = dst->layout.frame_stride;
    return run_pixels(f, dst->device_index, p, in[0]->layout.frame_stride, dst->base + (size_t)first * out_fs, out_fs, count, st);
}

static int stats_device(const vszip_filter* f, int kind, const vszip_dev_clip* a, const vszip_dev_clip* b, int32_t first, int32_t count,
                        void* out, void* stream) {
    cudaStream_t st;
    if (device_call(f, kind, {a, b, nullptr}, nullptr, first, count, stream, &st)) return -1;
    const int np = processed_planes(f);
    if (count == 0 || np == 0) return 0;
    const size_t fs = a->layout.frame_stride;
    AsyncScratch scratch_mem;
    const size_t sb = stats_scratch_bytes(count, np), rb = sizeof(StatsRaw) * (size_t)count * np;
    VSZ_CUDA(scratch_mem.alloc(sb + rb, st));
    StatsRaw* raw_dev = (StatsRaw*)(scratch_mem.p + sb);
    const int rc = run_stats(f, a->device_index, a->base + (size_t)first * fs, b ? b->base + (size_t)first * fs : nullptr, fs, count,
                             scratch_mem.p, raw_dev, st);
    if (!rc && out) {
        std::vector<StatsRaw> raw((size_t)count * np);
        VSZ_CUDA(cudaMemcpyAsync(raw.data(), raw_dev, rb, cudaMemcpyDeviceToHost, st));
        VSZ_CUDA(cudaStreamSynchronize(st));
        for (int i = 0; i < count; ++i) stats_finalize(f, raw.data() + (size_t)i * np, out, i);
    }
    return rc;
}

// =========================================================================== BoxBlur
vszip_filter* vszip_boxblur_create(const vszip_video_info* vi, const vszip_boxblur_args* a) {
    static const char* name = "BoxBlur";
    if (!basic_vi_ok(vi, name)) return nullptr;
    SampleKind kind;
    if (!select_kind(*vi, name, false, &kind)) return nullptr;
    bool process[3] = {true, true, true};
    if (!parse_planes(a->planes, a->num_planes, vi->num_planes, name, process)) return nullptr;
    const uint32_t hr = a->has_hradius ? sat_u32(a->hradius) : 1u;
    const uint32_t vr = a->has_vradius ? sat_u32(a->vradius) : 1u;
    const int32_t hp = a->has_hpasses ? sat_i32(a->hpasses) : 1;
    const int32_t vp = a->has_vpasses ? sat_i32(a->vpasses) : 1;
    const bool vblur = vr > 0 && vp > 0, hblur = hr > 0 && hp > 0;
    if (!vblur && !hblur) { set_error("BoxBlur: nothing to be performed"); return nullptr; }
    // the comptime kernel blurs both axes with `hradius` whenever it is selected (boxblur.zig:188),
    // so the size checks must hold for both axes there
    const bool use_rt = (hr != vr) || (hr > 22) || (hp > 1) || (vp > 1);
    for (int p = 0; p < vi->num_planes; ++p) {
        if (!process[p]) continue;
        const uint32_t pw = (uint32_t)vi->width >> (p ? vi->sub_sampling_w : 0);
        const uint32_t ph = (uint32_t)vi->height >> (p ? vi->sub_sampling_h : 0);
        if ((hblur || !use_rt) && (uint64_t)hr * 2 >= pw) { set_error("BoxBlur: hradius too large; 2*hradius must be < the (smallest processed) plane width."); return nullptr; }
        if ((vblur || !use_rt) && (uint64_t)vr * 2 >= ph) { set_error("BoxBlur: vradius too large; 2*vradius must be < the (smallest processed) plane height."); return nullptr; }
    }
    vszip_filter* f = new vszip_filter();
    f->kind = F_BOXBLUR;
    set_format(f, *vi, kind);
    for (int i = 0; i < 3; ++i) f->process[i] = process[i] && i < vi->num_planes;
    f->hradius = hr; f->vradius = vr; f->hpasses = hp; f->vpasses = vp;
    return f;
}

int vszip_boxblur_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, vszip_frame* dst) {
    return pixel_get_frame(f, F_BOXBLUR, n, {src, nullptr, nullptr}, dst);
}

int vszip_boxblur_device(const vszip_filter* f, const vszip_dev_clip* src, vszip_dev_clip* dst, int32_t first, int32_t count, void* stream) {
    return pixel_device(f, F_BOXBLUR, {src, nullptr, nullptr}, dst, first, count, stream);
}

// =========================================================================== Bilateral
vszip_filter* vszip_bilateral_create(const vszip_video_info* vi, const vszip_video_info* ref_vi, const vszip_bilateral_args* a) {
    static const char* name = "Bilateral";
    if (!basic_vi_ok(vi, name)) return nullptr;
    SampleKind kind;
    if (!select_kind(*vi, name, false, &kind)) return nullptr;
    vszip_filter* f = new vszip_filter();
    auto fail = [&]() { vszip_filter_free(f); return (vszip_filter*)nullptr; };
    f->kind = F_BILATERAL;
    set_format(f, *vi, kind);
    const bool yuv = vi->color_family == VSZIP_CF_YUV;
    f->hist_len = vi->sample_type == VSZIP_ST_INTEGER ? (1 << vi->bits_per_sample) : 65536;  // hz.getHistLen
    f->peak = (float)(f->hist_len - 1);

    double sigmaS[3], sigmaR[3];
    int32_t algorithm[3];
    uint32_t pbfic[3];
    for (int i = 0; i < 3; ++i) {  // bilateral.zig:104-125
        if (i < a->num_sigmaS) sigmaS[i] = a->sigmaS[i];
        else if (i == 0) sigmaS[0] = 3.0;
        else if (i == 1 && yuv && vi->sub_sampling_h != 0 && vi->sub_sampling_w != 0)
            sigmaS[1] = sigmaS[0] / std::sqrt((double)((1u << vi->sub_sampling_h) * (1u << vi->sub_sampling_w)));
        else sigmaS[i] = sigmaS[i - 1];
        if (sigmaS[i] < 0) { set_error("Bilateral: Invalid \"sigmaS\" assigned, must be non-negative float number"); return fail(); }
    }
    if (!get_array<double, double>(a->sigmaR, a->num_sigmaR, 0.02, 0.0, std::numeric_limits<double>::max(), "sigmaR", name, sigmaR, [](double v) { return v; })) return fail();
    if (!get_array<int32_t, int64_t>(a->algorithm, a->num_algorithm, 0, 0, 2, "algorithm", name, algorithm, [](int64_t v) { return sat_i32(v); })) return fail();
    if (!get_array<uint32_t, int64_t>(a->PBFICnum, a->num_PBFICnum, 0u, 0, 256, "PBFICnum", name, pbfic, [](int64_t v) { return sat_u32(v); })) return fail();
    bool process[3] = {true, true, true};
    if (!parse_planes(a->planes, a->num_planes, vi->num_planes, name, process)) return fail();
    for (int i = 0; i < 3; ++i)
        if (sigmaS[i] == 0 || sigmaR[i] == 0) process[i] = false;
    for (int i = 0; i < 3; ++i)
        if (pbfic[i] == 1) { set_error("Bilateral: Invalid \"PBFICnum\" assigned, must be integer ranges in [0,256] except 1"); return fail(); }
    for (int i = 0; i < 3; ++i) {  // bilateral.zig:147-162
        if (process[i] && pbfic[i] == 0) {
            if (sigmaR[i] >= 0.08) pbfic[i] = 4;
            else if (sigmaR[i] >= 0.015) pbfic[i] = std::min(16u, (uint32_t)std::trunc(4 * 0.08 / sigmaR[i] + 0.5));
            else pbfic[i] = std::min(32u, (uint32_t)std::trunc(16 * 0.015 / sigmaR[i] + 0.5));
            if (i > 0 && yuv && (pbfic[i] % 2 == 0) && pbfic[i] < 256) pbfic[i] += 1;
        }
    }
    for (int i = 0; i < 3; ++i) {  // bilateral.zig:164-199
        BilateralPlane& b = f->bl[i];
        b.sigmaS = sigmaS[i]; b.sigmaR = sigmaR[i]; b.algorithm = algorithm[i]; b.pbfic = pbfic[i];
        if (!process[i]) continue;
        const int orad = std::max((int)std::trunc(sigmaS[i] * 2 + 0.5), 1);
        b.step = orad < 4 ? 1 : (orad < 8 ? 2 : 3);
        b.samples = 1;
        b.radius = 1 + (b.samples - 1) * b.step;
        while (orad * 2 > (int)b.radius * 3) {
            b.samples += 1;
            b.radius = 1 + (b.samples - 1) * b.step;
            if ((int)b.radius >= orad && b.samples > 2) {
                b.samples -= 1;
                b.radius = 1 + (b.samples - 1) * b.step;
                break;
            }
        }
        if (b.algorithm <= 0)
            b.algorithm = (b.step == 1) ? 2 : ((sigmaR[i] < 0.08 && b.samples < 5) ? 2 : ((4 * b.samples * b.samples <= 15 * b.pbfic) ? 2 : 1));
    }
    for (int i = 0; i < vi->num_planes; ++i) {  // bilateral.zig:201-214
        if (process[i] && f->bl[i].algorithm == 2) {
            const uint32_t pw = (uint32_t)vi->width >> (i ? vi->sub_sampling_w : 0);
            const uint32_t ph = (uint32_t)vi->height >> (i ? vi->sub_sampling_h : 0);
            if (pw <= 2 * f->bl[i].radius || ph <= 2 * f->bl[i].radius) {
                set_error("Bilateral: plane too small for the spatial radius derived from sigmaS; lower sigmaS or use a larger clip.");
                return fail();
            }
        }
    }
    if (ref_vi && !compare_nodes(*vi, *ref_vi, name)) return fail();
    for (int i = 0; i < 3; ++i) f->process[i] = process[i] && i < vi->num_planes;
    f->has_input[0] = ref_vi != nullptr;
    // LUTs (src/filters/bilateral.zig:306-334), f64 math rounded to f32, uploaded to every device
    f->gs_host.resize(3); f->gr_host.resize(3);
    for (int i = 0; i < vi->num_planes; ++i) {
        if (!f->process[i]) continue;
        BilateralPlane& b = f->bl[i];
        const int upper = (int)b.radius + 1;
        f->gs_host[i].resize((size_t)upper * upper);
        for (int y = 0; y < upper; ++y)
            for (int x = 0; x < upper; ++x)
                f->gs_host[i][(size_t)y * upper + x] = (float)std::exp((double)(x * x + y * y) / (b.sigmaS * b.sigmaS * -2.0));
        const double range = (double)f->peak;
        const uint32_t top = (uint32_t)std::trunc(std::min(range, b.sigmaR * 8.0 * range + 0.5));
        const double norm = std::sqrt(2.0 * M_PI) * b.sigmaR;
        std::vector<float>& gr = f->gr_host[i];
        gr.resize((size_t)f->hist_len);
        uint32_t j = 0;
        for (; j <= top && j < (uint32_t)f->hist_len; ++j) {
            const double xx = ((double)j / range) / b.sigmaR;
            gr[j] = (float)(std::exp(xx * xx / -2.0) / norm);
        }
        const float tail = gr[std::min<uint32_t>(top, (uint32_t)f->hist_len - 1)];
        for (; j < (uint32_t)f->hist_len; ++j) gr[j] = tail;
        b.lut_len = (int)std::min<uint32_t>(top + 1, (uint32_t)f->hist_len);
        b.exact = (b.algorithm == 1) ? 1 : bilateral_weights_exact(b.lut_len);  // PBFIC always gathers the full LUT
    }
    return f;
}

int vszip_bilateral_get_info(const vszip_filter* f, vszip_bilateral_info* o) {
    if (!f || f->kind != F_BILATERAL) { set_error("Bilateral: bad filter handle"); return -1; }
    for (int i = 0; i < 3; ++i) {
        const BilateralPlane& b = f->bl[i];
        o->sigmaS[i] = b.sigmaS; o->sigmaR[i] = b.sigmaR; o->process[i] = f->process[i]; o->algorithm[i] = b.algorithm;
        o->PBFICnum[i] = b.pbfic; o->radius[i] = b.radius; o->samples[i] = b.samples; o->step[i] = b.step; o->exact_lut[i] = b.exact;
    }
    return 0;
}

// The weight tables are uploaded to a device the first time the instance runs there (create itself
// stays GPU-free so argument validation works anywhere).
static int bilateral_upload(const vszip_filter* cf, int dev_index) {
    vszip_filter* f = const_cast<vszip_filter*>(cf);
    std::lock_guard<std::mutex> lk(f->lut_mu);
    if (f->gr_dev.size() < (size_t)num_devices()) {
        f->gr_dev.resize(num_devices(), std::vector<float*>(3, nullptr));
        f->gs_dev.resize(num_devices(), std::vector<float*>(3, nullptr));
    }
    bool uploaded = false;
    for (int i = 0; i < f->vi.num_planes; ++i) {
        if (!f->process[i] || f->gr_dev[dev_index][i]) continue;
        const size_t gsb = f->gs_host[i].size() * sizeof(float), grb = f->gr_host[i].size() * sizeof(float);
        float *gs = nullptr, *gr = nullptr;
        // the pointers are published only after the copies have landed: the kernels run on non-blocking streams, which
        // are not ordered after a pageable cudaMemcpy on the default stream by themselves
        if (cudaMalloc((void**)&gs, gsb) != cudaSuccess || cudaMalloc((void**)&gr, grb) != cudaSuccess ||
            cudaMemcpy(gs, f->gs_host[i].data(), gsb, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(gr, f->gr_host[i].data(), grb, cudaMemcpyHostToDevice) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
            set_error("Bilateral: uploading the weight tables failed (%s)", cudaGetErrorString(cudaGetLastError()));
            cudaFree(gs); cudaFree(gr);
            return -1;
        }
        f->gs_dev[dev_index][i] = gs;
        f->gr_dev[dev_index][i] = gr;
        uploaded = true;
    }
    (void)uploaded;
    return 0;
}

static BilateralLaunch bilateral_launch(const vszip_filter* f, int dev_index) {
    BilateralLaunch bp{};
    bp.peak = f->peak;
    for (int i = 0; i < 3; ++i) {
        bp.gs[i] = f->gs_dev[dev_index][i]; bp.gr[i] = f->gr_dev[dev_index][i];
        bp.radius[i] = (int)f->bl[i].radius; bp.step[i] = (int)f->bl[i].step; bp.lut_len[i] = f->bl[i].lut_len;
        if (f->process[i]) {
            const double s = (double)f->peak * f->bl[i].sigmaR;
            bp.c2[i] = (float)(-1.4426950408889634 / (2.0 * s * s));
            bp.cnorm[i] = (float)(1.0 / (std::sqrt(2.0 * M_PI) * f->bl[i].sigmaR));
        }
    }
    return bp;
}

// Algorithm 2 planes go through the tiled kernel in one launch; algorithm 1 (PBFIC) planes one plane at a time.
static int bilateral_run(const vszip_filter* f, int dev_index, const char* src, size_t sfs, const char* ref, size_t rfs, char* dst,
                         size_t dfs, int count, cudaStream_t st) {
    bool mask2[3] = {false, false, false}, any2 = false;
    for (int i = 0; i < 3; ++i) { mask2[i] = f->process[i] && f->bl[i].algorithm == 2; any2 = any2 || mask2[i]; }
    if (any2) {
        const BilateralLaunch bp = bilateral_launch(f, dev_index);
        const int rc = run_bilateral(f->layout, mask2, src, sfs, ref, rfs, dst, dfs, count, bp, st);
        if (rc) return rc;
    }
    for (int i = 0; i < 3; ++i) {
        if (!f->process[i] || f->bl[i].algorithm != 1) continue;
        const int rc = run_pbfic(f->layout, i, src, sfs, ref, rfs, dst, dfs, count, f->gr_dev[dev_index][i], f->hist_len, f->bl[i].sigmaS,
                                 (int)f->bl[i].pbfic, f->peak, st);
        if (rc) return rc;
    }
    return 0;
}

int vszip_bilateral_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, const vszip_frame* ref, vszip_frame* dst) {
    return pixel_get_frame(f, F_BILATERAL, n, {src, ref, nullptr}, dst);
}

int vszip_bilateral_device(const vszip_filter* f, const vszip_dev_clip* src, const vszip_dev_clip* ref, vszip_dev_clip* dst,
                           int32_t first, int32_t count, void* stream) {
    return pixel_device(f, F_BILATERAL, {src, ref, nullptr}, dst, first, count, stream);
}

// =========================================================================== PlaneMinMax
vszip_filter* vszip_planeminmax_create(const vszip_video_info* vi, const vszip_video_info* clipb_vi, const vszip_planeminmax_args* a) {
    static const char* name = "PlaneMinMax";
    if (!basic_vi_ok(vi, name)) return nullptr;
    SampleKind kind;
    if (!select_kind(*vi, name, false, &kind)) return nullptr;
    if (clipb_vi && !compare_nodes(*vi, *clipb_vi, name)) return nullptr;
    bool process[3] = {true, false, false};
    if (!parse_planes(a->planes, a->num_planes, vi->num_planes, name, process)) return nullptr;
    const uint32_t hist_size = vi->sample_type == VSZIP_ST_FLOAT ? 65536u : (1u << vi->bits_per_sample);
    // getThr (planeminmax.zig:174-192): maxthr is read first
    const float maxthr = a->has_maxthr ? (float)a->maxthr : 0.0f;
    if (maxthr < 0 || maxthr > 1) { set_error("PlaneMinMax: maxthr should be a float between 0.0 and 1.0"); return nullptr; }
    const float minthr = a->has_minthr ? (float)a->minthr : 0.0f;
    if (minthr < 0 || minthr > 1) { set_error("PlaneMinMax: minthr should be a float between 0.0 and 1.0"); return nullptr; }
    const bool no_thr = maxthr == 0 && minthr == 0;
    const bool do_chroma = process[1] || process[2];
    if (do_chroma && !no_thr && vi->color_family == VSZIP_CF_YUV && vi->sample_type == VSZIP_ST_FLOAT) {
        set_error("PlaneMinMax: you can't use maxthr/minthr with float chroma, use planes=[0] or maxthr/minthr=0");
        return nullptr;
    }
    vszip_filter* f = new vszip_filter();
    f->kind = F_PLANEMINMAX;
    set_format(f, *vi, kind);
    for (int i = 0; i < 3; ++i) f->process[i] = process[i] && i < vi->num_planes;
    f->has_input[0] = clipb_vi != nullptr;
    f->minthr = minthr; f->maxthr = maxthr; f->hist_size = hist_size; f->no_thr = no_thr;
    return f;
}

static void minmax_finalize(const vszip_filter* f, const StatsRaw* raw, vszip_minmax_props* out) {
    const bool flt = f->sample == K_F16 || f->sample == K_F32;
    memset(out, 0, sizeof *out);
    out->is_float = flt; out->has_diff = f->has_input[0];
    const float peakf = (float)(f->hist_size - 1);  // planeminmax.zig:118-119
    int k = 0;
    for (int p = 0; p < f->layout.nplanes; ++p) {
        if (!f->process[p]) continue;
        const StatsRaw& r = raw[k];
        out->plane[k] = p;
        if (f->no_thr) {
            out->imin[k] = r.bin_min; out->imax[k] = r.bin_max;
            out->fmin[k] = (double)r.fmin; out->fmax[k] = (double)r.fmax;
        } else {
            out->imin[k] = r.bin_min; out->imax[k] = r.bin_max;
            out->fmin[k] = (double)((float)r.bin_min / 65535.0f);  // src/filters/planeminmax.zig:62-63
            out->fmax[k] = (double)((float)r.bin_max / 65535.0f);
        }
        if (f->has_input[0]) {
            const double total = (double)((uint32_t)f->layout.pl[p].w * (uint32_t)f->layout.pl[p].h);
            out->diff[k] = flt ? r.fdiff / total : (double)r.idiff / total / (double)peakf;
        }
        ++k;
    }
    out->count = k;
}

int vszip_planeminmax_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* a, const vszip_frame* b, vszip_minmax_props* out) {
    return stats_get_frame(f, F_PLANEMINMAX, n, a, b, out);
}

int vszip_planeminmax_device(const vszip_filter* f, const vszip_dev_clip* a, const vszip_dev_clip* b, int32_t first, int32_t count,
                             vszip_minmax_props* out, void* stream) {
    return stats_device(f, F_PLANEMINMAX, a, b, first, count, out, stream);
}

// =========================================================================== PlaneAverage
vszip_filter* vszip_planeaverage_create(const vszip_video_info* vi, const vszip_video_info* clipb_vi, const vszip_planeaverage_args* a) {
    static const char* name = "PlaneAverage";
    if (!basic_vi_ok(vi, name)) return nullptr;
    if (a->num_exclude < 0 || (a->num_exclude > 0 && !a->exclude)) {  // VapourSynth rejects a missing non-opt argument itself
        set_error("PlaneAverage: argument exclude is required");
        return nullptr;
    }
    const bool u32 = vi->sample_type == VSZIP_ST_INTEGER && vi->bytes_per_sample == 4;
    SampleKind kind = K_U16;
    if (!u32 && !select_kind(*vi, name, true, &kind)) return nullptr;
    if (clipb_vi && !compare_nodes(*vi, *clipb_vi, name)) return nullptr;
    bool process[3] = {true, false, false};
    if (!parse_planes(a->planes, a->num_planes, vi->num_planes, name, process)) return nullptr;
    if (u32) { set_error("PlaneAverage: exclude is not supported for 32-bit integer clips."); return nullptr; }
    vszip_filter* f = new vszip_filter();
    f->kind = F_PLANEAVERAGE;
    set_format(f, *vi, kind);
    for (int i = 0; i < 3; ++i) f->process[i] = process[i] && i < vi->num_planes;
    f->has_input[0] = clipb_vi != nullptr;
    f->avg_peak = (float)((1ull << vi->bits_per_sample) - 1ull);  // planeaverage.zig:112
    for (int i = 0; i < a->num_exclude; ++i) {
        f->exclude_f.push_back((float)a->exclude[i]);           // planeaverage.zig:122-125
        f->exclude_i.push_back(sat_i32(a->exclude[i]));         // math.lossyCast(i32, ..)
    }
    return f;
}

// Exclude lists longer than the 16 entries that travel in the kernel arguments are uploaded to a device the first
// time the instance runs there.
static int average_upload(const vszip_filter* cf, int dev_index, const int32_t** xi, const float** xf) {
    *xi = nullptr; *xf = nullptr;
    if (cf->exclude_i.size() <= 16) return 0;
    vszip_filter* f = const_cast<vszip_filter*>(cf);
    std::lock_guard<std::mutex> lk(f->lut_mu);
    if (f->exclude_i_dev.size() < (size_t)num_devices()) { f->exclude_i_dev.resize(num_devices(), nullptr); f->exclude_f_dev.resize(num_devices(), nullptr); }
    if (!f->exclude_i_dev[dev_index]) {
        const size_t n = f->exclude_i.size();
        int32_t* di = nullptr;
        float* df = nullptr;
        // published only once the copies have landed (the reductions run on non-blocking streams)
        if (cudaMalloc((void**)&di, n * sizeof(int32_t)) != cudaSuccess || cudaMalloc((void**)&df, n * sizeof(float)) != cudaSuccess ||
            cudaMemcpy(di, f->exclude_i.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(df, f->exclude_f.data(), n * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
            set_error("PlaneAverage: uploading the exclude list failed (%s)", cudaGetErrorString(cudaGetLastError()));
            cudaFree(di); cudaFree(df);
            return -1;
        }
        f->exclude_i_dev[dev_index] = di;
        f->exclude_f_dev[dev_index] = df;
    }
    *xi = f->exclude_i_dev[dev_index]; *xf = f->exclude_f_dev[dev_index];
    return 0;
}

static void average_finalize(const vszip_filter* f, const StatsRaw* raw, vszip_average_props* out) {
    const bool flt = f->sample == K_F16 || f->sample == K_F32;
    memset(out, 0, sizeof *out);
    out->has_diff = f->has_input[0];
    int k = 0;
    for (int p = 0; p < f->layout.nplanes; ++p) {
        if (!f->process[p]) continue;
        const StatsRaw& r = raw[k];
        out->plane[k] = p;
        const uint32_t all = (uint32_t)f->layout.pl[p].w * (uint32_t)f->layout.pl[p].h;
        const double total = (double)(all - r.excluded);
        // result() (src/filters/planeaverage.zig:16-24)
        if (total == 0) out->avg[k] = 0.0;
        else if (flt) out->avg[k] = r.fsum / total;
        else out->avg[k] = (double)r.isum / total / (double)f->avg_peak;
        if (f->has_input[0]) out->diff[k] = flt ? r.fdiff / (double)all : (double)r.idiff / (double)all / (double)f->avg_peak;
        ++k;
    }
    out->count = k;
}

int vszip_planeaverage_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* a, const vszip_frame* b, vszip_average_props* out) {
    return stats_get_frame(f, F_PLANEAVERAGE, n, a, b, out);
}

int vszip_planeaverage_device(const vszip_filter* f, const vszip_dev_clip* a, const vszip_dev_clip* b, int32_t first, int32_t count,
                              vszip_average_props* out, void* stream) {
    return stats_device(f, F_PLANEAVERAGE, a, b, first, count, out, stream);
}

// =========================================================================== dispatch
static int run_pixels(const vszip_filter* f, int dev_index, const char* const in[3], size_t in_fs, char* out, size_t out_fs, int count,
                      cudaStream_t st) {
    const FrameLayout& l = f->layout;
    const size_t fs = in_fs;  // every filter but ColorMap: out_fs == in_fs
    switch (f->kind) {
        case F_BOXBLUR:
            return run_boxblur(l, f->process, in[0], fs, out, fs, count, (int)f->hradius, f->hpasses, (int)f->vradius, f->vpasses, st);
        case F_BILATERAL:
            if (bilateral_upload(f, dev_index)) return -1;
            return bilateral_run(f, dev_index, in[0], fs, in[1], fs, out, fs, count, st);
        case F_LIMITER:
            return run_limiter(l, f->process, in[0], fs, out, fs, count, f->lim_lo, f->lim_hi, st);
        case F_LIMITFILTER:  // flt = the main input, src = the second, ref = the third
            return run_limitfilter(l, f->process, in[0], fs, in[1], fs, in[2], fs, out, fs, count, f->lf_dark, f->lf_bright, f->lf_elast, st);
        case F_CLAHE:
            return run_clahe(l, f->process, in[0], fs, out, fs, count, f->clahe_hs, f->clahe_limit, f->clahe_tiles[0], f->clahe_tiles[1], st);
        case F_COLORMAP:
            return run_colormap(l, in[0], in_fs, f->out_layout, out, out_fs, count, f->cmap_lut, st);
        default:  // AdaptiveBinarize: clip = the second input, clip2 = the main one
            return run_adaptivebinarize(l, in[1], fs, in[0], fs, out, fs, count, f->ab_c, st);
    }
}

static int run_stats(const vszip_filter* f, int dev_index, const char* a, const char* b, size_t fs, int count, void* scratch,
                     StatsRaw* raw, cudaStream_t st) {
    if (f->kind == F_PLANEMINMAX)
        return run_planeminmax(f->layout, f->process, a, fs, b, fs, count, f->no_thr, f->minthr, f->maxthr, f->hist_size, scratch, raw, st);
    const int32_t* xi; const float* xf;
    if (average_upload(f, dev_index, &xi, &xf)) return -1;
    return run_planeaverage(f->layout, f->process, a, fs, b, fs, count, f->exclude_i.data(), f->exclude_f.data(), (int)f->exclude_i.size(),
                            xi, xf, scratch, raw, st);
}

static void stats_finalize(const vszip_filter* f, const StatsRaw* raw, void* props, int i) {
    if (f->kind == F_PLANEMINMAX) minmax_finalize(f, raw, (vszip_minmax_props*)props + i);
    else average_finalize(f, raw, (vszip_average_props*)props + i);
}

// =========================================================================== PlaneMinMax + PlaneAverage from one read (SURVEY 8f rank 4)
// A PlaneMinMax and a PlaneAverage (either order) that one read can serve: the same planes, at least one of them, and an exclude
// list short enough for the fused kernels.
static bool stats_pair(const vszip_filter* x, const vszip_filter* y) {
    if (!((x->kind == F_PLANEMINMAX && y->kind == F_PLANEAVERAGE) || (x->kind == F_PLANEAVERAGE && y->kind == F_PLANEMINMAX))) return false;
    const vszip_filter* fa = x->kind == F_PLANEAVERAGE ? x : y;
    return x->process[0] == y->process[0] && x->process[1] == y->process[1] && x->process[2] == y->process[2] && processed_planes(x) > 0 &&
           fa->exclude_i.size() <= 16;
}

// PlaneMinMax and PlaneAverage, f and g in either order, over the same frames a; each reads the clipb b if it was created with it.
// One read when both read b (or neither does) and run_planestats_fused takes the pair (then *fused is set, if given), else f and
// then g on their own, in scratch_f and scratch_g.
static int run_stats_pair(const vszip_filter* f, const vszip_filter* g, int dev_index, const char* a, const char* b, size_t fs, int count,
                          bool same_float_sums, char* scratch_f, char* scratch_g, StatsRaw* raw_f, StatsRaw* raw_g, cudaStream_t st,
                          bool* fused) {
    const char* bf = f->has_input[0] ? b : nullptr;
    const char* bg = g->has_input[0] ? b : nullptr;
    if (stats_pair(f, g) && bf == bg) {
        const vszip_filter* fm = f->kind == F_PLANEMINMAX ? f : g;
        const vszip_filter* fa = f->kind == F_PLANEMINMAX ? g : f;
        const int rc = run_planestats_fused(fm->layout, fm->process, a, fs, bf, fs, count, fm->no_thr, fm->minthr, fm->maxthr, fm->hist_size,
                                            fa->exclude_i.data(), fa->exclude_f.data(), (int)fa->exclude_i.size(), same_float_sums, scratch_f,
                                            fm == f ? raw_f : raw_g, fm == f ? raw_g : raw_f, st);
        if (rc == 0 && fused) *fused = true;
        if (rc != 1) return rc;
    }
    int rc = 0;  // not eligible: the two reductions one after the other (two reads)
    if (processed_planes(f)) rc = run_stats(f, dev_index, a, bf, fs, count, scratch_f, raw_f, st);
    if (!rc && processed_planes(g)) rc = run_stats(g, dev_index, a, bg, fs, count, scratch_g, raw_g, st);
    return rc;
}

// b: the clipb clip (may be nullptr); a filter created without clipb ignores it.
static int planestats_run(const vszip_filter* fm, const vszip_filter* fa, const vszip_dev_clip* a, const vszip_dev_clip* b, int32_t first,
                          int32_t count, bool same_float_sums, vszip_minmax_props* mm_out, vszip_average_props* avg_out, int32_t* fused_out,
                          void* stream) {
    static const char* name = "PlaneStats";
    const vszip_dev_clip* clips[2] = {a, b};
    cudaStream_t st;
    if (!same_clip_shape(a, fa, name) || begin_device_call(fm, name, clips, b ? 2 : 1, first, count, stream, &st)) return -1;
    const int npm = processed_planes(fm), npa = processed_planes(fa);
    if (count == 0) return 0;
    const size_t fs = a->layout.frame_stride;
    const size_t sbm = stats_scratch_bytes(count, std::max(npm, 1)), sba = stats_scratch_bytes(count, std::max(npa, 1));
    const size_t rbm = sizeof(StatsRaw) * (size_t)count * npm, rba = sizeof(StatsRaw) * (size_t)count * npa;
    const size_t rbm_al = (rbm + 255) & ~(size_t)255;
    AsyncScratch scratch_mem;
    VSZ_CUDA(scratch_mem.alloc(sbm + sba + rbm_al + rba + 256, st));
    char* scratch = scratch_mem.p;
    StatsRaw* raw_m = (StatsRaw*)(scratch + sbm + sba);
    StatsRaw* raw_a = (StatsRaw*)(scratch + sbm + sba + rbm_al);
    bool fused = false;
    const int rc = run_stats_pair(fm, fa, a->device_index, a->base + (size_t)first * fs, b ? b->base + (size_t)first * fs : nullptr, fs, count,
                                  same_float_sums, scratch, scratch + sbm, raw_m, raw_a, st, &fused);
    if (fused && fused_out) *fused_out = 1;
    if (!rc && (mm_out || avg_out)) {
        std::vector<StatsRaw> hm((size_t)count * npm), ha((size_t)count * npa);
        if (mm_out && npm) VSZ_CUDA(cudaMemcpyAsync(hm.data(), raw_m, rbm, cudaMemcpyDeviceToHost, st));
        if (avg_out && npa) VSZ_CUDA(cudaMemcpyAsync(ha.data(), raw_a, rba, cudaMemcpyDeviceToHost, st));
        VSZ_CUDA(cudaStreamSynchronize(st));
        for (int i = 0; i < count; ++i) {
            if (mm_out) minmax_finalize(fm, hm.data() + (size_t)i * npm, mm_out + i);
            if (avg_out) average_finalize(fa, ha.data() + (size_t)i * npa, avg_out + i);
        }
    }
    return rc;
}

int vszip_planestats_device(const vszip_filter* fm, const vszip_filter* fa, const vszip_dev_clip* a, int32_t first, int32_t count,
                            vszip_minmax_props* mm_out, vszip_average_props* avg_out, int32_t* fused_out, void* stream) {
    if (fused_out) *fused_out = 0;
    if (!fm || fm->kind != F_PLANEMINMAX || !fa || fa->kind != F_PLANEAVERAGE) { set_error("PlaneStats: a PlaneMinMax and a PlaneAverage handle are required"); return -1; }
    if (fm->has_input[0] || fa->has_input[0]) { set_error("PlaneStats: filters created with clipb cannot be combined"); return -1; }
    return planestats_run(fm, fa, a, nullptr, first, count, false, mm_out, avg_out, fused_out, stream);
}

int vszip_planestats_device_b(const vszip_filter* fm, const vszip_filter* fa, const vszip_dev_clip* a, const vszip_dev_clip* b, int32_t first,
                              int32_t count, vszip_minmax_props* mm_out, vszip_average_props* avg_out, int32_t* fused_out, void* stream) {
    if (fused_out) *fused_out = 0;
    if (!fm || fm->kind != F_PLANEMINMAX || !fa || fa->kind != F_PLANEAVERAGE) { set_error("PlaneStats: a PlaneMinMax and a PlaneAverage handle are required"); return -1; }
    if ((fm->has_input[0] || fa->has_input[0]) != (b != nullptr)) { set_error("PlaneStats: clipb presence does not match the filter instances"); return -1; }
    return planestats_run(fm, fa, a, b, first, count, true, mm_out, avg_out, fused_out, stream);
}

// =========================================================================== Limiter
// Range tables of src/filters/limiter.zig:66-91: [lo|hi][plane] for full / tv-range YUV / tv-range RGB at 8 bits;
// deeper integer formats are the 8-bit values shifted left by (bits - 8), full range is (1 << bits) - 1.
static void limiter_table(const vszip_video_info& vi, bool tv_range, bool yuv, double lo[3], double hi[3]) {
    if (vi.sample_type == VSZIP_ST_FLOAT) {  // floats ignore tv_range (limiter.zig:53-54 of the filter file)
        for (int p = 0; p < 3; ++p) { lo[p] = (yuv && p > 0) ? -0.5 : 0.0; hi[p] = (yuv && p > 0) ? 0.5 : 1.0; }
        return;
    }
    const int sh = vi.bits_per_sample - 8;  // up to 24 (32-bit integer clips: full32 / yuv32 / rgb32 of src/filters/limiter.zig:72-91)
    for (int p = 0; p < 3; ++p) {
        if (!tv_range) { lo[p] = 0.0; hi[p] = (double)((1ull << vi.bits_per_sample) - 1ull); }
        else { lo[p] = (double)(16ull << sh); hi[p] = (double)(((yuv && p > 0) ? 240ull : 235ull) << sh); }
    }
}

vszip_filter* vszip_limiter_create(const vszip_video_info* vi, const vszip_limiter_args* a) {
    static const char* name = "Limiter";
    if (!basic_vi_ok(vi, name)) return nullptr;
    const int np = vi->num_planes;
    const bool is_int = vi->sample_type == VSZIP_ST_INTEGER;
    const double peak = is_int ? (double)(float)((1ll << vi->bits_per_sample) - 1) : 1.0;  // getPeakValue(.., false, .FULL) is f32
    bool process[3] = {true, true, true};
    if (!parse_planes(a->planes, a->num_planes, np, name, process)) return nullptr;
    double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
    const bool has_min = a->num_min >= 0, has_max = a->num_max >= 0;
    if (has_min) {  // limiter.zig:121-150
        if (a->num_min != np) { set_error("Limiter: min array must have the same number of elements as planes."); return nullptr; }
        for (int i = 0; i < np; ++i) {
            if (is_int) {
                const double t = std::trunc(a->min[i]);
                if (t < 0) { set_error("Limiter: min value must be greater than or equal to 0."); return nullptr; }
                if (a->min[i] > peak) { set_error("Limiter: min value must be less than or equal to peak value."); return nullptr; }
                lo[i] = t;
            } else {
                lo[i] = (double)(float)a->min[i];
            }
        }
    }
    if (has_max) {  // limiter.zig:152-181 (peak is tested before the sign here)
        if (a->num_max != np) { set_error("Limiter: max array must have the same number of elements as planes."); return nullptr; }
        for (int i = 0; i < np; ++i) {
            if (is_int) {
                const double t = std::trunc(a->max[i]);
                if (a->max[i] > peak) { set_error("Limiter: max value must be less than or equal to peak value."); return nullptr; }
                if (t < 0) { set_error("Limiter: max value must be greater than or equal to 0."); return nullptr; }
                hi[i] = t;
            } else {
                hi[i] = (double)(float)a->max[i];
            }
        }
    }
    if (has_min && !has_max) { set_error("Limiter: min array is set but max array is not."); return nullptr; }
    if (!has_min && has_max) { set_error("Limiter: max array is set but min array is not."); return nullptr; }
    if (has_min) {
        for (int p = 0; p < np; ++p)
            if (lo[p] > hi[p]) { set_error("Limiter: min value must be less than or equal to max value."); return nullptr; }
    }
    // BPSType.select (src/helper.zig:25-56)
    if (is_int) {
        const int b = vi->bits_per_sample;
        if (!(b == 8 || b == 9 || b == 10 || b == 12 || b == 14 || b == 16 || b == 32)) { set_error("Limiter: not supported Int format."); return nullptr; }
    } else if (!(vi->bits_per_sample == 16 || vi->bits_per_sample == 32)) {
        set_error("Limiter: not supported Float format.");
        return nullptr;
    }
    SampleKind kind;
    if (!select_kind(*vi, name, true, &kind)) return nullptr;
    if (kind == K_U32)  // the f32 peak of a 32-bit clip is 2^32: a bound that passed the check above may be one past the largest sample
        for (int i = 0; i < np; ++i) { lo[i] = std::min(lo[i], 4294967295.0); hi[i] = std::min(hi[i], 4294967295.0); }
    const bool tv_range = a->has_tv_range && a->tv_range != 0, maskf = a->has_mask && a->mask != 0;
    const bool yuv = vi->color_family == VSZIP_CF_YUV && !maskf;
    if (!has_min) limiter_table(*vi, tv_range, yuv, lo, hi);
    vszip_filter* f = new vszip_filter();
    f->kind = F_LIMITER;
    set_format(f, *vi, kind);
    for (int i = 0; i < 3; ++i) { f->process[i] = process[i] && i < np; f->lim_lo[i] = lo[i]; f->lim_hi[i] = hi[i]; }
    return f;
}

int vszip_limiter_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, vszip_frame* dst) {
    return pixel_get_frame(f, F_LIMITER, n, {src, nullptr, nullptr}, dst);
}

int vszip_limiter_device(const vszip_filter* f, const vszip_dev_clip* src, vszip_dev_clip* dst, int32_t first, int32_t count, void* stream) {
    return pixel_device(f, F_LIMITER, {src, nullptr, nullptr}, dst, first, count, stream);
}

// =========================================================================== LimitFilter
vszip_filter* vszip_limitfilter_create(const vszip_video_info* flt_vi, const vszip_video_info* src_vi, const vszip_video_info* ref_vi,
                                       const vszip_limitfilter_args* a) {
    static const char* name = "LimitFilter";
    if (!basic_vi_ok(flt_vi, name)) return nullptr;
    if (!src_vi) { set_error("LimitFilter: the src clip is required"); return nullptr; }
    static const vszip_limitfilter_args none = {nullptr, 0, nullptr, 0, nullptr, 0, nullptr, -1, -1};
    if (!a) a = &none;
    SampleKind kind;
    if (!select_kind(*flt_vi, name, false, &kind)) return nullptr;                     // limit_filter.zig:101
    if (!compare_nodes(*flt_vi, *src_vi, name, true)) return nullptr;                  // :107-108, SAME_LEN
    if (ref_vi && !compare_nodes(*flt_vi, *ref_vi, name, true)) return nullptr;
    bool process[3] = {true, true, true};
    if (!parse_planes(a->planes, a->num_planes, flt_vi->num_planes, name, process)) return nullptr;
    float dark[3], bright[3], elast[3];
    if (!get_array_f32(a->dark_thr, a->num_dark_thr, 1.0f, 0.0f, 255.0f, "dark_thr", name, dark)) return nullptr;
    if (!get_array_f32(a->bright_thr, a->num_bright_thr, 1.0f, 0.0f, 255.0f, "bright_thr", name, bright)) return nullptr;
    if (!get_array_f32(a->elast, a->num_elast, 2.0f, 0.0f, 65535.0f, "elast", name, elast)) return nullptr;
    // getColorRange (src/helper.zig:259-276) when the frame carries no _ColorRange
    const bool limited = a->color_range < 0 ? flt_vi->color_family != VSZIP_CF_RGB : a->color_range == 1;
    vszip_filter* f = new vszip_filter();
    f->kind = F_LIMITFILTER;
    set_format(f, *flt_vi, kind);
    for (int i = 0; i < 3; ++i) {
        f->process[i] = process[i] && i < flt_vi->num_planes;
        f->lf_dark[i] = scale_value8(dark[i], *flt_vi, limited);                       // :114-118
        f->lf_bright[i] = scale_value8(bright[i], *flt_vi, limited);
        f->lf_elast[i] = elast[i];
    }
    f->has_input[0] = true;
    f->has_input[1] = ref_vi != nullptr;
    return f;
}

int vszip_limitfilter_get_info(const vszip_filter* f, float dark_thr[3], float bright_thr[3], float elast[3]) {
    if (!f || f->kind != F_LIMITFILTER) { set_error("LimitFilter: bad filter handle"); return -1; }
    for (int i = 0; i < 3; ++i) { dark_thr[i] = f->lf_dark[i]; bright_thr[i] = f->lf_bright[i]; elast[i] = f->lf_elast[i]; }
    return 0;
}

int vszip_limitfilter_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* flt, const vszip_frame* src, const vszip_frame* ref,
                                vszip_frame* dst) {
    if (!flt || !src || !dst) { set_error("LimitFilter: flt, src and dst frames are required"); return -1; }
    return pixel_get_frame(f, F_LIMITFILTER, n, {flt, src, ref}, dst);
}

int vszip_limitfilter_device(const vszip_filter* f, const vszip_dev_clip* flt, const vszip_dev_clip* src, const vszip_dev_clip* ref,
                             vszip_dev_clip* dst, int32_t first, int32_t count, void* stream) {
    return pixel_device(f, F_LIMITFILTER, {flt, src, ref}, dst, first, count, stream);
}

// =========================================================================== AdaptiveBinarize
vszip_filter* vszip_adaptivebinarize_create(const vszip_video_info* vi, const vszip_video_info* clip2_vi, const vszip_adaptivebinarize_args* a) {
    static const char* name = "AdaptiveBinarize";
    if (!basic_vi_ok(vi, name)) return nullptr;
    if (!clip2_vi) { set_error("AdaptiveBinarize: clip2 is required"); return nullptr; }
    if (!compare_nodes(*vi, *clip2_vi, name)) return nullptr;                          // adaptive_binarize.zig:88-89, BIGGER_THAN
    if (vi->sample_type != VSZIP_ST_INTEGER || vi->bits_per_sample != 8) { set_error("AdaptiveBinarize: only 8 bit int format supported."); return nullptr; }
    const int64_t c = a && a->has_c ? (int64_t)sat_i32(a->c) : 3;                      // getValue(i32, "c") orelse 3
    vszip_filter* f = new vszip_filter();
    f->kind = F_ADAPTIVEBINARIZE;
    set_format(f, *vi, K_U8);
    for (int i = 0; i < 3; ++i) f->process[i] = i < vi->num_planes;
    f->ab_c = (int)std::min<int64_t>(std::max<int64_t>(c, -256), 256);               // :97-99
    f->has_input[0] = true;
    return f;
}

// In the chain's numbering clip2 is the main input (the one binarised) and clip the second.
int vszip_adaptivebinarize_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* clip, const vszip_frame* clip2, vszip_frame* dst) {
    if (!clip || !clip2 || !dst) { set_error("AdaptiveBinarize: clip, clip2 and dst frames are required"); return -1; }
    return pixel_get_frame(f, F_ADAPTIVEBINARIZE, n, {clip2, clip, nullptr}, dst);
}

int vszip_adaptivebinarize_device(const vszip_filter* f, const vszip_dev_clip* clip, const vszip_dev_clip* clip2, vszip_dev_clip* dst,
                                  int32_t first, int32_t count, void* stream) {
    return pixel_device(f, F_ADAPTIVEBINARIZE, {clip2, clip, nullptr}, dst, first, count, stream);
}

// =========================================================================== CLAHE
// OpenCV's CLAHE::apply on every plane (DESIGN.md §4.7).  The argument names, defaults and messages are this library's.
vszip_filter* vszip_clahe_create(const vszip_video_info* vi, const vszip_clahe_args* a) {
    static const char* name = "CLAHE";
    if (!basic_vi_ok(vi, name)) return nullptr;
    if (vi->sample_type != VSZIP_ST_INTEGER || vi->bits_per_sample < 8 || vi->bits_per_sample > 16) {
        set_error("CLAHE: only 8-16 bit int formats supported.");
        return nullptr;
    }
    SampleKind kind;
    if (!select_kind(*vi, name, false, &kind)) return nullptr;
    const double limit = a && a->has_limit ? a->limit : 15.0;
    if (!(limit >= 0)) { set_error("CLAHE: limit must be non-negative."); return nullptr; }
    const int n = a && a->tiles ? std::max(a->num_tiles, 0) : 0;
    if (n > 2) { set_error("CLAHE: tiles has too many elements (got %d, max 2).", n); return nullptr; }
    int64_t t[2] = {3, 3};
    if (n >= 1) t[0] = t[1] = a->tiles[0];
    if (n == 2) t[1] = a->tiles[1];
    if (t[0] < 1 || t[1] < 1) { set_error("CLAHE: tiles values must be at least 1."); return nullptr; }
    if (t[0] > 256 || t[1] > 256 || t[0] * t[1] > 256) { set_error("CLAHE: at most 256 tiles per plane (tiles[0] * tiles[1])."); return nullptr; }
    vszip_filter* f = new vszip_filter();
    f->kind = F_CLAHE;
    set_format(f, *vi, kind);
    for (int i = 0; i < 3; ++i) f->process[i] = i < vi->num_planes;
    f->clahe_limit = limit;
    f->clahe_tiles[0] = (int)t[0];
    f->clahe_tiles[1] = (int)t[1];
    f->clahe_hs = 1 << vi->bits_per_sample;
    return f;
}

int vszip_clahe_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, vszip_frame* dst) {
    return pixel_get_frame(f, F_CLAHE, n, {src, nullptr, nullptr}, dst);
}

int vszip_clahe_device(const vszip_filter* f, const vszip_dev_clip* src, vszip_dev_clip* dst, int32_t first, int32_t count, void* stream) {
    return pixel_device(f, F_CLAHE, {src, nullptr, nullptr}, dst, first, count, stream);
}

// =========================================================================== ColorMap
// OpenCV's applyColorMap on plane 0 (DESIGN.md §4.8): GRAY / YUV in, RGB24 out.  The argument names, default and messages are this
// library's.
vszip_filter* vszip_colormap_create(const vszip_video_info* vi, const vszip_colormap_args* a) {
    static const char* name = "ColorMap";
    if (!basic_vi_ok(vi, name)) return nullptr;
    if (vi->sample_type != VSZIP_ST_INTEGER || vi->bits_per_sample < 8 || vi->bits_per_sample > 16) {
        set_error("ColorMap: only 8-16 bit int formats supported.");
        return nullptr;
    }
    if (vi->color_family != VSZIP_CF_GRAY && vi->color_family != VSZIP_CF_YUV) { set_error("ColorMap: clip must be GRAY or YUV."); return nullptr; }
    const int64_t color = a && a->has_color ? a->color : 20;  // COLORMAP_TURBO
    if (color < 0 || color >= kColormapCount) { set_error("ColorMap: color must be between 0 and 21."); return nullptr; }
    SampleKind kind;
    if (!select_kind(*vi, name, false, &kind)) return nullptr;
    vszip_filter* f = new vszip_filter();
    f->kind = F_COLORMAP;
    set_format(f, *vi, kind);
    vszip_video_info o = *vi;  // RGB24 of the same size and length
    o.color_family = VSZIP_CF_RGB;
    o.sample_type = VSZIP_ST_INTEGER;
    o.bits_per_sample = 8;
    o.bytes_per_sample = 1;
    o.sub_sampling_w = o.sub_sampling_h = 0;
    o.num_planes = 3;
    f->out_vi = o;
    f->out_layout = make_layout(o, K_U8);
    for (int i = 0; i < 3; ++i) f->process[i] = i == 0;  // the planes it reads: the luma
    memcpy(f->cmap_lut, kColormapTables[color], sizeof f->cmap_lut);
    return f;
}

int vszip_colormap_get_lut(const vszip_filter* f, uint8_t rgb[768]) {
    if (!f || f->kind != F_COLORMAP || !rgb) { set_error("ColorMap: bad filter handle"); return -1; }
    for (int i = 0; i < 256; ++i)
        for (int c = 0; c < 3; ++c) rgb[3 * i + c] = (uint8_t)(f->cmap_lut[i] >> (8 * c));
    return 0;
}

int vszip_colormap_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, vszip_frame* dst) {
    return pixel_get_frame(f, F_COLORMAP, n, {src, nullptr, nullptr}, dst);
}

int vszip_colormap_device(const vszip_filter* f, const vszip_dev_clip* src, vszip_dev_clip* dst, int32_t first, int32_t count, void* stream) {
    return pixel_device(f, F_COLORMAP, {src, nullptr, nullptr}, dst, first, count, stream);
}

// =========================================================================== fused chains
// Values of a chain: 0 = the source frame, k >= 1 = the pixel output of element k - 1.  Every element reads its main input (the
// value it filters) and up to two extra inputs; the buffer plan gives every pixel output a frame buffer for as long as a later
// element reads it (DESIGN.md §5.1).  Buffers 0..2 are the slot's dev[0..2] (0 = the source, never written; 2 = the value the
// chain returns, the D2H source), buffers 3.. are the slot's device-only extras.  Every value has a format: value 0 filter 0's,
// value k the output format of element k - 1, which differs from its input's for ColorMap.
struct vszip_chain {
    std::vector<const vszip_filter*> fl;
    vsz::FrameLayout in_layout, out_layout;  // the source's and the returned value's
    bool written[3];
    int npixel;
    std::vector<int> in, in2, in3;  // buffer of each element's main / second / third input (-1: none)
    std::vector<int> out;           // buffer of each element's pixel output (-1: stats element)
    std::vector<char> fuse_next;    // stats element i runs together with element i + 1 from one read
    std::vector<char> used;         // buffers the plan uses (0..2: the slot's dev[], 3..: its device-only extras)
    std::vector<size_t> bytes;      // the size of each buffer: the frame stride of the largest value it holds
};

namespace {

const FrameLayout& value_layout(const vszip_filter* const* filters, int v) { return v == 0 ? filters[0]->layout : filters[v - 1]->out_layout; }

// Element i reads value v: it must have been created for that value's format.  The message names filter 0 when the value has its
// format (every value of a chain without a format-changing element does).
bool reads_ok(const vszip_filter* const* filters, int i, int v) {
    const vszip_video_info& fmt = v == 0 ? filters[0]->vi : filters[v - 1]->out_vi;
    if (same_format(filters[i]->vi, fmt)) return true;
    if (same_format(fmt, filters[0]->vi)) set_error("chain: filter %d was created for a different video format than filter 0", i);
    else set_error("chain: filter %d was created for a different video format than the value it reads", i);
    return false;
}

// input / second / third use the value numbering above; input == nullptr: every element reads the latest pixel output (or the source).
vszip_chain* chain_build(const vszip_filter* const* filters, int count, const int32_t* input, const int32_t* second, const int32_t* third) {
    const int nv = count + 1;
    std::vector<int> vin(count), v2(count), v3(count);
    std::vector<int> last_use(nv, -1), def(nv, -1);
    int cur = 0;
    for (int i = 0; i < count; ++i) {
        vin[i] = input ? input[i] : cur;
        v2[i] = second ? second[i] : -1;
        v3[i] = third ? third[i] : -1;
        if (is_pixel(filters[i])) { cur = i + 1; def[i + 1] = i; }
    }
    // the value the chain returns: the last element's pixel output, or the value a final stats element reads
    const vszip_filter* fl = filters[count - 1];
    const int result = is_pixel(fl) ? count : vin[count - 1];
    vszip_chain* c = new vszip_chain();
    c->fl.assign(filters, filters + count);
    c->in_layout = filters[0]->layout;
    c->out_layout = value_layout(filters, result);
    c->npixel = 0;
    for (int i = 0; i < count; ++i) {
        for (int v : {vin[i], v2[i], v3[i]}) if (v >= 0) last_use[v] = std::max(last_use[v], i);
        c->npixel += is_pixel(filters[i]) ? 1 : 0;
    }
    // planes in which each value differs from the source
    std::vector<std::array<bool, 3>> diff(nv, std::array<bool, 3>{false, false, false});
    for (int i = 0; i < count; ++i)
        if (is_pixel(filters[i])) {
            bool w[3];
            written_planes(filters[i], w);
            for (int p = 0; p < 3; ++p) diff[i + 1][p] = (!converts(filters[i]) && diff[vin[i]][p]) || w[p];
        }
    for (int p = 0; p < 3; ++p) c->written[p] = diff[result][p];
    // buffer plan: a value occupies its buffer from the element that writes it to the last element that reads it (both inclusive,
    // so an element never writes the buffer it reads).  The result goes to buffer 2 and lives to the end; the other pixel outputs,
    // latest first, take the lowest buffer >= 1 that is free over their whole span - for a linear chain that is the 1 / 2
    // alternation ending in 2.
    std::vector<int> buf(nv, -1);
    buf[0] = 0;
    std::vector<std::vector<std::pair<int, int>>> busy(3);
    if (result > 0) { buf[result] = 2; busy[2].push_back({def[result], count}); }
    for (int v = count; v >= 1; --v) {
        if (def[v] < 0 || v == result) continue;
        const int lo = def[v], hi = std::max(last_use[v], def[v]);
        int b = 1;
        for (;; ++b) {
            if ((int)busy.size() <= b) busy.resize(b + 1);
            bool free_ = true;
            for (auto& r : busy[b]) free_ = free_ && (hi < r.first || r.second < lo);
            if (free_) break;
        }
        buf[v] = b;
        busy[b].push_back({lo, hi});
    }
    c->used.assign(busy.size(), 0);
    c->used[0] = c->used[2] = 1;
    c->bytes.assign(busy.size(), 0);
    c->bytes[0] = c->in_layout.frame_stride;
    for (int v = 1; v < nv; ++v)
        if (buf[v] >= 0) {
            c->used[buf[v]] = 1;
            c->bytes[buf[v]] = std::max(c->bytes[buf[v]], value_layout(filters, v).frame_stride);
        }
    for (int i = 0; i < count; ++i) {
        c->in.push_back(buf[vin[i]]);
        c->in2.push_back(v2[i] >= 0 ? buf[v2[i]] : -1);
        c->in3.push_back(v3[i] >= 0 ? buf[v3[i]] : -1);
        c->out.push_back(is_pixel(filters[i]) ? buf[i + 1] : -1);
    }
    c->fuse_next.assign(count, 0);
    for (int i = 0; i + 1 < count; ++i) {
        if (stats_pair(filters[i], filters[i + 1]) && vin[i] == vin[i + 1] && v2[i] == v2[i + 1]) {
            c->fuse_next[i] = 1;
            ++i;
        }
    }
    return c;
}

}  // namespace

vszip_chain* vszip_chain_create(const vszip_filter* const* filters, int32_t count) {
    if (!filters || count < 1 || count > 16) { set_error("chain: between 1 and 16 filters are required"); return nullptr; }
    int32_t second[16];
    int cur = 0;  // the value element i filters: the latest pixel output, or the source
    for (int i = 0; i < count; ++i) {
        const vszip_filter* f = filters[i];
        if (!f) { set_error("chain: filter %d is NULL", i); return nullptr; }
        // LimitFilter (without ref) and AdaptiveBinarize take the chain's SOURCE frame as their second clip ("diamond" elements)
        const bool diamond = (f->kind == F_LIMITFILTER && !f->has_input[1]) || f->kind == F_ADAPTIVEBINARIZE;
        if (f->has_input[0] && !diamond) { set_error("chain: filter %d takes a second clip (ref/clipb); only single-input filters can be fused", i); return nullptr; }
        if (!reads_ok(filters, i, cur) || (diamond && !reads_ok(filters, i, 0))) return nullptr;
        second[i] = diamond ? 0 : -1;
        if (is_pixel(f)) cur = i + 1;
    }
    return chain_build(filters, count, nullptr, second, nullptr);
}

vszip_chain* vszip_chain_create2(const vszip_filter* const* filters, int32_t count, const int32_t* input, const int32_t* second,
                                 const int32_t* third) {
    if (!filters || count < 1 || count > 16) { set_error("chain: between 1 and 16 filters are required"); return nullptr; }
    const vszip_filter* f0 = filters[0];
    bool converted = false;  // an earlier element changed the format: the values no longer all have filter 0's
    int cur = 0;             // the value element i filters when input == NULL
    for (int i = 0; i < count; ++i) {
        const vszip_filter* f = filters[i];
        if (!f) { set_error("chain: filter %d is NULL", i); return nullptr; }
        if (!converted && !same_format(f0->vi, f->vi)) {
            set_error("chain: filter %d was created for a different video format than filter 0", i);
            return nullptr;
        }
        const KindInfo& info = kind_info(f->kind);
        const int32_t refs[3] = {input ? input[i] : 0, second ? second[i] : -1, third ? third[i] : -1};
        static const char* arr[3] = {"input", "second", "third"};
        static const char* none[3] = {"", "a second clip", "a third clip"};
        for (int k = 0; k < 3; ++k) {
            const int32_t v = refs[k];
            if (k > 0) {
                const char* what = info.input[k - 1] ? info.input[k - 1] : none[k];
                if (!f->has_input[k - 1] && v != -1) { set_error("chain: filter %d (%s) was created without %s; %s[%d] must be -1", i, info.name, what, arr[k], i); return nullptr; }
                if (f->has_input[k - 1] && v == -1) { set_error("chain: filter %d (%s) was created with %s; %s[%d] must name its input", i, info.name, what, arr[k], i); return nullptr; }
                if (v == -1) continue;
            }
            if (v < 0 || v > count) { set_error("chain: %s[%d] = %d is out of range (0 = the source, k = the output of filter k - 1)", arr[k], i, v); return nullptr; }
            if (v >= 1 && v - 1 >= i) { set_error("chain: %s[%d] names filter %d, which does not come before filter %d", arr[k], i, v - 1, i); return nullptr; }
            if (v >= 1 && !is_pixel(filters[v - 1])) { set_error("chain: %s[%d] names filter %d (%s), which has no pixel output", arr[k], i, v - 1, kind_info(filters[v - 1]->kind).name); return nullptr; }
        }
        for (int k = 0; k < 3; ++k)
            if (refs[k] >= 0 && !reads_ok(filters, i, k == 0 && !input ? cur : refs[k])) return nullptr;
        converted = converted || (is_pixel(f) && converts(f));
        if (is_pixel(f)) cur = i + 1;
    }
    return chain_build(filters, count, input, second, third);
}

void vszip_chain_free(vszip_chain* c) { delete c; }

int vszip_chain_planes(const vszip_chain* c, int32_t written[3]) {
    if (!c) { set_error("chain: bad handle"); return -1; }
    for (int p = 0; p < 3; ++p) written[p] = c->written[p] ? 1 : 0;
    return 0;
}

int vszip_chain_get_frame(const vszip_chain* c, int32_t n, const vszip_frame* src, vszip_frame* dst, void* const* props_out) {
    if (!c) { set_error("chain: bad handle"); return -1; }
    if (c->npixel > 0 && !dst) { set_error("chain: dst is required when the chain holds a pixel filter"); return -1; }
    DeviceCtx* d = route(n, "chain");
    if (!d) return -1;
    SlotGuard g(d);
    Slot* s = g.s;
    VSZ_CUDA(cudaSetDevice(d->ordinal));
    const FrameLayout& l = c->in_layout;
    if (slot_reserve(d, s, 0, c->bytes[0]) || slot_reserve(d, s, 2, c->bytes[2]) || (c->used[1] && slot_reserve(d, s, 1, c->bytes[1]))) return -1;
    for (int b = 3; b < (int)c->used.size(); ++b)
        if (slot_reserve_extra(d, s, b - 3, c->bytes[b])) return -1;
    auto B = [&](int b) -> char* { return b < 0 ? nullptr : (b < 3 ? s->dev[b] : s->xdev[b - 3]); };
    bool all[3] = {l.nplanes > 0, l.nplanes > 1, l.nplanes > 2};
    if (stage_in(s, 0, l, src, all)) return -1;  // later filters may read planes that earlier ones do not process
    const int dev_index = device_index_of(d);
    int stats_seen = 0;
    for (size_t i = 0; i < c->fl.size(); ++i) {
        const vszip_filter* f = c->fl[i];
        const char* in[3] = {B(c->in[i]), B(c->in2[i]), B(c->in3[i])};
        if (is_pixel(f)) {
            char* nxt = B(c->out[i]);
            const FrameLayout& fl = f->layout;
            for (int p = 0; p < fl.nplanes && !converts(f); ++p) {  // planes this filter passes through (none when it changes the format)
                if (f->process[p]) continue;
                VSZ_CUDA(cudaMemcpyAsync(nxt + fl.pl[p].offset, in[0] + fl.pl[p].offset, (size_t)fl.pl[p].pitch * fl.pl[p].h,
                                         cudaMemcpyDeviceToDevice, s->stream));
            }
            const int rc = run_pixels(f, dev_index, in, 0, nxt, 0, 1, s->stream);
            if (rc) return rc;
            continue;
        }
        // a PlaneMinMax and a PlaneAverage of the same value, planes and clipb run as a pair (one read when the kernels allow it)
        const int ne = c->fuse_next[i] ? 2 : 1;
        for (size_t e = i; e < i + ne; ++e)
            if (!props_out || !props_out[e]) { set_error("chain: props_out[%d] is required for a PlaneMinMax/PlaneAverage element", (int)e); return -1; }
        const int np = processed_planes(f);
        if (np == 0) { ++stats_seen; continue; }
        const size_t sb = stats_scratch_bytes(1, np);
        AsyncScratch stats_mem;
        VSZ_CUDA(stats_mem.alloc(sb * ne, s->stream));
        StatsRaw* raw_dev = (StatsRaw*)s->dev_small + (size_t)stats_seen * 3;
        const int rc = ne == 2 ? run_stats_pair(f, c->fl[i + 1], dev_index, in[0], in[1], 0, 1, true, stats_mem.p, stats_mem.p + sb, raw_dev,
                                                raw_dev + 3, s->stream, nullptr)
                               : run_stats(f, dev_index, in[0], in[1], 0, 1, stats_mem.p, raw_dev, s->stream);
        if (rc) return rc;
        VSZ_CUDA(cudaMemcpyAsync((StatsRaw*)s->pin_small + (size_t)stats_seen * 3, raw_dev, sizeof(StatsRaw) * (ne == 2 ? 6 : np),
                                 cudaMemcpyDeviceToHost, s->stream));
        stats_seen += ne;
        i += ne - 1;
    }
    bool direct[3] = {false, false, false};
    if (c->npixel > 0 && stage_out_begin(s, c->out_layout, dst, c->written, direct)) return -1;
    VSZ_CUDA(cudaStreamSynchronize(s->stream));
    if (c->npixel > 0) stage_out_finish(s, c->out_layout, dst, c->written, direct);
    stats_seen = 0;
    for (size_t i = 0; i < c->fl.size(); ++i) {
        const vszip_filter* f = c->fl[i];
        if (is_pixel(f)) continue;
        const StatsRaw* raw = (const StatsRaw*)s->pin_small + (size_t)stats_seen * 3;
        if (processed_planes(f) > 0) stats_finalize(f, raw, props_out[i], 0);
        else if (f->kind == F_PLANEMINMAX) ((vszip_minmax_props*)props_out[i])->count = 0;
        else ((vszip_average_props*)props_out[i])->count = 0;
        ++stats_seen;
    }
    return 0;
}

}  // extern "C"
