/* vszip_cuda.h — C ABI of the B200 (sm_100a) implementation of vszip's pixel hot path:
 * BoxBlur, Bilateral, PlaneMinMax, PlaneAverage.
 *
 * This is the drop-in boundary.  The reference (dnjulek/vapoursynth-zip 19.0.0) runs these four
 * filters as Zig functions called from its VapourSynth getFrame callbacks; a maintainer keeps
 * src/vszip.zig and the src/vapoursynth glue (names, argument strings, props) and replaces the
 * calls into src/filters/{boxblur_comptime,boxblur_runtime,bilateral,planeminmax,planeaverage}.zig
 * by the entry points below (see INTEGRATION.md for the Zig side).  Everything is plain C:
 * pointers, sizes, PODs.  No CUDA, torch or C++ types appear in any signature.
 *
 * Conventions
 *  - All functions are thread-safe; getFrame-style calls may be issued concurrently from many
 *    host threads (VapourSynth fmParallel) on one immutable filter handle.
 *  - Functions returning int return 0 on success and a negative code on failure; functions
 *    returning a pointer return NULL on failure.  vszip_cuda_last_error() then holds the message
 *    (thread-local).  Create-time validation messages are byte-identical to the reference's
 *    mapSetError strings so existing scripts/tests see the same errors.
 *  - There is no CPU fallback: without a usable sm_100 device every entry point fails.
 *  - Frame n is routed to device (n mod k) of the k devices given to vszip_cuda_init.
 */
#ifndef VSZIP_CUDA_H
#define VSZIP_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSZIP_CUDA_ABI_VERSION 5  /* 2: + vszip_chain_*, vszip_limiter_*; 3: + vszip_limitfilter_*, vszip_adaptivebinarize_*, vszip_planestats_device; 4: + vszip_cuda_host_forget, vszip_cuda_host_registered_bytes, vszip_cuda_host_register_limit; 5: + vszip_cuda_reserve, and additions that leave every earlier entry point unchanged: vszip_chain_create2, vszip_planestats_device_b, vszip_cuda_transfer_bytes, vszip_clahe_create, vszip_clahe_get_frame, vszip_clahe_device, vszip_colormap_create, vszip_colormap_get_frame, vszip_colormap_device, vszip_colormap_get_lut, vszip_filter_output_info (a caller that needs them resolves them by name) */

/* VapourSynth4.h values (VSColorFamily / VSSampleType) so the Zig glue can pass vi.format as is. */
enum { VSZIP_CF_GRAY = 1, VSZIP_CF_RGB = 2, VSZIP_CF_YUV = 3 };
enum { VSZIP_ST_INTEGER = 0, VSZIP_ST_FLOAT = 1 };

/* Subset of VSVideoInfo/VSVideoFormat the four create callbacks read
 * (src/vapoursynth/boxblur.zig:137-179, bilateral.zig:97-115, planeminmax.zig:105-140). */
typedef struct vszip_video_info {
    int32_t width, height, num_frames;
    int32_t color_family, sample_type, bits_per_sample, bytes_per_sample;
    int32_t sub_sampling_w, sub_sampling_h, num_planes;
} vszip_video_info;

/* One video frame in host memory as handed over by getReadPtr/getWritePtr/getStride
 * (stride in BYTES, may be negative-free arbitrary padding; pageable memory is fine). */
typedef struct vszip_frame {
    void* data[3];
    ptrdiff_t stride[3];
} vszip_frame;

typedef struct vszip_filter vszip_filter;     /* immutable after create */
typedef struct vszip_dev_clip vszip_dev_clip; /* frames resident in one GPU's HBM */

/* ------------------------------------------------------------------ runtime */

/* Selects the GPUs to use (CUDA ordinals); num_devices == 0 uses every visible device.
 * Returns the number of devices in use, or < 0.  Idempotent; replaces VapourSynthPluginInit2-time
 * setup (src/vszip.zig:35).  Each device gets a frame pool, pinned staging and a set of streams. */
int vszip_cuda_init(const int32_t* device_ids, int32_t num_devices);
void vszip_cuda_shutdown(void);
int vszip_cuda_device_count(void);
const char* vszip_cuda_last_error(void);
int vszip_cuda_abi_version(void);
/* Number of kernels this library has launched so far in this process (all threads). */
uint64_t vszip_cuda_kernel_launches(void);
/* Sample bytes (width * height * bytes per sample of each plane) of the frames this library has copied between host and GPU so far
 * in this process: direction 0 = host to device, 1 = device to host (the get_frame / chain staging and vszip_dev_clip_upload /
 * _download; not the small reduction results).  Any other direction returns 0. */
uint64_t vszip_cuda_transfer_bytes(int32_t direction);

/* Host frame buffers.  getFrame hands over pageable planes owned by the VapourSynth core (getReadPtr / getWritePtr,
 * src/helper.zig:510-531).  Planes that lie entirely inside memory the application page-locked are DMA'd in place; everything
 * else goes through the slots' pinned staging buffers.  Opt-in (vszip_cuda_host_register_limit(bytes > 0) or
 * VSZIP_HOST_REGISTER_MB): the library page-locks (cudaHostRegister) a pageable plane buffer the second time it sees its
 * address and DMAs it in place from then on.  Rule for the caller when this is switched on: before memory that was passed to a
 * *_get_frame call is freed or unmapped, call vszip_cuda_host_forget(ptr) with the plane pointer that was passed, or with NULL
 * to drop every entry - a registration left behind on an address range that is later mapped again makes the GPU copy from/to
 * the old pages.  vszip_cuda_shutdown() forgets everything. */
void vszip_cuda_host_forget(const void* ptr);
size_t vszip_cuda_host_registered_bytes(void);
/* Sets the cap on page-locked application memory in bytes (0 = never register; buffers registered so far stay registered until
 * they are forgotten) and returns the previous cap. */
size_t vszip_cuda_host_register_limit(size_t bytes);

/* Optional, from a filter's create callback: allocates the pinned + device staging buffers of every request slot on every GPU
 * for frames of this format (`buffers` of them per slot: 2 for one input clip + the output, 3 with a ref / second clip, 4 for
 * LimitFilter with ref) so that the first getFrame calls do not pay for cudaHostAlloc / cudaMalloc.  Blocks until no request is
 * in flight.  0 on success, -1 with vszip_cuda_last_error() otherwise.  Without it the buffers grow on first use (and on the
 * first larger format), exactly as before. */
int32_t vszip_cuda_reserve(const vszip_video_info* vi, int32_t buffers);

/* ------------------------------------------------------------------ BoxBlur
 * replaces boxBlurCreate / BoxBlurCT.getFrame / BoxBlurRT.getFrame (src/vapoursynth/boxblur.zig:27-212)
 * and the kernels in src/filters/boxblur_comptime.zig + boxblur_runtime.zig.
 * Argument string kept: "clip:vnode;planes:int[]:opt;hradius:int:opt;hpasses:int:opt;vradius:int:opt;vpasses:int:opt"
 * (src/vszip.zig:64).  has_* == 0 means "key absent" (defaults 1/1/1/1, boxblur.zig:145-148);
 * num_planes < 0 means "planes absent" (all planes). */
typedef struct vszip_boxblur_args {
    const int64_t* planes; int32_t num_planes;
    int32_t has_hradius; int64_t hradius;
    int32_t has_hpasses; int64_t hpasses;
    int32_t has_vradius; int64_t vradius;
    int32_t has_vpasses; int64_t vpasses;
} vszip_boxblur_args;

vszip_filter* vszip_boxblur_create(const vszip_video_info* vi, const vszip_boxblur_args* args);
/* getFrame(AllFramesReady): blurs the processed planes of src into dst (dst planes of unprocessed
 * planes are not touched: VapourSynth's newVideoFrame2 shares them).  Synchronous. */
int vszip_boxblur_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, vszip_frame* dst);

/* ------------------------------------------------------------------ Bilateral
 * replaces bilateralCreate / Bilateral.getFrame (src/vapoursynth/bilateral.zig:33-253) and
 * src/filters/bilateral.zig (algorithm 2).  Argument string kept:
 * "clip:vnode;ref:vnode:opt;sigmaS:float[]:opt;sigmaR:float[]:opt;planes:int[]:opt;algorithm:int[]:opt;PBFICnum:int[]:opt"
 * (src/vszip.zig:48).  num_* is the element count of each array key (0 = absent; planes: < 0 = absent). */
typedef struct vszip_bilateral_args {
    const double* sigmaS; int32_t num_sigmaS;
    const double* sigmaR; int32_t num_sigmaR;
    const int64_t* planes; int32_t num_planes;
    const int64_t* algorithm; int32_t num_algorithm;
    const int64_t* PBFICnum; int32_t num_PBFICnum;
} vszip_bilateral_args;

/* ref_vi == NULL: no joint clip. */
vszip_filter* vszip_bilateral_create(const vszip_video_info* vi, const vszip_video_info* ref_vi,
                                     const vszip_bilateral_args* args);
int vszip_bilateral_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src,
                              const vszip_frame* ref /* NULL unless joint */, vszip_frame* dst);

/* Derived per-plane parameters (for inspection/tests; bilateral.zig:147-199). */
typedef struct vszip_bilateral_info {
    double sigmaS[3], sigmaR[3];
    int32_t process[3], algorithm[3];
    uint32_t PBFICnum[3], radius[3], samples[3], step[3];
    int32_t exact_lut[3]; /* 1: range weights bit-identical to the reference LUT */
} vszip_bilateral_info;
int vszip_bilateral_get_info(const vszip_filter* f, vszip_bilateral_info* out);

/* ------------------------------------------------------------------ PlaneMinMax
 * replaces planeMinMaxCreate / PlaneMinMax.getFrame (src/vapoursynth/planeminmax.zig:34-192) and
 * src/filters/planeminmax.zig.  Argument string kept:
 * "clipa:vnode;minthr:float:opt;maxthr:float:opt;clipb:vnode:opt;planes:int[]:opt;prop:data:opt;"
 * (src/vszip.zig:194).  The prop-name prefix stays on the Zig side. */
typedef struct vszip_planeminmax_args {
    int32_t has_minthr; double minthr;
    int32_t has_maxthr; double maxthr;
    const int64_t* planes; int32_t num_planes;
} vszip_planeminmax_args;

/* Values to append, in plane order, to <prop>Min / <prop>Max / <prop>Diff
 * (planeminmax.zig:58-69 of src/filters): integer clips use imin/imax (setInt), float clips
 * fmin/fmax (setFloat). */
typedef struct vszip_minmax_props {
    int32_t count;      /* number of processed planes */
    int32_t plane[3];   /* their indices */
    int32_t is_float, has_diff;
    int64_t imin[3], imax[3];
    double fmin[3], fmax[3], diff[3];
} vszip_minmax_props;

vszip_filter* vszip_planeminmax_create(const vszip_video_info* vi, const vszip_video_info* clipb_vi,
                                       const vszip_planeminmax_args* args);
int vszip_planeminmax_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* clipa,
                                const vszip_frame* clipb /* NULL unless given */, vszip_minmax_props* out);

/* ------------------------------------------------------------------ PlaneAverage
 * replaces planeAverageCreate / PlaneAverage.getFrame (src/vapoursynth/planeaverage.zig:30-155) and
 * src/filters/planeaverage.zig.  Argument string kept:
 * "clipa:vnode;exclude:int[];clipb:vnode:opt;planes:int[]:opt;prop:data:opt;" (src/vszip.zig:186).
 * num_exclude < 0 means the (mandatory) key is absent -> error, as VapourSynth itself reports. */
typedef struct vszip_planeaverage_args {
    const int64_t* exclude; int32_t num_exclude;
    const int64_t* planes; int32_t num_planes;
} vszip_planeaverage_args;

typedef struct vszip_average_props {
    int32_t count;
    int32_t plane[3];
    int32_t has_diff;
    double avg[3], diff[3];
} vszip_average_props;

vszip_filter* vszip_planeaverage_create(const vszip_video_info* vi, const vszip_video_info* clipb_vi,
                                        const vszip_planeaverage_args* args);
int vszip_planeaverage_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* clipa,
                                 const vszip_frame* clipb, vszip_average_props* out);

/* ------------------------------------------------------------------ Limiter (SURVEY 8f rank 3: the pointwise neighbour of BoxBlur)
 * replaces limiterCreate / Limiter.getFrame / LimiterRT.getFrame (src/vapoursynth/limiter.zig:24-233) and the range
 * tables of src/filters/limiter.zig:66-91.  Argument string kept:
 * "clip:vnode;min:float[]:opt;max:float[]:opt;tv_range:int:opt;mask:int:opt;planes:int[]:opt;" (src/vszip.zig:162).
 * num_min / num_max / num_planes < 0 mean "key absent"; 32-bit integer clips are not supported by the CUDA path. */
typedef struct vszip_limiter_args {
    const double* min; int32_t num_min;
    const double* max; int32_t num_max;
    const int64_t* planes; int32_t num_planes;
    int32_t has_tv_range; int32_t tv_range;
    int32_t has_mask; int32_t mask;
} vszip_limiter_args;
vszip_filter* vszip_limiter_create(const vszip_video_info* vi, const vszip_limiter_args* args);
int vszip_limiter_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, vszip_frame* dst);

/* ------------------------------------------------------------------ LimitFilter (SURVEY 8f rank 3)
 * replaces limitFilterCreate / LimitFilter.getFrame (src/vapoursynth/limit_filter.zig:27-124) and
 * src/filters/limit_filter.zig:3-34.  Argument string kept:
 * "flt:vnode;src:vnode;ref:vnode:opt;dark_thr:float[]:opt;bright_thr:float[]:opt;elast:float[]:opt;planes:int[]:opt;"
 * num_* = element count of each array key (0 = absent; planes: < 0 = absent).
 * color_range: what hz.getColorRange(flt) returned on the Zig side (src/helper.zig:259-276: frame 0's _ColorRange,
 * 0 = full, 1 = limited); < 0 = "prop absent", resolved here like the reference (RGB -> full, else limited).  It only
 * matters for the 8-bit -> clip-depth scaling of dark_thr / bright_thr (hz.scaleValue, src/helper.zig:312-338). */
typedef struct vszip_limitfilter_args {
    const double* dark_thr; int32_t num_dark_thr;
    const double* bright_thr; int32_t num_bright_thr;
    const double* elast; int32_t num_elast;
    const int64_t* planes; int32_t num_planes;
    int32_t color_range;
} vszip_limitfilter_args;
/* src_vi is required, ref_vi == NULL: no ref clip (the difference is judged against src). */
vszip_filter* vszip_limitfilter_create(const vszip_video_info* flt_vi, const vszip_video_info* src_vi,
                                       const vszip_video_info* ref_vi, const vszip_limitfilter_args* args);
int vszip_limitfilter_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* flt, const vszip_frame* src,
                                const vszip_frame* ref /* NULL unless created with ref_vi */, vszip_frame* dst);
/* Thresholds after scaling, as the kernel uses them (for inspection/tests). */
int vszip_limitfilter_get_info(const vszip_filter* f, float dark_thr[3], float bright_thr[3], float elast[3]);

/* ------------------------------------------------------------------ AdaptiveBinarize (SURVEY 8f rank 3)
 * replaces adaptiveBinarizeCreate / adaptiveBinarizeGetFrame (src/vapoursynth/adaptive_binarize.zig:28-116):
 * every plane, dst = 255 where clip2 - clip >= c else 0, 8-bit integer clips only; the Zig side keeps setting
 * _ColorRange = full on the output frame.  Argument string kept: "clip:vnode;clip2:vnode;c:int:opt;". */
typedef struct vszip_adaptivebinarize_args {
    int32_t has_c; int64_t c;
} vszip_adaptivebinarize_args;
vszip_filter* vszip_adaptivebinarize_create(const vszip_video_info* vi, const vszip_video_info* clip2_vi,
                                            const vszip_adaptivebinarize_args* args);
int vszip_adaptivebinarize_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* clip, const vszip_frame* clip2,
                                     vszip_frame* dst);

/* ------------------------------------------------------------------ CLAHE
 * Contrast-limited adaptive histogram equalisation of every plane of an 8..16-bit integer clip, bit-exact with OpenCV's
 * cv::createCLAHE(limit, (tiles[0], tiles[1])).apply on each plane (histogram size 2^bits; samples above 2^bits - 1 count as
 * 2^bits - 1).  Argument string: "clip:vnode;limit:float:opt;tiles:int[]:opt;".  has_limit == 0: limit 15; num_tiles == 0:
 * tiles [3, 3]; one value applies to both axes.  limit >= 0 (0: no clipping), every tile count >= 1, tiles[0] * tiles[1] <= 256.
 * The names, defaults and messages are this library's (the reference's source is not part of this tree). */
typedef struct vszip_clahe_args {
    int32_t has_limit; double limit;
    const int64_t* tiles; int32_t num_tiles;
} vszip_clahe_args;
vszip_filter* vszip_clahe_create(const vszip_video_info* vi, const vszip_clahe_args* args);
int vszip_clahe_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, vszip_frame* dst);

/* ------------------------------------------------------------------ ColorMap
 * OpenCV's colormaps (cv::applyColorMap) on the luma of an 8..16-bit integer GRAY or YUV clip; the output is RGB24 of the same size
 * and length (vszip_filter_output_info), the first filter whose output format differs from its input's.  Plane 0 only is read:
 * i = min(x >> (bits - 8), 255), (R, G, B) = table[color][i]; for 8-bit input the result equals cv2.applyColorMap(y)[..., ::-1].
 * Argument string: "clip:vnode;color:int:opt;".  has_color == 0: color 20 (COLORMAP_TURBO); color is cv::ColormapTypes 0..21.
 * The Zig side sets _ColorRange = 0 and _Matrix = 0 on the output frame.  The names, default and messages are this library's. */
typedef struct vszip_colormap_args {
    int32_t has_color; int64_t color;
} vszip_colormap_args;
vszip_filter* vszip_colormap_create(const vszip_video_info* vi, const vszip_colormap_args* args);
/* dst: the three planes of an RGB24 frame, all written. */
int vszip_colormap_get_frame(const vszip_filter* f, int32_t n, const vszip_frame* src, vszip_frame* dst);
/* The selected table, rgb[3 * i + c] = channel c (R, G, B) of index i (for inspection and tests). */
int vszip_colormap_get_lut(const vszip_filter* f, uint8_t rgb[768]);

/* ------------------------------------------------------------------ common filter calls */
void vszip_filter_free(vszip_filter* f);                         /* replaces xxxFree */
int vszip_filter_planes(const vszip_filter* f, int32_t process[3]); /* d.planes after create: the planes the filter reads */
/* The format of the clip the filter's node returns (the output node's vi): the input format for every filter except ColorMap,
 * whose output is RGB24.  A filter that changes the format writes every plane of its output; any other pixel filter writes the
 * planes vszip_filter_planes reports and leaves the others to the input frame. */
int vszip_filter_output_info(const vszip_filter* f, vszip_video_info* out);

/* ------------------------------------------------------------------ device-resident clips
 * Frames that stay in HBM: used to chain vszip filters without PCIe round trips and to measure
 * kernels without transfers (batches of frames per launch).  `device` is an index into the
 * vszip_cuda_init list.  Plane pitch is chosen by the pool (multiple of 128 bytes). */
vszip_dev_clip* vszip_dev_clip_alloc(const vszip_video_info* vi, int32_t num_frames, int32_t device);
void vszip_dev_clip_free(vszip_dev_clip* c);
int vszip_dev_clip_upload(vszip_dev_clip* c, int32_t frame, const vszip_frame* host);
int vszip_dev_clip_download(const vszip_dev_clip* c, int32_t frame, vszip_frame* host);
/* Counter-based uniform noise keyed by (seed, frame number, plane, y, x): integer samples over the full
 * [0, 2^bits) range, float luma/RGB in [0,1), float chroma in [-0.5,0.5).  Frame i of the clip is frame number
 * first_frame_no + i*frame_no_stride of the synthetic source, so rank r of k can hold exactly the frames
 * n with n mod k == r (first = r, stride = k). */
int vszip_dev_clip_fill_noise(vszip_dev_clip* c, uint64_t seed, int32_t first_frame_no, int32_t frame_no_stride);
/* Sum over planes of width*height*bytes_per_sample (the algorithmic bytes of one frame). */
size_t vszip_dev_clip_frame_bytes(const vszip_dev_clip* c);
/* Raw device pointer / pitch of one plane (for interop with other CUDA code). */
void* vszip_dev_clip_plane_ptr(const vszip_dev_clip* c, int32_t frame, int32_t plane, ptrdiff_t* pitch_bytes);

/* Batched, asynchronous, device-resident execution on frames [first, first+count) of the clips.
 * `stream` is a cudaStream_t (as void*) on the clips' device, or NULL for the library's own stream
 * of that device; work is enqueued and NOT synchronised (use vszip_cuda_stream_sync or your own
 * event).  src and dst must have the same format/size and live on the same device; for ColorMap dst has the filter's output format
 * (vszip_filter_output_info). */
int vszip_boxblur_device(const vszip_filter* f, const vszip_dev_clip* src, vszip_dev_clip* dst,
                         int32_t first, int32_t count, void* stream);
int vszip_bilateral_device(const vszip_filter* f, const vszip_dev_clip* src, const vszip_dev_clip* ref,
                           vszip_dev_clip* dst, int32_t first, int32_t count, void* stream);
/* Results for frame first+i land in out[i] (host memory); these two calls synchronise the stream. */
int vszip_planeminmax_device(const vszip_filter* f, const vszip_dev_clip* clipa, const vszip_dev_clip* clipb,
                             int32_t first, int32_t count, vszip_minmax_props* out, void* stream);
int vszip_planeaverage_device(const vszip_filter* f, const vszip_dev_clip* clipa, const vszip_dev_clip* clipb,
                              int32_t first, int32_t count, vszip_average_props* out, void* stream);
/* PlaneMinMax + PlaneAverage over the same frames (SURVEY 8f rank 4; BASELINE config 4 runs both over the same plane).
 * When the pair is eligible - 8..16-bit integer clip, both filters created without clipb and for the same planes, thresholds
 * set, at most 4 distinct exclude values inside the sample range - ONE kernel reads each plane once and produces both
 * results; otherwise the two reductions run one after the other.  Results are identical to the two separate calls either
 * way.  *fused_out (may be NULL) reports which route ran.  Either out pointer may be NULL (results stay on the device and
 * the stream is not synchronised when both are). */
int vszip_planestats_device(const vszip_filter* minmax, const vszip_filter* average, const vszip_dev_clip* clipa,
                            int32_t first, int32_t count, vszip_minmax_props* minmax_out, vszip_average_props* average_out,
                            int32_t* fused_out, void* stream);
/* The same with clipb: clipb is the second clip of every filter of the pair that was created with clipb (and must be NULL when
 * neither was).  One read of each (clipa, clipb) plane pair when both filters were created with clipb and the pair is otherwise
 * eligible as above (plus: a float clip with thresholds only when its planes have row padding, so that every float sum is
 * accumulated in the same order as by the separate calls); Diff is accumulated once and reported to both.  Results are bit-identical
 * to the two separate calls either way. */
int vszip_planestats_device_b(const vszip_filter* minmax, const vszip_filter* average, const vszip_dev_clip* clipa,
                              const vszip_dev_clip* clipb, int32_t first, int32_t count, vszip_minmax_props* minmax_out,
                              vszip_average_props* average_out, int32_t* fused_out, void* stream);
int vszip_limiter_device(const vszip_filter* f, const vszip_dev_clip* src, vszip_dev_clip* dst,
                         int32_t first, int32_t count, void* stream);
int vszip_limitfilter_device(const vszip_filter* f, const vszip_dev_clip* flt, const vszip_dev_clip* src,
                             const vszip_dev_clip* ref, vszip_dev_clip* dst, int32_t first, int32_t count, void* stream);
int vszip_adaptivebinarize_device(const vszip_filter* f, const vszip_dev_clip* clip, const vszip_dev_clip* clip2,
                                  vszip_dev_clip* dst, int32_t first, int32_t count, void* stream);
int vszip_clahe_device(const vszip_filter* f, const vszip_dev_clip* src, vszip_dev_clip* dst,
                       int32_t first, int32_t count, void* stream);
int vszip_colormap_device(const vszip_filter* f, const vszip_dev_clip* src, vszip_dev_clip* dst,
                          int32_t first, int32_t count, void* stream);
int vszip_cuda_stream_sync(int32_t device, void* stream);

/* ------------------------------------------------------------------ fused chains of vszip filters (SURVEY 8f rank 1)
 * A linear chain A -> B -> C of single-input vszip filters evaluated for one frame with ONE upload and ONE download:
 * intermediates stay in HBM.  Meant for the Zig glue of a filter whose input node is itself a vszip CUDA filter
 * (a create-time registry node -> vszip_filter makes that visible, see INTEGRATION.md): its getFrame requests the
 * chain's SOURCE frame instead of its immediate input and calls this.  Results are identical to calling the
 * per-filter get_frame functions one after the other.
 *  - filters: 1..16 handles in evaluation order, each created for the format of the values it reads (the source's, or, after a
 *    ColorMap, RGB24) and without ref/clipb;
 *    the chain borrows them (they must outlive it).  Two "diamond" elements are accepted as well, with the chain's
 *    SOURCE frame as their second clip: a LimitFilter created without ref (flt = the chain's current value, src = the
 *    source frame: `flt = src.vszip.X(); flt.vszip.LimitFilter(src)`) and an AdaptiveBinarize (clip = the source frame,
 *    clip2 = the current value: `src.vszip.AdaptiveBinarize(src.vszip.BoxBlur())`, the reference's own usage).
 *  - props_out[i]: for a PlaneMinMax / PlaneAverage element a pointer to its vszip_minmax_props /
 *    vszip_average_props (required), for pixel filters ignored (may be NULL).
 *  - dst: receives the planes reported by vszip_chain_planes (the union of the planes the pixel filters process);
 *    the remaining planes equal the source's.  May be NULL when the chain holds no pixel filter. */
typedef struct vszip_chain vszip_chain;
vszip_chain* vszip_chain_create(const vszip_filter* const* filters, int32_t count);
/* A chain that is a small DAG: elements may read the source or an earlier element's pixel output as their extra clips, so
 * `m = src.BoxBlur().PlaneMinMax(clipb=src)` or `src.Bilateral(ref=src.BoxBlur())` also run with one upload and one download.
 * Values are numbered 0 = the chain's source frame, k >= 1 = the pixel output of element k - 1 (which must come before the reader
 * and be a pixel filter).  For element i:
 *  - input[i]: the clip it filters (its first clip).  input == NULL: every element reads the latest pixel output before it, or the
 *    source (the linear chain of vszip_chain_create).
 *  - second[i] / third[i]: its extra clips, -1 = none: PlaneMinMax / PlaneAverage clipb, Bilateral ref, LimitFilter src (second)
 *    and ref (third), AdaptiveBinarize clip (second; input is its clip2).  Exactly the clips the filter was created with must be
 *    given.  second / third == NULL: none anywhere.
 * The chain returns the last element's pixel output, or, when the last element is a PlaneMinMax / PlaneAverage, the value it reads;
 * vszip_chain_planes reports the planes in which that value differs from the source.  Intermediates live in HBM as long as a
 * later element reads them.  vszip_chain_create(f, n) equals vszip_chain_create2 with input == NULL and second[i] = 0 for its
 * diamond elements.  An adjacent PlaneMinMax + PlaneAverage that read the same value with the same planes and clipb (or none) share
 * one read when vszip_planestats_device_b would fuse them, with bit-identical results.  Value 0 has filter 0's format and value k
 * the output format of filter k - 1 (vszip_filter_output_info); every element must have been created for the format of each value
 * it reads.  After a ColorMap every plane of the result is written, and dst has the result's format. */
vszip_chain* vszip_chain_create2(const vszip_filter* const* filters, int32_t count, const int32_t* input, const int32_t* second,
                                 const int32_t* third);
void vszip_chain_free(vszip_chain* c);
int vszip_chain_planes(const vszip_chain* c, int32_t written[3]);
int vszip_chain_get_frame(const vszip_chain* c, int32_t n, const vszip_frame* src, vszip_frame* dst, void* const* props_out);

#ifdef __cplusplus
}
#endif
#endif /* VSZIP_CUDA_H */
