// filter.h — the immutable per-instance data of the ten filters (the CUDA-side twin of the
// reference's `Data` structs) and the kernel launchers each filter uses.
#pragma once

#include "common.h"

namespace vsz {

enum FilterKind { F_BOXBLUR = 1, F_BILATERAL = 2, F_PLANEMINMAX = 3, F_PLANEAVERAGE = 4, F_LIMITER = 5, F_LIMITFILTER = 6, F_ADAPTIVEBINARIZE = 7,
                  F_CLAHE = 8, F_COLORMAP = 9, F_PACKRGB = 10 };

struct BilateralPlane {
    double sigmaS = 0, sigmaR = 0;
    int algorithm = 0;
    unsigned pbfic = 0, radius = 0, samples = 0, step = 0;
    int lut_len = 0;      // entries of the range LUT that differ from its tail value (upper + 1)
    int exact = 0;        // weights bit-identical to the reference LUT
};

}  // namespace vsz

struct vszip_filter {
    int kind;
    vszip_video_info vi;
    vsz::SampleKind sample;
    vsz::FrameLayout layout;
    // the format of the frames the filter returns, and their layout: vi / layout for every filter except ColorMap (RGB24) and
    // PackRGB (GRAY32)
    vszip_video_info out_vi;
    vsz::FrameLayout out_layout;
    bool process[3];    // the planes the filter reads (and, unless it changes the format, writes)
    bool has_input[2];  // created with its second / third input (filters.cu's kind table names them)

    // BoxBlur (src/vapoursynth/boxblur.zig:16-25)
    uint32_t hradius, vradius;
    int32_t hpasses, vpasses;

    // Bilateral (src/vapoursynth/bilateral.zig:15-31)
    vsz::BilateralPlane bl[3];
    float peak;
    int hist_len;
    std::vector<std::vector<float>> gs_host, gr_host;  // [plane]
    std::vector<std::vector<float*>> gr_dev;           // [device][plane] full range LUT in HBM
    std::vector<std::vector<float*>> gs_dev;           // [device][plane]
    std::mutex lut_mu;                                 // guards the lazy per-device upload

    // PlaneMinMax (src/vapoursynth/planeminmax.zig:15-26)
    float minthr, maxthr;
    uint32_t hist_size;
    bool no_thr;

    // PlaneAverage (src/vapoursynth/planeaverage.zig:14-22)
    std::vector<int32_t> exclude_i;
    std::vector<float> exclude_f;

    // Limiter (src/vapoursynth/limiter.zig:16-23): per-plane bounds in the sample type, held as exact doubles
    double lim_lo[3], lim_hi[3];
    std::vector<int32_t*> exclude_i_dev;  // [device] copies of lists longer than 16 entries (lazy, guarded by lut_mu)
    std::vector<float*> exclude_f_dev;
    float avg_peak;

    // LimitFilter (src/vapoursynth/limit_filter.zig:15-25): thresholds already scaled to the clip's depth
    float lf_dark[3], lf_bright[3], lf_elast[3];
    // AdaptiveBinarize (src/vapoursynth/adaptive_binarize.zig:14-19)
    int ab_c;
    // CLAHE (DESIGN.md §4.7): clip limit, tiles along x / y, histogram size 2^bits
    double clahe_limit;
    int clahe_tiles[2];
    int clahe_hs;
    // ColorMap (DESIGN.md §4.8): the selected table, R | G << 8 | B << 16 per 8-bit index
    uint32_t cmap_lut[256];
};

namespace vsz {

// boxblur_kernels.cu
int run_boxblur(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs, int count,
                int hr, int hp, int vr, int vp, cudaStream_t st);

// The BoxBlur fast paths below return 0 = done, 1 = nothing was launched; the caller runs the streaming kernels
// (boxblur_kernels.cu), < 0 = error.
// boxblur_seg_{h,v,ct}.cu: 8- and 16-bit integer clips, radius 1..22, planes up to 1920x1080 (comptime path: up to 2048 wide).
int run_seg_h(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs, int count, int r,
              int passes, cudaStream_t st);
int run_seg_v(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs, int count, int r,
              int passes, cudaStream_t st);
int run_seg_ct(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs, int count, int r,
               cudaStream_t st);

// boxblur_ctf.cu: comptime float path (f16/f32), streaming accumulators, planes of at least 2r+1 rows and columns; tmp = scratch clip
// with the layout's frame stride
int run_ctf_stream(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* tmp, size_t tmp_fs, char* dst, size_t dst_fs,
                   int count, int r, cudaStream_t st);

// bilateral_kernels.cu
struct BilateralLaunch {
    const float* gs[3];
    const float* gr[3];
    int radius[3], step[3], lut_len[3];
    float c2[3], cnorm[3];  // computed-weight form: cnorm * 2^(c2 * idx^2)
    float peak;
};
int bilateral_weights_exact(int lut_len);
int run_bilateral(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, const char* ref, size_t ref_fs,
                  char* dst, size_t dst_fs, int count, const BilateralLaunch& bp, cudaStream_t st);

// pbfic_kernels.cu: Bilateral algorithm 1 on one plane of `count` frames (ref == nullptr: non-joint)
int run_pbfic(const FrameLayout& l, int plane, const char* src, size_t src_fs, const char* ref, size_t ref_fs, char* dst, size_t dst_fs,
              int count, const float* gr_dev, int hist_len, double sigmaS, int num, float peak, cudaStream_t st);

// pointwise_kernels.cu
int run_limiter(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs, int count,
                const double lo[3], const double hi[3], cudaStream_t st);

// flt/src/ref share the layout l; ref == nullptr: the difference is judged against src
int run_limitfilter(const FrameLayout& l, const bool mask[3], const char* flt, size_t flt_fs, const char* src, size_t src_fs,
                    const char* ref, size_t ref_fs, char* dst, size_t dst_fs, int count, const float dark[3], const float bright[3],
                    const float elast[3], cudaStream_t st);
int run_adaptivebinarize(const FrameLayout& l, const char* a, size_t a_fs, const char* b, size_t b_fs, char* dst, size_t dst_fs, int count,
                         int c, cudaStream_t st);

// clahe_kernels.cu: every processed plane of an 8..16-bit integer clip; hs = 2^bits, limit >= 0 (0: no clipping), tx * ty tiles.
// Scratch for the histograms and LUTs comes from the stream-ordered pool.
int run_clahe(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs, int count, int hs,
              double limit, int tx, int ty, cudaStream_t st);

// pointwise_kernels.cu: ColorMap, plane 0 of an 8..16-bit integer clip (layout in) into the three planes of RGB24 (layout out)
int run_colormap(const FrameLayout& in, const char* src, size_t src_fs, const FrameLayout& out, char* dst, size_t dst_fs, int count,
                 const uint32_t lut[256], cudaStream_t st);

// pointwise_kernels.cu: PackRGB, the three planes of an RGB24 / RGB30 clip (layout in) into the one plane of GRAY32 (layout out)
int run_packrgb(const FrameLayout& in, const char* src, size_t src_fs, const FrameLayout& out, char* dst, size_t dst_fs, int count,
                cudaStream_t st);

// planestats_kernels.cu
struct StatsRaw {  // one per (frame, processed plane), written by the kernels
    unsigned long long isum;   // integer sum of non-excluded samples / integer sum of |a-b|
    unsigned long long idiff;
    double fsum, fdiff;
    unsigned int excluded;
    unsigned int bin_min, bin_max;  // histogram bins (threshold path) or raw integer min/max
    float fmin, fmax;               // raw float min/max (no-threshold float path)
    unsigned int pad;
};
size_t stats_scratch_bytes(int count, int nplanes);
// a and the clipb b (nullptr when there is none) share the frame stride fs
int run_planeminmax(const FrameLayout& l, const bool mask[3], const char* a, const char* b, size_t fs, int count, bool no_thr,
                    float minthr, float maxthr, uint32_t hist_size, void* scratch, StatsRaw* out_dev, cudaStream_t st);
// PlaneMinMax + PlaneAverage of the same planes (and the same clipb b, or none) from one read: 0 done, 1 not eligible, < 0 error
int run_planestats_fused(const FrameLayout& l, const bool mask[3], const char* a, const char* b, size_t fs, int count, bool no_thr,
                         float minthr, float maxthr, uint32_t hist_size, const int32_t* excl, const float* excl_f, int nex,
                         bool same_float_sums, void* scratch, StatsRaw* out_mm, StatsRaw* out_avg, cudaStream_t st);
int run_planeaverage(const FrameLayout& l, const bool mask[3], const char* a, const char* b, size_t fs, int count, const int32_t* excl_i,
                     const float* excl_f, int nex, const int32_t* excl_i_dev, const float* excl_f_dev, void* scratch, StatsRaw* out_dev,
                     cudaStream_t st);

}  // namespace vsz
