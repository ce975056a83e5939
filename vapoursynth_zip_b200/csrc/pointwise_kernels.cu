// pointwise_kernels.cu — sm_100a kernels for the pointwise neighbours of the hot path (SURVEY 8f rank 3).
//
// vszip.Limiter (src/vapoursynth/limiter.zig:24-93): dst = min(max(lo, src), hi) per processed plane, bounds per plane
// in the sample type.  One read + one write per sample: HBM-bound by construction.  A CTA streams 4 rows of a plane
// with 16-byte vectors (4 independent loads in flight per thread), two 16-bit samples per VIMNMX.U16x2.
#include <cuda_fp16.h>

#include "filter.h"

namespace vsz {

struct LimiterParams {
    uint32_t lo_w[3], hi_w[3];  // bounds replicated into a 32-bit word of samples (u8 x4, u16 x2, f16 x2, f32 / u32 x1)
};

static constexpr int LNT = 256, LROWS = 4, LGROUPS = 4;  // a CTA streams LGROUPS groups of LROWS rows

template <typename T> __device__ __forceinline__ uint32_t clamp_word(uint32_t x, uint32_t lo, uint32_t hi);
template <> __device__ __forceinline__ uint32_t clamp_word<uint8_t>(uint32_t x, uint32_t lo, uint32_t hi) { return __vminu4(__vmaxu4(lo, x), hi); }
template <> __device__ __forceinline__ uint32_t clamp_word<uint16_t>(uint32_t x, uint32_t lo, uint32_t hi) { return __vminu2(__vmaxu2(lo, x), hi); }
template <> __device__ __forceinline__ uint32_t clamp_word<uint32_t>(uint32_t x, uint32_t lo, uint32_t hi) { return min(max(lo, x), hi); }
template <> __device__ __forceinline__ uint32_t clamp_word<__half>(uint32_t x, uint32_t lo, uint32_t hi) {
    // @max / @min return the other operand when one is NaN, like __hmax2 / __hmin2
    const __half2 r = __hmin2(__hmax2(*reinterpret_cast<const __half2*>(&lo), *reinterpret_cast<const __half2*>(&x)), *reinterpret_cast<const __half2*>(&hi));
    return *reinterpret_cast<const uint32_t*>(&r);
}
template <> __device__ __forceinline__ uint32_t clamp_word<float>(uint32_t x, uint32_t lo, uint32_t hi) {
    return __float_as_uint(fminf(fmaxf(__uint_as_float(lo), __uint_as_float(x)), __uint_as_float(hi)));
}

template <typename T>
__global__ void __launch_bounds__(LNT) limiter_kernel(const BatchJob job, const LimiterParams prm) {
    int k = job.nplanes - 1;
    while (k > 0 && (int)blockIdx.x < job.pl[k].cta_begin) --k;
    const PlaneJob& pj = job.pl[k];
    const int local = (int)blockIdx.x - pj.cta_begin;
    const int yc = local * (LROWS * LGROUPS);
    const char* src = job.src + (size_t)blockIdx.y * job.src_fs + pj.src_off;
    char* dst = job.dst + (size_t)blockIdx.y * job.dst_fs + pj.dst_off;
    const uint32_t lo = prm.lo_w[pj.aux], hi = prm.hi_w[pj.aux];
    const int row_bytes = pj.w * (int)sizeof(T);
    const int nvec = row_bytes / 16;
    for (int y0 = yc; y0 < min(yc + LROWS * LGROUPS, pj.h); y0 += LROWS) {
    for (int v = threadIdx.x; v < nvec; v += LNT) {
        uint4 x[LROWS];
#pragma unroll
        for (int r = 0; r < LROWS; ++r) {
            const int y = min(y0 + r, pj.h - 1);
            x[r] = __ldg(reinterpret_cast<const uint4*>(src + (size_t)y * pj.src_pitch) + v);
        }
#pragma unroll
        for (int r = 0; r < LROWS; ++r) {
            if (y0 + r < pj.h) {  // (a `break` here would keep the loop from unrolling and serialise the loads)
                uint4 o;
                o.x = clamp_word<T>(x[r].x, lo, hi); o.y = clamp_word<T>(x[r].y, lo, hi);
                o.z = clamp_word<T>(x[r].z, lo, hi); o.w = clamp_word<T>(x[r].w, lo, hi);
                reinterpret_cast<uint4*>(dst + (size_t)(y0 + r) * pj.dst_pitch)[v] = o;
            }
        }
    }
    // row tails (< 16 bytes): one sample per thread
    const int x0 = nvec * (16 / (int)sizeof(T)) + (int)threadIdx.x;
    if (x0 < pj.w) {
        constexpr int EPW = 4 / (int)sizeof(T);
        for (int r = 0; r < LROWS && y0 + r < pj.h; ++r) {
            const T s = reinterpret_cast<const T*>(src + (size_t)(y0 + r) * pj.src_pitch)[x0];
            uint32_t wv = 0u;
            reinterpret_cast<T*>(&wv)[0] = s;
            if (EPW > 1) { for (int e = 1; e < EPW; ++e) reinterpret_cast<T*>(&wv)[e] = s; }
            const uint32_t o = clamp_word<T>(wv, lo, hi);
            reinterpret_cast<T*>(dst + (size_t)(y0 + r) * pj.dst_pitch)[x0] = reinterpret_cast<const T*>(&o)[0];
        }
    }
    }
}

template <typename T>
static int launch_limiter_t(const BatchJob& job, const LimiterParams& prm, int count, cudaStream_t st) {
    for (int f0 = 0; f0 < count; f0 += 65535) {
        const int nf = std::min(65535, count - f0);
        BatchJob j = job;
        j.src += (size_t)f0 * job.src_fs; j.dst += (size_t)f0 * job.dst_fs;
        limiter_kernel<T><<<dim3(job.ctas_per_frame, nf), LNT, 0, st>>>(j, prm);
        count_launch();
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

// lo/hi: per plane bounds already rounded to the sample type (integers as exact doubles)
int run_limiter(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs, int count,
                const double lo[3], const double hi[3], cudaStream_t st) {
    if (count <= 0) return 0;
    BatchJob job = make_batch(l, mask, src, src_fs, nullptr, 0, dst, dst_fs, [](int, int h) { return (h + LROWS * LGROUPS - 1) / (LROWS * LGROUPS); });
    if (job.ctas_per_frame == 0) return 0;
    LimiterParams prm{};
    for (int p = 0; p < 3; ++p) {
        uint32_t a = 0, b = 0;
        switch (l.kind) {
            case K_U8: a = (uint32_t)lo[p] * 0x01010101u; b = (uint32_t)hi[p] * 0x01010101u; break;
            case K_U16: a = (uint32_t)lo[p] * 0x00010001u; b = (uint32_t)hi[p] * 0x00010001u; break;
            case K_F16: {
                const __half ha = __float2half_rn((float)lo[p]), hb = __float2half_rn((float)hi[p]);
                a = (uint32_t)(*reinterpret_cast<const uint16_t*>(&ha)) * 0x00010001u;
                b = (uint32_t)(*reinterpret_cast<const uint16_t*>(&hb)) * 0x00010001u;
                break;
            }
            case K_F32: {
                const float fa = (float)lo[p], fb = (float)hi[p];
                a = *reinterpret_cast<const uint32_t*>(&fa); b = *reinterpret_cast<const uint32_t*>(&fb);
                break;
            }
            case K_U32: a = (uint32_t)lo[p]; b = (uint32_t)hi[p]; break;
        }
        prm.lo_w[p] = a; prm.hi_w[p] = b;
    }
    switch (l.kind) {
        case K_U8: return launch_limiter_t<uint8_t>(job, prm, count, st);
        case K_U16: return launch_limiter_t<uint16_t>(job, prm, count, st);
        case K_F16: return launch_limiter_t<__half>(job, prm, count, st);
        case K_F32: return launch_limiter_t<float>(job, prm, count, st);
        case K_U32: return launch_limiter_t<uint32_t>(job, prm, count, st);
    }
    return -1;
}

// =========================================================================== LimitFilter
// src/filters/limit_filter.zig:3-34: per sample, in f32, d = flt - ref, thr1 = d > 0 ? bright : dark, thr2 = thr1 * elast;
// |d| <= thr1 keeps flt, |d| >= thr2 returns src, in between src + (flt - src) * (thr2 - |d|) / (thr2 - thr1) (IEEE divide,
// separate multiply and add - the file is built with -fmad=false); integers leave as trunc(out + 0.5), f16 by RN narrowing.
// Three reads (two without ref) + one write per sample: HBM-bound; same streaming shape as limiter_kernel.
struct LimitFilterParams {
    float dark[3], bright[3], elast[3];
    const char* third;  // the ref clip when it is a separate clip, laid out like src
    size_t third_fs;
};

template <typename T> __device__ __forceinline__ float lf_load(T v) { return (float)v; }
template <> __device__ __forceinline__ float lf_load<__half>(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T lf_store(float o) { return (T)__float2int_rz(o + 0.5f); }
template <> __device__ __forceinline__ __half lf_store<__half>(float o) { return __float2half_rn(o); }
template <> __device__ __forceinline__ float lf_store<float>(float o) { return o; }

__device__ __forceinline__ float limitfilter_core(float ff, float sf, float rf, float dark, float bright, float elast) {
    const float d = ff - rf;
    const float ad = fabsf(d);
    const float t1 = d > 0.0f ? bright : dark;
    const float t2 = t1 * elast;
    if (ad <= t1) return ff;
    if (ad >= t2) return sf;
    return sf + __fdiv_rn((ff - sf) * (t2 - ad), t2 - t1);
}

template <typename T>
__device__ __forceinline__ T limitfilter_sample(T f, T s, T r, float dark, float bright, float elast) {
    return lf_store<T>(limitfilter_core(lf_load<T>(f), lf_load<T>(s), lf_load<T>(r), dark, bright, elast));
}

// One 32-bit word of samples <-> floats without the conversion pipe (I2F / F2I run at a fraction of the FP32 rate and three of
// them per sample made the kernel conversion-bound): an integer x < 2^23 is the mantissa of the float 2^23 + x, so PRMT builds
// 0x4B000000 | x and one FADD removes the bias; on the way out FADD.RZ(out + 0.5, 2^23) leaves trunc(out + 0.5) in the mantissa.
template <typename T> struct WordIO;
template <> struct WordIO<uint8_t> {
    static constexpr int N = 4;
    static __device__ __forceinline__ void unpack(uint32_t w, float v[4]) {
        v[0] = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7650)) - 8388608.0f;
        v[1] = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7651)) - 8388608.0f;
        v[2] = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7652)) - 8388608.0f;
        v[3] = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7653)) - 8388608.0f;
    }
    static __device__ __forceinline__ uint32_t pack(const float o[4]) {
        uint32_t r[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) r[i] = __float_as_uint(__fadd_rz(o[i] + 0.5f, 8388608.0f));
        return __byte_perm(__byte_perm(r[0], r[1], 0x0040), __byte_perm(r[2], r[3], 0x0040), 0x5410);
    }
};
template <> struct WordIO<uint16_t> {
    static constexpr int N = 2;
    static __device__ __forceinline__ void unpack(uint32_t w, float v[2]) {
        v[0] = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7610)) - 8388608.0f;
        v[1] = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7632)) - 8388608.0f;
    }
    static __device__ __forceinline__ uint32_t pack(const float o[2]) {
        const uint32_t a = __float_as_uint(__fadd_rz(o[0] + 0.5f, 8388608.0f)), b = __float_as_uint(__fadd_rz(o[1] + 0.5f, 8388608.0f));
        return __byte_perm(a, b, 0x5410);
    }
};
template <> struct WordIO<__half> {
    static constexpr int N = 2;
    static __device__ __forceinline__ void unpack(uint32_t w, float v[2]) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w));
        v[0] = f.x; v[1] = f.y;
    }
    static __device__ __forceinline__ uint32_t pack(const float o[2]) {
        const __half2 h = __floats2half2_rn(o[0], o[1]);
        return *reinterpret_cast<const uint32_t*>(&h);
    }
};
template <> struct WordIO<float> {
    static constexpr int N = 1;
    static __device__ __forceinline__ void unpack(uint32_t w, float v[1]) { v[0] = __uint_as_float(w); }
    static __device__ __forceinline__ uint32_t pack(const float o[1]) { return __float_as_uint(o[0]); }
};

template <typename T, bool REF>
__device__ __forceinline__ uint32_t limitfilter_word(uint32_t f, uint32_t s, uint32_t r, float dark, float bright, float elast) {
    constexpr int N = WordIO<T>::N;
    float fv[N], sv[N], rv[N], o[N];
    WordIO<T>::unpack(f, fv);
    WordIO<T>::unpack(s, sv);
    if (REF) WordIO<T>::unpack(r, rv);
#pragma unroll
    for (int e = 0; e < N; ++e) o[e] = limitfilter_core(fv[e], sv[e], REF ? rv[e] : sv[e], dark, bright, elast);
    return WordIO<T>::pack(o);
}

template <typename T, bool REF>
__global__ void __launch_bounds__(LNT) limitfilter_kernel(const BatchJob job, const LimitFilterParams prm) {
    constexpr int EPV = 16 / (int)sizeof(T);
#ifndef VSZ_LF_ROWS
#define VSZ_LF_ROWS 2
#endif
    constexpr int ROWS = VSZ_LF_ROWS;  // 2 rows x 3 inputs = 6 independent 16-byte loads in flight per thread (1 row: -10 %, 4 rows: -20..45 %)
    int k = job.nplanes - 1;
    while (k > 0 && (int)blockIdx.x < job.pl[k].cta_begin) --k;
    const PlaneJob& pj = job.pl[k];
    const int local = (int)blockIdx.x - pj.cta_begin;
    const int yc = local * (LROWS * LGROUPS);
    const char* flt = job.src + (size_t)blockIdx.y * job.src_fs + pj.src_off;
    const char* src = job.ref + (size_t)blockIdx.y * job.ref_fs + pj.ref_off;
    const char* ref = REF ? prm.third + (size_t)blockIdx.y * prm.third_fs + pj.ref_off : src;
    char* dst = job.dst + (size_t)blockIdx.y * job.dst_fs + pj.dst_off;
    // (a ternary pick: indexing the parameter arrays with a run-time plane number would copy them to local memory)
    const int pa = pj.aux;
    const float dark = pa == 0 ? prm.dark[0] : (pa == 1 ? prm.dark[1] : prm.dark[2]);
    const float bright = pa == 0 ? prm.bright[0] : (pa == 1 ? prm.bright[1] : prm.bright[2]);
    const float elast = pa == 0 ? prm.elast[0] : (pa == 1 ? prm.elast[1] : prm.elast[2]);
    const int nvec = pj.w * (int)sizeof(T) / 16;
    const int yend = min(yc + LROWS * LGROUPS, pj.h);
    for (int y0 = yc; y0 < yend; y0 += ROWS) {
        for (int v = threadIdx.x; v < nvec; v += LNT) {
            union V { uint4 q; uint32_t w[4]; };
            V f[ROWS], s[ROWS], r[ROWS];
#pragma unroll
            for (int i = 0; i < ROWS; ++i) {
                const int y = min(y0 + i, pj.h - 1);
                f[i].q = __ldg(reinterpret_cast<const uint4*>(flt + (size_t)y * pj.src_pitch) + v);
                s[i].q = __ldg(reinterpret_cast<const uint4*>(src + (size_t)y * pj.ref_pitch) + v);
                if (REF) r[i].q = __ldg(reinterpret_cast<const uint4*>(ref + (size_t)y * pj.ref_pitch) + v);
            }
#pragma unroll
            for (int i = 0; i < ROWS; ++i) {
                if (y0 + i < yend) {
                    V o;
#pragma unroll
                    for (int e = 0; e < 4; ++e) o.w[e] = limitfilter_word<T, REF>(f[i].w[e], s[i].w[e], REF ? r[i].w[e] : 0u, dark, bright, elast);
                    reinterpret_cast<uint4*>(dst + (size_t)(y0 + i) * pj.dst_pitch)[v] = o.q;
                }
            }
        }
        // row tails (< 16 bytes): one sample per thread
        const int x0 = nvec * EPV + (int)threadIdx.x;
        if (x0 < pj.w) {
            for (int i = 0; i < ROWS && y0 + i < yend; ++i) {
                const size_t y = (size_t)(y0 + i);
                const T fv = reinterpret_cast<const T*>(flt + y * pj.src_pitch)[x0];
                const T sv = reinterpret_cast<const T*>(src + y * pj.ref_pitch)[x0];
                const T rv = REF ? reinterpret_cast<const T*>(ref + y * pj.ref_pitch)[x0] : sv;
                reinterpret_cast<T*>(dst + y * pj.dst_pitch)[x0] = limitfilter_sample<T>(fv, sv, rv, dark, bright, elast);
            }
        }
    }
}

template <typename T>
static int launch_limitfilter_t(const BatchJob& job, const LimitFilterParams& prm, int count, cudaStream_t st) {
    for (int f0 = 0; f0 < count; f0 += 65535) {
        const int nf = std::min(65535, count - f0);
        BatchJob j = job;
        LimitFilterParams p = prm;
        j.src += (size_t)f0 * job.src_fs; j.ref += (size_t)f0 * job.ref_fs; j.dst += (size_t)f0 * job.dst_fs;
        if (p.third) { p.third += (size_t)f0 * p.third_fs; limitfilter_kernel<T, true><<<dim3(job.ctas_per_frame, nf), LNT, 0, st>>>(j, p); }
        else limitfilter_kernel<T, false><<<dim3(job.ctas_per_frame, nf), LNT, 0, st>>>(j, p);
        count_launch();
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

int run_limitfilter(const FrameLayout& l, const bool mask[3], const char* flt, size_t flt_fs, const char* src, size_t src_fs,
                    const char* ref, size_t ref_fs, char* dst, size_t dst_fs, int count, const float dark[3], const float bright[3],
                    const float elast[3], cudaStream_t st) {
    if (count <= 0) return 0;
    BatchJob job = make_batch(l, mask, flt, flt_fs, src, src_fs, dst, dst_fs, [](int, int h) { return (h + LROWS * LGROUPS - 1) / (LROWS * LGROUPS); });
    if (job.ctas_per_frame == 0) return 0;
    LimitFilterParams prm{};
    for (int p = 0; p < 3; ++p) { prm.dark[p] = dark[p]; prm.bright[p] = bright[p]; prm.elast[p] = elast[p]; }
    prm.third = ref; prm.third_fs = ref_fs;
    switch (l.kind) {
        case K_U8: return launch_limitfilter_t<uint8_t>(job, prm, count, st);
        case K_U16: return launch_limitfilter_t<uint16_t>(job, prm, count, st);
        case K_F16: return launch_limitfilter_t<__half>(job, prm, count, st);
        case K_F32: return launch_limitfilter_t<float>(job, prm, count, st);
    }
    return -1;
}

// =========================================================================== AdaptiveBinarize
// src/vapoursynth/adaptive_binarize.zig:48-60: 8-bit, every plane, dst = (clip2 - clip >= c) ? 255 : 0.  Four samples per
// byte-SIMD instruction: for c > 0 the test is usat(b - a) >= c, for c <= 0 it is usat(a - b) <= -c (a negative a - b
// saturates to 0 and passes, as it must); c = 256 can never hold.  The compare instructions produce 0xff per true byte.
struct BinarizeParams { int mode; uint32_t k4; };  // mode 0: ge, 1: le, 2: constant 0

__device__ __forceinline__ uint32_t binarize_word(uint32_t a, uint32_t b, int mode, uint32_t k4) {
    if (mode == 0) return __vcmpgeu4(__vsubus4(b, a), k4);
    if (mode == 1) return __vcmpleu4(__vsubus4(a, b), k4);
    return 0u;
}

#ifndef VSZ_AB_ROWS
#define VSZ_AB_ROWS 2  // measured on B200: 1 row 71 %, 2 rows 97 %, 4 rows 91 %, 8 rows 84 % of the HBM peak (registers vs loads in flight)
#endif
__global__ void __launch_bounds__(LNT) adaptivebinarize_kernel(const BatchJob job, const BinarizeParams prm) {
    int k = job.nplanes - 1;
    while (k > 0 && (int)blockIdx.x < job.pl[k].cta_begin) --k;
    const PlaneJob& pj = job.pl[k];
    constexpr int ABR = VSZ_AB_ROWS;
    const int local = (int)blockIdx.x - pj.cta_begin;
    const int yc = local * ((LROWS * LGROUPS));
    const char* a = job.src + (size_t)blockIdx.y * job.src_fs + pj.src_off;
    const char* b = job.ref + (size_t)blockIdx.y * job.ref_fs + pj.ref_off;
    char* dst = job.dst + (size_t)blockIdx.y * job.dst_fs + pj.dst_off;
    const int nvec = pj.w / 16;
    const int yend = min(yc + (LROWS * LGROUPS), pj.h);
    for (int y0 = yc; y0 < yend; y0 += ABR) {
        for (int v = threadIdx.x; v < nvec; v += LNT) {
            uint4 x[ABR], z[ABR];
#pragma unroll
            for (int r = 0; r < ABR; ++r) {
                const int y = min(y0 + r, pj.h - 1);
                x[r] = __ldg(reinterpret_cast<const uint4*>(a + (size_t)y * pj.src_pitch) + v);
                z[r] = __ldg(reinterpret_cast<const uint4*>(b + (size_t)y * pj.ref_pitch) + v);
            }
#pragma unroll
            for (int r = 0; r < ABR; ++r) {
                if (y0 + r < yend) {
                    uint4 o;
                    o.x = binarize_word(x[r].x, z[r].x, prm.mode, prm.k4); o.y = binarize_word(x[r].y, z[r].y, prm.mode, prm.k4);
                    o.z = binarize_word(x[r].z, z[r].z, prm.mode, prm.k4); o.w = binarize_word(x[r].w, z[r].w, prm.mode, prm.k4);
                    reinterpret_cast<uint4*>(dst + (size_t)(y0 + r) * pj.dst_pitch)[v] = o;
                }
            }
        }
        const int x0 = nvec * 16 + (int)threadIdx.x;
        if (x0 < pj.w) {
            for (int r = 0; r < ABR && y0 + r < yend; ++r) {
                const size_t y = (size_t)(y0 + r);
                const uint32_t av = (uint8_t)a[y * pj.src_pitch + x0], bv = (uint8_t)b[y * pj.ref_pitch + x0];
                dst[y * pj.dst_pitch + x0] = (char)(binarize_word(av, bv, prm.mode, prm.k4) & 0xffu);
            }
        }
    }
}

int run_adaptivebinarize(const FrameLayout& l, const char* a, size_t a_fs, const char* b, size_t b_fs, char* dst, size_t dst_fs, int count,
                         int c, cudaStream_t st) {
    if (count <= 0) return 0;
    if (l.kind != K_U8) return -1;
    const bool all[3] = {true, true, true};
    BatchJob job = make_batch(l, all, a, a_fs, b, b_fs, dst, dst_fs, [](int, int h) { return (h + LROWS * LGROUPS - 1) / (LROWS * LGROUPS); });
    if (job.ctas_per_frame == 0) return 0;
    BinarizeParams prm{};
    if (c > 255) { prm.mode = 2; prm.k4 = 0u; }
    else if (c > 0) { prm.mode = 0; prm.k4 = (uint32_t)c * 0x01010101u; }
    else { prm.mode = 1; prm.k4 = (uint32_t)std::min(-c, 255) * 0x01010101u; }
    for (int f0 = 0; f0 < count; f0 += 65535) {
        const int nf = std::min(65535, count - f0);
        BatchJob j = job;
        j.src += (size_t)f0 * job.src_fs; j.ref += (size_t)f0 * job.ref_fs; j.dst += (size_t)f0 * job.dst_fs;
        adaptivebinarize_kernel<<<dim3(job.ctas_per_frame, nf), LNT, 0, st>>>(j, prm);
        count_launch();
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

// =========================================================================== ColorMap
// DESIGN.md §4.8: plane 0 of an 8..16-bit integer clip through one of OpenCV's colormaps into the three planes of RGB24,
// i = min(x >> (bits - 8), 255), (R, G, B) = table[i].  One 16-byte load (two for 9..16 bits) per 16 samples, 16 gathers, and
// three 16-byte stores: 1 + 3 bytes per sample at 8 bits, 2 + 3 above, HBM-bound by construction.  Every CTA copies the 1 KB
// table into shared memory once per bank, word [i][lane] (32 KB), so that each lane gathers from its own bank: a gather is
// conflict-free whatever the indices.  Work items (row, 16 samples) of a CTA's rows are spread over all threads, so rows
// narrower than 256 vectors keep every thread busy.
static constexpr int CMT = 256, CM_UNROLL = 4, CM_ITEMS = 8;  // CM_ITEMS: work items per thread a CTA's rows are sized for

struct ColorMapJob {
    const char* src;
    char* dst;
    size_t src_fs, dst_fs;
    size_t dst_off[3];     // R, G, B planes
    int src_pitch, dst_pitch;
    int w, h, rows;        // rows: per CTA
    int shift;             // bits - 8
    uint32_t lut[256];
};

// four table words -> the R, G and B bytes of four samples, one word per plane (7 PRMT)
__device__ __forceinline__ void cm_pack4(uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t& r, uint32_t& g, uint32_t& bl) {
    const uint32_t ab = __byte_perm(a, b, 0x5140), cd = __byte_perm(c, d, 0x5140);  // R0 R1 G0 G1 / R2 R3 G2 G3
    r = __byte_perm(ab, cd, 0x5410);
    g = __byte_perm(ab, cd, 0x7632);
    bl = __byte_perm(__byte_perm(a, b, 0x0062), __byte_perm(c, d, 0x0062), 0x5410);
}

template <typename T>
__device__ __forceinline__ uint32_t cm_index(uint32_t word, int e, int shift) {
    if (sizeof(T) == 1) return __byte_perm(word, 0u, 0x4440 | e);
    return min((e ? word >> 16 : word & 0xffffu) >> shift, 255u);
}

template <typename T>
__global__ void __launch_bounds__(CMT) colormap_kernel(const __grid_constant__ ColorMapJob job) {
    __shared__ uint32_t tab[256 * 32];
    for (int i = threadIdx.x; i < 256 * 32; i += CMT) tab[i] = job.lut[i >> 5];
    __syncthreads();
    const uint32_t* my = tab + (threadIdx.x & 31);
    constexpr int LOADS = (int)sizeof(T);  // 16-byte loads per 16 samples
    const int y0 = (int)blockIdx.x * job.rows, nrows = min(job.rows, job.h - y0);
    const char* src = job.src + (size_t)blockIdx.y * job.src_fs + (size_t)y0 * job.src_pitch;
    char* dst = job.dst + (size_t)blockIdx.y * job.dst_fs + (size_t)y0 * job.dst_pitch;
    char* const r_pl = dst + job.dst_off[0];
    char* const g_pl = dst + job.dst_off[1];
    char* const b_pl = dst + job.dst_off[2];
    const int nvec = job.w / 16, items = nrows * nvec;
    for (int it0 = threadIdx.x; it0 < items; it0 += CMT * CM_UNROLL) {
        uint4 x[CM_UNROLL][LOADS];
#pragma unroll
        for (int u = 0; u < CM_UNROLL; ++u) {
            const int it = min(it0 + u * CMT, items - 1);
            const int y = it / nvec, v = it - y * nvec;
            const uint4* p = reinterpret_cast<const uint4*>(src + (size_t)y * job.src_pitch) + v * LOADS;
#pragma unroll
            for (int l = 0; l < LOADS; ++l) x[u][l] = __ldg(p + l);
        }
#pragma unroll
        for (int u = 0; u < CM_UNROLL; ++u) {
            const int it = it0 + u * CMT;
            if (it < items) {
                const uint32_t* w = reinterpret_cast<const uint32_t*>(x[u]);
                constexpr int SPW = 4 / (int)sizeof(T);  // samples per input word
                uint32_t o[3][4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {  // output word q: samples 4q .. 4q + 3
                    uint32_t t[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int s = 4 * q + e;
                        t[e] = my[cm_index<T>(w[s / SPW], s % SPW, job.shift) << 5];
                    }
                    cm_pack4(t[0], t[1], t[2], t[3], o[0][q], o[1][q], o[2][q]);
                }
                const int y = it / nvec, v = it - y * nvec;
                const size_t off = (size_t)y * job.dst_pitch + (size_t)v * 16;
                *reinterpret_cast<uint4*>(r_pl + off) = make_uint4(o[0][0], o[0][1], o[0][2], o[0][3]);
                *reinterpret_cast<uint4*>(g_pl + off) = make_uint4(o[1][0], o[1][1], o[1][2], o[1][3]);
                *reinterpret_cast<uint4*>(b_pl + off) = make_uint4(o[2][0], o[2][1], o[2][2], o[2][3]);
            }
        }
    }
    // row tails (< 16 samples): one sample per thread
    const int tail = job.w - nvec * 16;
    for (int it = threadIdx.x; it < nrows * tail; it += CMT) {
        const int y = it / tail, x0 = nvec * 16 + (it - y * tail);
        const uint32_t s = reinterpret_cast<const T*>(src + (size_t)y * job.src_pitch)[x0];
        const uint32_t t = my[cm_index<T>(s, 0, job.shift) << 5];
        const size_t off = (size_t)y * job.dst_pitch + x0;
        r_pl[off] = (char)(t & 0xffu);
        g_pl[off] = (char)((t >> 8) & 0xffu);
        b_pl[off] = (char)((t >> 16) & 0xffu);
    }
}

int run_colormap(const FrameLayout& in, const char* src, size_t src_fs, const FrameLayout& out, char* dst, size_t dst_fs, int count,
                 const uint32_t lut[256], cudaStream_t st) {
    if (count <= 0) return 0;
    if ((in.kind != K_U8 && in.kind != K_U16) || out.kind != K_U8 || out.nplanes != 3) return -1;
    ColorMapJob job{};
    job.src = src; job.dst = dst; job.src_fs = src_fs; job.dst_fs = dst_fs;
    for (int p = 0; p < 3; ++p) job.dst_off[p] = out.pl[p].offset;
    job.src_pitch = in.pl[0].pitch; job.dst_pitch = out.pl[0].pitch;
    job.w = in.pl[0].w; job.h = in.pl[0].h;
    job.shift = in.bits - 8;
    job.rows = std::max(1, std::min(job.h, CMT * CM_ITEMS / std::max(1, job.w / 16)));
    for (int i = 0; i < 256; ++i) job.lut[i] = lut[i];
    const int ctas = (job.h + job.rows - 1) / job.rows;
    for (int f0 = 0; f0 < count; f0 += 65535) {
        const int nf = std::min(65535, count - f0);
        ColorMapJob j = job;
        j.src += (size_t)f0 * src_fs; j.dst += (size_t)f0 * dst_fs;
        if (in.kind == K_U8) colormap_kernel<uint8_t><<<dim3(ctas, nf), CMT, 0, st>>>(j);
        else colormap_kernel<uint16_t><<<dim3(ctas, nf), CMT, 0, st>>>(j);
        count_launch();
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace vsz
