// bilateral_kernels.cu — sm_100a kernel for vszip.Bilateral, algorithm 2 ("truncated" window).
//
// Semantics restated from src/filters/bilateral.zig:178-304: per output pixel, a centre tap plus
// (yy, xx) in {1, 1+step, ...} <= radius, four diagonal taps each, weights gs[yy][xx] * gr[range index],
// f32 accumulation with separate multiply/add in the reference's association order, replicate edges.
//
// Design: a CTA computes a 32x8 tile.  The tile plus halo is staged once in shared memory, already
// widened to f32 and with edge replication applied, so every tap is a conflict-free LDS.  The range
// weight comes from one of three sources, chosen per plane at create time:
//   W_SMEM    the reference's LUT copied to shared memory (8..12-bit clips, or small sigmaR where the LUT
//             is short): bit-identical weights;
//   W_COMPUTE C * 2^(c2 * idx^2) on the MUFU unit when the LUT (up to 256 KB) does not fit in shared
//             memory: weights within ~2 ulp, integer outputs within 1 LSB;
//   W_SCALED  W_COMPUTE for integer clips whose LUT is never clamped (sigmaR >= 1/8): the tile is staged already multiplied
//             by sqrt(-c2), so a tap's weight is 2^(-(a'-b')^2): FSUB, FMUL, MUFU instead of FSUB, FMNMX, FMUL, FMUL, MUFU;
//             also f32 clips with sigmaR >= ~1.95 (one FMNMX more per tap for the clamp of |a-b| to 1), where skipping the
//             quantisation of the range index moves the result by < 4e-6 relative;
//   W_GLOBAL  gathers from the full LUT in HBM/L2: bit-identical, slow (validation / VSZIP_BILATERAL_EXACT=1).
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "filter.h"

namespace vsz {

enum WeightMode { W_SMEM = 0, W_COMPUTE = 1, W_GLOBAL = 2, W_SCALED = 3 };

static constexpr int TW = 32, TH = 8, TILE = 32;

struct BilateralPlaneParams {
    const float* gs;   // (radius+1)^2, device
    const float* gr;   // full LUT, device
    int radius, step;
    int lut_len;       // entries [0, lut_len) are distinct; larger indices use gr[lut_len-1]
    int smem_lut;      // entries copied to shared memory (W_SMEM)
    float c2, cnorm;   // W_COMPUTE: weight = cnorm * exp2(c2 * idx^2)
    float scale, inv_scale;  // W_SCALED: sqrt(-c2) (x 65535 for f32 clips: the range index is |a-b|*65535 there) and its reciprocal
    float dmax;              // W_SCALED on f32 clips: the scaled difference of min(1, |a-b|) = 1
};

struct BilateralParams {
    BilateralPlaneParams pl[1];  // the launch's plane
    float peak;
    int tiles_x[3];              // 32x32 tiles per row, indexed like job.pl[]
    int strips_x[3];             // CTAs per tile row
    int strip;                   // tiles per CTA
};

// Integer samples reach f32 and come back without the conversion unit: I2F / F2I share the quarter-rate XU pipe with MUFU.EX2,
// which is the pipe that bounds this kernel (ncu: 16 EX2 + 2.5 conversions + 1 RCP per pixel on config 3).  x < 2^23 is the
// mantissa of the float 2^23 + x: OR in the exponent, subtract the bias (exact); on the way out FADD.RZ(v, 2^23) leaves trunc(v) in
// the mantissa for 0 <= v < 2^23.
template <typename T> __device__ __forceinline__ float widen(T v) { return __fsub_rn(__uint_as_float(0x4B000000u | (unsigned int)v), 8388608.0f); }
template <> __device__ __forceinline__ float widen<float>(float v) { return v; }
__device__ __forceinline__ unsigned int trunc_to_uint(float v) { return __float_as_uint(__fadd_rz(v, 8388608.0f)) & 0x7fffffu; }
template <> __device__ __forceinline__ float widen<__half>(__half v) { return __half2float(v); }

template <typename T> struct BTr { static constexpr bool flt = false; };
template <> struct BTr<__half> { static constexpr bool flt = true; };
template <> struct BTr<float> { static constexpr bool flt = true; };

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Range index (src/filters/bilateral.zig:15-22) as an exact non-negative integer held in a float:
// integer clips |a-b| (both < 2^16, exact); float clips trunc(min(1,|a-b|)*65535 + 0.5) with the
// subtraction rounded in T.  Keeping it in a float avoids an int<->float conversion pair per tap.
template <typename T> __device__ __forceinline__ float range_index_f(float a, float b) {
    float d = __fsub_rn(a, b);
    if constexpr (BTr<T>::flt) {
        if constexpr (sizeof(T) == 2) d = __half2float(__float2half_rn(d));  // the subtraction is rounded in f16
        const float m = fminf(1.0f, fabsf(d));
        return truncf(__fadd_rn(__fmul_rn(m, 65535.0f), 0.5f));
    } else {
        return fabsf(d);
    }
}

// weight of range index `fi` (an integer-valued float); `top` = lut_len - 1
template <int WM>
__device__ __forceinline__ float range_weight(float fi, float top, const BilateralPlaneParams& pp, const float* s_lut) {
    fi = fminf(fi, top);
    if constexpr (WM == W_COMPUTE) {
        return ex2_approx(__fmul_rn(__fmul_rn(fi, fi), pp.c2));  // un-normalised: the constant cancels in sum/wsum
    } else {
        const int idx = __float_as_int(__fadd_rn(fi, 8388608.0f)) & 0x7fffff;  // exact: fi is an integer < 2^23
        if constexpr (WM == W_SMEM) return s_lut[idx];
        else return __ldg(pp.gr + idx);
    }
}

// One CTA (32x8 threads) walks a horizontal strip of `prm.strip` 32x32-pixel tiles; every thread produces
// 4 pixels per tile (rows ty, ty+8, ty+16, ty+24).  The spatial table and - in W_SMEM mode - the range
// LUT are loaded once per CTA and reused by every tile of the strip.
// SAMPLES/STEP > 0: the tap pattern (radius = 1 + (SAMPLES-1)*STEP) is a compile-time constant, so the tile pitch
// and every tap offset become immediates and the tap loops unroll; SAMPLES == 0: any radius/step at run time.
template <typename T, bool JOINT, int WM, int SAMPLES, int STEP>
__global__ void __launch_bounds__(TW * TH) bilateral_kernel(const BatchJob job, const BilateralParams prm) {
    extern __shared__ float smem_f[];
    // one plane per launch (planes differ in radius, weight source and shared-memory size): its descriptors sit at index 0, so every
    // parameter is a constant-bank operand at a fixed offset (a run-time plane index cost 6.5 LDC per pixel in the ncu instruction mix)
    constexpr int k = 0;
    const PlaneJob& pj = job.pl[0];
    const BilateralPlaneParams& pp = prm.pl[0];
    const int local = blockIdx.x;
    const int strips_x = prm.strips_x[k];
    const int sx = local % strips_x, ty0 = local / strips_x;
    const int y0 = ty0 * TILE;
    constexpr bool FIXED = SAMPLES > 0;
    const int r = FIXED ? 1 + (SAMPLES - 1) * STEP : pp.radius, step = FIXED ? STEP : pp.step, r2 = r + 1;
    const int tw = TILE + 2 * r, th = TILE + 2 * r, tsize = tw * th;
    const uint32_t inv_tw = ((1u << 20) + (uint32_t)tw - 1u) / (uint32_t)tw;  // exact e / tw for e < 2^12

    float* s_src = smem_f;
    float* s_ref = JOINT ? s_src + tsize : s_src;
    float* s_gs = s_ref + tsize;
    float* s_lut = s_gs + r2 * r2;

    const char* src = job.src + (size_t)blockIdx.y * job.src_fs + pj.src_off;
    const char* ref = JOINT ? job.ref + (size_t)blockIdx.y * job.ref_fs + pj.ref_off : nullptr;
    char* dst = job.dst + (size_t)blockIdx.y * job.dst_fs + pj.dst_off;
    const int tid = threadIdx.y * TW + threadIdx.x;
    for (int i = tid; i < r2 * r2; i += TW * TH) s_gs[i] = pp.gs[i];
    if constexpr (WM == W_SMEM)
        for (int i = tid; i < pp.smem_lut; i += TW * TH) s_lut[i] = pp.gr[i];
    const float top = (float)(pp.lut_len - 1);

    const int tile_end = min((sx + 1) * prm.strip, prm.tiles_x[k]);
    // compile-time tap patterns: the tile size is a constant, so the NEXT tile's samples are fetched into registers
    // before the current tile's math (their latency is covered by ~300 instructions per pixel) and only written to
    // shared memory at the top of the next iteration
    constexpr int TSIZE_C = FIXED ? (TILE + 2 * (1 + (SAMPLES - 1) * STEP)) * (TILE + 2 * (1 + (SAMPLES - 1) * STEP)) : 1;
    constexpr int NPT = FIXED ? (TSIZE_C + TW * TH - 1) / (TW * TH) : 1;
    T pre_s[NPT], pre_r[JOINT ? NPT : 1];
    float sw_reg[FIXED ? SAMPLES : 1][FIXED ? SAMPLES : 1];  // the spatial weights of the pattern live in registers
    if constexpr (FIXED) {
#pragma unroll
        for (int a = 0; a < SAMPLES; ++a)
#pragma unroll
            for (int b = 0; b < SAMPLES; ++b) sw_reg[a][b] = __ldg(pp.gs + (1 + a * STEP) * r2 + (1 + b * STEP));
    }
    // per-thread staging geometry is the same for every tile of the strip: the (edge-clamped) row offset and the
    // column relative to the tile are computed once, a tile then costs an add, a clamp and the address per sample
    int row_off[NPT], ref_off[JOINT ? NPT : 1], lxr[NPT];
    if constexpr (FIXED) {
#pragma unroll
        for (int i = 0; i < NPT; ++i) {
            const int e = min(tid + i * (TW * TH), tsize - 1);
            const int ly = (int)(((uint32_t)e * inv_tw) >> 20);
            lxr[i] = e - ly * tw - r;
            const int gy = min(max(y0 + ly - r, 0), pj.h - 1);
            row_off[i] = gy * pj.src_pitch;
            if constexpr (JOINT) ref_off[i] = gy * pj.ref_pitch;
        }
    }
    auto fetch_tile = [&](int tx) {
        const int x0 = tx * TILE;
        const bool inner = x0 >= r && x0 + TILE + r <= pj.w;  // tile + halo inside the plane's columns: no clamps (most tiles)
#pragma unroll
        for (int i = 0; i < NPT; ++i) {
            if (i < NPT - 1 || tid + i * (TW * TH) < tsize) {   // only the last round of a tile is partial
                const int gx = inner ? x0 + lxr[i] : min(max(x0 + lxr[i], 0), pj.w - 1);
                pre_s[i] = reinterpret_cast<const T*>(src + row_off[i])[gx];
                if constexpr (JOINT) pre_r[i] = reinterpret_cast<const T*>(ref + ref_off[i])[gx];
            }
        }
    };
    if constexpr (FIXED) fetch_tile(sx * prm.strip);
    for (int tx = sx * prm.strip; tx < tile_end; ++tx) {
        const int x0 = tx * TILE;
        __syncthreads();  // previous tile fully consumed (and the tables visible on the first pass)
        // tile + halo, widened to f32, replicate edges (src/filters/bilateral.zig:281-289)
        if constexpr (FIXED) {
#pragma unroll
            for (int i = 0; i < NPT; ++i) {
                const int e = tid + i * (TW * TH);
                if (i < NPT - 1 || e < tsize) {
                    const float sv = widen<T>(pre_s[i]);
                    s_src[e] = (WM == W_SCALED && !JOINT) ? __fmul_rn(sv, pp.scale) : sv;
                    if constexpr (JOINT) {
                        const float rv = widen<T>(pre_r[i]);
                        s_ref[e] = (WM == W_SCALED) ? __fmul_rn(rv, pp.scale) : rv;
                    }
                }
            }
            if (tx + 1 < tile_end) fetch_tile(tx + 1);
        } else {
            for (int e = tid; e < tsize; e += TW * TH) {
                const int ly = (int)(((uint32_t)e * inv_tw) >> 20), lx = e - ly * tw;
                const int gy = min(max(y0 + ly - r, 0), pj.h - 1), gx = min(max(x0 + lx - r, 0), pj.w - 1);
                const float sv = widen<T>(reinterpret_cast<const T*>(src + (size_t)gy * pj.src_pitch)[gx]);
                s_src[e] = (WM == W_SCALED && !JOINT) ? __fmul_rn(sv, pp.scale) : sv;
                if constexpr (JOINT) {
                    const float rv = widen<T>(reinterpret_cast<const T*>(ref + (size_t)gy * pj.ref_pitch)[gx]);
                    s_ref[e] = (WM == W_SCALED) ? __fmul_rn(rv, pp.scale) : rv;
                }
            }
        }
        __syncthreads();
        const int x = x0 + threadIdx.x;
#pragma unroll
        for (int sub = 0; sub < TILE / TH; ++sub) {
            const int lyo = threadIdx.y + sub * TH, y = y0 + lyo;
            if (x >= pj.w || y >= pj.h) continue;
            const int cxy = (lyo + r) * tw + threadIdx.x + r;
            const float cref = s_ref[cxy];
            float wsum = (WM == W_SCALED) ? s_gs[0] : __fmul_rn(s_gs[0], range_weight<WM == W_SCALED ? W_COMPUTE : WM>(0.0f, top, pp, s_lut));
            float sum = __fmul_rn(s_src[cxy], wsum);
            auto taps = [&](int yy, int xx, float sw) {
                const int up = cxy - yy * tw, dn = cxy + yy * tw;
                const float r1 = s_ref[up + xx], r2v = s_ref[dn + xx], r3 = s_ref[up - xx], r4 = s_ref[dn - xx];
                const float v1 = JOINT ? s_src[up + xx] : r1, v2 = JOINT ? s_src[dn + xx] : r2v;
                const float v3 = JOINT ? s_src[up - xx] : r3, v4 = JOINT ? s_src[dn - xx] : r4;
                float g1, g2, g3, g4;
                if constexpr (WM == W_SCALED) {
                    float d1 = __fsub_rn(cref, r1), d2 = __fsub_rn(cref, r2v), d3 = __fsub_rn(cref, r3), d4 = __fsub_rn(cref, r4);
                    if constexpr (BTr<T>::flt) {  // rangeIndex clamps float differences to 1 (samples outside [0, 1] are legal)
                        d1 = fminf(fabsf(d1), pp.dmax); d2 = fminf(fabsf(d2), pp.dmax); d3 = fminf(fabsf(d3), pp.dmax); d4 = fminf(fabsf(d4), pp.dmax);
                    }
                    g1 = ex2_approx(__fmul_rn(-d1, d1)); g2 = ex2_approx(__fmul_rn(-d2, d2));
                    g3 = ex2_approx(__fmul_rn(-d3, d3)); g4 = ex2_approx(__fmul_rn(-d4, d4));
                } else {
                    g1 = range_weight<WM>(range_index_f<T>(cref, r1), top, pp, s_lut);
                    g2 = range_weight<WM>(range_index_f<T>(cref, r2v), top, pp, s_lut);
                    g3 = range_weight<WM>(range_index_f<T>(cref, r3), top, pp, s_lut);
                    g4 = range_weight<WM>(range_index_f<T>(cref, r4), top, pp, s_lut);
                }
                const float gsum = __fadd_rn(__fadd_rn(__fadd_rn(g1, g2), g3), g4);
                if constexpr (WM == W_SCALED) {
                    // computed weights are approximate anyway (<= 1 LSB bar): fused multiply-adds save 5 of 30 instructions
                    wsum = __fmaf_rn(sw, gsum, wsum);
                    const float psum = __fmaf_rn(v4, g4, __fmaf_rn(v3, g3, __fmaf_rn(v2, g2, __fmul_rn(v1, g1))));
                    sum = __fmaf_rn(sw, psum, sum);
                } else {
                    wsum = __fadd_rn(wsum, __fmul_rn(sw, gsum));
                    const float p1 = __fmul_rn(v1, g1), p2 = __fmul_rn(v2, g2), p3 = __fmul_rn(v3, g3), p4 = __fmul_rn(v4, g4);
                    const float psum = __fadd_rn(__fadd_rn(__fadd_rn(p1, p2), p3), p4);
                    sum = __fadd_rn(sum, __fmul_rn(sw, psum));
                }
            };
            if constexpr (FIXED) {
#pragma unroll
                for (int a = 0; a < SAMPLES; ++a)
#pragma unroll
                    for (int b = 0; b < SAMPLES; ++b) taps(1 + a * STEP, 1 + b * STEP, sw_reg[a][b]);
            } else {
                for (int yy = 1; yy < r2; yy += step)
                    for (int xx = 1; xx < r2; xx += step) taps(yy, xx, s_gs[yy * r2 + xx]);
            }
            float q;
            if constexpr (WM == W_SCALED) {
                // approximate-weights mode: reciprocal on the MUFU unit (2 ulp) instead of the IEEE divide sequence;
                // non-joint values were staged scaled, so the scale goes back in here
                float rw;
                asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rw) : "f"(wsum));
                if constexpr (!JOINT && !BTr<T>::flt) q = __fmaf_rn(__fmul_rn(sum, rw), pp.inv_scale, 0.5f);  // + 0.5: see the store below
                else q = __fmul_rn(sum, JOINT ? rw : __fmul_rn(rw, pp.inv_scale));
            } else {
                q = __fdiv_rn(sum, wsum);
            }
            T* out = reinterpret_cast<T*>(dst + (size_t)y * pj.dst_pitch) + x;
            if constexpr (std::is_same<T, float>::value) *out = q;
            else if constexpr (std::is_same<T, __half>::value) *out = __float2half_rn(q);
            else if constexpr (WM == W_SCALED && !JOINT) {
                // q = (sum * rw) * inv_scale was formed above; the rounding offset rides on the same multiply here instead
                // (approximate-weights mode): trunc(clamp(sum * rw * inv_scale + 0.5, 0, peak))
                *out = (T)trunc_to_uint(fminf(fmaxf(q, 0.0f), prm.peak));
            }
            else *out = (T)trunc_to_uint(fminf(fmaxf(__fadd_rn(q, 0.5f), 0.0f), prm.peak));  // trunc(clamp(q + 0.5, 0, peak))
        }
    }
}

// =========================================================================== host
static constexpr int kSmemLutMaxEntries = 12288;  // 48 KB

static int weight_mode_for(int lut_len) {
    static const bool force_exact = [] { const char* e = getenv("VSZIP_BILATERAL_EXACT"); return e && e[0] == '1'; }();
    if (lut_len <= kSmemLutMaxEntries) return W_SMEM;
    return force_exact ? W_GLOBAL : W_COMPUTE;
}

int bilateral_weights_exact(int lut_len) { return weight_mode_for(lut_len) != W_COMPUTE; }

template <typename T, bool JOINT, int WM, int SAMPLES, int STEP>
static int launch_one(const BatchJob& j, const BilateralParams& prm, int nf, size_t smem, cudaStream_t st) {
    auto kern = bilateral_kernel<T, JOINT, WM, SAMPLES, STEP>;
    VSZ_CUDA(allow_max_dynamic_smem(kern));
    kern<<<dim3(j.ctas_per_frame, nf), dim3(TW, TH), smem, st>>>(j, prm);
    count_launch();
    return 0;
}

template <typename T, bool JOINT>
static int launch_mode(int wm, int samples, int step, const BatchJob& j, const BilateralParams& prm, int nf, size_t smem, cudaStream_t st) {
    if constexpr (!JOINT) {
        // specialised tap patterns: sigmaS up to 7.5 (bilateral.zig:164-190 yields exactly these (samples, step) pairs)
#define VSZ_BL(SA, SE)                                                                                           \
        if (samples == SA && step == SE) {                                                                          \
            if (wm == W_SMEM) return launch_one<T, false, W_SMEM, SA, SE>(j, prm, nf, smem, st);                     \
            if (wm == W_COMPUTE) return launch_one<T, false, W_COMPUTE, SA, SE>(j, prm, nf, smem, st);               \
            if (wm == W_SCALED) return launch_one<T, false, W_SCALED, SA, SE>(j, prm, nf, smem, st);                 \
        }
        VSZ_BL(1, 1) VSZ_BL(2, 1) VSZ_BL(2, 2) VSZ_BL(3, 2) VSZ_BL(3, 3) VSZ_BL(4, 3)
#undef VSZ_BL
    }
    if (wm == W_SMEM) return launch_one<T, JOINT, W_SMEM, 0, 0>(j, prm, nf, smem, st);
    if (wm == W_COMPUTE) return launch_one<T, JOINT, W_COMPUTE, 0, 0>(j, prm, nf, smem, st);
    if (wm == W_SCALED) return launch_one<T, JOINT, W_SCALED, 0, 0>(j, prm, nf, smem, st);
    return launch_one<T, JOINT, W_GLOBAL, 0, 0>(j, prm, nf, smem, st);
}

template <typename T>
static int run_bilateral_t(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, const char* ref, size_t rfs, char* dst,
                           size_t dfs, int count, const BilateralLaunch& bp, cudaStream_t st) {
    // planes with different weight sources / radii need different shared-memory sizes: one launch per plane
    for (int p = 0; p < l.nplanes; ++p) {
        if (!mask[p]) continue;
        bool one[3] = {false, false, false};
        one[p] = true;
        BilateralParams prm{};
        prm.peak = bp.peak;
        BilateralPlaneParams& pp = prm.pl[0];
        pp.gs = bp.gs[p]; pp.gr = bp.gr[p];
        pp.radius = bp.radius[p]; pp.step = bp.step[p];
        pp.lut_len = bp.lut_len[p];
        int wm = weight_mode_for(pp.lut_len);
        pp.smem_lut = wm == W_SMEM ? pp.lut_len : 0;
        pp.c2 = bp.c2[p]; pp.cnorm = bp.cnorm[p];
        // integer clip, computed weights and a LUT that is never clamped (its last distinct entry is the peak index)
        if (wm == W_COMPUTE && !BTr<T>::flt && pp.lut_len - 1 >= (int)bp.peak) {
            wm = W_SCALED;
            pp.scale = std::sqrt(-pp.c2);
            pp.inv_scale = 1.0f / pp.scale;
        }
        // f32 clip with a very wide range kernel (BASELINE config 5: sigmaR = 2).  The reference quantises |a-b| to the index
        // idx = trunc(min(1,|a-b|)*65535 + 0.5); the scaled form uses t = min(1,|a-b|)*65535 itself.  |idx^2 - t^2| <= 65535, so a
        // weight changes by at most ln2 * |c2| * 65535 relative and the weighted mean by at most twice that: allowed while that
        // stays below 4e-6 (the bar is 1e-5 relative; the MUFU weights and the reciprocal add ~5e-7).  sigmaR = 2: 3.8e-6.
        // f16 clips round the difference in f16 first (bilateral.zig:15-22) and keep the computed-index path.
        if (wm == W_COMPUTE && std::is_same<T, float>::value && pp.lut_len - 1 >= 65535 && 2.0 * 0.6931472 * (double)(-pp.c2) * 65535.0 <= 4e-6) {
            wm = W_SCALED;
            pp.scale = std::sqrt(-pp.c2) * 65535.0f;
            pp.inv_scale = 1.0f / pp.scale;
            pp.dmax = pp.scale;
        }
        const int r = pp.radius;
        // strip length: whole tile rows when the batch alone fills the GPU, shorter strips for single frames
        const int tiles_x = (l.pl[p].w + TILE - 1) / TILE, tiles_y = (l.pl[p].h + TILE - 1) / TILE;
        // and never fewer than ~8 waves of CTAs (8 CTAs fit an SM), so that the last partial wave stays a small share
        int strip = tiles_x;
        while (strip > 1 && (long long)((tiles_x + strip - 1) / strip) * tiles_y * count < 4 * 148) strip = (strip + 1) / 2;
        while (strip > 8 && (long long)((tiles_x + strip - 1) / strip) * tiles_y * count < 8ll * 8 * 148) strip = (strip + 1) / 2;
        const int strips_x = (tiles_x + strip - 1) / strip;
        prm.strip = strip;
        prm.tiles_x[0] = tiles_x;
        prm.strips_x[0] = strips_x;
        BatchJob j = make_batch(l, one, src, sfs, ref, rfs, dst, dfs, [&](int, int) { return strips_x * tiles_y; });
        const size_t tile = (size_t)(TILE + 2 * r) * (TILE + 2 * r);
        const size_t smem = (tile * (ref ? 2 : 1) + (size_t)(r + 1) * (r + 1) + (size_t)pp.smem_lut) * sizeof(float);
        if (smem > (size_t)kMaxSmemPerCta) { set_error("Bilateral: spatial radius %d does not fit the shared-memory tile", r); return -2; }
        for (int f0 = 0; f0 < count; f0 += 65535) {
            const int nf = std::min(65535, count - f0);
            BatchJob jj = j;
            jj.src += (size_t)f0 * sfs; jj.dst += (size_t)f0 * dfs;
            if (ref) jj.ref += (size_t)f0 * rfs;
            const int samples = pp.step > 0 ? (pp.radius - 1) / pp.step + 1 : 0;
            const int rc = ref ? launch_mode<T, true>(wm, samples, pp.step, jj, prm, nf, smem, st) : launch_mode<T, false>(wm, samples, pp.step, jj, prm, nf, smem, st);
            if (rc) return rc;
        }
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

int run_bilateral(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, const char* ref, size_t ref_fs, char* dst,
                  size_t dst_fs, int count, const BilateralLaunch& bp, cudaStream_t st) {
    switch (l.kind) {
        case K_U8: return run_bilateral_t<uint8_t>(l, mask, src, src_fs, ref, ref_fs, dst, dst_fs, count, bp, st);
        case K_U16: return run_bilateral_t<uint16_t>(l, mask, src, src_fs, ref, ref_fs, dst, dst_fs, count, bp, st);
        case K_F16: return run_bilateral_t<__half>(l, mask, src, src_fs, ref, ref_fs, dst, dst_fs, count, bp, st);
        case K_F32: return run_bilateral_t<float>(l, mask, src, src_fs, ref, ref_fs, dst, dst_fs, count, bp, st);
    }
    return -1;
}

}  // namespace vsz
