// planestats_kernels.cu — sm_100a reductions for vszip.PlaneAverage and vszip.PlaneMinMax.
//
// Semantics restated from the reference:
//   PlaneAverage (src/filters/planeaverage.zig:26-84): acc = sum of samples not in `exclude`, count of
//       excluded samples, optional sum |a-b| over ALL samples (float |a-b| rounded in T).
//   PlaneMinMax  (src/filters/planeminmax.zig:11-133): raw min/max (no threshold) or a 65536-bin
//       histogram with two cumulative scans using strict '>' against trunc(total*thr).
//
// Design: both are single-read streaming reductions (16-byte loads, warp-shuffle trees, one partial per
// CTA, combined in CTA order by the last CTA to finish so float sums are run-to-run deterministic);
// 16-bit integer PlaneAverage with a short exclude list runs two samples per instruction (average_u16_kernel).
// The threshold path never materialises 65536 bins.  Default: a 1/16 line sample brackets both ranks, then ONE
// full read counts exactly what lies outside the brackets (packed 16-bit clamps) and histograms only what lies
// inside; the exact counts prove the result or hand the plane to the fallback.  Fallback (and
// VSZIP_MINMAX_EXACT=1): an exact two-level radix select - pass 1 histograms the top 8 bits of the bin index,
// pass 2 re-reads the plane and histograms the low bits of only the two coarse bins that contain the requested
// ranks.  Integer counts are exact on both routes, so the result is bit-identical to the reference's full scan.
#include <cuda_fp16.h>

#include <algorithm>
#include <type_traits>
#include <cstdlib>

#include "filter.h"

namespace vsz {

static constexpr int NT = 256;
static constexpr int MAX_CTAS_PER_PLANE = 512;

struct Partial {
    unsigned long long isum, idiff;
    double fsum, fdiff;
    unsigned int excluded, imin, imax;
    float fmin, fmax;
    unsigned int pad;
};

// Coarse-bin brackets guessed from a row sample (threshold fast path) and the "already resolved" flag.
// Both brackets are 2^kbits - 1 bins wide and start at bin 1 or above (see minmax_bracket_kernel).
struct Bracket { unsigned int l_min, u_min, l_max, u_max; unsigned int done; unsigned int kbits; unsigned int pad[2]; };  // [l, u) in bins
// (2048 bins: the per-CTA flush and the last CTA's scan are a visible part of the sampling pass; 4096 bins cost 4 % of the whole
// threshold path and bracket no tighter once the bracket is widened to 2^k - 1 bins)
#ifndef VSZ_SBITS
#define VSZ_SBITS 11
#endif
static constexpr int SBITS = VSZ_SBITS, SBINS = 1 << SBITS;   // bins of the sample histogram
static constexpr int FINE_KMAX = 10; // widest bracket the single-read kernel can histogram: 2^10 - 1 bins
static constexpr int FINE_W = 1 << FINE_KMAX;

struct StatsPlane {
    size_t a_off, b_off;
    int a_pitch, b_pitch;
    int w, h;
    int cta_begin, nctas;
    int s_cta_begin, s_nctas;  // CTAs of the sampling kernel
    int b_cta_begin, b_nctas;  // CTAs of the single-read bracket kernel
    int s_step, s_lpr;         // it reads every s_step-th 128-byte line; s_lpr lines per row
    unsigned int tmin, tmax;  // trunc(total * thr)
};

struct StatsJob {
    const char* a;
    const char* b;  // nullptr when there is no clipb
    size_t a_fs, b_fs;
    int nplanes, ctas_per_frame;
    StatsPlane pl[3];
    // scratch
    Partial* partials;        // [frame][plane][MAX_CTAS_PER_PLANE]
    unsigned int* counters;   // [frame][plane] completed-CTA counters of pass 1 / the single-pass kernels
    unsigned int* counters2;  // [frame][plane] completed-CTA counters of pass 2
    unsigned int* coarse;     // [frame][plane][256]
    unsigned int* fine;       // [frame][plane][2][256]
    unsigned int* counters3;  // [frame][plane] completed-CTA counters of the sampling kernel
    unsigned int* ssample;    // [frame][plane][SBINS] histogram of the line sample
    unsigned int* bfine;      // [frame][plane][2][FINE_W] exact histograms of the two brackets
    struct Bracket* brackets; // [frame][plane]
    int sample_ctas_per_frame, bracket_ctas_per_frame;
    int sshift;               // sample bin = bin >> sshift
    StatsRaw* out;            // [frame][plane]
    StatsRaw* out_avg;        // [frame][plane] PlaneAverage results of the fused bracket kernel (SURVEY 8f rank 4)
    // parameters
    int nex;
    int32_t excl_i[16];
    float excl_f[16];
    const int32_t* excl_i_more;  // when nex > 16 (device memory)
    const float* excl_f_more;
    unsigned int hist_size;
    int shift;  // fine bits = bin & ((1<<shift)-1); coarse = bin >> shift
};

__device__ __forceinline__ const StatsPlane& find_plane(const StatsJob& j, int cta, int& k, int& local) {
    k = j.nplanes - 1;
    while (k > 0 && cta < j.pl[k].cta_begin) --k;
    local = cta - j.pl[k].cta_begin;
    return j.pl[k];
}

// --------------------------------------------------------------------------- element helpers
template <typename T> struct El;
template <> struct El<uint8_t> { static constexpr bool flt = false; static constexpr int PER16 = 16; };
template <> struct El<uint16_t> { static constexpr bool flt = false; static constexpr int PER16 = 8; };
template <> struct El<__half> { static constexpr bool flt = true; static constexpr int PER16 = 8; };
template <> struct El<float> { static constexpr bool flt = true; static constexpr int PER16 = 4; };

template <typename T> __device__ __forceinline__ float as_float(T v) { return (float)v; }
template <> __device__ __forceinline__ float as_float<__half>(__half v) { return __half2float(v); }

// |a-b| as the reference computes it: integers exactly, floats rounded in T then widened.
template <typename T> __device__ __forceinline__ double abs_diff(T a, T b, unsigned int& idiff) {
    if constexpr (El<T>::flt) {
        if constexpr (sizeof(T) == 2) return (double)fabsf(__half2float(__hsub(a, b)));
        else return (double)fabsf(__fsub_rn(a, b));
    } else {
        idiff += (a > b) ? (unsigned)(a - b) : (unsigned)(b - a);
        return 0.0;
    }
}

// histogram bin of a sample (src/filters/planeminmax.zig:26,33): ints index directly, floats use
// sat_u16(trunc(f32(v)*65535 + 0.5)) with separate multiply and add.
// Float bins without the conversion unit and with one clamp instead of two: saturating the SAMPLE to [0, 1] (NaN -> 0) gives the same
// bin as clamping v*65535 + 0.5 to [0, 65535] - below 0 both truncate to 0, above 1 both give 65535 - and FADD.RZ(f, 2^23) leaves
// trunc(f) in the low mantissa bits for f in [0.5, 65535.5].  bin_bits returns that float's bit pattern (bin in bits 0..15).
template <typename T> __device__ __forceinline__ unsigned int bin_bits(T v) {
    const float f = __fadd_rn(__fmul_rn(__saturatef(as_float<T>(v)), 65535.0f), 0.5f);
    return __float_as_uint(__fadd_rz(f, 8388608.0f));
}
template <typename T> __device__ __forceinline__ unsigned int bin_of(T v) {
    if constexpr (El<T>::flt) {
        return bin_bits<T>(v) & 0xffffu;
    } else {
        return (unsigned int)v;
    }
}

// Visits every sample of rows [y0, y1) of a plane with 16-byte loads (+ scalar tail), calling
// fn(a_sample, b_sample) where b_sample == a_sample if there is no second clip.
template <typename T, bool HAS_B, class F>
__device__ __forceinline__ void for_each_sample(const char* a, int a_pitch, const char* b, int b_pitch, int w, int y0, int y1, F fn) {
    constexpr int V = El<T>::PER16;
    const int nvec = w / V;
    for (int y = y0; y < y1; ++y) {
        const uint4* ar = reinterpret_cast<const uint4*>(a + (size_t)y * a_pitch);
        const uint4* br = HAS_B ? reinterpret_cast<const uint4*>(b + (size_t)y * b_pitch) : nullptr;
        for (int v = threadIdx.x; v < nvec; v += NT) {
            const uint4 av = __ldg(ar + v);
            uint4 bv = av;
            if constexpr (HAS_B) bv = __ldg(br + v);
            const T* ae = reinterpret_cast<const T*>(&av);
            const T* be = reinterpret_cast<const T*>(&bv);
#pragma unroll
            for (int i = 0; i < V; ++i) fn(ae[i], be[i]);
        }
        const int x = nvec * V + threadIdx.x;
        if (x < w) {
            const T av = reinterpret_cast<const T*>(ar)[x];
            const T bv = HAS_B ? reinterpret_cast<const T*>(br)[x] : av;
            fn(av, bv);
        }
    }
}

__device__ __forceinline__ void rows_of_cta(const StatsPlane& p, int local, int& y0, int& y1) {
    const int per = (p.h + p.nctas - 1) / p.nctas;
    y0 = min(local * per, p.h);
    y1 = min(y0 + per, p.h);
}

// --------------------------------------------------------------------------- block reduction + last-CTA combine
__device__ __forceinline__ void warp_reduce(Partial& p) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        p.isum += __shfl_down_sync(0xffffffffu, p.isum, o);
        p.idiff += __shfl_down_sync(0xffffffffu, p.idiff, o);
        p.fsum += __shfl_down_sync(0xffffffffu, p.fsum, o);
        p.fdiff += __shfl_down_sync(0xffffffffu, p.fdiff, o);
        p.excluded += __shfl_down_sync(0xffffffffu, p.excluded, o);
        p.imin = min(p.imin, __shfl_down_sync(0xffffffffu, p.imin, o));
        p.imax = max(p.imax, __shfl_down_sync(0xffffffffu, p.imax, o));
        p.fmin = fminf(p.fmin, __shfl_down_sync(0xffffffffu, p.fmin, o));
        p.fmax = fmaxf(p.fmax, __shfl_down_sync(0xffffffffu, p.fmax, o));
    }
}

__device__ __forceinline__ void combine(Partial& a, const Partial& b) {
    a.isum += b.isum; a.idiff += b.idiff; a.fsum += b.fsum; a.fdiff += b.fdiff; a.excluded += b.excluded;
    a.imin = min(a.imin, b.imin); a.imax = max(a.imax, b.imax);
    a.fmin = fminf(a.fmin, b.fmin); a.fmax = fmaxf(a.fmax, b.fmax);
}

__device__ __forceinline__ Partial empty_partial() {
    Partial p;
    p.isum = p.idiff = 0ull; p.fsum = p.fdiff = 0.0; p.excluded = 0u;
    p.imin = 0xffffffffu; p.imax = 0u;
    p.fmin = __int_as_float(0x7f800000); p.fmax = __int_as_float(0xff800000);
    p.pad = 0;
    return p;
}

// Reduces `mine` over the CTA, stores the CTA partial and returns true in exactly one CTA per
// (frame, plane): the last one to finish, with `total` = all partials combined in CTA order.
__device__ bool block_finish(const StatsJob& j, int frame, int k, int local, int nctas, unsigned int* counter, Partial mine,
                             Partial& total) {
    __shared__ Partial s_part[NT / 32];
    __shared__ bool s_last;
    warp_reduce(mine);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s_part[warp] = mine;
    __syncthreads();
    Partial* slots = j.partials + ((size_t)frame * j.nplanes + k) * MAX_CTAS_PER_PLANE;
    if (threadIdx.x == 0) {
        Partial t = s_part[0];
        for (int i = 1; i < NT / 32; ++i) combine(t, s_part[i]);
        slots[local] = t;
        __threadfence();
        const unsigned int done = atomicAdd(counter, 1u);
        s_last = (done == (unsigned)nctas - 1u);
    }
    __syncthreads();
    if (!s_last) return false;
    __threadfence();
    if (threadIdx.x == 0) {
        Partial t = slots[0];
        for (int i = 1; i < nctas; ++i) combine(t, slots[i]);
        total = t;
    }
    return true;
}

// --------------------------------------------------------------------------- PlaneAverage / no-threshold PlaneMinMax
// LONGEX: the exclude list has more than 4 entries (entries 4..15 in the job, the rest in device memory); the usual
// short lists compile to four register compares per sample and nothing else.
// BOTH (with AVERAGE): the no-threshold PlaneMinMax of the same samples comes out of the same read (SURVEY 8f rank 4); the sum is
// accumulated exactly as without it, so the average is bit-identical to the separate call.
template <typename T, bool HAS_B, bool AVERAGE, bool LONGEX = false, bool BOTH = false>
__global__ void __launch_bounds__(NT) stats_kernel(const StatsJob j) {
    int k, local;
    const StatsPlane& p = find_plane(j, blockIdx.x, k, local);
    const int frame = blockIdx.y;
    const char* a = j.a + (size_t)frame * j.a_fs + p.a_off;
    const char* b = HAS_B ? j.b + (size_t)frame * j.b_fs + p.b_off : nullptr;
    int y0, y1;
    rows_of_cta(p, local, y0, y1);

    Partial acc = empty_partial();
    unsigned int isum32 = 0, idiff32 = 0;  // flushed to 64 bit after every group of rows
    const int nex = j.nex;
    // the exclude list lives in registers for the usual short lists (unused slots repeat the first value)
    int32_t xi[4];
    float xf[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { xi[i] = j.excl_i[i < nex ? i : 0]; xf[i] = j.excl_f[i < nex ? i : 0]; }

    auto visit = [&](T av, T bv) {
        if constexpr (AVERAGE) {
            bool found = false;
            if constexpr (El<T>::flt) {
                const float f = as_float<T>(av);
                if (nex > 0) found = (f == xf[0]) | (f == xf[1]) | (f == xf[2]) | (f == xf[3]);
                if constexpr (LONGEX) {
                    for (int i = 4; i < min(nex, 16); ++i) found |= (f == j.excl_f[i]);
                    for (int i = 16; i < nex; ++i) found |= (f == __ldg(j.excl_f_more + i));  // long lists: device copy
                }
                if (found) acc.excluded += 1; else acc.fsum += (double)f;
            } else {
                const int32_t iv = (int32_t)av;
                if (nex > 0) found = (iv == xi[0]) | (iv == xi[1]) | (iv == xi[2]) | (iv == xi[3]);
                if constexpr (LONGEX) {
                    for (int i = 4; i < min(nex, 16); ++i) found |= (iv == j.excl_i[i]);
                    for (int i = 16; i < nex; ++i) found |= (iv == __ldg(j.excl_i_more + i));
                }
                if (found) acc.excluded += 1; else isum32 += (unsigned)av;
            }
        }
        if constexpr (!AVERAGE || BOTH) {
            if constexpr (El<T>::flt) {
                const float f = as_float<T>(av);
                acc.fmin = fminf(acc.fmin, f); acc.fmax = fmaxf(acc.fmax, f);
            } else {
                acc.imin = min(acc.imin, (unsigned)av); acc.imax = max(acc.imax, (unsigned)av);
            }
        }
        if constexpr (HAS_B) acc.fdiff += abs_diff<T>(av, bv, idiff32);
    };

    // G rows per step: G independent 16-byte loads per clip are in flight before any sample is consumed
    constexpr int V = El<T>::PER16, G = HAS_B ? 2 : 4;
    const int nvec = p.w / V;
    for (int y = y0; y < y1; y += G) {
        for (int v = threadIdx.x; v < nvec; v += NT) {
            uint4 av[G], bv[G];
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int yy = min(y + g, y1 - 1);  // duplicates past the end are loaded but not visited
                av[g] = __ldg(reinterpret_cast<const uint4*>(a + (size_t)yy * p.a_pitch) + v);
                if constexpr (HAS_B) bv[g] = __ldg(reinterpret_cast<const uint4*>(b + (size_t)yy * p.b_pitch) + v);
                else bv[g] = av[g];
            }
#pragma unroll
            for (int g = 0; g < G; ++g) {
                if (y + g < y1) {
                    const T* ae = reinterpret_cast<const T*>(&av[g]);
                    const T* be = reinterpret_cast<const T*>(&bv[g]);
#pragma unroll
                    for (int i = 0; i < V; ++i) visit(ae[i], be[i]);
                }
            }
        }
        const int x = nvec * V + threadIdx.x;  // scalar tail of each row
        if (x < p.w) {
            for (int g = 0; g < G && y + g < y1; ++g) {
                const T at = reinterpret_cast<const T*>(a + (size_t)(y + g) * p.a_pitch)[x];
                const T bt = HAS_B ? reinterpret_cast<const T*>(b + (size_t)(y + g) * p.b_pitch)[x] : at;
                visit(at, bt);
            }
        }
        // per group a thread sees at most G*(ceil(w/NT)+1) samples: with w <= 65536 the u32 partials cannot overflow
        acc.isum += isum32; acc.idiff += idiff32;
        isum32 = idiff32 = 0;
    }
    Partial total;
    if (block_finish(j, frame, k, local, p.nctas, j.counters + (size_t)frame * j.nplanes + k, acc, total) && threadIdx.x == 0) {
        StatsRaw r{};
        r.isum = total.isum; r.idiff = total.idiff; r.fsum = total.fsum; r.fdiff = total.fdiff;
        r.excluded = total.excluded; r.bin_min = total.imin; r.bin_max = total.imax;
        r.fmin = total.fmin; r.fmax = total.fmax;
        if constexpr (BOTH) {
            j.out_avg[(size_t)frame * j.nplanes + k] = r;      // PlaneAverage reads isum / fsum / excluded
            r.isum = 0ull; r.fsum = 0.0; r.excluded = 0u;      // PlaneMinMax (no threshold) reads the raw minima / maxima
        }
        j.out[(size_t)frame * j.nplanes + k] = r;
    }
}

// --------------------------------------------------------------------------- PlaneAverage, 16-bit integer clips, short lists
// Two samples per instruction: IDP.2A adds both halves of a word to the running sum, and per distinct in-range exclude
// value e one XOR + VIMNMX.U16x2 turns a word into "1 per half that differs from e", accumulated as packed counts.
// The excluded samples are then removed arithmetically: count_e = seen - differing_e, sum -= e * count_e (all exact).
template <int NEX>
__global__ void __launch_bounds__(NT) average_u16_kernel(const StatsJob j) {
    int k, local;
    const StatsPlane& p = find_plane(j, blockIdx.x, k, local);
    const int frame = blockIdx.y;
    const char* a = j.a + (size_t)frame * j.a_fs + p.a_off;
    int y0, y1;
    rows_of_cta(p, local, y0, y1);
    unsigned int ee[NEX > 0 ? NEX : 1], pk[NEX > 0 ? NEX : 1], differing[NEX > 0 ? NEX : 1];
#pragma unroll
    for (int e = 0; e < NEX; ++e) { ee[e] = (unsigned)j.excl_i[e] * 0x10001u; pk[e] = 0u; differing[e] = 0u; }
    unsigned long long sum64 = 0ull;
    unsigned int s32 = 0u, seen = 0u;
    constexpr int G = 4;
    const int nvec = p.w / 8;
    for (int y = y0; y < y1; y += G) {
        for (int v = threadIdx.x; v < nvec; v += NT) {
            uint4 av[G];
#pragma unroll
            for (int g = 0; g < G; ++g) av[g] = __ldg(reinterpret_cast<const uint4*>(a + (size_t)min(y + g, y1 - 1) * p.a_pitch) + v);
#pragma unroll
            for (int g = 0; g < G; ++g) {
                if (y + g < y1) {
                    const unsigned int w[4] = {av[g].x, av[g].y, av[g].z, av[g].w};
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        s32 = __dp2a_lo(w[q], 0x0101u, s32);
#pragma unroll
                        for (int e = 0; e < NEX; ++e) pk[e] += __vminu2(w[q] ^ ee[e], 0x10001u);
                    }
                    seen += 8u;
                }
            }
        }
        const int x = nvec * 8 + threadIdx.x;  // scalar tail of each row
        if (x < p.w) {
            for (int g = 0; g < G && y + g < y1; ++g) {
                const unsigned int v = reinterpret_cast<const uint16_t*>(a + (size_t)(y + g) * p.a_pitch)[x];
                s32 += v;
#pragma unroll
                for (int e = 0; e < NEX; ++e) differing[e] += (v != (unsigned)j.excl_i[e]) ? 1u : 0u;
                seen += 1u;
            }
        }
        // per group a thread adds at most 4 * 32 * 4 to each packed half and 4 * 32 * 8 * 65535 to s32
        sum64 += s32; s32 = 0u;
#pragma unroll
        for (int e = 0; e < NEX; ++e) { differing[e] += (pk[e] & 0xffffu) + (pk[e] >> 16); pk[e] = 0u; }
    }
    Partial acc = empty_partial();
    unsigned long long removed = 0ull;
    unsigned int excluded = 0u;
#pragma unroll
    for (int e = 0; e < NEX; ++e) {
        const unsigned int cnt = seen - differing[e];
        excluded += cnt;
        removed += (unsigned long long)cnt * (unsigned)j.excl_i[e];
    }
    acc.isum = sum64 - removed;
    acc.excluded = excluded;
    Partial total;
    if (block_finish(j, frame, k, local, p.nctas, j.counters + (size_t)frame * j.nplanes + k, acc, total) && threadIdx.x == 0) {
        StatsRaw r{};
        r.isum = total.isum; r.excluded = total.excluded;
        j.out[(size_t)frame * j.nplanes + k] = r;
    }
}

// --------------------------------------------------------------------------- threshold path, pass 1
// warp-private 256-bin histograms in shared memory; a warp whose 32 lanes all hit the same bin
// (flat areas, blank clips) issues one atomic of 32 instead of 32 serialised ones.
__device__ __forceinline__ void hist_add(unsigned int* h, unsigned int key, bool valid) {
    // (MATCH.ANY would aggregate arbitrary groups but was measured 3x slower than this on B200)
    const unsigned int active = __ballot_sync(0xffffffffu, valid);
    if (active == 0u) return;
    const int leader = __ffs(active) - 1;
    const unsigned int k0 = __shfl_sync(0xffffffffu, key, leader);
    const unsigned int same = __ballot_sync(0xffffffffu, valid && key == k0);
    if (same == active) {
        if ((int)(threadIdx.x & 31) == leader) atomicAdd(&h[k0], (unsigned)__popc(active));
    } else if (valid) {
        atomicAdd(&h[key], 1u);
    }
}

template <typename T, bool HAS_B>
__device__ __forceinline__ void hist_coarse_body(const StatsJob& j, const int frame) {
    __shared__ unsigned int s_hist[NT / 32][256];
    int k, local;
    const StatsPlane& p = find_plane(j, blockIdx.x, k, local);
    if (j.brackets[(size_t)frame * j.nplanes + k].done) return;  // resolved by the sampled fast path
    const char* a = j.a + (size_t)frame * j.a_fs + p.a_off;
    const char* b = HAS_B ? j.b + (size_t)frame * j.b_fs + p.b_off : nullptr;
    int y0, y1;
    rows_of_cta(p, local, y0, y1);
    for (int i = threadIdx.x; i < (NT / 32) * 256; i += NT) (&s_hist[0][0])[i] = 0u;
    __syncthreads();

    unsigned int* mine = s_hist[threadIdx.x >> 5];
    Partial acc = empty_partial();
    unsigned int idiff32 = 0;
    const unsigned int hist_size = j.hist_size;
    const int shift = j.shift;
    // whole warps walk the rows together so the ballot in hist_add is always convergent
    constexpr int V = El<T>::PER16;
    const int nvec = p.w / V;
    const int nvec_pad = (nvec + NT - 1) / NT * NT;
    for (int y = y0; y < y1; ++y) {
        const uint4* ar = reinterpret_cast<const uint4*>(a + (size_t)y * p.a_pitch);
        const uint4* br = HAS_B ? reinterpret_cast<const uint4*>(b + (size_t)y * p.b_pitch) : nullptr;
        for (int v = threadIdx.x; v < nvec_pad; v += NT) {
            const bool ok = v < nvec;
            uint4 av = make_uint4(0, 0, 0, 0), bv = av;
            if (ok) { av = __ldg(ar + v); if constexpr (HAS_B) bv = __ldg(br + v); }
            const T* ae = reinterpret_cast<const T*>(&av);
            const T* be = reinterpret_cast<const T*>(&bv);
#pragma unroll
            for (int i = 0; i < V; ++i) {
                const unsigned int bin = bin_of<T>(ae[i]);
                hist_add(mine, bin >> shift, ok && bin < hist_size);
                if constexpr (HAS_B) { if (ok) acc.fdiff += abs_diff<T>(ae[i], be[i], idiff32); }
            }
        }
        {
            const int x = nvec * V + (int)threadIdx.x;
            const bool ok = x < p.w;
            if (__any_sync(0xffffffffu, ok)) {
                T av{}, bv{};
                if (ok) { av = reinterpret_cast<const T*>(ar)[x]; if constexpr (HAS_B) bv = reinterpret_cast<const T*>(br)[x]; }
                const unsigned int bin = bin_of<T>(av);
                hist_add(mine, bin >> shift, ok && bin < hist_size);
                if constexpr (HAS_B) { if (ok) acc.fdiff += abs_diff<T>(av, bv, idiff32); }
            }
        }
        acc.idiff += idiff32; idiff32 = 0;
    }
    __syncthreads();
    unsigned int* coarse = j.coarse + ((size_t)frame * j.nplanes + k) * 256;
    for (int i = threadIdx.x; i < 256; i += NT) {
        unsigned int s = 0;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) s += s_hist[w][i];
        if (s) atomicAdd(&coarse[i], s);
    }
    if constexpr (HAS_B) {
        Partial total;
        if (block_finish(j, frame, k, local, p.nctas, j.counters + (size_t)frame * j.nplanes + k, acc, total) && threadIdx.x == 0) {
            StatsRaw& r = j.out[(size_t)frame * j.nplanes + k];
            r.idiff = total.idiff; r.fdiff = total.fdiff;
        }
    }
}

// Finds, from a 256-entry histogram with `base` samples already counted before it, the first entry
// (scanning upward if UP, downward otherwise) at which the running count exceeds `thr`.
// Returns the entry index or -1; *before = running count before that entry.  Single thread.
template <bool UP>
__device__ int scan_rank(const unsigned int* h, int n, unsigned int base, unsigned int thr, unsigned int* before) {
    unsigned int c = base;
    for (int s = 0; s < n; ++s) {
        const int i = UP ? s : n - 1 - s;
        const unsigned int next = c + h[i];
        if (next > thr) { *before = c; return i; }
        c = next;
    }
    *before = c;
    return -1;
}

// --------------------------------------------------------------------------- threshold path, pass 2
template <typename T>
__device__ __forceinline__ void hist_fine_body(const StatsJob& j, const int frame) {
    __shared__ unsigned int s_fine[2][256];
    __shared__ int s_bmin, s_bmax;
    __shared__ unsigned int s_cmin, s_cmax;
    __shared__ bool s_last;
    int k, local;
    const StatsPlane& p = find_plane(j, blockIdx.x, k, local);
    if (j.brackets[(size_t)frame * j.nplanes + k].done) return;  // resolved by the sampled fast path
    const char* a = j.a + (size_t)frame * j.a_fs + p.a_off;
    const unsigned int* coarse = j.coarse + ((size_t)frame * j.nplanes + k) * 256;
    const int shift = j.shift;
    const int ncoarse = (int)((j.hist_size + (1u << shift) - 1) >> shift);
    const int nfine = 1 << shift;
    for (int i = threadIdx.x; i < 512; i += NT) (&s_fine[0][0])[i] = 0u;
    if (threadIdx.x == 0) s_bmin = scan_rank<true>(coarse, ncoarse, 0u, p.tmin, &s_cmin);
    if (threadIdx.x == 32) s_bmax = scan_rank<false>(coarse, ncoarse, 0u, p.tmax, &s_cmax);
    __syncthreads();
    const int bmin = s_bmin, bmax = s_bmax;

    if (shift > 0 && (bmin >= 0 || bmax >= 0)) {
        int y0, y1;
        rows_of_cta(p, local, y0, y1);
        const unsigned int fmask = (unsigned)nfine - 1u;
        for_each_sample<T, false>(a, p.a_pitch, nullptr, 0, p.w, y0, y1, [&](T av, T) {
            const unsigned int bin = bin_of<T>(av);
            const int c = (int)(bin >> shift);
            if (bin < j.hist_size) {
                if (c == bmin) atomicAdd(&s_fine[0][bin & fmask], 1u);
                if (c == bmax) atomicAdd(&s_fine[1][bin & fmask], 1u);
            }
        });
    }
    __syncthreads();
    unsigned int* fine = j.fine + ((size_t)frame * j.nplanes + k) * 512;
    if (shift > 0) {
        for (int i = threadIdx.x; i < 512; i += NT) {
            const unsigned int s = (&s_fine[0][0])[i];
            if (s) atomicAdd(&fine[i], s);
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int done = atomicAdd(j.counters2 + (size_t)frame * j.nplanes + k, 1u);
        s_last = (done == (unsigned)p.nctas - 1u);
    }
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    const unsigned int peak = j.hist_size - 1u;
    unsigned int lo = peak, hi = 0u, dummy;
    if (bmin >= 0) {
        if (shift == 0) lo = (unsigned)bmin;
        else {
            const int f = scan_rank<true>(const_cast<const unsigned int*>(fine), nfine, s_cmin, p.tmin, &dummy);
            lo = ((unsigned)bmin << shift) + (unsigned)f;  // f >= 0: the coarse bin is known to cross the rank
        }
    }
    if (bmax >= 0) {
        if (shift == 0) hi = (unsigned)bmax;
        else {
            const int f = scan_rank<false>(const_cast<const unsigned int*>(fine + 256), nfine, s_cmax, p.tmax, &dummy);
            hi = ((unsigned)bmax << shift) + (unsigned)f;
        }
    }
    StatsRaw& r = j.out[(size_t)frame * j.nplanes + k];
    r.bin_min = lo; r.bin_max = hi;
}

// The exact kernels walk the frames of a batch with a grid-stride loop: when the fast path below is on they are
// only a fallback, so the launcher gives them a few frame rows instead of one CTA per (chunk, frame) that would
// exit at once.
template <typename T, bool HAS_B>
__global__ void __launch_bounds__(NT) hist_coarse_kernel(const StatsJob j, const int nframes) {
    for (int frame = blockIdx.y; frame < nframes; frame += gridDim.y) {
        hist_coarse_body<T, HAS_B>(j, frame);
        __syncthreads();
    }
}
template <typename T>
__global__ void __launch_bounds__(NT) hist_fine_kernel(const StatsJob j, const int nframes) {
    for (int frame = blockIdx.y; frame < nframes; frame += gridDim.y) {
        hist_fine_body<T>(j, frame);
        __syncthreads();
    }
}

// --------------------------------------------------------------------------- threshold path, sampled fast path
// The exact two-pass select above costs two full reads and one shared-memory atomic per sample.  The fast path
// brackets, from a 1/16 sample of the plane's 128-byte lines (2048-bin histogram), the bin range that must hold each
// requested rank and then makes ONE full pass that (a) counts exactly how many samples lie below / above the
// brackets with packed 16-bit min/max arithmetic (no atomics, content independent) and (b) builds exact histograms
// of the (few) samples inside the brackets.  If the true rank lies inside its bracket - which the exact counts
// prove or disprove - the bin is resolved exactly; otherwise the plane is left to the exact two-pass kernels,
// which return immediately when `done`.
template <typename T>
__global__ void __launch_bounds__(NT) hist_sample_kernel(const StatsJob j) {
    __shared__ unsigned int s_h[SBINS];
    __shared__ unsigned int s_scan[NT];
    __shared__ int s_res[4];
    __shared__ bool s_last;
    // sample CTAs have their own plane map (far fewer CTAs than the full-read kernels)
    int k = j.nplanes - 1;
    while (k > 0 && (int)blockIdx.x < j.pl[k].s_cta_begin) --k;
    const StatsPlane& p = j.pl[k];
    const int local = (int)blockIdx.x - p.s_cta_begin;
    const int frame = blockIdx.y;
    const size_t fp = (size_t)frame * j.nplanes + k;
    const char* a = j.a + (size_t)frame * j.a_fs + p.a_off;
    for (int i = threadIdx.x; i < SBINS; i += NT) s_h[i] = 0u;
    __syncthreads();

    constexpr int V = El<T>::PER16, U = 4;
    const int nvec = p.w / V;
    const int sshift = j.sshift;
    const unsigned int hist_size = j.hist_size;
    // The sample is every s_step-th 128-byte line of the plane in raster order; s_step is coprime with the lines per
    // row, so consecutive rows are sampled at shifting columns.  8 lanes read one line, a warp 4 lines, U in flight.
    const long long nlines = (long long)p.h * p.s_lpr;
    const long long nsl = (nlines + p.s_step - 1) / p.s_step;  // sampled lines
    const int sub = threadIdx.x & 7;
    const long long first = (long long)local * (NT / 8) + (threadIdx.x >> 3);
    const long long stride = (long long)p.s_nctas * (NT / 8);
    for (long long s0 = first; s0 < nsl; s0 += stride * U) {
        uint4 av[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long s = s0 + u * stride;
            const long long line = s * p.s_step;
            const int r = (int)(line / p.s_lpr), c = (int)(line - (long long)r * p.s_lpr);
            const int v = c * 8 + sub;
            ok[u] = s < nsl && v < nvec;
            if (ok[u]) av[u] = __ldg(reinterpret_cast<const uint4*>(a + (size_t)r * p.a_pitch) + v);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!ok[u]) continue;
            const T* e = reinterpret_cast<const T*>(&av[u]);
            bool flat = (av[u].x == av[u].y) & (av[u].y == av[u].z) & (av[u].z == av[u].w);
            if (sizeof(T) <= 2) flat = flat & (__byte_perm(av[u].x, 0u, 0x1032) == av[u].x);
            if (sizeof(T) == 1) flat = flat & (__byte_perm(av[u].x, 0u, 0x0321) == av[u].x);
            if (flat) {  // constant vector: one atomic (flat areas would otherwise serialise on one address)
                const unsigned int bin = bin_of<T>(e[0]);
                if (bin < hist_size) atomicAdd(&s_h[bin >> sshift], (unsigned)V);
            } else {
#pragma unroll
                for (int i = 0; i < V; ++i) {
                    const unsigned int bin = bin_of<T>(e[i]);
                    if (bin < hist_size) atomicAdd(&s_h[bin >> sshift], 1u);
                }
            }
        }
    }
    __syncthreads();
    unsigned int* sh = j.ssample + fp * SBINS;
    for (int i = threadIdx.x; i < SBINS; i += NT) {
        const unsigned int c = s_h[i];
        if (c) atomicAdd(&sh[i], c);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(j.counters3 + fp, 1u) == (unsigned)p.s_nctas - 1u);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // ---- last sample CTA of the plane: bracket both ranks.  Each thread owns SBINS/NT consecutive bins.
    constexpr int PER = SBINS / NT;
    unsigned int mine[PER], local_sum = 0u;
#pragma unroll
    for (int i = 0; i < PER; ++i) { mine[i] = __ldcg(sh + threadIdx.x * PER + i); local_sum += mine[i]; }
    s_scan[threadIdx.x] = local_sum;
    if (threadIdx.x < 4) s_res[threadIdx.x] = -1;
    __syncthreads();
    for (int o = 1; o < NT; o <<= 1) {  // inclusive Hillis-Steele scan
        const unsigned int add = (int)threadIdx.x >= o ? s_scan[threadIdx.x - o] : 0u;
        __syncthreads();
        s_scan[threadIdx.x] += add;
        __syncthreads();
    }
    const unsigned int ns = s_scan[NT - 1];
    const unsigned int before = s_scan[threadIdx.x] - local_sum;
    // requested ranks scaled to the sample, +- a margin of 4.5 binomial sigmas + 0.05 % (pictures are not i.i.d.)
    const double npx = (double)p.w * (double)p.h, scale = (double)ns / npx;
    double q[4];
    {
        const double full = (p.s_step == 1 && nvec * V == p.w) ? 0.0 : 1.0;  // complete sample: no margin
        const double f_lo = fmin((double)p.tmin / npx, 1.0), f_hi = fmin((double)p.tmax / npx, 1.0);
        const double dmin = full * (4.5 * sqrt((double)ns * f_lo * (1.0 - f_lo)) + 0.0005 * ns + 2.0);
        const double dmax = full * (4.5 * sqrt((double)ns * f_hi * (1.0 - f_hi)) + 0.0005 * ns + 2.0);
        const double tmin_s = (double)p.tmin * scale, top = (double)ns - 1.0 - (double)p.tmax * scale;
        q[0] = tmin_s - dmin; q[1] = tmin_s + dmin; q[2] = top - dmax; q[3] = top + dmax;
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const double qc = fmin(fmax(q[t], 0.0), (double)ns - 1.0);
        const unsigned int qi = ns ? (unsigned int)qc : 0u;
        if (local_sum && qi >= before && qi < before + local_sum) {
            unsigned int c = before;
            int hit = PER - 1;
#pragma unroll
            for (int i = 0; i < PER; ++i) { c += mine[i]; if (qi < c) { hit = i; break; } }
            s_res[t] = (int)threadIdx.x * PER + hit;
        }
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const int nsb = (int)((hist_size + (1u << sshift) - 1u) >> sshift);
    // The full-read kernel wants both brackets 2^k - 1 bins wide with one k, and bin l - 1 >= 0 below each of them:
    // the sampled ranges are widened to the next such width around their middle (a range wider than 2^FINE_KMAX - 1
    // keeps its middle; a range that starts at bin 0 loses bin 0 - the exactness check of the full-read kernel
    // resolves a rank that falls into that single bin, and sends everything else it cannot prove to the exact path).
    auto sampled = [&](int lo_sb, int hi_sb, unsigned int& l, unsigned int& u) {
        if (lo_sb < 0) lo_sb = 0;
        if (hi_sb < 0) hi_sb = nsb - 1;
        l = (unsigned)lo_sb << sshift;
        u = min((unsigned)(hi_sb + 1) << sshift, hist_size);
    };
    unsigned int l0, u0, l1, u1;
    sampled(s_res[0], s_res[1], l0, u0);
    sampled(s_res[2], s_res[3], l1, u1);
    unsigned int kbits = 1u;
    while (kbits < (unsigned)FINE_KMAX && (1u << kbits) - 1u < max(u0 - l0, u1 - l1)) ++kbits;
    const int width = (1 << kbits) - 1;
    auto place = [&](unsigned int l, unsigned int u, unsigned int& lo, unsigned int& hi) {
        int start = (int)l - (width - (int)(u - l)) / 2;   // needed range in the middle of the window (negative slack: its middle)
        start = max(1, min(start, 65536 - width));
        lo = (unsigned)start; hi = (unsigned)(start + width);
    };
    Bracket br;
    place(l0, u0, br.l_min, br.u_min);
    place(l1, u1, br.l_max, br.u_max);
    br.done = 0u; br.kbits = kbits; br.pad[0] = br.pad[1] = 0u;
    j.brackets[fp] = br;
}

// Packs the histogram bins of one 16-byte vector two per 32-bit word so that the per-sample work below runs on
// VIMNMX.U16x2 (two samples per instruction).
template <typename T> __device__ __forceinline__ void pack_bins(const uint4& v, unsigned int (&w)[El<T>::PER16 / 2]) {
    if constexpr (sizeof(T) == 2 && !El<T>::flt) {
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    } else if constexpr (sizeof(T) == 1) {
        const unsigned int s[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) { w[2 * q] = __byte_perm(s[q], 0u, 0x4140); w[2 * q + 1] = __byte_perm(s[q], 0u, 0x4342); }
    } else {
        const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
        for (int q = 0; q < El<T>::PER16 / 2; ++q) w[q] = __byte_perm(bin_bits<T>(e[2 * q]), bin_bits<T>(e[2 * q + 1]), 0x5410);  // low halves of both
    }
}

// Per bracket [l, u) with u - l = 2^k - 1 and A = l - 1:  h = min(max(x, A) - A, 2^k)  (VIMNMX.U16x2 + VIADDMNMX.U16x2, two
// samples per instruction) is 0 below the bracket, 2^k at or above u and x - A in 1 .. 2^k - 1 inside.  So
//   - a word holds a sample inside a bracket iff the OR of its two h values has one of the low k bits set (one LOP3 with a
//     predicate result per word), and
//   - the sum of h over everything a lane has visited (IDP.2A) is 2^k * (samples >= u) + sum(x - A) over its inside samples;
//     the lane visits those one by one anyway (the fine histograms), subtracts their part and has the exact count.
// Words with an inside sample go to a LANE-PRIVATE queue in shared memory (a predicated store and a predicated add: no ballot, no
// prefix, no __syncwarp); when a lane has 16 waiting the warp drains, every lane its own words.
// TRACK = false: every bin is valid (full-depth integer or float clip) and both ranks are > 0, so the exact
// min/max tracking drops out of the per-sample work.  With TRACK the packed min/max give the answers for zero
// ranks and detect samples above the format's peak (such planes are left to the exact two-pass kernels).
// AVG >= 0: the same single read also yields PlaneAverage with AVG distinct in-range exclude values (SURVEY 8f rank 4).  8..16-bit
// integer clips: IDP.2A sums both halves of a word, one XOR + VIMNMX.U16x2 per exclude value counts the halves that differ from it
// (the arithmetic of average_u16_kernel); sum and excluded count travel in the Partial's idiff / excluded fields - with clipb idiff
// carries Diff, so the sum travels in fsum instead (a whole plane's sum is below 2^47: exact in a double).  With clipb the one Diff
// accumulated here is both filters' Diff.
template <typename T, bool HAS_B, bool TRACK, int AVG = -1>
__global__ void __launch_bounds__(NT) minmax_bracket_kernel(const StatsJob j) {
    constexpr bool FAVG = AVG >= 0 && El<T>::flt;  // float clips: per sample AVG compares against the exclude values and one f64 add
    constexpr int V = El<T>::PER16, NW = V / 2, G = HAS_B ? 2 : 4;
    constexpr int NEX = AVG > 0 ? AVG : 1;
    unsigned int ee[NEX], differing[NEX];
#pragma unroll
    for (int e = 0; e < NEX; ++e) { ee[e] = AVG > 0 ? (unsigned)j.excl_i[e] * 0x10001u : 0u; differing[e] = 0u; }
    unsigned int s32 = 0u, seen = 0u;
    unsigned long long sum64 = 0ull;
    float xf[NEX];
#pragma unroll
    for (int e = 0; e < NEX; ++e) xf[e] = AVG > 0 ? j.excl_f[e] : 0.f;
    double fsum = 0.0;
    unsigned int fexcluded = 0u;
    auto favg = [&](float f) {
        bool found = false;
#pragma unroll
        for (int e = 0; e < AVG; ++e) found |= (f == xf[e]);
        if (found) fexcluded += 1u; else fsum += (double)f;
    };
    // lane-private queue of QCAP words, looked at after every step of G vectors (after every vector where a step could overflow it:
    // 8-bit clips) and drained when some lane could not take another such portion
    constexpr int QCAP = 32;
    constexpr bool PER_VEC = G * NW > QCAP / 2;
    constexpr int QDRAIN = QCAP - (PER_VEC ? NW : G * NW) + 1;
    static_assert(QDRAIN >= 1 && NW <= QCAP, "queue too small");
    __shared__ unsigned int s_fine[2][FINE_W];
    __shared__ unsigned int s_q[NT / 32][QCAP][32];  // [warp][entry][lane]: a lane only ever touches bank `lane`
    // own plane map: in large batches this kernel uses fewer, longer-running CTAs than the other reductions
    int k = j.nplanes - 1;
    while (k > 0 && (int)blockIdx.x < j.pl[k].b_cta_begin) --k;
    const StatsPlane& p = j.pl[k];
    const int local = (int)blockIdx.x - p.b_cta_begin;
    const int frame = blockIdx.y;
    const size_t fp = (size_t)frame * j.nplanes + k;
    const char* a = j.a + (size_t)frame * j.a_fs + p.a_off;
    const char* b = HAS_B ? j.b + (size_t)frame * j.b_fs + p.b_off : nullptr;
    const Bracket br = j.brackets[fp];
    const int rows_per = (p.h + p.b_nctas - 1) / p.b_nctas;
    const int y0 = min(local * rows_per, p.h), y1 = min(y0 + rows_per, p.h);
    for (int i = threadIdx.x; i < 2 * FINE_W; i += NT) (&s_fine[0][0])[i] = 0u;
    __syncthreads();
    const unsigned int hist_size = j.hist_size;
    const unsigned int l_min = br.l_min, u_min = br.u_min, l_max = br.l_max, u_max = br.u_max;  // [l, u) in bins
    const unsigned int kbits = br.kbits, w_min = u_min - l_min, w_max = u_max - l_max;           // both 2^kbits - 1
    const unsigned int a_min = l_min - 1u, a_max = l_max - 1u;
    const unsigned int pkA0 = a_min * 0x10001u, pkN0 = ((65536u - a_min) & 0xffffu) * 0x10001u;
    const unsigned int pkA1 = a_max * 0x10001u, pkN1 = ((65536u - a_max) & 0xffffu) * 0x10001u;
    const unsigned int pkW = (1u << kbits) * 0x10001u, pk_low = ((1u << kbits) - 1u) * 0x10001u;

    Partial acc = empty_partial();
    unsigned int ge_lmin = 0, ge_umax = 0, idiff32 = 0;    // scalar row tails: samples with bin >= l_min / >= u_max
    unsigned int sum_h0 = 0, sum_h1 = 0;                   // sums of h over both halves of the words of one group of rows
    unsigned long long tot_h0 = 0ull, tot_h1 = 0ull;       // ... of the lane's whole share
    unsigned long long in_h0 = 0ull, in_h1 = 0ull;         // sum(x - A) over the inside samples this lane drained
    unsigned int in_n0 = 0u;                               // how many were inside the min bracket
    unsigned int pk_min = 0xffffffffu, pk_max = 0u;
    const int lane = threadIdx.x & 31;
    unsigned int* myq = &s_q[threadIdx.x >> 5][0][lane];   // entry e at myq[e * 32]
    unsigned int qn = 0u;                                   // words waiting in this lane's queue

    auto fine_add = [&](unsigned int bin, unsigned int n) {
        if (bin - l_min < w_min) atomicAdd(&s_fine[0][bin - l_min], n);
        if (bin - l_max < w_max) atomicAdd(&s_fine[1][bin - l_max], n);
    };
    auto visit_vec = [&](const uint4& av, const uint4& bv) {
        unsigned int w[NW];
        pack_bins<T>(av, w);
#pragma unroll
        for (int q = 0; q < NW; ++q) {
            const unsigned int h0 = __viaddmin_u16x2(__vmaxu2(w[q], pkA0), pkN0, pkW);
            const unsigned int h1 = __viaddmin_u16x2(__vmaxu2(w[q], pkA1), pkN1, pkW);
            sum_h0 = __dp2a_lo(h0, 0x0101u, sum_h0);
            sum_h1 = __dp2a_lo(h1, 0x0101u, sum_h1);
            if (((h0 | h1) & pk_low) != 0u) { myq[qn * 32u] = w[q]; qn += 1u; }  // (packed bins: the drain needs no conversion)
            if constexpr (TRACK) { pk_min = __vminu2(pk_min, w[q]); pk_max = __vmaxu2(pk_max, w[q]); }
            if constexpr (AVG >= 0 && !FAVG) {
                s32 = __dp2a_lo(w[q], 0x0101u, s32);
#pragma unroll
                for (int e = 0; e < AVG; ++e) differing[e] = __dp2a_lo(__vminu2(w[q] ^ ee[e], 0x10001u), 0x0101u, differing[e]);  // + 1 per half that differs
            }
        }
        if constexpr (AVG >= 0 && !FAVG) seen += (unsigned)V;
        if constexpr (FAVG) {
            const T* ae = reinterpret_cast<const T*>(&av);
#pragma unroll
            for (int i = 0; i < V; ++i) favg(as_float<T>(ae[i]));
        }
        if constexpr (HAS_B) {
            const T* ae = reinterpret_cast<const T*>(&av);
            const T* be = reinterpret_cast<const T*>(&bv);
#pragma unroll
            for (int i = 0; i < V; ++i) acc.fdiff += abs_diff<T>(ae[i], be[i], idiff32);
        }
    };
    // every lane walks its own queued words: the fine histogram(s) each half belongs to, and the inside samples' share of the h sums
    auto drain = [&]() {
        const unsigned int most = __reduce_max_sync(0xffffffffu, qn);
        for (unsigned int e = 0; e < most; ++e) {
            if (e < qn) {
                const unsigned int w = myq[e * 32u];
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const unsigned int bin = half ? (w >> 16) : (w & 0xffffu);
                    const unsigned int d0 = bin - l_min, d1 = bin - l_max;
                    if (d0 < w_min) { atomicAdd(&s_fine[0][d0], 1u); in_h0 += d0 + 1u; in_n0 += 1u; }
                    if (d1 < w_max) { atomicAdd(&s_fine[1][d1], 1u); in_h1 += d1 + 1u; }
                }
            }
        }
        qn = 0u;
    };
    auto visit_one = [&](T at, T bt) {  // scalar row tails
        const unsigned int bin = bin_of<T>(at);
        ge_lmin += bin >= l_min ? 1u : 0u;
        ge_umax += bin >= u_max ? 1u : 0u;
        fine_add(bin, 1u);
        if constexpr (TRACK) { pk_min = __vminu2(pk_min, bin * 0x10001u); pk_max = __vmaxu2(pk_max, bin * 0x10001u); }
        if constexpr (HAS_B) acc.fdiff += abs_diff<T>(at, bt, idiff32);
        if constexpr (AVG >= 0 && !FAVG) {
            s32 += bin;
#pragma unroll
            for (int e = 0; e < AVG; ++e) differing[e] += (bin != (unsigned)j.excl_i[e]) ? 1u : 0u;
            seen += 1u;
        }
        if constexpr (FAVG) favg(as_float<T>(at));
    };

    const int nvec = p.w / V;
    const int iters = (nvec + NT - 1) / NT;
    auto flush32 = [&]() {  // the 32-bit running sums go to 64 bit
        tot_h0 += sum_h0; tot_h1 += sum_h1;
        sum_h0 = sum_h1 = 0u;
        acc.idiff += idiff32; idiff32 = 0;
        if constexpr (AVG >= 0 && !FAVG) { sum64 += s32; s32 = 0u; }
    };
    bool contiguous = nvec > 0 && p.a_pitch == nvec * 16;  // rows back to back (the pitch is the row: no tail samples either)
    if constexpr (HAS_B) contiguous = contiguous && p.b_pitch == p.a_pitch;
    if (contiguous) {
        // the CTA's rows as one run of vectors: every thread gets the same share whatever the width (per row, 480 vectors over 256
        // threads leave an eighth of the lanes idle in every second step)
        const long long total = (long long)(y1 - y0) * nvec;
        const uint4* abase = reinterpret_cast<const uint4*>(a + (size_t)y0 * p.a_pitch);
        const uint4* bbase = HAS_B ? reinterpret_cast<const uint4*>(b + (size_t)y0 * p.b_pitch) : nullptr;
        int step = 0;
        for (long long i0 = 0; i0 < total; i0 += (long long)NT * G, ++step) {
            uint4 av[G], bv[G];
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const long long idx = i0 + (long long)g * NT + threadIdx.x;
                if (idx < total) {
                    av[g] = __ldg(abase + idx);
                    if constexpr (HAS_B) bv[g] = __ldg(bbase + idx);
                    else bv[g] = av[g];
                }
            }
#pragma unroll
            for (int g = 0; g < G; ++g) {
                if (i0 + (long long)g * NT + threadIdx.x < total) visit_vec(av[g], bv[g]);
                if constexpr (PER_VEC) { if (__any_sync(0xffffffffu, qn >= (unsigned)QDRAIN)) drain(); }
            }
            if constexpr (!PER_VEC) { if (__any_sync(0xffffffffu, qn >= (unsigned)QDRAIN)) drain(); }
            // a step adds at most G * NW * 2 * 2^FINE_KMAX to the h sums and G * V * 65535 to s32: far below 2^32 in 32 steps
            if ((step & 31) == 31) flush32();
        }
        flush32();
    } else
    for (int y = y0; y < y1; y += G) {
        for (int it = 0; it < iters; ++it) {
            const int v = it * NT + (int)threadIdx.x;
            uint4 av[G], bv[G];
            if (v < nvec) {
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    const int yy = min(y + g, y1 - 1);
                    av[g] = __ldg(reinterpret_cast<const uint4*>(a + (size_t)yy * p.a_pitch) + v);
                    if constexpr (HAS_B) bv[g] = __ldg(reinterpret_cast<const uint4*>(b + (size_t)yy * p.b_pitch) + v);
                    else bv[g] = av[g];
                }
            }
#pragma unroll
            for (int g = 0; g < G; ++g) {
                if (v < nvec && y + g < y1) visit_vec(av[g], bv[g]);
                if constexpr (PER_VEC) { if (__any_sync(0xffffffffu, qn >= (unsigned)QDRAIN)) drain(); }
            }
            if constexpr (!PER_VEC) { if (__any_sync(0xffffffffu, qn >= (unsigned)QDRAIN)) drain(); }
        }
        const int x = nvec * V + threadIdx.x;
        if (x < p.w) {
            for (int g = 0; g < G && y + g < y1; ++g) {
                const T at = reinterpret_cast<const T*>(a + (size_t)(y + g) * p.a_pitch)[x];
                const T bt = HAS_B ? reinterpret_cast<const T*>(b + (size_t)(y + g) * p.b_pitch)[x] : at;
                visit_one(at, bt);
            }
        }
        // a thread visits at most G * iters * NW <= 4 * 32 * 8 words per group of rows, each adds at most 2 * 2^FINE_KMAX: below 2^22
        tot_h0 += sum_h0; tot_h1 += sum_h1;
        sum_h0 = sum_h1 = 0u;
        acc.idiff += idiff32; idiff32 = 0;
        if constexpr (AVG >= 0 && !FAVG) {  // same bound: <= 4 * 32 * 8 * 65535 in s32 per group of rows
            sum64 += s32; s32 = 0u;
        }
    }
    if constexpr (FAVG) {
        acc.fsum = fsum;
        acc.excluded = fexcluded;
    } else if constexpr (AVG >= 0) {
        unsigned long long removed = 0ull;
        unsigned int excluded = 0u;
#pragma unroll
        for (int e = 0; e < AVG; ++e) {
            const unsigned int cnt = seen - differing[e];
            excluded += cnt;
            removed += (unsigned long long)cnt * (unsigned)j.excl_i[e];
        }
        if constexpr (HAS_B) acc.fsum = (double)(sum64 - removed);
        else acc.idiff = sum64 - removed;
        acc.excluded = excluded;
    }
    drain();
    // exact counts of the lane's vector samples: (sum of h - the inside samples' share) / 2^k are at or above u; those at or above
    // l_min are the ones at or above u_min plus the inside ones
    ge_lmin += (unsigned int)((tot_h0 - in_h0) >> kbits) + in_n0;
    ge_umax += (unsigned int)((tot_h1 - in_h1) >> kbits);
    acc.isum = (unsigned long long)ge_lmin + ((unsigned long long)ge_umax << 32);
    acc.imin = min(pk_min & 0xffffu, pk_min >> 16);
    acc.imax = max(pk_max & 0xffffu, pk_max >> 16);
    __syncthreads();
    unsigned int* gf = j.bfine + fp * (2 * FINE_W);
    for (int i = threadIdx.x; i < 2 * FINE_W; i += NT) {
        const unsigned int c = (&s_fine[0][0])[i];
        if (c) atomicAdd(&gf[i], c);
    }
    Partial total;
    if (!block_finish(j, frame, k, local, p.b_nctas, j.counters + fp, acc, total)) return;
    // ---- last CTA: resolve both ranks exactly if they lie inside their brackets (warp 0: min, warp 1: max)
    __shared__ unsigned int s_cnt[2], s_ans[2];
    __shared__ int s_okk[2];
    if (threadIdx.x == 0) {
        StatsRaw& r = j.out[fp];
        if constexpr (AVG >= 0) {
            StatsRaw ra{};
            if constexpr (HAS_B && !FAVG) ra.isum = (unsigned long long)total.fsum;
            else { ra.isum = total.idiff; ra.fsum = total.fsum; }
            ra.excluded = total.excluded;
            if constexpr (HAS_B) { ra.idiff = r.idiff = total.idiff; ra.fdiff = r.fdiff = total.fdiff; }
            j.out_avg[fp] = ra;
        } else {
            r.idiff = total.idiff; r.fdiff = total.fdiff;
        }
        const unsigned long long npx0 = (unsigned long long)p.w * p.h;
        s_cnt[0] = (unsigned int)(npx0 - (total.isum & 0xffffffffull));  // samples below l_min
        s_cnt[1] = (unsigned int)(total.isum >> 32);                     // samples at or above u_max
        s_okk[0] = s_okk[1] = 0;
        s_ans[0] = total.imin; s_ans[1] = total.imax;
    }
    for (int i = threadIdx.x; i < 2 * FINE_W; i += NT) (&s_fine[0][0])[i] = __ldcg(gf + i);
    __syncthreads();
    const bool above_peak = TRACK && s_ans[1] >= hist_size;
    __syncthreads();  // every thread has read s_ans before warps 0/1 overwrite it below (racecheck)
    if (above_peak) return;  // samples above the peak: exact path
    const unsigned long long npx = (unsigned long long)p.w * p.h;
    const int side = threadIdx.x >> 5;
    if (side < 2) {
        const unsigned int thr = side == 0 ? p.tmin : p.tmax;
        const unsigned int width = side == 0 ? w_min : w_max;
        const unsigned int outside = s_cnt[side];
        // bins in scan order: ascending for the min rank, descending for the max rank
        constexpr int PER = FINE_W / 32;
        unsigned int mine[PER], sum = 0u;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const unsigned int o = (unsigned)(lane * PER + i);
            mine[i] = o < width ? s_fine[side][side == 0 ? o : width - 1u - o] : 0u;
            sum += mine[i];
        }
        unsigned int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        const unsigned int before = outside + incl - sum;
        const unsigned int inside_total = __shfl_sync(0xffffffffu, incl, 31);
        if ((unsigned long long)thr >= npx) { if (lane == 0) { s_okk[side] = 1; s_ans[side] = side == 0 ? hist_size - 1u : 0u; } }  // planeminmax.zig:44-48
        else if (thr == 0u) { if (lane == 0) s_okk[side] = TRACK ? 1 : 0; }  // first / last non-empty bin (already in s_ans)
        else if (side == 0 && l_min == 1u && outside > thr) { if (lane == 0) { s_okk[0] = 1; s_ans[0] = 0u; } }  // "below the bracket" is bin 0 alone
        else if (side == 1 && l_max == 1u && outside + inside_total <= thr) { if (lane == 0) { s_okk[1] = 1; s_ans[1] = 0u; } }  // ditto, scanning down
        else if (outside <= thr && before <= thr && before + sum > thr) {
            unsigned int c = before;
#pragma unroll
            for (int i = 0; i < PER; ++i) {
                c += mine[i];
                if (c > thr) {
                    const unsigned int o = (unsigned)(lane * PER + i);
                    s_ans[side] = side == 0 ? l_min + o : l_max + (width - 1u - o);
                    s_okk[side] = 1;
                    break;
                }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0 && s_okk[0] && s_okk[1]) {
        StatsRaw& r = j.out[fp];
        r.bin_min = s_ans[0]; r.bin_max = s_ans[1];
        j.brackets[fp].done = 1u;
    }
}

// =========================================================================== host launchers
static constexpr int MAX_BATCH = 32768;  // frames per call

static size_t align256(size_t v) { return (v + 255) / 256 * 256; }
// The scratch regions, laid out from base (n = frames * planes): stats_scratch_bytes walks them from 0, make_job from the scratch
// buffer.  Everything before `partials` is zeroed before each call.  Returns the bytes they take.
static size_t lay_out_scratch(StatsJob& j, uintptr_t base, size_t n) {
    uintptr_t p = base;
    auto take = [&](size_t bytes) { const uintptr_t r = p; p += align256(bytes); return r; };
    const uintptr_t c = take(3 * n * 4);  // counters, counters2, counters3
    j.counters = (unsigned int*)c; j.counters2 = (unsigned int*)(c + n * 4); j.counters3 = (unsigned int*)(c + 2 * n * 4);
    j.coarse = (unsigned int*)take(n * 256 * 4);
    j.ssample = (unsigned int*)take(n * SBINS * 4);
    j.fine = (unsigned int*)take(n * 512 * 4);
    j.bfine = (unsigned int*)take(n * 2 * FINE_W * 4);
    j.brackets = (Bracket*)take(n * sizeof(Bracket));
    j.partials = (Partial*)take(n * MAX_CTAS_PER_PLANE * sizeof(Partial));
    return p - base;
}
size_t stats_scratch_bytes(int count, int np) {
    StatsJob j;
    return lay_out_scratch(j, 0, (size_t)count * np);
}
// zeroes the scratch regions before `partials`
static cudaError_t clear_scratch(const StatsJob& j, void* scratch, cudaStream_t st) {
    return cudaMemsetAsync(scratch, 0, (const char*)j.partials - (const char*)scratch, st);
}

// a and b (clipb, nullptr when there is none) share the frame stride fs
static StatsJob make_job(const FrameLayout& l, const bool mask[3], const char* a, const char* b, size_t fs, int count, void* scratch,
                         StatsRaw* out) {
    StatsJob j{};
    j.a = a; j.b = b; j.a_fs = j.b_fs = fs;
    int cta = 0, scta = 0, bcta = 0, k = 0;
    for (int p = 0; p < l.nplanes; ++p) {
        if (!mask[p]) continue;
        StatsPlane& s = j.pl[k++];
        s.a_off = s.b_off = l.pl[p].offset;
        s.a_pitch = s.b_pitch = l.pl[p].pitch;
        s.w = l.pl[p].w; s.h = l.pl[p].h;
        // ~32K samples per CTA keeps >= 2 waves on 148 SMs for a single 4K plane and bounds the
        // per-thread u32 partial sums
        const long long px = (long long)s.w * s.h;
        int n = (int)std::min<long long>(MAX_CTAS_PER_PLANE, std::max<long long>(1, (px + 32767) / 32768));
        // once the batch alone fills the GPU many times over, 4x longer CTAs amortise the per-CTA reduction epilogue
        if ((long long)count * n >= 4096) n = std::max(1, n / 4);
        n = std::min(n, s.h);
        s.cta_begin = cta; s.nctas = n;
        cta += n;
        // line sample of the threshold fast path: planes under 1 M samples are sampled completely
        s.s_lpr = (s.w * l.bps + 127) / 128;
        s.s_step = 1;
        if (px >= (1ll << 20)) {
            s.s_step = 16;
            if (s.s_lpr % 2 == 0) s.s_step = s.s_lpr % 17 ? 17 : 19;  // coprime with the lines per row
        }
        const long long nsl = ((long long)s.h * s.s_lpr + s.s_step - 1) / s.s_step;
        s.s_nctas = (int)std::min<long long>(16, std::max<long long>(1, nsl / (NT / 8 * 8)));
        s.s_cta_begin = scta;
        scta += s.s_nctas;
        s.b_nctas = n;  // the bracket kernel keeps its own plane map (historical; same partition as the other kernels now)
        s.b_cta_begin = bcta;
        bcta += s.b_nctas;
    }
    j.nplanes = k; j.ctas_per_frame = cta; j.sample_ctas_per_frame = scta; j.bracket_ctas_per_frame = bcta;
    lay_out_scratch(j, (uintptr_t)scratch, (size_t)count * k);
    j.out = out;
    return j;
}

// hist_size and the thresholds of PlaneMinMax as the threshold kernels read them
static void set_thresholds(StatsJob& j, uint32_t hist_size, float minthr, float maxthr) {
    j.hist_size = hist_size;
    int bits = 0;
    while ((1u << bits) < hist_size) ++bits;
    j.shift = bits > 8 ? bits - 8 : 0;
    j.sshift = bits > SBITS ? bits - SBITS : 0;
    for (int k = 0; k < j.nplanes; ++k) {
        const double total = (double)((uint32_t)j.pl[k].w * (uint32_t)j.pl[k].h);
        j.pl[k].tmin = (unsigned int)(total * (double)minthr);  // trunc (src/filters/planeminmax.zig:40-41)
        j.pl[k].tmax = (unsigned int)(total * (double)maxthr);
    }
}

// Whether the threshold path may start with the line sample: every plane under 2^31 samples, and VSZIP_MINMAX_EXACT is not 1 (read on
// every call; the tests set it to exercise the exact kernels).
static bool sampled_path_allowed(const StatsJob& j) {
    const char* ev = getenv("VSZIP_MINMAX_EXACT");
    if (ev && ev[0] == '1') return false;
    for (int k = 0; k < j.nplanes; ++k)
        if ((long long)j.pl[k].w * j.pl[k].h >= (1ll << 31)) return false;
    return true;
}

// The exclude values that can match a sample of this kind, each once: integers outside the sample range are dropped, float lists are
// deduplicated as floats.  Writes them to ex / exf and returns how many; -1 when there are more than 4 or the list has more than 16
// entries.
static int distinct_exclude(SampleKind kind, const int32_t* excl, const float* excl_f, int nex, int32_t* ex, float* exf) {
    if (nex > 16) return -1;
    const bool flt = kind == K_F16 || kind == K_F32;
    const int32_t top = kind == K_U8 ? 255 : 65535;
    int m = 0;
    for (int i = 0; i < nex; ++i) {
        const int32_t v = excl[i];
        if (!flt && (v < 0 || v > top)) continue;  // can never match a sample
        bool dup = false;
        for (int t = 0; t < m; ++t) dup = dup || (flt ? exf[t] == excl_f[i] : ex[t] == v);
        if (dup) continue;
        if (m == 4) return -1;
        ex[m] = v; exf[m] = excl_f[i];
        ++m;
    }
    return m;
}

// Calls launch(Type<T>{}, std::bool_constant<HAS_B>{}) for the clip's sample type and whether a clipb is read, then checks the launches.
template <typename T> struct Type { using type = T; };
template <class F> static int dispatch(SampleKind kind, bool has_b, F&& launch) {
    auto with_b = [&](auto t) { if (has_b) launch(t, std::true_type{}); else launch(t, std::false_type{}); };
    switch (kind) {
        case K_U8: with_b(Type<uint8_t>{}); break;
        case K_U16: with_b(Type<uint16_t>{}); break;
        case K_F16: with_b(Type<__half>{}); break;
        case K_F32: with_b(Type<float>{}); break;
        default: return -1;
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

// The single-read kernel: raw min/max (PlaneMinMax without thresholds), PlaneAverage, or both (BOTH).
template <typename T, bool HAS_B, bool AVERAGE, bool BOTH = false>
static void launch_stats(const StatsJob& j, int count, cudaStream_t st) {
    const dim3 grid(j.ctas_per_frame, count);
    if constexpr (!AVERAGE) stats_kernel<T, HAS_B, false><<<grid, NT, 0, st>>>(j);
    else if (j.nex > 4) stats_kernel<T, HAS_B, true, true, BOTH><<<grid, NT, 0, st>>>(j);
    else stats_kernel<T, HAS_B, true, false, BOTH><<<grid, NT, 0, st>>>(j);
    count_launch();
}

// The threshold path of PlaneMinMax, with PlaneAverage's exclude compares unrolled AVG times in the bracket kernel (-1: PlaneMinMax
// alone).  Sampled: the line sample brackets both ranks, one full read resolves most planes, and the exact two-pass select takes the
// rest.  Otherwise (PlaneMinMax alone): the exact two-pass select on every plane.
template <typename T, bool HAS_B, int AVG>
static void launch_threshold(const StatsJob& j, int count, bool sampled, cudaStream_t st) {
    // Pass 2 re-reads what pass 1 read.  Running the pair on L2-sized chunks (<= 64 MB) was measured SLOWER on
    // B200 (3-frame launches leave the GPU under-filled and add launch gaps: 42 k vs 77 k fps on 4K GRAY16), so the
    // whole batch goes through each pass; single frames (<= 64 MB) still hit L2 on the second read.
    if (sampled) {
        hist_sample_kernel<T><<<dim3(j.sample_ctas_per_frame, count), NT, 0, st>>>(j);  // 1/16 of the lines
        // one full read (also Diff); the lean variant needs every bin valid and both ranks > 0 on every plane
        bool lean = (j.hist_size == 65536u) || (sizeof(T) == 1 && j.hist_size == 256u);
        for (int k = 0; k < j.nplanes; ++k) lean = lean && j.pl[k].tmin > 0u && j.pl[k].tmax > 0u;
        const dim3 bgrid(j.bracket_ctas_per_frame, count);
        if (lean) minmax_bracket_kernel<T, HAS_B, false, AVG><<<bgrid, NT, 0, st>>>(j);
        else minmax_bracket_kernel<T, HAS_B, true, AVG><<<bgrid, NT, 0, st>>>(j);
        count_launch(2);
    }
    // exact two-pass select: after the sampled path only for the planes it could not resolve (else immediate exit)
    const dim3 xgrid(j.ctas_per_frame, sampled ? std::min(count, 8) : count);
    if (sampled) hist_coarse_kernel<T, false><<<xgrid, NT, 0, st>>>(j, count);  // Diff came from the bracket kernel
    else hist_coarse_kernel<T, HAS_B><<<xgrid, NT, 0, st>>>(j, count);
    hist_fine_kernel<T><<<xgrid, NT, 0, st>>>(j, count);
    count_launch(2);
}

int run_planeminmax(const FrameLayout& l, const bool mask[3], const char* a, const char* b, size_t fs, int count, bool no_thr,
                    float minthr, float maxthr, uint32_t hist_size, void* scratch, StatsRaw* out_dev, cudaStream_t st) {
    StatsJob j = make_job(l, mask, a, b, fs, count, scratch, out_dev);
    if (j.ctas_per_frame == 0) return 0;
    VSZ_CUDA(clear_scratch(j, scratch, st));
    VSZ_CUDA(cudaMemsetAsync(out_dev, 0, sizeof(StatsRaw) * (size_t)count * j.nplanes, st));
    if (count > MAX_BATCH) { set_error("PlaneMinMax: batches above %d frames are not supported", MAX_BATCH); return -2; }
    set_thresholds(j, hist_size, minthr, maxthr);
    return dispatch(l.kind, b != nullptr, [&](auto t, auto hb) {
        using T = typename decltype(t)::type;
        if (no_thr) launch_stats<T, decltype(hb)::value, false>(j, count, st);
        else launch_threshold<T, decltype(hb)::value, -1>(j, count, sampled_path_allowed(j), st);
    });
}

// PlaneMinMax + PlaneAverage of the same planes from ONE read (SURVEY 8f rank 4).  run_planestats_fused returns 1 when the
// combination is not eligible (the caller then runs the two reductions separately), 0 on success, < 0 on error.
// Eligible: at most 32768 frames; without thresholds any sample type and up to 16 exclude values; with thresholds (sampled fast
// path enabled) at most 4 distinct exclude values that can match a sample.  b (clipb, may be nullptr): both filters read it; Diff
// is accumulated once, in the order of the separate kernels.  same_float_sums: fuse a float clip with thresholds only when its float
// sums come out bit-identical to the separate calls - the bracket kernel walks a plane whose rows are back to back (no row padding)
// as one run of vectors, which the separate PlaneAverage kernel does not, so such planes are not fused.  Always on with clipb, so
// that a float Diff is the same whichever route ran.
int run_planestats_fused(const FrameLayout& l, const bool mask[3], const char* a, const char* b, size_t fs, int count, bool no_thr,
                         float minthr, float maxthr, uint32_t hist_size, const int32_t* excl, const float* excl_f, int nex,
                         bool same_float_sums, void* scratch, StatsRaw* out_mm, StatsRaw* out_avg, cudaStream_t st) {
    if (count <= 0 || count > MAX_BATCH) return 1;
    StatsJob j = make_job(l, mask, a, b, fs, count, scratch, out_mm);
    if (j.ctas_per_frame == 0) return 1;
    j.out_avg = out_avg;
    if (no_thr) {
        if (nex > 16) return 1;
        VSZ_CUDA(clear_scratch(j, scratch, st));
        j.nex = nex;
        for (int i = 0; i < nex; ++i) { j.excl_i[i] = excl[i]; j.excl_f[i] = excl_f[i]; }
        return dispatch(l.kind, b != nullptr, [&](auto t, auto hb) {
            launch_stats<typename decltype(t)::type, decltype(hb)::value, true, true>(j, count, st);
        });
    }
    j.nex = distinct_exclude(l.kind, excl, excl_f, nex, j.excl_i, j.excl_f);
    if (j.nex < 0 || !sampled_path_allowed(j)) return 1;
    const bool flt = l.kind == K_F16 || l.kind == K_F32;
    for (int k = 0; k < j.nplanes; ++k) {
        const int nvec = j.pl[k].w / (16 / l.bps);  // minmax_bracket_kernel's `contiguous` test
        if (flt && (same_float_sums || b) && nvec > 0 && j.pl[k].a_pitch == nvec * 16) return 1;
    }
    VSZ_CUDA(clear_scratch(j, scratch, st));
    VSZ_CUDA(cudaMemsetAsync(out_mm, 0, sizeof(StatsRaw) * (size_t)count * j.nplanes, st));
    set_thresholds(j, hist_size, minthr, maxthr);
    return dispatch(l.kind, b != nullptr, [&](auto t, auto hb) {
        using T = typename decltype(t)::type;
        constexpr bool HAS_B = decltype(hb)::value;
        switch (j.nex) {
            case 0: launch_threshold<T, HAS_B, 0>(j, count, true, st); break;
            case 1: launch_threshold<T, HAS_B, 1>(j, count, true, st); break;
            case 2: launch_threshold<T, HAS_B, 2>(j, count, true, st); break;
            case 3: launch_threshold<T, HAS_B, 3>(j, count, true, st); break;
            default: launch_threshold<T, HAS_B, 4>(j, count, true, st); break;
        }
    });
}

int run_planeaverage(const FrameLayout& l, const bool mask[3], const char* a, const char* b, size_t fs, int count, const int32_t* excl_i,
                     const float* excl_f, int nex, const int32_t* excl_i_dev, const float* excl_f_dev, void* scratch, StatsRaw* out_dev,
                     cudaStream_t st) {
    StatsJob j = make_job(l, mask, a, b, fs, count, scratch, out_dev);
    if (j.ctas_per_frame == 0) return 0;
    if (nex > 16 && (!excl_i_dev || !excl_f_dev)) { set_error("PlaneAverage: internal error, long exclude list not uploaded"); return -2; }
    VSZ_CUDA(clear_scratch(j, scratch, st));
    if (count > MAX_BATCH) { set_error("PlaneAverage: batches above %d frames are not supported", MAX_BATCH); return -2; }
    j.nex = nex;
    for (int i = 0; i < std::min(nex, 16); ++i) { j.excl_i[i] = excl_i[i]; j.excl_f[i] = excl_f[i]; }
    j.excl_i_more = excl_i_dev; j.excl_f_more = excl_f_dev;  // the whole list (entries >= 16 are read from here)
    return dispatch(l.kind, b != nullptr, [&](auto t, auto hb) {
        using T = typename decltype(t)::type;
        constexpr bool HAS_B = decltype(hb)::value;
        // packed path for 16-bit integer clips: at most 4 distinct exclude values inside the sample range
        if constexpr (std::is_same<T, uint16_t>::value && !HAS_B) {
            StatsJob q = j;
            const int m = distinct_exclude(l.kind, excl_i, excl_f, nex, q.excl_i, q.excl_f);
            const dim3 grid(j.ctas_per_frame, count);
            switch (m) {
                case 0: average_u16_kernel<0><<<grid, NT, 0, st>>>(q); break;
                case 1: average_u16_kernel<1><<<grid, NT, 0, st>>>(q); break;
                case 2: average_u16_kernel<2><<<grid, NT, 0, st>>>(q); break;
                case 3: average_u16_kernel<3><<<grid, NT, 0, st>>>(q); break;
                case 4: average_u16_kernel<4><<<grid, NT, 0, st>>>(q); break;
            }
            if (m >= 0) { count_launch(); return; }
        }
        launch_stats<T, HAS_B, true>(j, count, st);
    });
}

}  // namespace vsz
