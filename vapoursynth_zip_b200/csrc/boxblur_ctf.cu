// boxblur_ctf.cu — vszip.BoxBlur, comptime FLOAT path (hradius == vradius <= 22, one pass each) on f16 / f32 clips.
//
// Reference (src/filters/boxblur_comptime.zig:161-263): V first, then H; every output is the tap-ordered sum
//     acc = 0;  for k in 0..2r:  acc = acc + div * v[k]            (f32, separate multiply and add)
// with reflect-101 indexing at the low edge and the reference's "m - over" rule at the high edge (r101q in
// boxblur_kernels.cu), narrowed to T after each direction.  Neighbouring outputs share no partial sums (each has its own
// rounding history), so bit-exactness costs 2r+1 dependent adds per output and direction.  The kernels here spend exactly
// those adds and almost nothing else:
//
//   A thread walks ALONG a line and keeps the 2r+1 outputs whose windows contain the current sample in registers.  Every new
//   sample p = div*v is added to all of them (2r+1 independent FADDs: the ILP that keeps the FP32 pipe full with few warps),
//   the oldest one is complete and leaves, a new one starts (acc = 0 + p).  Each output still adds its taps in the
//   reference's order, so results are bit-identical.  Per sample: one load, one multiply, 2r+1 adds, one store.
//   The loop is unrolled by 2r+1 so that the rotating accumulators have static register names.
//
//   ctf_v_kernel  columns: thread = column (f16: two columns), rows arrive by coalesced loads that are issued one whole block
//                 of 2r+1 rows ahead into the registers the consumed samples leave behind.
//   ctf_h_kernel  rows: thread = row; a CTA owns 128 rows and streams along them in tiles of 2r+1 columns that the TMA engine
//                 (cp.async.bulk.tensor, mbarrier completion, double buffered) drops into shared memory with a row pitch that makes the
//                 per-row 16-byte reads conflict-free; results collect in a per-row shared-memory ring that a fifth warp
//                 drains to global memory in whole aligned 128-byte lines underneath the arithmetic.
//   The first / last r outputs of a line (mirrored windows) are computed from 2r samples held in registers with compile-time
//   tap indices.  Long lines are cut into segments (each pays 2r warm-up samples) so that single-frame calls fill the GPU too.
//
// Planes with fewer than 2r+1 rows or columns keep the tiled kernel of boxblur_kernels.cu.
#include <cuda_fp16.h>

#include <algorithm>
#include <type_traits>
#include <utility>

#include "boxblur_host.h"
#include "boxblur_tma.h"
#include "common.h"
#include "filter.h"

namespace vsz {

namespace {

constexpr int kThreads = 128;
#ifndef VSZ_CTF_HROWS
#define VSZ_CTF_HROWS 64
#endif
// rows (= row threads) per CTA of the H kernel.  64 rows and 2 TMA stages need 44 KB of shared memory (f32, r = 13): 5 CTAs of 3 warps per SM
// instead of 2 CTAs of 5 warps with 128 rows and 3 stages (4K YUV444PS r = 13: 84.3 -> 81.4 us per frame, r = 22: 171 -> 146, 1080p GRAYS 7.4 -> 7.0;
// 32 rows: 101 us - one store warp per 32 row threads is too many)
constexpr int kHRows = VSZ_CTF_HROWS;

struct CtfPlane {
    size_t src_off, dst_off;
    int src_pitch, dst_pitch;
    int w, h;
    int cta_begin;
    int cross_blocks;   // CTAs across the axis that is not blurred
    int segs, seg_len;  // pieces along the blurred axis; piece s owns the interior outputs [r + s*seg_len, r + (s+1)*seg_len)
};
struct CtfJob {
    const char* src;
    char* dst;
    size_t src_fs, dst_fs;
    int nplanes, ctas_per_frame;
    float div;
    CtfPlane pl[3];
};
struct CtfMaps { CUtensorMap in[3]; };

__device__ __forceinline__ const CtfPlane& ctf_plane(const CtfJob& b, int cta, int& local) {
    int k = b.nplanes - 1;
    while (k > 0 && cta < b.pl[k].cta_begin) --k;
    local = cta - b.pl[k].cta_begin;
    return b.pl[k];
}

// compile-time loop: f(std::integral_constant<int, I>) for I in [0, N)
template <int I, int N, class F>
__device__ __forceinline__ void static_for(F&& f) {
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, N>(f);
    }
}

// ---- sample packs: what one thread of the V kernel loads per row
template <typename T> struct Smp;
template <> struct Smp<float> {
    static constexpr int NC = 1;
    using Pack = float;
    static __device__ __forceinline__ void unpack(Pack v, float (&f)[1]) { f[0] = v; }
    static __device__ __forceinline__ Pack pack(const float (&f)[1]) { return f[0]; }
};
template <> struct Smp<__half> {
    static constexpr int NC = 2;
    using Pack = __half2;
    static __device__ __forceinline__ void unpack(Pack v, float (&f)[2]) { const float2 t = __half22float2(v); f[0] = t.x; f[1] = t.y; }
    static __device__ __forceinline__ Pack pack(const float (&f)[2]) { return __floats2half2_rn(f[0], f[1]); }
};

// ---- mirrored windows with compile-time tap indices (lines of at least 2r+1 samples)
// low edge: output i in [0, r), taps k = 0..2r read sample |i + k - r| of e[0..2r) = samples 0..2r-1 (reflect-101)
template <int R, int NC, int I>
__device__ __forceinline__ void edge_low_i(const float (&pe)[2 * R][NC], float (&a)[NC]) {
#pragma unroll
    for (int c = 0; c < NC; ++c) a[c] = 0.f;
#pragma unroll
    for (int k = 0; k <= 2 * R; ++k) {
        const int j = (I + k - R) < 0 ? -(I + k - R) : (I + k - R);
#pragma unroll
        for (int c = 0; c < NC; ++c) a[c] = __fadd_rn(a[c], pe[j][c]);
    }
}
// high edge: output n-1-D (D in [0, r)), e[0..2r) = samples n-2r..n-1.  Taps before the centre read i+k-r; taps after it read
// i+over while that stays inside the line and n-1-over afterwards (boxblur_comptime.zig:228-230,257-259).
template <int R, int NC, int D>
__device__ __forceinline__ void edge_high_d(const float (&pe)[2 * R][NC], float (&a)[NC]) {
#pragma unroll
    for (int c = 0; c < NC; ++c) a[c] = 0.f;
#pragma unroll
    for (int k = 0; k <= 2 * R; ++k) {
        const int over = k - R;
        const int j = k < R ? (R - 1 - D + k) : (D < over ? 2 * R - 1 - over : 2 * R - 1 - D + over);
#pragma unroll
        for (int c = 0; c < NC; ++c) a[c] = __fadd_rn(a[c], pe[j][c]);
    }
}
template <int R, int NC, int I, class F>
__device__ __forceinline__ void edge_low_all(const float (&pe)[2 * R][NC], F&& emit) {
    if constexpr (I < R) {
        float a[NC];
        edge_low_i<R, NC, I>(pe, a);
        emit(I, a);
        edge_low_all<R, NC, I + 1>(pe, emit);
    }
}
template <int R, int NC, int D, class F>
__device__ __forceinline__ void edge_high_all(const float (&pe)[2 * R][NC], F&& emit) {  // emit(distance from the last sample, value)
    if constexpr (D < R) {
        float a[NC];
        edge_high_d<R, NC, D>(pe, a);
        emit(D, a);
        edge_high_all<R, NC, D + 1>(pe, emit);
    }
}

// ---- the streaming step: sample p enters every live window; slot FRESH starts over with it
template <int K, int NC, int FRESH>
__device__ __forceinline__ void push(float (&acc)[K][NC], const float (&p)[NC]) {
#pragma unroll
    for (int s = 0; s < K; ++s)
#pragma unroll
        for (int c = 0; c < NC; ++c) acc[s][c] = __fadd_rn(s == FRESH ? 0.f : acc[s][c], p[c]);
}

// =========================================================================== V
template <typename T, int R>
__global__ void __launch_bounds__(kThreads) ctf_v_kernel(const CtfJob job) {
    constexpr int K = 2 * R + 1, NC = Smp<T>::NC;
    using Pack = typename Smp<T>::Pack;
    int local;
    const CtfPlane& pj = ctf_plane(job, blockIdx.y, local);
    const int cb = local % pj.cross_blocks, sg = local / pj.cross_blocks;
    const int x = (cb * kThreads + threadIdx.x) * NC;
    if (x >= pj.w) return;  // (a second column beyond an odd width lands in the pitch padding: a don't-care lane)
    const char* src = job.src + (size_t)blockIdx.x * job.src_fs + pj.src_off + (size_t)x * sizeof(T);
    char* dst = job.dst + (size_t)blockIdx.x * job.dst_fs + pj.dst_off + (size_t)x * sizeof(T);
    const int h = pj.h;
    const uint32_t sp = (uint32_t)pj.src_pitch, dp = (uint32_t)pj.dst_pitch;
    const float div = job.div;
    auto ld = [&](int row) { return *reinterpret_cast<const Pack*>(src + (size_t)((uint32_t)row * sp)); };
    auto st = [&](int row, const float (&a)[NC]) { *reinterpret_cast<Pack*>(dst + (size_t)((uint32_t)row * dp)) = Smp<T>::pack(a); };
    auto mul = [&](Pack v, float (&p)[NC]) {
        float f[NC];
        Smp<T>::unpack(v, f);
#pragma unroll
        for (int c = 0; c < NC; ++c) p[c] = __fmul_rn(div, f[c]);
    };

    const int ys = R + sg * pj.seg_len, ye = min(ys + pj.seg_len, h - R);  // interior outputs of this piece
    const int ts = ys - R, n = ye - ys + 2 * R;                            // rows ts .. ts+n-1 are consumed, n >= 2r+1
    Pack cv[K];
#pragma unroll
    for (int u = 0; u < K; ++u) cv[u] = ld(ts + u);                        // n >= K

    if (sg == 0) {  // rows 0..r-1 from rows 0..2r-1, which are the first samples of this piece
        float pe[2 * R][NC];
#pragma unroll
        for (int j = 0; j < 2 * R; ++j) mul(cv[j], pe[j]);
        edge_low_all<R, NC, 0>(pe, [&](int i, const float (&a)[NC]) { st(i, a); });
    }

    float acc[K][NC];
#pragma unroll
    for (int s = 0; s < K; ++s)
#pragma unroll
        for (int c = 0; c < NC; ++c) acc[s][c] = 0.f;
    // step t (row ts+t) uses slot t mod K as its fresh slot; the window that started at step t-2r (slot (t+1) mod K) is complete.
    // Whole blocks only: the steps past the piece's end run on rows clamped to the plane and store nothing (every load is
    // unconditional and lands in the register its consumer reads a block later - a predicated load would go through a
    // temporary that the next step has to wait for).
    const int last = h - 1;
    for (int base = 0; base < n; base += K) {
        static_for<0, K>([&](auto uc) {
            constexpr int U = decltype(uc)::value;
            const int t = base + U;
            const Pack v = cv[U];
            cv[U] = ld(min(ts + t + K, last));
            float p[NC];
            mul(v, p);
            push<K, NC, U>(acc, p);
            if (t >= 2 * R && t < n) st(ts + t - R, acc[(U + 1) % K]);
        });
    }

    if (sg == pj.segs - 1) {  // rows h-r..h-1 from rows h-2r..h-1
        float pe[2 * R][NC];
#pragma unroll
        for (int j = 0; j < 2 * R; ++j) mul(ld(h - 2 * R + j), pe[j]);
        edge_high_all<R, NC, 0>(pe, [&](int d, const float (&a)[NC]) { st(h - 1 - d, a); });
    }
}

// =========================================================================== H
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "CTF_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra CTF_WAIT_DONE;\n"
        "bra CTF_WAIT_LOOP;\n"
        "CTF_WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* sdst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                     smem_u32(sdst)),
                 "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
                 : "memory");
}

// Tile geometry.  The TMA engine wants the first byte of a box row 16-byte aligned, i.e. the box's x coordinate a multiple of VEC
// samples, while block i of a line starts at sample a_i = xs + r + i*(2r+1) (odd step): the box starts at a_i rounded down and the
// thread skips PH = a_i mod VEC samples (a switch over VEC compile-time variants of "copy the tile's registers").  A tile row holds NV
// 16-byte vectors - enough for the worst phase, and an ODD number so that the 8 threads of a quarter-warp, one row each, cover
// all 32 banks with their 16-byte accesses.
#ifndef VSZ_CTF_STAGES
#define VSZ_CTF_STAGES 2
#endif
template <typename T, int R> struct HTile {
    static constexpr int K = 2 * R + 1;
    static constexpr int VEC = 16 / (int)sizeof(T);
    static constexpr int MB = K >= 32 ? 1 : 32 / K;               // blocks of 2r+1 steps per tile (small radii: fewer, larger tiles)
    static constexpr int TS = MB * K;                            // samples a tile advances along the row
    static constexpr int NVR = (TS + VEC - 1 + VEC - 1) / VEC;  // vectors a thread reads: covers PH + TS samples for every PH < VEC
    static constexpr int NV = NVR | 1;
    static constexpr int TW = NV * VEC;                          // samples per input tile row (TMA box width)
    static constexpr int ROW_BYTES = NV * 16;
    // results: a ring of RCH aligned 128-byte chunks per row (+ one vector of padding: odd pitch again); the store warp writes a
    // chunk to global memory once all of it has been produced, so global stores are whole aligned 128-byte lines
    static constexpr int CH = 128 / (int)sizeof(T);              // samples per chunk
    static constexpr int RCH = (2 * TS + CH - 1 + CH - 1) / CH;  // chunks: two tiles may be in flight behind an incomplete chunk
    static constexpr int RV = RCH * 8;                           // ring vectors per row
    static constexpr int OROW_BYTES = (RV + 1) * 16;
    static constexpr int STAGES = VSZ_CTF_STAGES;
    static constexpr int TILE_BYTES = kHRows * ROW_BYTES;
    static constexpr int RING_BYTES = kHRows * OROW_BYTES;
    static constexpr int SMEM = STAGES * TILE_BYTES + RING_BYTES;
};

// xv[u] = e[PH + u], PH known at compile time
template <int K, int PH, int N>
__device__ __forceinline__ void take_from(const float (&e)[N], float (&xv)[K]) {
#pragma unroll
    for (int u = 0; u < K; ++u) xv[u] = e[PH + u];
}
template <int K, int VEC, int N>
__device__ __forceinline__ void take_phase(const float (&e)[N], float (&xv)[K], int ph) {
    static_assert(VEC == 4 || VEC == 8, "16-byte vectors of f32 or f16");
    switch (ph) {
        case 0: take_from<K, 0>(e, xv); break;
        case 1: take_from<K, 1>(e, xv); break;
        case 2: take_from<K, 2>(e, xv); break;
        case 3: take_from<K, 3>(e, xv); break;
        default:
            if constexpr (VEC == 8) {
                switch (ph) {
                    case 4: take_from<K, 4>(e, xv); break;
                    case 5: take_from<K, 5>(e, xv); break;
                    case 6: take_from<K, 6>(e, xv); break;
                    default: take_from<K, 7>(e, xv); break;
                }
            }
            break;
    }
}

template <typename T> __device__ __forceinline__ void vec_to_floats(const uint4& q, float* f);
template <> __device__ __forceinline__ void vec_to_floats<float>(const uint4& q, float* f) {
    f[0] = __uint_as_float(q.x); f[1] = __uint_as_float(q.y); f[2] = __uint_as_float(q.z); f[3] = __uint_as_float(q.w);
}
template <> __device__ __forceinline__ void vec_to_floats<__half>(const uint4& q, float* f) {
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
        f[2 * i] = t.x; f[2 * i + 1] = t.y;
    }
}
template <typename T> __device__ __forceinline__ uint4 floats_to_vec(const float* f);
template <> __device__ __forceinline__ uint4 floats_to_vec<float>(const float* f) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
}
template <> __device__ __forceinline__ uint4 floats_to_vec<__half>(const float* f) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __half2 h = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}
template <typename T> __device__ __forceinline__ float ld1(const T* p);
template <> __device__ __forceinline__ float ld1<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ld1<__half>(const __half* p) { return __half2float(*p); }
template <typename T> __device__ __forceinline__ T cvt1(float v);
template <> __device__ __forceinline__ float cvt1<float>(float v) { return v; }
template <> __device__ __forceinline__ __half cvt1<__half>(float v) { return __float2half_rn(v); }

// Appends the TS results of a tile to the row's ring.  The first of them sits PH samples into a 16-byte vector; the PH samples
// before it are the tail of the previous tile, kept in `carry`, so only whole vectors are written.  hv = ring index of that vector.
template <typename T, int TS, int VEC, int RV, int PH>
__device__ __forceinline__ void ring_put_case(const float (&xv)[TS], float (&carry)[VEC - 1], uint4* rowring, int hv) {
    constexpr int NVP = (PH + TS + VEC - 1) / VEC, NPH = (PH + TS) % VEC;
    float o[NVP * VEC];
#pragma unroll
    for (int j = 0; j < NVP * VEC; ++j) o[j] = j < PH ? carry[j < VEC - 1 ? j : 0] : (j - PH < TS ? xv[j - PH < TS ? j - PH : 0] : 0.f);
#pragma unroll
    for (int v = 0; v < NVP; ++v) {
        int idx = hv + v;
        if (idx >= RV) idx -= RV;
        rowring[idx] = floats_to_vec<T>(o + v * VEC);
    }
#pragma unroll
    for (int j = 0; j < NPH; ++j) carry[j] = xv[TS - NPH + j];
}
template <typename T, int TS, int VEC, int RV>
__device__ __forceinline__ void ring_put(const float (&xv)[TS], float (&carry)[VEC - 1], uint4* rowring, int hv, int ph) {
    switch (ph) {
        case 0: ring_put_case<T, TS, VEC, RV, 0>(xv, carry, rowring, hv); break;
        case 1: ring_put_case<T, TS, VEC, RV, 1>(xv, carry, rowring, hv); break;
        case 2: ring_put_case<T, TS, VEC, RV, 2>(xv, carry, rowring, hv); break;
        case 3: ring_put_case<T, TS, VEC, RV, 3>(xv, carry, rowring, hv); break;
        default:
            if constexpr (VEC == 8) {
                switch (ph) {
                    case 4: ring_put_case<T, TS, VEC, RV, 4>(xv, carry, rowring, hv); break;
                    case 5: ring_put_case<T, TS, VEC, RV, 5>(xv, carry, rowring, hv); break;
                    case 6: ring_put_case<T, TS, VEC, RV, 6>(xv, carry, rowring, hv); break;
                    default: ring_put_case<T, TS, VEC, RV, 7>(xv, carry, rowring, hv); break;
                }
            }
            break;
    }
}

// named barriers (bar 0 is __syncthreads): the full / empty hand-over of the output ring between the row threads and the store warp
constexpr int kStoreThreads = 32, kHThreads = kHRows + kStoreThreads;
enum { BAR_FULL = 2, BAR_EMPTY = 4 };
__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// Warps 0-3: one row per thread (the arithmetic); their results go into a per-row ring in shared memory.  Warp 4 writes the
// ring to global memory in whole aligned 128-byte lines (16 bytes per lane, 4 rows per store instruction) while the row threads
// are busy with the next tile.  Measured on 4K YUV444PS, r = 13: with every tile's 27 results per row stored as they came
// (108 bytes at a 4-byte alignment) the stores alone took 27 of the kernel's 58 us per frame.
template <typename T, int R>
__global__ void __launch_bounds__(kHThreads) ctf_h_kernel(const CtfJob job, const __grid_constant__ CtfMaps maps) {
    using G = HTile<T, R>;
    constexpr int K = G::K, VEC = G::VEC, TS = G::TS;
    extern __shared__ __align__(128) unsigned char ctf_smem[];
    __shared__ uint64_t full[G::STAGES], consumed[G::STAGES];  // per input stage: TMA has landed / all 128 row threads have read it
    int local;
    const CtfPlane& pj = ctf_plane(job, blockIdx.y, local);
    const int plane = (int)(&pj - job.pl);
    const int rb = local % pj.cross_blocks, sg = local / pj.cross_blocks;
    const int tid = threadIdx.x, lane = tid & 31;
    const int row0 = rb * kHRows;
    const int w = pj.w, f = blockIdx.x;
    const int xs = R + sg * pj.seg_len, xe = min(xs + pj.seg_len, w - R);  // interior outputs of this piece
    const int ntiles = (xe - xs + TS - 1) / TS;                            // tile i: inputs xs+r+i*TS.., outputs xs+i*TS..
    unsigned char* in_tiles = ctf_smem;
    unsigned char* ring = ctf_smem + G::STAGES * G::TILE_BYTES;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < G::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&consumed[s], kHRows); }
        fence_mbar_init();
    }
    __syncthreads();
    // the store warp is also the TMA producer: the row threads never wait for each other, only for their data
    auto issue = [&](int i) {  // one thread
        const int s = i % G::STAGES;
        mbar_expect_tx(&full[s], (uint32_t)G::TILE_BYTES);
        tma_load_3d(in_tiles + s * G::TILE_BYTES, &maps.in[plane], (xs + R + i * TS) & ~(VEC - 1), row0, f, &full[s]);
    };

    // the ring's sample 0 is plane sample xbase: the 128-byte line that holds the piece's first output
    const int xbase = xs & ~(G::CH - 1);
    if (tid >= kHRows) {  // ---- store warp
        char* dplane = job.dst + (size_t)f * job.dst_fs + pj.dst_off + (size_t)row0 * pj.dst_pitch;
        const int rows = min(kHRows, pj.h - row0);
        const uint32_t dp = (uint32_t)pj.dst_pitch;
        const int sub = lane >> 3, vq = lane & 7;
        int chunk = 0;  // next chunk to store
        if (lane == 0)
            for (int i = 0; i < min(G::STAGES, ntiles); ++i) issue(i);
        for (int i = 0; i < ntiles; ++i) {
            const int b = i & 1;
            if (lane == 0 && i + G::STAGES < ntiles) {  // tile i has been read into registers by every row thread: refill its stage
                mbar_wait(&consumed[i % G::STAGES], (uint32_t)(i / G::STAGES) & 1u);
                issue(i + G::STAGES);
            }
            __syncwarp();
            bar_sync(BAR_FULL + b, kHThreads);
            const int done = min(xs + (i + 1) * TS, xe) - xbase;  // results [xs - xbase, done) are in the ring
            while ((chunk + 1) * G::CH <= done || (i == ntiles - 1 && chunk * G::CH < done)) {
                const int x0 = xbase + chunk * G::CH;              // first plane sample of the chunk
                const unsigned char* rc = ring + (chunk % G::RCH) * 128;
                if (x0 >= xs && x0 + G::CH <= xe) {  // whole lines: 8 lanes x 16 bytes per row, 4 rows per instruction
                    char* g = dplane + (size_t)x0 * sizeof(T) + vq * 16;
                    int rr = sub;
                    for (; rr + 12 < rows; rr += 16) {
                        uint4 v[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) v[q] = *reinterpret_cast<const uint4*>(rc + (rr + 4 * q) * G::OROW_BYTES + vq * 16);
#pragma unroll
                        for (int q = 0; q < 4; ++q) *reinterpret_cast<uint4*>(g + (size_t)((uint32_t)(rr + 4 * q) * dp)) = v[q];
                    }
                    for (; rr < rows; rr += 4)
                        *reinterpret_cast<uint4*>(g + (size_t)((uint32_t)rr * dp)) = *reinterpret_cast<const uint4*>(rc + rr * G::OROW_BYTES + vq * 16);
                } else {  // the piece's first / last line: sample by sample, inside [xs, xe) only
                    for (int c = lane; c < G::CH; c += 32) {
                        const int x = x0 + c;
                        if (x < xs || x >= xe) continue;
                        for (int rr = 0; rr < rows; ++rr)
                            reinterpret_cast<T*>(dplane + (size_t)((uint32_t)rr * dp))[x] = reinterpret_cast<const T*>(rc + rr * G::OROW_BYTES)[c];
                    }
                }
                ++chunk;
            }
            bar_arrive(BAR_EMPTY + b, kHThreads);
        }
        return;
    }

    // ---- row threads
    const int row = row0 + tid;
    const bool live = row < pj.h;
    const float div = job.div;
    const T* srow = reinterpret_cast<const T*>(job.src + (size_t)f * job.src_fs + pj.src_off + (size_t)min(row, pj.h - 1) * pj.src_pitch);
    T* drow = reinterpret_cast<T*>(job.dst + (size_t)f * job.dst_fs + pj.dst_off + (size_t)min(row, pj.h - 1) * pj.dst_pitch);
    // warm-up: the 2r samples before the first tile, straight from global memory (also the low edge's samples for piece 0)
    float acc[K][1];
#pragma unroll
    for (int s = 0; s < K; ++s) acc[s][0] = 0.f;
    {
        float pe[2 * R][1];
#pragma unroll
        for (int j = 0; j < 2 * R; ++j) pe[j][0] = __fmul_rn(div, ld1<T>(srow + xs - R + j));
        if (sg == 0 && live) edge_low_all<R, 1, 0>(pe, [&](int i, const float (&a)[1]) { drow[i] = cvt1<T>(a[0]); });
        static_for<0, 2 * R>([&](auto uc) { constexpr int U = decltype(uc)::value; push<K, 1, U>(acc, pe[U]); });
    }

    float carry[VEC - 1];
#pragma unroll
    for (int j = 0; j < VEC - 1; ++j) carry[j] = 0.f;
    for (int i = 0; i < ntiles; ++i) {
        const int s = i % G::STAGES, b = i & 1;
        mbar_wait(&full[s], (uint32_t)(i / G::STAGES) & 1u);
        float xv[TS];
        {
            float e[G::NVR * VEC];
            const uint4* q = reinterpret_cast<const uint4*>(in_tiles + s * G::TILE_BYTES + tid * G::ROW_BYTES);
#pragma unroll
            for (int v = 0; v < G::NVR; ++v) vec_to_floats<T>(q[v], e + v * VEC);
            take_phase<TS, VEC>(e, xv, (xs + R + i * TS) & (VEC - 1));
        }
        mbar_arrive(&consumed[s]);  // (the values are in registers: shared-memory reads complete before a dependent instruction issues)
        // tile step j = b*K + u is global step 2r + i*TS + j: fresh slot (u - 1) mod K, complete slot u
        static_for<0, TS>([&](auto jc) {
            constexpr int J = decltype(jc)::value, U = J % K;
            const float p[1] = {__fmul_rn(div, xv[J])};
            push<K, 1, (U + K - 1) % K>(acc, p);
            xv[J] = acc[U][0];
        });
        if (i >= 2) bar_sync(BAR_EMPTY + b, kHThreads);  // the store warp has dealt with tile i-2: the ring has room for this one
        {
            const int rel = xs + i * TS - xbase;
            ring_put<T, TS, VEC, G::RV>(xv, carry, reinterpret_cast<uint4*>(ring + tid * G::OROW_BYTES), (rel / VEC) % G::RV, rel & (VEC - 1));
        }
        bar_arrive(BAR_FULL + b, kHThreads);             // hand the tile's results to the store warp
    }

    if (sg == pj.segs - 1 && live) {  // outputs w-r..w-1 from samples w-2r..w-1
        float pe[2 * R][1];
#pragma unroll
        for (int j = 0; j < 2 * R; ++j) pe[j][0] = __fmul_rn(div, ld1<T>(srow + w - 2 * R + j));
        edge_high_all<R, 1, 0>(pe, [&](int d, const float (&a)[1]) { drow[w - 1 - d] = cvt1<T>(a[0]); });
    }
}

// --------------------------------------------------------------------------- host side
// pieces along the blurred axis: as many as it takes to give the GPU ~3 waves of CTAs, each a multiple of `quantum` long
// and at least 8 blocks of 2r+1 samples (a piece pays 2r warm-up samples)
void cut_line(int interior, int quantum, int ctas_without_cut, int sms, int& segs, int& seg_len) {
    const int want = std::max(1, (3 * 3 * sms + ctas_without_cut - 1) / std::max(1, ctas_without_cut));
    const int max_segs = std::max(1, interior / (8 * quantum));
    segs = std::min(want, max_segs);
    seg_len = ((interior + segs - 1) / segs + quantum - 1) / quantum * quantum;
    segs = (interior + seg_len - 1) / seg_len;
}

template <typename T, int R>
int launch_ctf(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* tmp, size_t tfs, char* dst, size_t dfs, int count,
               cudaStream_t st) {
    constexpr int K = 2 * R + 1, NC = Smp<T>::NC;
    using G = HTile<T, R>;
    if (!tensor_map_encoder()) return 1;
    const int sms = current_sm_count();
    if (sms < 0) return sms;
    CtfJob jv{}, jh{};
    jv.src = src; jv.src_fs = sfs; jv.dst = tmp; jv.dst_fs = tfs;
    jh.src = tmp; jh.src_fs = tfs; jh.dst = dst; jh.dst_fs = dfs;
    jv.div = jh.div = 1.0f / (float)K;
    int k = 0, base_v = 0, base_h = 0;
    for (int p = 0; p < l.nplanes; ++p) {
        if (!mask[p]) continue;
        if (l.pl[p].w < K || l.pl[p].h < K) return 1;
        CtfPlane& a = jv.pl[k];
        CtfPlane& b = jh.pl[k];
        a.src_off = a.dst_off = b.src_off = b.dst_off = l.pl[p].offset;
        a.src_pitch = a.dst_pitch = b.src_pitch = b.dst_pitch = l.pl[p].pitch;
        a.w = b.w = l.pl[p].w; a.h = b.h = l.pl[p].h;
        a.cross_blocks = (a.w + kThreads * NC - 1) / (kThreads * NC);
        b.cross_blocks = (b.h + kHRows - 1) / kHRows;
        base_v += a.cross_blocks; base_h += b.cross_blocks;
        ++k;
    }
    if (k == 0) return 0;
    jv.nplanes = jh.nplanes = k;
    int cv = 0, ch = 0;
    for (int q = 0; q < k; ++q) {
        cut_line(jv.pl[q].h - 2 * R, K, base_v * count, sms, jv.pl[q].segs, jv.pl[q].seg_len);
        cut_line(jh.pl[q].w - 2 * R, G::TS, base_h * count, sms, jh.pl[q].segs, jh.pl[q].seg_len);
        jv.pl[q].cta_begin = cv; cv += jv.pl[q].cross_blocks * jv.pl[q].segs;
        jh.pl[q].cta_begin = ch; ch += jh.pl[q].cross_blocks * jh.pl[q].segs;
    }
    jv.ctas_per_frame = cv; jh.ctas_per_frame = ch;
    VSZ_CUDA(allow_max_dynamic_smem(ctf_h_kernel<T, R>));
    for (int f0 = 0; f0 < count; f0 += 32768) {
        const int nf = std::min(32768, count - f0);
        CtfJob a = jv, b = jh;
        a.src += (size_t)f0 * sfs; a.dst += (size_t)f0 * tfs;
        b.src += (size_t)f0 * tfs; b.dst += (size_t)f0 * dfs;
        CtfMaps maps;
        for (int q = 0; q < k; ++q) {
            const CtfPlane& pl = b.pl[q];
            const int rc = encode_plane_map(&maps.in[q], sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_UINT32 : CU_TENSOR_MAP_DATA_TYPE_UINT16,
                                            b.src + pl.src_off, pl.w, pl.h, pl.src_pitch, b.src_fs, nf, G::TW, kHRows);
            if (rc) return rc;
        }
        ctf_v_kernel<T, R><<<dim3(nf, a.ctas_per_frame), kThreads, 0, st>>>(a);
        ctf_h_kernel<T, R><<<dim3(nf, b.ctas_per_frame), kHThreads, G::SMEM, st>>>(b, maps);
        count_launch(2);
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace

int run_ctf_stream(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* tmp, size_t tfs, char* dst, size_t dfs,
                   int count, int r, cudaStream_t st) {
    return with_radius(r, [&](auto radius) {
        constexpr int R = decltype(radius)::value;
        if (l.kind == K_F32) return launch_ctf<float, R>(l, mask, src, sfs, tmp, tfs, dst, dfs, count, st);
        if (l.kind == K_F16) return launch_ctf<__half, R>(l, mask, src, sfs, tmp, tfs, dst, dfs, count, st);
        return 1;
    });
}

}  // namespace vsz
