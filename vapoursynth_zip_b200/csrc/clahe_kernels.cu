// clahe_kernels.cu — sm_100a kernels of CLAHE (contrast-limited adaptive histogram equalisation), bit-exact with OpenCV's
// cv::CLAHE::apply on 8..16-bit integer planes (DESIGN.md §4.7).  Three phases per chunk of frames, each one launch over every
// (frame, processed plane):
//  A  tile histograms of the padded plane (reflect-101 at the padded edges): a CTA counts one segment of a tile (at most 65535
//     samples) in shared memory and adds its non-empty bins to the tile's u32 histogram in global memory;
//  B  one CTA per tile: clip, closed-form redistribution of the excess, exact block scan, the rounded LUT (u16);
//  C  bilinear interpolation of the four surrounding tiles' LUTs per sample: row terms once per row, column terms once per
//     column, four gathers (from shared memory when the LUTs a CTA needs fit there, else from L2), rounded store.
// A chunk holds as many frames as keep their planes, histograms and LUTs inside the L2 between A and C.
#include <algorithm>

#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "filter.h"

namespace vsz {

namespace {

constexpr int ANT = 1024;            // phase A threads: one warp per row of a segment
constexpr int ASEG_SAMPLES = 65535;  // samples per phase-A CTA: packed u16 counters cannot overflow
constexpr int ASEG_COLS = 2048;
constexpr int BNT = 1024;            // phase B threads: each scans hs / BNT consecutive bins
constexpr int CNT = 256, CVEC = 4, CROWS = 16;  // phase C: 4 adjacent samples per thread, 16 rows per CTA
constexpr int CCOLS = CNT * CVEC;
constexpr int kLutSmemCap = 64 * 1024;       // phase C gathers from shared memory when its LUTs fit in this
constexpr size_t kL2ChunkBytes = 64ull << 20;  // per chunk: planes read + written + histograms + LUTs

struct ClahePlane {
    size_t src_off, dst_off;  // bytes from the frame base (src and dst share the layout)
    size_t hist_off;          // elements from the frame's histogram / LUT base
    int pitch, w, h;
    int tw, th;               // tile size in the padded plane
    int cw, rb, segx, segy;   // phase A segments: cw columns x rb rows, segx x segy of them per tile
    int cchunks;              // phase C column chunks
    int a_begin, b_begin, c_begin;  // first blockIdx.x of this plane in phases A, B and C
    unsigned clip;            // clip limit in counts, 0: no clipping
    float lut_scale;          // f32(hs - 1) / f32(tw * th)
};

struct ClaheJob {
    const char* src;
    char* dst;
    size_t src_fs, dst_fs;
    unsigned* hist;     // [frame][plane][tile][hs]
    uint16_t* lut;      // same shape
    size_t tab_fs;      // elements per frame of hist / lut
    int nplanes, tx, ty, hs;
    ClahePlane pl[3];
};

template <int ClahePlane::*BEGIN>
__device__ __forceinline__ int plane_of(const ClaheJob& job) {
    int k = job.nplanes - 1;
    while (k > 0 && (int)blockIdx.x < job.pl[k].*BEGIN) --k;
    return k;
}

// cv::borderInterpolate(p, n, BORDER_REFLECT_101) for p >= 0
__device__ __forceinline__ int reflect101(int p, int n) {
    if (p < n) return p;
    if (n == 1) return 0;
    do {
        p = 2 * n - 2 - p;
        if (p < 0) p = -p;
    } while (p >= n);
    return p;
}

// One count for each valid lane.  A warp whose lanes all hit one bin (flat areas, blank clips) issues one atomic of n instead of
// n serialised ones, as planestats_kernels.cu's hist_add.  PACKED: two u16 counters per word (bin b in half b & 1).
template <bool PACKED>
__device__ __forceinline__ void hist_add(unsigned* h, unsigned key, bool valid) {
    const unsigned active = __ballot_sync(0xffffffffu, valid);
    if (active == 0u) return;
    const int leader = __ffs(active) - 1;
    const unsigned k0 = __shfl_sync(0xffffffffu, key, leader);
    const unsigned same = __ballot_sync(0xffffffffu, valid && key == k0);
    unsigned n = 1u;
    if (same == active) {
        if ((int)(threadIdx.x & 31) != leader) return;
        n = (unsigned)__popc(active);
    } else if (!valid) {
        return;
    }
    if (PACKED) atomicAdd(&h[key >> 1], n << ((key & 1u) * 16u));
    else atomicAdd(&h[key], n);
}

template <typename T, bool PACKED>
__global__ void __launch_bounds__(ANT) clahe_hist_kernel(const ClaheJob job) {
    extern __shared__ unsigned s_h[];
    const ClahePlane& p = job.pl[plane_of<&ClahePlane::a_begin>(job)];
    const int local = (int)blockIdx.x - p.a_begin;
    const int per_tile = p.segx * p.segy;
    const int tile = local / per_tile, seg = local % per_tile;
    const int ti = tile / job.tx, tj = tile % job.tx;
    const int x0 = tj * p.tw + (seg % p.segx) * p.cw, x1 = min(x0 + p.cw, (tj + 1) * p.tw);
    const int y0 = ti * p.th + (seg / p.segx) * p.rb, y1 = min(y0 + p.rb, (ti + 1) * p.th);
    const int words = PACKED ? job.hs / 2 : job.hs;
    for (int i = threadIdx.x; i < words; i += ANT) s_h[i] = 0u;
    __syncthreads();
    const char* src = job.src + (size_t)blockIdx.y * job.src_fs + p.src_off;
    const unsigned top = (unsigned)job.hs - 1u;
    const int lane = threadIdx.x & 31;
    for (int y = y0 + (int)(threadIdx.x >> 5); y < y1; y += ANT / 32) {
        const T* row = reinterpret_cast<const T*>(src + (size_t)reflect101(y, p.h) * p.pitch);
        for (int xb = x0; xb < x1; xb += 32) {
            const int x = xb + lane;
            const bool valid = x < x1;
            const unsigned v = valid ? min((unsigned)row[reflect101(x, p.w)], top) : 0u;
            hist_add<PACKED>(s_h, v, valid);
        }
    }
    __syncthreads();
    unsigned* gh = job.hist + (size_t)blockIdx.y * job.tab_fs + p.hist_off + (size_t)tile * job.hs;
    for (int i = threadIdx.x; i < words; i += ANT) {
        const unsigned c = s_h[i];
        if (PACKED) {
            if (c & 0xffffu) atomicAdd(&gh[2 * i], c & 0xffffu);
            if (c >> 16) atomicAdd(&gh[2 * i + 1], c >> 16);
        } else if (c) {
            atomicAdd(&gh[i], c);
        }
    }
}

// One tile: clipped histogram -> exact inclusive scan -> LUT.  Thread t owns bins [t * per, (t + 1) * per).
__global__ void __launch_bounds__(BNT) clahe_lut_kernel(const ClaheJob job) {
    using Reduce = cub::BlockReduce<unsigned long long, BNT>;
    using Scan = cub::BlockScan<unsigned, BNT>;
    __shared__ union { typename Reduce::TempStorage r; typename Scan::TempStorage s; } tmp;
    __shared__ unsigned long long s_clipped;
    const ClahePlane& p = job.pl[plane_of<&ClahePlane::b_begin>(job)];
    const int tile = (int)blockIdx.x - p.b_begin;
    const int hs = job.hs;
    const size_t base = (size_t)blockIdx.y * job.tab_fs + p.hist_off + (size_t)tile * hs;
    const unsigned* gh = job.hist + base;
    uint16_t* lut = job.lut + base;
    const int per = (hs + BNT - 1) / BNT;
    const int i0 = min((int)threadIdx.x * per, hs), i1 = min(i0 + per, hs);
    const unsigned c = p.clip;
    unsigned long long excess = 0;
    if (c)
        for (int i = i0; i < i1; ++i) excess += gh[i] > c ? gh[i] - c : 0u;
    const unsigned long long clipped_all = Reduce(tmp.r).Sum(excess);
    if (threadIdx.x == 0) s_clipped = clipped_all;
    __syncthreads();
    // every bin gets clipped / hs; the remainder res goes one count each to bins 0, step, 2 step, ... (res of them)
    const unsigned long long clipped = s_clipped;
    const unsigned batch = (unsigned)(clipped / (unsigned)hs);
    const int res = (int)(clipped % (unsigned)hs);
    const int step = res ? max(hs / res, 1) : 1;
    auto value = [&](int i) -> unsigned {
        unsigned h = gh[i];
        if (c) h = min(h, c) + batch + ((res && i % step == 0 && i / step < res) ? 1u : 0u);
        return h;
    };
    unsigned sum = 0;
    for (int i = i0; i < i1; ++i) sum += value(i);
    unsigned cdf;
    Scan(tmp.s).ExclusiveSum(sum, cdf);
    const int top = hs - 1;
    for (int i = i0; i < i1; ++i) {
        cdf += value(i);
        const int v = __float2int_rn(__fmul_rn(__uint2float_rn(cdf), p.lut_scale));
        lut[i] = (uint16_t)min(max(v, 0), top);
    }
}

// Tile coordinate of position x along an axis of n tiles of size t (inv = f32(1 / t)): the two tiles and the weight of the second.
__device__ __forceinline__ void tile_pos(int x, float inv, int n, int& t1, int& t2, float& a) {
    const float f = __fsub_rn(__fmul_rn((float)x, inv), 0.5f);
    const int i = (int)floorf(f);
    a = __fsub_rn(f, (float)i);
    t1 = max(i, 0);
    t2 = min(i + 1, n - 1);
}

template <typename T> struct Vec4;
template <> struct Vec4<uint8_t> { using type = uint32_t; };
template <> struct Vec4<uint16_t> { using type = uint2; };

template <typename T>
__global__ void __launch_bounds__(CNT) clahe_apply_kernel(const ClaheJob job, int smem_bytes) {
    extern __shared__ __align__(16) uint16_t s_lut[];
    const ClahePlane& p = job.pl[plane_of<&ClahePlane::c_begin>(job)];
    const int local = (int)blockIdx.x - p.c_begin;
    const int y0 = (local / p.cchunks) * CROWS, y1 = min(y0 + CROWS, p.h);
    const int xc0 = (local % p.cchunks) * CCOLS, xc1 = min(xc0 + CCOLS, p.w);
    const int hs = job.hs;
    const float inv_tw = __fdiv_rn(1.0f, (float)p.tw), inv_th = __fdiv_rn(1.0f, (float)p.th);
    // the tiles this CTA reads: positions are monotone in x and y, so the corners bound them
    int c_lo, c_hi, r_lo, r_hi, dummy;
    float fd;
    tile_pos(xc0, inv_tw, job.tx, c_lo, dummy, fd);
    tile_pos(xc1 - 1, inv_tw, job.tx, dummy, c_hi, fd);
    tile_pos(y0, inv_th, job.ty, r_lo, dummy, fd);
    tile_pos(y1 - 1, inv_th, job.ty, dummy, r_hi, fd);
    const int ncols = c_hi - c_lo + 1, nrows = r_hi - r_lo + 1;
    const uint16_t* glut = job.lut + (size_t)blockIdx.y * job.tab_fs + p.hist_off;
    const uint16_t* base;  // LUT of tile (r_lo, c_lo); tile (r, c) is at base + (r - r_lo) * rstride + (c - c_lo) * hs
    size_t rstride;
    if ((size_t)nrows * ncols * hs * sizeof(uint16_t) <= (size_t)smem_bytes) {
        const int per_tile = hs / 8;  // 16-byte vectors
        const int nvec = nrows * ncols * per_tile;
        for (int v = threadIdx.x; v < nvec; v += CNT) {
            const int t = v / per_tile, e = v % per_tile;
            const int r = r_lo + t / ncols, c = c_lo + t % ncols;
            reinterpret_cast<uint4*>(s_lut)[v] = reinterpret_cast<const uint4*>(glut + ((size_t)r * job.tx + c) * hs)[e];
        }
        __syncthreads();
        base = s_lut;
        rstride = (size_t)ncols * hs;
    } else {
        base = glut + ((size_t)r_lo * job.tx + c_lo) * hs;
        rstride = (size_t)job.tx * hs;
    }
    const int xt = xc0 + (int)threadIdx.x * CVEC;
    if (xt >= xc1) return;
    int o1[CVEC], o2[CVEC];
    float xa[CVEC], xa1[CVEC];
#pragma unroll
    for (int e = 0; e < CVEC; ++e) {
        // a lane past the plane's last column (not stored) takes that column's tiles: its own could lie past the last tile
        int t1, t2;
        tile_pos(min(xt + e, xc1 - 1), inv_tw, job.tx, t1, t2, xa[e]);
        xa1[e] = __fsub_rn(1.0f, xa[e]);
        o1[e] = (t1 - c_lo) * hs;
        o2[e] = (t2 - c_lo) * hs;
    }
    const bool full = xt + CVEC <= xc1;
    const unsigned top = (unsigned)hs - 1u;
    const char* src = job.src + (size_t)blockIdx.y * job.src_fs + p.src_off;
    char* dst = job.dst + (size_t)blockIdx.y * job.dst_fs + p.dst_off;
    using V = typename Vec4<T>::type;
    for (int y = y0; y < y1; ++y) {
        int r1, r2;
        float ya;
        tile_pos(y, inv_th, job.ty, r1, r2, ya);
        const float ya1 = __fsub_rn(1.0f, ya);
        const uint16_t* l1 = base + (size_t)(r1 - r_lo) * rstride;
        const uint16_t* l2 = base + (size_t)(r2 - r_lo) * rstride;
        // a vector read stays inside the row's pitch: x is a multiple of 4 and the pitch a multiple of 128 bytes
        union { V v; T s[CVEC]; } in, out;
        in.v = *reinterpret_cast<const V*>(src + (size_t)y * p.pitch + (size_t)xt * sizeof(T));
#pragma unroll
        for (int e = 0; e < CVEC; ++e) {
            const unsigned s = min((unsigned)in.s[e], top);
            const float a = (float)l1[o1[e] + s], b = (float)l1[o2[e] + s];
            const float c = (float)l2[o1[e] + s], d = (float)l2[o2[e] + s];
            const float t0 = __fadd_rn(__fmul_rn(a, xa1[e]), __fmul_rn(b, xa[e]));
            const float t1 = __fadd_rn(__fmul_rn(c, xa1[e]), __fmul_rn(d, xa[e]));
            const int v = __float2int_rn(__fadd_rn(__fmul_rn(t0, ya1), __fmul_rn(t1, ya)));
            out.s[e] = (T)min(max(v, 0), (int)top);
        }
        T* drow = reinterpret_cast<T*>(dst + (size_t)y * p.pitch);
        if (full) {
            *reinterpret_cast<V*>(drow + xt) = out.v;
        } else {
#pragma unroll
            for (int e = 0; e < CVEC; ++e)
                if (xt + e < xc1) drow[xt + e] = out.s[e];
        }
    }
}

template <typename T>
int launch_clahe_t(const ClaheJob& job0, int a_ctas, int b_ctas, int c_ctas, int c_smem, int count, int chunk, unsigned* hist,
                   uint16_t* lut, cudaStream_t st) {
    const bool packed = job0.hs > 4096;
    const int a_smem = packed ? job0.hs * 2 : job0.hs * 4;
    auto ka = packed ? clahe_hist_kernel<T, true> : clahe_hist_kernel<T, false>;
    VSZ_CUDA(allow_max_dynamic_smem(ka));
    VSZ_CUDA(allow_max_dynamic_smem(clahe_apply_kernel<T>));
    for (int f0 = 0; f0 < count; f0 += chunk) {
        const int nf = std::min(chunk, count - f0);
        ClaheJob j = job0;
        j.src += (size_t)f0 * job0.src_fs;
        j.dst += (size_t)f0 * job0.dst_fs;
        j.hist = hist;
        j.lut = lut;
        VSZ_CUDA(cudaMemsetAsync(hist, 0, (size_t)nf * job0.tab_fs * sizeof(unsigned), st));
        ka<<<dim3(a_ctas, nf), ANT, a_smem, st>>>(j);
        clahe_lut_kernel<<<dim3(b_ctas, nf), BNT, 0, st>>>(j);
        clahe_apply_kernel<T><<<dim3(c_ctas, nf), CNT, c_smem, st>>>(j, c_smem);
        count_launch(3);
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace

int run_clahe(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs, int count, int hs,
              double limit, int tx, int ty, cudaStream_t st) {
    if (count <= 0) return 0;
    if (l.kind != K_U8 && l.kind != K_U16) return -1;
    ClaheJob job{};
    job.src = src; job.dst = dst; job.src_fs = src_fs; job.dst_fs = dst_fs;
    job.tx = tx; job.ty = ty; job.hs = hs;
    int a = 0, b = 0, c = 0, c_smem = 0;
    size_t tab = 0;
    for (int pi = 0; pi < l.nplanes; ++pi) {
        if (!mask[pi]) continue;
        ClahePlane& p = job.pl[job.nplanes++];
        const PlaneGeom& g = l.pl[pi];
        p.src_off = p.dst_off = g.offset;
        p.pitch = g.pitch; p.w = g.w; p.h = g.h;
        // OpenCV pads both axes (by a whole tile on an axis that divides) as soon as one of them does not divide
        const bool pad = g.w % tx != 0 || g.h % ty != 0;
        const int pw = pad ? g.w + tx - g.w % tx : g.w, ph = pad ? g.h + ty - g.h % ty : g.h;
        p.tw = pw / tx; p.th = ph / ty;
        const double n = (double)p.tw * (double)p.th;
        if (limit > 0) {
            const double cl = limit * n / (double)hs;
            p.clip = cl >= 2147483647.0 ? 2147483647u : (unsigned)std::max((int)cl, 1);
        }
        p.lut_scale = (float)(hs - 1) / (float)(p.tw * p.th);
        p.cw = std::min(p.tw, ASEG_COLS);
        p.rb = std::max(1, std::min(p.th, ASEG_SAMPLES / p.cw));
        p.segx = (p.tw + p.cw - 1) / p.cw;
        p.segy = (p.th + p.rb - 1) / p.rb;
        p.cchunks = (g.w + CCOLS - 1) / CCOLS;
        p.a_begin = a; a += tx * ty * p.segx * p.segy;
        p.b_begin = b; b += tx * ty;
        p.c_begin = c; c += p.cchunks * ((g.h + CROWS - 1) / CROWS);
        p.hist_off = tab;
        tab += (size_t)tx * ty * hs;
        if (hs <= 4096) {  // the most LUTs one phase-C CTA can need: the tiles its columns and rows reach
            const int nc = std::min(tx, (std::min(CCOLS, g.w) + p.tw - 1) / p.tw + 2);
            const int nr = std::min(ty, (std::min(CROWS, g.h) + p.th - 1) / p.th + 2);
            c_smem = std::max(c_smem, std::min(nc * nr * hs * (int)sizeof(uint16_t), kLutSmemCap));
        }
    }
    if (job.nplanes == 0) return 0;
    job.tab_fs = (tab + 127) & ~(size_t)127;  // keeps every frame's tables 512-byte aligned
    const size_t tab_bytes = job.tab_fs * (sizeof(unsigned) + sizeof(uint16_t));
    const size_t per_frame = 2 * layout_algorithmic_bytes(l) + tab_bytes;
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>({kL2ChunkBytes / per_frame, (size_t)count, 65535}));
    AsyncScratch mem;
    VSZ_CUDA(mem.alloc((size_t)chunk * tab_bytes, st));
    unsigned* hist = reinterpret_cast<unsigned*>(mem.p);
    uint16_t* lut = reinterpret_cast<uint16_t*>(mem.p + (size_t)chunk * job.tab_fs * sizeof(unsigned));
    if (l.kind == K_U8) return launch_clahe_t<uint8_t>(job, a, b, c, c_smem, count, chunk, hist, lut, st);
    return launch_clahe_t<uint16_t>(job, a, b, c, c_smem, count, chunk, hist, lut, st);
}

}  // namespace vsz
