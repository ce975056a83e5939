// boxblur_seg_v.cu — vseg_kernel: vertical passes on 64-column strips (see boxblur_seg.cuh for the design of the segment kernels).
#include "boxblur_seg.cuh"
#include "boxblur_tma.h"

namespace vsz {

namespace {

// =========================================================================== V
// LV = rows per thread.  90 rows x 12 warps (1080 rows) leave 168 registers per thread; the general 60-row variant runs
// up to 18 warps, which the register file only grants 96 registers each (allocation is per 4 warps).
template <int LV> struct VSegShape;
template <> struct VSegShape<90> { static constexpr int MAX_WARPS = 12; };
template <> struct VSegShape<60> { static constexpr int MAX_WARPS = 18; };

// U8 (both V kernels): a lane's pair of columns is two BYTES per row; they are widened into the packed 16-bit word on the way in
// and narrowed on the way out, the passes in between are the 16-bit kernel.
__device__ __forceinline__ uint32_t widen2(uint32_t b2) { return __byte_perm(b2, 0u, 0x4140); }    // bytes 0,1 -> halves
__device__ __forceinline__ uint16_t narrow2(uint32_t w) { return (uint16_t)__byte_perm(w, 0u, 0x4420); }  // low bytes of both halves
template <bool U8> __device__ __forceinline__ uint32_t ld_pair(const char* p) {
    if constexpr (U8) return widen2(*reinterpret_cast<const uint16_t*>(p));
    else return *reinterpret_cast<const uint32_t*>(p);
}
template <bool U8> __device__ __forceinline__ void st_pair(char* p, uint32_t w) {
    if constexpr (U8) *reinterpret_cast<uint16_t*>(p) = narrow2(w);
    else *reinterpret_cast<uint32_t*>(p) = w;
}

template <int R, int LV, bool U8>
__global__ void __launch_bounds__(VSegShape<LV>::MAX_WARPS * 32, 1) vseg_kernel(const SegJob job) {
    using Gm = VGeom<R, LV>;
    extern __shared__ __align__(128) unsigned char seg_smem[];
    uint32_t* tile = reinterpret_cast<uint32_t*>(seg_smem);  // row y of the strip at tile[(R + y) * 32 + lane]
    const int s = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    int local;
    const SegPlane& pj = seg_plane(job, blockIdx.y, local);
    const int S = pj.S, n = pj.h;
    uint32_t* cbuf = tile + (size_t)(R + LV * S + R + 1) * 32;  // [2][32] line constants
    const int cw = local * 32 + lane;                           // pair of columns
    const bool colok = cw * 2 < pj.w;
    const bool segok = s < S;
    const bool exact = (n % LV) == 0;
    const char* src = job.src + (size_t)blockIdx.x * job.src_fs + pj.src_off + (size_t)cw * (U8 ? 2 : 4);
    char* dst = job.dst + (size_t)blockIdx.x * job.dst_fs + pj.dst_off + (size_t)cw * (U8 ? 2 : 4);

    uint32_t e[Gm::NW];
#pragma unroll
    for (int i = 0; i < Gm::NW; ++i) e[i] = 0u;
    if (colok && segok) {
        const int y0 = LV * s;
        if (y0 + LV <= n) {
#pragma unroll
            for (int i = 0; i < LV; ++i) e[R + i] = ld_pair<U8>(src + (size_t)(y0 + i) * pj.src_pitch);
        } else {
#pragma unroll
            for (int i = 0; i < LV; ++i) e[R + i] = ld_pair<U8>(src + (size_t)min(y0 + i, n - 1) * pj.src_pitch);
        }
    }
    for (int p = 0; p < job.passes; ++p) {
        if (s == 0) {  // the line constants of this pass, from rows 0..r of the pass input
            uint32_t Wl, Wh;
            v_window0<R, LV>(e, Wl, Wh);
            cbuf[lane] = line_const(Wl, job.inv, job.inv2);
            cbuf[32 + lane] = line_const(Wh, job.inv, job.inv2);
        }
        if (segok) {
            uint32_t* t = tile + (size_t)(R + LV * s) * 32 + lane;
            if (exact) {
#pragma unroll
                for (int j = 0; j < R; ++j) { t[j * 32] = e[R + j]; t[(LV - R + j) * 32] = e[R + LV - R + j]; }
            } else {
#pragma unroll
                for (int i = 0; i < LV; ++i) t[i * 32] = e[R + i];
            }
        }
        __syncthreads();
        if (!exact) {  // SYM mirror rows either side of the strip
            for (int k = s; k < R; k += nwarps) {
                tile[(R - 1 - k) * 32 + lane] = tile[(R + k) * 32 + lane];
                tile[(R + n + k) * 32 + lane] = tile[(R + n - 1 - k) * 32 + lane];
            }
            __syncthreads();
        }
        if (segok) {
            const uint32_t* t = tile + (size_t)(LV * s) * 32 + lane;  // row LV*s - R
            if (exact && s == 0) {
#pragma unroll
                for (int k = 0; k < R; ++k) e[R - 1 - k] = e[R + k];
            } else {
#pragma unroll
                for (int j = 0; j < R; ++j) e[j] = t[j * 32];
            }
            if (exact && s == S - 1) {
#pragma unroll
                for (int k = 0; k < R; ++k) e[R + LV + k] = e[R + LV - 1 - k];
            } else {
#pragma unroll
                for (int j = 0; j < R; ++j) e[R + LV + j] = t[(R + LV + j) * 32];
            }
            if (!exact && s == S - 1) {
#pragma unroll
                for (int i = 0; i < LV; ++i) e[R + i] = t[(R + i) * 32];
            }
            const uint32_t Cl = cbuf[lane], Ch = cbuf[32 + lane];
            uint32_t Wl, Wh;
            v_window<R, LV>(e, Wl, Wh);
            uint32_t out[LV];
            v_slide<R, LV, kAllDp>(e, out, Wl, Wh, Cl, Ch, job.inv2);
#pragma unroll
            for (int i = 0; i < LV; ++i) e[R + i] = out[i];
        }
        __syncthreads();  // halos and constants consumed: the tile may be overwritten
    }
    if (colok && segok) {
        const int y0 = LV * s;
        if (y0 + LV <= n) {
#pragma unroll
            for (int i = 0; i < LV; ++i) st_pair<U8>(dst + (size_t)(y0 + i) * pj.dst_pitch, e[R + i]);
        } else {
#pragma unroll
            for (int i = 0; i < LV; ++i)
                if (y0 + i < n) st_pair<U8>(dst + (size_t)(y0 + i) * pj.dst_pitch, e[R + i]);
        }
    }
}

// --------------------------------------------------------------------------- V, plane heights that are multiples of 90 rows
// (1080, 540, 720, ...): persistent CTAs.  A CTA walks over 64-column strips; the strip's [rows x 128 bytes] tile is brought
// into shared memory by the TMA engine (cp.async.bulk.tensor.3d, one 90-row box per warp, mbarrier completion) while the
// previous strip is being blurred, each thread copies its 90 words into registers with immediate-offset LDS, and per pass only
// the first and last r rows of every segment go through (double-buffered) shared memory: one __syncthreads per pass.
constexpr int LVT = 90;
struct VTiles { CUtensorMap map[3]; };

__device__ __forceinline__ void tma_load_3d(void* sdst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                     smem_u32(sdst)),
                 "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
                 : "memory");
}

template <int R, bool U8>
__global__ void __launch_bounds__(VSegShape<LVT>::MAX_WARPS * 32, 1)
    vseg_tile_kernel(const SegJob job, const __grid_constant__ VTiles tiles, int strips, int nitems) {
    using Gm = VGeom<R, LVT>;
    extern __shared__ __align__(128) unsigned char seg_smem[];
    __shared__ uint64_t tile_bar;
    const int s = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int S = blockDim.x >> 5;
    constexpr int ROWB = U8 ? 64 : 128;                              // bytes of a tile row: 64 columns
    unsigned char* tile = seg_smem;                                  // [S * 90 rows][64 columns]
    uint32_t* halo = reinterpret_cast<uint32_t*>(seg_smem + (size_t)S * LVT * ROWB);  // [2][S][2r][32]: first r and last r rows of every segment
    uint32_t* cbuf = halo + (size_t)2 * S * 2 * R * 32;              // [2][2][32] line constants
    const uint32_t tile_bytes = (uint32_t)S * LVT * ROWB;

    if (threadIdx.x == 0) {
        mbar_init(&tile_bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto issue = [&](int item) {  // thread 0: one box per warp segment
        const int strip = item % strips, k = (item / strips) % job.nplanes, f = item / (strips * job.nplanes);
        mbar_expect_tx(&tile_bar, tile_bytes);
        for (int q = 0; q < S; ++q) tma_load_3d(tile + (size_t)q * LVT * ROWB, &tiles.map[k], strip * 64, q * LVT, f, &tile_bar);
    };
    if (threadIdx.x == 0 && (int)blockIdx.x < nitems) issue(blockIdx.x);

    uint32_t ea[Gm::NW], eb[Gm::NW];  // pass input / output, swapping roles every pass (no register copies)
    int hb = 0;
    uint32_t phase = 0;
    // one pass: in[] own rows -> halo exchange -> emit(i, word) for the 90 rows of the segment
    auto pass = [&](uint32_t (&in)[Gm::NW], auto emit) {
        uint32_t* hw = halo + (size_t)(hb * S + s) * (2 * R * 32) + lane;
        if (s == 0) {  // the line constants of this pass, from rows 0..r of the pass input
            uint32_t Wl, Wh;
            v_window0<R, LVT>(in, Wl, Wh);
            cbuf[hb * 64 + lane] = line_const(Wl, job.inv, job.inv2);
            cbuf[hb * 64 + 32 + lane] = line_const(Wh, job.inv, job.inv2);
        }
#pragma unroll
        for (int j = 0; j < R; ++j) { hw[j * 32] = in[R + j]; hw[(R + j) * 32] = in[R + LVT - R + j]; }
        __syncthreads();
        if (s == 0) {
#pragma unroll
            for (int j = 0; j < R; ++j) in[R - 1 - j] = in[R + j];                      // SYM mirror above row 0
        } else {
            const uint32_t* hr = hw - 2 * R * 32 + R * 32;                               // last r rows of the segment above
#pragma unroll
            for (int j = 0; j < R; ++j) in[j] = hr[j * 32];
        }
        if (s == S - 1) {
#pragma unroll
            for (int j = 0; j < R; ++j) in[R + LVT + j] = in[R + LVT - 1 - j];          // SYM mirror below the last row
        } else {
            const uint32_t* hr = hw + 2 * R * 32;                                        // first r rows of the segment below
#pragma unroll
            for (int j = 0; j < R; ++j) in[R + LVT + j] = hr[j * 32];
        }
        const uint32_t Cl = cbuf[hb * 64 + lane], Ch = cbuf[hb * 64 + 32 + lane];
        uint32_t Wl, Wh;
        v_window<R, LVT>(in, Wl, Wh);
        v_slide_emit<R, LVT, kAllDp>(in, Wl, Wh, Cl, Ch, job.inv2, emit);
        hb ^= 1;
    };
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int strip = item % strips, k = (item / strips) % job.nplanes, f = item / (strips * job.nplanes);
        const SegPlane& pj = job.pl[k];
        const int cw = strip * 32 + lane;
        mbar_wait(&tile_bar, phase);
        phase ^= 1u;
        {
            if constexpr (U8) {
                const uint16_t* t = reinterpret_cast<const uint16_t*>(tile + (size_t)s * LVT * ROWB) + lane;
#pragma unroll
                for (int i = 0; i < LVT; ++i) ea[R + i] = widen2(t[i * 32]);
            } else {
                const uint32_t* t = reinterpret_cast<const uint32_t*>(tile + (size_t)s * LVT * ROWB) + lane;
#pragma unroll
                for (int i = 0; i < LVT; ++i) ea[R + i] = t[i * 32];
            }
        }
        __syncthreads();  // the tile is in registers
        if (threadIdx.x == 0 && item + (int)gridDim.x < nitems) {
            fence_proxy_async();
            issue(item + gridDim.x);
        }
        // Every call site has fixed roles for the two register arrays, so at most one and a bit of them is live at any time.
        // In the last pass the results leave for global memory as they are produced (idle columns of the last strip write nowhere).
        char* const q = job.dst + (size_t)f * job.dst_fs + pj.dst_off + (size_t)(s * LVT) * pj.dst_pitch + (size_t)cw * (U8 ? 2 : 4);
        const uint32_t dp = (uint32_t)pj.dst_pitch;
        auto store = [&](int i, uint32_t v) { st_pair<U8>(q + (size_t)((uint32_t)i * dp), v); };  // strips are whole (w % 64 == 0)
        auto to_a = [&](int i, uint32_t v) { ea[R + i] = v; };
        auto to_b = [&](int i, uint32_t v) { eb[R + i] = v; };
        int left = job.passes;
        for (; left > 2; left -= 2) {
            pass(ea, to_b);
            pass(eb, to_a);
        }
        if (left == 2) {
            pass(ea, to_b);
            pass(eb, store);
        } else {
            pass(ea, store);
        }
    }
}

template <int R, bool U8> size_t vseg_tile_smem(int S) { return (size_t)S * LVT * (U8 ? 64 : 128) + ((size_t)2 * S * 2 * R * 32 + 128) * 4; }

// Whether the tile kernel can run planes of height h (S = h / 90 warps): 0 = yes, with `resident` CTAs on the GPU at once;
// 1 = no (no tensor-map encoder in this driver, too much shared memory or no resident CTA); < 0 = error
template <int R, bool U8>
int vseg_tile_fit(int h, int& resident) {
    if (!tensor_map_encoder()) return 1;
    const int S = h / LVT;
    const size_t smem = vseg_tile_smem<R, U8>(S);
    if (smem > (size_t)kMaxSmemPerCta) return 1;
    auto kern = vseg_tile_kernel<R, U8>;
    VSZ_CUDA(allow_max_dynamic_smem(kern));
    const int sms = current_sm_count();
    if (sms < 0) return sms;
    int per_sm = 1;
    VSZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, S * 32, smem));
    if (per_sm < 1) return 1;
    resident = sms * per_sm;
    return 0;
}

template <int R, bool U8>
int launch_vseg_tile(const SegJob& job, int count, int resident, cudaStream_t st) {
    const int S = job.pl[0].h / LVT, strips = ((job.pl[0].w + 1) / 2 + 31) / 32;
    for (int f0 = 0; f0 < count; f0 += 32768) {
        const int nf = std::min(32768, count - f0);
        SegJob j = job;
        j.src += (size_t)f0 * job.src_fs; j.dst += (size_t)f0 * job.dst_fs;
        VTiles tiles;
        for (int k = 0; k < j.nplanes; ++k) {
            const SegPlane& pl = j.pl[k];
            const int rc = encode_plane_map(&tiles.map[k], U8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_UINT16, j.src + pl.src_off,
                                            pl.w, pl.h, pl.src_pitch, j.src_fs, nf, 64, LVT);
            if (rc) return rc;
        }
        const int nitems = nf * j.nplanes * strips;
        vseg_tile_kernel<R, U8><<<std::min(nitems, resident), S * 32, vseg_tile_smem<R, U8>(S), st>>>(j, tiles, strips, nitems);
        count_launch();
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

template <int LV> bool vseg_fits(int h) { return (h + LV - 1) / LV <= VSegShape<LV>::MAX_WARPS; }
inline bool vseg_long(int w, int h) { return h % 90 == 0 && vseg_fits<90>(h) && w % 64 == 0; }  // whole strips, whole segments

template <int R, int LV, bool U8>
int launch_vseg_shape(SegJob job, int count, cudaStream_t st) {
    int cta = 0;
    const int S = (job.pl[0].h + LV - 1) / LV;
    for (int k = 0; k < job.nplanes; ++k) {
        SegPlane& s = job.pl[k];
        s.S = S;
        s.cta_begin = cta;
        cta += ((s.w + 1) / 2 + 31) / 32;
    }
    job.ctas_per_frame = cta;
    const size_t smem = ((size_t)(R + LV * S + R + 1) * 32 + 64) * 4;
    return launch_frames(vseg_kernel<R, LV, U8>, job, count, S * 32, smem, st);
}

// Every shape group's kernel (tile or plain) is settled before the first launch, so that 1 means nothing was launched.
template <int R, bool U8>
int launch_vseg(const SegJob& whole, int count, cudaStream_t st) {
    for (int k = 0; k < whole.nplanes; ++k)
        if (!vseg_long(whole.pl[k].w, whole.pl[k].h) && !vseg_fits<60>(whole.pl[k].h)) return 1;
    SegJob groups[3];
    const int ngroups = shape_groups(whole, groups);
    int resident[3] = {0, 0, 0};  // tile kernel: resident CTAs; 0 = plain kernel
    for (int g = 0; g < ngroups; ++g) {
        const SegPlane& p = groups[g].pl[0];
        if (!vseg_long(p.w, p.h)) continue;
        const int rc = vseg_tile_fit<R, U8>(p.h, resident[g]);
        if (rc) return rc;
    }
    for (int g = 0; g < ngroups; ++g) {
        const int rc = resident[g] ? launch_vseg_tile<R, U8>(groups[g], count, resident[g], st) : launch_vseg_shape<R, 60, U8>(groups[g], count, st);
        if (rc) return rc;
    }
    return 0;
}

}  // namespace

int run_seg_v(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int count, int r, int passes,
              cudaStream_t st) {
    if ((l.kind != K_U16 && l.kind != K_U8) || passes < 1) return 1;
    const SegJob job = base_job(l, mask, src, sfs, dst, dfs, r, passes);
    const bool u8 = l.kind == K_U8;
    return with_radius(r, [&](auto radius) {
        constexpr int R = decltype(radius)::value;
        return u8 ? launch_vseg<R, true>(job, count, st) : launch_vseg<R, false>(job, count, st);
    });
}

}  // namespace vsz
