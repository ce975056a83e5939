// boxblur_seg_ct.cu — ctfused_kernel: the comptime path in one read and one write (see boxblur_seg.cuh for the design of the segment kernels).
#include <type_traits>

#include "boxblur_seg.cuh"

namespace vsz {

namespace {

// =========================================================================== comptime path, fused
constexpr int CTF_WARPS = 8;

// CPT consecutive samples of a row as CPT / 2 packed 16-bit words; 8-bit rows are widened on the way in
// (`PRMT`), so that everything after the load is the 16-bit code.
template <int CPT, bool U8>
__device__ __forceinline__ void load_cols(const void* p, uint32_t (&w)[CPT / 2]) {
    if constexpr (!U8) {
        if constexpr (CPT == 8) { const uint4 v = *reinterpret_cast<const uint4*>(p); w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w; }
        else { const uint2 v = *reinterpret_cast<const uint2*>(p); w[0] = v.x; w[1] = v.y; }
    } else {
        if constexpr (CPT == 8) {
            const uint2 v = *reinterpret_cast<const uint2*>(p);
            w[0] = __byte_perm(v.x, 0u, 0x4140); w[1] = __byte_perm(v.x, 0u, 0x4342);
            w[2] = __byte_perm(v.y, 0u, 0x4140); w[3] = __byte_perm(v.y, 0u, 0x4342);
        } else {
            const uint32_t v = *reinterpret_cast<const uint32_t*>(p);
            w[0] = __byte_perm(v, 0u, 0x4140); w[1] = __byte_perm(v, 0u, 0x4342);
        }
    }
}

template <int R, int CPT, bool U8, int NWARPS = CTF_WARPS>
__global__ void __launch_bounds__(NWARPS * 32, NWARPS == 4 ? 4 : 2) ctfused_kernel(const SegJob job) {
    using Gm = HGeom<R>;
    using CV = typename std::conditional<CPT == 8, uint4, uint2>::type;  // CPT 16-bit means
    constexpr int CW = CPT / 2, BPS = U8 ? 1 : 2;
    extern __shared__ __align__(128) unsigned char seg_smem[];
    __shared__ uint64_t ring_bar;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int local;
    const SegPlane& pj = seg_plane(job, blockIdx.y, local);
    const int G = pj.G, RPW = 32 / G, sub = lane / G, sg0 = lane % G;
    const int GR = NWARPS * RPW;  // rows per group
    const bool act = sg0 < pj.S;
    const int sg = act ? sg0 : 0;
    const int w = pj.w, h = pj.h;
    const int y0 = local * pj.per_cta, y1 = min(y0 + pj.per_cta, h);
    const uint32_t row_bytes = (uint32_t)((w * BPS + 15) & ~15);
    unsigned char* ring = seg_smem;                                  // [2*GR][row_bytes]: rows entering (0..GR-1) and leaving (GR..) the window
    unsigned char* tmpb = seg_smem + (size_t)2 * GR * row_bytes;     // [GR][rowbuf]: rounded column means, then the finished rows
    const char* src = job.src + (size_t)blockIdx.x * job.src_fs + pj.src_off;
    char* dst = job.dst + (size_t)blockIdx.x * job.dst_fs + pj.dst_off;
    const int c0 = threadIdx.x * CPT;
    const bool vact = c0 < w;

    if (threadIdx.x == 0) {
        mbar_init(&ring_bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    // A row enters the window once and leaves it 2r+1 rows later: it is fetched from HBM the first time and kept in L2
    // (evict_last) until the second, last read (evict_first); finished rows are written evict_first as well, so that the
    // windows of all resident CTAs (~30 MB) are what stays in L2.
    const uint64_t keep = l2_evict_last(), drop = l2_evict_first();
    auto issue_ring = [&](int yg) {  // thread 0
        mbar_expect_tx(&ring_bar, (uint32_t)(2 * GR) * row_bytes);
        for (int j = 0; j < GR; ++j) {
            const int y = min(yg + j, h - 1);
            bulk_g2s_hint(ring + (size_t)j * row_bytes, src + (size_t)ct_add_row(y, R, h) * pj.src_pitch, row_bytes, &ring_bar, keep);
            bulk_g2s_hint(ring + (size_t)(GR + j) * row_bytes, src + (size_t)ct_sub_row(y, R) * pj.src_pitch, row_bytes, &ring_bar, drop);
        }
    };
    if (threadIdx.x == 0) issue_ring(y0);

    // exact column sums of row y0: the 2r+1 R101q taps, straight from global memory
    uint32_t col[CPT];
#pragma unroll
    for (int k = 0; k < CPT; ++k) col[k] = 0u;
    if (vact) {
        constexpr int NB = 9;
        for (int k0 = 0; k0 <= 2 * R; k0 += NB) {
            uint32_t v[NB][CW];
#pragma unroll
            for (int u = 0; u < NB; ++u) {
                const int k = min(k0 + u, 2 * R);
                load_cols<CPT, U8>(src + (size_t)ct_tap_row(y0, k, R, h) * pj.src_pitch + (size_t)c0 * BPS, v[u]);
            }
#pragma unroll
            for (int u = 0; u < NB; ++u) {
                if (k0 + u <= 2 * R) {
#pragma unroll
                    for (int m = 0; m < CW; ++m) { col[2 * m] = dp2a(v[u][m], ADD_LO, col[2 * m]); col[2 * m + 1] += v[u][m] >> 16; }
                }
            }
        }
    }

    uint32_t e[Gm::NW], eo[Gm::NW];
    int gi = 0;
    for (int yg = y0; yg < y1; yg += GR, ++gi) {
        // ---- V: rounded means of GR rows into tmpb, column sums stepped row by row
        mbar_wait(&ring_bar, (uint32_t)gi & 1u);
        if (vact) {
            for (int j0 = 0; j0 < GR; j0 += 8) {
#pragma unroll
                for (int j8 = 0; j8 < 8; ++j8) {
                    const int j = j0 + j8;
                    uint32_t m[CPT];
#pragma unroll
                    for (int k = 0; k < CPT; ++k) m[k] = ct_mean(col[k], job.inv);
                    CV t;
                    if constexpr (CPT == 8) t = make_uint4(pack_lo(m[0], m[1]), pack_lo(m[2], m[3]), pack_lo(m[4], m[5]), pack_lo(m[6], m[7]));
                    else t = make_uint2(pack_lo(m[0], m[1]), pack_lo(m[2], m[3]));
                    *reinterpret_cast<CV*>(tmpb + (size_t)j * pj.rowbuf + (size_t)(Gm::PAD + c0) * 2) = t;
                    uint32_t a[CW], b[CW];
                    load_cols<CPT, U8>(ring + (size_t)j * row_bytes + (size_t)c0 * BPS, a);
                    load_cols<CPT, U8>(ring + (size_t)(GR + j) * row_bytes + (size_t)c0 * BPS, b);
#pragma unroll
                    for (int q = 0; q < CW; ++q) {
                        col[2 * q] = dp2a(b[q], SUB_LO, dp2a(a[q], ADD_LO, col[2 * q]));
                        col[2 * q + 1] = col[2 * q + 1] + (a[q] >> 16) - (b[q] >> 16);
                    }
                }
            }
        }
        __syncthreads();  // tmpb complete, ring consumed
        if (threadIdx.x == 0 && yg + GR < y1) {
            fence_proxy_async();
            issue_ring(yg + GR);
        }
        // ---- H: each lane group blurs one row of means (SYM closed form), in place in tmpb
        {
            uint16_t* row = reinterpret_cast<uint16_t*>(tmpb + (size_t)(warp * RPW + sub) * pj.rowbuf);
            hseg_load_row<R>(e, row, w, sg, G, pj.S, true, act, lane);
            const uint32_t W = h_window<R>(e);
            const uint32_t C = __shfl_sync(0xffffffffu, line_const(W, job.inv, job.inv2), lane & ~(G - 1));
            h_slide<R, kCtChains, false>(e, eo, W, C, job.inv2);
            __syncwarp();  // every lane has read its halos: the staged row may be overwritten
            if (act) h_store_own<R>(eo, row + Gm::PAD + L * sg);
            __syncwarp();
            // coalesced copy-out of the warp's rows
            for (int s2 = 0; s2 < RPW; ++s2) {
                const int y = yg + warp * RPW + s2;
                if (y < y1) {
                    const unsigned char* from = tmpb + (size_t)(warp * RPW + s2) * pj.rowbuf + Gm::PAD * 2;
                    char* to = dst + (size_t)y * pj.dst_pitch;
                    if constexpr (!U8) {
                        for (uint32_t off = lane * 16; off < row_bytes; off += 512) st_global_hint(to + off, *reinterpret_cast<const uint4*>(from + off), drop);
                    } else {  // 16 bytes of 16-bit results -> 8 bytes of the 8-bit row
                        for (uint32_t off = lane * 8; off < (uint32_t)((w + 7) & ~7); off += 256) {  // (the same extent of tmpb as the 16-bit copy)
                            const uint4 t = *reinterpret_cast<const uint4*>(from + 2 * off);
                            __stcs(reinterpret_cast<uint2*>(to + off), make_uint2(__byte_perm(t.x, t.y, 0x6420), __byte_perm(t.z, t.w, 0x6420)));
                        }
                    }
                }
            }
        }
        __syncthreads();  // tmpb free
    }
}

template <int R, bool U8>
int launch_ctfused(const SegJob& whole, int count, cudaStream_t st) {
    using Gm = HGeom<R>;
    for (int k = 0; k < whole.nplanes; ++k)
        if (whole.pl[k].w > CTF_WARPS * 32 * 8 || (whole.pl[k].w + L - 1) / L > 32) return 1;
    SegJob groups[3];
    const int ngroups = shape_groups(whole, groups);
    for (int g = 0; g < ngroups; ++g) {
        SegJob& job = groups[g];
        const int w = job.pl[0].w, h = job.pl[0].h;
        // planes up to 960 wide (1080p chroma): 4 warps x 8 columns per thread and 4 CTAs per SM instead of 8 warps x 4 columns and 2 -
        // the two CTA-wide barriers per group of rows cost less across 4 warps, and 4 CTAs interleave their V and H phases
        // (1080p YUV420P16, r = 13: 2.96 -> 2.74 us per frame)
        const bool narrow = w <= 16 * L;   // at most 16 lanes per row: 2 or 4 rows per warp, so a group is still a multiple of 8 rows
        const int nwarps = narrow ? 4 : CTF_WARPS;
        const int S = (w + L - 1) / L, G = lanes_per_row(S), RPW = 32 / G, GR = nwarps * RPW;
        const int rowbuf = rowbuf_bytes(Gm::row_samples(S), G);
        const size_t row_bytes = (size_t)((w * (U8 ? 1 : 2) + 15) & ~15);
        const size_t smem = (size_t)2 * GR * row_bytes + (size_t)GR * rowbuf;
        // rows per band: the first 2r rows of a band are read twice, so bands are as tall as the batch allows while the launch
        // still has ~4 waves of CTAs (a whole plane per CTA for big batches, 2 groups per band for a lone frame)
        const long planes = (long)count * job.nplanes;
        int nb = (int)std::min<long>((4 * 296 + planes - 1) / planes, (h + 2 * GR - 1) / (2 * GR));
        nb = std::max(nb, 1);
        const int band = (((h + nb - 1) / nb + GR - 1) / GR) * GR;
        int cta = 0;
        for (int k = 0; k < job.nplanes; ++k) {
            SegPlane& s = job.pl[k];
            s.S = S; s.G = G; s.rowbuf = rowbuf; s.per_cta = band;
            s.cta_begin = cta;
            cta += (h + band - 1) / band;
        }
        job.ctas_per_frame = cta;
        const int rc = narrow ? launch_frames(ctfused_kernel<R, 8, U8, 4>, job, count, 4 * 32, smem, st)
                              : launch_frames(ctfused_kernel<R, 8, U8>, job, count, CTF_WARPS * 32, smem, st);
        if (rc) return rc;
    }
    return 0;
}

}  // namespace

int run_seg_ct(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int count, int r, cudaStream_t st) {
    if ((l.kind != K_U16 && l.kind != K_U8) || src == dst) return 1;
    const SegJob job = base_job(l, mask, src, sfs, dst, dfs, r, 1);
    const bool u8 = l.kind == K_U8;
    return with_radius(r, [&](auto radius) {
        constexpr int R = decltype(radius)::value;
        return u8 ? launch_ctfused<R, true>(job, count, st) : launch_ctfused<R, false>(job, count, st);
    });
}

}  // namespace vsz
