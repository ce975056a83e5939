// boxblur_seg_h.cu — hseg_kernel: horizontal passes, TMA-staged rows (see boxblur_seg.cuh for the design of the segment kernels).
#include "boxblur_seg.cuh"

namespace vsz {

namespace {

// =========================================================================== H
constexpr int HSEG_WARPS = 8;
#ifndef VSZ_HSEG_MINB
#define VSZ_HSEG_MINB 2
#endif

// U8: 8-bit clips run the same 16-bit arithmetic (the closed form is the same for every integer sample type,
// src/filters/boxblur_runtime.zig:10-41, and its results fit a byte).  The TMA engine moves BYTE rows; a lane widens its 60 bytes into
// the packed 16-bit registers after the load and narrows them before the store, everything in between is the 16-bit kernel.
template <int R, bool U8>
__global__ void __launch_bounds__(HSEG_WARPS * 32, VSZ_HSEG_MINB) hseg_kernel(const SegJob job) {
    using Gm = HGeom<R>;
    extern __shared__ __align__(128) unsigned char seg_smem[];
    __shared__ uint64_t bars[HSEG_WARPS][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int local;
    const SegPlane& pj = seg_plane(job, blockIdx.y, local);
    const int G = pj.G, RPW = 32 / G, sub = lane / G, sg0 = lane % G;
    const bool act = sg0 < pj.S;
    const int sg = act ? sg0 : 0;  // idle lanes shadow lane 0 (loads only)
    const int n = pj.w;
    const int groups = (pj.h + RPW - 1) / RPW;
    const int g_end = min((local + 1) * pj.per_cta, groups);
    const uint32_t row_bytes = (uint32_t)((n * (U8 ? 1 : 2) + 15) & ~15);   // what the TMA engine moves per row
    const uint32_t bytebuf = U8 ? (uint32_t)((pj.S * L + 15) & ~15) : 0u;     // U8: a byte row (whole segments) next to every staged 16-bit row
    unsigned char* wbase = seg_smem + (size_t)warp * (2 * RPW * (pj.rowbuf + bytebuf));
    unsigned char* bbase = wbase + (size_t)2 * RPW * pj.rowbuf;
    const char* src = job.src + (size_t)blockIdx.x * job.src_fs + pj.src_off;
    char* dst = job.dst + (size_t)blockIdx.x * job.dst_fs + pj.dst_off;

    if (lane == 0) {
        mbar_init(&bars[warp][0], 1);
        mbar_init(&bars[warp][1], 1);
        fence_mbar_init();
    }
    __syncwarp();
    auto issue = [&](int g, int b) {  // lane 0: stage the rows of group g into buffer b
        const int rows = min(RPW, pj.h - g * RPW);
        mbar_expect_tx(&bars[warp][b], (uint32_t)rows * row_bytes);
        for (int s2 = 0; s2 < rows; ++s2)
            bulk_g2s(U8 ? bbase + (size_t)(b * RPW + s2) * bytebuf : wbase + (size_t)(b * RPW + s2) * pj.rowbuf + Gm::PAD * 2,
                     src + (size_t)(g * RPW + s2) * pj.src_pitch, row_bytes, &bars[warp][b]);
    };
    int g = local * pj.per_cta + warp;
    if (lane == 0 && g < g_end) issue(g, 0);
    uint32_t e[Gm::NW], pa[NP], pb[NP], xs[2 * Gm::HW], out[LW];
    for (int it = 0; g < g_end; g += HSEG_WARPS, ++it) {
        const int b = it & 1;
        uint16_t* row = reinterpret_cast<uint16_t*>(wbase + (size_t)(b * RPW + sub) * pj.rowbuf);
        uint16_t* own = row + Gm::PAD + L * sg;
        mbar_wait(&bars[warp][b], (uint32_t)(it >> 1) & 1u);
        uint32_t* bown = reinterpret_cast<uint32_t*>(bbase + (size_t)(b * RPW + sub) * bytebuf + L * sg);  // the lane's 60 bytes
        if constexpr (U8) {
#pragma unroll
            for (int j = 0; j < L / 4; ++j) {
                const uint32_t w4 = bown[j];
                e[Gm::HW + 2 * j] = __byte_perm(w4, 0u, 0x4140);
                e[Gm::HW + 2 * j + 1] = __byte_perm(w4, 0u, 0x4342);
            }
        }
        hseg_load_pairs<R>(e, pa, row, n, sg, G, pj.S, !U8, act, lane);
        if (lane == 0 && g + HSEG_WARPS < g_end) {
            bulk_wait_read0();  // the other buffer's previous rows have left shared memory
            fence_proxy_async();
            issue(g + HSEG_WARPS, b ^ 1);
        }
        // Every call site has fixed roles for pa / pb, so that passes need no register copies.
        auto mid = [&](uint32_t (&in)[NP], uint32_t (&next)[NP]) {
            uint32_t C;
            const uint32_t W = hseg_window<R>(in, lane, G, job.inv, job.inv2, C);
            h_slide_next<R>(in, next, xs, W, C, job.inv2);
            hseg_next_pairs<R>(e, next, xs, row, n, sg, G, pj.S, act, lane);
        };
        auto last = [&](uint32_t (&in)[NP]) {
            uint32_t C;
            const uint32_t W = hseg_window<R>(in, lane, G, job.inv, job.inv2, C);
            h_slide_out<R>(in, out, W, C, job.inv2);
        };
        int left = job.passes;
        for (; left > 2; left -= 2) {
            mid(pa, pb);
            mid(pb, pa);
        }
        if (left == 2) {
            mid(pa, pb);
            last(pb);
        } else {
            last(pa);
        }
        if (act) {
            if constexpr (U8) {
#pragma unroll
                for (int j = 0; j < L / 4; ++j) bown[j] = __byte_perm(out[2 * j], out[2 * j + 1], 0x6420);
            } else {
                h_store_words(out, own);
            }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
            const int rows = min(RPW, pj.h - g * RPW);
            for (int s2 = 0; s2 < rows; ++s2)
                bulk_s2g(dst + (size_t)(g * RPW + s2) * pj.dst_pitch,
                         U8 ? bbase + (size_t)(b * RPW + s2) * bytebuf : wbase + (size_t)(b * RPW + s2) * pj.rowbuf + Gm::PAD * 2, row_bytes);
            bulk_commit();
        }
    }
    if (lane == 0) bulk_wait0();  // shared memory must outlive the last bulk stores
}

template <int R, bool U8>
int launch_hseg(SegJob job, int count, cudaStream_t st) {
    using Gm = HGeom<R>;
    size_t smem = 0;
    int cta = 0;
    for (int k = 0; k < job.nplanes; ++k) {
        SegPlane& s = job.pl[k];
        s.S = (s.w + L - 1) / L;
        if (s.S > 32) return 1;
        s.G = lanes_per_row(s.S);
        const int RPW = 32 / s.G;
        s.rowbuf = rowbuf_bytes(Gm::row_samples(s.S), s.G);
        smem = std::max(smem, (size_t)HSEG_WARPS * 2 * RPW * (s.rowbuf + (U8 ? ((s.S * L + 15) & ~15) : 0)));
        const int groups = (s.h + RPW - 1) / RPW;
        // ~4 row groups per warp and CTA; fewer when a lone frame would leave SMs idle
        int per_warp = 4;
        if (count * ((groups + HSEG_WARPS * per_warp - 1) / (HSEG_WARPS * per_warp)) < 2 * 148) per_warp = 1;
        s.per_cta = HSEG_WARPS * per_warp;
        s.cta_begin = cta;
        cta += (groups + s.per_cta - 1) / s.per_cta;
    }
    job.ctas_per_frame = cta;
    if (smem > (size_t)kMaxSmemPerCta) return 1;
    return launch_frames(hseg_kernel<R, U8>, job, count, HSEG_WARPS * 32, smem, st);
}

}  // namespace

int run_seg_h(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int count, int r, int passes,
              cudaStream_t st) {
    if ((l.kind != K_U16 && l.kind != K_U8) || passes < 1) return 1;
    const SegJob job = base_job(l, mask, src, sfs, dst, dfs, r, passes);
    const bool u8 = l.kind == K_U8;
    return with_radius(r, [&](auto radius) {
        constexpr int R = decltype(radius)::value;
        return u8 ? launch_hseg<R, true>(job, count, st) : launch_hseg<R, false>(job, count, st);
    });
}

}  // namespace vsz
