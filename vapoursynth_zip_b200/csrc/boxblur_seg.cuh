// boxblur_seg.cuh — shared by boxblur_seg_{h,v,ct}.cu: sm_100a "segment" kernels for vszip.BoxBlur on 8- and 16-bit integer clips.
//
// Integer BoxBlur has a closed form per pass (boxblur_seg_core.h; src/filters/boxblur_runtime.zig:10-41), so a line
// does not have to be walked by one thread.  Here a thread owns a segment of 60 consecutive samples of a line, keeps
// it in registers across ALL passes of the axis, and per pass only exchanges the r samples either side of the segment:
//
//   hseg_kernel    rows.  A warp owns a row (32 lanes x 60 samples = 1920; narrower planes pack 2 or 4 rows per warp).
//                  Rows are staged by the TMA engine: one cp.async.bulk (global -> shared, mbarrier completion) per row
//                  into a per-warp double buffer, one cp.async.bulk (shared -> global) per finished row.  No thread
//                  issues a global load or store; halo exchange is warp-local (shared memory + __syncwarp).
//   vseg_kernel    columns.  A CTA owns a 64-column strip of a plane; lane = pair of columns (one 32-bit word per row),
//                  warp = 60-row segment.  Global access is coalesced by construction (128 bytes per warp and row).
//   ctfused_kernel the comptime path (hradius == vradius <= 22, one pass each; src/filters/boxblur_comptime.zig:10-159)
//                  in ONE read and ONE write of the plane: a CTA streams down a band of rows keeping exact column sums in
//                  registers (8 columns per thread); the rows entering and leaving the window arrive through a TMA-fed
//                  shared-memory ring; the rounded means of 8 (16) rows go to shared memory and each warp then runs the
//                  horizontal closed form on one (two) of them.
//
// The radius is a template parameter (1..22: every comptime radius); other radii, float clips and planes wider
// than 1920 / taller than 1080 keep the streaming kernels of boxblur_kernels.cu.  8-bit clips run the same kernels: bytes are widened
// after the TMA load and narrowed before the store (template parameter U8).
#pragma once

#include <algorithm>

#include "boxblur_host.h"
#include "boxblur_seg_core.h"
#include "common.h"
#include "filter.h"

namespace vsz {

namespace {

using namespace seg;

// --------------------------------------------------------------------------- job descriptors
struct SegPlane {
    size_t src_off, dst_off;
    int src_pitch, dst_pitch;
    int w, h;
    int cta_begin;
    int S;       // segments (threads) along the blurred axis
    int G;       // H: lanes per row (8 / 16 / 32)
    int rowbuf;  // H: bytes between staged rows
    int per_cta; // H: row groups per CTA; ctfused: rows per band
};
struct SegJob {
    const char* src;
    char* dst;
    size_t src_fs, dst_fs;
    int nplanes, ctas_per_frame, passes;
    uint32_t inv, inv2;
    SegPlane pl[3];
};

__device__ __forceinline__ const SegPlane& seg_plane(const SegJob& b, int cta, int& local) {
    int k = b.nplanes - 1;
    while (k > 0 && cta < b.pl[k].cta_begin) --k;
    local = cta - b.pl[k].cta_begin;
    return b.pl[k];
}

// --------------------------------------------------------------------------- TMA (bulk async copy) + mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
// global -> shared, completion counted in bytes on the mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sdst)), "l"(gsrc),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global, tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
// L2 eviction priorities: rows that will be read again soon are kept (evict_last), data that is dead after this access
// leaves first (evict_first)
__device__ __forceinline__ uint64_t l2_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s_hint(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(sdst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void st_global_hint(void* g, const uint4& v, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(g), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

#ifndef VSZ_SEG_ALL_DP
#define VSZ_SEG_ALL_DP false
#endif
constexpr bool kAllDp = VSZ_SEG_ALL_DP;
constexpr int kCtChains = 2;  // independent running sums per thread in the comptime path's H pass

// The lane's view ext[] of the staged row(s) of a lane group (sample 0 at row + PAD), halos included.
//   e[] = the lane's registers: its own samples are loaded from the row here (from_row), or are given (two consecutive samples
//   per word) and published to the row.  Mirrors: when the row ends exactly at a segment end the first and last lane write them
//   from registers; ragged rows copy them inside the staged row and the last lane reloads its span (which contains mirrored
//   samples).  The row may be overwritten after the next __syncwarp.
template <int R>
__device__ __forceinline__ void hseg_load_row(uint32_t (&e)[HGeom<R>::NW], uint16_t* row, int n, int sg, int G, int S, bool from_row, bool act,
                                              int lane) {
    using Gm = HGeom<R>;
    uint16_t* own = row + Gm::PAD + L * sg;
    const int lig = lane & (G - 1);
    if (from_row) h_load_own<R>(e, own);
    else if (act) h_store_own<R>(e, own);
    if (L * S == n) {
        if (lig == 0) h_write_left_pad<R>(e, row + Gm::PAD);
        if (lig == S - 1) h_write_right_pad<R>(e, row + Gm::PAD + n);
        __syncwarp();
    } else {
        __syncwarp();
#pragma unroll
        for (int t = 0; t < 3; ++t) {  // r <= 22 < 3 * 8 lanes
            const int k = lig + t * G;
            if (k < R) {
                row[Gm::PAD - 1 - k] = row[Gm::PAD + k];
                row[Gm::PAD + n + k] = row[Gm::PAD + n - 1 - k];
            }
        }
        __syncwarp();
        if (lig == S - 1) h_load_own<R>(e, own);
    }
    h_load_halos<R>(e, own);
}
// ... and the words of the H pass from it; ends with every lane past its reads of the row, so the row may be overwritten
template <int R>
__device__ __forceinline__ void hseg_load_pairs(uint32_t (&e)[HGeom<R>::NW], uint32_t (&p)[NP], uint16_t* row, int n, int sg, int G, int S,
                                                bool from_row, bool act, int lane) {
    hseg_load_row<R>(e, row, n, sg, G, S, from_row, act, lane);
    h_pairs<R>(e, p);
    __syncwarp();
}

// The words of the next H pass from h_slide_next's q[] and xs[].  Rows that end at a segment end exchange only the edges: every
// lane publishes its first and last HW words (the first / last lane their mirrors too) and completes its edge words from the
// neighbours'.  Ragged rows go through hseg_load_pairs with the lane's own samples.
template <int R>
__device__ __forceinline__ void hseg_next_pairs(uint32_t (&e)[HGeom<R>::NW], uint32_t (&q)[NP], const uint32_t (&xs)[2 * HGeom<R>::HW],
                                                uint16_t* row, int n, int sg, int G, int S, bool act, int lane) {
    using Gm = HGeom<R>;
    if (L * S == n) {
        uint16_t* own = row + Gm::PAD + L * sg;
        const int lig = lane & (G - 1);
        if (act) h_store_edges<R>(xs, own);
        if (lig == 0) h_write_left_pad_words<R>(xs, row + Gm::PAD);
        if (lig == S - 1) h_write_right_pad_words<R>(xs + 2 * Gm::HW, row + Gm::PAD + n);
        __syncwarp();
        h_load_halos<R>(e, own);
        __syncwarp();
        h_complete_edges<R>(q, e);
    } else {
        h_own_words<R>(q, e + Gm::HW);
        hseg_load_pairs<R>(e, q, row, n, sg, G, S, false, act, lane);
    }
}

// window sum at own[0] and the line constant C of the pass (the group's first lane holds the window at position 0)
template <int R>
__device__ __forceinline__ uint32_t hseg_window(const uint32_t (&p)[NP], int lane, int G, uint32_t inv, uint32_t inv2, uint32_t& C) {
    const uint32_t W = pair_window<R>(p);
    C = __shfl_sync(0xffffffffu, line_const(W, inv, inv2), lane & ~(G - 1));
    return W;
}

// --------------------------------------------------------------------------- host side
SegJob base_job(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int r, int passes) {
    SegJob j{};
    j.src = src; j.dst = dst; j.src_fs = sfs; j.dst_fs = dfs; j.passes = passes;
    axis_consts(r, j.inv, j.inv2);
    int k = 0;
    for (int p = 0; p < l.nplanes; ++p) {
        if (!mask[p]) continue;
        SegPlane& s = j.pl[k++];
        s.src_off = s.dst_off = l.pl[p].offset;
        s.src_pitch = s.dst_pitch = l.pl[p].pitch;
        s.w = l.pl[p].w; s.h = l.pl[p].h;
    }
    j.nplanes = k;
    return j;
}

int lanes_per_row(int S) { return S > 16 ? 32 : (S > 8 ? 16 : 8); }

// bytes between staged rows: a multiple of 16, and for 8-lane groups 16 words off a multiple of 32 words so that the two
// groups of a half-warp fall on disjoint banks
int rowbuf_bytes(int samples, int G) {
    int words = (samples + 1) / 2;
    words = (words + 3) & ~3;
    if (G == 8) while ((words & 31) != 16) words += 4;
    return words * 4;
}

// Planes of different shapes want different CTA shapes (V: warps = segments per column; comptime: columns per thread), so a
// job is launched once per group of equally shaped planes.  Returns the number of groups.
int shape_groups(const SegJob& job, SegJob (&groups)[3]) {
    bool done[3] = {false, false, false};
    int n = 0;
    for (int k = 0; k < job.nplanes; ++k) {
        if (done[k]) continue;
        SegJob& sub = groups[n++];
        sub = job;
        sub.nplanes = 0;
        for (int q = k; q < job.nplanes; ++q)
            if (!done[q] && job.pl[q].w == job.pl[k].w && job.pl[q].h == job.pl[k].h) { sub.pl[sub.nplanes++] = job.pl[q]; done[q] = true; }
    }
    return n;
}

}  // namespace

}  // namespace vsz
