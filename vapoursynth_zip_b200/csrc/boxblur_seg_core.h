// boxblur_seg_core.h — per-thread arithmetic of the "segment" integer BoxBlur kernels (boxblur_seg_kernels.cu).
//
// Integer BoxBlur is exactly parallelisable (SURVEY §7.2): one runtime-path pass over a line is
//     out[x] = (S0 + inv2*(W_x - W_0)) >> 16 = (C + inv2*W_x) >> 16,      C = S0 - inv2*W_0 (mod 2^32),
// with W_x the 2r+1 window sum under SYM mirroring and S0 = (W_0*inv + 2^31) >> 16
// (src/filters/boxblur_runtime.zig:10-41; the u64 running sum stays below 2^32, so u32 arithmetic is exact).
// A thread therefore owns a SEGMENT of L = 60 consecutive samples of a line, keeps it in registers across all
// passes, and only exchanges the r samples either side of the segment with its neighbours per pass.
//
// 16-bit samples stay packed two per 32-bit word; `dp2a` (IDP.2A) adds or subtracts the halves of a word to a 32-bit sum
// in one instruction, so samples are never unpacked.  H passes pair each sample with the one 2r+1 further on (see h_pairs),
// so that one window step is one dp2a.
//
// Everything here is __host__ __device__: tests/sim/boxblur_seg_sim.cpp runs the same code lane by lane on the
// CPU against the oracle (the container that builds this has no GPU).
#pragma once

#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define VSZ_HD __host__ __device__ __forceinline__
#else
#define VSZ_HD inline
#endif

namespace vsz {
namespace seg {

constexpr int L = 60;       // samples of a line one thread owns
constexpr int LW = L / 2;   // ... in 32-bit words when the word packs two consecutive samples (H)

// selectors for dp2a: bytes 0/1 are the signed weights of the low/high 16-bit half
constexpr uint32_t ADD_LO = 0x0001u, ADD_HI = 0x0100u, ADD_BOTH = 0x0101u, SUB_LO = 0x00ffu, SUB_HI = 0xff00u;
constexpr uint32_t ADD2_LO = 0x0002u, ADD2_HI = 0x0200u;

// c + a.lo16 * (int8)sel.b0 + a.hi16 * (int8)sel.b1   (mod 2^32)
VSZ_HD uint32_t dp2a(uint32_t a, uint32_t sel, uint32_t c) {
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("dp2a.lo.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(sel), "r"(c));
    return d;
#else
    const int32_t b0 = (int8_t)(sel & 0xffu), b1 = (int8_t)((sel >> 8) & 0xffu);
    return c + (a & 0xffffu) * (uint32_t)b0 + (a >> 16) * (uint32_t)b1;
#endif
}

// (x >> 16) | (y & 0xffff0000): the two 16.16 results of a word, packed
VSZ_HD uint32_t pack_hi(uint32_t x, uint32_t y) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, 0x7632);
#else
    return (x >> 16) | (y & 0xffff0000u);
#endif
}
// (x & 0xffff) | (y << 16)
VSZ_HD uint32_t pack_lo(uint32_t x, uint32_t y) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, 0x5410);
#else
    return (x & 0xffffu) | (y << 16);
#endif
}

// 8-byte aligned 64-bit access to staged samples
VSZ_HD void ld64(const uint16_t* p, uint32_t& a, uint32_t& b) {
#if defined(__CUDA_ARCH__)
    const uint2 v = *reinterpret_cast<const uint2*>(p);
    a = v.x; b = v.y;
#else
    uint32_t v[2];
    memcpy(v, p, 8);
    a = v[0]; b = v[1];
#endif
}
VSZ_HD void st64(uint16_t* p, uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    *reinterpret_cast<uint2*>(p) = make_uint2(a, b);
#else
    const uint32_t v[2] = {a, b};
    memcpy(p, v, 8);
#endif
}

// the per-line constant C of the closed form, from the window sum at position 0
VSZ_HD uint32_t line_const(uint32_t w0, uint32_t inv, uint32_t inv2) {
    const uint32_t s0 = (uint32_t)(((uint64_t)w0 * inv + 0x80000000ull) >> 16);
    return s0 - inv2 * w0;
}

// =========================================================================== H
// ext[] is the thread's view of its row as staged in shared memory: [prev halo | own 60 samples | next halo], two consecutive
// samples per word, whole 64-bit units.
template <int R>
struct HGeom {
    static_assert(R >= 1 && 2 * R + 2 <= L, "segment kernels need 1 <= r <= 29");
    static constexpr int HW = 2 * ((R + 3) / 4);   // words of either halo (>= r samples, loaded as 64-bit units)
    static constexpr int NW = HW + LW + HW;
    static constexpr int J0 = 2 * HW;              // sample index of own[0] inside ext[]
    static constexpr int PAD = 8 * ((R + 7) / 8);  // samples in front of a staged row (multiple of 16 bytes)
    static constexpr int PADR = 2 * HW;            // samples behind the last segment that a thread may read
    // samples of one staged row: pad, S segments, tail
    static constexpr int row_samples(int S) { return PAD + L * S + PADR; }
};

// A pass holds one word per window step of the segment [x0, x0 + 60): both samples of that step,
//     p[k] = (lo16: s[x0 + k + r + 1], hi16: s[x0 + k - r]),   k = 0 .. NP-1,
// so that a step is one dp2a, W_{k+1} = W_k + lo16(p[k]) - hi16(p[k]), and an output one IMAD, o_k = W_k * inv2 + C (16.16:
// the sample is hi16(o_k)).  The words of the next pass are two 16.16 outputs 2r+1 apart, pack_hi(o_{k+r+1}, o_{k-r}) (PRMT).
// The first r words take their high half from the left neighbour's last r outputs, the last r words their low half from the
// right neighbour's first r outputs; between passes they hold the lane's own 16.16 output alone (h_complete_edges fills in
// the other half once the neighbours have published theirs).
constexpr int NP = L - 1;
constexpr uint32_t STEP = 0xff01u;  // dp2a selector: + low half - high half

// byte permute: bytes 0-3 of x, 4-7 of y, one selector nibble per result byte
VSZ_HD uint32_t prmt(uint32_t x, uint32_t y, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, sel);
#else
    const uint64_t v = ((uint64_t)y << 32) | x;
    uint32_t d = 0;
    for (int b = 0; b < 4; ++b) d |= (uint32_t)((v >> (8 * ((sel >> (4 * b)) & 7u))) & 0xffu) << (8 * b);
    return d;
#endif
}

// the words of a pass from the staged samples in ext[]
template <int R>
VSZ_HD void h_pairs(const uint32_t (&ext)[HGeom<R>::NW], uint32_t (&p)[NP]) {
    using G = HGeom<R>;
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const int a = G::J0 + k + R + 1, b = G::J0 + k - R;  // entering / leaving sample (a - b is odd: opposite halves)
        p[k] = prmt(ext[a >> 1], ext[b >> 1], (a & 1) ? 0x5432u : 0x7610u);
    }
}

// the edge words, from the neighbours' samples in the halo part of ext[] (the own part is not read)
template <int R>
VSZ_HD void h_complete_edges(uint32_t (&p)[NP], const uint32_t (&ext)[HGeom<R>::NW]) {
    using G = HGeom<R>;
#pragma unroll
    for (int k = 0; k < R; ++k) {
        const int b = G::J0 + k - R;
        p[k] = prmt(p[k], ext[b >> 1], (b & 1) ? 0x7632u : 0x5432u);
    }
#pragma unroll
    for (int k = NP - R; k < NP; ++k) {
        const int a = G::J0 + k + R + 1;
        p[k] = prmt(ext[a >> 1], p[k], (a & 1) ? 0x7632u : 0x7610u);
    }
}

// window sum of the samples [-r, r] around the segment's first sample: the high halves of p[0..2r]
template <int R, int N>
VSZ_HD uint32_t pair_window(const uint32_t (&p)[N]) {
    uint32_t W = 0;
#pragma unroll
    for (int k = 0; k <= 2 * R; ++k) W = dp2a(p[k], ADD_HI, W);
    return W;
}

// One pass over a segment of N + 1 samples that feeds another: emit(i, o_i) gets the 16.16 outputs, q[] receives the next
// pass's words (edge words holding the own output only).
template <int R, int N, class Emit>
VSZ_HD void pair_slide_next(const uint32_t (&p)[N], uint32_t (&q)[N], uint32_t W, uint32_t C, uint32_t inv2, Emit emit) {
    uint32_t o[N + 1];
#pragma unroll
    for (int i = 0; i <= N; ++i) {
        o[i] = W * inv2 + C;
        if (i < N) W = dp2a(p[i], STEP, W);
        if (i > 2 * R) q[i - R - 1] = pack_hi(o[i], o[i - 2 * R - 1]);
        else if (i > R) q[i - R - 1] = o[i];                    // first r words: the high half comes from the segment before
        if (i >= N - 2 * R && i < N - R) q[i + R] = o[i];     // last r words: the low half comes from the segment after
        emit(i, o[i]);
    }
}
// The last pass: emit(i, o_i) only.
template <int R, int N, class Emit>
VSZ_HD void pair_slide_out(const uint32_t (&p)[N], uint32_t W, uint32_t C, uint32_t inv2, Emit emit) {
#pragma unroll
    for (int i = 0; i <= N; ++i) {
        emit(i, W * inv2 + C);
        if (i < N) W = dp2a(p[i], STEP, W);
    }
}

// H, a pass that feeds another: also xs[], the first and the last HW words of the own samples (two consecutive samples per
// word) that the neighbours need.
template <int R>
VSZ_HD void h_slide_next(const uint32_t (&p)[NP], uint32_t (&q)[NP], uint32_t (&xs)[2 * HGeom<R>::HW], uint32_t W, uint32_t C,
                         uint32_t inv2) {
    constexpr int HW = HGeom<R>::HW;
    uint32_t prev = 0;
    pair_slide_next<R>(p, q, W, C, inv2, [&](int i, uint32_t o) {
        if (i & 1) {
            if (i < 2 * HW) xs[i >> 1] = pack_hi(prev, o);
            if (i >= L - 2 * HW) xs[HW + ((i - (L - 2 * HW)) >> 1)] = pack_hi(prev, o);
        }
        prev = o;
    });
}

// H, the last pass: the outputs packed two consecutive samples per word.
template <int R>
VSZ_HD void h_slide_out(const uint32_t (&p)[NP], uint32_t (&out)[LW], uint32_t W, uint32_t C, uint32_t inv2) {
    uint32_t prev = 0;
    pair_slide_out<R>(p, W, C, inv2, [&](int i, uint32_t o) {
        if (i & 1) out[i >> 1] = pack_hi(prev, o);
        prev = o;
    });
}

// window sum of the samples [-R, R] around own[0]
template <int R>
VSZ_HD uint32_t h_window(const uint32_t (&ext)[HGeom<R>::NW]) {
    using G = HGeom<R>;
    constexpr int a = G::J0 - R, b = G::J0 + R;
    uint32_t W = 0;
#pragma unroll
    for (int k = a >> 1; k <= (b >> 1); ++k) {
        const bool lo = 2 * k >= a, hi = 2 * k + 1 <= b;
        W = dp2a(ext[k], (lo ? ADD_LO : 0u) | (hi ? ADD_HI : 0u), W);
    }
    return W;
}

// The single H pass of the comptime path (ctfused_kernel) works on ext[] as staged: with no next pass to feed, building the
// pair words would cost a PRMT per sample that nothing reuses.
// One pass over the owned segment.  The segment is cut into NCH independent chains (each with its own running window
// sum, started from a window computed out of registers) so that a thread always has NCH dependency chains in flight.
// Within a chain two steps are taken together:  W1 = t -/+ hi,  W2 = u + hiA - hiB  with t, u the dp2a (low-half)
// updates, so the chain is 3 dependent operations per 2 samples and the high-half terms are one 3-input add.
template <int R>
VSZ_HD uint32_t h_window_at(const uint32_t (&ext)[HGeom<R>::NW], int i0) {  // window sum around own[i0] (i0 compile-time after unrolling)
    using G = HGeom<R>;
    const int a = G::J0 + i0 - R, b = G::J0 + i0 + R;
    uint32_t W = 0;
#pragma unroll
    for (int k = a >> 1; k <= (b >> 1); ++k) {
        const bool lo = 2 * k >= a, hi = 2 * k + 1 <= b;
        W = dp2a(ext[k], (lo ? ADD_LO : 0u) | (hi ? ADD_HI : 0u), W);
    }
    return W;
}

// HI_DP: the high-half terms go through dp2a as well (4 dp2a per 2 samples, all on the full-rate FMA pipe) instead of
// shift + add (ALU pipe, which issues at half the rate on sm_100).
template <int R, int NCH, bool HI_DP>
VSZ_HD void h_slide(const uint32_t (&ext)[HGeom<R>::NW], uint32_t (&out)[HGeom<R>::NW], uint32_t W0, uint32_t C, uint32_t inv2) {  // results -> own part of out[]
    using G = HGeom<R>;
    constexpr int CL = L / NCH;  // samples per chain (even)
    static_assert(L % NCH == 0 && CL % 2 == 0, "chains must hold whole words");
    uint32_t W[NCH];
    W[0] = W0;
#pragma unroll
    for (int c = 1; c < NCH; ++c) W[c] = h_window_at<R>(ext, c * CL);
#pragma unroll
    for (int i = 0; i < CL; i += 2) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int x = c * CL + i;  // even
            const int ja = G::J0 + x + R + 1, jb = G::J0 + x - R;  // samples entering / leaving at the step x -> x+1
            uint32_t t, W1;
            const uint32_t o0 = W[c] * inv2 + C;
            if ((ja & 1) == 0) {  // entering sample is a low half, leaving one a high half
                t = dp2a(ext[ja >> 1], ADD_LO, W[c]);
                W1 = HI_DP ? dp2a(ext[jb >> 1], SUB_HI, t) : t - (ext[jb >> 1] >> 16);
            } else {
                t = dp2a(ext[jb >> 1], SUB_LO, W[c]);
                W1 = HI_DP ? dp2a(ext[ja >> 1], ADD_HI, t) : t + (ext[ja >> 1] >> 16);
            }
            out[G::HW + (x >> 1)] = pack_hi(o0, W1 * inv2 + C);
            if (i + 2 < CL) {
                // step x+1 -> x+2: the entering sample is ja+1, the leaving one jb+1
                uint32_t u;
                if ((ja & 1) == 0) u = dp2a(ext[(jb + 1) >> 1], SUB_LO, t);
                else u = dp2a(ext[(ja + 1) >> 1], ADD_LO, t);
                // the two high halves of these two steps: one entering, one leaving
                const int ha = (ja & 1) ? ja : ja + 1, hb = (jb & 1) ? jb : jb + 1;
                if (HI_DP) W[c] = dp2a(ext[hb >> 1], SUB_HI, dp2a(ext[ha >> 1], ADD_HI, u));
                else W[c] = u + (ext[ha >> 1] >> 16) - (ext[hb >> 1] >> 16);
            }
        }
    }
}

// The own samples of h_slide_next's q[] (before h_complete_edges), packed two consecutive samples per word: sample i is hi16 of
// q[i + r] for i < NP - r, else (i - r - 1 >= r + 1) hi16 of a left edge word or lo16 of a complete word.
template <int R>
VSZ_HD void h_own_words(const uint32_t (&q)[NP], uint32_t* own) {
    auto at = [](int i, int& w, bool& hi) {
        if (i < NP - R) { w = i + R; hi = true; }
        else { w = i - R - 1; hi = w < R; }
    };
#pragma unroll
    for (int m = 0; m < LW; ++m) {
        int wa, wb;
        bool ha, hb;
        at(2 * m, wa, ha);
        at(2 * m + 1, wb, hb);
        own[m] = prmt(q[wa], q[wb], (ha ? 0x32u : 0x10u) | ((hb ? 0x76u : 0x54u) << 8));
    }
}

// Loads.  `own` points at the thread's first sample inside the staged row (8-byte aligned).
template <int R>
VSZ_HD void h_load_halos(uint32_t (&ext)[HGeom<R>::NW], const uint16_t* own) {
    using G = HGeom<R>;
#pragma unroll
    for (int k = 0; k < G::HW; k += 2) {
        ld64(own - 2 * G::HW + 2 * k, ext[k], ext[k + 1]);
        ld64(own + L + 2 * k, ext[G::HW + LW + k], ext[G::HW + LW + k + 1]);
    }
}
template <int R>
VSZ_HD void h_load_own(uint32_t (&ext)[HGeom<R>::NW], const uint16_t* own) {
    using G = HGeom<R>;
#pragma unroll
    for (int k = 0; k < LW; k += 2) {
        ld64(own + 2 * k, ext[G::HW + k], ext[G::HW + k + 1]);
    }
}
// w = LW words of own samples
VSZ_HD void h_store_words(const uint32_t* w, uint16_t* own) {
#pragma unroll
    for (int k = 0; k < LW; k += 2) st64(own + 2 * k, w[k], w[k + 1]);
}
template <int R>
VSZ_HD void h_store_own(const uint32_t (&ext)[HGeom<R>::NW], uint16_t* own) {
    h_store_words(ext + HGeom<R>::HW, own);
}
// the neighbours' part of h_slide_next's xs[]: the first and the last HW words of the own samples
template <int R>
VSZ_HD void h_store_edges(const uint32_t (&xs)[2 * HGeom<R>::HW], uint16_t* own) {
    using G = HGeom<R>;
#pragma unroll
    for (int k = 0; k < G::HW; k += 2) {
        st64(own + 2 * k, xs[k], xs[k + 1]);
        st64(own + L - 2 * G::HW + 2 * k, xs[G::HW + k], xs[G::HW + k + 1]);
    }
}

// SYM mirror pads of a staged row written straight from the registers of the lanes that own the samples (no shared-memory
// read-modify-write): the first lane writes samples -1-k = own[k], the last lane (when the row ends exactly at its segment end)
// samples n+k = own[59-k], k = 0..r-1 (one sample more when r is odd; the pads are sized for it).
VSZ_HD uint32_t halfswap(uint32_t w) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, w, 0x1032);
#else
    return (w >> 16) | (w << 16);
#endif
}
VSZ_HD void st32(uint16_t* p, uint32_t a) {
#if defined(__CUDA_ARCH__)
    *reinterpret_cast<uint32_t*>(p) = a;
#else
    memcpy(p, &a, 4);
#endif
}
// first = the lane's first own words (two consecutive samples each), at least (r + 1) / 2 of them
template <int R>
VSZ_HD void h_write_left_pad_words(const uint32_t* first, uint16_t* row0) {  // row0 = sample 0 of the staged row
    constexpr int NWD = (R + 1) / 2;
#pragma unroll
    for (int m = 0; m + 1 < NWD; m += 2) st64(row0 - 4 - 2 * m, halfswap(first[m + 1]), halfswap(first[m]));
    if (NWD & 1) st32(row0 - 2 * NWD, halfswap(first[NWD - 1]));
}
// end = one past the lane's last own word
template <int R>
VSZ_HD void h_write_right_pad_words(const uint32_t* end, uint16_t* row_end) {  // row_end = sample n (= end of the lane's segment)
    constexpr int NWD = (R + 1) / 2;
#pragma unroll
    for (int m = 0; m + 1 < NWD; m += 2) st64(row_end + 2 * m, halfswap(end[-1 - m]), halfswap(end[-2 - m]));
    if (NWD & 1) st32(row_end + 2 * (NWD - 1), halfswap(end[-NWD]));
}

template <int R>
VSZ_HD void h_write_left_pad(const uint32_t (&ext)[HGeom<R>::NW], uint16_t* row0) {
    h_write_left_pad_words<R>(ext + HGeom<R>::HW, row0);
}
template <int R>
VSZ_HD void h_write_right_pad(const uint32_t (&ext)[HGeom<R>::NW], uint16_t* row_end) {
    h_write_right_pad_words<R>(ext + HGeom<R>::HW + LW, row_end);
}

// =========================================================================== V: a word = the same row of two columns
// ext[] = [r rows above | own LV rows | r rows below], one word (two adjacent columns) per row.  LV = rows a thread owns
// (90 when the plane height is a multiple of 90, e.g. 1080 and 540: 12 / 6 warps per column strip; else 60).
template <int R, int LV>
struct VGeom {
    static_assert(R >= 1 && R < LV, "segment kernels need 1 <= r < segment length");
    static constexpr int NW = R + LV + R;
    static constexpr int J0 = R;
};

// The high-half column goes through shift + add (ALU pipe) and the low-half one through dp2a (FMA pipe) so that both
// pipes, which issue at the same rate, stay busy while all warps of a CTA are in this phase together.
template <int R, int LV>
VSZ_HD void v_window(const uint32_t (&ext)[VGeom<R, LV>::NW], uint32_t& Wl, uint32_t& Wh) {
    Wl = 0; Wh = 0;
#pragma unroll
    for (int j = 0; j <= 2 * R; ++j) {
        Wl = dp2a(ext[j], ADD_LO, Wl);
        Wh += ext[j] >> 16;
    }
}

// window sum at line position 0 under SYM mirroring, from the rows the first segment owns: s[r] + 2*sum(s[0..r-1])
template <int R, int LV>
VSZ_HD void v_window0(const uint32_t (&ext)[VGeom<R, LV>::NW], uint32_t& Wl, uint32_t& Wh) {
    Wl = dp2a(ext[R + R], ADD_LO, 0u);
    Wh = ext[R + R] >> 16;
#pragma unroll
    for (int j = 0; j < R; ++j) {
        Wl = dp2a(ext[R + j], ADD2_LO, Wl);
        Wh += (ext[R + j] >> 16) * 2u;
    }
}

// emit(i, word) receives the packed results of row i of the segment (into registers, or straight to global memory in the
// last pass)
template <int R, int LV, bool ALL_DP, class Emit>
VSZ_HD void v_slide_emit(const uint32_t (&ext)[VGeom<R, LV>::NW], uint32_t Wl, uint32_t Wh, uint32_t Cl, uint32_t Ch, uint32_t inv2, Emit emit) {
#pragma unroll
    for (int i = 0; i < LV; ++i) {
        emit(i, pack_hi(Wl * inv2 + Cl, Wh * inv2 + Ch));
        if (i + 1 < LV) {
            const uint32_t A = ext[R + i + R + 1], B = ext[i];
            Wl = dp2a(A, ADD_LO, Wl);
            Wl = dp2a(B, SUB_LO, Wl);
            if (ALL_DP) { Wh = dp2a(A, ADD_HI, Wh); Wh = dp2a(B, SUB_HI, Wh); }
            else Wh = Wh + (A >> 16) - (B >> 16);
        }
    }
}
template <int R, int LV, bool ALL_DP>
VSZ_HD void v_slide(const uint32_t (&ext)[VGeom<R, LV>::NW], uint32_t (&out)[LV], uint32_t Wl, uint32_t Wh, uint32_t Cl, uint32_t Ch,
                    uint32_t inv2) {
    v_slide_emit<R, LV, ALL_DP>(ext, Wl, Wh, Cl, Ch, inv2, [&](int i, uint32_t v) { out[i] = v; });
}

// =========================================================================== comptime path, vertical part
// Exact column sums under R101q mirroring (src/filters/boxblur_comptime.zig:50-109): the window of row i+1 is the
// window of row i minus row ct_sub_row(i) plus row ct_add_row(i) (as multisets of source rows).
VSZ_HD int ct_tap_row(int i, int k, int r, int n) {  // source row of tap k (0..2r) of output row i
    if (k < r) {
        const int need = r - k;
        return (i < need) ? ((need - i < n - 1) ? need - i : n - 1) : i - need;
    }
    const int over = k - r, room = n - 1 - i;
    if (room < over) { const int d = over - room; return i - (d < i ? d : i); }
    return i + over;
}
VSZ_HD int ct_sub_row(int i, int r) { return i < r ? r - i : i - r; }
VSZ_HD int ct_add_row(int i, int r, int n) { return (i + 1 + r <= n - 1) ? i + 1 + r : i; }

// rounded mean of an exact column sum: (col*inv + 2^31) >> 32 (boxblur_comptime.zig:111-128)
VSZ_HD uint32_t ct_mean(uint32_t col, uint32_t inv) { return (uint32_t)(((uint64_t)col * inv + 0x80000000ull) >> 32); }

}  // namespace seg
}  // namespace vsz
