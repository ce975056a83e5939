// CPU lane-by-lane simulation of the H passes of the segment BoxBlur kernels (vapoursynth_zip_b200/csrc/boxblur_seg_h.cu, the H
// part of boxblur_seg_ct.cu).  TEST INFRASTRUCTURE: it runs the product's own per-thread arithmetic (boxblur_seg_core.h: pair
// words, one dp2a per window step) with the kernels' orchestration (edge exchange, mirror pads, ragged rows) replayed
// sequentially, so that tests/test_seg_pairs_sim.py can check it against the oracle without a GPU.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

#include "boxblur_seg_core.h"

using namespace vsz::seg;

namespace {

struct Axis { uint32_t inv, inv2; };
Axis axis(int r) {
    const uint64_t inv = ((1ull << 32) + (uint64_t)r) / (uint64_t)(2 * r + 1);
    return {(uint32_t)inv, (uint32_t)(inv >> 16)};
}

// ---- hseg_kernel: one row, `passes` passes, the way a group of lanes runs it (hseg_load_pairs, h_slide_next, hseg_next_pairs,
// h_slide_out)
template <int R>
void h_row(const uint16_t* src, uint16_t* dst, int n, int passes) {
    using G = HGeom<R>;
    using Ext = uint32_t[G::NW];
    using Pairs = uint32_t[NP];
    const Axis ax = axis(R);
    const int S = (n + L - 1) / L;
    const bool exact = L * S == n;
    std::vector<uint16_t> buf(G::row_samples(S) + 8, 0xdead);
    uint16_t* row = buf.data() + G::PAD;
    // the bulk copy brings round16(n*2) bytes; model the garbage tail
    memcpy(row, src, (size_t)n * 2);
    std::vector<std::vector<uint32_t>> ext(S, std::vector<uint32_t>(G::NW, 0xabababab)), p(S, std::vector<uint32_t>(NP, 0xcdcdcdcd)),
        xs(S, std::vector<uint32_t>(2 * G::HW, 0xefefefef));
    auto E = [&](int s) -> Ext& { return *reinterpret_cast<Ext*>(ext[s].data()); };
    auto P = [&](int s) -> Pairs& { return *reinterpret_cast<Pairs*>(p[s].data()); };
    // hseg_load_pairs: own samples in ext[] (from the row on the first pass, else published here), mirrors, halos, words
    auto load_pairs = [&](bool from_row) {
        for (int s = 0; s < S; ++s) {
            if (from_row) h_load_own<R>(E(s), row + L * s);
            else h_store_own<R>(E(s), row + L * s);
        }
        if (exact) {
            h_write_left_pad<R>(E(0), row);
            h_write_right_pad<R>(E(S - 1), row + n);
        } else {
            for (int k = 0; k < R; ++k) { row[-1 - k] = row[k]; row[n + k] = row[n - 1 - k]; }
            h_load_own<R>(E(S - 1), row + L * (S - 1));
        }
        for (int s = 0; s < S; ++s) {
            h_load_halos<R>(E(s), row + L * s);
            h_pairs<R>(E(s), P(s));
        }
    };
    load_pairs(true);
    std::vector<uint32_t> out(LW);
    for (int pass = 0; pass < passes; ++pass) {
        const uint32_t C = line_const(pair_window<R>(P(0)), ax.inv, ax.inv2);
        if (pass + 1 == passes) {
            for (int s = 0; s < S; ++s) {
                h_slide_out<R>(P(s), *reinterpret_cast<uint32_t(*)[LW]>(out.data()), pair_window<R>(P(s)), C, ax.inv2);
                h_store_words(out.data(), row + L * s);
            }
            break;
        }
        // hseg_next_pairs
        for (int s = 0; s < S; ++s) {
            uint32_t q[NP];
            h_slide_next<R>(P(s), q, *reinterpret_cast<uint32_t(*)[2 * G::HW]>(xs[s].data()), pair_window<R>(P(s)), C, ax.inv2);
            memcpy(P(s), q, sizeof q);
        }
        if (exact) {
            for (int s = 0; s < S; ++s) h_store_edges<R>(*reinterpret_cast<uint32_t(*)[2 * G::HW]>(xs[s].data()), row + L * s);
            h_write_left_pad_words<R>(xs[0].data(), row);
            h_write_right_pad_words<R>(xs[S - 1].data() + 2 * G::HW, row + n);
            for (int s = 0; s < S; ++s) {
                h_load_halos<R>(E(s), row + L * s);
                h_complete_edges<R>(P(s), E(s));
            }
        } else {
            for (int s = 0; s < S; ++s) h_own_words<R>(P(s), E(s) + G::HW);
            load_pairs(false);
        }
    }
    memcpy(dst, row, (size_t)n * 2);
}

// ---- ctfused_kernel, H part: its single pass over one row (hseg_load_row, h_window, h_slide with two chains)
template <int R>
void h_row_single(const uint16_t* src, uint16_t* dst, int n) {
    using G = HGeom<R>;
    using Ext = uint32_t[G::NW];
    const Axis ax = axis(R);
    const int S = (n + L - 1) / L;
    std::vector<uint16_t> buf(G::row_samples(S) + 8, 0xdead);
    uint16_t* row = buf.data() + G::PAD;
    memcpy(row, src, (size_t)n * 2);
    std::vector<std::vector<uint32_t>> ext(S, std::vector<uint32_t>(G::NW, 0xabababab)), out(S, std::vector<uint32_t>(G::NW));
    auto E = [&](int s) -> Ext& { return *reinterpret_cast<Ext*>(ext[s].data()); };
    for (int s = 0; s < S; ++s) h_load_own<R>(E(s), row + L * s);
    if (L * S == n) {
        h_write_left_pad<R>(E(0), row);
        h_write_right_pad<R>(E(S - 1), row + n);
    } else {
        for (int k = 0; k < R; ++k) { row[-1 - k] = row[k]; row[n + k] = row[n - 1 - k]; }
        h_load_own<R>(E(S - 1), row + L * (S - 1));
    }
    for (int s = 0; s < S; ++s) h_load_halos<R>(E(s), row + L * s);
    const uint32_t C = line_const(h_window<R>(E(0)), ax.inv, ax.inv2);
    for (int s = 0; s < S; ++s) {
        Ext& o = *reinterpret_cast<Ext*>(out[s].data());
        const uint32_t W = h_window<R>(E(s));
        h_slide<R, 2, false>(E(s), o, W, C, ax.inv2);
        h_store_own<R>(o, row + L * s);
    }
    memcpy(dst, row, (size_t)n * 2);
}

template <int R>
int run(int what, const uint16_t* src, uint16_t* dst, int w, int h, int passes) {
    for (int y = 0; y < h; ++y) {
        if (what == 0) h_row<R>(src + (size_t)y * w, dst + (size_t)y * w, w, passes);
        else h_row_single<R>(src + (size_t)y * w, dst + (size_t)y * w, w);
    }
    return 0;
}

}  // namespace

// what: 0 = hseg_kernel's H passes, 1 = ctfused_kernel's single H pass (passes ignored).  Returns -1 for an unsupported radius.
extern "C" int seg_pairs_sim_u16(int what, const uint16_t* src, uint16_t* dst, int w, int h, int r, int passes) {
    switch (r) {
#define CASE(R) case R: return run<R>(what, src, dst, w, h, passes);
        CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9) CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15)
        CASE(16) CASE(17) CASE(18) CASE(19) CASE(20) CASE(21) CASE(22)
#undef CASE
    }
    return -1;
}
