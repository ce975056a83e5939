// boxblur_kernels.cu — sm_100a kernels for vszip.BoxBlur.
//
// Semantics restated from the reference (see DESIGN.md §BoxBlur for the derivation):
//   runtime path  (src/filters/boxblur_runtime.zig:10-119): per line and pass a running box sum with
//       SYM (edge-repeating) mirroring; integer S += inv2*(a-b), out = S>>16; float S += (a-b)*div.
//   comptime path (src/filters/boxblur_comptime.zig:10-159): V first with exact R101q column sums and a
//       rounded mean, then the runtime H pass; float uses direct tap-ordered sums (:161-263).
//
// Design: a line (row or column) is owned by exactly one thread, which streams along it once and
// pipelines all `P` passes of that axis: at time t stage p works on position t - p*r, its "add"
// operand is the value stage p-1 produced in the same step (a register), its "sub" operand is the
// value stage p-1 produced 2r+1 steps ago.  Every stage keeps those last 2r+1 values in a shared-
// memory delay ring and all stages share one slot index (t mod (2r+1)), so a stage costs one LDS, one
// STS (the same address: an exchange) and the multiply-adds; no pass ever touches HBM for
// intermediates.  Lines are packed 4/sizeof(T) per thread into 32-bit words so ring traffic and global
// accesses are 32-bit per lane.  The arithmetic per line is the reference's own op sequence, hence
// bit-exact for integer AND float formats.
//
//   blur_v_kernel : lines = columns, thread = 32-bit column group; global access coalesced by construction.
//   blur_h_kernel : lines = rows; a CTA owns NT*NL rows and stages 32-position tiles through shared
//                   memory (coalesced row segments in, transposed so each thread reads its own rows).
//   ctf_*_kernel  : comptime float path (direct sums, R101q).
#include <cuda_fp16.h>

#include "boxblur_host.h"
#include "common.h"
#include "filter.h"

namespace vsz {

enum BlurMode { MODE_RT = 0, MODE_CTV = 1 };

// --------------------------------------------------------------------------- pixel traits
template <typename T> struct Px;
template <> struct Px<uint8_t> { static constexpr int NL = 4; using Acc = uint32_t; static constexpr bool flt = false; };
template <> struct Px<uint16_t> { static constexpr int NL = 2; using Acc = uint32_t; static constexpr bool flt = false; };
template <> struct Px<__half> { static constexpr int NL = 2; using Acc = float; static constexpr bool flt = true; };
template <> struct Px<float> { static constexpr int NL = 1; using Acc = float; static constexpr bool flt = true; };

template <typename T> __device__ __forceinline__ void unpack(uint32_t w, typename Px<T>::Acc (&v)[Px<T>::NL]);
template <> __device__ __forceinline__ void unpack<uint8_t>(uint32_t w, uint32_t (&v)[4]) {
    v[0] = w & 0xffu; v[1] = (w >> 8) & 0xffu; v[2] = (w >> 16) & 0xffu; v[3] = w >> 24;
}
template <> __device__ __forceinline__ void unpack<uint16_t>(uint32_t w, uint32_t (&v)[2]) {
    v[0] = w & 0xffffu; v[1] = w >> 16;
}
template <> __device__ __forceinline__ void unpack<__half>(uint32_t w, float (&v)[2]) {
    const __half2 h = *reinterpret_cast<const __half2*>(&w);
    const float2 f = __half22float2(h);
    v[0] = f.x; v[1] = f.y;
}
template <> __device__ __forceinline__ void unpack<float>(uint32_t w, float (&v)[1]) { v[0] = __uint_as_float(w); }

// Parameters of one axis, uniform over the launch.
struct AxisParams {
    int r;          // radius
    int ring;       // 2r+1
    uint32_t inv2;  // inv >> 16
    uint32_t inv;   // floor((2^32 + r) / (2r+1))  (fits u32 for r >= 1)
    float div;      // 1 / (2r+1) in f32
};

// --------------------------------------------------------------------------- one stage's arithmetic
// Integer stages keep S = 16.16 fixed point in u32: the reference's u64 running sum stays below 2^32
// (its Debug build would trap on the narrowing cast otherwise), so modular u32 arithmetic is exact.
template <typename T, int MODE>
struct StageOps {
    using X = Px<T>;
    using Acc = typename X::Acc;
    static constexpr int NL = X::NL;

    // returns the packed output word after folding (a - b) into S
    static __device__ __forceinline__ uint32_t update(Acc (&S)[NL], uint32_t aw, uint32_t bw, const AxisParams& ap) {
        Acc a[NL], b[NL];
        unpack<T>(aw, a);
        unpack<T>(bw, b);
#pragma unroll
        for (int l = 0; l < NL; ++l) {
            if constexpr (X::flt) {
                const float d = __fsub_rn(a[l], b[l]);
                S[l] = __fadd_rn(S[l], __fmul_rn(d, ap.div));
            } else if constexpr (MODE == MODE_CTV) {
                S[l] = S[l] + a[l] - b[l];
            } else {
                S[l] = S[l] + ap.inv2 * (a[l] - b[l]);
            }
        }
        return emit(S, ap);
    }

    // packed output of the current state
    static __device__ __forceinline__ uint32_t emit(const Acc (&S)[NL], const AxisParams& ap) {
        if constexpr (std::is_same<T, float>::value) {
            return __float_as_uint(S[0]);
        } else if constexpr (std::is_same<T, __half>::value) {
            const __half2 h = __floats2half2_rn(S[0], S[1]);
            return *reinterpret_cast<const uint32_t*>(&h);
        } else {
            uint32_t o[NL];
#pragma unroll
            for (int l = 0; l < NL; ++l) {
                if constexpr (MODE == MODE_CTV)
                    o[l] = (uint32_t)(((uint64_t)S[l] * ap.inv + 0x80000000ull) >> 32);  // rounded mean
                else
                    o[l] = S[l] >> 16;
            }
            if constexpr (NL == 2) return o[0] | (o[1] << 16);
            else return o[0] | (o[1] << 8) | (o[2] << 16) | (o[3] << 24);
        }
    }

    // start-of-line state from the first r+1 samples of the previous stage (read through `rd(pos)`)
    template <class RD>
    static __device__ __forceinline__ void init(Acc (&S)[NL], const AxisParams& ap, RD rd) {
        Acc v[NL];
        if constexpr (X::flt) {
            // sum = in[r]; sum += in[x]*2 for x = 0..r-1 (in that order); sum *= div
            unpack<T>(rd(ap.r), v);
#pragma unroll
            for (int l = 0; l < NL; ++l) S[l] = v[l];
            for (int x = 0; x < ap.r; ++x) {
                unpack<T>(rd(x), v);
#pragma unroll
                for (int l = 0; l < NL; ++l) S[l] = __fadd_rn(S[l], __fmul_rn(v[l], 2.0f));
            }
#pragma unroll
            for (int l = 0; l < NL; ++l) S[l] = __fmul_rn(S[l], ap.div);
        } else if constexpr (MODE == MODE_CTV) {
            // reflect-101 window at row 0: in[0] + 2*sum(in[1..r])
            unpack<T>(rd(0), v);
#pragma unroll
            for (int l = 0; l < NL; ++l) S[l] = v[l];
            for (int x = 1; x <= ap.r; ++x) {
                unpack<T>(rd(x), v);
#pragma unroll
                for (int l = 0; l < NL; ++l) S[l] += 2u * v[l];
            }
        } else {
            // W0 = in[r] + 2*sum(in[0..r-1]);  S0 = (W0*inv + 2^31) >> 16
            unpack<T>(rd(ap.r), v);
            uint32_t w0[NL];
#pragma unroll
            for (int l = 0; l < NL; ++l) w0[l] = v[l];
            for (int x = 0; x < ap.r; ++x) {
                unpack<T>(rd(x), v);
#pragma unroll
                for (int l = 0; l < NL; ++l) w0[l] += 2u * v[l];
            }
#pragma unroll
            for (int l = 0; l < NL; ++l) S[l] = (uint32_t)(((uint64_t)w0[l] * ap.inv + 0x80000000ull) >> 16);
        }
    }
};

// compile-time loop: f(std::integral_constant<int, 0>{}), ..., f(std::integral_constant<int, N-1>{})
template <class F, int... Is>
__device__ __forceinline__ void static_for_impl(std::integer_sequence<int, Is...>, F& f) { (f(std::integral_constant<int, Is>{}), ...); }
template <int N, class F>
__device__ __forceinline__ void static_for(F&& f) { static_for_impl(std::make_integer_sequence<int, N>{}, f); }

// --------------------------------------------------------------------------- the per-thread pipeline
// Skewed schedule: stage p (1..P) works at time t on position x = t - p*D, D = r+1.  Its operands are
// what stage p-1 published one step earlier: a = v_{p-1}(t-1) (position x+r) and b = the ring entry that
// publication displaced (position x-r-1, written 2r+1 steps before).  Both are carried in registers, so
// within one step all P stages (x NL packed lines) are independent instruction chains.
//
// Edges cost nothing in the steady state because the mirrors are materialised in the rings:
//   low edge : when stage p starts (x = 0) it seeds its state from positions 0..r of ring p-1 and writes
//              the mirrored samples into the ring slots of the virtual positions -r..-1, so the b operands
//              of x = 1..r come out of the ordinary exchange;
//   high edge: after its last real sample a stage keeps publishing r mirrored samples (virtual positions
//              n..n+r-1, read back from its own ring), so the a operands of x >= n-r are ordinary too.
// Idle or drained stages just compute on don't-care values.  Ring layout: word ((slot*P + q)*NT + tid),
// slot = t mod (2r+1) shared by all stages, so stage offsets are compile-time immediates.
// W = 32-bit words per thread and ring cell (1 or 2): with W = 2 a thread owns twice as many lines, ring and
// global accesses are 64-bit, and the per-step bookkeeping is amortised over twice the pixels.
template <int W> struct alignas(4 * W) Vec { uint32_t v[W]; };

template <typename T, int P, int MODE, int NT, int W = 1>
struct LinePipe {
    using Ops = StageOps<T, MODE>;
    using Acc = typename Px<T>::Acc;
    using V = Vec<W>;
    static constexpr int NL = Px<T>::NL;
    static constexpr int SLOT_WORDS = P * NT * W;

    // u16 runtime path: the low 16-bit line of va[] is also carried unpacked (it falls out of the previous stage's
    // S >> 16) and the subtrahend's low line is folded in arithmetically, which moves three unpack operations per
    // word and stage from the ALU pipe (the bound of these kernels on B200) to IMADs on the FMA pipe.
    static constexpr bool SPLIT = std::is_same<T, uint16_t>::value && MODE == MODE_RT;
    Acc S[P][W][NL];
    uint32_t alo[P][W];  // SPLIT only: va[q].v[w] & 0xffff
    V va[P], vb[P];   // operands of stage q+1 for the next step
    V pa[P], pb[P];   // ring cells of slot(t) and slot(t+1), fetched two / one step(s) ahead of their exchange
    uint32_t* ring;   // &ring_base[tid * W]
    uint32_t* cur;    // ring + slot(t) * SLOT_WORDS
    uint32_t* cur2;   // ring + slot(t+2) * SLOT_WORDS
    int slot;         // t mod (2r+1)
    int n, D;         // line length, stage delay r+1
    AxisParams ap;

    __device__ __forceinline__ void start(uint32_t* ring_, int n_, const AxisParams& ap_) {
        ring = ring_; n = n_; ap = ap_; D = ap_.r + 1;
        slot = 0; cur = ring; cur2 = ring + 2 * SLOT_WORDS;  // ring >= 3 slots
#pragma unroll
        for (int q = 0; q < P; ++q)
#pragma unroll
            for (int w = 0; w < W; ++w) {
                va[q].v[w] = vb[q].v[w] = pa[q].v[w] = pb[q].v[w] = 0u;
                alo[q][w] = 0u;
#pragma unroll
                for (int l = 0; l < NL; ++l) S[q][w][l] = Acc(0);
            }
    }
    __device__ __forceinline__ int lag() const { return P * D; }
    __device__ __forceinline__ int fast_begin() const { return P * D + 1; }  // first t with every stage at x >= 1
    __device__ __forceinline__ V& cell(int s, int q) { return *reinterpret_cast<V*>(ring + (s * P + q) * (NT * W)); }
    static __device__ __forceinline__ V& at(uint32_t* base, int q) { return *reinterpret_cast<V*>(base + q * (NT * W)); }
    // slot k steps behind slot(t) (0 <= k <= ring)
    __device__ __forceinline__ int back(int k) const { const int s = slot - k; return s < 0 ? s + ap.ring : s; }
    __device__ __forceinline__ void advance() {
        ++slot; cur += SLOT_WORDS;
        if (slot == ap.ring) { slot = 0; cur = ring; }
        cur2 += SLOT_WORDS;
        if (cur2 == ring + ap.ring * SLOT_WORDS) cur2 = ring;
    }
    static __device__ __forceinline__ uint32_t mad_lo(uint32_t a, uint32_t b, uint32_t c) {
        uint32_t d;
        asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
        return d;
    }
    // one stage update; lo[w] = low 16-bit line of the result (SPLIT only)
    __device__ __forceinline__ V update(int q, const V& a, const V& b, uint32_t (&lo)[W]) {
        V o;
        if constexpr (SPLIT) {
            const uint32_t inv2 = ap.inv2, ninv2 = 0u - ap.inv2, inv2s = ap.inv2 << 16;
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const uint32_t aw = a.v[w], bw = b.v[w];
                const uint32_t bhi = bw >> 16;
                // S_lo += inv2*a_lo - inv2*b_lo with b_lo = bw - (bhi << 16), all modulo 2^32
                uint32_t s0 = mad_lo(alo[q][w], inv2, S[q][w][0]);
                s0 = mad_lo(bw, ninv2, s0);
                s0 = mad_lo(bhi, inv2s, s0);
                const uint32_t s1 = mad_lo((aw >> 16) - bhi, inv2, S[q][w][1]);
                S[q][w][0] = s0; S[q][w][1] = s1;
                lo[w] = s0 >> 16;
                o.v[w] = (s1 & 0xffff0000u) | lo[w];
            }
        } else {
#pragma unroll
            for (int w = 0; w < W; ++w) { o.v[w] = Ops::update(S[q][w], a.v[w], b.v[w], ap); lo[w] = 0u; }
        }
        return o;
    }
    __device__ __forceinline__ V update(int q, const V& a, const V& b) {
        uint32_t lo[W];
        return update(q, a, b, lo);
    }

    // publish v as stage q's value of this step: exchange with the ring cell of slot(t) (already in pa[q],
    // loaded two steps ago so no shared-memory latency sits on the critical path) and keep the look-ahead going.
    __device__ __forceinline__ void publish(int q, const V& v) {
        vb[q] = pa[q];
        va[q] = v;
        if constexpr (SPLIT) {
#pragma unroll
            for (int w = 0; w < W; ++w) alo[q][w] = v.v[w] & 0xffffu;
        }
        at(cur, q) = v;
    }
    __device__ __forceinline__ void publish(int q, const V& v, const uint32_t (&lo)[W]) {  // lo = known low lines of v
        vb[q] = pa[q];
        va[q] = v;
        if constexpr (SPLIT) {
#pragma unroll
            for (int w = 0; w < W; ++w) alo[q][w] = lo[w];
        }
        at(cur, q) = v;
    }
    __device__ __forceinline__ void rotate(int q) {
        pa[q] = pb[q];
        pb[q] = at(cur2, q);
    }

    // steady state, t in [fast_begin, n).  Returns stage P's output for position t - P*D.
    __device__ __forceinline__ V step_fast(const V& v_in) {
        V nv[P];
        uint32_t nlo[P][W];
#pragma unroll
        for (int q = 0; q < P; ++q) nv[q] = update(q, va[q], vb[q], nlo[q]);
#pragma unroll
        for (int q = 0; q < P; ++q) {
            if (q == 0) publish(0, v_in);
            else publish(q, nv[q > 0 ? q - 1 : 0], nlo[q > 0 ? q - 1 : 0]);
            rotate(q);
        }
        advance();
        return nv[P - 1];
    }

    // ---- edge steps with a compile-time set of live stages (no per-stage branching) -------------------------
    // Start-up phase k (t in [kD, (k+1)D)): stages 1..k are live, stage k itself starts (x = 0) on the first
    // step of the phase; producers 0..k publish.  Requires n >= fast_begin().
    __device__ __forceinline__ V seed(int Q) {
        const int r = ap.r;
        V out;
#pragma unroll
        for (int w = 0; w < W; ++w) {
            // ring Q holds positions -r..r of stage Q; position p sits (r - p + 1) slots behind slot(t)
            Ops::init(S[Q][w], ap, [&](int pos) { return cell(back(r - pos + 1), Q).v[w]; });
        }
        for (int k = 1; k <= r; ++k) {  // virtual position -k: SYM -> k-1, reflect-101 (comptime V) -> k
            const int from = (MODE == MODE_CTV) ? k : k - 1;
            cell(back(r + k + 1), Q) = cell(back(r - from + 1), Q);
        }
        pa[Q] = cell(slot, Q);  // the seeding rewrote slot(t) and slot(t+1) of ring Q
        pb[Q] = cell(slot + 1 == ap.ring ? 0 : slot + 1, Q);
        const V c = cell(back(1), Q);
#pragma unroll
        for (int w = 0; w < W; ++w) {
            if constexpr (MODE == MODE_CTV) out.v[w] = Ops::emit(S[Q][w], ap);
            else out.v[w] = Ops::update(S[Q][w], c.v[w], c.v[w], ap);  // the reference's x = 0 step adds in[r] - in[r]
        }
        return out;
    }

    template <int ACT, bool INIT>
    __device__ __forceinline__ V step_start(const V& v_in) {
        V nv[P];
        static_for<P>([&](auto qc) {
            constexpr int q = decltype(qc)::value;
            if constexpr (INIT && q == ACT - 1) nv[q] = seed(q);
            else if constexpr (q < ACT) nv[q] = update(q, va[q], vb[q]);
            else nv[q] = V{};
        });
        static_for<P>([&](auto qc) {
            constexpr int q = decltype(qc)::value;
            if constexpr (q <= ACT) publish(q, (q == 0) ? v_in : nv[q > 0 ? q - 1 : 0]);
            if constexpr (q < ACT) rotate(q);
        });
        advance();
        return nv[P - 1];
    }

    // Drain phase K (t in [n + KD, n + (K+1)D)): producer K is in its mirrored tail (first r steps of the phase,
    // j = step index inside the phase), producers > K still publish real samples, consumers K+1..P are live.
    template <int K, bool MIRROR>
    __device__ __forceinline__ V step_drain(int j) {
        V nv[P];
        static_for<P>([&](auto qc) {
            constexpr int q = decltype(qc)::value;
            if constexpr (q >= K) nv[q] = update(q, va[q], vb[q]);
            else nv[q] = V{};
        });
        static_for<P>([&](auto qc) {
            constexpr int q = decltype(qc)::value;
            if constexpr (q == K) {
                if constexpr (MIRROR) publish(q, cell(back((MODE == MODE_CTV) ? 1 + ap.r : 1 + 2 * j), q));
                rotate(q);
            } else if constexpr (q > K) {
                publish(q, nv[q > 0 ? q - 1 : 0]);
                rotate(q);
            }
        });
        advance();
        return nv[P - 1];
    }

    // Runs steps [t, t_end) for callers that cannot structure their loops by phase (the tiled H kernel walks the line
    // in 32-step chunks): the phase dispatch is hoisted out of the per-step loops, so every inner loop contains one
    // compile-time step variant.  in(t) -> V is the input sample of step t, out(t, V) receives stage P's result.
    // Requires n >= fast_begin().
    template <class IN, class OUT>
    __device__ __forceinline__ void run_steps(int t, const int t_end, IN in, OUT out) {
        while (t < t_end) {
            if (t < n) {
                if (t >= fast_begin()) {
                    const int e = min(t_end, n);
                    for (; t < e; ++t) out(t, step_fast(in(t)));
                    continue;
                }
                const int k = t / D, j = t - k * D;  // start-up phase k (0..P), step j inside it
                static_for<P + 1>([&](auto kc) {
                    constexpr int K = decltype(kc)::value;
                    if (k == K) {
                        if constexpr (K >= 1) {
                            if (j == 0) { out(t, step_start<K, true>(in(t))); ++t; }
                        }
                        const int e = min((K == P) ? K * D + 1 : (K + 1) * D, t_end);
                        for (; t < e; ++t) out(t, step_start<K, false>(in(t)));
                    }
                });
            } else {
                const int k = (t - n) / D;  // drain phase k (0..P-1)
                static_for<P>([&](auto kc) {
                    constexpr int K = decltype(kc)::value;
                    if (k == K) {
                        const int base = n + K * D, e = min(base + D, t_end);
                        const int em = min(base + ap.r, e);  // mirrored-tail steps of this phase come first
                        for (; t < em; ++t) out(t, step_drain<K, true>(t - base));
                        for (; t < e; ++t) out(t, step_drain<K, false>(0));
                    }
                });
                if (k >= P) t = t_end;  // nothing left to compute
            }
        }
    }

    // any t, any n (tiny lines): also seeds stages that start at this step and publishes mirrored tails.  v_in is
    // the input sample for time t (ignored once t >= n).  The result is meaningful iff 0 <= t - P*D < n.
    __device__ __forceinline__ V step_edge(int t, const V& v_in) {
        V nv[P];
        const int r = ap.r;
#pragma unroll
        for (int q = 0; q < P; ++q) {
            const int x = t - (q + 1) * D;  // position of stage q+1
            if (x == 0) nv[q] = seed(q);
            else if (x > 0 && x < n) nv[q] = update(q, va[q], vb[q]);
            else nv[q] = V{};  // not started yet / already drained: nothing to compute
        }
#pragma unroll
        for (int q = 0; q < P; ++q) {
            const int y = t - q * D;  // position stage q publishes now
            if (y >= 0 && y < n + r) {
                V v = (q == 0) ? v_in : nv[q > 0 ? q - 1 : 0];
                if (y >= n) {
                    // mirrored tail, re-read from the stage's own ring (never from global memory: the kernels
                    // run in place).  SYM: position 2n-1-y; comptime V (R101q): position y-r-1.
                    v = cell(back((MODE == MODE_CTV) ? 1 + r : 1 + 2 * (y - n)), q);
                }
                publish(q, v);
            }
            rotate(q);
        }
        advance();
        return nv[P - 1];
    }
};

__device__ __forceinline__ const PlaneJob& find_plane(const BatchJob& b, int cta, int& local) {
    int k = b.nplanes - 1;
    while (k > 0 && cta < b.pl[k].cta_begin) --k;
    local = cta - b.pl[k].cta_begin;
    return b.pl[k];
}

// 4/8-byte asynchronous global->shared copies (LDGSTS): their completion is tracked by commit groups, not
// by the register scoreboards the ring traffic uses, so deep input prefetch never stalls the math.
template <int BYTES>
__device__ __forceinline__ void cp_async(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// --------------------------------------------------------------------------- V: lines are columns
// 12 slots = AHEAD rows in flight + the U rows being consumed: with 16 the W = 2, P = 5, r = 13 kernel needs 38.5 KB per CTA and only 5 CTAs
// fit an SM; 12 slots bring it to 37.6 KB = 6 CTAs (the kernel is bound by resident warps).
template <int NT, int W> struct VStage { static constexpr int AHEAD = 8, SLOTS = 12, WORDS = SLOTS * NT * W; };

template <typename T, int P, int MODE, int NT, int W>
__global__ void __launch_bounds__(NT) blur_v_kernel(const BatchJob job, const AxisParams ap) {
    extern __shared__ uint32_t smem[];
    constexpr int NL = Px<T>::NL;
    using Pipe = LinePipe<T, P, MODE, NT, W>;
    using V = Vec<W>;
    using ST = VStage<NT, W>;
    int local;
    const PlaneJob& pj = find_plane(job, blockIdx.y, local);
    const int g = local * NT + threadIdx.x;  // (32*W)-bit column group
    if (g * NL * W >= pj.w) return;           // no block-level sync in this kernel
    const char* src = job.src + (size_t)blockIdx.x * job.src_fs + pj.src_off + (size_t)g * 4 * W;
    char* dst = job.dst + (size_t)blockIdx.x * job.dst_fs + pj.dst_off + (size_t)g * 4 * W;
    const int sp = pj.src_pitch, dp = pj.dst_pitch;

    uint32_t* stage = smem + threadIdx.x * W;               // [SLOTS][NT] input rows in flight
    Pipe pipe;
    pipe.start(smem + ST::WORDS + threadIdx.x * W, pj.h, ap);
    const int n = pj.h, lag = pipe.lag(), total = n + lag;
    const int t_fast = min(pipe.fast_begin(), n);

    // one commit group per input row, AHEAD rows in flight
    auto slot_at = [&](int sl) -> V& { return *reinterpret_cast<V*>(stage + sl * (NT * W)); };
    auto staged = [&](int row) -> V& { return slot_at((int)((unsigned)row % (unsigned)ST::SLOTS)); };
    auto fetch = [&](int row) {
        cp_async<4 * W>(&staged(row), src + (size_t)min(row, n - 1) * sp);
        cp_async_commit();
    };
    auto store = [&](int x, const V& v) { *reinterpret_cast<V*>(dst + (size_t)x * dp) = v; };
#pragma unroll
    for (int i = 0; i < ST::AHEAD; ++i) fetch(i);

    int t = 0;
    const bool phased = (n >= pipe.fast_begin());
    if (phased) {
        // start-up: phase k has exactly k live stages (compile-time), stage k is seeded on the phase's first step
        static_for<P + 1>([&](auto kc) {
            constexpr int k = decltype(kc)::value;
            const int steps = (k == P) ? 1 : pipe.D;
            for (int j = 0; j < steps; ++j, ++t) {
                fetch(t + ST::AHEAD);
                cp_async_wait<ST::AHEAD>();
                const V v = staged(t);
                V o;
                if (j == 0 && k >= 1) o = pipe.template step_start<k, (k >= 1)>(v);
                else o = pipe.template step_start<k, false>(v);
                if (k == P) store(0, o);
            }
        });
    } else {
        for (; t < t_fast; ++t) {  // tiny lines: generic edge step
            fetch(t + ST::AHEAD);
            cp_async_wait<ST::AHEAD>();
            const V o = pipe.step_edge(t, staged(t));
            const int x = t - lag;
            if (x >= 0 && x < n) store(x, o);
        }
    }
    // steady state: U steps per iteration with running pointers (no per-step 64-bit multiplies, no
    // clamping: every prefetched row is < n here).  U = 4 keeps the loop body inside the L0 i-cache.
    constexpr int U = 4;
    {
        const char* fsrc = src + (size_t)(t + ST::AHEAD) * sp;  // next row to prefetch
        char* fdst = dst + (size_t)(t - lag) * dp;              // next row to store
        int sr = (int)((unsigned)t % (unsigned)ST::SLOTS), sf = (int)((unsigned)(t + ST::AHEAD) % (unsigned)ST::SLOTS);  // running slots
        // 1-3 fused passes are close to memory-bound: an L2 prefetch 24 rows further ahead lets the cp.async find its line
        // in L2 instead of HBM (V1 -6 %, V2 -12 %); with 4-5 passes the kernel is issue-bound and the extra instruction only costs
        constexpr int L2_AHEAD = 24;
        for (; t + ST::AHEAD + U <= n; t += U) {
            if (P <= 3 && t + ST::AHEAD + U + L2_AHEAD <= n) {
#pragma unroll
                for (int i = 0; i < U; ++i) asm volatile("prefetch.global.L2 [%0];" ::"l"(fsrc + (size_t)(L2_AHEAD + i) * sp));
            }
#pragma unroll
            for (int i = 0; i < U; ++i) {
                cp_async<4 * W>(&slot_at(sf), fsrc);
                cp_async_commit();
                fsrc += sp;
                sf = (sf + 1 == ST::SLOTS) ? 0 : sf + 1;
            }
            cp_async_wait<ST::AHEAD>();
#pragma unroll
            for (int i = 0; i < U; ++i) {
                *reinterpret_cast<V*>(fdst) = pipe.step_fast(slot_at(sr));
                fdst += dp;
                sr = (sr + 1 == ST::SLOTS) ? 0 : sr + 1;
            }
        }
    }
    for (; t < n; ++t) {
        fetch(t + ST::AHEAD);
        cp_async_wait<ST::AHEAD>();
        store(t - lag, pipe.step_fast(staged(t)));
    }
    cp_async_wait<0>();
    if (phased) {
        // drain: phase k has producer k in its mirrored tail and stages k+1..P live
        static_for<P>([&](auto kc) {
            constexpr int k = decltype(kc)::value;
            for (int j = 0; j < pipe.D; ++j, ++t) {
                const V o = (j < ap.r) ? pipe.template step_drain<k, true>(j) : pipe.template step_drain<k, false>(0);
                store(t - lag, o);
            }
        });
    } else {
        for (; t < total; ++t) {
            const V o = pipe.step_edge(t, V{});
            const int x = t - lag;
            if (x >= 0 && x < n) store(x, o);
        }
    }
}

// --------------------------------------------------------------------------- H: lines are rows
// CTA = NT threads = NT*NL rows.  Tiles are [position][row] in T units with (NT*NL + PAD) row pitch so
// that both the coalesced side (32 lanes = 32 positions of one row) and the line side (32 lanes = 32
// consecutive row groups) are bank-conflict free.
template <typename T, int NT> struct HTile {
    static constexpr int NL = Px<T>::NL;
    static constexpr int CH = 32;                        // positions per input tile
    static constexpr int OUT = 64;                       // positions in the output ring (two blocks)
    static constexpr int PITCH_W = NT + 1;               // words per position (odd)
    static constexpr int IN_WORDS = CH * PITCH_W;
    static constexpr int OUT_WORDS = OUT * PITCH_W;
};

template <typename T, int P, int NT>
__global__ void __launch_bounds__(NT) blur_h_kernel(const BatchJob job, const AxisParams ap) {
    extern __shared__ uint32_t smem[];
    using TL = HTile<T, NT>;
    using Pipe = LinePipe<T, P, MODE_RT, NT>;
    constexpr int NL = Px<T>::NL;
    constexpr int ROWS = NT * NL;
    constexpr int NWARP = NT / 32;
    int local;
    const PlaneJob& pj = find_plane(job, blockIdx.y, local);
    const int row0 = local * ROWS;
    const int nrows = min(ROWS, pj.h - row0);
    const char* src = job.src + (size_t)blockIdx.x * job.src_fs + pj.src_off + (size_t)row0 * pj.src_pitch;
    char* dst = job.dst + (size_t)blockIdx.x * job.dst_fs + pj.dst_off + (size_t)row0 * pj.dst_pitch;
    const int sp = pj.src_pitch, dp = pj.dst_pitch;

    uint32_t* ring = smem;
    uint32_t* in_tile = ring + ap.ring * P * NT;
    uint32_t* out_tile = in_tile + TL::IN_WORDS;
    T* in_t = reinterpret_cast<T*>(in_tile);
    T* out_t = reinterpret_cast<T*>(out_tile);

    Pipe pipe;
    pipe.start(ring + threadIdx.x, pj.w, ap);
    const int n = pj.w, lag = pipe.lag(), total = n + lag;
    const int t_fast = min(pipe.fast_begin(), n);
    const bool phased = (n >= pipe.fast_begin());

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int flushed = 0;  // output positions [0, flushed) are already in global memory
    const int nchunks = (total + TL::CH - 1) / TL::CH;

    // Input staging: 32-bit coalesced loads of the NEXT 32-position tile are issued before the current
    // tile's math and parked in registers, so their latency is covered by a whole chunk of work; they are
    // scattered (transposed) into shared memory at the top of the next iteration.
    constexpr int EPW = 4 / (int)sizeof(T);      // samples per 32-bit word
    constexpr int WPR = TL::CH / EPW;            // words per row per tile: 8 / 16 / 32
    constexpr int RPI = 32 / WPR;                // rows covered by one warp-wide load
    constexpr int NLD = ROWS / (RPI * NWARP);    // loads per thread per tile
    const int lw = lane % WPR, lr = lane / WPR;
    uint32_t pre[NLD];
    // 16-bit samples, one warp: load i fetches row 4*(i/2) + 2*lr + (i%2), so a thread holds both rows of a packed
    // row pair at the same two positions and the 2x2 transpose happens in registers (2 PRMT + 2 32-bit STS per pair
    // of loads instead of 4 16-bit STS; the same in reverse when flushing).
    // Measured on B200: a gain for 1-2 fused passes (staging dominates), a loss from 3 passes up (register pressure).
    constexpr bool PAIR = (P <= 2 && sizeof(T) == 2 && NWARP == 1);
    auto row_of = [&](int i) { return PAIR ? 4 * (i >> 1) + 2 * lr + (i & 1) : (i * NWARP + warp) * RPI + lr; };
    // generic mapping: row rr_i = (i*NWARP + warp)*RPI + lr, word lw: running 64-bit pointers, one add per load
    const bool full = (nrows == ROWS);
    const char* lsrc = src + (size_t)row_of(0) * sp + (size_t)lw * 4;
    char* ldst = dst + (size_t)row_of(0) * dp + (size_t)lw * 4;
    const size_t lstep_s = (size_t)(NWARP * RPI) * sp, lstep_d = (size_t)(NWARP * RPI) * dp;
    auto issue_loads = [&](int t0) {
        const char* p = lsrc + (size_t)t0 * sizeof(T);
        if (t0 + lw * EPW >= n) return;  // this lane's word lies beyond the line: keeps stale data, never consumed
        if constexpr (PAIR) {
#pragma unroll
            for (int i = 0; i < NLD; i += 2) {
                if (full || row_of(i) < nrows) pre[i] = *reinterpret_cast<const uint32_t*>(p);
                if (full || row_of(i + 1) < nrows) pre[i + 1] = *reinterpret_cast<const uint32_t*>(p + sp);
                p += 4 * (size_t)sp;
            }
        } else if (full) {
#pragma unroll
            for (int i = 0; i < NLD; ++i) { pre[i] = *reinterpret_cast<const uint32_t*>(p); p += lstep_s; }
        } else {
#pragma unroll
            for (int i = 0; i < NLD; ++i) {
                if (row_of(i) < nrows) pre[i] = *reinterpret_cast<const uint32_t*>(p);
                p += lstep_s;
            }
        }
    };
#pragma unroll
    for (int i = 0; i < NLD; ++i) pre[i] = 0u;
    issue_loads(0);

    for (int c = 0; c < nchunks; ++c) {
        const int t0 = c * TL::CH;
        // ---- scatter the prefetched tile (positions [t0, t0+32) of every row) and prefetch the next one
        if constexpr (PAIR) {
#pragma unroll
            for (int i = 0; i < NLD; i += 2) {
                const int tw = (i >> 1) * 2 + lr;  // the thread that owns rows (row_of(i), row_of(i) + 1)
                in_tile[(lw * 2) * TL::PITCH_W + tw] = __byte_perm(pre[i], pre[i + 1], 0x5410);
                in_tile[(lw * 2 + 1) * TL::PITCH_W + tw] = __byte_perm(pre[i], pre[i + 1], 0x7632);
            }
        } else {
#pragma unroll
            for (int i = 0; i < NLD; ++i) {
                const int rr = row_of(i);
                const T* e = reinterpret_cast<const T*>(&pre[i]);
#pragma unroll
                for (int k = 0; k < EPW; ++k) in_t[((lw * EPW + k) * TL::PITCH_W) * NL + rr] = e[k];
            }
        }
        if (t0 + TL::CH < n) issue_loads(t0 + TL::CH);
        __syncthreads();
        // ---- every thread advances its own rows by up to 32 steps
        const int t1 = min(t0 + TL::CH, total);
        if (t0 >= t_fast && t1 <= n) {
            // whole tile in the steady state: no per-step branches, unrolled so the look-ahead rotation is free
            const int x0 = t0 - lag;  // >= 1
#pragma unroll 4
            for (int i = 0; i < TL::CH; ++i)
                out_tile[((x0 + i) & (TL::OUT - 1)) * TL::PITCH_W + threadIdx.x] = pipe.step_fast(Vec<1>{{in_tile[i * TL::PITCH_W + threadIdx.x]}}).v[0];
        } else {
            auto in = [&](int t) { return Vec<1>{{in_tile[(t - t0) * TL::PITCH_W + threadIdx.x]}}; };
            auto out = [&](int t, const Vec<1>& o) {
                const int x = t - lag;
                if (x >= 0 && x < n) out_tile[(x & (TL::OUT - 1)) * TL::PITCH_W + threadIdx.x] = o.v[0];
            };
            if (phased) {
                pipe.run_steps(t0, t1, in, out);
            } else {
                for (int t = t0; t < t1; ++t) {
                    if (t >= t_fast && t < n) out(t, pipe.step_fast(in(t)));
                    else out(t, pipe.step_edge(t, in(t)));
                }
            }
        }
        __syncthreads();
        // ---- flush every complete 32-position output block (and the tail at the very end)
        const int produced = min(max(t1 - lag, 0), n);
        const int upto = (t1 == total) ? n : (produced / 32) * 32;
        for (int xb = flushed; xb < upto; xb += 32) {
            // one 32-bit store per EPW samples, same lane->(row, word) mapping as the loads
            const int x = xb + lw * EPW;
            char* q = ldst + (size_t)xb * sizeof(T);
            if (full && xb + 32 <= upto) {
                // common case (full CTA, complete block): branch-free, all shared-memory reads issued before the stores
                uint32_t wv[NLD];
                if constexpr (PAIR) {
#pragma unroll
                    for (int i = 0; i < NLD; i += 2) {
                        const int tw = (i >> 1) * 2 + lr;
                        const uint32_t o0 = out_tile[(x & (TL::OUT - 1)) * TL::PITCH_W + tw];
                        const uint32_t o1 = out_tile[((x + 1) & (TL::OUT - 1)) * TL::PITCH_W + tw];
                        wv[i] = __byte_perm(o0, o1, 0x5410);
                        wv[i + 1] = __byte_perm(o0, o1, 0x7632);
                    }
#pragma unroll
                    for (int i = 0; i < NLD; i += 2) {
                        *reinterpret_cast<uint32_t*>(q) = wv[i];
                        *reinterpret_cast<uint32_t*>(q + dp) = wv[i + 1];
                        q += 4 * (size_t)dp;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < NLD; ++i) {
                        const int rr = row_of(i);
                        T e[EPW];
#pragma unroll
                        for (int k = 0; k < EPW; ++k) e[k] = out_t[(((x + k) & (TL::OUT - 1)) * TL::PITCH_W) * NL + rr];
                        wv[i] = *reinterpret_cast<const uint32_t*>(e);
                    }
#pragma unroll
                    for (int i = 0; i < NLD; ++i) { *reinterpret_cast<uint32_t*>(q) = wv[i]; q += lstep_d; }
                }
            } else if (x < upto) {
                const bool whole = (x + EPW <= upto);
#pragma unroll 4
                for (int i = 0; i < NLD; ++i) {
                    const int rr = row_of(i);
                    char* qi = PAIR ? dst + (size_t)rr * dp + (size_t)lw * 4 + (size_t)xb * sizeof(T) : q;
                    if (rr < nrows) {
                        T e[EPW];
#pragma unroll
                        for (int k = 0; k < EPW; ++k) e[k] = out_t[(((x + k) & (TL::OUT - 1)) * TL::PITCH_W) * NL + rr];
                        if (whole) {
                            *reinterpret_cast<uint32_t*>(qi) = *reinterpret_cast<const uint32_t*>(e);
                        } else {
                            for (int k = 0; k < EPW && x + k < upto; ++k) reinterpret_cast<T*>(qi)[k] = e[k];
                        }
                    }
                    q += lstep_d;
                }
            }
        }
        flushed = max(flushed, upto);
        // the next iteration's __syncthreads (after its load) orders these reads before new out_tile writes
    }
}

// --------------------------------------------------------------------------- comptime float path
// Direct tap-ordered sums with R101q indexing (src/filters/boxblur_comptime.zig:161-263):
// acc = 0; for k in 0..2r: acc = acc + div * v_k; narrowed to T.  One thread per output sample.
__device__ __forceinline__ int r101q(int i, int k, int r, int n) {
    if (k < r) {
        const int need = r - k;
        return (i < need) ? min(need - i, n - 1) : i - need;
    }
    const int over = k - r, room = n - 1 - i;
    return (room < over) ? i - min(over - room, i) : i + over;
}

template <typename T> __device__ __forceinline__ float ld_f(const T* p) { return (float)*p; }
template <> __device__ __forceinline__ float ld_f<__half>(const __half* p) { return __half2float(*p); }
template <typename T> __device__ __forceinline__ T st_f(float v);
template <> __device__ __forceinline__ float st_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __half st_f<__half>(float v) { return __float2half_rn(v); }

// Tiled version.  "Line axis" = the blurred direction (y for the V pass, x for the H pass), "cross axis" the
// other one.  A CTA of 128 threads owns 128 cross positions x TL line positions.  The products div*v of the
// TL + 2r line positions it needs are staged once in shared memory as [line][cross] (pitch 129: the H pass
// fills it with lanes along the line axis, every pass reads it with lanes along the cross axis, both
// conflict-free).  A thread then produces its line in groups of 4 outputs that share one sweep over 2r+4
// products, each output adding its 2r+1 products in tap order (acc = 0 + m0 + m1 + ...): bit-exact.
// Edge outputs (within r of either end) take the generic R101q tap loop.
static constexpr int CTF_NT = 128, CTF_TL = 32, CTF_PITCH = 129;

template <typename T, bool HORIZ>
__global__ void __launch_bounds__(CTF_NT) ctf_kernel(const BatchJob job, int r, float div, int3 line_blocks) {
    extern __shared__ float ctf_smem[];
    int local;
    const PlaneJob& pj = find_plane(job, blockIdx.x, local);
    const int k = (int)(&pj - job.pl);
    const int nlb = k == 0 ? line_blocks.x : (k == 1 ? line_blocks.y : line_blocks.z);
    const int lb = local % nlb, cb = local / nlb;
    const int n = HORIZ ? pj.w : pj.h, ncross = HORIZ ? pj.h : pj.w;
    const int l0 = lb * CTF_TL, l1 = min(l0 + CTF_TL, n);
    const int c0 = cb * CTF_NT;
    const int lo = max(l0 - r, 0), hi = min(l1 - 1 + r, n - 1), cnt = hi - lo + 1;
    const char* src = job.src + (size_t)blockIdx.y * job.src_fs + pj.src_off;
    char* dst = job.dst + (size_t)blockIdx.y * job.dst_fs + pj.dst_off;
    float* P = ctf_smem;                               // [cnt][129] products
    const int c = threadIdx.x;
    const bool live = (c0 + c) < ncross;

    if constexpr (!HORIZ) {
        // every thread stages (and later reads) only its own column: no barrier needed
        if (live) {
            const char* col = src + (size_t)lo * pj.src_pitch + (size_t)(c0 + c) * sizeof(T);
            int j = 0;
            for (; j + 8 <= cnt; j += 8) {  // 8 independent loads in flight per thread
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = ld_f<T>(reinterpret_cast<const T*>(col + (size_t)(j + u) * pj.src_pitch));
#pragma unroll
                for (int u = 0; u < 8; ++u) P[(j + u) * CTF_PITCH + c] = __fmul_rn(div, v[u]);
            }
            for (; j < cnt; ++j) P[j * CTF_PITCH + c] = __fmul_rn(div, ld_f<T>(reinterpret_cast<const T*>(col + (size_t)j * pj.src_pitch)));
        }
    } else {
        const int lane = c & 31, warp = c >> 5;
        // 4 rows x up to 4 lane-strided segments = up to 16 independent loads in flight per thread
        for (int rr0 = warp * 4; rr0 < CTF_NT; rr0 += CTF_NT / 8) {
            float v[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int rr = min(rr0 + u, CTF_NT - 1);
                const T* row = reinterpret_cast<const T*>(src + (size_t)min(c0 + rr, ncross - 1) * pj.src_pitch) + lo;
#pragma unroll
                for (int s2 = 0; s2 < 4; ++s2) v[u][s2] = ld_f<T>(row + min(lane + 32 * s2, cnt - 1));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int s2 = 0; s2 < 4; ++s2)
                    if (lane + 32 * s2 < cnt) P[(lane + 32 * s2) * CTF_PITCH + rr0 + u] = __fmul_rn(div, v[u][s2]);
        }
        __syncthreads();
    }

    if (live) {
        const float* Pc = P + c;
        // four results of one line leave as a vector (H: the thread owns row c0 + c; the other half of the 32-byte
        // sector follows with the next group, so L2 merges them) or as four coalesced row stores (V)
        auto emit4 = [&](int i0, float r0, float r1, float r2, float r3) {
            const float res[4] = {r0, r1, r2, r3};
            if constexpr (HORIZ) {
                T* out = reinterpret_cast<T*>(dst + (size_t)(c0 + c) * pj.dst_pitch) + i0;
                if (i0 + 3 < l1) {
                    if constexpr (sizeof(T) == 4) {
                        *reinterpret_cast<float4*>(out) = make_float4(res[0], res[1], res[2], res[3]);
                    } else {
                        const __half2 h01 = __floats2half2_rn(res[0], res[1]), h23 = __floats2half2_rn(res[2], res[3]);
                        uint2 pk;
                        pk.x = *reinterpret_cast<const uint32_t*>(&h01); pk.y = *reinterpret_cast<const uint32_t*>(&h23);
                        *reinterpret_cast<uint2*>(out) = pk;
                    }
                } else {
                    for (int g = 0; g < 4 && i0 + g < l1; ++g) out[g] = st_f<T>(res[g]);
                }
            } else {
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const int i = i0 + g;
                    if (i < l1) reinterpret_cast<T*>(dst + (size_t)i * pj.dst_pitch)[c0 + c] = st_f<T>(res[g]);
                }
            }
        };
        // outputs i0 .. i0+3: one sweep over products i0-r .. i0+3+r, each output adding its 2r+1 taps in tap order
        auto group4 = [&](int i0) {
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
            const bool interior4 = (i0 >= r) && (i0 + 3 + r < n) && (i0 + 3 < l1);
            if (interior4) {
                const float* q = Pc + (i0 - r - lo) * CTF_PITCH;
                const int m = 2 * r;  // output g adds products g .. g + 2r of this sweep
                float v = q[0]; a0 = __fadd_rn(a0, v);
                v = q[CTF_PITCH]; a0 = __fadd_rn(a0, v); a1 = __fadd_rn(a1, v);
                v = q[2 * CTF_PITCH]; a0 = __fadd_rn(a0, v); a1 = __fadd_rn(a1, v); a2 = __fadd_rn(a2, v);
                q += 3 * CTF_PITCH;
                for (int t = 3; t <= m; ++t, q += CTF_PITCH) {
                    v = q[0];
                    a0 = __fadd_rn(a0, v); a1 = __fadd_rn(a1, v); a2 = __fadd_rn(a2, v); a3 = __fadd_rn(a3, v);
                }
                // t = m+1, m+2, m+3 (for r == 1, m = 2: the loop above did not run and a0 is already complete)
                v = q[0]; a1 = __fadd_rn(a1, v); a2 = __fadd_rn(a2, v); a3 = __fadd_rn(a3, v);
                v = q[CTF_PITCH]; a2 = __fadd_rn(a2, v); a3 = __fadd_rn(a3, v);
                v = q[2 * CTF_PITCH]; a3 = __fadd_rn(a3, v);
            } else {
                float* acc[4] = {&a0, &a1, &a2, &a3};
                for (int g = 0; g < 4 && i0 + g < l1; ++g) {
                    float a = 0.f;
                    const int i = i0 + g;
                    for (int t = 0; t <= 2 * r; ++t) a = __fadd_rn(a, Pc[(r101q(i, t, r, n) - lo) * CTF_PITCH]);
                    *acc[g] = a;
                }
            }
            emit4(i0, a0, a1, a2, a3);
        };
        // outputs i0 .. i0+7 away from the edges, r >= 4: every product is read once per 8 outputs
        auto group8 = [&](int i0) {
            float a[8];
#pragma unroll
            for (int g = 0; g < 8; ++g) a[g] = 0.f;
            const float* q = Pc + (i0 - r - lo) * CTF_PITCH;
            const int m = 2 * r;  // >= 8
#pragma unroll
            for (int t = 0; t < 7; ++t) {  // products 0..6: output g takes product t iff g <= t
                const float v = q[t * CTF_PITCH];
#pragma unroll
                for (int g = 0; g < 8; ++g) if (g <= t) a[g] = __fadd_rn(a[g], v);
            }
            q += 7 * CTF_PITCH;
            for (int t = 7; t <= m; ++t, q += CTF_PITCH) {
                const float v = q[0];
#pragma unroll
                for (int g = 0; g < 8; ++g) a[g] = __fadd_rn(a[g], v);
            }
#pragma unroll
            for (int u = 1; u <= 7; ++u) {  // products m+1..m+7: output g takes product m+u iff g >= u
                const float v = q[(u - 1) * CTF_PITCH];
#pragma unroll
                for (int g = 0; g < 8; ++g) if (g >= u) a[g] = __fadd_rn(a[g], v);
            }
            emit4(i0, a[0], a[1], a[2], a[3]);
            emit4(i0 + 4, a[4], a[5], a[6], a[7]);
        };
        for (int i0 = l0; i0 < l1; i0 += 8) {
            if (r >= 4 && i0 >= r && i0 + 7 + r < n && i0 + 7 < l1) {
                group8(i0);
            } else {
                group4(i0);
                if (i0 + 4 < l1) group4(i0 + 4);
            }
        }
    }
}

// =========================================================================== host-side launchers
static AxisParams axis_params(int r) {
    AxisParams a{};
    a.r = r;
    a.ring = 2 * r + 1;
    axis_consts(r, a.inv, a.inv2);
    a.div = 1.0f / (float)(2 * r + 1);
    return a;
}

#ifndef VSZ_NT_V
#define VSZ_NT_V 64
#endif
#ifndef VSZ_NT_H
#define VSZ_NT_H 32
#endif
static constexpr int NT_V = VSZ_NT_V;
static constexpr int NT_H = VSZ_NT_H;

#ifndef VSZ_V_WORDS
#define VSZ_V_WORDS 2
#endif
static constexpr int V_W = VSZ_V_WORDS, V_NT = NT_V / V_W;  // same shared memory per CTA for W = 1 and W = 2

// dynamic shared memory of blur_v_kernel / blur_h_kernel with P fused passes at radius r: one 2r+1-slot delay ring per pass and
// thread, then the input stage (V) or the input and output tiles (H)
static size_t v_smem(int r, int P) { return ((size_t)(2 * r + 1) * P * V_NT * V_W + VStage<V_NT, V_W>::WORDS) * 4; }
template <typename T>
static size_t h_smem(int r, int P) { return ((size_t)(2 * r + 1) * P * NT_H + HTile<T, NT_H>::IN_WORDS + HTile<T, NT_H>::OUT_WORDS) * 4; }

template <typename T, int P, int MODE>
static int launch_v(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs,
                    int count, int r, cudaStream_t st) {
    constexpr int NL = Px<T>::NL;
    const BatchJob job = make_batch(l, mask, src, src_fs, nullptr, 0, dst, dst_fs,
                                    [](int w, int) { return ((w + NL * V_W - 1) / (NL * V_W) + V_NT - 1) / V_NT; });
    return launch_frames(blur_v_kernel<T, P, MODE, V_NT, V_W>, job, count, V_NT, v_smem(r, P), st, axis_params(r));
}

template <typename T, int P>
static int launch_h(const FrameLayout& l, const bool mask[3], const char* src, size_t src_fs, char* dst, size_t dst_fs,
                    int count, int r, cudaStream_t st) {
    constexpr int NL = Px<T>::NL;
    const BatchJob job = make_batch(l, mask, src, src_fs, nullptr, 0, dst, dst_fs,
                                    [](int, int h) { return (h + NT_H * NL - 1) / (NT_H * NL); });
    return launch_frames(blur_h_kernel<T, P, NT_H>, job, count, NT_H, h_smem<T>(r, P), st, axis_params(r));
}

// largest number of passes one launch can fuse for this radius (shared-memory bound), at most 5
template <typename T, bool H>
static int max_fused(int r) {
    int p = 5;
    while (p > 0 && (H ? h_smem<T>(r, p) : v_smem(r, p)) > (size_t)kMaxSmemPerCta) --p;
    return p;
}

template <typename T, bool H>
static int launch_axis_p(int P, const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs,
                         int count, int r, cudaStream_t st) {
    const int rc = with_constant(std::integer_sequence<int, 1, 2, 3, 4, 5>{}, P, [&](auto passes) {
        if constexpr (H) return launch_h<T, decltype(passes)::value>(l, mask, src, sfs, dst, dfs, count, r, st);
        else return launch_v<T, decltype(passes)::value, MODE_RT>(l, mask, src, sfs, dst, dfs, count, r, st);
    });
    if (rc != 1) return rc;  // launch_h / launch_v return 0 or an error: 1 = P is not in 1..5
    set_error("BoxBlur: internal error, bad fused pass count %d", P);
    return -3;
}

// --------------------------------------------------------------------------- very large radii
// When even one 2r+1-slot delay ring per line does not fit in shared memory (r in the hundreds), a pass is
// run straight from global memory: one thread per packed line group, the reference's own index rules
// (src/filters/boxblur_runtime.zig:24-40), out of place.  Slow (two dependent global reads per step, the
// H direction uncoalesced) but bit-exact; it only exists so that no legal radius is rejected.
template <typename T, bool HORIZ>
__global__ void __launch_bounds__(128) blur_global_kernel(const BatchJob job, const AxisParams ap) {
    using Ops = StageOps<T, MODE_RT>;
    using Acc = typename Px<T>::Acc;
    constexpr int NL = Px<T>::NL;
    int local;
    const PlaneJob& pj = find_plane(job, blockIdx.x, local);
    const int g = local * 128 + threadIdx.x;  // packed line group
    const int n = HORIZ ? pj.w : pj.h, nlines = HORIZ ? pj.h : pj.w;
    if (g * NL >= nlines) return;
    const char* src = job.src + (size_t)blockIdx.y * job.src_fs + pj.src_off;
    char* dst = job.dst + (size_t)blockIdx.y * job.dst_fs + pj.dst_off;
    auto load = [&](int pos) -> uint32_t {
        if constexpr (!HORIZ) return *reinterpret_cast<const uint32_t*>(src + (size_t)pos * pj.src_pitch + (size_t)g * 4);
        T e[NL];
#pragma unroll
        for (int l = 0; l < NL; ++l) e[l] = reinterpret_cast<const T*>(src + (size_t)min(g * NL + l, nlines - 1) * pj.src_pitch)[pos];
        uint32_t w; memcpy(&w, e, 4); return w;
    };
    auto store = [&](int pos, uint32_t w) {
        if constexpr (!HORIZ) { *reinterpret_cast<uint32_t*>(dst + (size_t)pos * pj.dst_pitch + (size_t)g * 4) = w; return; }
        T e[NL]; memcpy(e, &w, 4);
#pragma unroll
        for (int l = 0; l < NL; ++l) if (g * NL + l < nlines) reinterpret_cast<T*>(dst + (size_t)(g * NL + l) * pj.dst_pitch)[pos] = e[l];
    };
    Acc S[NL];
    const int r = ap.r;
    Ops::init(S, ap, load);
    for (int x = 0; x < n; ++x) {
        int ia, ib;
        if (x <= r) { ia = r + x; ib = r - x; }
        else if (x < n - r) { ia = r + x; ib = x - r - 1; }
        else { ia = 2 * n - r - x - 1; ib = x - r - 1; }
        store(x, Ops::update(S, load(ia), load(ib), ap));
    }
}

template <typename T, bool H>
static int launch_global(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int count, int r, cudaStream_t st) {
    constexpr int NL = Px<T>::NL;
    BatchJob job = make_batch(l, mask, src, sfs, nullptr, 0, dst, dfs,
                              [](int w, int h) { return (((H ? h : w) + NL - 1) / NL + 127) / 128; });
    if (job.ctas_per_frame == 0) return 0;
    const AxisParams ap = axis_params(r);
    for (int f0 = 0; f0 < count; f0 += 65535) {
        const int nf = std::min(65535, count - f0);
        BatchJob j = job;
        j.src += (size_t)f0 * sfs; j.dst += (size_t)f0 * dfs;
        blur_global_kernel<T, H><<<dim3(job.ctas_per_frame, nf), 128, 0, st>>>(j, ap);
        count_launch();
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

// `passes` runtime-path passes along one axis.  The first launch reads src, later ones run in place on
// dst (a line is owned by one thread and outputs trail inputs, so in-place is race-free).
template <typename T, bool H>
static int run_axis(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int count,
                    int r, int passes, cudaStream_t st) {
    const int cap = max_fused<T, H>(r);
    if (cap < 1) {
        // out-of-place passes from global memory, ping-ponging two scratch clips so the last pass lands in dst
        AsyncScratch scratch;
        const size_t bytes = l.frame_stride * (size_t)count, tfs = l.frame_stride;
        VSZ_CUDA(scratch.alloc(2 * bytes, st));
        char* t1 = scratch.p;
        char* t2 = t1 + bytes;
        const char* cur = src;
        size_t cur_fs = sfs;
        int rc = 0;
        for (int p = 1; p <= passes && !rc; ++p) {
            char* out = (p == passes && cur != dst) ? dst : ((p & 1) ? t1 : t2);
            const size_t ofs = (out == dst) ? dfs : tfs;
            rc = launch_global<T, H>(l, mask, cur, cur_fs, out, ofs, count, r, st);
            cur = out; cur_fs = ofs;
        }
        if (!rc && cur != dst) {  // single pass whose input was dst itself: copy the result back plane by plane
            for (int f = 0; f < count && !rc; ++f)
                for (int pl = 0; pl < l.nplanes; ++pl)
                    if (mask[pl] && cudaMemcpyAsync(dst + (size_t)f * dfs + l.pl[pl].offset, cur + (size_t)f * cur_fs + l.pl[pl].offset,
                                                    (size_t)l.pl[pl].pitch * l.pl[pl].h, cudaMemcpyDeviceToDevice, st) != cudaSuccess) rc = -1;
        }
        return rc;
    }
    const char* cur = src;
    size_t cur_fs = sfs;
    while (passes > 0) {
        const int p = passes < cap ? passes : cap;
        const int rc = launch_axis_p<T, H>(p, l, mask, cur, cur_fs, dst, dfs, count, r, st);
        if (rc) return rc;
        cur = dst; cur_fs = dfs;
        passes -= p;
    }
    return 0;
}

template <typename T>
static int run_ct_float(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* tmp, size_t tfs, char* dst,
                        size_t dfs, int count, int r, cudaStream_t st) {
    const float div = 1.0f / (float)(2 * r + 1);
    auto blocks = [](int len) { return (len + CTF_TL - 1) / CTF_TL; };
    auto cross = [](int len) { return (len + CTF_NT - 1) / CTF_NT; };
    BatchJob jv = make_batch(l, mask, src, sfs, nullptr, 0, tmp, tfs, [&](int w, int h) { return blocks(h) * cross(w); });
    BatchJob jh = make_batch(l, mask, tmp, tfs, nullptr, 0, dst, dfs, [&](int w, int h) { return blocks(w) * cross(h); });
    if (jv.ctas_per_frame == 0) return 0;
    int3 lbv = make_int3(1, 1, 1), lbh = make_int3(1, 1, 1);
    for (int k = 0; k < jv.nplanes; ++k) {
        (k == 0 ? lbv.x : (k == 1 ? lbv.y : lbv.z)) = blocks(jv.pl[k].h);
        (k == 0 ? lbh.x : (k == 1 ? lbh.y : lbh.z)) = blocks(jh.pl[k].w);
    }
    const size_t smem_v = (size_t)(CTF_TL + 2 * r) * CTF_PITCH * sizeof(float);
    const size_t smem_h = smem_v;  // the H pass stores its outputs straight from registers
    VSZ_CUDA(allow_max_dynamic_smem(ctf_kernel<T, false>));
    VSZ_CUDA(allow_max_dynamic_smem(ctf_kernel<T, true>));
    for (int f0 = 0; f0 < count; f0 += 65535) {
        const int nf = std::min(65535, count - f0);
        BatchJob a = jv, b = jh;
        a.src += (size_t)f0 * sfs; a.dst += (size_t)f0 * tfs;
        b.src += (size_t)f0 * tfs; b.dst += (size_t)f0 * dfs;
        ctf_kernel<T, false><<<dim3(jv.ctas_per_frame, nf), CTF_NT, smem_v, st>>>(a, r, div, lbv);
        ctf_kernel<T, true><<<dim3(jh.ctas_per_frame, nf), CTF_NT, smem_h, st>>>(b, r, div, lbh);
        count_launch(2);
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

// 8- and 16-bit integer clips take the segment kernels (boxblur_seg_{h,v,ct}.cu) where they apply
template <typename T, bool H>
static int run_axis_any(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int count, int r,
                        int passes, cudaStream_t st) {
    if constexpr (std::is_same<T, uint16_t>::value || std::is_same<T, uint8_t>::value) {
        const int rc = H ? run_seg_h(l, mask, src, sfs, dst, dfs, count, r, passes, st)
                         : run_seg_v(l, mask, src, sfs, dst, dfs, count, r, passes, st);
        if (rc <= 0) return rc;  // done, or a CUDA error; 1 = nothing launched
    }
    return run_axis<T, H>(l, mask, src, sfs, dst, dfs, count, r, passes, st);
}

template <typename T>
static int run_boxblur_t(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int count,
                         int hr, int hp, int vr, int vp, cudaStream_t st) {
    // dispatch rule of src/vapoursynth/boxblur.zig:188
    const bool use_rt = (hr != vr) || (hr > 22) || (hp > 1) || (vp > 1);
    if (use_rt) {
        const bool hb = hr > 0 && hp > 0, vb = vr > 0 && vp > 0;
        // "all H passes, then all V passes" (boxblur.zig:93-112), V in place on dst
        if (hb) { const int rc = run_axis_any<T, true>(l, mask, src, sfs, dst, dfs, count, hr, hp, st); if (rc) return rc; }
        if (vb) return run_axis_any<T, false>(l, mask, hb ? dst : src, hb ? dfs : sfs, dst, dfs, count, vr, vp, st);
        return 0;
    }
    if constexpr (Px<T>::flt) {
        AsyncScratch tmp;
        VSZ_CUDA(tmp.alloc(l.frame_stride * (size_t)count, st));
        // streaming accumulators (boxblur_ctf.cu); planes smaller than the window keep the tiled kernel
        const int rc = run_ctf_stream(l, mask, src, sfs, tmp.p, l.frame_stride, dst, dfs, count, hr, st);
        if (rc <= 0) return rc;
        return run_ct_float<T>(l, mask, src, sfs, tmp.p, l.frame_stride, dst, dfs, count, hr, st);
    } else {
        // comptime integer path: exact R101q column sums + rounded mean, then the SYM H pass
        if constexpr (std::is_same<T, uint16_t>::value || std::is_same<T, uint8_t>::value) {
            const int rc = run_seg_ct(l, mask, src, sfs, dst, dfs, count, hr, st);  // one read, one write
            if (rc <= 0) return rc;
        }
        int rc = launch_v<T, 1, MODE_CTV>(l, mask, src, sfs, dst, dfs, count, hr, st);
        if (rc) return rc;
        return launch_h<T, 1>(l, mask, dst, dfs, dst, dfs, count, hr, st);
    }
}

int run_boxblur(const FrameLayout& l, const bool mask[3], const char* src, size_t sfs, char* dst, size_t dfs, int count, int hr,
                int hp, int vr, int vp, cudaStream_t st) {
    switch (l.kind) {
        case K_U8: return run_boxblur_t<uint8_t>(l, mask, src, sfs, dst, dfs, count, hr, hp, vr, vp, st);
        case K_U16: return run_boxblur_t<uint16_t>(l, mask, src, sfs, dst, dfs, count, hr, hp, vr, vp, st);
        case K_F16: return run_boxblur_t<__half>(l, mask, src, sfs, dst, dfs, count, hr, hp, vr, vp, st);
        case K_F32: return run_boxblur_t<float>(l, mask, src, sfs, dst, dfs, count, hr, hp, vr, vp, st);
    }
    return -1;
}

}  // namespace vsz
