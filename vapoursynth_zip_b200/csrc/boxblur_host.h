// boxblur_host.h — host-side helpers shared by the BoxBlur launchers (boxblur_kernels.cu, boxblur_seg_{h,v,ct}.cu, boxblur_ctf.cu).
#pragma once

#include <algorithm>
#include <type_traits>
#include <utility>

#include "common.h"

namespace vsz {

// The radii the segment kernels and the streaming comptime-float kernels are compiled for: every comptime radius.  A/B builds
// (scripts/build_variant.sh, VSZ_SEG_DEV13) compile radius 13 only, which takes seconds.
#ifdef VSZ_SEG_DEV13
using CompiledRadii = std::integer_sequence<int, 13>;
#else
using CompiledRadii = std::integer_sequence<int, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22>;
#endif

// f(std::integral_constant<int, V>{}) for the V of Vs that equals v; 1 when none does
template <int... Vs, class F>
int with_constant(std::integer_sequence<int, Vs...>, int v, F&& f) {
    int rc = 1;
    (void)((v == Vs && ((rc = f(std::integral_constant<int, Vs>{})), true)) || ...);
    return rc;
}

// f at compile-time radius r; 1 (not applicable) for a radius no kernel is compiled for
template <class F>
int with_radius(int r, F&& f) {
    return with_constant(CompiledRadii{}, r, f);
}

// floor((2^32 + r) / (2r+1)) and its top 16 bits: the reference's integer reciprocal of the window size
inline void axis_consts(int r, uint32_t& inv, uint32_t& inv2) {
    const uint64_t v = ((1ull << 32) + (uint64_t)r) / (uint64_t)(2 * r + 1);
    inv = (uint32_t)v;
    inv2 = (uint32_t)(v >> 16);
}

// SMs of the current device, < 0 = error
inline int current_sm_count() {
    int dev = 0, sms = 0;
    VSZ_CUDA(cudaGetDevice(&dev));
    VSZ_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    return sms;
}

// kern<<<(frames, ctas_per_frame), threads, smem>>>(job, args...) over chunks of at most 65535 frames.  Job is a batch descriptor
// with src / dst frame bases and strides.
template <class K, class Job, class... Args>
int launch_frames(K kern, const Job& job, int count, int threads, size_t smem, cudaStream_t st, const Args&... args) {
    VSZ_CUDA(allow_max_dynamic_smem(kern));
    if (job.ctas_per_frame == 0) return 0;
    for (int f0 = 0; f0 < count; f0 += 65535) {
        const int nf = std::min(65535, count - f0);
        Job j = job;
        j.src += (size_t)f0 * job.src_fs; j.dst += (size_t)f0 * job.dst_fs;
        // grid.x = frame, grid.y = CTA within the frame: CTAs are scheduled x-fastest, so every frame's (long) luma CTAs start
        // before any (short) chroma CTA and the tail of the launch is made of short CTAs
        kern<<<dim3(nf, job.ctas_per_frame), threads, smem, st>>>(j, args...);
        count_launch();
    }
    VSZ_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace vsz
