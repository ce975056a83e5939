// boxblur_tma.h — tensor maps for the BoxBlur kernels that stage tiles with the TMA engine (boxblur_seg_v.cu, boxblur_ctf.cu).
#pragma once

#include <cuda.h>  // CUtensorMap types only: the encoder comes from cudaGetDriverEntryPoint, libcuda is not linked

#include "common.h"

namespace vsz {

using TensorMapEncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                       const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                       CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled, looked up once; nullptr when the driver does not provide it (the failed query's error is cleared, so
// that it is not reported by the next launch check)
inline TensorMapEncodeFn tensor_map_encoder() {
    static const TensorMapEncodeFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            p = nullptr;
        }
        return reinterpret_cast<TensorMapEncodeFn>(p);
    }();
    return fn;
}

// The [w, h, frames] map of one plane in a chunk of `frames` frames (plane base, row pitch and frame stride in bytes), read in
// boxes of box_w x box_h samples of one frame.  Requires tensor_map_encoder() != nullptr.
inline int encode_plane_map(CUtensorMap* map, CUtensorMapDataType type, const char* plane, int w, int h, int pitch, size_t fs, int frames,
                            int box_w, int box_h) {
    const cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)frames};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch, (cuuint64_t)fs};
    const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, 1}, estr[3] = {1, 1, 1};
    const CUresult rc = tensor_map_encoder()(map, type, 3, const_cast<char*>(plane), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) { set_error("BoxBlur: cuTensorMapEncodeTiled failed (%d)", (int)rc); return -1; }
    return 0;
}

}  // namespace vsz
