// gp_epilogue.cuh — device helpers shared by the dense epilogue (gp_epilogue.cu) and the feature-store gather
// (gp_fstore.cu): the value of a reached column and the x half of concat_into_features.
#pragma once

#include "gp_common.cuh"

#ifdef __CUDACC__

// Reference value convention (utils.py:72-76): 1/len(path) = 1/(d+1) in IEEE fp32.
static __device__ __forceinline__ float inv_hops(u32 d)
{
    return __fdiv_rn(1.0f, __uint2float_rn(d + 1u));
}

// concat_into_features' copy of one x row (utils.py:133-134) by a warp: out[0:F] = x[0:F].  The loads of a
// chunk are all issued before its stores — written as `o4[i] = x4[i]` the compiler must assume the two rows
// alias and keeps ONE 512-byte load in flight per warp, which left the epilogue at 65 % of the HBM peak.
// Streaming loads / stores: both rows are touched once.
static __device__ __forceinline__ void copy_x_row(const float *xrow, float *orow, int f, int lane, int vec_x)
{
    constexpr int T = 4;  // float4 loads in flight per lane
    if (vec_x) {
        const float4 *x4 = reinterpret_cast<const float4 *>(xrow);
        float4 *o4 = reinterpret_cast<float4 *>(orow);
        const int q = f >> 2;
        for (int i0 = 0; i0 < q; i0 += 32 * T) {
            float4 v[T];
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const int i = i0 + lane + 32 * t;
                if (i < q) v[t] = __ldcs(x4 + i);
            }
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const int i = i0 + lane + 32 * t;
                if (i < q) __stcs(o4 + i, v[t]);
            }
        }
        for (int i = (q << 2) + lane; i < f; i += 32) orow[i] = __ldcs(xrow + i);
    } else {
        for (int i0 = 0; i0 < f; i0 += 32 * T) {
            float v[T];
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const int i = i0 + lane + 32 * t;
                if (i < f) v[t] = __ldcs(xrow + i);
            }
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const int i = i0 + lane + 32 * t;
                if (i < f) __stcs(orow + i, v[t]);
            }
        }
    }
}

#endif  // __CUDACC__
