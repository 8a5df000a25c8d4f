// pcl_nn.cuh -- the nearest-neighbour arithmetic shared by pcl_knn.cu (kNN, ball query) and pcl_icp.cu (ICP's K = 1
// search), so that their distances and tie rule stay bit-identical.
#pragma once
#include "pcl_common.cuh"

namespace pcl {

// The key of a (distance, index) candidate: the distance's bits in the upper half (for +0, positive, +inf and NaN the
// unsigned order is the float order; every NaN becomes 0x7fffffff, ranked after +inf), the index in the lower half.
__device__ __forceinline__ unsigned long long knn_key(float d, int j) {
    const unsigned b = (d != d) ? 0x7fffffffu : __float_as_uint(d);
    return ((unsigned long long)b << 32) | (unsigned)j;
}
__device__ __forceinline__ float key_dist(unsigned long long k) { return __uint_as_float((unsigned)(k >> 32)); }  // ~0 -> NaN

// the Chamfer arithmetic (sqdist3 / chamfer_nnD_kernel of pcl_chamfer.cu): d = 0; per channel d = d + df*df or fma(df, df, d)
template <bool FMA, int D>
__device__ __forceinline__ float sqdist(const float (&q)[D], const float *t) {
    float d = 0.f;
#pragma unroll
    for (int c = 0; c < D; c++) {
        const float df = __fsub_rn(q[c], t[c]);
        if constexpr (FMA) d = __fmaf_rn(df, df, d);
        else d = __fadd_rn(d, __fmul_rn(df, df));
    }
    return d;
}

}  // namespace pcl
