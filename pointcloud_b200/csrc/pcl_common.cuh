// pcl_common.cuh -- shared helpers for libpcl_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/pcl.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libpcl_b200 is written for sm_100a (B200) only"
#endif

namespace pcl {

// thread-local last error text (pcl_last_error)
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);

#define PCL_CUDA(call)                                        \
    do {                                                      \
        cudaError_t _e = (call);                              \
        if (_e != cudaSuccess) return pcl::cuda_fail(_e, #call); \
    } while (0)

struct DeviceInfo {
    int sm_count, cc_major, cc_minor, max_smem_optin;
};
int device_info(DeviceInfo *out);  // cached per device

// A strided (B, P, D) point array of fp32 / fp16 / bf16 elements.
struct Pts {
    const void *p;
    int64_t bs, rs;  // element strides
    int dtype;
};

template <int DT>
__device__ __forceinline__ float ld_elem(const void *p, int64_t i) {
    if constexpr (DT == PCL_F32) return __ldg(reinterpret_cast<const float *>(p) + i);
    else if constexpr (DT == PCL_F16) return __half2float(__ldg(reinterpret_cast<const __half *>(p) + i));
    else return __bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16 *>(p) + i));
}

// runtime-dtype element load (used in staging loops that are not on the critical path)
__device__ __forceinline__ float ld_any(const Pts &a, int64_t i) {
    if (a.dtype == PCL_F32) return ld_elem<PCL_F32>(a.p, i);
    if (a.dtype == PCL_F16) return ld_elem<PCL_F16>(a.p, i);
    return ld_elem<PCL_BF16>(a.p, i);
}

__device__ __forceinline__ float3 ld_xyz(const Pts &a, int64_t b, int64_t row) {
    const int64_t o = b * a.bs + row * a.rs;
    return make_float3(ld_any(a, o), ld_any(a, o + 1), ld_any(a, o + 2));
}

// length of cloud n (len nullable: P), clamped to [0, P]: pytorch3d raises on lengths > P; a kernel cannot, but it must not
// read past the cloud
__device__ __forceinline__ int len_of(const int64_t *len, int n, int P) {
    if (!len) return P;
    const int64_t v = len[n];
    return (int)(v < 0 ? 0 : (v > P ? P : v));
}

// Chamfer backward with the upstream gradients either on the device (grad_out != nullptr) or as immediates (pcl_chamfer.cu)
int chamfer_bwd_impl(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len, const void *y, int y_dtype,
                     int64_t y_bs, int64_t y_rs, const int64_t *y_len, int B, int P1, int P2, int D, const int32_t *idx_x,
                     const int32_t *idx_y, const float *grad_out, float g_imm_x, float g_imm_y, float *grad_x, float *grad_y,
                     cudaStream_t st, bool outputs_are_zero = false);  // outputs_are_zero: the caller has zero-filled grad_x / grad_y on `st` already

// pcl_emd_fwd_fused with a say on the worker launch of the ticket path (pcl_emd.cu)
enum { EMD_WORKERS_AUTO = 0, EMD_WORKERS_NONE_DEDICATED = 1 };
int emd_fwd_fused_impl(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1, const void *xyz2, int dtype2, int64_t bs2, int64_t rs2, int B,
                       int N, float eps, int iters, float *dist, int32_t *assignment, int32_t *stats, float grad_scale, float *grad_xyz1,
                       float *sums, void *workspace, size_t workspace_bytes, void *stream, int worker_policy);

static inline bool dtype_ok(int dt) { return dt == PCL_F32 || dt == PCL_F16 || dt == PCL_BF16; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace pcl
