// Shared-memory poison and canary for the stale-state tests (tests/test_stale_state_gpu.py).  TEST INFRASTRUCTURE ONLY.
// smem_poison: CTAs of 1024 threads with the device's opt-in maximum of dynamic shared memory fill all of it with a 32-bit
//   pattern and count, per %smid, the CTAs that ran there.  Launched with a few times the SM count of CTAs, every SM runs one.
// smem_peek:   the canary -- the same launch shape reads its dynamic shared memory without writing it and counts, per %smid,
//   the CTAs that found a word other than the pattern.
#include <cuda_runtime.h>
#include <stdint.h>

__device__ __forceinline__ unsigned smid() {
    unsigned v;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(v));
    return v;
}

__device__ __forceinline__ unsigned dynamic_smem_bytes() {
    unsigned v;
    asm volatile("mov.u32 %0, %%dynamic_smem_size;" : "=r"(v));
    return v;
}

__global__ void __launch_bounds__(1024, 1) poison_kernel(uint32_t pattern, unsigned *sm_hits) {
    extern __shared__ __align__(16) uint4 sm[];
    const unsigned n = dynamic_smem_bytes() / 16;
    const uint4 v = make_uint4(pattern, pattern, pattern, pattern);
    for (unsigned i = threadIdx.x; i < n; i += blockDim.x) sm[i] = v;
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(sm_hits + smid(), 1u);
}

__global__ void __launch_bounds__(1024, 1) peek_kernel(uint32_t pattern, unsigned *sm_hits, unsigned *sm_bad) {
    extern __shared__ __align__(16) uint4 sm[];
    const volatile uint4 *vs = sm;
    const unsigned n = dynamic_smem_bytes() / 16;
    bool bad = false;
    for (unsigned i = threadIdx.x; i < n; i += blockDim.x) {
        const uint4 w = make_uint4(vs[i].x, vs[i].y, vs[i].z, vs[i].w);
        bad |= w.x != pattern || w.y != pattern || w.z != pattern || w.w != pattern;
    }
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) {
        atomicAdd(sm_hits + smid(), 1u);
        if (bad) atomicAdd(sm_bad + smid(), 1u);
    }
}

template <typename Kernel>
static int configure(Kernel k, int *smem) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return -1;
    if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, *smem) != cudaSuccess) return -2;
    if (cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, 100) != cudaSuccess) return -3;
    return 0;
}

// sm_hits: unsigned[1024] on the device, indexed by %smid; returns 0 or a negative code (a CUDA call failed)
extern "C" int smem_poison(uint32_t pattern, int ctas, unsigned *sm_hits, void *stream) {
    int smem = 0, rc = configure(poison_kernel, &smem);
    if (rc) return rc;
    poison_kernel<<<ctas, 1024, smem, (cudaStream_t)stream>>>(pattern, sm_hits);
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}

// sm_hits, sm_bad: unsigned[1024] on the device, indexed by %smid
extern "C" int smem_peek(uint32_t pattern, int ctas, unsigned *sm_hits, unsigned *sm_bad, void *stream) {
    int smem = 0, rc = configure(peek_kernel, &smem);
    if (rc) return rc;
    peek_kernel<<<ctas, 1024, smem, (cudaStream_t)stream>>>(pattern, sm_hits, sm_bad);
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}
