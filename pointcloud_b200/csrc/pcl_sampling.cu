// pcl_sampling.cu -- farthest point sampling and ball query for sm_100a (SURVEY.md 8f rows 1 and 3: the callers on
// the producer side of the loss path -- PointNet2's sample_and_group, models/pointnet2_utils.py:89-144 -- and the
// dataset / sensor sampler, utils.py:86-94).
//
// FPS replaces pointnet2_ops._ext.furthest_point_sampling / pytorch3d.ops.sample_farthest_points (third party, absent):
// start at index 0, keep the running minimum squared distance of every point to the selected set (initial 1e10),
// select the point with the largest running minimum, lowest index on ties -- the torch algorithm the reference keeps
// as a comment (pointnet2_utils.py:64-86).  One thread-block cluster of CS CTAs per cloud (CS = 1, 2, 4, 8, 16); point k
// of the cloud belongs to thread k mod 512 of CTA (k / 512) mod CS, so every CTA gets an equal share of a ragged cloud.
// The points and their running minima stay on chip: PPT <= 16 points per thread in REGISTERS, up to 16 more in shared
// memory (16384 points per CTA, 262144 per cluster of 16).  Per selected point: each warp reduces its lanes with REDUX
// (maximum distance bits, then the lowest index attaining it) and writes its (bits, index, xyz) partial into slot
// [buf][rank][warp] of every CTA of the cluster (distributed shared memory); ONE barrier (__syncthreads for CS = 1,
// barrier.cluster.arrive.release / wait.acquire otherwise); every warp then re-reduces all CS x 16 partials redundantly
// and takes the selected point's xyz from its partial, so no round reads global memory.  The slots are double-buffered:
// a CTA reaches round j+2's writes only after every CTA passed barrier j+1, which each CTA does after reading round j.
// The order-independent selection rule makes the result bit-identical for every CS.
//
// AUTO cluster size (fps_pick_cluster): the smallest CS whose CTAs hold N points (N <= 16384 * CS), doubled while every
// CTA of the doubled cluster still gets at least FPS_AUTO_MIN_CTA_POINTS = 4096 points of the padded width N, the doubled
// cluster has at most FPS_AUTO_MAX_CLUSTER = 8 CTAs and B clusters of it are resident at once (occupancy query); a cloud
// that fits one CTA's registers (N <= 8192) stays on one CTA.
// Splitting a cloud shortens each round's scan but adds the cluster barrier and a longer partial reduction.  Measured on
// a B200 (tools/fps_time.py, profiles/r4_fps_time.txt): a cluster barrier round costs ~0.5 us more than a __syncthreads
// round, so N <= 8192 stays on one CTA (N = 8192: 1.89 ms on one CTA, 2.07 ms on two); the best splits of N = 16384 / 32768 / 65536 leave 4096 / 4096 / 8192 points
// per CTA (clusters of 4 / 8 / 8), and a cluster of 16 is slower than one of 8 wherever 8 holds the cloud (65536 points:
// 3.60 vs 3.09 ms for 2048 samples), so 16 is only taken when N > 131072 needs it.
//
// Ball query replaces query_ball_point (pointnet2_utils.py:93-113, a full sort over N per centroid): one warp per
// centroid scans the cloud in index order with ballot compaction and stops after nsample hits.
#include <cooperative_groups.h>

#include "pcl_common.cuh"

namespace cg = cooperative_groups;

namespace pcl {
namespace {

constexpr int FPS_THREADS = 512;
constexpr int FPS_WARPS = FPS_THREADS / 32;
constexpr int FPS_REG_PPT = 16;                                 // points per thread held in registers
constexpr int FPS_MAX_PPT = 32;                                 // ... plus up to 16 in shared memory
constexpr int FPS_CTA_POINTS = FPS_THREADS * FPS_MAX_PPT;       // 16384
constexpr int FPS_MAX_CLUSTER = 16;                             // non-portable cluster size
constexpr int FPS_MAX_POINTS = FPS_MAX_CLUSTER * FPS_CTA_POINTS;  // 262144
constexpr int FPS_AUTO_MIN_CTA_POINTS = 4096;
constexpr int FPS_AUTO_MAX_CLUSTER = 8;

// dynamic shared memory of an instantiation: x, y, z and the running minimum of the points beyond the registers
constexpr size_t fps_smem_bytes(int ppt) { return ppt > FPS_REG_PPT ? (size_t)(ppt - FPS_REG_PPT) * FPS_THREADS * sizeof(float4) : 0; }

__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// 32-bit shared-memory address kept in a register: without the empty asm the compiler recomputes it from %cgactaid on
// every round, on the path from the barrier to the partial loads
__device__ __forceinline__ unsigned smem_addr(const void *p) {
    unsigned a = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("" : "+r"(a));
    return a;
}
__device__ __forceinline__ int2 lds_int2(unsigned a) {
    int2 v;
    asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float4 lds_float4(unsigned a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}

__device__ __forceinline__ bool at_origin(float3 p) {
    return __fadd_rn(__fadd_rn(__fmul_rn(p.x, p.x), __fmul_rn(p.y, p.y)), __fmul_rn(p.z, p.z)) <= 1e-3f;
}

// A point that can never be selected (index >= n_b, or at the origin with skip_origin) starts with running minimum -1:
// `d < -1` is false for every distance (NaN included), so it stays -1 and never beats `best` (initially -1).
// pad != 0 (pcl_fps_ragged): cloud b runs s_b = min(n_b, k_b) rounds and fills slots s_b..npoint-1 with -1;
// pad == 0 (pcl_fps): npoint rounds on all N points (index 0 repeats once every running minimum is 0).
template <int CS, int PPT>
__global__ void __launch_bounds__(FPS_THREADS)
fps_cluster_kernel(Pts xyz, const int64_t *__restrict__ lengths, int N, const int64_t *__restrict__ K, int npoint, int pad,
                   const int *__restrict__ start, int skip_origin, int *__restrict__ out) {
    constexpr int RPT = PPT < FPS_REG_PPT ? PPT : FPS_REG_PPT, SPT = PPT - RPT;
    constexpr int NP = CS * FPS_WARPS;        // partials per round
    constexpr int STRIDE = CS * FPS_THREADS;  // between the points of one thread
    __shared__ int2 p_key[2][NP];             // (distance bits, index)
    __shared__ float4 p_pos[2][NP];           // xyz of that point
    extern __shared__ float4 s_pts[];         // [SPT][FPS_THREADS]: x, y, z, running minimum
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int rank = CS > 1 ? (int)cg::this_cluster().block_rank() : 0;
    const int cloud = blockIdx.x / CS, g = rank * FPS_THREADS + tid;
    const int n = len_of(lengths, cloud, N);
    int s = npoint;
    if (K) {
        const int64_t k = K[cloud];
        s = (int)(k < 0 ? 0 : (k > npoint ? npoint : k));
    }
    if (pad) s = min(s, n);
    int *o = out + (size_t)cloud * npoint;

    float px[RPT], py[RPT], pz[RPT], mind[RPT];
#pragma unroll
    for (int i = 0; i < RPT; i++) {
        const int k = g + i * STRIDE;
        float3 p = make_float3(0.f, 0.f, 0.f);
        if (s > 0 && k < n) p = ld_xyz(xyz, cloud, k);
        px[i] = p.x; py[i] = p.y; pz[i] = p.z;
        mind[i] = (s > 0 && k < n && !(skip_origin && at_origin(p))) ? 1e10f : -1.f;
    }
#pragma unroll
    for (int i = 0; i < SPT; i++) {
        const int k = g + (RPT + i) * STRIDE;
        float3 p = make_float3(0.f, 0.f, 0.f);
        if (s > 0 && k < n) p = ld_xyz(xyz, cloud, k);
        s_pts[i * FPS_THREADS + tid] = make_float4(p.x, p.y, p.z, (s > 0 && k < n && !(skip_origin && at_origin(p))) ? 1e10f : -1.f);
    }
    int last = 0;
    float3 lp = make_float3(0.f, 0.f, 0.f);
    if (s > 0) {
        last = start ? start[cloud] : 0;
        last = min(max(last, 0), n - 1);
        lp = ld_xyz(xyz, cloud, last);
    }
    if constexpr (CS > 1) cluster_barrier();  // every CTA of the cluster runs before a peer writes into its shared memory
    // shared addresses of this thread's slots, computed once (buffer 1 is NP entries further)
    int2 *const w_key = &p_key[0][rank * FPS_WARPS + wid];
    float4 *const w_pos = &p_pos[0][rank * FPS_WARPS + wid];
    const unsigned r_key = smem_addr(&p_key[0][lane]), r_pos = smem_addr(&p_pos[0][0]);
    int buf = 0;
    for (int j = 0; j < s; j++) {
        if (g == 0) o[j] = last;
        if (j == s - 1) break;
        float best = -1.f, bx = 0.f, by = 0.f, bz = 0.f;
        int besti = 0x7fffffff;
#pragma unroll
        for (int i = 0; i < RPT; i++) {  // ascending k: the strict > keeps the lowest index on ties
            const float dx = __fsub_rn(px[i], lp.x), dy = __fsub_rn(py[i], lp.y), dz = __fsub_rn(pz[i], lp.z);
            const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
            const float m = d < mind[i] ? d : mind[i];
            mind[i] = m;
            if (m > best) { best = m; besti = g + i * STRIDE; bx = px[i]; by = py[i]; bz = pz[i]; }
        }
#pragma unroll
        for (int i = 0; i < SPT; i++) {
            float4 *q = &s_pts[i * FPS_THREADS + tid];
            const float4 v = *q;
            const float dx = __fsub_rn(v.x, lp.x), dy = __fsub_rn(v.y, lp.y), dz = __fsub_rn(v.z, lp.z);
            const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
            float m = v.w;
            if (d < m) { m = d; q->w = d; }
            if (m > best) { best = m; besti = g + (RPT + i) * STRIDE; bx = v.x; by = v.y; bz = v.z; }
        }
        // warp: maximum value (non-negative floats and -1 order like their int bits), then the lowest index attaining it
        const int bits = __float_as_int(best);
        const int wmax = __reduce_max_sync(0xffffffffu, bits);
        const int wmin = __reduce_min_sync(0xffffffffu, bits == wmax ? besti : 0x7fffffff);
        if constexpr (CS == 1) {
            // exactly one lane (indices are unique), or, when nothing in the warp is selectable, every lane with the same
            // (-1, INT_MAX, 0, 0, 0)
            if (bits == wmax && besti == wmin) { w_key[buf * NP] = make_int2(wmax, wmin); w_pos[buf * NP] = make_float4(bx, by, bz, 0.f); }
            __syncthreads();
        } else {
            const int src = __ffs(__ballot_sync(0xffffffffu, bits == wmax && besti == wmin)) - 1;
            bx = __shfl_sync(0xffffffffu, bx, src); by = __shfl_sync(0xffffffffu, by, src); bz = __shfl_sync(0xffffffffu, bz, src);
            if (lane < CS) {  // lane r writes this warp's partial into CTA r
                cg::cluster_group cl = cg::this_cluster();
                *cl.map_shared_rank(w_key + buf * NP, lane) = make_int2(wmax, wmin);
                *cl.map_shared_rank(w_pos + buf * NP, lane) = make_float4(bx, by, bz, 0.f);
            }
            cluster_barrier();
        }
        // every warp reduces the NP partials redundantly: no second barrier, buffers alternate
        int lb = (int)0x80000000, li = 0x7fffffff, lq = lane;
        if (NP >= 32 || lane < NP) { const int2 kv = lds_int2(r_key + buf * NP * sizeof(int2)); lb = kv.x; li = kv.y; }
#pragma unroll
        for (int q = lane + 32; q < NP; q += 32) {
            const int2 kv = lds_int2(r_key + (buf * NP + q - lane) * sizeof(int2));
            if (kv.x > lb || (kv.x == lb && kv.y < li)) { lb = kv.x; li = kv.y; lq = q; }
        }
        const int gmax = __reduce_max_sync(0xffffffffu, lb);
        const int gmin = __reduce_min_sync(0xffffffffu, lb == gmax ? li : 0x7fffffff);
        if (gmin == 0x7fffffff) {  // no selectable point at all (skip_origin removed everything): index 0, like the oracle
            last = 0;
            lp = ld_xyz(xyz, cloud, 0);
        } else {
            const int who = __ffs(__ballot_sync(0xffffffffu, lb == gmax && li == gmin)) - 1;
            const float4 v = lds_float4(r_pos + (buf * NP + (NP <= 32 ? who : __shfl_sync(0xffffffffu, lq, who))) * sizeof(float4));
            last = gmin;
            lp = make_float3(v.x, v.y, v.z);
        }
        buf ^= 1;
    }
    for (int j = s + g; j < npoint; j += STRIDE) o[j] = -1;
    if constexpr (CS > 1) cluster_barrier();  // no CTA leaves while a peer may still write into its shared memory
}

using FpsKernel = decltype(&fps_cluster_kernel<1, 1>);
#define PCL_FPS_ROW(CS) {fps_cluster_kernel<CS, 1>, fps_cluster_kernel<CS, 2>, fps_cluster_kernel<CS, 4>, fps_cluster_kernel<CS, 8>, \
                         fps_cluster_kernel<CS, 16>, fps_cluster_kernel<CS, 32>}
const FpsKernel fps_kernels[5][6] = {PCL_FPS_ROW(1), PCL_FPS_ROW(2), PCL_FPS_ROW(4), PCL_FPS_ROW(8), PCL_FPS_ROW(16)};  // [log2 CS][log2 PPT]
#undef PCL_FPS_ROW

int ilog2(int v) { int l = 0; while ((1 << l) < v) l++; return l; }
// log2 of the points per thread for N points on a cluster of cs CTAs (power of two, <= 32 when N <= 16384 * cs)
int fps_ppt_log2(int N, int cs) { return ilog2((N + cs * FPS_THREADS - 1) / (cs * FPS_THREADS)); }

// the kernel attributes, once per device and thread
int fps_set_attributes() {
    static thread_local int attr_dev = -1;
    int dev = 0;
    PCL_CUDA(cudaGetDevice(&dev));
    if (attr_dev == dev) return PCL_OK;
    for (int c = 0; c < 5; c++) {
        for (int p = 0; p < 6; p++) {
            PCL_CUDA(cudaFuncSetAttribute(fps_kernels[c][p], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fps_smem_bytes(1 << p)));
            if (c > 0) PCL_CUDA(cudaFuncSetAttribute(fps_kernels[c][p], cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        }
    }
    attr_dev = dev;
    return PCL_OK;
}

// B clusters of cs CTAs for N points resident at the same time?
bool fps_coresident(int B, int N, int cs, cudaStream_t st) {
    const int p = fps_ppt_log2(N, cs);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(B * cs); cfg.blockDim = dim3(FPS_THREADS); cfg.dynamicSmemBytes = fps_smem_bytes(1 << p); cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int ncl = 0;
    const cudaError_t e = cudaOccupancyMaxActiveClusters(&ncl, fps_kernels[ilog2(cs)][p], &cfg);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return ncl >= B;
}

// AUTO cluster size (header comment): remembered per (device, B, N) -- the occupancy query costs microseconds of host time
int fps_pick_cluster(int B, int N, int sm_count, cudaStream_t st) {
    struct Memo { int dev, B, N, cs; };
    static thread_local Memo memo[8];
    static thread_local int memo_n = 0, memo_next = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); dev = -1; }
    for (int i = 0; i < memo_n; i++)
        if (memo[i].dev == dev && memo[i].B == B && memo[i].N == N) return memo[i].cs;
    int cs = 1;
    while ((long)cs * FPS_CTA_POINTS < N) cs <<= 1;
    while (N > FPS_THREADS * FPS_REG_PPT && 2 * cs <= FPS_AUTO_MAX_CLUSTER && N / (2 * cs) >= FPS_AUTO_MIN_CTA_POINTS && (long)B * 2 * cs <= sm_count && fps_coresident(B, N, 2 * cs, st))
        cs <<= 1;
    memo[memo_next] = Memo{dev, B, N, cs};
    memo_next = (memo_next + 1) % 8;
    if (memo_n < 8) memo_n++;
    return cs;
}

int fps_impl(const void *xyz, int dtype, int64_t bs, int64_t rs, const int64_t *lengths, int B, int N, const int64_t *K, int npoint,
             const int32_t *start_idx, int skip_origin, int cluster, int pad, int32_t *idx_out, void *stream, const char *who) {
    if (B < 0 || N < 1 || npoint < 0) { set_error("%s: bad size B=%d N=%d npoint=%d", who, B, N, npoint); return PCL_E_SHAPE; }
    if (cluster != 0 && cluster != 1 && cluster != 2 && cluster != 4 && cluster != 8 && cluster != 16) {
        set_error("%s: cluster=%d (0 = auto, or 1, 2, 4, 8, 16)", who, cluster);
        return PCL_E_ARG;
    }
    if (N > FPS_MAX_POINTS) { set_error("%s: N=%d > %d points per cloud is not supported", who, N, FPS_MAX_POINTS); return PCL_E_UNSUPPORTED; }
    if (cluster && (long)cluster * FPS_CTA_POINTS < N) {
        set_error("%s: a cluster of %d CTAs holds at most %d points per cloud (N=%d)", who, cluster, cluster * FPS_CTA_POINTS, N);
        return PCL_E_UNSUPPORTED;
    }
    if (!dtype_ok(dtype)) { set_error("%s: bad dtype", who); return PCL_E_ARG; }
    if (B == 0 || npoint == 0) return PCL_OK;
    if (!xyz || !idx_out) { set_error("%s: null argument", who); return PCL_E_ARG; }
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    if ((rc = fps_set_attributes())) return rc;
    const Pts p{xyz, bs, rs, dtype};
    cudaStream_t st = (cudaStream_t)stream;
    const int cs = cluster ? cluster : fps_pick_cluster(B, N, di.sm_count, st);
    const int pl = fps_ppt_log2(N, cs);
    const FpsKernel k = fps_kernels[ilog2(cs)][pl];
    const int *start = start_idx;
    if (cs == 1) {
        k<<<B, FPS_THREADS, fps_smem_bytes(1 << pl), st>>>(p, lengths, N, K, npoint, pad, start, skip_origin, idx_out);
    } else {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(B * cs); cfg.blockDim = dim3(FPS_THREADS); cfg.dynamicSmemBytes = fps_smem_bytes(1 << pl); cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        PCL_CUDA(cudaLaunchKernelEx(&cfg, k, p, lengths, N, K, npoint, pad, start, skip_origin, idx_out));
    }
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

// one warp per centroid; group_idx (B, S, nsample) int32
__global__ void __launch_bounds__(256)
ball_query_kernel(Pts xyz, Pts centers, int N, int S, float r2, int nsample, int *__restrict__ group_idx) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.y;
    if (warp >= S) return;
    const float3 c = ld_xyz(centers, b, warp);
    int *out = group_idx + ((size_t)b * S + warp) * nsample;
    int cnt = 0, first = N;  // N = "nothing within the radius" (pointnet2_utils.py:107-112 leaves N in that case)
    for (int k0 = 0; k0 < N && cnt < nsample; k0 += 32) {
        const int k = k0 + lane;
        bool in = false;
        if (k < N) {
            const float3 p = ld_xyz(xyz, b, k);
            const float dx = __fsub_rn(c.x, p.x), dy = __fsub_rn(c.y, p.y), dz = __fsub_rn(c.z, p.z);
            const float d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
            in = !(d > r2);  // group_idx[sqrdists > radius ** 2] = N
        }
        const unsigned m = __ballot_sync(0xffffffffu, in);
        if (m) {
            if (first == N) first = k0 + __ffs(m) - 1;
            const int pos = cnt + __popc(m & ((1u << lane) - 1u));
            if (in && pos < nsample) out[pos] = k;
            cnt += __popc(m);
        }
    }
    cnt = min(cnt, nsample);
    for (int p = cnt + lane; p < nsample; p += 32) out[p] = first;  // pad with the first hit (pointnet2_utils.py:110-112)
}

}  // namespace
}  // namespace pcl

using namespace pcl;

extern "C" int pcl_fps_max_points(void) { return FPS_MAX_POINTS; }

extern "C" int pcl_fps(const void *xyz, int dtype, int64_t bs, int64_t rs, int B, int N, int npoint, const int32_t *start_idx,
                       int skip_origin, int32_t *idx_out, void *stream) {
    return fps_impl(xyz, dtype, bs, rs, nullptr, B, N, nullptr, npoint, start_idx, skip_origin, 0, 0, idx_out, stream, "fps");
}

extern "C" int pcl_fps_ragged(const void *xyz, int dtype, int64_t bs, int64_t rs, const int64_t *lengths, int B, int N, const int64_t *K,
                              int npoint, const int32_t *start_idx, int skip_origin, int cluster, int32_t *idx_out, void *stream) {
    return fps_impl(xyz, dtype, bs, rs, lengths, B, N, K, npoint, start_idx, skip_origin, cluster, 1, idx_out, stream, "fps_ragged");
}

extern "C" int pcl_ball_query(const void *xyz, int dtype, int64_t bs, int64_t rs, const void *new_xyz, int ndtype, int64_t nbs,
                              int64_t nrs, int B, int N, int S, float radius2, int nsample, int32_t *group_idx, void *stream) {
    if (B < 0 || N < 1 || S < 0 || nsample < 1) { set_error("ball_query: bad size B=%d N=%d S=%d nsample=%d", B, N, S, nsample); return PCL_E_SHAPE; }
    if (!dtype_ok(dtype) || !dtype_ok(ndtype)) { set_error("ball_query: bad dtype"); return PCL_E_ARG; }
    if (B == 0 || S == 0) return PCL_OK;
    if (B > 65535) { set_error("ball_query: B=%d > 65535", B); return PCL_E_SHAPE; }
    if (!xyz || !new_xyz || !group_idx) { set_error("ball_query: null argument"); return PCL_E_ARG; }
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    const Pts p{xyz, bs, rs, dtype}, c{new_xyz, nbs, nrs, ndtype};
    ball_query_kernel<<<dim3((S * 32 + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(p, c, N, S, radius2, nsample, group_idx);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}
