// pcl_knn.cu -- exact K-nearest-neighbour search (forward + backward) for sm_100a.
//
// Replaces pytorch3d.ops.knn_points / knn_points_backward for norm=2 (SURVEY.md App. B restates their semantics for
// K=1; the K > 1 contract is in include/pcl.h): squared L2 with the Chamfer arithmetic (mode UNFUSED or FMA), the K
// smallest targets j < len2[n] of every query i < len1[n], ranked and sorted by the key (distance, index).
//
// The key is one unsigned 64-bit integer: the distance's bit pattern in the upper half (distances are +0, positive,
// +inf or NaN, and for those the unsigned integer order is the float order; every NaN is mapped to 0x7fffffff, i.e.
// ranked after +inf) and the target index in the lower half.  All keys of one query are distinct, so "the K smallest
// keys" is one set whatever order the targets are visited in -- which lets warps scan different targets of the same
// queries and merge their lists at the end with bit-exact results.
//
// Forward kernel: one lane per query, 32 queries per CTA, and `parts` warps that scan interleaved targets of the same 32
// queries (parts > 1 when B*P1 is too small to fill the GPU).  The target cloud streams through shared memory in tiles.
// Every lane keeps its sorted list of K keys in shared memory and the K-th key in a register as the admission threshold;
// a target whose distance is not above the threshold distance is compared by key and, if it is smaller, appended to a
// small per-lane candidate buffer.  When some lane's buffer may overflow, the whole warp drains its buffers into the
// sorted lists (insertion, threshold refreshed after each key).  Draining together bounds the time a warp spends in the
// divergent insertion code by the busiest lane's admissions -- about K (1 + ln(P2/K)) for random order -- instead of one
// insertion for every target that ANY of the 32 queries admits, which early in the scan is nearly every target.
#include <climits>

#include "pcl_common.cuh"
#include "pcl_nn.cuh"

namespace pcl {
namespace {

typedef unsigned long long u64;

#ifndef PCL_KNN_MAX_PARTS
#define PCL_KNN_MAX_PARTS 16
#endif
constexpr int KNN_MAX_K = 64;
constexpr int KNN_MAX_PARTS = PCL_KNN_MAX_PARTS;     // warps per CTA that share the 32 queries
constexpr int KNN_TILE = 512;                         // targets per shared-memory tile
constexpr int KNN_BUF = 16;                           // candidate buffer per lane, drained when a lane may not have
constexpr int KNN_UNROLL = 4;                         // room for the next KNN_UNROLL targets
constexpr int KNN_LIST_BYTES = 64 * 1024;             // sorted lists of one CTA: parts * 32 * K * 8 bytes at most
constexpr u64 KNN_NONE = ~0ull;                       // empty list slot: above every key
constexpr int KNN_BWD_THREADS = 128;

// element load with a runtime dtype: one 32-bit or one 16-bit load (bf16 -> fp32 is exact: the bits move up by 16).  Fewer
// branches than ld_any, which makes ptxas spill a few bytes in these kernels.
__device__ __forceinline__ float ld_pt(const Pts &a, int64_t i) {
    if (a.dtype == PCL_F32) return __ldg(reinterpret_cast<const float *>(a.p) + i);
    const unsigned short h = __ldg(reinterpret_cast<const unsigned short *>(a.p) + i);
    return (a.dtype == PCL_F16) ? __half2float(__ushort_as_half(h)) : __uint_as_float((unsigned)h << 16);
}

// knn_key, key_dist and sqdist<FMA, D>: pcl_nn.cuh (shared with pcl_icp.cu)

// insert `key` (< my[K-1]) into the ascending list my[0], my[32], ..., my[32 (K-1)]; returns the new K-th key
__device__ __forceinline__ u64 list_insert(u64 *my, int K, u64 key) {
    int p = K - 1;
    for (; p > 0; p--) {
        const u64 prev = my[(p - 1) * 32];
        if (prev < key) break;
        my[p * 32] = prev;
    }
    my[p * 32] = key;
    return my[(K - 1) * 32];
}

// grid (ceil(P1 / 32), B); block 32 * parts; dynamic shared memory: the tile, then per warp 32 x K list keys and
// 32 x KNN_BUF buffered keys (lane-interleaved: conflict-free).
template <bool FMA, int D>
__global__ void __launch_bounds__(32 * KNN_MAX_PARTS, 1)
knn_fwd_kernel(Pts p1, const int64_t *__restrict__ len1, Pts p2, const int64_t *__restrict__ len2, int P1, int P2, int K,
               float *__restrict__ dists, int *__restrict__ idx) {
    constexpr int DS = (D == 3) ? 4 : D;  // tile row stride in floats (D = 3: one LDS.128 per target)
    extern __shared__ __align__(16) unsigned char knn_smem[];
    float *tile = reinterpret_cast<float *>(knn_smem);
    const int parts = blockDim.x >> 5, part = threadIdx.x >> 5, lane = threadIdx.x & 31, n = blockIdx.y;
    u64 *lists = reinterpret_cast<u64 *>(knn_smem + KNN_TILE * DS * sizeof(float));
    u64 *my = lists + (size_t)part * 32 * (K + KNN_BUF) + lane;  // list slot k: my[32 k]
    u64 *buf = my + 32 * K;                                        // buffer slot b: buf[32 b]
    const int i0 = blockIdx.x * 32, i = i0 + lane;
    const int lq = len_of(len1, n, P1), lt = len_of(len2, n, P2);
    const int kv = min(K, lt);  // slots that receive a neighbour; the others are 0 / 0
    const size_t out0 = ((size_t)n * P1 + i0) * K;
    const int nout = min(32, P1 - i0) * K;  // this CTA's rows are one contiguous block of the outputs
    if (i0 >= lq || kv == 0) {  // CTA-uniform: padded rows only, or nothing to find
        for (int e = threadIdx.x; e < nout; e += blockDim.x) { dists[out0 + e] = 0.f; idx[out0 + e] = 0; }
        return;
    }
    float q[D];
#pragma unroll
    for (int c = 0; c < D; c++) q[c] = (i < lq) ? ld_pt(p1, (int64_t)n * p1.bs + (int64_t)i * p1.rs + c) : 0.f;  // surplus lanes: discarded
    for (int k = 0; k < K; k++) my[32 * k] = KNN_NONE;
    u64 thr = KNN_NONE;                 // K-th key of the list
    float thr_d = key_dist(thr);        // its distance: NaN (empty slot or NaN key) lets every target through to the key test
    int nb = 0;
    auto drain = [&]() {
        for (int b = 0; b < nb; b++) {
            const u64 key = buf[32 * b];
            if (key < thr) thr = list_insert(my, K, key);
        }
        nb = 0;
        thr_d = key_dist(thr);
    };
    for (int t0 = 0; t0 < lt; t0 += KNN_TILE) {
        const int cnt = min(KNN_TILE, lt - t0);
        __syncthreads();  // the previous tile is consumed
        for (int e = threadIdx.x; e < cnt * D; e += blockDim.x) {
            const int j = e / D, c = e - j * D;
            tile[j * DS + c] = ld_pt(p2, (int64_t)n * p2.bs + (int64_t)(t0 + j) * p2.rs + c);
        }
        __syncthreads();
        for (int e0 = part * KNN_UNROLL; e0 < cnt; e0 += parts * KNN_UNROLL) {  // warp-uniform
#pragma unroll
            for (int u = 0; u < KNN_UNROLL; u++) {
                const int e = e0 + u;
                if (e < cnt) {
                    const float d = sqdist<FMA, D>(q, tile + e * DS);
                    if (!(d > thr_d)) {
                        const u64 key = knn_key(d, t0 + e);
                        if (key < thr) { buf[32 * nb] = key; nb++; }
                    }
                }
            }
            if (__any_sync(0xffffffffu, nb > KNN_BUF - KNN_UNROLL)) drain();
        }
    }
    drain();
    // merge the other warps' lists into warp 0's (each is sorted: stop at the first key that is not admitted)
    __syncthreads();
    if (part == 0) {
        for (int s = 1; s < parts; s++) {
            const u64 *o = lists + (size_t)s * 32 * (K + KNN_BUF) + lane;
            for (int k = 0; k < K; k++) {
                const u64 key = o[32 * k];
                if (!(key < thr)) break;
                thr = list_insert(my, K, key);
            }
        }
    }
    __syncthreads();
    const u64 *l0 = lists + 0;  // warp 0's lists: row r, slot k at l0[32 k + r]
    for (int e = threadIdx.x; e < nout; e += blockDim.x) {
        const int r = e / K, k = e - r * K;
        const bool ok = (i0 + r < lq) && (k < kv);
        const u64 key = ok ? l0[32 * k + r] : 0ull;
        dists[out0 + e] = ok ? key_dist(key) : 0.f;
        idx[out0 + e] = ok ? (int)(unsigned)key : 0;
    }
}

// Backward: one thread per (n, i).  grad_p1[n, i] = sum_k diff_k in ascending k (fp32, in registers, then one store;
// padded rows get 0); grad_p2[n, idx] -= diff_k with red.global.add onto the zero-filled grad_p2.  Slots whose idx is -1
// contribute nothing.
template <int D>
__global__ void __launch_bounds__(KNN_BWD_THREADS, 4)
knn_bwd_kernel(Pts p1, const int64_t *__restrict__ len1, Pts p2, const int64_t *__restrict__ len2, int P1, int P2, int K,
               const int *__restrict__ idx, const float *__restrict__ grad_dists, float *__restrict__ grad_p1,
               float *__restrict__ grad_p2) {
    const int n = blockIdx.y, i = blockIdx.x * KNN_BWD_THREADS + threadIdx.x;
    if (i >= P1) return;
    const int lq = len_of(len1, n, P1), lt = len_of(len2, n, P2);
    const int kv = (i < lq) ? min(K, lt) : 0;
    float acc[D], q[D];
#pragma unroll
    for (int c = 0; c < D; c++) {
        acc[c] = 0.f;
        q[c] = kv ? ld_pt(p1, (int64_t)n * p1.bs + (int64_t)i * p1.rs + c) : 0.f;
    }
    const size_t r0 = ((size_t)n * P1 + i) * K;
    for (int k = 0; k < kv; k++) {
        const int j = __ldg(idx + r0 + k);
        if (j < 0) continue;  // a ball-query pad (pcl_knn_fwd never writes -1)
        const float g2 = __fmul_rn(2.0f, __ldg(grad_dists + r0 + k));
        const int64_t to = (int64_t)n * p2.bs + (int64_t)j * p2.rs;
        float *gt = grad_p2 + ((size_t)n * P2 + j) * D;
#pragma unroll
        for (int c = 0; c < D; c++) {
            const float diff = __fmul_rn(g2, __fsub_rn(q[c], ld_pt(p2, to + c)));
            acc[c] = __fadd_rn(acc[c], diff);
            atomicAdd(gt + c, -diff);
        }
    }
    float *gq = grad_p1 + ((size_t)n * P1 + i) * D;
#pragma unroll
    for (int c = 0; c < D; c++) gq[c] = acc[c];
}

// ------------------------------------------------------------------ ball query
// pytorch3d.ops.ball_query (include/pcl.h, "ball query"): for a query i < len1[n], the first K targets j < len2[n] in
// ascending index order with sqdist<FMA, D> < radius2, then (0, -1) pads.
//
// One lane per query, 32 queries per CTA.  When B * ceil(P1 / 32) warps cannot fill the GPU, `parts` warps of the CTA
// scan `parts` contiguous, ascending ranges of the targets [0, len2) (range p = [p c, (p+1) c), c = ceil(len2 / parts)),
// each collecting the first K hits of its own range.  Part 0 appends its hits straight to the output row; part p >= 1
// keeps the indices of its hits in shared memory (distances are recomputed by the same sqdist when merged, so they are
// bit-identical).  Warp 0 then appends parts 1, 2, ... in order until the row holds K hits.  Because the ranges are
// contiguous and ordered, the first K hits of the concatenation are the first K hits of the whole scan: the result does
// not depend on `parts`.  Split rule (bq_parts_for): double `parts` while the GPU has fewer than 8 query warps per SM,
// parts <= BQ_MAX_PARTS, every part keeps at least BQ_MIN_RANGE of the P2 targets, and the buffered indices
// (parts - 1) * 32 * K * 4 bytes fit BQ_BUF_BYTES -- so K <= 960 may split in two and K <= 64 in sixteen.  The unsplit
// path has no bound on K.
//
// Each warp streams its range through its own shared-memory tile (no CTA barrier in the scan) and stops once all its
// lanes have K hits, or once the lower parts already hold K hits for every lane: per-lane hit counts are published in
// shared memory after every tile, and since they only grow, a stale read only delays the exit.
constexpr int BQ_MAX_PARTS = 16;
constexpr int BQ_TILE = 128;                // targets per warp tile
constexpr int BQ_MIN_RANGE = 256;           // targets per part at least
constexpr int BQ_BUF_BYTES = 120 * 1024;    // buffered hit indices of parts 1.. (15 parts x 32 lanes x K = 64 x 4 bytes)

// grid (ceil(P1 / 32), B); block 32 * parts; dynamic shared memory: parts tiles of BQ_TILE x DS floats, hit counts
// [part][lane], then buffered indices [part - 1][k][lane].
template <bool FMA, int D>
__global__ void __launch_bounds__(32 * BQ_MAX_PARTS, 1)
ball_query_fwd_kernel(Pts p1, const int64_t *__restrict__ len1, Pts p2, const int64_t *__restrict__ len2, int P1, int P2,
                      int K, float r2, float *__restrict__ dists, int *__restrict__ idx) {
    constexpr int DS = (D == 3) ? 4 : D;
    extern __shared__ __align__(16) unsigned char bq_sm[];
    const int parts = blockDim.x >> 5, part = threadIdx.x >> 5, lane = threadIdx.x & 31, n = blockIdx.y;
    float *tile = reinterpret_cast<float *>(bq_sm) + part * BQ_TILE * DS;
    volatile int *counts = reinterpret_cast<volatile int *>(bq_sm + (size_t)parts * BQ_TILE * DS * sizeof(float));
    int *bufs = const_cast<int *>(counts) + parts * 32;
    const int i0 = blockIdx.x * 32, i = i0 + lane;
    const int lq = len_of(len1, n, P1), lt = len_of(len2, n, P2);
    const size_t out0 = ((size_t)n * P1 + i0) * K;
    const int nout = min(32, P1 - i0) * K;  // this CTA's rows are one contiguous block of the outputs
    if (i0 >= lq) {  // CTA-uniform: padded rows only
        for (int e = threadIdx.x; e < nout; e += blockDim.x) { dists[out0 + e] = 0.f; idx[out0 + e] = -1; }
        return;
    }
    const bool active = i < lq;
    float q[D];
#pragma unroll
    for (int c = 0; c < D; c++) q[c] = active ? ld_pt(p1, (int64_t)n * p1.bs + (int64_t)i * p1.rs + c) : 0.f;
    float *drow = dists + out0 + (size_t)lane * K;
    int *irow = idx + out0 + (size_t)lane * K;
    int *buf = bufs + (size_t)(part - 1) * K * 32 + lane;  // part >= 1: hit k at buf[32 k]
    const int chunk = (lt + parts - 1) / parts;
    const int lo = min(lt, part * chunk), hi = min(lt, lo + chunk);
    int cnt = active ? 0 : K;  // surplus lanes count as done
    counts[part * 32 + lane] = cnt;
    __syncthreads();
    for (int t0 = lo; t0 < hi; t0 += BQ_TILE) {
        int below = 0;
        for (int s = 0; s < part; s++) below += counts[s * 32 + lane];
        if (__all_sync(0xffffffffu, cnt >= K || below >= K)) break;  // warp-uniform
        const int m = min(BQ_TILE, hi - t0);
        __syncwarp();  // the previous tile is consumed
        for (int e = lane; e < m * D; e += 32) {
            const int j = e / D, c = e - j * D;
            tile[j * DS + c] = ld_pt(p2, (int64_t)n * p2.bs + (int64_t)(t0 + j) * p2.rs + c);
        }
        __syncwarp();
#pragma unroll 4
        for (int e = 0; e < m; e++) {
            const float d = sqdist<FMA, D>(q, tile + e * DS);
            if (d < r2 && cnt < K) {  // NaN is never < r2
                if (part == 0) { drow[cnt] = d; irow[cnt] = t0 + e; }
                else buf[32 * cnt] = t0 + e;
                cnt++;
            }
        }
        counts[part * 32 + lane] = cnt;
    }
    __syncthreads();
    if (part == 0) {
        for (int s = 1; s < parts && cnt < K; s++) {
            const int ns = counts[s * 32 + lane];
            const int *ob = bufs + (size_t)(s - 1) * K * 32 + lane;
            for (int k = 0; k < ns && cnt < K; k++) {
                const int j = ob[32 * k];
                float t[D];
#pragma unroll
                for (int c = 0; c < D; c++) t[c] = ld_pt(p2, (int64_t)n * p2.bs + (int64_t)j * p2.rs + c);
                drow[cnt] = sqdist<FMA, D>(q, t);
                irow[cnt] = j;
                cnt++;
            }
        }
        counts[lane] = cnt;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nout; e += blockDim.x) {  // pads, coalesced over the CTA's block of rows
        const int r = e / K, k = e - r * K;
        if (i0 + r >= lq || k >= counts[r]) { dists[out0 + e] = 0.f; idx[out0 + e] = -1; }
    }
}

inline int parts_for(int B, int P1, int P2, int K, int sm_count) {
    // Split the targets over more warps only while the GPU is short of warps (fewer than 8 per SM), every warp keeps at least
    // 32 K targets (below that the list insertions cost more than the scan saves) and the lists fit KNN_LIST_BYTES.
    const long long qwarps = (long long)B * ((P1 + 31) / 32);
    int parts = 1;
    while (parts * 2 <= KNN_MAX_PARTS && qwarps * parts < 8LL * sm_count && P2 / (parts * 2) >= 32 * K &&
           (size_t)parts * 2 * 32 * (K + KNN_BUF) * sizeof(u64) <= (size_t)KNN_LIST_BYTES)
        parts *= 2;
    return parts;
}

inline size_t fwd_smem(int D, int K, int parts) {
    return (size_t)KNN_TILE * (D == 3 ? 4 : D) * sizeof(float) + (size_t)parts * 32 * (K + KNN_BUF) * sizeof(u64);
}

template <bool FMA, int D>
int launch_fwd_d(const Pts &a, const int64_t *len1, const Pts &b, const int64_t *len2, int B, int P1, int P2, int K, int parts,
                 float *dists, int *idx, cudaStream_t st) {
    const size_t smem = fwd_smem(D, K, parts);
    static thread_local int attr_dev = -1;  // per instantiation: the opt-in to more than 48 KB of dynamic shared memory
    int dev = 0;
    PCL_CUDA(cudaGetDevice(&dev));
    if (attr_dev != dev) {  // parts_for keeps the lists within KNN_LIST_BYTES (one warp's lists at K = 64 need 20 KB)
        PCL_CUDA(cudaFuncSetAttribute(knn_fwd_kernel<FMA, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fwd_smem(D, 0, 0) + KNN_LIST_BYTES));
        attr_dev = dev;
    }
    knn_fwd_kernel<FMA, D><<<dim3((P1 + 31) / 32, B), 32 * parts, smem, st>>>(a, len1, b, len2, P1, P2, K, dists, idx);
    return PCL_OK;
}

template <bool FMA>
int launch_fwd(const Pts &a, const int64_t *len1, const Pts &b, const int64_t *len2, int B, int P1, int P2, int D, int K, int parts,
               float *dists, int *idx, cudaStream_t st) {
    switch (D) {
#define PCL_KNN_FWD(DD) case DD: return launch_fwd_d<FMA, DD>(a, len1, b, len2, B, P1, P2, K, parts, dists, idx, st)
        PCL_KNN_FWD(1); PCL_KNN_FWD(2); PCL_KNN_FWD(3); PCL_KNN_FWD(4);
        PCL_KNN_FWD(5); PCL_KNN_FWD(6); PCL_KNN_FWD(7); PCL_KNN_FWD(8);
#undef PCL_KNN_FWD
    }
    set_error("knn: D=%d unsupported (1..8)", D);
    return PCL_E_UNSUPPORTED;
}

inline int bq_parts_for(int B, int P1, int P2, int K, int sm_count) {
    const long long qwarps = (long long)B * ((P1 + 31) / 32);
    int parts = 1;
    while (parts * 2 <= BQ_MAX_PARTS && qwarps * parts < 8LL * sm_count && P2 / (parts * 2) >= BQ_MIN_RANGE &&
           (long long)(parts * 2 - 1) * 32 * K * sizeof(int) <= BQ_BUF_BYTES)
        parts *= 2;
    return parts;
}

inline size_t bq_smem(int D, int K, int parts) {
    return (size_t)parts * BQ_TILE * (D == 3 ? 4 : D) * sizeof(float) + (size_t)parts * 32 * sizeof(int) +
           (size_t)(parts - 1) * 32 * K * sizeof(int);
}

template <bool FMA, int D>
int launch_bq_d(const Pts &a, const int64_t *len1, const Pts &b, const int64_t *len2, int B, int P1, int P2, int K, float r2,
                int parts, float *dists, int *idx, cudaStream_t st) {
    static thread_local int attr_dev = -1;  // per instantiation: the opt-in to more than 48 KB of dynamic shared memory
    int dev = 0;
    PCL_CUDA(cudaGetDevice(&dev));
    if (attr_dev != dev) {  // bq_parts_for keeps the buffers within BQ_BUF_BYTES
        PCL_CUDA(cudaFuncSetAttribute(ball_query_fwd_kernel<FMA, D>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(bq_smem(D, 0, BQ_MAX_PARTS) + BQ_BUF_BYTES)));
        attr_dev = dev;
    }
    ball_query_fwd_kernel<FMA, D><<<dim3((P1 + 31) / 32, B), 32 * parts, bq_smem(D, K, parts), st>>>(a, len1, b, len2, P1, P2, K,
                                                                                                    r2, dists, idx);
    return PCL_OK;
}

template <bool FMA>
int launch_bq(const Pts &a, const int64_t *len1, const Pts &b, const int64_t *len2, int B, int P1, int P2, int D, int K, float r2,
              int parts, float *dists, int *idx, cudaStream_t st) {
    switch (D) {
#define PCL_BQ_FWD(DD) case DD: return launch_bq_d<FMA, DD>(a, len1, b, len2, B, P1, P2, K, r2, parts, dists, idx, st)
        PCL_BQ_FWD(1); PCL_BQ_FWD(2); PCL_BQ_FWD(3); PCL_BQ_FWD(4);
        PCL_BQ_FWD(5); PCL_BQ_FWD(6); PCL_BQ_FWD(7); PCL_BQ_FWD(8);
#undef PCL_BQ_FWD
    }
    set_error("ball_query: D=%d unsupported (1..8)", D);
    return PCL_E_UNSUPPORTED;
}

// kmax: the largest K accepted (KNN_MAX_K for kNN; ball query has no bound but sizes)
int check_args(const char *who, const void *p1, int dtype1, const void *p2, int dtype2, int B, int P1, int P2, int D, int K,
               int kmax) {
    if (B < 0 || P1 < 0 || P2 < 0) { set_error("%s: negative size B=%d P1=%d P2=%d", who, B, P1, P2); return PCL_E_SHAPE; }
    if (D < 1 || D > 8) { set_error("%s: D=%d unsupported (1..8)", who, D); return PCL_E_UNSUPPORTED; }
    if (K < 1) { set_error("%s: K=%d must be at least 1", who, K); return PCL_E_SHAPE; }
    if (K > kmax) { set_error("%s: K=%d > pcl_knn_max_k() = %d", who, K, kmax); return PCL_E_UNSUPPORTED; }
    if (B > 65535) { set_error("%s: B=%d > 65535", who, B); return PCL_E_SHAPE; }
    if (!dtype_ok(dtype1) || !dtype_ok(dtype2)) { set_error("%s: bad dtype", who); return PCL_E_ARG; }
    if (B > 0 && ((P1 > 0 && !p1) || (P2 > 0 && !p2))) { set_error("%s: null input", who); return PCL_E_ARG; }
    return PCL_OK;
}

}  // namespace
}  // namespace pcl

using namespace pcl;

extern "C" int pcl_knn_max_k(void) { return KNN_MAX_K; }

extern "C" int pcl_knn_fwd(const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
                           const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2,
                           int B, int P1, int P2, int D, int K, int mode, float *dists, int32_t *idx, void *stream) {
    int rc = check_args("knn", p1, dtype1, p2, dtype2, B, P1, P2, D, K, KNN_MAX_K);
    if (rc) return rc;
    if (mode != PCL_CHAMFER_UNFUSED && mode != PCL_CHAMFER_FMA) { set_error("knn: bad mode %d", mode); return PCL_E_ARG; }
    if (B > 0 && P1 > 0 && (!dists || !idx)) { set_error("knn: null output"); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0 || P1 == 0) return PCL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const Pts a{p1, bs1, rs1, dtype1}, b{p2, bs2, rs2, dtype2};
    const int parts = parts_for(B, P1, P2, K, di.sm_count);
    rc = (mode == PCL_CHAMFER_FMA) ? launch_fwd<true>(a, len1, b, len2, B, P1, P2, D, K, parts, dists, (int *)idx, st)
                                   : launch_fwd<false>(a, len1, b, len2, B, P1, P2, D, K, parts, dists, (int *)idx, st);
    if (rc) return rc;
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

namespace {
// pcl_knn_bwd and pcl_ball_query_bwd: the same kernel, with kNN's or ball query's bound on K
int bwd_impl(const char *who, int kmax, const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
             const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2, int B, int P1, int P2, int D, int K,
             const int32_t *idx, const float *grad_dists, float *grad_p1, float *grad_p2, void *stream) {
    int rc = check_args(who, p1, dtype1, p2, dtype2, B, P1, P2, D, K, kmax);
    if (rc) return rc;
    if (B > 0 && ((P1 > 0 && (!idx || !grad_dists || !grad_p1)) || (P2 > 0 && !grad_p2))) {
        set_error("%s: null argument", who); return PCL_E_ARG;
    }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0) return PCL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (P2 > 0) PCL_CUDA(cudaMemsetAsync(grad_p2, 0, (size_t)B * P2 * D * sizeof(float), st));
    if (P1 == 0) return PCL_OK;
    const Pts a{p1, bs1, rs1, dtype1}, b{p2, bs2, rs2, dtype2};
    const dim3 grid((P1 + KNN_BWD_THREADS - 1) / KNN_BWD_THREADS, B);
    switch (D) {
#define PCL_KNN_BWD(DD) \
    case DD: knn_bwd_kernel<DD><<<grid, KNN_BWD_THREADS, 0, st>>>(a, len1, b, len2, P1, P2, K, (const int *)idx, grad_dists, grad_p1, grad_p2); break
        PCL_KNN_BWD(1); PCL_KNN_BWD(2); PCL_KNN_BWD(3); PCL_KNN_BWD(4);
        PCL_KNN_BWD(5); PCL_KNN_BWD(6); PCL_KNN_BWD(7); PCL_KNN_BWD(8);
#undef PCL_KNN_BWD
    }
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}
}  // namespace

extern "C" int pcl_knn_bwd(const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
                           const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2,
                           int B, int P1, int P2, int D, int K, const int32_t *idx, const float *grad_dists,
                           float *grad_p1, float *grad_p2, void *stream) {
    return bwd_impl("knn_bwd", KNN_MAX_K, p1, dtype1, bs1, rs1, len1, p2, dtype2, bs2, rs2, len2, B, P1, P2, D, K, idx,
                    grad_dists, grad_p1, grad_p2, stream);
}

extern "C" int pcl_ball_query_fwd(const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
                                  const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2,
                                  int B, int P1, int P2, int D, int K, float radius2, int mode, float *dists, int32_t *idx,
                                  void *stream) {
    int rc = check_args("ball_query", p1, dtype1, p2, dtype2, B, P1, P2, D, K, INT_MAX);
    if (rc) return rc;
    if (mode != PCL_CHAMFER_UNFUSED && mode != PCL_CHAMFER_FMA) { set_error("ball_query: bad mode %d", mode); return PCL_E_ARG; }
    if (B > 0 && P1 > 0 && (!dists || !idx)) { set_error("ball_query: null output"); return PCL_E_ARG; }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0 || P1 == 0) return PCL_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const Pts a{p1, bs1, rs1, dtype1}, b{p2, bs2, rs2, dtype2};
    const int parts = bq_parts_for(B, P1, P2, K, di.sm_count);
    rc = (mode == PCL_CHAMFER_FMA) ? launch_bq<true>(a, len1, b, len2, B, P1, P2, D, K, radius2, parts, dists, (int *)idx, st)
                                   : launch_bq<false>(a, len1, b, len2, B, P1, P2, D, K, radius2, parts, dists, (int *)idx, st);
    if (rc) return rc;
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_ball_query_bwd(const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
                                  const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2,
                                  int B, int P1, int P2, int D, int K, const int32_t *idx, const float *grad_dists,
                                  float *grad_p1, float *grad_p2, void *stream) {
    return bwd_impl("ball_query_bwd", INT_MAX, p1, dtype1, bs1, rs1, len1, p2, dtype2, bs2, rs2, len2, B, P1, P2, D, K, idx,
                    grad_dists, grad_p1, grad_p2, stream);
}
