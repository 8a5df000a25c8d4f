// pcl_chamfer.cu -- Chamfer distance forward/backward for sm_100a.
//
// Replaces the native layer under pytorch3d.loss.chamfer_distance as the reference calls it
// (pointcloud_vision/utils.py:211,228): knn_points(K=1) in both directions, squared L2, lowest
// index on exact ties, variable lengths, point-mean + batch-mean; backward scatters
// 2*g*(p - q[idx]) to both clouds (SURVEY.md App. B).
//
// Forward kernel (D == 3): one CTA = 128 threads x QPT register-resident queries of one cloud and one direction; the
// target cloud streams through shared memory in tiles stored per PAIR of targets ({x0,x1,y0,y1}, {z0,z1,|t0|^2,|t1|^2}:
// the operand layout of FFMA2).  The scan evaluates an APPROXIMATE expanded-form distance with packed FFMA2 and only
// remembers which 32-target chunks can hold the nearest neighbour; those chunks are re-scanned with the oracle's
// arithmetic (explicit __fsub_rn/__fmul_rn/__fadd_rn/__fmaf_rn), which alone decides distance, index and the
// lowest-index tie rule (derivation above chamfer_nn3_kernel and in DESIGN.md 3.2).
#include <stdlib.h>

#include "pcl_common.cuh"

namespace pcl {
namespace {

constexpr int CH_THREADS = 128;  // the generic-D kernel and the partial-sum layout: one slot per 128 queries
#ifndef PCL_C3_QPT
#define PCL_C3_QPT 2
#endif
#ifndef PCL_C3_WQ
#define PCL_C3_WQ 4
#endif
#ifndef PCL_C3_PARTS
#define PCL_C3_PARTS 1
#endif
constexpr int C3_QPT = PCL_C3_QPT;      // D == 3 kernel: register-resident queries per lane ...
constexpr int C3_WQ = PCL_C3_WQ;        // ... warps with different queries ...
constexpr int C3_PARTS = PCL_C3_PARTS;  // ... and warps that share the queries but scan different chunks of the targets (merged at the end)
constexpr int C3_QUERIES = 32 * C3_QPT * C3_WQ;  // queries per CTA
constexpr int C3_THREADS = 32 * C3_WQ * C3_PARTS;
constexpr int C3_TILE = 1024;    // targets per shared-memory tile (16 KB), cut into ...
constexpr int C3_CHUNK = 32;     // ... chunks of 32: the granularity of the approximate minimum and of the exact re-scan
#ifndef PCL_C3_GROUP
#define PCL_C3_GROUP 4
#endif
#ifndef PCL_C3_MINB
#define PCL_C3_MINB 5  // CTAs per SM the register budget is set for: 5 x 128 threads x 96 registers (4 x 128: 6-10 % slower at every size, 6 x 80: spills)
#endif
constexpr int C3_GROUP = PCL_C3_GROUP;      // pairs of targets per register buffer of the scan (double-buffered: hides the LDS latency)

typedef unsigned long long u64;
// sm_100a packed FP32: FFMA2 = two IEEE-rounded FMAs per instruction, same FLOP rate as FFMA at half the issue slots
// (tools/microbench_packed.cu).  Only the approximate scan uses it: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into
// FFMA2 (even with -fmad=false), so the oracle's unfused sums cannot be written with packed instructions.
__device__ __forceinline__ u64 pk2(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ float lo2(u64 v) { return __uint_as_float((unsigned)v); }
__device__ __forceinline__ float hi2(u64 v) { return __uint_as_float((unsigned)(v >> 32)); }
__device__ __forceinline__ u64 ffma2(u64 a, u64 b, u64 c) { u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ float fmin3(float a, float b, float c) { float r; asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r; }  // NaN operands are ignored

template <bool FMA>
__device__ __forceinline__ float sqdist3(float qx, float qy, float qz, const float4 &t) {
    const float dx = __fsub_rn(qx, t.x), dy = __fsub_rn(qy, t.y), dz = __fsub_rn(qz, t.z);
    if constexpr (FMA) return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
    else return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// length of cloud n, clamped to [0, P]: pytorch3d raises on lengths > P; a kernel cannot, but it must not read past the cloud
__device__ __forceinline__ int len_of(const int64_t *len, int n, int P) {
    if (!len) return P;
    const int64_t v = len[n];
    return (int)(v < 0 ? 0 : (v > P ? P : v));
}

// Tail of both forward kernels: the CTA's partial sum goes to the workspace; the CTA that takes the LAST ticket of the grid
// (zeroed by the host call) then forms  loss_xy[dir] = sum_n (sum_i dist / clamp(len,1)) / max(B,1)  from all partials in a
// fixed order (deterministic scalar, fp64) -- no memset of the partials and no second launch.  Needs >= 64 threads per CTA.
__device__ __forceinline__ void finish_block(float s /* valid on thread 0 */, float *__restrict__ partial, int nblk, int dir, int n,
                                             unsigned *__restrict__ ticket, int P1, int P2, const int64_t *__restrict__ x_len,
                                             const int64_t *__restrict__ y_len, float *__restrict__ loss_xy) {
    __shared__ int last_flag;
    const int B = (int)gridDim.y;
    if (threadIdx.x == 0) {
        partial[((size_t)dir * B + n) * nblk + blockIdx.x] = s;
        __threadfence();
        last_flag = (atomicAdd(ticket, 1u) == gridDim.x * gridDim.y * gridDim.z - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!last_flag || threadIdx.x >= 64) return;
    __threadfence();
    __shared__ double acc[2][32];
    const int d = threadIdx.x >> 5, lane = threadIdx.x & 31;  // one warp per direction
    double a = 0.0;
    for (int c = lane; c < B; c += 32) {
        double t = 0.0;
        for (int k = 0; k < (int)gridDim.x; k++) t += (double)__ldcg(&partial[((size_t)d * B + c) * nblk + k]);
        const int len = d ? len_of(y_len, c, P2) : len_of(x_len, c, P1);
        a += t / (double)(len > 1 ? len : 1);
    }
    acc[d][lane] = a;
    __syncwarp();
    if (lane == 0) {
        double t = 0.0;
        for (int k = 0; k < 32; k++) t += acc[d][k];
        loss_xy[d] = (float)(t / (double)(B > 1 ? B : 1));
        loss_xy[2 + d] = (float)t;  // the un-normalised batch sum: what a batch-sharded caller all-reduces
    }
}

template <int NWARPS>
__device__ __forceinline__ float block_sum(float v, float *red /* >= NWARPS floats */) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) red[w] = v;
    __syncthreads();
    float s = 0.f;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < NWARPS; i++) s += red[i];  // fixed order
    }
    return s;  // valid on thread 0
}

__device__ __forceinline__ float finite_or_inf(float v) { return (v <= 3.0e38f) ? v : __int_as_float(0x7f800000); }  // NaN -> +inf

// Exact re-scan of chunk c of the tile for one query.  Phase A evaluates the approximate distance once more (same
// bound, same threshold thr = running minimum + E2) and collects the pairs of targets that pass it -- the exact nearest
// neighbour always does; phase B gives those (one or two) the oracle's arithmetic and folds them into (best, bi) with the
// explicit rule "smaller distance, then lower index", the order-independent form of knn's ascending strict-'<' scan.
// Lanes re-scan DIFFERENT chunks; rotating the pair order by the lane id keeps the 8 lanes of an LDS.128 phase on 8
// different bank groups.
template <bool FMA>
__device__ __forceinline__ void rescan_chunk(const float4 *tA, const float4 *tB, bool act, int c, int cnt, int t0, float qx,
                                             float qy, float qz, u64 nqx, u64 nqy, u64 nqz, float thr, float &best, int &bi) {
    unsigned pm = 0;
    const int base = c * (C3_CHUNK / 2), rot = (int)threadIdx.x;
#pragma unroll
    for (int pp = 0; pp < C3_CHUNK / 2; pp++) {
        const int o = (pp + rot) & (C3_CHUNK / 2 - 1);
        const float4 a = tA[base + o], b = tB[base + o];
        const u64 v = ffma2(pk2(b.x, b.y), nqz, ffma2(pk2(a.z, a.w), nqy, ffma2(pk2(a.x, a.y), nqx, pk2(b.z, b.w))));
        pm |= (unsigned)(!(fminf(lo2(v), hi2(v)) > thr)) << o;
    }
    if (!act) pm = 0;
    while (__any_sync(0xffffffffu, pm != 0)) {
        if (pm) {
            const int o = __ffs(pm) - 1;
            pm &= pm - 1;
            const float4 a = tA[base + o], b = tB[base + o];
            const int j0 = 2 * (base + o), i0 = t0 + j0;
            const float d0 = sqdist3<FMA>(qx, qy, qz, make_float4(a.x, a.z, b.x, 0.f));
            const float d1 = sqdist3<FMA>(qx, qy, qz, make_float4(a.y, a.w, b.y, 0.f));
            if (j0 < cnt && (d0 < best || (d0 == best && i0 < bi))) { best = d0; bi = i0; }
            if (j0 + 1 < cnt && (d1 < best || (d1 == best && i0 + 1 < bi))) { best = d1; bi = i0 + 1; }
        }
    }
}

// Forward kernel for D == 3.  grid: (ceil(maxP / C3_QUERIES), B, 2 directions); block: WQ x PARTS warps, QPT queries per lane.
//
// The scan over the targets runs on an APPROXIMATE distance in expanded form,
//     a(q,t) = |t|^2 - 2 q.t  =  fma(tz, -2qz, fma(ty, -2qy, fma(tx, -2qx, |t|^2)))      (= |q-t|^2 - |q|^2),
// three FFMA2 per two targets instead of eight FP32 operations per target, and keeps only the minimum of a per
// (query, 32-target chunk).  Results never depend on it: with u = 2^-24, |a + |q|^2 - d| <= u (21 |t|^2 + 15 |q|^2) for
// the oracle's fp32 distance d (3 roundings in |t|^2, 3 in the FMAs on partial sums <= 2|t|^2 + |q|^2, <= 6 relative
// roundings in d <= 2|q|^2 + 2|t|^2), so the chunk that holds the exact nearest neighbour k* satisfies, when it is
// scanned and at any later time,
//     chunk minimum <= (running minimum of a) + E2,   E2 = 2^-18 (max|t|^2 seen so far + |q|^2)   (> twice that bound).
// Such a chunk is remembered per query when it is scanned (the most recent one in registers; when it is displaced and
// still qualifies it moves into a bit mask), and before the tile leaves shared memory the remembered chunks (one,
// rarely two) are re-scanned with the oracle's arithmetic (rescan_chunk), which alone decides
// distance and index.  Non-finite or huge coordinates make E2 infinite, i.e. everything is re-scanned: slower, still exact.
template <bool FMA>
__global__ void __launch_bounds__(C3_THREADS, PCL_C3_MINB)
chamfer_nn3_kernel(Pts x, const int64_t *__restrict__ x_len, Pts y, const int64_t *__restrict__ y_len, int P1, int P2,
                   float *__restrict__ dist_x, int *__restrict__ idx_x, float *__restrict__ dist_y,
                   int *__restrict__ idx_y, float *__restrict__ partial, int nblk, unsigned *__restrict__ ticket,
                   float *__restrict__ loss_xy) {
    __shared__ float4 tA[C3_TILE / 2 + C3_GROUP];  // per pair of targets {x0, x1, y0, y1} (+ slack for the read-ahead)
    __shared__ float4 tB[C3_TILE / 2 + C3_GROUP];  //                     {z0, z1, |t0|^2, |t1|^2}
    constexpr int C3_PPT = C3_TILE / C3_THREADS;   // staged points per thread and tile
    constexpr int CP = C3_CHUNK / 2;               // pairs per chunk
    __shared__ float red[C3_THREADS / 32];
    __shared__ int tmax_bits;
    const int dir = blockIdx.z, n = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wq = (tid >> 5) % C3_WQ, part = (tid >> 5) / C3_WQ;
    const Pts q = dir ? y : x, t = dir ? x : y;
    const int PQ = dir ? P2 : P1;
    const int q0 = blockIdx.x * C3_QUERIES;
    if (q0 >= PQ) {  // block-uniform: beyond the shorter cloud -- contributes a zero partial (and may be the last CTA)
        finish_block(0.f, partial, nblk, dir, n, ticket, P1, P2, x_len, y_len, loss_xy);
        return;
    }
    const int lq = dir ? len_of(y_len, n, P2) : len_of(x_len, n, P1);
    const int lt = dir ? len_of(x_len, n, P1) : len_of(y_len, n, P2);
    float *dist = (dir ? dist_y : dist_x) + (size_t)n * PQ;
    int *idx = (dir ? idx_y : idx_x) + (size_t)n * PQ;
    const float INF = __int_as_float(0x7f800000);

    // query r of a lane: q0 + 32 (r WQ + wq) + lane; the PARTS warps with the same wq hold the same queries
    float qx[C3_QPT], qy[C3_QPT], qz[C3_QPT], q2[C3_QPT], best[C3_QPT], mrun[C3_QPT];
    u64 nqx[C3_QPT], nqy[C3_QPT], nqz[C3_QPT];
    int bi[C3_QPT];
#pragma unroll
    for (int r = 0; r < C3_QPT; r++) {
        const int i = q0 + (r * C3_WQ + wq) * 32 + lane;
        float3 p = make_float3(0.f, 0.f, 0.f);
        if (i < lq) p = ld_xyz(q, n, i);
        qx[r] = p.x; qy[r] = p.y; qz[r] = p.z;
        q2[r] = finite_or_inf(__fmaf_rn(p.z, p.z, __fmaf_rn(p.y, p.y, __fmul_rn(p.x, p.x))));
        nqx[r] = pk2(-2.f * p.x, -2.f * p.x); nqy[r] = pk2(-2.f * p.y, -2.f * p.y); nqz[r] = pk2(-2.f * p.z, -2.f * p.z);
        best[r] = INF; bi[r] = 0x7fffffff; mrun[r] = INF;
    }
    if (q0 < lq && lt > 0) {  // block-uniform: blocks made only of padded rows skip the scan
        if (tid == 0) tmax_bits = 0;
        float3 pre[C3_PPT];  // points of the next tile: loaded before the exact re-scans of the current one, stored after them
        auto prefetch = [&](int t0) {
#pragma unroll
            for (int k = 0; k < C3_PPT; k++) {
                const int j = t0 + k * C3_THREADS + tid;
                pre[k] = (j < lt) ? ld_xyz(t, n, j) : make_float3(0.f, 0.f, 0.f);
            }
        };
        prefetch(0);
        __syncthreads();
        for (int t0 = 0; t0 < lt; t0 += C3_TILE) {
            const int cnt = min(C3_TILE, lt - t0);
            const int nch = (cnt + C3_CHUNK - 1) / C3_CHUNK;
            {   // registers -> shared memory (pair layout), |t|^2, running maximum of |t|^2; padding: a = +inf, never a minimum
                float wmax = 0.f;
                float *fA = reinterpret_cast<float *>(tA), *fB = reinterpret_cast<float *>(tB);
#pragma unroll
                for (int k = 0; k < C3_PPT; k++) {
                    const int j = k * C3_THREADS + tid;
                    const float3 p = pre[k];
                    float w = __fmaf_rn(p.z, p.z, __fmaf_rn(p.y, p.y, __fmul_rn(p.x, p.x)));
                    if (j < cnt) wmax = fmaxf(wmax, finite_or_inf(w)); else w = INF;
                    const int o = (j >> 1) * 4 + (j & 1);
                    fA[o] = p.x; fA[o + 2] = p.y; fB[o] = p.z; fB[o + 2] = w;
                }
                const int wm = __reduce_max_sync(0xffffffffu, __float_as_int(wmax));  // wmax >= 0: integer order == float order
                if (lane == 0) atomicMax(&tmax_bits, wm);
            }
            __syncthreads();
            const float tmax = __int_as_float(tmax_bits);
            float e2[C3_QPT], thr[C3_QPT], lm[C3_QPT];
            int lcid[C3_QPT];       // chunk of the most recent candidate (lm = its approximate minimum)
            unsigned dmask[C3_QPT]; // displaced candidates that still qualified when they were displaced
#pragma unroll
            for (int r = 0; r < C3_QPT; r++) {
                e2[r] = fmaxf(__fmul_ru(__fadd_ru(tmax, q2[r]), 3.8147e-6f /* > 2^-18 */), 1e-36f);
                thr[r] = __fadd_ru(mrun[r], e2[r]);
                lm[r] = INF; lcid[r] = 0; dmask[r] = 0;
            }
            float4 ga[C3_GROUP], gb[C3_GROUP];  // current group of pairs; the next one is loaded while this one is used
#pragma unroll
            for (int i = 0; i < C3_GROUP; i++) { ga[i] = tA[part * CP + i]; gb[i] = tB[part * CP + i]; }
            for (int c = part; c < nch; c += C3_PARTS) {
                float mc[C3_QPT];
#pragma unroll
                for (int r = 0; r < C3_QPT; r++) mc[r] = INF;
#pragma unroll
                for (int g = 0; g < CP / C3_GROUP; g++) {
                    float4 na[C3_GROUP], nb[C3_GROUP];
                    // next group of this chunk, or the first group of this warp's next chunk (clamped into the slack at the end)
                    const int nxt = min((g + 1 < CP / C3_GROUP) ? c * CP + (g + 1) * C3_GROUP : (c + C3_PARTS) * CP, C3_TILE / 2);
#pragma unroll
                    for (int i = 0; i < C3_GROUP; i++) { na[i] = tA[nxt + i]; nb[i] = tB[nxt + i]; }
#pragma unroll
                    for (int i = 0; i < C3_GROUP; i++) {
                        const u64 tx = pk2(ga[i].x, ga[i].y), ty = pk2(ga[i].z, ga[i].w), tz = pk2(gb[i].x, gb[i].y), tw = pk2(gb[i].z, gb[i].w);
#pragma unroll
                        for (int r = 0; r < C3_QPT; r++) {
                            const u64 v = ffma2(tz, nqz[r], ffma2(ty, nqy[r], ffma2(tx, nqx[r], tw)));
                            mc[r] = fmin3(mc[r], lo2(v), hi2(v));
                        }
                    }
#pragma unroll
                    for (int i = 0; i < C3_GROUP; i++) { ga[i] = na[i]; gb[i] = nb[i]; }
                }
#pragma unroll
                for (int r = 0; r < C3_QPT; r++) {  // branch-free: a chunk that may hold the exact nearest neighbour becomes the candidate
                    const bool cand = !(mc[r] > thr[r]);
                    const float nm = fminf(mrun[r], mc[r]);     // == mrun unless cand
                    const float nthr = __fadd_ru(nm, e2[r]);
                    const bool keep = cand && !(lm[r] > nthr);  // the displaced candidate still qualifies (lm = +inf: none yet)
                    dmask[r] |= keep ? (1u << lcid[r]) : 0u;
                    lm[r] = cand ? mc[r] : lm[r];
                    lcid[r] = cand ? c : lcid[r];
                    mrun[r] = nm; thr[r] = nthr;
                }
            }
            if (t0 + C3_TILE < lt) prefetch(t0 + C3_TILE);
            // exact re-scan of the remembered chunks while the tile is resident
#pragma unroll
            for (int r = 0; r < C3_QPT; r++) {
                unsigned m = dmask[r];
                if (!(lm[r] > thr[r])) m |= 1u << lcid[r];
                if (q0 + (r * C3_WQ + wq) * 32 + lane >= lq) m = 0;
                while (__any_sync(0xffffffffu, m != 0)) {
                    const bool act = m != 0;
                    const int c = act ? (__ffs(m) - 1) : 0;
                    m &= m - 1;
                    rescan_chunk<FMA>(tA, tB, act, c, cnt, t0, qx[r], qy[r], qz[r], nqx[r], nqy[r], nqz[r], thr[r], best[r], bi[r]);
                }
            }
            __syncthreads();
        }
    }
    // merge the parts (smaller distance, then lower index) -- the tile buffers are free now
    if constexpr (C3_PARTS > 1) {
        static_assert((C3_PARTS - 1) * C3_QUERIES * 4 <= (int)sizeof(float4) * (C3_TILE / 2), "merge buffer fits into a tile array");
        float *mb = reinterpret_cast<float *>(tA);
        int *mi = reinterpret_cast<int *>(tB);
        if (part > 0) {
#pragma unroll
            for (int r = 0; r < C3_QPT; r++) {
                mb[(part - 1) * C3_QUERIES + (r * C3_WQ + wq) * 32 + lane] = best[r];
                mi[(part - 1) * C3_QUERIES + (r * C3_WQ + wq) * 32 + lane] = bi[r];
            }
        }
        __syncthreads();
        if (part == 0) {
#pragma unroll
            for (int r = 0; r < C3_QPT; r++) {
#pragma unroll
                for (int pp = 1; pp < C3_PARTS; pp++) {
                    const float ob = mb[(pp - 1) * C3_QUERIES + (r * C3_WQ + wq) * 32 + lane];
                    const int oi = mi[(pp - 1) * C3_QUERIES + (r * C3_WQ + wq) * 32 + lane];
                    if (ob < best[r] || (ob == best[r] && oi < bi[r])) { best[r] = ob; bi[r] = oi; }
                }
            }
        }
    }
    float s = 0.f;
    if (part == 0) {
#pragma unroll
        for (int r = 0; r < C3_QPT; r++) {
            const int i = q0 + (r * C3_WQ + wq) * 32 + lane;
            if (i < PQ) {
                const bool valid = (i < lq) && (lt > 0);
                const float d = valid ? best[r] : 0.f;
                dist[i] = d; idx[i] = (valid && bi[r] != 0x7fffffff && best[r] < INF) ? bi[r] : 0;  // no finite distance: knn's initial index 0
                s += d;
            }
        }
    }
    s = block_sum<C3_THREADS / 32>(s, red);
    finish_block(s, partial, nblk, dir, n, ticket, P1, P2, x_len, y_len, loss_xy);
}


// ---- spatially pruned nearest neighbour for D == 3 (large clouds) ------------------------------------------------------------------
// The brute-force scan above is O(P1 * P2).  Here both clouds are first put into Morton order (cells of a 32^3 grid over their common
// bounding box; counting sort in shared memory; cell mates ranked by original index, so the order is a deterministic function of the
// input) and cut into tiles of 32 points with bounding boxes; then a warp of 32 neighbouring queries visits only the tiles whose box can
// still hold a nearer point: 32 tiles are box-tested per ballot against the warp's query box and its largest running minimum, survivors
// get the per-query test, and what is left is scanned with the ORACLE's arithmetic and the explicit rule "smaller distance, then lower
// original index".  A tile is skipped only when its box distance (shrunk by 2^-20 relative against rounding) is STRICTLY larger than the
// running minimum of every query, so distances, indices and the lowest-index tie rule are exactly the brute-force ones; non-finite
// coordinates switch the pruning off for the tiles / queries they touch (slower, still exact).
constexpr int PR_THREADS = 512;                 // sort kernel
constexpr int PR_CELL_BITS = 15;                // 32^3 Morton cells
constexpr int PR_CELLS = 1 << PR_CELL_BITS;
constexpr int PR_MAX_P = 16384;                 // shared memory of the sort: 128 KB histogram + 4 B per point
constexpr int PR_NN_WARPS = 4;                  // nearest-neighbour kernel: 4 warps x 32 queries per CTA

struct PruneWs {                                // workspace regions, per direction d (0: cloud x, 1: cloud y)
    float4 *pts[2];                             // B x Ppad sorted points {x, y, z, original index bits}, Ppad = P rounded up to 32
    float4 *box[2];                             // B x NT x 2: {min xyz, flag (1: some point of the tile is not finite)}, {max xyz, -}
    int ppad[2], nt[2];
};

__device__ __forceinline__ unsigned spread5(unsigned v) {  // 5 bits -> every third bit
    v = (v | (v << 8)) & 0x0000100Fu;
    v = (v | (v << 4)) & 0x000010C3u;
    v = (v | (v << 2)) & 0x00001249u;
    return v;
}
__device__ __forceinline__ bool finite3(float3 p) { return fabsf(p.x) <= 3.0e38f && fabsf(p.y) <= 3.0e38f && fabsf(p.z) <= 3.0e38f; }

// grid (B, 2): CTA (n, d) sorts the first len points of cloud d of batch element n and zero-fills the outputs of its padded rows.
__global__ void __launch_bounds__(PR_THREADS, 1)
chamfer_sort_kernel(Pts x, const int64_t *__restrict__ x_len, Pts y, const int64_t *__restrict__ y_len, int P1, int P2, PruneWs W,
                    float *__restrict__ dist_x, int *__restrict__ idx_x, float *__restrict__ dist_y, int *__restrict__ idx_y) {
    extern __shared__ __align__(16) unsigned char pr_smem[];
    int *hist = reinterpret_cast<int *>(pr_smem);                 // PR_CELLS cell counts, then offsets | arrivals << 16
    unsigned *tmp = reinterpret_cast<unsigned *>(hist + PR_CELLS + 32);  // P (cell-ordered original indices)
    __shared__ float red[6][PR_THREADS / 32];
    __shared__ float bb[6];
    const int n = blockIdx.x, d = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const Pts me = d ? y : x, other = d ? x : y;
    const int P = d ? P2 : P1;
    const int len = d ? len_of(y_len, n, P2) : len_of(x_len, n, P1), olen = d ? len_of(x_len, n, P1) : len_of(y_len, n, P2);
    float *dist = (d ? dist_y : dist_x) + (size_t)n * P;
    int *idx = (d ? idx_y : idx_x) + (size_t)n * P;
    for (int i = len + tid; i < P; i += PR_THREADS) { dist[i] = 0.f; idx[i] = 0; }  // padded rows (knn leaves them at 0)
    // common bounding box of both clouds (finite coordinates only): the two directions use the same grid
    float lo[3] = {3e38f, 3e38f, 3e38f}, hi[3] = {-3e38f, -3e38f, -3e38f};
    for (int pass = 0; pass < 2; pass++) {
        const Pts &c = pass ? other : me;
        const int l = pass ? olen : len;
        for (int i = tid; i < l; i += PR_THREADS) {
            const float3 p = ld_xyz(c, n, i);
            if (finite3(p)) {
                lo[0] = fminf(lo[0], p.x); lo[1] = fminf(lo[1], p.y); lo[2] = fminf(lo[2], p.z);
                hi[0] = fmaxf(hi[0], p.x); hi[1] = fmaxf(hi[1], p.y); hi[2] = fmaxf(hi[2], p.z);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o)); hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o)); }
        if (lane == 0) { red[k][wid] = lo[k]; red[3 + k][wid] = hi[k]; }
    }
    for (int c = tid; c < PR_CELLS + 32; c += PR_THREADS) hist[c] = 0;
    __syncthreads();
    if (tid < 6) {
        float v = red[tid][0];
        for (int w = 1; w < PR_THREADS / 32; w++) v = tid < 3 ? fminf(v, red[tid][w]) : fmaxf(v, red[tid][w]);
        bb[tid] = v;
    }
    __syncthreads();
    float sc[3];
#pragma unroll
    for (int k = 0; k < 3; k++) sc[k] = (bb[3 + k] > bb[k]) ? 32.f / (bb[3 + k] - bb[k]) : 0.f;
    auto cell_of = [&](float3 p) -> int {
        if (!finite3(p)) return PR_CELLS - 1;
        const unsigned qx = (unsigned)min(max((int)((p.x - bb[0]) * sc[0]), 0), 31), qy = (unsigned)min(max((int)((p.y - bb[1]) * sc[1]), 0), 31),
                       qz = (unsigned)min(max((int)((p.z - bb[2]) * sc[2]), 0), 31);
        return (int)(spread5(qx) | (spread5(qy) << 1) | (spread5(qz) << 2));
    };
    for (int i = tid; i < len; i += PR_THREADS) atomicAdd(&hist[cell_of(ld_xyz(me, n, i))], 1);
    __syncthreads();
    {   // exclusive prefix sum over the cells: 64 consecutive cells per thread + block scan
        constexpr int CPT = PR_CELLS / PR_THREADS;
        int sum = 0;
        for (int i = 0; i < CPT; i++) sum += hist[tid * CPT + i];
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
        __shared__ int wsum[PR_THREADS / 32];
        if (lane == 31) wsum[wid] = incl;
        __syncthreads();
        int base = incl - sum;
        for (int w = 0; w < wid; w++) base += wsum[w];
        for (int i = 0; i < CPT; i++) { const int v = hist[tid * CPT + i]; hist[tid * CPT + i] = base; base += v; }
    }
    __syncthreads();
    // Cell mates in arrival order (tmp), then every point takes the rank of its original index among them: a deterministic order
    // (the per-CTA partial sums of the loss depend on it).  The arrival counter of a cell lives in the upper half of its offset word
    // (offsets and counts are <= 16384 = PR_MAX_P).
    for (int i = tid; i < len; i += PR_THREADS) {
        const int c = cell_of(ld_xyz(me, n, i));
        const unsigned old = (unsigned)atomicAdd(&hist[c], 0x10000);
        tmp[(old & 0xffffu) + (old >> 16)] = (unsigned)i;
    }
    __syncthreads();
    float4 *out = W.pts[d] + (size_t)n * W.ppad[d];
    for (int i = tid; i < len; i += PR_THREADS) {
        const float3 p = ld_xyz(me, n, i);
        const unsigned h = (unsigned)hist[cell_of(p)];
        const int s0 = (int)(h & 0xffffu), s1 = s0 + (int)(h >> 16);
        int pos = s0;
        for (int q = s0; q < s1; q++) pos += (tmp[q] < (unsigned)i) ? 1 : 0;
        out[pos] = make_float4(p.x, p.y, p.z, __int_as_float(i));
    }
    const int NT = W.nt[d];
    for (int i = len + tid; i < NT * 32 && i < W.ppad[d]; i += PR_THREADS) out[i] = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7fffffff));  // tail of the last tile (never read as a point: j < cnt)
    __threadfence_block();
    __syncthreads();
    float4 *box = W.box[d] + (size_t)n * NT * 2;
    for (int t = wid; t * 32 < len; t += PR_THREADS / 32) {
        const int i = t * 32 + lane;
        const bool ok = i < len;
        const float4 p = ok ? out[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        const bool fin = !ok || finite3(make_float3(p.x, p.y, p.z));
        float l0 = (ok && fin) ? p.x : 3e38f, l1 = (ok && fin) ? p.y : 3e38f, l2 = (ok && fin) ? p.z : 3e38f;
        float h0 = (ok && fin) ? p.x : -3e38f, h1 = (ok && fin) ? p.y : -3e38f, h2 = (ok && fin) ? p.z : -3e38f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            l0 = fminf(l0, __shfl_xor_sync(0xffffffffu, l0, o)); l1 = fminf(l1, __shfl_xor_sync(0xffffffffu, l1, o)); l2 = fminf(l2, __shfl_xor_sync(0xffffffffu, l2, o));
            h0 = fmaxf(h0, __shfl_xor_sync(0xffffffffu, h0, o)); h1 = fmaxf(h1, __shfl_xor_sync(0xffffffffu, h1, o)); h2 = fmaxf(h2, __shfl_xor_sync(0xffffffffu, h2, o));
        }
        const bool anybad = __any_sync(0xffffffffu, !fin);
        if (lane == 0) { box[2 * t] = make_float4(l0, l1, l2, anybad ? 1.f : 0.f); box[2 * t + 1] = make_float4(h0, h1, h2, 0.f); }
    }
}

// squared distance between two boxes / a point and a box (0 inside); NaN-free for finite boxes
__device__ __forceinline__ float box_gap2(float alo, float ahi, float blo, float bhi) {
    const float g = fmaxf(fmaxf(blo - ahi, alo - bhi), 0.f);
    return g * g;
}

// grid (ceil(maxP / 128), B, 2): warp = 32 consecutive queries of the SORTED query cloud.
template <bool FMA>
__global__ void __launch_bounds__(PR_NN_WARPS * 32)
chamfer_nn3_pruned_kernel(const int64_t *__restrict__ x_len, const int64_t *__restrict__ y_len, int P1, int P2, PruneWs W,
                          float *__restrict__ dist_x, int *__restrict__ idx_x, float *__restrict__ dist_y, int *__restrict__ idx_y,
                          float *__restrict__ partial, int nblk, unsigned *__restrict__ ticket, float *__restrict__ loss_xy) {
    __shared__ float red[PR_NN_WARPS];
    const int dir = blockIdx.z, n = blockIdx.y, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int PQ = dir ? P2 : P1;
    const int q0 = (blockIdx.x * PR_NN_WARPS + wid) * 32;
    const int lq = dir ? len_of(y_len, n, P2) : len_of(x_len, n, P1);
    const int lt = dir ? len_of(x_len, n, P1) : len_of(y_len, n, P2);
    const int dq = dir, dt = dir ^ 1;
    const float INF = __int_as_float(0x7f800000);
    float s = 0.f;
    if (q0 < lq) {  // warp-uniform
        const float4 *qp = W.pts[dq] + (size_t)n * W.ppad[dq];
        const float4 *tp = W.pts[dt] + (size_t)n * W.ppad[dt];
        const float4 *tb = W.box[dt] + (size_t)n * W.nt[dt] * 2;
        const bool valid = q0 + lane < lq;
        const float4 q = valid ? qp[q0 + lane] : qp[q0];           // surplus lanes shadow the first query (results discarded)
        const int qi = __float_as_int(q.w);
        float best = INF;
        int bi = 0x7fffffff;
        if (lt > 0) {
            const int NTt = (lt + 31) >> 5;
            // the warp's query box; a non-finite query makes it infinite (nothing is pruned by the bulk test)
            const bool qfin = finite3(make_float3(q.x, q.y, q.z));
            float bl0 = q.x, bl1 = q.y, bl2 = q.z, bh0 = q.x, bh1 = q.y, bh2 = q.z;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                bl0 = fminf(bl0, __shfl_xor_sync(0xffffffffu, bl0, o)); bl1 = fminf(bl1, __shfl_xor_sync(0xffffffffu, bl1, o)); bl2 = fminf(bl2, __shfl_xor_sync(0xffffffffu, bl2, o));
                bh0 = fmaxf(bh0, __shfl_xor_sync(0xffffffffu, bh0, o)); bh1 = fmaxf(bh1, __shfl_xor_sync(0xffffffffu, bh1, o)); bh2 = fmaxf(bh2, __shfl_xor_sync(0xffffffffu, bh2, o));
            }
            const bool allfin = __all_sync(0xffffffffu, qfin);
            auto scan = [&](int tl) {
                const int cnt = min(32, lt - tl * 32);
                const float4 *tt = tp + (size_t)tl * 32;
#pragma unroll 4
                for (int j = 0; j < cnt; j++) {
                    const float4 t = __ldg(tt + j);
                    const float dd = sqdist3<FMA>(q.x, q.y, q.z, t);
                    const int ti = __float_as_int(t.w);
                    if (dd < best || (dd == best && ti < bi)) { best = dd; bi = ti; }
                }
            };
            auto lane_skips = [&](const float4 &lo, const float4 &hi) -> bool {  // this query cannot find anything nearer (or equal) in the tile
                const float d2 = box_gap2(q.x, q.x, lo.x, hi.x) + box_gap2(q.y, q.y, lo.y, hi.y) + box_gap2(q.z, q.z, lo.z, hi.z);
                return lo.w == 0.f && (d2 * 0.999999f > best);
            };
            // Seed: the tile whose box is nearest to the warp's query box (32 boxes per round, warp arg-min) gives every query a tight
            // running minimum before the candidates are collected; the guess by rank (both clouds are sorted along the same curve) is
            // the fall-back when no finite box distance exists.
            int tg = min((int)(((long long)q0 * NTt) / max(lq, 1)), NTt - 1);
            {
                float dmin = INF;
                int tmin = -1;
                for (int tb0 = 0; tb0 < NTt; tb0 += 32) {
                    const int tl = tb0 + lane;
                    if (tl < NTt) {
                        const float4 lo = __ldg(tb + 2 * tl), hi = __ldg(tb + 2 * tl + 1);
                        const float d2 = box_gap2(bl0, bh0, lo.x, hi.x) + box_gap2(bl1, bh1, lo.y, hi.y) + box_gap2(bl2, bh2, lo.z, hi.z);
                        if (lo.w == 0.f && d2 < dmin) { dmin = d2; tmin = tl; }
                    }
                }
                const int key = __reduce_min_sync(0xffffffffu, (dmin < INF) ? __float_as_int(dmin) : 0x7f800000);  // d2 >= 0: integer order == float order
                const unsigned who = __ballot_sync(0xffffffffu, tmin >= 0 && __float_as_int(dmin) == key);
                if (allfin && who) tg = __shfl_sync(0xffffffffu, tmin, __ffs(who) - 1);
            }
            scan(tg);
            for (int tb0 = 0; tb0 < NTt; tb0 += 32) {
                const int tl = tb0 + lane;
                // largest running minimum of the warp (best >= 0 or +inf / NaN-free: integer order == float order)
                const float bmax = __int_as_float(__reduce_max_sync(0xffffffffu, __float_as_int(best)));
                bool cand = false;
                if (tl < NTt && tl != tg) {
                    const float4 lo = __ldg(tb + 2 * tl), hi = __ldg(tb + 2 * tl + 1);
                    const float d2 = box_gap2(bl0, bh0, lo.x, hi.x) + box_gap2(bl1, bh1, lo.y, hi.y) + box_gap2(bl2, bh2, lo.z, hi.z);
                    cand = !(allfin && lo.w == 0.f && d2 * 0.999999f > bmax);
                }
                unsigned cm = __ballot_sync(0xffffffffu, cand);
                while (cm) {
                    const int t2 = tb0 + __ffs(cm) - 1;
                    cm &= cm - 1;
                    const float4 lo = __ldg(tb + 2 * t2), hi = __ldg(tb + 2 * t2 + 1);
                    if (__all_sync(0xffffffffu, lane_skips(lo, hi))) continue;
                    scan(t2);
                }
            }
        }
        if (valid) {
            const bool ok = lt > 0;
            const float dres = ok ? best : 0.f;
            float *dist = (dir ? dist_y : dist_x) + (size_t)n * PQ;
            int *idx = (dir ? idx_y : idx_x) + (size_t)n * PQ;
            dist[qi] = dres;
            idx[qi] = (ok && bi != 0x7fffffff && best < INF) ? bi : 0;
            s = dres;
        }
    }
    s = block_sum<PR_NN_WARPS>(s, red);
    finish_block(s, partial, nblk, dir, n, ticket, P1, P2, x_len, y_len, loss_xy);
}

// Generic feature width (ChamferDistance over all channels, utils.py:209-211).  One query per thread.
template <bool FMA, int D>
__global__ void __launch_bounds__(CH_THREADS)
chamfer_nnD_kernel(Pts x, const int64_t *__restrict__ x_len, Pts y, const int64_t *__restrict__ y_len, int P1, int P2,
                   float *__restrict__ dist_x, int *__restrict__ idx_x, float *__restrict__ dist_y,
                   int *__restrict__ idx_y, float *__restrict__ partial, int nblk, unsigned *__restrict__ ticket,
                   float *__restrict__ loss_xy) {
    constexpr int TILE = 512;
    __shared__ float tile[TILE * D];
    __shared__ float red[4];
    const int dir = blockIdx.z, n = blockIdx.y;
    const Pts q = dir ? y : x, t = dir ? x : y;
    const int PQ = dir ? P2 : P1;
    const int q0 = blockIdx.x * CH_THREADS;
    if (q0 >= PQ) {
        finish_block(0.f, partial, nblk, dir, n, ticket, P1, P2, x_len, y_len, loss_xy);
        return;
    }
    const int lq = dir ? len_of(y_len, n, P2) : len_of(x_len, n, P1);
    const int lt = dir ? len_of(x_len, n, P1) : len_of(y_len, n, P2);
    float *dist = (dir ? dist_y : dist_x) + (size_t)n * PQ;
    int *idx = (dir ? idx_y : idx_x) + (size_t)n * PQ;
    const int i = q0 + threadIdx.x;
    float qv[D];
#pragma unroll
    for (int c = 0; c < D; c++) qv[c] = (i < lq) ? ld_any(q, (int64_t)n * q.bs + (int64_t)i * q.rs + c) : 0.f;
    float best = __int_as_float(0x7f800000);
    int bi = 0;
    if (q0 < lq) {
        for (int t0 = 0; t0 < lt; t0 += TILE) {
            const int cnt = min(TILE, lt - t0);
            for (int e = threadIdx.x; e < cnt * D; e += CH_THREADS) {
                const int j = e / D, c = e - j * D;
                tile[e] = ld_any(t, (int64_t)n * t.bs + (int64_t)(t0 + j) * t.rs + c);
            }
            __syncthreads();
#pragma unroll 2
            for (int j = 0; j < cnt; j++) {
                float d = 0.f;
#pragma unroll
                for (int c = 0; c < D; c++) {
                    const float df = __fsub_rn(qv[c], tile[j * D + c]);
                    if constexpr (FMA) d = __fmaf_rn(df, df, d);
                    else d = __fadd_rn(d, __fmul_rn(df, df));
                }
                if (d < best) { best = d; bi = t0 + j; }
            }
            __syncthreads();
        }
    }
    float s = 0.f;
    if (i < PQ) {
        const bool valid = (i < lq) && (lt > 0);
        s = valid ? best : 0.f;
        dist[i] = s; idx[i] = valid ? bi : 0;
    }
    s = block_sum<4>(s, red);
    finish_block(s, partial, nblk, dir, n, ticket, P1, P2, x_len, y_len, loss_xy);
}

// Backward: grid (ceil(maxP/256), B, 2).  All contributions go through fp32 red.global.add onto
// zero-filled outputs (same accumulation model as pytorch3d's CUDA knn backward).
__global__ void __launch_bounds__(256)
chamfer_bwd_kernel(Pts x, const int64_t *__restrict__ x_len, Pts y, const int64_t *__restrict__ y_len, int B, int P1,
                   int P2, int D, const int *__restrict__ idx_x, const int *__restrict__ idx_y,
                   const float *__restrict__ grad_out, float g_imm_x, float g_imm_y, float *__restrict__ grad_x,
                   float *__restrict__ grad_y) {
    const int dir = blockIdx.z, n = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const Pts q = dir ? y : x, t = dir ? x : y;
    const int PQ = dir ? P2 : P1, PT = dir ? P1 : P2;
    const int lq = dir ? len_of(y_len, n, P2) : len_of(x_len, n, P1);
    const int lt = dir ? len_of(x_len, n, P1) : len_of(y_len, n, P2);
    if (i >= lq || lt <= 0) return;
    const float g = grad_out ? __ldg(grad_out + dir) : (dir ? g_imm_y : g_imm_x);  // upstream gradient: device scalar or immediate
    const float gd = g / (float)(B > 1 ? B : 1) / (float)(lq > 1 ? lq : 1);
    const int j = (dir ? idx_y : idx_x)[(size_t)n * PQ + i];
    float *gq = (dir ? grad_y : grad_x) + ((size_t)n * PQ + i) * D;
    float *gt = (dir ? grad_x : grad_y) + ((size_t)n * PT + j) * D;
    const int64_t qo = (int64_t)n * q.bs + (int64_t)i * q.rs, to = (int64_t)n * t.bs + (int64_t)j * t.rs;
    for (int c = 0; c < D; c++) {
        const float diff = __fmul_rn(__fmul_rn(2.0f, gd), __fsub_rn(ld_any(q, qo + c), ld_any(t, to + c)));
        atomicAdd(gq + c, diff);
        atomicAdd(gt + c, -diff);
    }
}

template <bool FMA>
int launch_fwd(const Pts &x, const int64_t *x_len, const Pts &y, const int64_t *y_len, int B, int P1, int P2, int D,
               float *dist_x, int *idx_x, float *dist_y, int *idx_y, float *partial, int nblk, unsigned *ticket, float *loss_xy,
               cudaStream_t st) {
    const int maxP = P1 > P2 ? P1 : P2;
    if (D == 3) {
        dim3 grid((maxP + C3_QUERIES - 1) / C3_QUERIES, B, 2);
        chamfer_nn3_kernel<FMA><<<grid, C3_THREADS, 0, st>>>(x, x_len, y, y_len, P1, P2, dist_x, idx_x, dist_y, idx_y, partial, nblk, ticket, loss_xy);
    } else {
        dim3 grid((maxP + CH_THREADS - 1) / CH_THREADS, B, 2);
#define PCL_LAUNCH_NND(DD) \
    case DD: chamfer_nnD_kernel<FMA, DD><<<grid, CH_THREADS, 0, st>>>(x, x_len, y, y_len, P1, P2, dist_x, idx_x, dist_y, idx_y, partial, nblk, ticket, loss_xy); break
        switch (D) {
            PCL_LAUNCH_NND(1); PCL_LAUNCH_NND(2); PCL_LAUNCH_NND(4); PCL_LAUNCH_NND(5);
            PCL_LAUNCH_NND(6); PCL_LAUNCH_NND(7); PCL_LAUNCH_NND(8);
            default: set_error("chamfer: D=%d unsupported (1..8)", D); return PCL_E_UNSUPPORTED;
        }
#undef PCL_LAUNCH_NND
    }
    return PCL_OK;
}

int check_args(const void *x, int x_dtype, const void *y, int y_dtype, int B, int P1, int P2, int D) {
    if (B < 0 || P1 < 0 || P2 < 0) { set_error("chamfer: negative size B=%d P1=%d P2=%d", B, P1, P2); return PCL_E_SHAPE; }
    if (D < 1 || D > 8) { set_error("chamfer: D=%d unsupported (1..8)", D); return PCL_E_UNSUPPORTED; }
    if (B > 65535) { set_error("chamfer: B=%d > 65535", B); return PCL_E_SHAPE; }
    if (!dtype_ok(x_dtype) || !dtype_ok(y_dtype)) { set_error("chamfer: bad dtype"); return PCL_E_ARG; }
    if (B > 0 && ((P1 > 0 && !x) || (P2 > 0 && !y))) { set_error("chamfer: null input"); return PCL_E_ARG; }
    return PCL_OK;
}

// workspace of the pruned path, behind [ticket][partials]: sorted clouds and tile boxes of both directions
inline size_t prune_bytes(int B, int P1, int P2) {
    if (B <= 0 || P1 <= 0 || P2 <= 0 || P1 > PR_MAX_P || P2 > PR_MAX_P) return 0;
    size_t o = 0;
    for (int d = 0; d < 2; d++) {
        const size_t ppad = (size_t)((d ? P2 : P1) + 31) / 32 * 32;
        o += align_up((size_t)B * ppad * sizeof(float4), 256) + align_up((size_t)B * (ppad / 32) * 2 * sizeof(float4), 256);
    }
    return o;
}
inline PruneWs prune_ws(unsigned char *base, int B, int P1, int P2) {
    PruneWs W;
    size_t o = 0;
    for (int d = 0; d < 2; d++) {
        const size_t ppad = (size_t)((d ? P2 : P1) + 31) / 32 * 32;
        W.ppad[d] = (int)ppad; W.nt[d] = (int)(ppad / 32);
        W.pts[d] = reinterpret_cast<float4 *>(base + o); o += align_up((size_t)B * ppad * sizeof(float4), 256);
        W.box[d] = reinterpret_cast<float4 *>(base + o); o += align_up((size_t)B * (ppad / 32) * 2 * sizeof(float4), 256);
    }
    return W;
}
// smallest min(P1, P2) that takes the pruned path (0: never).  Measured on B200 (profiles/r2_s2_chamfer_pruned.txt): the brute-force
// kernel evaluates a pair in 2.5 instructions, the pruned scan in ~12 (oracle arithmetic) on the ~30 % / 6 % of the pairs that survive
// at N = 2048 / 16384 -- the crossover is near 6000 points.  pcl_chamfer_set_prune_min overrides it.
int g_prune_min = -1;
inline int prune_min() { return g_prune_min >= 0 ? g_prune_min : 6144; }

inline int nblk_for(int P1, int P2) {
    const int maxP = P1 > P2 ? P1 : P2;
    constexpr int G = C3_QUERIES < CH_THREADS ? C3_QUERIES : CH_THREADS;  // queries per CTA of the finer-grained kernel
    return (maxP + G - 1) / G + 1;
}

}  // namespace
}  // namespace pcl

using namespace pcl;

extern "C" int pcl_chamfer_set_prune_min(int min_points) {
    g_prune_min = min_points;  // < 0: back to the default
    return PCL_OK;
}

extern "C" size_t pcl_chamfer_workspace_bytes(int B, int P1, int P2) {
    if (B <= 0) return 256;
    return 256 + align_up((size_t)2 * B * nblk_for(P1, P2) * sizeof(float), 256) + prune_bytes(B, P1, P2);  // [ticket][per-CTA partial sums][sorted clouds + tile boxes of the pruned path]
}

extern "C" int pcl_chamfer_fwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len,
                               const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *y_len, int B,
                               int P1, int P2, int D, int mode, float *dist_x, int32_t *idx_x, float *dist_y,
                               int32_t *idx_y, float *loss_xy, void *workspace, size_t workspace_bytes, void *stream) {
    int rc = check_args(x, x_dtype, y, y_dtype, B, P1, P2, D);
    if (rc) return rc;
    if (mode != PCL_CHAMFER_UNFUSED && mode != PCL_CHAMFER_FMA) { set_error("chamfer: bad mode %d", mode); return PCL_E_ARG; }
    if (!loss_xy || (B > 0 && ((P1 > 0 && (!dist_x || !idx_x)) || (P2 > 0 && (!dist_y || !idx_y))))) {
        set_error("chamfer: null output"); return PCL_E_ARG;
    }
    if (workspace_bytes < pcl_chamfer_workspace_bytes(B, P1, P2) || !workspace) {
        set_error("chamfer: workspace too small (%zu < %zu)", workspace_bytes, pcl_chamfer_workspace_bytes(B, P1, P2));
        return PCL_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    if (B == 0 || (P1 == 0 && P2 == 0)) {
        PCL_CUDA(cudaMemsetAsync(loss_xy, 0, 4 * sizeof(float), st));
        return PCL_OK;
    }
    const Pts xp{x, x_bs, x_rs, x_dtype}, yp{y, y_bs, y_rs, y_dtype};
    unsigned *ticket = (unsigned *)workspace;
    float *partial = (float *)((unsigned char *)workspace + 256);
    const int nblk = nblk_for(P1, P2);
    PCL_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned), st));  // every CTA writes its partial (zeros beyond the shorter cloud); the last one sums
    const int pmin = P1 < P2 ? P1 : P2;
    if (D == 3 && prune_min() > 0 && pmin >= prune_min() && prune_bytes(B, P1, P2) > 0) {
        // large clouds: Morton order + tile boxes, then a nearest-neighbour scan that only visits the tiles that can matter
        const PruneWs W = prune_ws((unsigned char *)workspace + 256 + align_up((size_t)2 * B * nblk * sizeof(float), 256), B, P1, P2);
        const int maxP = P1 > P2 ? P1 : P2;
        const size_t smem = (size_t)(PR_CELLS + 32) * sizeof(int) + (size_t)maxP * sizeof(unsigned);
        static thread_local int attr_dev = -1;
        int dev = 0;
        PCL_CUDA(cudaGetDevice(&dev));
        if (attr_dev != dev) {
            PCL_CUDA(cudaFuncSetAttribute(chamfer_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((PR_CELLS + 32) * sizeof(int) + PR_MAX_P * sizeof(unsigned))));
            attr_dev = dev;
        }
        chamfer_sort_kernel<<<dim3(B, 2), PR_THREADS, smem, st>>>(xp, x_len, yp, y_len, P1, P2, W, dist_x, (int *)idx_x, dist_y, (int *)idx_y);
        PCL_CUDA(cudaGetLastError());
        const dim3 grid((maxP + PR_NN_WARPS * 32 - 1) / (PR_NN_WARPS * 32), B, 2);
        if (mode == PCL_CHAMFER_FMA)
            chamfer_nn3_pruned_kernel<true><<<grid, PR_NN_WARPS * 32, 0, st>>>(x_len, y_len, P1, P2, W, dist_x, (int *)idx_x, dist_y, (int *)idx_y, partial, nblk, ticket, loss_xy);
        else
            chamfer_nn3_pruned_kernel<false><<<grid, PR_NN_WARPS * 32, 0, st>>>(x_len, y_len, P1, P2, W, dist_x, (int *)idx_x, dist_y, (int *)idx_y, partial, nblk, ticket, loss_xy);
        PCL_CUDA(cudaGetLastError());
        return PCL_OK;
    }
    rc = (mode == PCL_CHAMFER_FMA)
             ? launch_fwd<true>(xp, x_len, yp, y_len, B, P1, P2, D, dist_x, idx_x, dist_y, idx_y, partial, nblk, ticket, loss_xy, st)
             : launch_fwd<false>(xp, x_len, yp, y_len, B, P1, P2, D, dist_x, idx_x, dist_y, idx_y, partial, nblk, ticket, loss_xy, st);
    if (rc) return rc;
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

// shared by pcl_chamfer_bwd (upstream gradients on the device) and the composite step (immediate upstream gradients)
int pcl::chamfer_bwd_impl(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len, const void *y, int y_dtype,
                          int64_t y_bs, int64_t y_rs, const int64_t *y_len, int B, int P1, int P2, int D, const int32_t *idx_x,
                          const int32_t *idx_y, const float *grad_out, float g_imm_x, float g_imm_y, float *grad_x, float *grad_y,
                          cudaStream_t st, bool outputs_are_zero) {
    int rc = check_args(x, x_dtype, y, y_dtype, B, P1, P2, D);
    if (rc) return rc;
    if (B > 0 && ((P1 > 0 && (!grad_x || !idx_x)) || (P2 > 0 && (!grad_y || !idx_y)))) {
        set_error("chamfer_bwd: null argument"); return PCL_E_ARG;
    }
    if (B == 0) return PCL_OK;
    if (!outputs_are_zero) {
        if (P1 > 0) PCL_CUDA(cudaMemsetAsync(grad_x, 0, (size_t)B * P1 * D * sizeof(float), st));
        if (P2 > 0) PCL_CUDA(cudaMemsetAsync(grad_y, 0, (size_t)B * P2 * D * sizeof(float), st));
    }
    if (P1 == 0 || P2 == 0) return PCL_OK;
    const Pts xp{x, x_bs, x_rs, x_dtype}, yp{y, y_bs, y_rs, y_dtype};
    const int maxP = P1 > P2 ? P1 : P2;
    dim3 grid((maxP + 255) / 256, B, 2);
    chamfer_bwd_kernel<<<grid, 256, 0, st>>>(xp, x_len, yp, y_len, B, P1, P2, D, idx_x, idx_y, grad_out, g_imm_x, g_imm_y, grad_x, grad_y);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_chamfer_bwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len,
                               const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *y_len, int B,
                               int P1, int P2, int D, const int32_t *idx_x, const int32_t *idx_y,
                               const float *grad_out, float *grad_x, float *grad_y, void *stream) {
    if (!grad_out) { set_error("chamfer_bwd: null argument"); return PCL_E_ARG; }
    return chamfer_bwd_impl(x, x_dtype, x_bs, x_rs, x_len, y, y_dtype, y_bs, y_rs, y_len, B, P1, P2, D, idx_x, idx_y, grad_out, 0.f, 0.f,
                            grad_x, grad_y, (cudaStream_t)stream);
}
