// pcl_emd_core.cuh -- shared device code of the auction kernels (pcl_emd.cu: cluster-per-cloud kernel, pcl_emd_team.cu: owner + worker
// kernel): shared-memory layout of one cloud's auction state, the bit-faithful bid arithmetic, the exact-safe FP32 filter, the tile
// scan, seeds and the order-independent top-2 update.  See the header comment of pcl_emd.cu and DESIGN.md "Why skipping is exact".
#pragma once
#include <cooperative_groups.h>
#include <stdlib.h>

#include "pcl_common.cuh"

#ifndef PCL_WPB_CHUNK
#define PCL_WPB_CHUNK 4
#endif
#ifndef PCL_SCAN_UNROLL
#define PCL_SCAN_UNROLL 4  // swept 1, 2, 4, 8 on config 2
#endif

namespace cg = cooperative_groups;

constexpr int kScanUnroll = PCL_SCAN_UNROLL;  // groups of 4 targets per loop trip in the tile scan

namespace pcl {
namespace {

#ifndef PCL_EMD_THREADS
#define PCL_EMD_THREADS 512
#endif
constexpr int EMD_THREADS = PCL_EMD_THREADS;
constexpr int EMD_WARPS = EMD_THREADS / 32;
#ifndef PCL_EMD_THREADS_WIDE
#define PCL_EMD_THREADS_WIDE 640
#endif
constexpr int EMD_THREADS_WIDE = PCL_EMD_THREADS_WIDE;  // the cluster kernel's second build: 20 warps at 80 registers for clusters of <= 4 CTAs
constexpr int EMD_MAX_N = 8192;      // EMD_SMEM_ONLY_N+1..8192: the cold half of the state lives in a per-CTA global-memory region (L2)
constexpr int EMD_SMEM_ONLY_N = 3584;  // up to here the whole auction state (58 B/point + 9 KB) fits into 227 KB of shared memory
constexpr int TILE = 32;  // targets per spatial tile (one bounding box per tile)
constexpr int EMD_WPB_MAX = 6 * EMD_WARPS;  // at most this many bidders per CTA: warp-per-bidder scan (swept on config 2: 48..128)
constexpr unsigned short NONE16 = 0xffffu;
constexpr unsigned NOLAST = 0xffffffffu;
constexpr float FILTER_MARGIN = 2e-6f;  // keeps T_m below T; the directed rounding below, not this size, makes skipping exact

// flags of the launch (what fits into shared memory for this N)
constexpr int EMD_F_SORT = 1;  // clouds are re-ordered along a Morton curve inside the kernel
constexpr int EMD_F_X1 = 2;    // predictions are cached in shared memory
constexpr int EMD_F_COLD = 4;  // bids / per-object maxima / assignment arrays live in global memory (large N)

struct EmdSmem {
    float4 *tgt;            // n32 {x, y, z, c = RU(3 - price)}, internal (sorted) target order, padded with far sentinels
    uint2 *pub;             // 2N  published bids {object | second<<16, increment bits}, double-buffered (sort scratch at init)
    float *pf;              // n32 price (fp32, as in the reference); padding targets keep price 0
    float *maxinc;          // N   per-object running max increment (reference: max_increments)
    int *maxidx;            // N   per-object winning bidder, ORIGINAL index (reference: max_idx), -1 = none
    unsigned *last;         // N   previous bid of every bidder (object | second<<16), NOLAST = never bid
    unsigned *last34;       // N   two more recent candidates of that bid (third | fourth<<16): extra seeds, never affect results
    unsigned short *asg;    // N8  assignment (pred -> target, internal indices), NONE16 = unassigned; padded with 0
    unsigned short *inv;    // N   assignment_inv (target -> pred), NONE16 = free
    unsigned short *unass;  // N   compacted list of unassigned bidders (internal pred indices, ascending)
    float *pbest, *pbetter; // pcap slice partials (pcap = 32 * max work items with a partial)
    unsigned *pbi, *pbi34;  // pcap
    int *wsum;              // 64: [0..31] warp sums, [48] work counter
    unsigned long long *evals;  // 1   executed evaluations of the whole cluster (accumulated in rank 0's copy)
    float4 *tlo, *thi;      // NT  tile boxes: lo = {min xyz, max c of the tile}, hi = {max xyz, -}
    unsigned short *tperm;  // N   internal target index -> original index (nullptr: identity)
    unsigned short *pperm;  // N   internal pred index -> original index (nullptr: identity)
    float4 *x1;             // N   predictions {x,y,z,0} in internal order (nullptr: read from global/L2)
};

// bytes of the "cold" arrays (touched O(U) times per iteration): pub 16, maxinc 4, maxidx 4, last 4 + 4, asg/inv/unass 6
__host__ __device__ inline size_t emd_cold_bytes(int N) {
    const size_t n8 = (size_t)(N + 7) / 8 * 8;
    return n8 * (16 + 4 + 4 + 4 + 4) + n8 * 2 * 3;
}
__host__ __device__ inline size_t emd_smem_bytes(int N, int flags, int pcap = EMD_THREADS) {
    const size_t n8 = (size_t)(N + 7) / 8 * 8, n32 = (size_t)(N + 31) / 32 * 32, nt = n32 / 32;
    return n32 * 16 + n32 * 4 + ((flags & EMD_F_COLD) ? 0 : emd_cold_bytes(N)) + (size_t)pcap * 16 + 64 * 4 + 16 + nt * 32 +
           ((flags & EMD_F_SORT) ? n8 * 4 : 0) + ((flags & EMD_F_X1) ? n8 * 16 : 0) + 64;
}

__device__ inline EmdSmem carve(unsigned char *base, unsigned char *cold, int N, int flags, int pcap) {
    const size_t n8 = (size_t)(N + 7) / 8 * 8, n32 = (size_t)(N + 31) / 32 * 32, nt = n32 / 32;
    EmdSmem s;
    unsigned char *p = base;
    s.tgt = (float4 *)p; p += n32 * 16;
    s.tlo = (float4 *)p; p += nt * 16;
    s.thi = (float4 *)p; p += nt * 16;
    s.x1 = (flags & EMD_F_X1) ? (float4 *)p : nullptr; p += (flags & EMD_F_X1) ? n8 * 16 : 0;
    s.tperm = (flags & EMD_F_SORT) ? (unsigned short *)p : nullptr; p += (flags & EMD_F_SORT) ? n8 * 2 : 0;
    s.pperm = (flags & EMD_F_SORT) ? (unsigned short *)p : nullptr; p += (flags & EMD_F_SORT) ? n8 * 2 : 0;
    s.pf = (float *)p; p += n32 * 4;    // n32: the padding targets of the last tile are priced too (0)
    s.pbest = (float *)p; p += (size_t)pcap * 4;
    s.pbetter = (float *)p; p += (size_t)pcap * 4;
    s.pbi = (unsigned *)p; p += (size_t)pcap * 4;
    s.pbi34 = (unsigned *)p; p += (size_t)pcap * 4;
    s.wsum = (int *)p; p += 64 * 4;
    s.evals = (unsigned long long *)p; p += 16;
    unsigned char *c = (flags & EMD_F_COLD) ? cold : p;  // same layout in shared memory or in the CTA's global region
    s.pub = (uint2 *)c; c += n8 * 16;
    s.asg = (unsigned short *)c; c += n8 * 2;   // 16-byte aligned for the uint4 reads of the compaction
    s.inv = (unsigned short *)c; c += n8 * 2;
    s.unass = (unsigned short *)c; c += n8 * 2;
    s.maxinc = (float *)c; c += n8 * 4;
    s.maxidx = (int *)c; c += n8 * 4;
    s.last = (unsigned *)c; c += n8 * 4;
    s.last34 = (unsigned *)c; c += n8 * 4;
    return s;
}

// float max that is correct for mixed signs (reference: CAS loop, emd_cuda.cu:10-20)
__device__ __forceinline__ void atomic_max_float(float *addr, float v) {
    if (v >= 0.f) atomicMax((int *)addr, __float_as_int(v));
    else atomicMin((unsigned *)addr, __float_as_uint(v));
}

__device__ __forceinline__ float sq3_ref(float dx, float dy, float dz) {  // the reference's contracted x*x+y*y+z*z
    return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

// exact value of a target for a bidder (emd_cuda.cu:146), given the exact squared distance
__device__ __forceinline__ float bid_value_exact(float s, float price) {
    return __double2float_rn(__dsub_rn(__dsub_rn(3.0, (double)__fsqrt_rn(s)), (double)price));
}

// 18-bit Morton key (6 bits per axis over [0,1]); only the spatial coherence of the internal order depends on it, never a
// result.  Any prefix of it is a valid cell number: ordering by (cell, key) == ordering by key
__device__ __forceinline__ unsigned spread6(unsigned v) {
    v = (v | (v << 8)) & 0x0000300Fu;
    v = (v | (v << 4)) & 0x000030C3u;
    v = (v | (v << 2)) & 0x00009249u;
    return v;
}
__device__ __forceinline__ unsigned morton18(float3 p) {
    const unsigned qx = (unsigned)min(max((int)(p.x * 64.f), 0), 63), qy = (unsigned)min(max((int)(p.y * 64.f), 0), 63),
                   qz = (unsigned)min(max((int)(p.z * 64.f), 0), 63);
    return spread6(qx) | (spread6(qy) << 1) | (spread6(qz) << 2);
}

// The skip rule of every Bid scan (DESIGN.md "Why skipping is exact"): for T a proven lower bound of the bidder's final second
// best, c >= 3 - price and s (a lower bound of) the squared distance, u = filter_u(c, filter_threshold(T)) and
// fma(u, u, -s) < 0 prove value < T.  Both subtractions round in the safe direction -- T_m down, u up -- so that the proof
// needs no bound on the magnitude of coordinates, prices or values.
__device__ __forceinline__ float filter_threshold(float T) { return __fsub_rd(T, FILTER_MARGIN); }
__device__ __forceinline__ float filter_u(float c, float tm) { return __fsub_ru(c, tm); }

struct Top2 {
    float best, better;  // emd_cuda.cu:112
    int bi, bi2;         // internal index of the bid (first argmax in ORIGINAL index order) and of the runner-up
    int bio;             // original index of bi (tie rule: lowest original index among equal maxima)
    int k3, k4;          // the two most recent "also-rans" (displaced runner-ups / survivors that missed the top two): seeds
    float tm;            // filter threshold: (lower bound of the final second best) - margin
};

// Exact update.  Order-independent restatement of emd_cuda.cu:147-154 scanned in ascending original index:
// best = max value, its index = lowest original index attaining it, better = second largest counting duplicates.
__device__ __forceinline__ void top2_exact(const EmdSmem &S, Top2 &r, float s, int k) {
    const float v = bid_value_exact(s, S.pf[k]);
    const int ko = S.tperm ? (int)S.tperm[k] : k;
    if (v > r.best || (v == r.best && ko < r.bio)) { r.k4 = r.k3; r.k3 = r.bi2; r.better = r.best; r.bi2 = r.bi; r.best = v; r.bi = k; r.bio = ko; }
    else if (v > r.better) { r.k4 = r.k3; r.k3 = r.bi2; r.better = v; r.bi2 = k; }
    else { r.k4 = r.k3; r.k3 = k; }
    r.tm = fmaxf(r.tm, filter_threshold(r.better));
}

// One tile of 32 targets for the bidder at (ax,ay,az).  e = u*u - s with u = filter_u(c_k, tm): e < 0 proves
// value_k < (final second best), so the candidate cannot change best / second best / argmax.
__device__ __forceinline__ void scan_tile(const EmdSmem &S, int k0, float ax, float ay, float az, Top2 &r) {
#define PCL_FILTER(T_, S_, E_)                                                                   \
    const float4 T_ = S.tgt[k_];                                                                 \
    const float S_ = sq3_ref(__fsub_rn(T_.x, ax), __fsub_rn(T_.y, ay), __fsub_rn(T_.z, az));     \
    const float u_##E_ = filter_u(T_.w, r.tm);                                                   \
    const float E_ = __fmaf_rn(u_##E_, u_##E_, -S_);
#pragma unroll kScanUnroll
    for (int k = k0; k < k0 + TILE; k += 4) {
        float e0, e1, e2, e3, s0, s1, s2, s3;
        { const int k_ = k;     PCL_FILTER(t, s, e) e0 = e; s0 = s; }
        { const int k_ = k + 1; PCL_FILTER(t, s, e) e1 = e; s1 = s; }
        { const int k_ = k + 2; PCL_FILTER(t, s, e) e2 = e; s2 = s; }
        { const int k_ = k + 3; PCL_FILTER(t, s, e) e3 = e; s3 = s; }
        if (!(fmaxf(fmaxf(e0, e1), fmaxf(e2, e3)) < 0.f)) {  // rare: some candidate may be in the top 2
            if (!(e0 < 0.f)) top2_exact(S, r, s0, k);
            if (!(e1 < 0.f)) top2_exact(S, r, s1, k + 1);
            if (!(e2 < 0.f)) top2_exact(S, r, s2, k + 2);
            if (!(e3 < 0.f)) top2_exact(S, r, s3, k + 3);
        }
    }
#undef PCL_FILTER
}

// Can the whole tile be skipped for this bidder?  Lower bound of s over the tile = squared distance to the
// tile's box (the same monotone fp32 operations as s, shrunk by 1e-6 relative on top), upper bound of c = tile max.
__device__ __forceinline__ bool tile_skippable(const float4 &lo, const float4 &hi, float ax, float ay, float az, float tm) {
    const float dx = fmaxf(fmaxf(__fsub_rn(lo.x, ax), __fsub_rn(ax, hi.x)), 0.f);
    const float dy = fmaxf(fmaxf(__fsub_rn(lo.y, ay), __fsub_rn(ay, hi.y)), 0.f);
    const float dz = fmaxf(fmaxf(__fsub_rn(lo.z, az), __fsub_rn(az, hi.z)), 0.f);
    const float d2 = __fmul_rn(__fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy))), 0.999999f);
    const float u = filter_u(lo.w, tm);
    return (u < 0.f) || (__fmaf_rn(u, u, -d2) < 0.f);
}

// Start of a scan: seed the threshold with the exact CURRENT values of up to four objects this bidder met at its
// previous bid (its top two and two also-rans; prices may have risen since).  The second largest of the values of
// distinct objects is a valid lower bound of the final second best.
__device__ __forceinline__ float seed_value(const EmdSmem &S, int k, float ax, float ay, float az) {
    const float4 t = S.tgt[k];
    return bid_value_exact(sq3_ref(__fsub_rn(t.x, ax), __fsub_rn(t.y, ay), __fsub_rn(t.z, az)), S.pf[k]);
}
// Seeds of a bidder that has not bid yet (the first iteration): both clouds are in Morton order, so the targets of
// similar rank are spatial neighbours.  Like all seeds they only tighten the filter threshold, never a result.
__device__ __forceinline__ void first_seeds(int jp, int N, unsigned &lastpack, unsigned &last34) {
    if (lastpack != NOLAST || N < 4) return;
    const int k1 = min(max(jp, 1), N - 3);
    lastpack = (unsigned)k1 | ((unsigned)(k1 - 1) << 16);
    last34 = (unsigned)(k1 + 1) | ((unsigned)(k1 + 2) << 16);
}

// Filter threshold from the seeds: (second largest of the exact current values of up to four distinct objects) - margin
__device__ __forceinline__ float seed_threshold(const EmdSmem &S, unsigned lastpack, unsigned last34, int N, float ax, float ay, float az) {
    float tm = -1e9f;
    const int k1 = (int)(lastpack & 0xffffu), k2 = (int)(lastpack >> 16);
    if (lastpack != NOLAST && k1 < N && k2 < N && k1 != k2) {
        float hi = seed_value(S, k1, ax, ay, az), lo = seed_value(S, k2, ax, ay, az);  // hi >= lo: the two largest so far
        if (lo > hi) { const float t = hi; hi = lo; lo = t; }
        const int k3 = (int)(last34 & 0xffffu), k4 = (int)(last34 >> 16);
        if (k3 < N && k3 != k1 && k3 != k2) {
            const float v = seed_value(S, k3, ax, ay, az);
            if (v > hi) { lo = hi; hi = v; } else if (v > lo) lo = v;
        }
        if (k4 < N && k4 != k1 && k4 != k2 && k4 != k3) {
            const float v = seed_value(S, k4, ax, ay, az);
            if (v > hi) { lo = hi; hi = v; } else if (v > lo) lo = v;
        }
        tm = filter_threshold(lo);
    }
    return tm;
}
// The same threshold for a bidder scanned by a whole warp: lanes 0..3 evaluate up to four seeds in parallel (warp-uniform result).
__device__ __forceinline__ float warp_seed_threshold(const EmdSmem &S, unsigned lastpack, unsigned last34, int N, float ax, float ay, float az) {
    const int lane = threadIdx.x & 31;
    float tm = -1e9f;
    const int k1 = (int)(lastpack & 0xffffu), k2 = (int)(lastpack >> 16);
    if (lastpack != NOLAST && k1 < N && k2 < N && k1 != k2) {
        const int k3 = (int)(last34 & 0xffffu), k4 = (int)(last34 >> 16);
        const bool ok3 = k3 < N && k3 != k1 && k3 != k2, ok4 = k4 < N && k4 != k1 && k4 != k2 && k4 != k3;
        float v = -3e38f;
        const int ks = lane == 0 ? k1 : lane == 1 ? k2 : lane == 2 ? k3 : k4;
        if (lane < 2 || (lane == 2 && ok3) || (lane == 3 && ok4)) v = seed_value(S, ks, ax, ay, az);
        // second largest of the (up to) four values
        const float v0 = __shfl_sync(0xffffffffu, v, 0), v1 = __shfl_sync(0xffffffffu, v, 1),
                    v2 = __shfl_sync(0xffffffffu, v, 2), v3 = __shfl_sync(0xffffffffu, v, 3);
        const float hi01 = fmaxf(v0, v1), lo01 = fminf(v0, v1), hi23 = fmaxf(v2, v3), lo23 = fminf(v2, v3);
        tm = filter_threshold(fmaxf(fminf(hi01, hi23), fmaxf(lo01, lo23)));
    }
    return tm;
}
__device__ __forceinline__ Top2 top2_init(float tm) {
    Top2 r;
    r.best = -1e9f; r.better = -1e9f; r.bi = -1; r.bi2 = -1; r.bio = 0x7fffffff; r.k3 = -1; r.k4 = -1; r.tm = tm;
    return r;
}

// prediction jp (internal index) of the cloud: from the shared-memory copy, else from global memory / L2
__device__ __forceinline__ float3 pred_xyz(const EmdSmem &S, const Pts &xyz1, int cloud, int jp) {
    if (S.x1) { const float4 q = S.x1[jp]; return make_float3(q.x, q.y, q.z); }
    return ld_xyz(xyz1, cloud, S.pperm ? (int)S.pperm[jp] : jp);
}

// Start of iteration t: prices moved in the previous iteration, so refresh the per-tile upper bound of c.  A stale, higher bound
// stays valid, so with at most 32 bidders left (have_list) only every fourth iteration does it.
template <int THREADS>
__device__ __forceinline__ void refresh_tile_bounds(const EmdSmem &S, int NT, int t, bool have_list) {
    constexpr int NW = THREADS / 32;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (t > 0 && (!have_list || (t & 3) == 0)) {
        for (int t0 = wid; t0 < NT; t0 += 4 * NW) {  // four independent tiles per trip
            // warp maximum with one REDUX on an order-preserving integer image of the float (c may be negative: padding)
            int b[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int tl = min(t0 + i * NW, NT - 1);
                b[i] = __float_as_int(S.tgt[tl * TILE + lane].w);
                b[i] ^= (b[i] >> 31) & 0x7fffffff;
            }
#pragma unroll
            for (int i = 0; i < 4; i++) b[i] = __reduce_max_sync(0xffffffffu, b[i]);
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int tl = t0 + i * NW;
                b[i] ^= (b[i] >> 31) & 0x7fffffff;
                if (lane == 0 && tl < NT) S.tlo[tl].w = __int_as_float(b[i]);
            }
        }
    }
}

// Set-up of one CTA's replica (emd_module.py:45-56 + the internal order): both clouds in Morton order, target tiles with their
// boxes, empty auction state.  Ends WITHOUT a barrier: the caller synchronises (cluster or block) before anyone reads the state.
template <int THREADS>
__device__ __forceinline__ void emd_setup(const EmdSmem &S, const Pts &xyz1, const Pts &xyz2, int cloud, int N, int flags) {
    const int tid = threadIdx.x, T = THREADS, lane = tid & 31, wid = tid >> 5;
    const int n8 = (N + 7) / 8 * 8, n32 = (N + 31) / 32 * 32, NT = n32 / TILE;
    if (tid == 0) *S.evals = 0ull;
    if (flags & EMD_F_SORT) {
        // Counting sort by Morton cell (histogram with shared-memory atomics, block scan, scatter, in-cell ranking).
        // Every tie rule uses original indices, so results never depend on the internal order (the parity tests run it
        // sorted, in natural order and with N > 4096); it only has to be the SAME order in all CTAs of a cluster.
        // Scratch: the cold arrays (bids, assignment, per-object maxima, seeds: 38 B/point) are not in use yet.  The more
        // cells, the cheaper the quadratic in-cell ranking for clustered clouds: cells = 8 N rounded down to a power of two,
        // 4096..16384 (a prefix of the 18-bit key, so that ordering by (cell, key) == ordering by key).
        int cbits = 12;
        while (cbits < 14 && (1 << (cbits + 1)) <= 8 * N) cbits++;
        const int ncell = 1 << cbits, cshift = 18 - cbits;
        int *hist = reinterpret_cast<int *>(S.pub);                              // ncell ints, one pad word per 32: cell c lives at H(c)
        unsigned *tmp = reinterpret_cast<unsigned *>(hist + ncell + ncell / 32); // N keys
        unsigned short *rnk = reinterpret_cast<unsigned short *>(S.pbest);       // N arrival ranks inside the cell (partials buffer: >= 8 KB)
        auto H = [](int c) -> int { return c + (c >> 5); };  // a thread scans 8..32 consecutive cells: the pad keeps the lanes on different banks
        for (int pass = 0; pass < 2; pass++) {  // 0: targets, 1: predictions
            const Pts &src = pass ? xyz1 : xyz2;
            for (int c = tid; c < ncell + ncell / 32; c += T) hist[c] = 0;
            __syncthreads();
            for (int k = tid; k < N; k += T) rnk[k] = (unsigned short)atomicAdd(&hist[H((int)(morton18(ld_xyz(src, cloud, k)) >> cshift))], 1);
            __syncthreads();
            {   // exclusive prefix sum over the cells: ncell / T consecutive cells per thread + block scan
                const int cpt = (ncell + THREADS - 1) / THREADS;  // (exact for 512 threads; other CTA sizes leave the last threads idle)
                int sum = 0;
                for (int i = 0; i < cpt; i++) sum += (tid * cpt + i < ncell) ? hist[H(tid * cpt + i)] : 0;
                int incl2 = sum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int u = __shfl_up_sync(0xffffffffu, incl2, o);
                    if (lane >= o) incl2 += u;
                }
                if (lane == 31) S.wsum[wid] = incl2;
                __syncthreads();
                int base = incl2 - sum;
                for (int w = 0; w < wid; w++) base += S.wsum[w];
                for (int i = 0; i < cpt; i++) {
                    if (tid * cpt + i < ncell) { const int v = hist[H(tid * cpt + i)]; hist[H(tid * cpt + i)] = base; base += v; }
                }
            }
            __syncthreads();
            // scatter (fine key | original index) in arrival order, then rank every point among its cell mates by that
            // unique key: the final internal order is the full Morton order, a deterministic function of the input and
            // hence identical in every CTA of the cluster (the replicas exchange internal indices)
            for (int k = tid; k < N; k += T) {
                const float3 p = ld_xyz(src, cloud, k);
                const unsigned k18 = morton18(p);
                tmp[hist[H((int)(k18 >> cshift))] + (int)rnk[k]] = (k18 << 12) | (unsigned)k;
            }
            __syncthreads();
            for (int k = tid; k < N; k += T) {
                const float3 p = ld_xyz(src, cloud, k);
                const unsigned k18 = morton18(p);
                const int cell = (int)(k18 >> cshift);
                const unsigned key = (k18 << 12) | (unsigned)k;
                const int lo = hist[H(cell)], hi = (cell + 1 < ncell) ? hist[H(cell + 1)] : N;
                int pos = lo;
                for (int q = lo; q < hi; q++) pos += (tmp[q] < key) ? 1 : 0;
                if (pass == 0) { S.tperm[pos] = (unsigned short)k; S.tgt[pos] = make_float4(p.x, p.y, p.z, 3.0f); }
                else { S.pperm[pos] = (unsigned short)k; if (S.x1) S.x1[pos] = make_float4(p.x, p.y, p.z, 0.f); }
            }
            __syncthreads();
        }
    } else {
        for (int k = tid; k < N; k += T) {
            const float3 p = ld_xyz(xyz2, cloud, k);
            S.tgt[k] = make_float4(p.x, p.y, p.z, 3.0f);
            if (S.x1) { const float3 q = ld_xyz(xyz1, cloud, k); S.x1[k] = make_float4(q.x, q.y, q.z, 0.f); }
        }
    }
    for (int k = N + tid; k < n32; k += T) S.tgt[k] = make_float4(1e18f, 1e18f, 1e18f, -1e30f);  // far away: never a bid
    // Every lane of a candidate tile evaluates its target, the padding ones of the last tile included: their price must be a
    // defined 0 (value 3 - sqrt(3e36) -- never a bid) rather than whatever the previous kernel left in shared memory.
    for (int j = n8 + tid; j < n32; j += T) S.pf[j] = 0.f;
    for (int j = tid; j < n8; j += T) {
        S.pf[j] = 0.f;
        S.asg[j] = (j < N) ? NONE16 : (unsigned short)0;
        S.inv[j] = NONE16;
        S.maxinc[j] = 0.f;
        S.maxidx[j] = -1;
        S.last[j] = NOLAST;
        S.last34[j] = NOLAST;
    }
    __syncthreads();
    for (int t = wid; t < NT; t += THREADS / 32) {  // tile boxes
        const int k = t * TILE + lane;
        const float4 p = S.tgt[k];
        const bool ok = k < N;
        float lx = ok ? p.x : 3e38f, ly = ok ? p.y : 3e38f, lz = ok ? p.z : 3e38f;
        float hx = ok ? p.x : -3e38f, hy = ok ? p.y : -3e38f, hz = ok ? p.z : -3e38f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lx = fminf(lx, __shfl_xor_sync(0xffffffffu, lx, o)); ly = fminf(ly, __shfl_xor_sync(0xffffffffu, ly, o));
            lz = fminf(lz, __shfl_xor_sync(0xffffffffu, lz, o)); hx = fmaxf(hx, __shfl_xor_sync(0xffffffffu, hx, o));
            hy = fmaxf(hy, __shfl_xor_sync(0xffffffffu, hy, o)); hz = fmaxf(hz, __shfl_xor_sync(0xffffffffu, hz, o));
        }
        if (lane == 0) { S.tlo[t] = make_float4(lx, ly, lz, 3.0f); S.thi[t] = make_float4(hx, hy, hz, 0.f); }
    }
}

}  // namespace
}  // namespace pcl
