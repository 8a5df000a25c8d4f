// pcl_emd_tasks.cuh -- the task protocol shared by the auction kernels: a cloud's Bid phase (emd_cuda.cu:95-179) cut into tasks that any
// CTA can execute from a copy of the cloud's hot state (targets with c = RU(3 - price), prices, tile boxes, original target indices).
//   publisher (the cloud's owner / lead CTA): writes bidder records + boxes + price updates into the cloud's L2 mirror, then release-stores
//             (iteration, ticket limit);
//   executor  (owner, cluster member or worker CTA): claims a ticket with a CAS while next < limit, runs the task, writes 16-byte bid
//             records by list position, fence + atomicAdd(done);
//   the publisher waits for done == limit and reads the bids back.
// See pcl_emd_team.cu (owner + worker kernel, worker kernel) and pcl_emd.cu (cluster kernel with exported lane-per-bidder iterations).
#pragma once
#include "pcl_emd_core.cuh"

namespace pcl {
namespace {

struct __align__(128) TeamCtl {  // one per cloud; zeroed by the host call before every launch
    unsigned long long avail;    // ((iteration + 1) << 32) | ticket limit, release-stored by the owner
    unsigned next;               // next ticket (claimed by CAS while next < limit)
    unsigned done;               // finished tickets
    int t, U, TB, KS, mode, base, prog, pad2;  // header of the iteration the tickets [base, limit) belong to; prog: iteration the cloud is in (lag estimate)
    unsigned long long evals;    // evaluations executed by workers for this cloud (statistics)
    unsigned pad1[18];
};
static_assert(sizeof(TeamCtl) == 128, "TeamCtl is one 128-byte line");

struct __align__(16) TeamWs {  // 16-byte aligned: as a kernel parameter, pairs of its fields are read with one 128-bit constant load
    TeamCtl *ctl;          // B control lines
    unsigned *finished;    // number of owners that are done
    unsigned char *clouds; // per-cloud mirror regions
    size_t stride, o_tgt, o_pf, o_tperm, o_box, o_brec, o_pub, o_jp;
    int nworkers;          // worker CTAs of this launch (0: nobody reads the mirror)
};

__host__ __device__ inline size_t team_cloud_bytes(int N, size_t *o_tgt, size_t *o_pf, size_t *o_tperm, size_t *o_box, size_t *o_brec,
                                                   size_t *o_pub, size_t *o_jp) {
    const size_t n8 = (size_t)(N + 7) / 8 * 8, n32 = (size_t)(N + 31) / 32 * 32, nt = n32 / 32;
    size_t o = 0;
    auto put = [&](size_t *where, size_t bytes) { if (where) *where = o; o += (bytes + 255) / 256 * 256; };
    put(o_tgt, n32 * 16); put(o_pf, n8 * 4); put(o_tperm, n8 * 2); put(o_box, nt * 32); put(o_brec, n8 * 16); put(o_pub, n8 * 16);
    put(o_jp, n8 * 2);
    return o;
}

// The task workspace: [control block: B + 1 lines, zeroed before every launch][B mirror regions]
inline size_t team_ctl_bytes(int B) { return align_up((size_t)(B + 1) * sizeof(TeamCtl), 256); }
inline TeamWs team_ws_make(void *team_ws, int B, int N, int nworkers) {
    TeamWs W;
    W.ctl = reinterpret_cast<TeamCtl *>(team_ws);
    W.finished = reinterpret_cast<unsigned *>(W.ctl + B);
    W.clouds = reinterpret_cast<unsigned char *>(team_ws) + team_ctl_bytes(B);
    W.stride = team_cloud_bytes(N, &W.o_tgt, &W.o_pf, &W.o_tperm, &W.o_box, &W.o_brec, &W.o_pub, &W.o_jp);
    W.nworkers = nworkers;
    return W;
}

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// 16-byte copies global (L2, never the possibly stale L1) -> shared
__device__ __forceinline__ void copy16_in(void *dst, const void *src, int n16) {
    for (int i = threadIdx.x; i < n16; i += (int)blockDim.x) reinterpret_cast<uint4 *>(dst)[i] = __ldcg(reinterpret_cast<const uint4 *>(src) + i);
}
__device__ __forceinline__ void copy16_out(void *dst, const void *src, int n16) {
    for (int i = threadIdx.x; i < n16; i += (int)blockDim.x) reinterpret_cast<uint4 *>(dst)[i] = reinterpret_cast<const uint4 *>(src)[i];
}

// One bidder scanned by one warp, one lane per target of a tile (the warp-per-bidder mode of pcl_emd.cu): 32 boxes per ballot, up to
// PCL_WPB_CHUNK candidate tiles per step, rare filter survivors folded into a warp-uniform top two.  Returns the bid of the bidder.
struct WarpBid { float best, better; int bi, bi2, k3, k4; };
__device__ __forceinline__ WarpBid warp_scan_bidder(const EmdSmem &S, int NT, float ax, float ay, float az, float tm, unsigned long long &my_evals) {
    const int lane = threadIdx.x & 31;
    float best = -1e9f, better = -1e9f;
    int bi = -1, bi2 = -1, bio = 0x7fffffff, k3 = -1, k4 = -1;
    for (int tb = 0; tb < NT; tb += 32) {
        const int tl = tb + lane;
        bool cand = false;
        if (tl < NT) cand = !tile_skippable(S.tlo[tl], S.thi[tl], ax, ay, az, tm);
        unsigned cm = __ballot_sync(0xffffffffu, cand);
        constexpr int WC = PCL_WPB_CHUNK;
        while (cm) {
            int tix[WC];
            bool have[WC];
#pragma unroll
            for (int i = 0; i < WC; i++) {
                have[i] = cm != 0;
                tix[i] = tb + (have[i] ? __ffs(cm) - 1 : 0);
                cm &= cm - 1;
            }
            float sq[WC], cw[WC];
            bool pass[WC];
            bool any = false;
#pragma unroll
            for (int i = 0; i < WC; i++) {
                const float4 tq = S.tgt[tix[i] * TILE + lane];
                sq[i] = sq3_ref(__fsub_rn(tq.x, ax), __fsub_rn(tq.y, ay), __fsub_rn(tq.z, az));
                cw[i] = tq.w;
                const float u = __fsub_rn(tq.w, tm);
                pass[i] = have[i] && !(__fmaf_rn(u, u, -sq[i]) < 0.f);
                any |= pass[i];
            }
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < WC; i++) my_evals += have[i] ? TILE : 0;
            }
            if (!__any_sync(0xffffffffu, any)) continue;
            do {
                int sel = -1;
#pragma unroll
                for (int i = WC - 1; i >= 0; i--) sel = pass[i] ? i : sel;
                float ssel = 0.f;
                int ksel = 0;
#pragma unroll
                for (int i = 0; i < WC; i++) {
                    if (sel == i) { ssel = sq[i]; ksel = tix[i] * TILE + lane; pass[i] = false; }
                }
                float v = 0.f;
                int ko = 0;
                if (sel >= 0) { v = bid_value_exact(ssel, S.pf[ksel]); ko = S.tperm ? (int)S.tperm[ksel] : ksel; }
                unsigned pm = __ballot_sync(0xffffffffu, sel >= 0);
                if (__popc(pm) > 3) {  // many survivors: only the two largest can change (best, better)
                    const float vc = __fadd_rn(v, 0.f);
                    int key = __float_as_int(vc);
                    key ^= (key >> 31) & 0x7fffffff;
                    if (!(sel >= 0 && vc == vc)) key = (int)0x80000000;
                    const int key1 = __reduce_max_sync(0xffffffffu, key);
                    if (key1 != (int)0x80000000) {
                        const int ko1 = __reduce_min_sync(0xffffffffu, (key == key1) ? ko : 0x7fffffff);
                        const int l1 = __ffs(__ballot_sync(0xffffffffu, key == key1 && ko == ko1)) - 1;
                        const int keyr = (lane == l1) ? (int)0x80000000 : key;
                        const int key2 = __reduce_max_sync(0xffffffffu, keyr);
                        const int l2 = (key2 != (int)0x80000000) ? __ffs(__ballot_sync(0xffffffffu, keyr == key2)) - 1 : l1;
                        const float va = __shfl_sync(0xffffffffu, v, l1), vb = __shfl_sync(0xffffffffu, v, l2);
                        const int ka = __shfl_sync(0xffffffffu, ksel, l1), kb = __shfl_sync(0xffffffffu, ksel, l2);
                        const int kob = __shfl_sync(0xffffffffu, ko, l2);
                        if (va > best || (va == best && ko1 < bio)) { k4 = k3; k3 = bi2; better = best; bi2 = bi; best = va; bi = ka; bio = ko1; }
                        else if (va > better) { k4 = k3; k3 = bi2; better = va; bi2 = ka; }
                        else { k4 = k3; k3 = ka; }
                        if (key2 != (int)0x80000000) {
                            if (vb > best || (vb == best && kob < bio)) { k4 = k3; k3 = bi2; better = best; bi2 = bi; best = vb; bi = kb; bio = kob; }
                            else if (vb > better) { k4 = k3; k3 = bi2; better = vb; bi2 = kb; }
                            else { k4 = k3; k3 = kb; }
                        }
                    }
                    pm = 0;
                }
                while (pm) {
                    const int l = __ffs(pm) - 1;
                    pm &= pm - 1;
                    const float vl = __shfl_sync(0xffffffffu, v, l);
                    const int kol = __shfl_sync(0xffffffffu, ko, l), kl = __shfl_sync(0xffffffffu, ksel, l);
                    if (vl > best || (vl == best && kol < bio)) { k4 = k3; k3 = bi2; better = best; bi2 = bi; best = vl; bi = kl; bio = kol; }
                    else if (vl > better) { k4 = k3; k3 = bi2; better = vl; bi2 = kl; }
                    else { k4 = k3; k3 = kl; }
                }
                tm = fmaxf(tm, __fsub_rn(better, FILTER_MARGIN));
                any = false;
#pragma unroll
                for (int i = 0; i < WC; i++) {
                    const float u = __fsub_rn(cw[i], tm);
                    pass[i] = pass[i] && !(__fmaf_rn(u, u, -sq[i]) < 0.f);
                    any |= pass[i];
                }
            } while (__any_sync(0xffffffffu, any));
        }
    }
    return WarpBid{best, better, bi, bi2, k3, k4};
}

struct TaskHdr { int U, TB, KS, mode; };
// How an iteration with U bidders is cut into tasks: about `tasks_target` tasks, each with ~32 work items for the 16 warps.
__device__ __forceinline__ TaskHdr task_policy(int U, bool wpb, int tasks_target, int NT, int pcap) {
    TaskHdr h;
    h.U = U;
    h.mode = wpb ? 1 : 0;
    if (wpb) {  // warp-per-bidder: tasks of 16..64 bidders (one to four rounds of the 16 warps)
        h.TB = 16 * max(1, min(4, (U + 16 * tasks_target - 1) / (16 * tasks_target)));
        h.KS = 1;
    } else {    // lane-per-bidder: tasks of 1..8 groups of 32 bidders, ~32 work items (group x tile slice) per task
        const int Gn = (U + 31) >> 5, tg = max(1, min(8, (Gn + tasks_target - 1) / tasks_target));
        h.TB = tg * 32;
        h.KS = max(1, min(min(32 / tg, NT), pcap / h.TB));
    }
    return h;
}  // bidders of the iteration, bidders per task, tile slices per group, scan mode

// One task of a cloud's Bid phase, executed by a whole CTA whose shared memory holds the cloud's targets / prices / boxes (the
// owner's replica or a worker's copy of the mirror): TB consecutive bidders of the list.  mode 0: lane-per-bidder -- groups of 32
// neighbouring bidders, every group scanned in KS tile slices (TB/32*KS work items for the 16 warps, dynamic queue, slice partials
// merged by the tree of pcl_emd.cu == emd_cuda.cu:165-173).  mode 1: warp-per-bidder -- one bidder per warp at a time.
// Bids go to pub[list position] = {object | second << 16, increment bits, third | fourth << 16, 0}.
template <int THREADS>
__device__ __forceinline__ void team_run_task(const EmdSmem &S, int NT, float eps, const TaskHdr &h, int task,
                                              const float4 *__restrict__ brec, const unsigned short *__restrict__ bjp,
                                              uint4 *__restrict__ pub, unsigned long long &my_evals) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int *const work_ctr = S.wsum + 48;
    const int b0 = task * h.TB;                            // first list position of the task
    const int nb = min(h.TB, h.U - b0);                    // bidders of the task
    if (tid == 0) *work_ctr = THREADS / 32;
    __syncthreads();
    if (h.mode == 1) {
        for (int i = wid;;) {
            if (i >= nb) break;
            const float4 rec = __ldcg(&brec[b0 + i]);
            const WarpBid w = warp_scan_bidder(S, NT, rec.x, rec.y, rec.z, rec.w, my_evals);
            if (lane == 0) {
                const float inc = __fadd_rn(__fsub_rn(w.best, w.better), eps);  // emd_cuda.cu:175
                pub[b0 + i] = make_uint4((unsigned)(w.bi & 0xffff) | ((unsigned)(w.bi2 & 0xffff) << 16), __float_as_uint(inc),
                                         (unsigned)(w.k3 & 0xffff) | ((unsigned)(w.k4 & 0xffff) << 16), 0u);
                i = atomicAdd(work_ctr, 1);
            }
            i = __shfl_sync(0xffffffffu, i, 0);
        }
        return;
    }
    const int ng = (nb + 31) >> 5, KS = h.KS, GS = ng * 32;
    for (int it = wid;;) {
        if (it >= ng * KS) break;
        const int g = it % ng, sl = it / ng;
        const int bl = min(g * 32 + lane, nb - 1);        // surplus lanes shadow the last bidder (results discarded)
        const bool active = (g * 32 + lane) < nb;
        const float4 rec = __ldcg(&brec[b0 + bl]);
        const float ax = rec.x, ay = rec.y, az = rec.z;
        Top2 r = top2_init(rec.w);
        const int ntl = (NT - sl + KS - 1) / KS;           // tiles of this slice: sl, sl+KS, ...
        const int jp0 = (int)__ldcg(&bjp[b0 + g * 32]);
        const int home = min(max((jp0 / TILE - sl + KS / 2) / KS, 0), ntl - 1);
        for (int m = 0; m < ntl; m++) {                    // zig-zag outwards from the tile next to the bidders
            int q = home + ((m & 1) ? ((m + 1) >> 1) : -(m >> 1));
            q += (q < 0) ? ntl : 0;
            q -= (q >= ntl) ? ntl : 0;
            const int tl = sl + q * KS;
            if (__all_sync(0xffffffffu, tile_skippable(S.tlo[tl], S.thi[tl], ax, ay, az, r.tm))) continue;
            scan_tile(S, tl * TILE, ax, ay, az, r);
            my_evals += active ? TILE : 0;
        }
        const unsigned pack = (unsigned)(r.bi & 0xffff) | ((unsigned)(r.bi2 & 0xffff) << 16);
        const unsigned pack34 = (unsigned)(r.k3 & 0xffff) | ((unsigned)(r.k4 & 0xffff) << 16);
        if (KS == 1) {
            if (active) pub[b0 + bl] = make_uint4(pack, __float_as_uint(__fadd_rn(__fsub_rn(r.best, r.better), eps)), pack34, 0u);
        } else if (active) {
            S.pbest[sl * GS + bl] = r.best; S.pbetter[sl * GS + bl] = r.better; S.pbi[sl * GS + bl] = pack; S.pbi34[sl * GS + bl] = pack34;
        }
        if (lane == 0) it = atomicAdd(work_ctr, 1);
        it = __shfl_sync(0xffffffffu, it, 0);
    }
    if (KS > 1) {
        __syncthreads();
        int span = 1;
        while (span < KS) span <<= 1;
        for (int st = span >> 1; st >= 1; st >>= 1) {
            const int rows = min(st, KS - st);  // slices c in [0, rows) absorb slice c + st
            for (int idx = tid; idx < rows * nb; idx += THREADS) {
                const int c = idx / nb, b = idx - c * nb;
                const int me = c * GS + b, ot = (c + st) * GS + b;
                float best = S.pbest[me], better = S.pbetter[me];
                unsigned pk = S.pbi[me], pk34 = S.pbi34[me];
                const float ob = S.pbest[ot], obt = S.pbetter[ot];
                const unsigned opk = S.pbi[ot];
                bool other_wins = ob > best;
                if (ob == best && (opk & 0xffffu) != 0xffffu) {
                    const unsigned mine = pk & 0xffffu;
                    if (mine == 0xffffu) other_wins = true;
                    else {
                        const unsigned mo = S.tperm ? S.tperm[mine] : mine, oo = S.tperm ? S.tperm[opk & 0xffffu] : (opk & 0xffffu);
                        other_wins = oo < mo;
                    }
                }
                if (other_wins) {
                    const unsigned second = (best >= obt) ? (pk & 0xffffu) : (opk >> 16);
                    better = fmaxf(best, obt);
                    best = ob;
                    pk = (opk & 0xffffu) | (second << 16);
                    pk34 = S.pbi34[ot];
                } else if (ob > better) {
                    better = ob;
                    pk = (pk & 0xffffu) | ((opk & 0xffffu) << 16);
                }
                S.pbest[me] = best; S.pbetter[me] = better; S.pbi[me] = pk; S.pbi34[me] = pk34;
            }
            __syncthreads();
        }
        for (int b = tid; b < nb; b += THREADS)
            pub[b0 + b] = make_uint4(S.pbi[b], __float_as_uint(__fadd_rn(__fsub_rn(S.pbest[b], S.pbetter[b]), eps)), S.pbi34[b], 0u);
    }
}

// spin guard: a protocol bug must end in a trap (an error the host sees), never in a hung GPU
#define PCL_SPIN_LIMIT (1u << 25)

// widx: index of this worker (home cloud = widx mod B); idle_limit: leave after this many cycles without a ticket (0: never)
template <int THREADS>
__device__ void team_worker(const EmdSmem &S, const TeamWs &W, int B, int N, float eps, int widx, long long idle_limit) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n8 = (N + 7) / 8 * 8, n32 = (N + 31) / 32 * 32, NT = n32 / TILE;
    int cached_c = -1, cached_t = -1;
    const int home = widx % B;
    long long last_work = clock64();
    unsigned long long my_evals = 0ull;
    for (;;) {
        if (wid == 0) {
            // Which task next?  First the worker's HOME cloud (workers are dealt to the clouds round-robin: one control line, no
            // contention with the workers of other clouds); else steal from the cloud that is furthest behind, ties broken by the
            // distance from home so that idle workers spread over the clouds instead of all racing for the same ticket.
            int c_sel = -1;
            unsigned ticket = 0;
            for (unsigned spin = 0;; spin++) {
                unsigned bestkey = 0xffffffffu, bestnx = 0;
                int bestc = -1;
                {
                    const unsigned long long av = ld_relaxed_u64(&W.ctl[home].avail);
                    const unsigned nx = ld_relaxed_u32(&W.ctl[home].next);
                    if (nx < (unsigned)av) { bestc = home; bestnx = nx; bestkey = 0; }
                }
                if (bestc < 0) {
                    for (int c0 = 0; c0 < B; c0 += 32) {
                        const int r = c0 + lane;                       // rotated position: cloud (home + 1 + r) mod B
                        int c = home + 1 + r;
                        c -= (c >= B) ? B : 0;
                        unsigned key = 0xffffffffu, nx = 0;
                        if (r < B - 1) {
                            const unsigned long long av = ld_relaxed_u64(&W.ctl[c].avail);
                            nx = ld_relaxed_u32(&W.ctl[c].next);
                            if (nx < (unsigned)av) key = ((unsigned)(av >> 32) << 16) | (unsigned)(r & 0xffff);
                        }
                        const unsigned k = __reduce_min_sync(0xffffffffu, key);
                        if (k < bestkey) {
                            bestkey = k;
                            const int src = __ffs(__ballot_sync(0xffffffffu, key == k)) - 1;
                            bestc = __shfl_sync(0xffffffffu, c, src);
                            bestnx = __shfl_sync(0xffffffffu, nx, src);
                        }
                    }
                }
                if (bestc >= 0) {
                    unsigned got = 0;
                    if (lane == 0) got = (atomicCAS(&W.ctl[bestc].next, bestnx, bestnx + 1) == bestnx) ? 1u : 0u;
                    got = __shfl_sync(0xffffffffu, got, 0);
                    if (got) { c_sel = bestc; ticket = bestnx; break; }
                    continue;  // lost the race: look again at once
                }
                if (ld_relaxed_u32(W.finished) >= (unsigned)B) break;  // every auction is over (or past its exported iterations)
                // Nothing to do for a long time while some cloud has not even started: this worker may be sitting on an SM that
                // cloud's CTAs are waiting for -- give it back.  (finished[1] counts the clouds whose CTAs are running.)
                if (idle_limit > 0 && clock64() - last_work > idle_limit && ld_relaxed_u32(W.finished + 1) < (unsigned)B) break;
                if (spin > PCL_SPIN_LIMIT) __trap();
                __nanosleep(100);
            }
            __threadfence();  // acquire side of the owner's release store: the ticket's iteration header, records and mirror are visible
            if (lane == 0) { S.wsum[56] = c_sel; S.wsum[57] = (int)ticket; }
        }
        __syncthreads();
        const int c = S.wsum[56];
        if (c < 0) return;
        const unsigned ticket = (unsigned)S.wsum[57];
        last_work = clock64();
        const TeamCtl *ctl = &W.ctl[c];
        TaskHdr h;
        h.U = __ldcg(&ctl->U); h.TB = __ldcg(&ctl->TB); h.KS = __ldcg(&ctl->KS); h.mode = __ldcg(&ctl->mode);
        const int t = __ldcg(&ctl->t), base = __ldcg(&ctl->base);
        const unsigned char *cl = W.clouds + (size_t)c * W.stride;
        if (c != cached_c || t != cached_t) {  // this CTA's copy of the cloud's hot state is for another cloud / iteration
            // targets + prices + boxes (+ original indices for a new cloud): every thread has all its 16-byte loads in flight at once
            const int c_tgt = n32, c_pf = n8 / 4, c_box = 2 * NT, c_tp = (c != cached_c && S.tperm) ? n8 / 8 : 0;
            const int total = c_tgt + c_pf + c_box + c_tp;
            constexpr int PER = 8;  // 16 B x 8 x 512 threads = 64 KB per round
            for (int base = 0; base < total; base += PER * THREADS) {
                uint4 v[PER];
#pragma unroll
                for (int i = 0; i < PER; i++) {
                    const int e = base + i * THREADS + tid;
                    const unsigned char *src = nullptr;
                    if (e < c_tgt) src = cl + W.o_tgt + (size_t)e * 16;
                    else if (e < c_tgt + c_pf) src = cl + W.o_pf + (size_t)(e - c_tgt) * 16;
                    else if (e < c_tgt + c_pf + c_box) src = cl + W.o_box + (size_t)(e - c_tgt - c_pf) * 16;
                    else if (e < total) src = cl + W.o_tperm + (size_t)(e - c_tgt - c_pf - c_box) * 16;
                    if (src) v[i] = __ldcg(reinterpret_cast<const uint4 *>(src));
                }
#pragma unroll
                for (int i = 0; i < PER; i++) {
                    const int e = base + i * THREADS + tid;
                    unsigned char *dst = nullptr;
                    if (e < c_tgt) dst = reinterpret_cast<unsigned char *>(S.tgt) + (size_t)e * 16;
                    else if (e < c_tgt + c_pf) dst = reinterpret_cast<unsigned char *>(S.pf) + (size_t)(e - c_tgt) * 16;
                    else if (e < c_tgt + c_pf + c_box) dst = reinterpret_cast<unsigned char *>(S.tlo) + (size_t)(e - c_tgt - c_pf) * 16;  // tlo, thi adjacent
                    else if (e < total) dst = reinterpret_cast<unsigned char *>(S.tperm) + (size_t)(e - c_tgt - c_pf - c_box) * 16;
                    if (dst) *reinterpret_cast<uint4 *>(dst) = v[i];
                }
            }
            cached_c = c; cached_t = t;
            __syncthreads();
        }
        // (team_run_task starts with a block barrier: the copies are visible to every warp before the first scan)
        team_run_task<THREADS>(S, NT, eps, h, (int)ticket - base, reinterpret_cast<const float4 *>(cl + W.o_brec),
                      reinterpret_cast<const unsigned short *>(cl + W.o_jp), reinterpret_cast<uint4 *>(const_cast<unsigned char *>(cl) + W.o_pub), my_evals);
        // statistics: evaluations executed for cloud c (before the task counts as done: the owner reads the total at the end)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my_evals += __shfl_xor_sync(0xffffffffu, my_evals, o);
        if (lane == 0 && my_evals) atomicAdd(&W.ctl[c].evals, my_evals);
        my_evals = 0ull;
        __threadfence();   // this thread's bids are visible device-wide ...
        __syncthreads();   // ... for every thread of the CTA, before the task counts as done
        if (tid == 0) { __threadfence(); atomicAdd(&W.ctl[c].done, 1u); }
    }
}

}  // namespace
}  // namespace pcl
