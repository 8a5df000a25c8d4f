// pcl_emd.cu -- auction-based approximate Earth Mover's Distance for sm_100a.
//
// Replaces the reference's 7*iters+1 launches (pointcloud_vision/loss/emd/emd_cuda.cu:256-269:
// clear, calc_unass_cnt, calc_unass_cnt_sum, calc_unass_idx, Bid, GetMax, Assign, CalcDist) with ONE
// persistent kernel.  A cloud is owned by a thread-block cluster of CS CTAs (CS in {1,2,4,8,16}: the largest size
// for which all B clusters are resident at once; 640-thread CTAs for CS <= 4, 512 otherwise).  This file holds the cluster
// kernel (and its EXPORT variant, whose heavy iterations are shared with worker CTAs) and the host entry points that pick
// between it and the owner + worker kernel of pcl_emd_team.cu (pcl_emd_set_path, DESIGN.md 3.1b).
// Every CTA keeps the whole auction state of its cloud in shared memory
// (targets, prices, assignment, inverse assignment) as a REPLICA:
//   0. set-up: both clouds are put into an internal Morton order (counting sort over up to 16384 cells + in-cell ranking),
//      targets are cut into tiles of 32 with a bounding box; every tie rule is evaluated on ORIGINAL indices, so the order never changes a result;
//   1. every CTA compacts the list of unassigned bidders from its replica (identical in all CTAs);
//   2. the bidders are dealt to the CTAs of the cluster and scanned through a dynamic work queue, either with one
//      lane per bidder (a warp = 32 neighbouring bidders x a slice of tiles, broadcast LDS.128, whole tiles skipped
//      when all 32 lanes prove them irrelevant) or, for few bidders, with one warp per bidder (32 boxes tested per
//      ballot, one lane per target); slice partials are merged by a tree equivalent to emd_cuda.cu:165-173;
//   3. finished bids (object, increment) are written into EVERY CTA's bid arrays through distributed
//      shared memory, followed by the one cluster barrier of the iteration;
//   4. every CTA resolves all bids redundantly (GetMax / Assign, emd_cuda.cu:181-215) on its replica with
//      shared-memory atomics, so prices and assignments never have to be exchanged.
//
// Bid arithmetic is bit-faithful to the reference's SASS (SURVEY.md App. A):
//   s = fma(dz,dz,fma(dx,dx,dy*dy)), r = sqrt.rn(s), v = (float)((3.0 - (double)r) - (double)price).
// Only the two largest values of a scan matter, so the expensive part (IEEE sqrt, two F2F conversions, two
// DADDs -- the XU pipe runs at 16 lanes/clk/SM on B200 and bounds the reference's Bid) is evaluated only
// for candidates that pass an exact-safe FP32 filter in the squared domain:
//   skip k  <=>  s_k > u^2,  u = RU(c_k - RD(T - margin)),  c_k = RU(3 - price_k) kept in the target tile's .w,
// where T is a proven lower bound of the bidder's final second-best value (its running second best, seeded
// with the exact current values of the two objects it preferred at its previous bid); a whole tile is skipped with
// the same inequality on bounds (distance to the tile's box, tile maximum of c).  Skipped candidates are strictly
// below the final second best, so best / second-best / argmax are exactly the reference's (derivation in DESIGN.md
// "Why skipping is exact").
// Per-iteration fixed costs are kept short because late iterations have only a handful of bidders: the tile maxima are
// refreshed with one REDUX per tile, decide + commit of the resolve phase is one pass, many filter survivors of a
// warp-per-bidder step are reduced to their top two with warp reductions, the first work item of a warp needs no atomic,
// and with at most 32 bidders left warp 0 writes the next list of unassigned bidders while it commits the bids.
// The reference's GetMax race (last writer wins inside a +-1e-6 window) is resolved as
// "largest bidder index wins" (atomicMax), identical to oracle/emd_oracle.c.
// Clouds of 3585..8192 points (EMD_SMEM_ONLY_N < N <= EMD_MAX_N) keep the hot half of the state (targets, prices) in
// shared memory and the cold half (bids, per-object maxima, assignment arrays) in a per-CTA global-memory region.
#include "pcl_emd_tasks.cuh"

namespace pcl {
namespace {

// EXPORT: the lane-per-bidder iterations run as TICKETS (pcl_emd_tasks.cuh): the bidders' records go to the cloud's L2 region, the
// CTAs of the cluster claim tasks dynamically (no static dealing, no waiting for the slowest CTA of the cluster), worker CTAs of a
// second launch (emd_worker_kernel) claim them too -- they take work from the clouds that are furthest behind, which is what
// shortens the launch: it ends with its slowest cloud -- and the bids come back as 16-byte records by list position (no scattered
// distributed-shared-memory stores).  Iterations with few bidders keep the cluster-local warp-per-bidder path.
// THREADS: 512, or 640 for clusters of at most 4 CTAs (their iterations are dominated by the lane-per-bidder scan, which gains from 20
// warps at 80 registers: -4..9 % on early-training inputs for B >= 16; bigger clusters spend their time in the latency-bound
// warp-per-bidder mode, where the 16-warp / 103-register build is 2-6 % faster -- profiles/r2_s2_auction_experiments.txt).
template <bool EXPORT, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
emd_auction_kernel(Pts xyz1, Pts xyz2, int N, float eps, int iters, int flags, int pcap, int wpb_max, int items_target,
                   float *__restrict__ dist,
                   int *__restrict__ assignment, int *__restrict__ stats,
                   unsigned char *__restrict__ cold_ws, float grad_scale, float *__restrict__ grad_xyz1,
                   double *__restrict__ part, unsigned *__restrict__ ticket, float *__restrict__ sums_out, TeamWs W, int tasks_target, int export_pct, int lag_min_q, int lag_slope) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cg::cluster_group cluster = cg::this_cluster();
    const int cs = (int)cluster.num_blocks(), rank = (int)cluster.block_rank(), csl = __ffs(cs) - 1;  // cs is a power of two
    const int cloud = blockIdx.x / cs;
    constexpr int NW = THREADS / 32;  // warps per CTA
    const int tid = threadIdx.x, T = THREADS, lane = tid & 31, wid = tid >> 5;
    const size_t cold_stride = (emd_cold_bytes(N) + 255) / 256 * 256;
    const EmdSmem S = carve(smem_raw, (flags & EMD_F_COLD) ? cold_ws + (size_t)blockIdx.x * cold_stride : nullptr, N, flags, pcap);
    int *const work_ctr = S.wsum + 48;  // dynamic work-item counter of the bid phase (wsum[0..31] = warp sums)
    const int n8 = (N + 7) / 8 * 8, n32 = (N + 31) / 32 * 32, NT = n32 / TILE;

    // ---- init: internal (Morton) order of both clouds, tiles, auction state (emd_module.py:45-56) ----------
    emd_setup<THREADS>(S, xyz1, xyz2, cloud, N, flags);
    TeamCtl *const ctl = EXPORT ? &W.ctl[cloud] : nullptr;
    unsigned char *const cl = EXPORT ? W.clouds + (size_t)cloud * W.stride : nullptr;
    if constexpr (EXPORT) {
        if (rank == 0 && W.nworkers > 0) {  // the mirror the workers load: targets (c = 3: price 0), prices, original target indices
            __syncthreads();
            copy16_out(cl + W.o_tgt, S.tgt, n32);
            copy16_out(cl + W.o_pf, S.pf, n32 / 4);
            if (S.tperm) copy16_out(cl + W.o_tperm, S.tperm, n8 / 8);
        }
    }
    if constexpr (EXPORT) {
        if (rank == 0 && tid == 0) atomicAdd(W.finished + 1, 1u);  // this cloud's CTAs are running (the workers' idle rule, pcl_emd_tasks.cuh)
    }
    unsigned tk_limit = 0;       // tickets published so far (identical in every CTA of the cluster)
    bool told_workers = false;   // this cloud has no more exported iterations: said so once (rank 0)
    cluster.sync();  // every CTA's arrays exist before anyone writes remote bids

    long long sum_u = 0;
    unsigned long long my_evals = 0ull;  // evaluations this lane really executed (tiles that were not skipped)
    int iters_run = 0, extra_qualifiers = 0, cur = 0;
    bool have_list = false;  // the list of unassigned bidders of the next iteration already exists (written during the commit)
    const int E = (n8 / 8 + T - 1) / T * 8;  // contiguous elements per thread in the compaction (multiple of 8, <= 32)

    for (int t = 0; t < iters; t++) {
        const bool last = (t == iters - 1);
        // ---- 1. list of unassigned bidders (emd_cuda.cu:23-93), ascending, identical in every CTA -------
        refresh_tile_bounds<THREADS>(S, NT, t, have_list);
        int U = 0;
        if (have_list) {
            // At most 32 bidders were left: warp 0 wrote the next list (the losers in list order, then the evicted owners)
            // while it committed the bids -- identical in every CTA, and the dealing does not need it sorted.
            U = S.wsum[40];
            if (U == 0) break;
            if (tid == 0) *work_ctr = NW;
        } else {
        unsigned fl = 0;
        {
            const int base = tid * E;
            for (int e = 0; e < E; e += 8) {
                if (base + e < n8) {
                    const uint4 a = *reinterpret_cast<const uint4 *>(S.asg + base + e);
                    const unsigned w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                    for (int h = 0; h < 4; h++) {
                        fl |= (unsigned)((w[h] & 0xffffu) == NONE16) << (e + 2 * h);
                        fl |= (unsigned)((w[h] >> 16) == NONE16) << (e + 2 * h + 1);
                    }
                }
            }
        }
        const int cnt = __popc(fl);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) S.wsum[wid] = incl;
        __syncthreads();
        int wbase = 0;
#pragma unroll
        for (int w = 0; w < NW; w++) {
            const int v = S.wsum[w];
            if (w < wid) wbase += v;
            U += v;
        }
        if (U == 0) break;  // uniform across the cluster: replicas are identical
        if (tid == 0) *work_ctr = NW;  // the first work item of warp w is item w (no atomic on the critical path), the rest is dynamic
        {
            int pos = wbase + incl - cnt;
            const int base = tid * E;
            while (fl) {
                const int e = __ffs(fl) - 1;
                fl &= fl - 1;
                S.unass[pos++] = (unsigned short)(base + e);
            }
        }
        }
        __syncthreads();
        sum_u += U;
        iters_run = t + 1;

        // ---- 2. Bid (emd_cuda.cu:95-179) for this CTA's share of the bidders ----------------------------
        // A warp owns 32 consecutive (= spatially close) bidders and one interleaved slice of the target tiles;
        // a tile is skipped when every lane proves that none of its 32 targets can reach the lane's top 2.
        // The (spatially sorted) list is dealt to the CTAs of the cluster in an interleaved way -- single bidders when
        // there are few (warp-per-bidder mode), blocks of 32 neighbours otherwise -- so that every CTA sees the
        // same mix of easy and hard regions.  list position of local bidder b:  pos(b).
        // (cluster size and dealing granularity are powers of two: shifts instead of integer divisions, which every thread
        // would otherwise execute in every iteration)
        const bool wpb = (U > 0 && ((U + cs - 1) >> csl) <= wpb_max);
        // EXPORT: in a lane-per-bidder iteration the LAST blocks of the list (a share of export_pct percent) become tickets for the
        // worker CTAs; the cluster deals the first Ud bidders among its CTAs as usual and serves the tickets the workers left over.
        int Ud = U;
        if constexpr (EXPORT) {
            // How much is exported depends on how far this cloud lags behind the others (decided by rank 0 during the previous
            // iteration, wsum[58..59] in every CTA): clouds that keep up export nothing and pay nothing, the slow ones -- the launch
            // ends with the slowest -- hand up to export_pct percent of their bidders to the workers.
            const int pct = (t > 0) ? S.wsum[58 + (t & 1)] : 0;  // two slots: rank 0 may write the next decision while a slow CTA still reads this one
            if (!wpb && W.nworkers > 0 && pct > 0) Ud = (((U + 31) >> 5) - ((((U + 31) >> 5) * pct) / 100)) << 5;  // pct <= 60: Ud >= 32
            Ud = min(Ud, U);
        }
        const bool ticketed = Ud < U;
        const int gsl = wpb ? 0 : 5, gsz = 1 << gsl;        // dealing granularity: 1 or 32 bidders
        const int nblk = (Ud + gsz - 1) >> gsl;             // blocks in the (statically dealt part of the) list
        const int myblk = (nblk > rank) ? ((nblk - rank + cs - 1) >> csl) : 0;  // blocks rank, rank+cs, ...
        int Uc = myblk << gsl;
        if (myblk > 0 && (rank + (myblk - 1) * cs) == nblk - 1) Uc -= (nblk << gsl) - Ud;  // the last block may be short
        auto pos = [&](int b) -> int { return ((((b >> gsl) << csl) + rank) << gsl) + (b & (gsz - 1)); };
        const int Gn = (Uc + 31) >> 5;                                   // bidder groups (warps' worth)
        // tile slices per group: aim at ~2 work items per warp (dynamic queue), bounded by the partial buffer
        int KS = 1;
        if (!wpb && Gn > 0 && Gn < items_target) KS = max(1, min(min((items_target + Gn - 1) / Gn, NT), pcap / (Gn * 32)));
        const int GS = Gn * 32;                                          // partial stride of one slice
        uint2 *pub_cur = S.pub + cur * n8;

        auto publish = [&](int jp, float best, float better, unsigned pack, unsigned pack34) {
            const float inc = __fadd_rn(__fsub_rn(best, better), eps);  // emd_cuda.cu:175
            const uint2 v = make_uint2(pack, __float_as_uint(inc));
            if (flags & EMD_F_COLD) {  // peers' bid buffers are global-memory regions: plain stores, ordered by the cluster barrier
                const size_t off = (size_t)(pub_cur - S.pub) + (size_t)jp;
                for (int c = 0; c < cs; c++) {
                    unsigned char *peer = cold_ws + ((size_t)cloud * cs + c) * cold_stride;
                    reinterpret_cast<uint2 *>(peer)[off] = v;
                    reinterpret_cast<unsigned *>(peer + ((unsigned char *)S.last34 - (unsigned char *)S.pub))[jp] = pack34;
                }
            } else {
                for (int c = 0; c < cs; c++) {
                    cluster.map_shared_rank(pub_cur, c)[jp] = v;
                    cluster.map_shared_rank(S.last34, c)[jp] = pack34;  // read next in the bid phase after the coming barrier
                }
            }
        };

        TaskHdr th = {};
        unsigned tk_base = 0;
        int prog_sum = 0;
        if constexpr (EXPORT) {
            if (rank == 0 && W.nworkers > 0) {  // progress of this cloud out, progress of all clouds in (consumed at the end of the bid phase)
                if (tid == 0) *reinterpret_cast<volatile int *>(&ctl->prog) = wpb ? iters : t;
                if (wid == NW - 1)
                    for (int c = lane; c < (int)gridDim.x / cs; c += 32) prog_sum += (int)ld_relaxed_u32(reinterpret_cast<const unsigned *>(&W.ctl[c].prog));
            }
            if (rank == 0 && tid == 0 && !told_workers && wpb) atomicAdd(W.finished, 1u);  // U never grows: no exported iteration will follow
            told_workers |= wpb;
            if (ticketed) {
                // The publisher of this iteration (the role rotates through the cluster) writes the exported bidders' records
                // {x, y, z, seed threshold} and the boxes, then release-stores the ticket limit; no cluster barrier is needed.
                const int Ux = U - Ud;
                th = task_policy(Ux, false, tasks_target, NT, pcap);
                tk_base = tk_limit;
                tk_limit += (unsigned)((Ux + th.TB - 1) / th.TB);
                if (rank == (t & (cs - 1))) {
                    float4 *const g_brec = reinterpret_cast<float4 *>(cl + W.o_brec);
                    unsigned short *const g_jp = reinterpret_cast<unsigned short *>(cl + W.o_jp);
                    for (int i = tid; i < Ux; i += T) {
                        const int jp = S.unass[Ud + i];
                        const float3 a = pred_xyz(S, xyz1, cloud, jp);
                        unsigned lp = S.last[jp], lp34 = S.last34[jp];
                        if (flags & EMD_F_SORT) first_seeds(jp, N, lp, lp34);
                        g_brec[i] = make_float4(a.x, a.y, a.z, seed_threshold(S, lp, lp34, N, a.x, a.y, a.z));
                        g_jp[i] = (unsigned short)jp;
                    }
                    copy16_out(cl + W.o_box, S.tlo, 2 * NT);  // boxes with this iteration's upper bounds of c
                    __threadfence();
                    __syncthreads();
                    if (tid == 0) {
                        ctl->t = t; ctl->U = th.U; ctl->TB = th.TB; ctl->KS = th.KS; ctl->mode = th.mode; ctl->base = (int)tk_base;
                        __threadfence();
                        st_release_u64(&ctl->avail, ((unsigned long long)(unsigned)(t + 1) << 32) | (unsigned long long)tk_limit);
                    }
                }
            }
        }
        if (wpb) {
            // ---- few bidders: one WARP per bidder, one lane per target of a tile: the scan of warp_scan_bidder (pcl_emd_tasks.cuh),
            // written out here because routing it through the shared function slowed this kernel (profiles/r10_emd_shared_phases_ab.txt)
            for (int b = wid;;) {
                if (b >= Uc) break;
                const int jp = S.unass[pos(b)];
                const float3 a = pred_xyz(S, xyz1, cloud, jp);
                unsigned lp = S.last[jp], lp34 = S.last34[jp];
                if (flags & EMD_F_SORT) first_seeds(jp, N, lp, lp34);
                float tm = warp_seed_threshold(S, lp, lp34, N, a.x, a.y, a.z);
                float best = -1e9f, better = -1e9f;
                int bi = -1, bi2 = -1, bio = 0x7fffffff, k3 = -1, k4 = -1;
                for (int tb = 0; tb < NT; tb += 32) {
                    const int tl = tb + lane;
                    bool cand = false;
                    if (tl < NT) cand = !tile_skippable(S.tlo[tl], S.thi[tl], a.x, a.y, a.z, tm);
                    unsigned cm = __ballot_sync(0xffffffffu, cand);
                    constexpr int WC = PCL_WPB_CHUNK;
                    while (cm) {  // up to WC candidate tiles per step: WC independent filter chains per lane, one vote
                        int tix[WC];
                        bool have[WC];
#pragma unroll
                        for (int i = 0; i < WC; i++) {
                            have[i] = cm != 0;
                            tix[i] = tb + (have[i] ? __ffs(cm) - 1 : 0);
                            cm &= cm - 1;  // cm == 0 stays 0
                        }
                        float sq[WC], cw[WC];
                        bool pass[WC];
                        bool any = false;
#pragma unroll
                        for (int i = 0; i < WC; i++) {
                            const float4 tq = S.tgt[tix[i] * TILE + lane];
                            sq[i] = sq3_ref(__fsub_rn(tq.x, a.x), __fsub_rn(tq.y, a.y), __fsub_rn(tq.z, a.z));
                            cw[i] = tq.w;
                            const float u = filter_u(tq.w, tm);
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
                            if (__popc(pm) > 3) {
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
                            tm = fmaxf(tm, filter_threshold(better));  // re-test the leftovers against the tightened threshold
                            any = false;
#pragma unroll
                            for (int i = 0; i < WC; i++) {
                                const float u = filter_u(cw[i], tm);
                                pass[i] = pass[i] && !(__fmaf_rn(u, u, -sq[i]) < 0.f);
                                any |= pass[i];
                            }
                        } while (__any_sync(0xffffffffu, any));
                    }
                }
                if (lane == 0) publish(jp, best, better, (unsigned)(bi & 0xffff) | ((unsigned)(bi2 & 0xffff) << 16),
                                       (unsigned)(k3 & 0xffff) | ((unsigned)(k4 & 0xffff) << 16));
                if (lane == 0) b = atomicAdd(work_ctr, 1);  // next bidder of this warp
                b = __shfl_sync(0xffffffffu, b, 0);
            }
        } else {
        // seed thresholds once per bidder (not once per slice item): parked in the increment field of the bidder's own
        // bid slot, which nobody else touches before this CTA publishes that bid
        for (int b = tid; b < Uc; b += T) {
            const int jp = S.unass[pos(b)];
            const float3 a = pred_xyz(S, xyz1, cloud, jp);
            unsigned lp = S.last[jp], lp34 = S.last34[jp];
            if (flags & EMD_F_SORT) first_seeds(jp, N, lp, lp34);
            pub_cur[jp].y = __float_as_uint(seed_threshold(S, lp, lp34, N, a.x, a.y, a.z));
        }
        __syncthreads();
        for (int it = wid;;) {
            if (it >= Gn * KS) break;
            const int g = it % Gn, sl = it / Gn;
            const int b = min(g * 32 + lane, Uc - 1);          // surplus lanes shadow the last bidder (results discarded)
            const bool active = (g * 32 + lane) < Uc;
            const int jp = S.unass[pos(b)];
            const float3 a = pred_xyz(S, xyz1, cloud, jp);
            Top2 r = top2_init(__uint_as_float(pub_cur[jp].y));
            const int ntl = (NT - sl + KS - 1) / KS;           // tiles of this slice: sl, sl+KS, ...
            const int home = min(max((__shfl_sync(0xffffffffu, jp, 0) / TILE - sl + KS / 2) / KS, 0), ntl - 1);
            for (int m = 0; m < ntl; m++) {                    // zig-zag outwards from the tile next to the bidders
                int q = home + ((m & 1) ? ((m + 1) >> 1) : -(m >> 1));
                q += (q < 0) ? ntl : 0;
                q -= (q >= ntl) ? ntl : 0;
                const int tl = sl + q * KS;
                if (__all_sync(0xffffffffu, tile_skippable(S.tlo[tl], S.thi[tl], a.x, a.y, a.z, r.tm))) continue;
                scan_tile(S, tl * TILE, a.x, a.y, a.z, r);
                my_evals += active ? TILE : 0;
            }
            const unsigned pack = (unsigned)(r.bi & 0xffff) | ((unsigned)(r.bi2 & 0xffff) << 16);
            const unsigned pack34 = (unsigned)(r.k3 & 0xffff) | ((unsigned)(r.k4 & 0xffff) << 16);
            if (KS == 1) {
                if (active) publish(jp, r.best, r.better, pack, pack34);
            } else if (active) {
                S.pbest[sl * GS + b] = r.best; S.pbetter[sl * GS + b] = r.better; S.pbi[sl * GS + b] = pack; S.pbi34[sl * GS + b] = pack34;
            }
            if (lane == 0) it = atomicAdd(work_ctr, 1);  // next work item of this warp
            it = __shfl_sync(0xffffffffu, it, 0);
        }
        }
        if (!wpb && KS > 1) {
            merge_slices<THREADS>(S, KS, Uc, GS);
            for (int b = tid; b < Uc; b += T) publish(S.unass[pos(b)], S.pbest[b], S.pbetter[b], S.pbi[b], S.pbi34[b]);
        }
        if constexpr (EXPORT) {
            if (!wpb && rank == 0 && wid == NW - 1 && W.nworkers > 0) {  // export share of the NEXT iteration from the mean lag (in iterations)
                const int nb = (int)gridDim.x / cs;
                const float lag = (float)__reduce_add_sync(0xffffffffu, prog_sum) / (float)nb - (float)t;
                int pct = 0;
                if (lag >= 0.25f * (float)lag_min_q) pct = min(export_pct, 20 + (int)(lag * (float)lag_slope));
                if (lane < cs) *cluster.map_shared_rank(S.wsum + 58 + ((t + 1) & 1), lane) = pct;  // read after the coming cluster barrier
            }
            if (ticketed) {
                // tickets the workers have not taken: every CTA of the cluster serves them from its own replica
                float4 *const g_brec = reinterpret_cast<float4 *>(cl + W.o_brec);
                unsigned short *const g_jp = reinterpret_cast<unsigned short *>(cl + W.o_jp);
                uint4 *const g_pub = reinterpret_cast<uint4 *>(cl + W.o_pub);
                for (;;) {
                    __syncthreads();  // the CTA is through with its own bids (partials, work counter) / with the previous ticket
                    if (tid == 0) {
                        int got = -1;
                        for (;;) {
                            const unsigned long long av = ld_acquire_u64(&ctl->avail);
                            if ((unsigned)(av >> 32) != (unsigned)(t + 1)) { __nanosleep(32); continue; }  // the publisher is not there yet
                            const unsigned nx = ld_relaxed_u32(&ctl->next);
                            if (nx >= tk_limit) break;
                            if (atomicCAS(&ctl->next, nx, nx + 1) == nx) { got = (int)(nx - tk_base); break; }
                        }
                        S.wsum[56] = got;
                    }
                    __syncthreads();
                    const int task = S.wsum[56];
                    if (task < 0) break;
                    team_run_task<THREADS>(S, NT, eps, th, task, g_brec, g_jp, g_pub, my_evals);
                    __threadfence();
                    __syncthreads();
                    if (tid == 0) { __threadfence(); atomicAdd(&ctl->done, 1u); }
                }
                if (rank == 0 && tid == 0) {  // the tickets other CTAs hold (the barrier below makes the whole cluster wait with this thread)
                    for (unsigned spin = 0; ld_acquire_u32(&ctl->done) < tk_limit; spin++) {
                        if (spin > PCL_SPIN_LIMIT) __trap();
                        __nanosleep(32);
                    }
                }
            }
        }
        cluster.sync();  // all bids of this iteration are visible in every CTA
        if constexpr (EXPORT) {
            if (ticketed) {  // all bids of the iteration are in the cloud's L2 region: bring them home, indexed by bidder
                const uint4 *const g_pub = reinterpret_cast<const uint4 *>(cl + W.o_pub);
                for (int q = tid; q < U - Ud; q += T) {
                    const uint4 rec = __ldcg(&g_pub[q]);
                    const int jp = S.unass[Ud + q];
                    pub_cur[jp] = make_uint2(rec.x, rec.y);
                    S.last34[jp] = rec.z;
                }
                __syncthreads();
            }
        }

        // ---- 3. GetMax + Assign (emd_cuda.cu:181-215), replicated in every CTA -------------------------
        for (int q = tid; q < U; q += T) {
            const int jp = S.unass[q];
            const uint2 pb = pub_cur[jp];
            S.last[jp] = pb.x;
            atomic_max_float(&S.maxinc[pb.x & 0xffffu], __uint_as_float(pb.y));  // emd_cuda.cu:176
        }
        __syncthreads();
        for (int q = tid; q < U; q += T) {
            const int jp = S.unass[q];
            const uint2 pb = pub_cur[jp];
            const int o = (int)(pb.x & 0xffffu);
            const double bi = (double)__uint_as_float(pb.y), mi = (double)S.maxinc[o];
            if (bi - 1e-6 <= mi && mi <= bi + 1e-6) {  // :188-191; the largest ORIGINAL bidder index wins
                atomicMax(&S.maxidx[o], S.pperm ? (int)S.pperm[jp] : jp);
                extra_qualifiers += (rank == 0) ? 1 : 0;  // statistics: bidders inside the window (the winners are subtracted below)
            }
        }
        __syncthreads();
        // Decide and commit in one pass: a decision reads only max_idx[o], which nobody but the winner of o writes again
        // (its reset to -1 makes every later reader of o a non-winner, which is what it is).
        unsigned keep = NONE16;  // with at most 32 bidders (one per lane of warp 0): the bidder this lane leaves unassigned
        bool loser = false;
        for (int q = tid; q < U; q += T) {
            const int jp = S.unass[q];
            const uint2 pb = pub_cur[jp];
            const int o = (int)(pb.x & 0xffffu);  // emd_cuda.cu:203-211
            const bool winner = (S.maxidx[o] == (S.pperm ? (int)S.pperm[jp] : jp));
            extra_qualifiers -= (winner && rank == 0) ? 1 : 0;
            if (!(last || winner)) { keep = (unsigned)jp; loser = true; continue; }  // emd_cuda.cu:201: a loser stays unassigned
            const unsigned prev = S.inv[o];
            if (!last && prev != NONE16) { S.asg[prev] = NONE16; keep = prev; }  // the evicted owner becomes unassigned
            S.inv[o] = (unsigned short)jp;
            S.asg[jp] = (unsigned short)o;
            const float pnew = __fadd_rn(S.pf[o], __uint_as_float(pb.y));
            S.pf[o] = pnew;
            const float cnew = __fsub_ru(3.0f, pnew);  // c = RU(3 - price): upper bound used by the filter
            S.tgt[o].w = cnew;
            if constexpr (EXPORT) {
                if (!wpb && W.nworkers > 0 && rank == ((t + 1) & (cs - 1))) {  // an exported iteration may follow (whether or not this one was): its publisher keeps the workers' mirror current (its own fence + release order these stores)
                    reinterpret_cast<float *>(cl + W.o_pf)[o] = pnew;
                    reinterpret_cast<float4 *>(cl + W.o_tgt)[o].w = cnew;
                }
            }
            if (!last) {  // (in the last iteration every bidder commits: resetting here would hide the winner from the statistics of a later thread)
                S.maxinc[o] = -1e9f;
                S.maxidx[o] = -1;
            }
        }
        have_list = (U <= 32);
        if (have_list && wid == 0) {  // losers in list order, then evicted owners in list order: ballot compaction inside warp 0
            const unsigned lose = __ballot_sync(0xffffffffu, loser);
            const unsigned evic = __ballot_sync(0xffffffffu, keep != NONE16) & ~lose;
            const unsigned below = (1u << lane) - 1u;
            const int p = ((lose >> lane) & 1u) ? __popc(lose & below) : __popc(lose) + __popc(evic & below);
            __syncwarp();  // every lane has read its entry of the old list
            if (keep != NONE16) S.unass[p] = (unsigned short)keep;
            if (lane == 0) S.wsum[40] = __popc(lose) + __popc(evic);
        }
        __syncthreads();
        cur ^= 1;
    }

    if constexpr (EXPORT) {
        if (rank == 0 && tid == 0 && !told_workers) atomicAdd(W.finished, 1u);  // the auction ended inside its exported iterations
    }
    // ---- CalcDist (emd_cuda.cu:217-226) + outputs in ORIGINAL index order; points split over the cluster ----
    // Fused loss epilogue of the unweighted EMD (utils.py:304 with weights == 1; emd_module.py:63-72 + emd_cuda.cu:284-300):
    //   grad_xyz1 = grad_scale * d(sum sqrt(dist)) / d xyz1 = 2 * (grad_scale / (2 sqrt(dist))) * (xyz1 - xyz2[assignment])
    // in the operation order of torch's sqrt backward followed by NmDistanceGradKernel, and sum sqrt(dist) in fp64.
    __syncthreads();
    double sq_sum = 0.0;
    for (int jp = rank * T + tid; jp < N; jp += cs * T) {
        const unsigned k = S.asg[jp];
        float d = 0.f;
        float3 gr = make_float3(0.f, 0.f, 0.f);
        if (k != NONE16) {
            const float3 a = pred_xyz(S, xyz1, cloud, jp);
            const float4 tp = S.tgt[k];
            const float dx = __fsub_rn(a.x, tp.x), dy = __fsub_rn(a.y, tp.y), dz = __fsub_rn(a.z, tp.z);
            d = sq3_ref(dx, dy, dz);
            if (grad_xyz1) {
                const float g2 = __fmul_rn(__fdiv_rn(grad_scale, __fmul_rn(2.f, __fsqrt_rn(d))), 2.f);  // d == 0: inf, like the reference
                gr = make_float3(__fmul_rn(g2, dx), __fmul_rn(g2, dy), __fmul_rn(g2, dz));
            }
        }
        const int jo = S.pperm ? (int)S.pperm[jp] : jp;
        const size_t o = (size_t)cloud * N + jo;
        dist[o] = d;
        assignment[o] = (k != NONE16) ? (S.tperm ? (int)S.tperm[k] : (int)k) : -1;
        if (grad_xyz1) { grad_xyz1[o * 3 + 0] = gr.x; grad_xyz1[o * 3 + 1] = gr.y; grad_xyz1[o * 3 + 2] = gr.z; }
        sq_sum += (double)__fsqrt_rn(d);
    }
    if (part) {
        // per-CTA partial in a fixed order, then the CTA that takes the last ticket adds the partials of the whole grid in
        // index order: one deterministic scalar without a second launch (the ticket is zeroed by the host call)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq_sum += __shfl_xor_sync(0xffffffffu, sq_sum, o);
        double *red = reinterpret_cast<double *>(S.pbest);  // the slice-partial buffer is free now (8-byte aligned, >= 2 KB)
        if (lane == 0) red[wid] = sq_sum;
        __syncthreads();
        if (tid == 0) {
            double b = 0.0;
            for (int w = 0; w < NW; w++) b += red[w];
            part[blockIdx.x] = b;
            __threadfence();
            S.wsum[41] = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
        }
        __syncthreads();
        if (S.wsum[41] && wid == 0) {
            __threadfence();
            double b = 0.0;
            for (int i = lane; i < (int)gridDim.x; i += 32) b += __ldcg(&part[i]);  // lane-strided, then a fixed shuffle tree
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
            if (lane == 0) {
                const float total = (float)b, count = (float)((double)(gridDim.x / cs) * (double)N);
                sums_out[0] = total; sums_out[1] = count; sums_out[2] = total / count;
            }
        }
    }
    if (stats) {  // uniform over the grid
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            extra_qualifiers += __shfl_xor_sync(0xffffffffu, extra_qualifiers, o);
            my_evals += __shfl_xor_sync(0xffffffffu, my_evals, o);
        }
        if (lane == 0) {
            atomicAdd(cluster.map_shared_rank(S.evals, 0), my_evals);
            S.wsum[wid] = extra_qualifiers;
        }
        cluster.sync();
        if (rank == 0 && tid == 0) {
            int e = 0;
            for (int w = 0; w < NW; w++) e += S.wsum[w];
            int *st = stats + (size_t)cloud * 8;
            st[0] = (int)sum_u; st[1] = iters_run; st[2] = e; st[3] = cs;
            unsigned long long ce = *S.evals;
            if constexpr (EXPORT) ce += atomicAdd(&ctl->evals, 0ull);  // evaluations the workers executed for this cloud
            st[4] = (int)(ce & 0xffffffffull); st[5] = (int)(ce >> 32);
            st[6] = flags; st[7] = NT;
        }
    }
    if constexpr (EXPORT) {
        // This cloud is done: its CTAs serve the tickets of the clouds that are still running (the launch ends with the slowest cloud,
        // and by now that cloud exports a large share of its iterations) until every cloud is past its exported iterations.
        if (W.nworkers > 0) {
            __syncthreads();
            team_worker<THREADS>(S, W, (int)gridDim.x / cs, N, eps, (int)blockIdx.x, 0);
        }
    }
}

// NmDistanceGradKernel (emd_cuda.cu:284-300) without the atomics (one writer per address) and without
// the zero-fill: grad = (2*graddist) * (xyz1 - xyz2[assignment]).
__global__ void __launch_bounds__(256)
emd_bwd_kernel(Pts xyz1, Pts xyz2, int N, const int *__restrict__ assignment, const float *__restrict__ graddist,
               float *__restrict__ grad) {
    const int b = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    const size_t o = (size_t)b * N + j;
    const int k = assignment[o];
    const float g = __fmul_rn(graddist[o], 2.f);
    const float3 a = ld_xyz(xyz1, b, j);
    float3 r = make_float3(0.f, 0.f, 0.f);
    if (k >= 0 && k < N) {
        const float3 tpt = ld_xyz(xyz2, b, k);
        r = make_float3(__fmul_rn(g, __fsub_rn(a.x, tpt.x)), __fmul_rn(g, __fsub_rn(a.y, tpt.y)),
                        __fmul_rn(g, __fsub_rn(a.z, tpt.z)));
    }
    grad[o * 3 + 0] = r.x; grad[o * 3 + 1] = r.y; grad[o * 3 + 2] = r.z;
}

// ---- loss epilogue (utils.py:257-304) ----------------------------------------------------------------
__global__ void __launch_bounds__(256)
emd_match_hist_kernel(Pts label, const int *__restrict__ assignment, int B, int N, int C,
                      unsigned long long *__restrict__ hist, int *__restrict__ matched) {
    extern __shared__ unsigned int sh[];
    for (int c = threadIdx.x; c < C; c += blockDim.x) sh[c] = 0;
    __syncthreads();
    const size_t total = (size_t)B * N;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / N);
        const int k = assignment[e];
        int lab = -1;
        if (k >= 0 && k < N) lab = (int)ld_any(label, (int64_t)b * label.bs + (int64_t)k * label.rs);  // .long(): truncation
        if (matched) matched[e] = lab;
        if (lab >= 0 && lab < C) atomicAdd(&sh[lab], 1u);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x)
        if (sh[c]) atomicAdd(&hist[c], (unsigned long long)sh[c]);
}

// sums[0] = sum w*sqrt(d), sums[1] = sum w.  Two-stage, fixed order => deterministic.
constexpr int RED_BLOCKS = 64;
__global__ void __launch_bounds__(256)
emd_wreduce_stage1(const float *__restrict__ dist, const int *__restrict__ matched, const float *__restrict__ cw,
                   size_t total, int C, double *__restrict__ part) {
    __shared__ double s0[8], s1[8];
    double a0 = 0.0, a1 = 0.0;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        float w = 1.f;
        if (cw) { const int l = matched[e]; w = (l >= 0 && l < C) ? cw[l] : 0.f; }
        a0 += (double)__fmul_rn(__fsqrt_rn(dist[e]), w);
        a1 += (double)w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o); }
    if ((threadIdx.x & 31) == 0) { s0[threadIdx.x >> 5] = a0; s1[threadIdx.x >> 5] = a1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double b0 = 0.0, b1 = 0.0;
        for (int w = 0; w < 8; w++) { b0 += s0[w]; b1 += s1[w]; }
        part[blockIdx.x * 2] = b0; part[blockIdx.x * 2 + 1] = b1;
    }
}
__global__ void emd_wreduce_stage2(const double *__restrict__ part, int nb, float *__restrict__ sums) {
    if (threadIdx.x == 0) {
        double b0 = 0.0, b1 = 0.0;
        for (int i = 0; i < nb; i++) { b0 += part[i * 2]; b1 += part[i * 2 + 1]; }
        sums[0] = (float)b0; sums[1] = (float)b1;
    }
}

__global__ void __launch_bounds__(256)
emd_weighted_bwd_kernel(Pts xyz1, Pts xyz2, int N, const int *__restrict__ assignment, const float *__restrict__ dist,
                        const int *__restrict__ matched, const float *__restrict__ cw, int C,
                        const float *__restrict__ sums, const float *__restrict__ grad_out, float *__restrict__ grad) {
    const int b = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    const size_t o = (size_t)b * N + j;
    const int k = assignment[o];
    float w = 1.f;
    if (cw) { const int l = matched[o]; w = (l >= 0 && l < C) ? cw[l] : 0.f; }
    // d/d dist of  g * sum(w*sqrt(dist)) / sum(w)   (torch: sqrt backward = grad / (2*sqrt))
    const float up = __fdiv_rn(__fmul_rn(__ldg(grad_out), w), __ldg(sums + 1));
    const float gd = __fdiv_rn(up, __fmul_rn(2.f, __fsqrt_rn(dist[o])));
    const float g = __fmul_rn(gd, 2.f);
    const float3 a = ld_xyz(xyz1, b, j);
    float3 r = make_float3(0.f, 0.f, 0.f);
    if (k >= 0 && k < N) {
        const float3 tpt = ld_xyz(xyz2, b, k);
        r = make_float3(__fmul_rn(g, __fsub_rn(a.x, tpt.x)), __fmul_rn(g, __fsub_rn(a.y, tpt.y)),
                        __fmul_rn(g, __fsub_rn(a.z, tpt.z)));
    }
    grad[o * 3 + 0] = r.x; grad[o * 3 + 1] = r.y; grad[o * 3 + 2] = r.z;
}

// cluster size wanted for B clouds on sm_count SMs: the largest power of two <= 16 with B * cs <= sm_count
int cluster_size_for(int B, int sm_count) {
    int cs = 16;
    while (cs > 1 && (long)B * cs > sm_count) cs >>= 1;
    return cs;
}
// SM count of the current device; 148 (B200) when no device can be queried (size queries on a CPU-only host)
int sm_count_or_default() {
    DeviceInfo di;
    if (device_info(&di) != PCL_OK) return 148;
    return di.sm_count;
}

// cluster size of the launch: cluster_size_for, halved until B clusters of it are resident at once with `smem` bytes per CTA
int pick_cluster(int B, int sm_count, size_t smem, cudaStream_t st) {
    // the occupancy query costs a few microseconds of host time: remembered per (device, B, shared-memory size)
    struct Memo { int dev, B; size_t smem; int cs; };
    static thread_local Memo memo[8];
    static thread_local int memo_n = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); dev = -1; }
    for (int i = 0; i < memo_n; i++)
        if (memo[i].dev == dev && memo[i].B == B && memo[i].smem == smem) return memo[i].cs;
    int cs = cluster_size_for(B, sm_count);
    // Are B clusters of this size resident at the same time with this much shared memory?  A cluster lives inside one GPC, so
    // fewer clusters than B * cs <= SM count suggests may fit (8 clusters of 16 never do on a B200); a second wave would
    // double the time of the launch, half the cluster size costs far less.
    while (cs > 1) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(B * cs); cfg.blockDim = dim3(EMD_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int ncl = 0;
        cudaError_t e = cudaOccupancyMaxActiveClusters(&ncl, emd_auction_kernel<false, EMD_THREADS>, &cfg);
        if (e == cudaSuccess && ncl >= B) break;
        (void)cudaGetLastError();
        cs >>= 1;
    }
    memo[memo_n < 8 ? memo_n++ : (memo_n = 8, 7)] = Memo{dev, B, smem, cs};
    return cs;
}

// the instantiations of the cluster kernel, by [EXPORT][THREADS == EMD_THREADS_WIDE]
using AuctionKernel = decltype(&emd_auction_kernel<false, EMD_THREADS>);
const AuctionKernel auction_kernels[2][2] = {{emd_auction_kernel<false, EMD_THREADS>, emd_auction_kernel<false, EMD_THREADS_WIDE>},
                                             {emd_auction_kernel<true, EMD_THREADS>, emd_auction_kernel<true, EMD_THREADS_WIDE>}};

}  // namespace

// pcl_emd_team.cu
size_t emd_team_workspace_bytes(int B, int N);
int emd_team_launch(const Pts &p1, const Pts &p2, int B, int N, float eps, int iters, int flags, int pcap, int wpb_max, int tasks_target,
                    int local_max, int grid, size_t smem, float *dist, int *assignment, int *stats, void *team_ws, float grad_scale,
                    float *grad_xyz1, double *part, unsigned *ticket, float *sums, cudaStream_t st);

int emd_worker_launch(void *team_ws, int B, int N, float eps, int flags, int pcap, int nworkers, size_t smem, cudaStream_t st);

static int g_emd_path = PCL_EMD_PATH_AUTO;  // pcl_emd_set_path

// library-owned stream for the worker launch of the ticket path (forked from / joined to the caller's stream with events)
struct WorkerStream {
    int dev = -1;
    cudaStream_t side = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
static int worker_stream(WorkerStream **out) {
    static thread_local WorkerStream ws;
    int dev = 0;
    PCL_CUDA(cudaGetDevice(&dev));
    if (ws.dev != dev) {
        if (ws.side) { cudaStreamDestroy(ws.side); cudaEventDestroy(ws.fork); cudaEventDestroy(ws.join); ws = WorkerStream(); }
        PCL_CUDA(cudaStreamCreateWithFlags(&ws.side, cudaStreamNonBlocking));
        PCL_CUDA(cudaEventCreateWithFlags(&ws.fork, cudaEventDisableTiming));
        PCL_CUDA(cudaEventCreateWithFlags(&ws.join, cudaEventDisableTiming));
        ws.dev = dev;
    }
    *out = &ws;
    return PCL_OK;
}
}  // namespace pcl

using namespace pcl;

extern "C" int pcl_emd_max_points(void) { return EMD_MAX_N; }

extern "C" int pcl_emd_set_path(int path) {
    if (path < PCL_EMD_PATH_AUTO || path > PCL_EMD_PATH_TICKETS) { set_error("emd_set_path: %d", path); return PCL_E_ARG; }
    g_emd_path = path;
    return PCL_OK;
}

// workspace layout: [ticket, 256 B][per-CTA partial sums of the fused epilogue, fp64][reduction partials of
// pcl_emd_weighted_reduce | cold auction state for large N][task workspace of the team / ticket paths]
static size_t emd_fused_bytes(int B) {
    const size_t ctas = (size_t)(B > 256 ? B : 256);  // grid = B * cs <= max(SM count, B)
    return 256 + align_up(ctas * sizeof(double), 256);
}

extern "C" size_t pcl_emd_workspace_bytes(int B, int N) {
    const size_t red = (size_t)RED_BLOCKS * 2 * sizeof(double);
    size_t cold = 0;
    if (N > EMD_SMEM_ONLY_N && B > 0) {  // large clouds: per-CTA global region for the cold state, sized for the largest cluster
        const int cs = cluster_size_for(B, sm_count_or_default());  // the same rule pick_cluster starts from (it can only go down)
        cold = (size_t)B * cs * ((emd_cold_bytes(N) + 255) / 256 * 256);
    }
    return emd_fused_bytes(B) + align_up(red > cold ? red : cold, 256) + emd_team_workspace_bytes(B, N);  // the team region is the tail
}

static int emd_check(const void *xyz1, int dtype1, const void *xyz2, int dtype2, int B, int N, const char *who) {
    if (B < 0 || N < 1) { set_error("%s: bad size B=%d N=%d", who, B, N); return PCL_E_SHAPE; }
    if (N > EMD_MAX_N) { set_error("%s: N=%d > %d points per cloud is not supported", who, N, EMD_MAX_N); return PCL_E_UNSUPPORTED; }
    if (!dtype_ok(dtype1) || !dtype_ok(dtype2)) { set_error("%s: bad dtype", who); return PCL_E_ARG; }
    if (B > 0 && (!xyz1 || !xyz2)) { set_error("%s: null input", who); return PCL_E_ARG; }
    return PCL_OK;
}

extern "C" int pcl_emd_fwd(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1, const void *xyz2, int dtype2,
                           int64_t bs2, int64_t rs2, int B, int N, float eps, int iters, float *dist,
                           int32_t *assignment, int32_t *stats, void *workspace, size_t workspace_bytes, void *stream) {
    return pcl_emd_fwd_fused(xyz1, dtype1, bs1, rs1, xyz2, dtype2, bs2, rs2, B, N, eps, iters, dist, assignment, stats, 0.f, nullptr,
                             nullptr, workspace, workspace_bytes, stream);
}

extern "C" int pcl_emd_fwd_fused(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1, const void *xyz2, int dtype2,
                                 int64_t bs2, int64_t rs2, int B, int N, float eps, int iters, float *dist,
                                 int32_t *assignment, int32_t *stats, float grad_scale, float *grad_xyz1, float *sums,
                                 void *workspace, size_t workspace_bytes, void *stream) {
    return pcl::emd_fwd_fused_impl(xyz1, dtype1, bs1, rs1, xyz2, dtype2, bs2, rs2, B, N, eps, iters, dist, assignment, stats, grad_scale, grad_xyz1,
                                   sums, workspace, workspace_bytes, stream, EMD_WORKERS_AUTO);
}

// worker_policy EMD_WORKERS_NONE_DEDICATED: the caller runs other kernels next to the auction (the composite step's Chamfer on the SMs the
// clusters leave free), so no dedicated worker CTAs are launched; finished clusters still help the slow clouds.
int pcl::emd_fwd_fused_impl(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1, const void *xyz2, int dtype2, int64_t bs2, int64_t rs2, int B,
                            int N, float eps, int iters, float *dist, int32_t *assignment, int32_t *stats, float grad_scale, float *grad_xyz1,
                            float *sums, void *workspace, size_t workspace_bytes, void *stream, int worker_policy) {
    int rc = emd_check(xyz1, dtype1, xyz2, dtype2, B, N, "emd_fwd");
    if (rc) return rc;
    if (iters < 0) { set_error("emd_fwd: iters=%d", iters); return PCL_E_ARG; }
    if (B > 0 && (!dist || !assignment)) { set_error("emd_fwd: null output"); return PCL_E_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0) {
        if (sums) PCL_CUDA(cudaMemsetAsync(sums, 0, 3 * sizeof(float), st));
        return PCL_OK;
    }
    if (sums && (!workspace || workspace_bytes < pcl_emd_workspace_bytes(B, N))) {
        set_error("emd_fwd: the fused sum needs a workspace of %zu bytes (pcl_emd_workspace_bytes)", pcl_emd_workspace_bytes(B, N));
        return PCL_E_WORKSPACE;
    }
    DeviceInfo di;
    if ((rc = device_info(&di))) return rc;
    int flags = 0;
    if (N > EMD_SMEM_ONLY_N) {
        flags |= EMD_F_COLD;
        if (!workspace || workspace_bytes < pcl_emd_workspace_bytes(B, N)) {
            set_error("emd_fwd: N=%d needs a workspace of %zu bytes (pcl_emd_workspace_bytes)", N, pcl_emd_workspace_bytes(B, N));
            return PCL_E_WORKSPACE;
        }
    }
    if (N >= 1024 && N <= EMD_SMEM_ONLY_N && emd_smem_bytes(N, EMD_F_SORT) <= (size_t)di.max_smem_optin) flags |= EMD_F_SORT;
    if (N <= EMD_SMEM_ONLY_N && emd_smem_bytes(N, flags | EMD_F_X1) <= (size_t)di.max_smem_optin) flags |= EMD_F_X1;
    static thread_local int attr_dev = -1;
    int dev = 0;
    PCL_CUDA(cudaGetDevice(&dev));
    if (attr_dev != dev) {
        for (const auto &by_threads : auction_kernels) {
            for (const AuctionKernel k : by_threads) {
                PCL_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, di.max_smem_optin));
                PCL_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
                // The largest shared-memory carveout (228 KB) instead of the smallest that holds the 183 KB state (196 KB): the 44 KB that
                // are left let one CTA of another kernel (Chamfer in the composite step: 17 KB, 96 registers) share the SM with an auction
                // CTA.  Late-training steps, where Chamfer on the 20 free SMs ends the step, 376 -> 357 us; early-training steps
                // 1514 -> 1529 us (the guest competes for issue slots).  Training spends most of its steps in the late regime.
                PCL_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            }
        }
        attr_dev = dev;
    }
    // cluster size first (with the 512-thread configuration), then the CTA size that goes with it
    int pcap = 2 * EMD_THREADS;  // room for 32 work items with partials; fall back to 16 when shared memory is tight
    while (pcap > EMD_THREADS && emd_smem_bytes(N, flags, pcap) > (size_t)di.max_smem_optin) pcap -= EMD_THREADS;
    size_t smem = emd_smem_bytes(N, flags, pcap);
    if (smem > (size_t)di.max_smem_optin) { set_error("emd_fwd: N=%d needs %zu B shared memory (> %d)", N, smem, di.max_smem_optin); return PCL_E_UNSUPPORTED; }
    const int cs = pick_cluster(B, di.sm_count, smem, st);
    const int pcap512 = pcap;  // the team kernel always runs 512 threads
    const size_t smem512 = smem;
    int threads = EMD_THREADS;
    unsigned *ticket = sums ? (unsigned *)workspace : nullptr;
    double *part = sums ? (double *)((unsigned char *)workspace + 256) : nullptr;
    if (sums) PCL_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned), st));
    const Pts p1{xyz1, bs1, rs1, dtype1}, p2{xyz2, bs2, rs2, dtype2};
    // Which kernel (include/pcl.h, pcl_emd_set_path):
    //   tickets: cluster kernel whose lane-per-bidder iterations run as tickets + worker CTAs on the SMs the clusters leave free;
    //   team:    one owner CTA per cloud + workers (pcl_emd_team.cu);
    //   cluster: the plain cluster kernel (the only one for large clouds, B >= SM count or without a workspace).
    int path = g_emd_path;
    const size_t team_bytes = emd_team_workspace_bytes(B, N), all_bytes = pcl_emd_workspace_bytes(B, N);
    const bool can = !(flags & EMD_F_COLD) && B < di.sm_count && team_bytes > 0 && workspace && workspace_bytes >= all_bytes;
    if ((path == PCL_EMD_PATH_TEAM || path == PCL_EMD_PATH_TICKETS) && !can) {
        set_error("emd_fwd: the team / ticket paths need N <= %d, B < %d and a workspace of pcl_emd_workspace_bytes", EMD_SMEM_ONLY_N, di.sm_count);
        return PCL_E_UNSUPPORTED;
    }
    if (path == PCL_EMD_PATH_AUTO) {
        // Measured on B200 over B = 1..128, N = 1024 / 2048 / 3584, early- and late-training inputs (profiles/r2_s2_path_sweep*.txt), judged
        // on the sum of both regimes: big clouds are throughput-bound -> owner + workers; many clouds in small clusters (B >= 38: clusters
        // of 2 or 1) -> clusters + workers on the free SMs + finished clusters helping the slow ones (-10..20 %); otherwise (and for the
        // B = 32 launch of the benchmark) the plain cluster kernel, whose distributed-shared-memory exchange has the lowest latency per
        // iteration.
        path = PCL_EMD_PATH_CLUSTER;
        if (can && N >= 3072 && B >= 8) path = PCL_EMD_PATH_TEAM;
        else if (can && N >= 1536 && cs <= 2) path = PCL_EMD_PATH_TICKETS;  // (clusters of 4 with many free SMs gain 1-3 % on the mix: not worth the second launch)
    }
    // CTA size: 640 threads where the lane-per-bidder scan dominates (plain clusters of <= 4 CTAs, ticket path with clusters of <= 2)
    if (!(flags & EMD_F_COLD) && ((path == PCL_EMD_PATH_CLUSTER && cs <= 4) || (path == PCL_EMD_PATH_TICKETS && cs <= 2))) {
        const int pc = 2 * EMD_THREADS_WIDE;
        if (emd_smem_bytes(N, flags, pc) <= (size_t)di.max_smem_optin) { threads = EMD_THREADS_WIDE; pcap = pc; smem = emd_smem_bytes(N, flags, pcap); }
    }
    const int warps = threads / 32;
    const int wpb_max = 6 * warps;  // at most this many bidders per CTA: warp-per-bidder scan (swept on config 2: 48..128 at 16 warps)
    const int items_target = 2 * warps;  // work items per CTA and iteration in the lane-per-bidder mode (dynamic queue; swept 8..128 on config 2)
    void *team_ws = can ? (unsigned char *)workspace + (all_bytes - team_bytes) : nullptr;
    if (path == PCL_EMD_PATH_TEAM) {
        const int grid = max(di.sm_count, B);
        const int tasks_target = (3 * grid / B + 1) / 2;  // ~1.5 tasks per CTA that can work on a cloud
        const int local_max = 32;                         // the owner works alone with at most this many bidders
        const int team_wpb = 4 * EMD_WPB_MAX;             // warp-per-bidder tasks with at most this many bidders
        return emd_team_launch(p1, p2, B, N, eps, iters, flags, pcap512, team_wpb, tasks_target, local_max, grid, smem512, dist, (int *)assignment,
                               (int *)stats, team_ws, grad_scale, grad_xyz1, part, ticket, sums, st);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(B * cs); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    unsigned char *cold_ws = (flags & EMD_F_COLD) ? (unsigned char *)workspace + emd_fused_bytes(B) : nullptr;  // behind the fused-epilogue header
    const bool exported = path == PCL_EMD_PATH_TICKETS;
    TeamWs W = {};  // zero for the plain cluster kernel, like the four ticket-path parameters below
    int tasks_target = 0, export_pct = 0, lag_min_q = 0, lag_slope = 0, nworkers = 0;
    WorkerStream *ws = nullptr;
    if (exported) {
        // dedicated worker CTAs (a second launch) on the SMs the clusters leave free; besides them, the CTAs of every cluster whose
        // auction is over serve tickets until the last cloud is done (W.nworkers > 0 switches the export machinery on)
        nworkers = di.sm_count - B * cs;
        if (nworkers < 0 || worker_policy == EMD_WORKERS_NONE_DEDICATED) nworkers = 0;
        tasks_target = max(4, (2 * (nworkers > 0 ? nworkers : di.sm_count - B * cs) + B - 1) / B);  // exported tickets per cloud and iteration: ~2 per worker that serves the cloud, at least 4 (swept 2..8 at B=32)
        export_pct = 50;  // upper limit of the exported share (percent; the kernel needs <= 60)
        lag_min_q = 4;    // a cloud exports when it lags >= this many quarter iterations behind the mean
        lag_slope = 5;    // exported percent = 20 + slope * lag
        W = team_ws_make(team_ws, B, N, nworkers > 0 ? nworkers : 1);
        PCL_CUDA(cudaMemsetAsync(team_ws, 0, team_ctl_bytes(B), st));
        if (nworkers > 0) {
            int rc2 = worker_stream(&ws);
            if (rc2) return rc2;
            PCL_CUDA(cudaEventRecord(ws->fork, st));  // the workers need the zeroed control block, nothing else
        }
    }
    PCL_CUDA(cudaLaunchKernelEx(&cfg, auction_kernels[exported][threads == EMD_THREADS_WIDE], p1, p2, N, eps, iters, flags, pcap, wpb_max,
                                items_target, dist, (int *)assignment, (int *)stats, cold_ws, grad_scale, grad_xyz1, part, ticket, sums, W,
                                tasks_target, export_pct, lag_min_q, lag_slope));
    if (nworkers > 0) {
        // Launched AFTER the clusters (they must not find their SMs taken) on a stream of their own; a worker leaves when every
        // cloud is past its exported iterations, or after ~100 us without a ticket (so it can never starve a cluster of its SM).
        PCL_CUDA(cudaStreamWaitEvent(ws->side, ws->fork, 0));
        int rc2 = emd_worker_launch(team_ws, B, N, eps, flags, pcap, nworkers, smem, ws->side);
        if (rc2) return rc2;
        PCL_CUDA(cudaEventRecord(ws->join, ws->side));
        PCL_CUDA(cudaStreamWaitEvent(st, ws->join, 0));  // the caller's next operation on `stream` comes after the workers
    }
    return PCL_OK;
}

extern "C" int pcl_emd_bwd(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1, const void *xyz2, int dtype2,
                           int64_t bs2, int64_t rs2, int B, int N, const int32_t *assignment, const float *graddist,
                           float *grad_xyz1, void *stream) {
    if (B < 0 || N < 1) { set_error("emd_bwd: bad size B=%d N=%d", B, N); return PCL_E_SHAPE; }
    if (!dtype_ok(dtype1) || !dtype_ok(dtype2)) { set_error("emd_bwd: bad dtype"); return PCL_E_ARG; }
    if (B == 0) return PCL_OK;
    if (!xyz1 || !xyz2 || !assignment || !graddist || !grad_xyz1) { set_error("emd_bwd: null argument"); return PCL_E_ARG; }
    if (B > 65535) { set_error("emd_bwd: B=%d > 65535", B); return PCL_E_SHAPE; }
    const Pts p1{xyz1, bs1, rs1, dtype1}, p2{xyz2, bs2, rs2, dtype2};
    emd_bwd_kernel<<<dim3((N + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(p1, p2, N, assignment, graddist, grad_xyz1);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_emd_match_hist(const void *target_label, int dtype, int64_t bs, int64_t rs, const int32_t *assignment,
                                  int B, int N, int C, int64_t *hist, int32_t *matched_label, void *stream) {
    if (B < 0 || N < 1 || C < 1 || C > 4096) { set_error("emd_match_hist: bad size B=%d N=%d C=%d", B, N, C); return PCL_E_SHAPE; }
    if (!dtype_ok(dtype) || !hist) { set_error("emd_match_hist: bad argument"); return PCL_E_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    PCL_CUDA(cudaMemsetAsync(hist, 0, (size_t)C * sizeof(int64_t), st));
    if (B == 0) return PCL_OK;
    if (!target_label || !assignment) { set_error("emd_match_hist: null argument"); return PCL_E_ARG; }
    const Pts lab{target_label, bs, rs, dtype};
    const size_t total = (size_t)B * N;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 296) blocks = 296;
    emd_match_hist_kernel<<<blocks, 256, C * sizeof(unsigned), st>>>(lab, assignment, B, N, C, (unsigned long long *)hist, matched_label);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_emd_weighted_reduce(const float *dist, const int32_t *matched_label, const float *class_weights, int B,
                                       int N, int C, float *sums, void *workspace, size_t workspace_bytes, void *stream) {
    if (B < 0 || N < 1) { set_error("emd_weighted_reduce: bad size B=%d N=%d", B, N); return PCL_E_SHAPE; }
    if (!sums || (B > 0 && !dist) || (class_weights && !matched_label)) { set_error("emd_weighted_reduce: null argument"); return PCL_E_ARG; }
    if (!workspace || workspace_bytes < pcl_emd_workspace_bytes(B, N)) { set_error("emd_weighted_reduce: workspace too small"); return PCL_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    double *part = (double *)((unsigned char *)workspace + emd_fused_bytes(B));
    emd_wreduce_stage1<<<RED_BLOCKS, 256, 0, st>>>(dist, matched_label, class_weights, (size_t)B * N, C, part);
    PCL_CUDA(cudaGetLastError());
    emd_wreduce_stage2<<<1, 32, 0, st>>>(part, RED_BLOCKS, sums);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

extern "C" int pcl_emd_weighted_bwd(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1, const void *xyz2, int dtype2,
                                    int64_t bs2, int64_t rs2, int B, int N, const int32_t *assignment, const float *dist,
                                    const int32_t *matched_label, const float *class_weights, int C, const float *sums,
                                    const float *grad_out, float *grad_xyz1, void *stream) {
    if (B < 0 || N < 1) { set_error("emd_weighted_bwd: bad size B=%d N=%d", B, N); return PCL_E_SHAPE; }
    if (!dtype_ok(dtype1) || !dtype_ok(dtype2)) { set_error("emd_weighted_bwd: bad dtype"); return PCL_E_ARG; }
    if (B == 0) return PCL_OK;
    if (!xyz1 || !xyz2 || !assignment || !dist || !sums || !grad_out || !grad_xyz1 || (class_weights && !matched_label)) {
        set_error("emd_weighted_bwd: null argument"); return PCL_E_ARG;
    }
    if (B > 65535) { set_error("emd_weighted_bwd: B=%d > 65535", B); return PCL_E_SHAPE; }
    const Pts p1{xyz1, bs1, rs1, dtype1}, p2{xyz2, bs2, rs2, dtype2};
    emd_weighted_bwd_kernel<<<dim3((N + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(
        p1, p2, N, assignment, dist, matched_label, class_weights, C, sums, grad_out, grad_xyz1);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}
