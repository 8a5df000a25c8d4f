// pcl_emd_team.cu -- auction EMD as ONE persistent launch of owner and worker CTAs (sm_100a).
//
// Same algorithm, arithmetic and tie rules as pcl_emd.cu (reference: pointcloud_vision/loss/emd/emd_cuda.cu:23-282), different
// distribution of the work.  The cluster kernel gives every cloud a fixed cluster of CTAs for the whole auction: the launch ends
// with its slowest cloud (Table-shaped clouds: 3.6 M cycles against a mean of 2.7 M), 20 of the 148 SMs stay empty at B=32 and a
// small batch cannot use more than 16 SMs per cloud.  Here the grid is one CTA per SM:
//   * CTA c < B is the OWNER of cloud c.  It keeps the complete auction state in shared memory exactly like a cluster of one:
//     set-up sort, list of unassigned bidders, seed thresholds, GetMax / Assign (emd_cuda.cu:181-215), CalcDist and the fused epilogue.
//   * The Bid phase (emd_cuda.cu:95-179) of an iteration is cut into TASKS -- a block of bidders x all target tiles -- that ANY CTA
//     can execute: the owner itself, or one of the gridDim.x - B WORKER CTAs, which pull tasks of whichever cloud is furthest behind.
//     What a task needs is small and lives in an L2-resident mirror the owner keeps up to date: targets with c = RU(3 - price),
//     prices, tile boxes (46 KB at N=2048, loaded into the worker's shared memory per (cloud, iteration)) and one 16-byte record per
//     bidder {x, y, z, seed threshold}.  Bids come back as 16-byte records indexed by list position.
//   * Synchronisation is per cloud and one-directional: the owner publishes an iteration with a release store of
//     (iteration, ticket limit); tickets are claimed with a CAS; a finished task is a fence + atomicAdd on `done`; the owner serves
//     its own tickets while it waits, so it never depends on a CTA that is not running (no co-residency assumption, no deadlock
//     with fewer SMs than CTAs).  With at most `local_max` (32) bidders left the owner finishes the auction alone.
// Results are independent of who executes a task and in which order (order-independent top-2 update, tie rules on original
// indices): bit-exact against oracle/emd_oracle.c like the cluster kernel.
#include "pcl_emd_tasks.cuh"

namespace pcl {
namespace {


__global__ void __launch_bounds__(EMD_THREADS, 1)
emd_team_kernel(Pts xyz1, Pts xyz2, int B, int N, float eps, int iters, int flags, int pcap, int wpb_max, int tasks_target, int local_max,
                float *__restrict__ dist, int *__restrict__ assignment, int *__restrict__ stats, TeamWs W, float grad_scale,
                float *__restrict__ grad_xyz1, double *__restrict__ part, unsigned *__restrict__ ticket, float *__restrict__ sums_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, T = EMD_THREADS, lane = tid & 31, wid = tid >> 5;
    // each branch carves its own view of shared memory: one carve before the branch keeps values live into the worker loop, which
    // runs at the 128-register limit and would spill them
    if ((int)blockIdx.x >= B) { team_worker<EMD_THREADS>(carve(smem_raw, nullptr, N, flags, pcap), W, B, N, eps, (int)blockIdx.x - B, 0); return; }
    const EmdSmem S = carve(smem_raw, nullptr, N, flags, pcap);

    const int cloud = blockIdx.x;
    int *const work_ctr = S.wsum + 48;
    const int n8 = (N + 7) / 8 * 8, n32 = (N + 31) / 32 * 32, NT = n32 / TILE;
    TeamCtl *const ctl = &W.ctl[cloud];
    unsigned char *const cl = W.clouds + (size_t)cloud * W.stride;
    float4 *const g_tgt = reinterpret_cast<float4 *>(cl + W.o_tgt);
    float *const g_pf = reinterpret_cast<float *>(cl + W.o_pf);
    float4 *const g_brec = reinterpret_cast<float4 *>(cl + W.o_brec);
    unsigned short *const g_jp = reinterpret_cast<unsigned short *>(cl + W.o_jp);
    uint4 *const g_pub = reinterpret_cast<uint4 *>(cl + W.o_pub);

    emd_setup<EMD_THREADS>(S, xyz1, xyz2, cloud, N, flags);
    __syncthreads();
    // the mirror of the hot state: targets (c = 3: price 0), prices, original target indices, tile boxes
    copy16_out(g_tgt, S.tgt, n32);
    copy16_out(g_pf, S.pf, n8 / 4);
    if (S.tperm) copy16_out(cl + W.o_tperm, S.tperm, n8 / 8);

    auto pred_xyz = [&](int jp) -> float3 {
        if (S.x1) { const float4 q = S.x1[jp]; return make_float3(q.x, q.y, q.z); }
        return ld_xyz(xyz1, cloud, S.pperm ? (int)S.pperm[jp] : jp);
    };
    long long sum_u = 0;
    unsigned long long my_evals = 0ull;
    int iters_run = 0, extra_qualifiers = 0;
    unsigned limit = 0;      // tickets handed out so far (== finished tickets between iterations)
    bool have_list = false;
    const int E = (n8 / 8 + T - 1) / T * 8;
    uint2 *const pub_cur = S.pub;  // bids of the current iteration by bidder (no double buffering: nobody else writes it)

    for (int t = 0; t < iters; t++) {
        const bool last = (t == iters - 1);
        // ---- 1. list of unassigned bidders (emd_cuda.cu:23-93) and the per-tile upper bound of c ----------------
        if (t > 0 && (!have_list || (t & 3) == 0)) {
            for (int t0 = wid; t0 < NT; t0 += 4 * EMD_WARPS) {
                int b[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int tl = min(t0 + i * EMD_WARPS, NT - 1);
                    b[i] = __float_as_int(S.tgt[tl * TILE + lane].w);
                    b[i] ^= (b[i] >> 31) & 0x7fffffff;
                }
#pragma unroll
                for (int i = 0; i < 4; i++) b[i] = __reduce_max_sync(0xffffffffu, b[i]);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int tl = t0 + i * EMD_WARPS;
                    b[i] ^= (b[i] >> 31) & 0x7fffffff;
                    if (lane == 0 && tl < NT) S.tlo[tl].w = __int_as_float(b[i]);
                }
            }
        }
        int U = 0;
        if (have_list) {
            U = S.wsum[40];
            if (U == 0) break;
            if (tid == 0) *work_ctr = EMD_WARPS;
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
            for (int w = 0; w < EMD_WARPS; w++) {
                const int v = S.wsum[w];
                if (w < wid) wbase += v;
                U += v;
            }
            if (U == 0) break;
            if (tid == 0) *work_ctr = EMD_WARPS;
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

        // ---- 2. Bid (emd_cuda.cu:95-179) ------------------------------------------------------------------------
        const bool team = U > local_max;
        if (!team) {
            // few bidders: the owner scans them itself, one warp per bidder (a trip through L2 and a worker would cost more)
            for (int b = wid;;) {
                if (b >= U) break;
                const int jp = S.unass[b];
                const float3 a = pred_xyz(jp);
                unsigned lp = S.last[jp], lp34 = S.last34[jp];
                if (flags & EMD_F_SORT) first_seeds(jp, N, lp, lp34);
                float tm = -1e9f;
                {
                    const int k1 = (int)(lp & 0xffffu), k2 = (int)(lp >> 16);
                    if (lp != NOLAST && k1 < N && k2 < N && k1 != k2) {  // seeds: lanes 0..3 evaluate up to four of them in parallel
                        const int k3 = (int)(lp34 & 0xffffu), k4 = (int)(lp34 >> 16);
                        const bool ok3 = k3 < N && k3 != k1 && k3 != k2, ok4 = k4 < N && k4 != k1 && k4 != k2 && k4 != k3;
                        float v = -3e38f;
                        const int ks = lane == 0 ? k1 : lane == 1 ? k2 : lane == 2 ? k3 : k4;
                        if (lane < 2 || (lane == 2 && ok3) || (lane == 3 && ok4)) v = seed_value(S, ks, a.x, a.y, a.z);
                        const float v0 = __shfl_sync(0xffffffffu, v, 0), v1 = __shfl_sync(0xffffffffu, v, 1),
                                    v2 = __shfl_sync(0xffffffffu, v, 2), v3 = __shfl_sync(0xffffffffu, v, 3);
                        const float hi01 = fmaxf(v0, v1), lo01 = fminf(v0, v1), hi23 = fmaxf(v2, v3), lo23 = fminf(v2, v3);
                        tm = __fsub_rn(fmaxf(fminf(hi01, hi23), fmaxf(lo01, lo23)), FILTER_MARGIN);
                    }
                }
                const WarpBid w = warp_scan_bidder(S, NT, a.x, a.y, a.z, tm, my_evals);
                if (lane == 0) {
                    pub_cur[jp] = make_uint2((unsigned)(w.bi & 0xffff) | ((unsigned)(w.bi2 & 0xffff) << 16),
                                             __float_as_uint(__fadd_rn(__fsub_rn(w.best, w.better), eps)));
                    S.last34[jp] = (unsigned)(w.k3 & 0xffff) | ((unsigned)(w.k4 & 0xffff) << 16);
                    b = atomicAdd(work_ctr, 1);
                }
                b = __shfl_sync(0xffffffffu, b, 0);
            }
            __syncthreads();
        } else {
            // bidder records {x, y, z, seed threshold} by list position + the internal index (scan start hint) ...
            for (int b = tid; b < U; b += T) {
                const int jp = S.unass[b];
                const float3 a = pred_xyz(jp);
                unsigned lp = S.last[jp], lp34 = S.last34[jp];
                if (flags & EMD_F_SORT) first_seeds(jp, N, lp, lp34);
                g_brec[b] = make_float4(a.x, a.y, a.z, seed_threshold(S, lp, lp34, N, a.x, a.y, a.z));
                g_jp[b] = (unsigned short)jp;
            }
            // ... and the tile boxes with this iteration's upper bounds of c
            copy16_out(cl + W.o_box, S.tlo, 2 * NT);
            const TaskHdr h = task_policy(U, U <= wpb_max, tasks_target, NT, pcap);
            const int ntasks = (U + h.TB - 1) / h.TB;
            __threadfence();  // mirror updates of the previous commit, records and boxes: visible before the iteration is published
            __syncthreads();
            if (tid == 0) {
                ctl->t = t; ctl->U = h.U; ctl->TB = h.TB; ctl->KS = h.KS; ctl->mode = h.mode; ctl->base = (int)limit;
                __threadfence();
                st_release_u64(&ctl->avail, ((unsigned long long)(unsigned)(t + 1) << 32) | (unsigned long long)(limit + (unsigned)ntasks));
            }
            const unsigned base = limit;
            limit += (unsigned)ntasks;
            // serve own tickets while any is left, then wait for the tasks the workers took
            for (;;) {
                if (tid == 0) {
                    int got = -1;
                    for (;;) {
                        const unsigned nx = ld_relaxed_u32(&ctl->next);
                        if (nx >= limit) break;
                        if (atomicCAS(&ctl->next, nx, nx + 1) == nx) { got = (int)(nx - base); break; }
                    }
                    S.wsum[56] = got;
                }
                __syncthreads();
                const int task = S.wsum[56];
                if (task < 0) break;
                team_run_task<EMD_THREADS>(S, NT, eps, h, task, g_brec, g_jp, g_pub, my_evals);
                __threadfence();
                __syncthreads();
                if (tid == 0) { __threadfence(); atomicAdd(&ctl->done, 1u); }
            }
            if (tid == 0) {
                for (unsigned spin = 0; ld_acquire_u32(&ctl->done) < limit; spin++) {
                    if (spin > PCL_SPIN_LIMIT) __trap();
                    __nanosleep(100);
                }
            }
            __syncthreads();
            // all bids of the iteration are in the mirror: bring them home, indexed by bidder as GetMax / Assign expect them
            for (int q = tid; q < U; q += T) {
                const uint4 rec = __ldcg(&g_pub[q]);
                const int jp = S.unass[q];
                pub_cur[jp] = make_uint2(rec.x, rec.y);
                S.last34[jp] = rec.z;
            }
            __syncthreads();
        }

        // ---- 3. GetMax + Assign (emd_cuda.cu:181-215) -------------------------------------------------------------
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
                extra_qualifiers += 1;
            }
        }
        __syncthreads();
        unsigned keep = NONE16;
        bool loser = false;
        for (int q = tid; q < U; q += T) {
            const int jp = S.unass[q];
            const uint2 pb = pub_cur[jp];
            const int o = (int)(pb.x & 0xffffu);  // emd_cuda.cu:203-211
            const bool winner = (S.maxidx[o] == (S.pperm ? (int)S.pperm[jp] : jp));
            extra_qualifiers -= winner ? 1 : 0;
            if (!(last || winner)) { keep = (unsigned)jp; loser = true; continue; }
            const unsigned prev = S.inv[o];
            if (!last && prev != NONE16) { S.asg[prev] = NONE16; keep = prev; }
            S.inv[o] = (unsigned short)jp;
            S.asg[jp] = (unsigned short)o;
            const float pnew = __fadd_rn(S.pf[o], __uint_as_float(pb.y));
            const float cnew = __fsub_ru(3.0f, pnew);  // c = RU(3 - price): upper bound used by the filter
            S.pf[o] = pnew;
            S.tgt[o].w = cnew;
            if (team) { g_pf[o] = pnew; g_tgt[o].w = cnew; }  // U never grows: once the owner works alone the mirror is not read again
            if (!last) {  // (in the last iteration every bidder commits: resetting here would hide the winner from the statistics of a later thread)
                S.maxinc[o] = -1e9f;
                S.maxidx[o] = -1;
            }
        }
        have_list = (U <= 32);
        if (have_list && wid == 0) {
            const unsigned lose = __ballot_sync(0xffffffffu, loser);
            const unsigned evic = __ballot_sync(0xffffffffu, keep != NONE16) & ~lose;
            const unsigned below = (1u << lane) - 1u;
            const int p = ((lose >> lane) & 1u) ? __popc(lose & below) : __popc(lose) + __popc(evic & below);
            __syncwarp();
            if (keep != NONE16) S.unass[p] = (unsigned short)keep;
            if (lane == 0) S.wsum[40] = __popc(lose) + __popc(evic);
        }
        __syncthreads();
    }

    // ---- CalcDist (emd_cuda.cu:217-226) + outputs in ORIGINAL index order + fused loss epilogue (see pcl_emd.cu) ----
    __syncthreads();
    double sq_sum = 0.0;
    for (int jp = tid; jp < N; jp += T) {
        const unsigned k = S.asg[jp];
        float d = 0.f;
        float3 gr = make_float3(0.f, 0.f, 0.f);
        if (k != NONE16) {
            const float3 a = pred_xyz(jp);
            const float4 tp = S.tgt[k];
            const float dx = __fsub_rn(a.x, tp.x), dy = __fsub_rn(a.y, tp.y), dz = __fsub_rn(a.z, tp.z);
            d = sq3_ref(dx, dy, dz);
            if (grad_xyz1) {
                const float g2 = __fmul_rn(__fdiv_rn(grad_scale, __fmul_rn(2.f, __fsqrt_rn(d))), 2.f);
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
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq_sum += __shfl_xor_sync(0xffffffffu, sq_sum, o);
        double *red = reinterpret_cast<double *>(S.pbest);
        if (lane == 0) red[wid] = sq_sum;
        __syncthreads();
        if (tid == 0) {
            double b = 0.0;
            for (int w = 0; w < EMD_WARPS; w++) b += red[w];
            part[cloud] = b;
            __threadfence();
            S.wsum[41] = (atomicAdd(ticket, 1u) == (unsigned)B - 1u) ? 1 : 0;
        }
        __syncthreads();
        if (S.wsum[41] && wid == 0) {
            __threadfence();
            double b = 0.0;
            for (int i = lane; i < B; i += 32) b += __ldcg(&part[i]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
            if (lane == 0) {
                const float total = (float)b, count = (float)((double)B * (double)N);
                sums_out[0] = total; sums_out[1] = count; sums_out[2] = total / count;
            }
        }
    }
    if (stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            extra_qualifiers += __shfl_xor_sync(0xffffffffu, extra_qualifiers, o);
            my_evals += __shfl_xor_sync(0xffffffffu, my_evals, o);
        }
        __syncthreads();
        if (lane == 0) { S.wsum[wid] = extra_qualifiers; if (my_evals) atomicAdd(&ctl->evals, my_evals); }
        __syncthreads();
        if (tid == 0) {
            int e = 0;
            for (int w = 0; w < EMD_WARPS; w++) e += S.wsum[w];
            __threadfence();
            int *st = stats + (size_t)cloud * 8;
            st[0] = (int)sum_u; st[1] = iters_run; st[2] = e; st[3] = 0;  // cluster size 0 = team kernel
            const unsigned long long ce = atomicAdd(&ctl->evals, 0ull);
            st[4] = (int)(ce & 0xffffffffull); st[5] = (int)(ce >> 32);
            st[6] = flags; st[7] = NT;
        }
    }
    __syncthreads();
    if (tid == 0) { __threadfence(); atomicAdd(W.finished, 1u); }  // the workers leave when every owner is here
}

// Worker CTAs for the cluster kernel's exported iterations (pcl_emd.cu, EXPORT): launched next to it on a second stream.
__global__ void __launch_bounds__(EMD_THREADS, 1)
emd_worker_kernel(TeamWs W, int B, int N, float eps, int flags, int pcap, long long idle_limit) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const EmdSmem S = carve(smem_raw, nullptr, N, flags, pcap);
    team_worker<EMD_THREADS>(S, W, B, N, eps, (int)blockIdx.x, idle_limit);
}

}  // namespace

int emd_worker_launch(void *team_ws, int B, int N, float eps, int flags, int pcap, int nworkers, size_t smem, cudaStream_t st) {
    static thread_local int attr_dev = -1;
    int dev = 0;
    PCL_CUDA(cudaGetDevice(&dev));
    if (attr_dev != dev) {
        DeviceInfo di;
        int rc = device_info(&di);
        if (rc) return rc;
        PCL_CUDA(cudaFuncSetAttribute(emd_worker_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, di.max_smem_optin));
        attr_dev = dev;
    }
    emd_worker_kernel<<<nworkers, EMD_THREADS, smem, st>>>(team_ws_make(team_ws, B, N, nworkers), B, N, eps, flags, pcap,
                                                           200000LL);  // a worker leaves after ~100 us without a ticket
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

size_t emd_team_workspace_bytes(int B, int N) {
    if (B <= 0 || N > EMD_SMEM_ONLY_N) return 0;
    return team_ctl_bytes(B) + (size_t)B * team_cloud_bytes(N, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
}

// Launches the team kernel on `st`.  team_ws: emd_team_workspace_bytes(B, N) bytes.  Everything else as emd_auction_kernel.
int emd_team_launch(const Pts &p1, const Pts &p2, int B, int N, float eps, int iters, int flags, int pcap, int wpb_max, int tasks_target,
                    int local_max, int grid, size_t smem, float *dist, int *assignment, int *stats, void *team_ws, float grad_scale,
                    float *grad_xyz1, double *part, unsigned *ticket, float *sums, cudaStream_t st) {
    const TeamWs W = team_ws_make(team_ws, B, N, grid - B);
    const size_t ctl_bytes = team_ctl_bytes(B);
    PCL_CUDA(cudaMemsetAsync(team_ws, 0, ctl_bytes, st));
    static thread_local int attr_dev = -1;
    int dev = 0;
    PCL_CUDA(cudaGetDevice(&dev));
    if (attr_dev != dev) {
        DeviceInfo di;
        int rc = device_info(&di);
        if (rc) return rc;
        PCL_CUDA(cudaFuncSetAttribute(emd_team_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, di.max_smem_optin));
        attr_dev = dev;
    }
    emd_team_kernel<<<grid, EMD_THREADS, smem, st>>>(p1, p2, B, N, eps, iters, flags, pcap, wpb_max, tasks_target, local_max, dist, assignment,
                                                      stats, W, grad_scale, grad_xyz1, part, ticket, sums);
    PCL_CUDA(cudaGetLastError());
    return PCL_OK;
}

}  // namespace pcl
