#!/usr/bin/env python
"""bench.py -- Chamfer + EMD forward+backward throughput (BASELINE.json metric) on N B200s.

One "step" = one pass of the loss hot path over one batch of B=32 synthetic Table-shaped cloud pairs
(N=M=2048): Chamfer fwd + bwd and auction EMD (eps=0.005, 50 iterations, cfg.py:36-37) fwd + bwd with the
reference's sqrt-mean reduction (utils.py:304, weights == 1), through pointcloud_b200.ShardedChamferEmdStep: one C-ABI
call (three kernels) per rank and, at N > 1, the one all-reduce of the batch sums INSIDE the timed region.

  value : whole-job clouds/s, WEAK scaling (32 clouds per rank), inputs resident in HBM, CUDA events, max over ranks
  strong_scaling : the same step with B=32 GLOBAL (32/N clouds per rank)
  e2e   : the same metric through the C-ABI host-buffer entry point (pcl_chamfer_emd_step_host): pinned HOST inputs
          copied in, loss scalars copied back and the stream synchronised inside the timed region, every step
          (e2e.python_api: the same through the Python loss functions; sharded_api: the loss CLASSES through ShardedLoss)
  parity_checked : the timed step's outputs against the CPU oracle (outside the timed regions)
  roofline / roofline_bwd / cpu_baseline / reference_gpu : see DESIGN.md "Measurement"

`--impl reference` times the reference's CPU path (the oracle port: the reference EMD has no CPU
implementation and pytorch3d is absent) on the host cores, on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step returned to its caller (see dump_outputs) as DIR/<name>.npy; the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, NPTS, EPS, ITERS = 32, 2048, 0.005, 50
METRIC = "chamfer+emd fwd+bwd clouds/sec (B=32,N=2048)"
UNIT = "clouds/s"
WORKLOAD = ("config2: Chamfer+EMD fwd+bwd, B=32 per GPU, N=M=2048, Table-shaped synthetic clouds, "
            "regimes independent/noisy alternating, eps=0.005, iters=50")
FLOP_PER_EMD_EVAL = 11   # SURVEY.md 8d: 8 (distance) + sqrt + 2 adds
FLOP_PER_CHAMFER_EVAL = 8
NCU_AUCTION_DRAM_BYTES = 1670656  # ncu --set full, one launch (profiles/r1_s2_emd_auction_full.txt)
KERNELS_PER_STEP = 3  # emd_auction_kernel (fused epilogue) | chamfer_nn3_kernel, chamfer_bwd_kernel (side stream); + 4 small memsets


def peaks():
    p = {}
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    return p


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except Exception:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:  # region shorter than one sample period: take the samples nearest to it
            near = sorted(self.lines, key=lambda tl: min(abs(tl[0] - t0), abs(tl[0] - t1)))[:3]
            for ts, line in near:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except Exception:
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ inputs
def make_pool(torch, synth, device, rank, n_sets):
    """n_sets (pred, target) pairs whose total size exceeds the 126 MB L2: 8 seeded base batches (4 'independent'
    = early training, 4 'noisy' = late training) replicated with random point permutations."""
    bases = []
    for s in range(4):
        for regime in ("independent", "noisy"):
            p, t = synth.table_clouds(B_PER_GPU, NPTS, seed=1000 * rank + s, regime=regime)
            bases.append((p.to(device), t[:, :, :3].contiguous().to(device), regime))
    g = torch.Generator(device="cpu").manual_seed(rank)
    pool = []
    for i in range(n_sets):
        p, t, regime = bases[i % len(bases)]
        if i >= len(bases):
            pp = torch.randperm(NPTS, generator=g).to(device)
            tp = torch.randperm(NPTS, generator=g).to(device)
            p, t = p[:, pp].contiguous(), t[:, tp].contiguous()
        pool.append((p, t, regime))
    return pool


class DeviceKernels:
    """The separate C-ABI entry points with preallocated outputs, for the per-phase breakdown and the kernel rooflines."""

    def __init__(self, torch, _lib, device, b=B_PER_GPU, n=NPTS):
        self.torch, self.lib, self.L, self.b, self.n = torch, _lib, _lib.lib(), b, n
        f32, i32 = torch.float32, torch.int32
        e = lambda *s, dt=f32: torch.empty(*s, device=device, dtype=dt)
        self.dist_x, self.dist_y, self.idx_x, self.idx_y = e(b, n), e(b, n), e(b, n, dt=i32), e(b, n, dt=i32)
        self.loss_xy, self.ones = e(4), torch.ones(2, device=device)
        self.gx, self.gy = e(b, n, 3), e(b, n, 3)
        self.dist, self.asg, self.stats = e(b, n), e(b, n, dt=i32), e(b, 8, dt=i32)
        self.sums, self.gemd, self.graddist = e(4), e(b, n, 3), torch.full((b, n), 1.0 / (b * n), device=device)
        self.cws = self.L.pcl_chamfer_workspace_bytes(b, n, n); self.cw = torch.empty(self.cws, device=device, dtype=torch.uint8)
        self.ews = self.L.pcl_emd_workspace_bytes(b, n); self.ew = torch.empty(self.ews, device=device, dtype=torch.uint8)

    def chamfer_fwd(self, p, t, st):
        A, b, n = self.lib.pts_args, self.b, self.n
        return self.L.pcl_chamfer_fwd(*A(p), None, *A(t), None, b, n, n, 3, 0, self.dist_x.data_ptr(), self.idx_x.data_ptr(),
                                      self.dist_y.data_ptr(), self.idx_y.data_ptr(), self.loss_xy.data_ptr(), self.cw.data_ptr(), self.cws, st)

    def chamfer_bwd(self, p, t, st):
        A, b, n = self.lib.pts_args, self.b, self.n
        return self.L.pcl_chamfer_bwd(*A(p), None, *A(t), None, b, n, n, 3, self.idx_x.data_ptr(), self.idx_y.data_ptr(),
                                      self.ones.data_ptr(), self.gx.data_ptr(), self.gy.data_ptr(), st)

    def emd_fused(self, p, t, st, stats=True):
        """auction + CalcDist + sqrt-mean + gradient of the mean: the whole EMD side of the step, one kernel"""
        A, b, n = self.lib.pts_args, self.b, self.n
        return self.L.pcl_emd_fwd_fused(*A(p), *A(t), b, n, EPS, ITERS, self.dist.data_ptr(), self.asg.data_ptr(),
                                        self.stats.data_ptr() if stats else None, 1.0 / (b * n), self.gemd.data_ptr(), self.sums.data_ptr(),
                                        self.ew.data_ptr(), self.ews, st)

    def emd_bwd(self, p, t, st):
        """the module-level backward (emdFunction.backward): gather/scatter kernel alone"""
        A, b, n = self.lib.pts_args, self.b, self.n
        return self.L.pcl_emd_bwd(*A(p), *A(t), b, n, self.asg.data_ptr(), self.graddist.data_ptr(), self.gemd.data_ptr(), st)


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_step(oracle, np, x1, x2, threads):
    """The same step on the host cores with the oracle port (Chamfer fwd+bwd, EMD fwd, sqrt-mean, EMD bwd)."""
    c = oracle.chamfer_forward(x1, x2, nthreads=threads)
    oracle.chamfer_backward(x1, x2, c["idx_x"], c["idx_y"], 1.0)
    r = oracle.emd_forward(x1, x2, EPS, ITERS, nthreads=threads)
    d = r["dist"]
    gd = (1.0 / d.size) / (2.0 * np.sqrt(d))
    oracle.emd_backward(x1, x2, r["assignment"], gd.astype(np.float32))
    return r


def cpu_baseline(sample_clouds, steps, warmup):
    import numpy as np
    import oracle
    from pointcloud_b200 import synth
    threads = os.cpu_count() or 1
    half = max(1, sample_clouds // 2)
    pa, ta = synth.table_clouds(half, NPTS, seed=0, regime="independent")
    pb, tb = synth.table_clouds(sample_clouds - half, NPTS, seed=0, regime="noisy") if sample_clouds > half else (pa[:0], ta[:0])
    x1 = np.ascontiguousarray(np.concatenate([pa.numpy(), pb.numpy()]))
    x2 = np.ascontiguousarray(np.concatenate([ta[:, :, :3].numpy(), tb[:, :, :3].numpy()]))
    order = np.argsort(np.concatenate([np.arange(half) * 2, np.arange(sample_clouds - half) * 2 + 1]), kind="stable")
    x1, x2 = np.ascontiguousarray(x1[order]), np.ascontiguousarray(x2[order])  # interleave heavy/light clouds over the threads
    for _ in range(warmup):
        cpu_step(oracle, np, x1, x2, threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_step(oracle, np, x1, x2, threads)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return {"value": sample_clouds / dt, "unit": UNIT, "cores": min(threads, sample_clouds), "kind": "port",
            "sample": f"{sample_clouds} clouds (half independent, half noisy) of the same workload per step, {steps} steps, "
                      f"oracle C port (oracle/*.c), {threads} host threads available, batch-parallel",
            "ms_per_step": dt * 1e3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = 16
    steps, warm = args.steps, max(1, min(args.warmup, 2))
    cb = cpu_baseline(sample, steps, warm)
    line = {"metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference", "config": {"workload": WORKLOAD, "sample_clouds_per_step": sample},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "reference EMD has no CPU implementation (CUDA only) and pytorch3d is absent: this arm is the CPU oracle port of "
                    "both; the unmodified reference CUDA extension is timed on the GPU in the default arm (key reference_gpu)"}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ parity / reference
def parity_check(torch, np, pcl, pool, device):
    """Outside every timed region: the composite step of the first early-training and the first late-training batch of the
    pool against the CPU oracle (bit-exact assignment and distances, loss scalars and gradients within 1e-5 relative)."""
    import oracle
    step = pcl.ShardedChamferEmdStep(B_PER_GPU, NPTS, device, EPS, ITERS, process_group=None)
    step.world = 1
    kern_dist = torch.empty(B_PER_GPU, NPTS, device=device)
    out = {}
    for p, t, regime in pool[:2]:
        step.step(p, t)
        torch.cuda.synchronize()
        got = step.out.cpu().double().numpy()
        x1, x2 = p.cpu(), t.cpu()
        o = oracle.emd_forward(x1, x2, EPS, ITERS, nthreads=os.cpu_count() or 1)
        d, a, _ = pcl.emd_forward_raw(p, t, EPS, ITERS)
        exact = bool(np.array_equal(a.cpu().numpy(), o["assignment"]) and np.array_equal(d.cpu().numpy(), o["dist"]))
        sq = np.sqrt(o["dist"].astype(np.float64))
        emd_ok = abs(got[6] - sq.mean()) <= 1e-5 * sq.mean() and abs(got[4] - sq.sum()) <= 1e-5 * sq.sum() and got[5] == B_PER_GPU * NPTS
        gd = ((1.0 / o["dist"].size) / (2.0 * np.sqrt(o["dist"]))).astype(np.float32)
        g1, _ = oracle.emd_backward(x1, x2, o["assignment"], gd)
        ge = step.grad_emd.cpu().numpy()
        grad_emd_ok = bool(np.allclose(ge, g1, rtol=1e-5, atol=1e-12))
        c = oracle.chamfer_forward(x1, x2, nthreads=os.cpu_count() or 1)
        ch_ok = abs(got[0] + got[1] - float(c["loss"])) <= 1e-5 * float(c["loss"])
        gx, _ = oracle.chamfer_backward(x1, x2, c["idx_x"], c["idx_y"], 1.0)
        gc = step.grad_chamfer.cpu().numpy()
        grad_ch_ok = bool(np.allclose(gc, gx, rtol=1e-5, atol=1e-6 * float(np.abs(gx).max())))
        out[regime] = {"emd_assignment_and_dist_bit_exact": exact, "emd_loss": bool(emd_ok), "emd_grad": grad_emd_ok,
                       "chamfer_loss": bool(ch_ok), "chamfer_grad": grad_ch_ok, "race_free_clouds": int((o["race_events"] == 0).sum())}
    ok = all(v for r in out.values() for k, v in r.items() if k != "race_free_clouds")
    return ok, out


def reference_gpu_step(torch, pool, ev, emd_ms_ours):
    """The UNMODIFIED reference CUDA extension (oracle/_ref/emd.so) driven exactly like the reference's emd_module.py drives it --
    emdFunction.forward (12 zero-filled scratch tensors + emd.forward, emd_module.py:33-61), `dists.sqrt().mean()` (utils.py:304
    with weights == 1) and its backward through emdFunction.backward (2 more zero fills + emd.backward, :63-72) -- on the same
    B200, over the same pool, both regimes, >= 20 steps each.  Context for the speed-up, outside our timed regions."""
    from oracle import build_ref
    ref = build_ref.load_ref()
    if ref is None:
        return {"unavailable": "oracle/_ref/emd.so was not built (needs /root/reference at build time)"}
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import RefEmdFunction
    out = {"what": "unmodified reference emd extension (oracle/_ref/emd.so) under a restatement of emdFunction (tests/helpers.py): forward "
                   "(12 torch.zeros + 351 launches) + dists.sqrt().mean() + backward, same B200, same pool"}
    for regime in ("independent", "noisy"):
        sets = [(p, t) for p, t, r in pool if r == regime][:24]
        ts = []
        for i, (p, t) in enumerate(sets):
            x = p.detach().clone().requires_grad_()
            a, b_ = ev(), ev()
            a.record()
            dist, _ = RefEmdFunction.apply(ref, x, t, EPS, ITERS)
            dist.sqrt().mean().backward()
            b_.record()
            torch.cuda.synchronize()
            if i >= 4:
                ts.append(a.elapsed_time(b_))
        out[f"emd_step_ms_{regime}"] = statistics.mean(ts)
        out[f"steps_{regime}"] = len(ts)
    out["emd_step_ms"] = 0.5 * (out["emd_step_ms_independent"] + out["emd_step_ms_noisy"])
    out["ours_emd_step_ms"] = emd_ms_ours
    out["emd_step_speedup"] = out["emd_step_ms"] / emd_ms_ours
    return out


def dump_outputs(out_dir, step):
    """What the caller of the timed step holds after its last call (rank 0's shard), as float32 arrays:
    losses       the first 7 entries of the `losses` vector of pcl_chamfer_emd_step (include/pcl.h; [2:6] all-reduced over the ranks),
    grad_chamfer (B,N,3) d Chamfer loss / d pred,
    grad_emd     (B,N,3) d EMD loss / d pred."""
    import numpy as np
    step.wait()
    arrays = {"losses": step.out[:7], "grad_chamfer": step.grad_chamfer, "grad_emd": step.grad_emd}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy().astype(np.float32))


# ------------------------------------------------------------------------------------------------ main arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300, help="timed steps of the measured step (`value`)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile", action="store_true", help="value leg only (short command for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU step; the reference arm has none")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)  # before the run: an unusable DIR fails in a second, not after it

    import numpy as np
    import torch
    import torch.distributed as dist

    import pointcloud_b200 as pcl
    from pointcloud_b200 import _lib, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator is created; stdout must carry only the JSON line,
        # so file descriptor 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def timed(fn, k, w):
        """w untimed + k timed calls of fn(i), barrier + synchronise on both sides, CUDA events, max over ranks -> total ms"""
        for i in range(w):
            fn(i)
        barrier()
        e0, e1 = ev(), ev()
        e0.record()
        for i in range(k):
            fn(w + i)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    K, W = args.steps, args.warmup
    sampler = ClockSampler(local)
    sampler.start()  # started early: nvidia-smi needs a few hundred ms before its first sample
    n_sets = 96  # 96 * 1.57 MB of inputs = 151 MB > 126 MB L2: every step reads inputs that are not L2-resident
    pool = make_pool(torch, synth, device, rank, n_sets)
    st = torch.cuda.current_stream().cuda_stream
    ev = lambda: torch.cuda.Event(enable_timing=True)

    # ---- value (weak scaling, 32 clouds per GPU): the sharded config-2 step of the product package.  Per step and rank: ONE C-ABI
    #      call (three kernels: auction with fused epilogue | Chamfer forward, Chamfer backward on the side stream) + at N > 1 ONE
    #      NCCL all-reduce of the four batch sums, INSIDE the timed region --------------------------------------------------------
    step = pcl.ShardedChamferEmdStep(B_PER_GPU, NPTS, device, EPS, ITERS)
    t_wall0 = time.time()
    # the last timed step sees pool[(W + K - 1) % n_sets]: tests/test_bench_gpu.py recomputes it to check --dump-outputs
    ms_total = timed(lambda i: step.step(*pool[i % n_sets][:2]), K, W)
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step)
    ms_per_step = ms_total / K
    value = world * B_PER_GPU * K / (ms_total * 1e-3)
    if args.profile:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "ms_per_step": ms_per_step, "profile_only": True}))
        if world > 1:
            dist.destroy_process_group()
        return

    # the collective alone, and the sharded step against one GPU on the gathered batch (outside the timed regions)
    coll_ms, sharded_equals_single = None, None
    if world > 1:
        tiny = torch.zeros(4, device=device)
        coll_ms = timed(lambda i: dist.all_reduce(tiny), 200, 20) / 200
        p, t, _ = pool[0]
        step.step(p, t)
        got = step.losses()
        gp = [torch.empty_like(p) for _ in range(world)]
        gt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(gp, p.contiguous()); dist.all_gather(gt, t.contiguous())
        if rank == 0:
            single = pcl.ShardedChamferEmdStep(world * B_PER_GPU, NPTS, device, EPS, ITERS)
            single.world = 1
            single.step(torch.cat(gp), torch.cat(gt))
            want = single.losses()
            sharded_equals_single = {k: abs(got[k] - want[k]) <= 1e-5 * abs(want[k]) for k in want}
            lo = rank * B_PER_GPU
            sharded_equals_single["grad_emd"] = bool(torch.allclose(step.grad_emd, single.grad_emd[lo:lo + B_PER_GPU] * world, rtol=1e-5, atol=1e-12))
            sharded_equals_single["grad_chamfer"] = bool(torch.allclose(step.grad_chamfer, single.grad_chamfer[lo:lo + B_PER_GPU] * world, rtol=1e-5, atol=1e-9))
            assert all(sharded_equals_single.values()), sharded_equals_single
            del single
        barrier()

    # ---- strong scaling (BASELINE.json: "(B=32,N=2048) at 1/2/4/8 B200" read as B=32 GLOBAL): 32 / N clouds per rank ------------
    strong = None
    if B_PER_GPU % world == 0:
        bl = B_PER_GPU // world
        sstep = pcl.ShardedChamferEmdStep(bl, NPTS, device, EPS, ITERS)
        lo = rank * bl
        if world == 1:
            spool = [(p, t) for p, t, _ in pool]
        else:  # every rank holds its slice of the SAME global batches: rank 0's pool
            spool = []
            for p, t, _ in pool[:32]:
                pp, tt = p.clone(), t.clone()
                dist.broadcast(pp, 0); dist.broadcast(tt, 0)
                spool.append((pp[lo:lo + bl].contiguous(), tt[lo:lo + bl].contiguous()))
        Ks = min(K, 200)
        s_ms = timed(lambda i: sstep.step(*spool[i % len(spool)]), Ks, W)
        strong = {"global_batch": B_PER_GPU, "clouds_per_gpu": bl, "steps": Ks, "ms_per_step": s_ms / Ks, "value": B_PER_GPU * Ks / (s_ms * 1e-3),
                  "unit": UNIT, "scaling": "strong",
                  "note": "same sharded step, B=32 split over the ranks; the auction takes B_r*cs SMs with cs <= 16 (cluster limit): "
                          f"{bl} clouds per GPU use at most {min(148, bl * 16)} of 148 SMs"}
        del sstep, spool

    # ---- per-kernel breakdown on rank 0's stream (explains `value`; the phases run one after the other here, whereas the
    #      timed step overlaps Chamfer with the auction) ----
    kern = DeviceKernels(torch, _lib, device)
    phases = {"chamfer_fwd": [], "chamfer_bwd": [], "emd_fused_fwd_bwd": [], "emd_bwd_kernel_alone": []}
    per_regime = {"independent": [], "noisy": []}
    sum_u, executed = [], []
    for i in range(min(K, 32)):
        p, t, regime = pool[(W + i) % n_sets]
        # the short kernels (5-80 us) are timed as the average of REP back-to-back launches on rotating inputs: an event pair around a
        # single launch would add the event / launch gap (~10 us) to every one of them
        REP = 8
        batch = [pool[(W + i * REP + j) % n_sets][:2] for j in range(REP)]
        m = [ev() for _ in range(6)]
        rc = 0
        m[0].record()
        for pj, tj in batch:
            rc |= kern.chamfer_fwd(pj, tj, st)
        m[1].record()
        for pj, tj in batch:
            rc |= kern.chamfer_bwd(pj, tj, st)
        m[2].record()
        rc |= kern.emd_fused(p, t, st); m[3].record()
        for pj, tj in batch:
            rc |= kern.emd_bwd(pj, tj, st)
        m[4].record()
        torch.cuda.synchronize()
        if rc:
            raise RuntimeError(_lib.lib().pcl_last_error().decode())
        for name, a, b_, div in zip(phases, m[:-1], m[1:], (REP, REP, 1, REP)):
            phases[name].append(a.elapsed_time(b_) / div)
        e_a, e_b = ev(), ev()
        e_a.record(); step.step(p, t); e_b.record()
        torch.cuda.synchronize()
        per_regime[regime].append(e_a.elapsed_time(e_b))
        sum_u.append(int(kern.stats[:, 0].sum().item()))
        executed.append(int(((kern.stats[:, 4].long() & 0xffffffff) + (kern.stats[:, 5].long() << 32)).sum().item()))
    emd_ms = statistics.mean(phases["emd_fused_fwd_bwd"])
    evals = statistics.mean(sum_u) * NPTS  # pair evaluations one auction launch stands for (sum_t U_t * N over the batch)
    sm_count = ctypes.c_int(0)
    _lib.lib().pcl_device_info(ctypes.byref(sm_count), None, None, None)
    pk = peaks()
    sm_max = pk.get("sm_max_mhz") or clocks.get("sm_max_mhz") or 1965.0
    hbm_peak = pk.get("hbm_gbs") or 6532.0
    fp32_peak_tflops = sm_count.value * 128 * 2 * sm_max * 1e6 / 1e12
    achieved = FLOP_PER_EMD_EVAL * evals / (emd_ms * 1e-3) / 1e12
    roofline = {"kernel": "emd_auction_kernel (with the fused CalcDist / sqrt-mean / gradient epilogue)", "bound": "fp32-cuda-core", "achieved": achieved,
                "peak": fp32_peak_tflops, "unit": "TFLOP/s", "frac": achieved / fp32_peak_tflops, "traffic": NCU_AUCTION_DRAM_BYTES,
                "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, profiles/ (algorithmic: 1.57 MB inputs + 1.3 MB "
                                  "outputs; the auction state never leaves shared memory)",
                "peak_source": f"{sm_count.value} SMs x 128 lanes x 2 FLOP x {sm_max:.0f} MHz (MEASURED_PEAKS.json sm_max_mhz); "
                               "contraction depth 3 => CUDA-core bound, neither hbm nor tensor (SURVEY.md 8d)",
                "algorithmic": f"{FLOP_PER_EMD_EVAL} FLOP x N x sum_t U_t = {FLOP_PER_EMD_EVAL * evals:.3e} FLOP per launch",
                "pair_evals_per_s": evals / (emd_ms * 1e-3), "avg_launch_ms": emd_ms,
                "executed_fraction": statistics.mean(executed) / evals,
                "executed_note": "algorithmic = every (bidder, target) pair of the reference's Bid (N * sum_t U_t); the kernel proves "
                                 "whole 32-target tiles irrelevant with an exact bounding-box test and really evaluates only this fraction"}
    ch_evals = 2.0 * B_PER_GPU * NPTS * NPTS
    ch_ms = statistics.mean(phases["chamfer_fwd"])
    ch_achieved = FLOP_PER_CHAMFER_EVAL * ch_evals / (ch_ms * 1e-3) / 1e12
    roofline_chamfer = {"kernel": "chamfer_nn3_kernel (one launch incl. the final reduction; + a 4-byte ticket memset); average of 8 back-to-back launches on rotating inputs", "bound": "fp32-cuda-core",
                        "achieved": ch_achieved, "peak": fp32_peak_tflops, "unit": "TFLOP/s", "frac": ch_achieved / fp32_peak_tflops, "traffic": None,
                        "avg_launch_ms": ch_ms,
                        "algorithmic": f"{FLOP_PER_CHAMFER_EVAL} FLOP x 2*B*N*M directed evaluations = {FLOP_PER_CHAMFER_EVAL * ch_evals:.3e} FLOP per launch",
                        "executed_fma_lane_ops_frac": 3 * ch_evals / (ch_ms * 1e-3) / (fp32_peak_tflops * 1e12 / 2)}
    # backward kernels: gather / scatter, bounded by the memory system (SURVEY.md 8d: 56 B per point and direction for Chamfer, 44 B per
    # point for EMD).  The whole working set (3-7 MB) is L2-resident, so HBM never sees most of it: the fraction of the HBM copy peak is
    # reported as asked, the limiter is L2 / atomic latency, not DRAM bandwidth (ncu lts counters in profiles/).
    chb_ms, emb_ms = statistics.mean(phases["chamfer_bwd"]), statistics.mean(phases["emd_bwd_kernel_alone"])
    chb_bytes, emb_bytes = 2.0 * B_PER_GPU * NPTS * 56, 1.0 * B_PER_GPU * NPTS * 44
    roofline_bwd = {
        "chamfer_bwd_kernel (+ 2 zero fills)": {"bound": "hbm", "achieved": chb_bytes / (chb_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                                "frac": chb_bytes / (chb_ms * 1e-3) / 1e9 / hbm_peak, "avg_launch_ms": chb_ms,
                                                "algorithmic": f"2*B*N*56 B = {chb_bytes / 1e6:.2f} MB per launch", "traffic": None},
        "emd_bwd_kernel": {"bound": "hbm", "achieved": emb_bytes / (emb_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                           "frac": emb_bytes / (emb_ms * 1e-3) / 1e9 / hbm_peak, "avg_launch_ms": emb_ms,
                           "algorithmic": f"B*N*44 B = {emb_bytes / 1e6:.2f} MB per launch", "traffic": None,
                           "note": "module-level emdFunction.backward only; in the timed step the EMD gradient is written by the auction kernel's epilogue"},
        "note": "both working sets are L2-resident (126 MB L2): latency / atomic bound, not DRAM bound"}
    breakdown = {k: statistics.mean(v) for k, v in phases.items()}
    breakdown["ms_per_step_independent"] = statistics.mean(per_regime["independent"]) if per_regime["independent"] else None
    breakdown["ms_per_step_noisy"] = statistics.mean(per_regime["noisy"]) if per_regime["noisy"] else None
    breakdown["chamfer_directed_pair_evals_per_s"] = ch_evals / (ch_ms * 1e-3)
    breakdown["ms_per_step_phases_run_sequentially"] = breakdown["chamfer_fwd"] + breakdown["chamfer_bwd"] + breakdown["emd_fused_fwd_bwd"]
    breakdown["collective_ms"] = coll_ms

    # ---- e2e: HOST buffers in, HOST results out, every step, through the C ABI (pcl_chamfer_emd_step_host) ------
    # timed region per step: H2D of that step's pinned inputs, the three kernels, (N > 1: the all-reduce of the batch sums,) D2H of the
    # loss vector, stream sync
    host = [(p.cpu().pin_memory(), t.cpu().pin_memory()) for p, t, _ in pool[:16]]
    L = _lib.lib()
    nbytes = L.pcl_loss_host_scratch_bytes(B_PER_GPU, NPTS)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=device)
    loss_h = torch.zeros(8).pin_memory()
    red_d, red_h = torch.zeros(4, device=device), torch.zeros(4).pin_memory()
    cur_stream = torch.cuda.current_stream()

    def host_step(i):
        ph, th = host[i % len(host)]
        rc = L.pcl_chamfer_emd_step_host(ph.data_ptr(), th.data_ptr(), B_PER_GPU, NPTS, EPS, ITERS, 0, loss_h.data_ptr(), None, None,
                                         scratch.data_ptr(), nbytes, st)
        if rc:
            raise RuntimeError(L.pcl_last_error().decode())
        cur_stream.synchronize()  # the caller reads loss_h now
        if world > 1:             # the sharded caller's collective on the four batch sums, result read back
            red_d.copy_(loss_h[2:6], non_blocking=True)
            dist.all_reduce(red_d)
            red_h.copy_(red_d, non_blocking=True)
            cur_stream.synchronize()
            return float(red_h[2] / red_h[3])
        return float(loss_h[0]) + float(loss_h[1]) + float(loss_h[6])

    Ke = max(8, min(K, 200))
    serial_ms = timed(host_step, Ke, 3)

    # The same step the way a training loop issues it: a data loader that prefetches ONE batch -- the next batch's host->device copy runs
    # on a copy stream while the current step computes; the kernels of consecutive steps stay serialised on the compute stream (a
    # step's prediction depends on the previous optimiser step, so compute must not overlap), and every step's loss vector is read on
    # the host.  Every step copies its own inputs from pinned host memory inside the timed region.
    copy_stream = torch.cuda.Stream(device=device)
    estep = pcl.ShardedChamferEmdStep(B_PER_GPU, NPTS, device, EPS, ITERS)
    slots = [{"p": torch.empty(B_PER_GPU, NPTS, 3, device=device), "t": torch.empty(B_PER_GPU, NPTS, 3, device=device),
              "copied": torch.cuda.Event(), "free": torch.cuda.Event(), "loss_h": torch.zeros(4).pin_memory()} for _ in range(2)]
    for sl in slots:
        sl["free"].record(cur_stream)

    def prefetch(i):
        sl = slots[i & 1]
        ph, th = host[i % len(host)]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(sl["free"])          # the step that last read this slot is done with it
            sl["p"].copy_(ph, non_blocking=True)
            sl["t"].copy_(th, non_blocking=True)
            sl["copied"].record(copy_stream)

    def compute_and_read(i):
        sl = slots[i & 1]
        cur_stream.wait_event(sl["copied"])
        estep.step(sl["p"], sl["t"])                     # the three kernels (+ the all-reduce of the batch sums at N > 1)
        sl["free"].record(cur_stream)
        sl["loss_h"].copy_(estep.wait(), non_blocking=True)   # the loss is read every step here: the stream waits for the collective
        prefetch(i + 1)                                  # copy of the NEXT step's inputs: issued while this step's kernels run
        cur_stream.synchronize()                         # the caller reads the loss now
        return float(sl["loss_h"][2] / sl["loss_h"][3])

    def prefetched(k, w):
        prefetch(0)
        for i in range(w):
            compute_and_read(i)
        barrier()
        e0, e1 = ev(), ev()
        e0.record()
        for i in range(w, w + k):
            compute_and_read(i)
        e1.record()
        barrier()
        copy_stream.synchronize()
        return max_over_ranks(e0.elapsed_time(e1))

    e2e_ms = prefetched(Ke, 4)

    # Two independent batches in flight (two streams, two scratch areas; e.g. micro-batches of a gradient-accumulation step or a
    # validation loop): the second batch's clusters start on the SMs the first batch's fast clouds free, which the single-batch launch
    # cannot do.  Reported separately -- it is not what a strictly sequential training step sees.
    side = torch.cuda.Stream(device=device)
    lanes = [(cur_stream, scratch, loss_h), (side, torch.empty(nbytes, dtype=torch.uint8, device=device), torch.zeros(8).pin_memory())]
    pending = []

    def read_back(lane):
        stream_, _, lh = lane
        stream_.synchronize()
        return float(lh[0]) + float(lh[1]) + float(lh[6])

    def issue(i):
        lane = lanes[i & 1]
        ph, th = host[i % len(host)]
        rc = L.pcl_chamfer_emd_step_host(ph.data_ptr(), th.data_ptr(), B_PER_GPU, NPTS, EPS, ITERS, 0, lane[2].data_ptr(), None, None,
                                         lane[1].data_ptr(), nbytes, lane[0].cuda_stream)
        if rc:
            raise RuntimeError(L.pcl_last_error().decode())
        return lane

    def two_in_flight(k, w):
        for i in range(w):
            read_back(issue(i))
        barrier()
        e0, e1 = ev(), ev()
        e0.record()
        pending.clear()
        for i in range(k):
            pending.append(issue(w + i))
            if len(pending) == 2:
                read_back(pending.pop(0))
        while pending:
            read_back(pending.pop(0))
        e1.record()  # after the host has the last step's result: both streams are idle
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    two_ms = two_in_flight(Ke, 4) if world == 1 else None
    e2e = {"value": world * B_PER_GPU * Ke / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 2 * B_PER_GPU * NPTS * 3 * 4,
           "d2h_bytes_per_step": 16, "steps": Ke, "ms_per_step": e2e_ms / Ke,
           "path": "pinned host inputs -> H2D on a copy stream (the NEXT step's copy overlaps this step's kernels: one prefetched batch) -> C ABI "
                   "pcl_chamfer_emd_step: auction with fused epilogue | Chamfer fwd, Chamfer bwd (+ the all-reduce of the batch sums at N > 1) -> "
                   "D2H of the loss sums -> host reads them, every step; compute of consecutive steps is serialised (gradients stay on the device, "
                   "as in training)",
           "serial": {"value": world * B_PER_GPU * Ke / (serial_ms * 1e-3), "ms_per_step": serial_ms / Ke,
                      "path": "C ABI pcl_chamfer_emd_step_host, strictly one step at a time: copy, kernels, read back, then the next copy"}}
    if two_ms is not None:
        e2e["two_batches_in_flight"] = {
            "value": B_PER_GPU * Ke / (two_ms * 1e-3), "ms_per_step": two_ms / Ke,
            "path": "pcl_chamfer_emd_step_host on two streams, the loss of step i read while step i+1 runs: kernels of two independent batches "
                    "overlap (the second batch's clusters fill the SMs the first batch's fast clouds free)"}

    # ---- the same through the Python loss API (autograd Functions), for the torch user -----------------------------
    emd_mod = pcl.emdModule()

    def api_step(i):
        ph, th = host[i % len(host)]
        p = ph.to(device, non_blocking=True).requires_grad_()
        t = th.to(device, non_blocking=True)
        closs, _ = pcl.chamfer_distance(p, t)
        d, _ = emd_mod(p, t, EPS, ITERS)
        eloss = d.sqrt().mean()
        (closs + eloss).backward()
        return torch.stack([closs.detach(), eloss.detach()]).cpu()  # device -> host read of the step's result (synchronises)

    def api_fused_step(i):
        ph, th = host[i % len(host)]
        p = ph.to(device, non_blocking=True).requires_grad_()
        t = th.to(device, non_blocking=True)
        closs, eloss = pcl.chamfer_emd_loss(p, t, EPS, ITERS)
        (closs + eloss).backward()
        return torch.stack([closs.detach(), eloss.detach()]).cpu()  # device -> host read of the step's result (synchronises)

    # the same with one prefetched batch (copy stream), like the C-ABI e2e leg: what a DataLoader with pinned memory gives the trainer
    loss2_h = [torch.zeros(2).pin_memory() for _ in range(2)]

    def api_prefetched_step(i):
        sl = slots[i & 1]
        cur_stream.wait_event(sl["copied"])
        p = sl["p"].detach().requires_grad_()
        closs, eloss = pcl.chamfer_emd_loss(p, sl["t"], EPS, ITERS)
        (closs + eloss).backward()
        sl["free"].record(cur_stream)
        loss2_h[i & 1].copy_(torch.stack([closs.detach(), eloss.detach()]), non_blocking=True)
        prefetch(i + 1)
        cur_stream.synchronize()
        return float(loss2_h[i & 1][0]) + float(loss2_h[i & 1][1])

    def api_prefetched(k, w):
        copy_stream.synchronize(); cur_stream.synchronize()
        for sl in slots:
            sl["free"].record(cur_stream)
        prefetch(0)
        for i in range(w):
            api_prefetched_step(i)
        barrier()
        e0, e1 = ev(), ev()
        e0.record()
        for i in range(w, w + k):
            api_prefetched_step(i)
        e1.record()
        barrier()
        copy_stream.synchronize()
        return max_over_ranks(e0.elapsed_time(e1))

    Kp = max(8, min(K, 40))
    api_ms = timed(api_step, Kp, 3)
    apis_ms = timed(api_fused_step, Kp, 3)
    apif_ms = api_prefetched(Kp, 4)
    e2e["python_api"] = {"value": world * B_PER_GPU * Kp / (apif_ms * 1e-3), "ms_per_step": apif_ms / Kp, "steps": Kp,
                         "path": "pointcloud_b200.chamfer_emd_loss (one autograd Function over pcl_chamfer_emd_step) + backward; pinned host "
                                 "inputs copied every step on a copy stream (one prefetched batch, as in `e2e`), both losses read back every step",
                         "serial": {"value": world * B_PER_GPU * Kp / (apis_ms * 1e-3), "ms_per_step": apis_ms / Kp,
                                    "path": "the same Function, copy -> forward -> backward -> read back strictly one step at a time"},
                         "separate_calls": {"value": world * B_PER_GPU * Kp / (api_ms * 1e-3), "ms_per_step": api_ms / Kp,
                                            "path": "pointcloud_b200.chamfer_distance + emdModule + autograd (two calls on one stream, "
                                                    "the reference's module-level surface), same copies and read-back"}}

    # ---- the loss CLASSES train.py uses, through ShardedLoss, fwd + bwd, collectives inside the timed region (config 3 = Segmenter) ----
    def class_leg(make_batch, loss_fn):
        sh = pcl.ShardedLoss(loss_fn)
        data = []
        for s_ in range(2):
            for regime in ("independent", "noisy"):
                pr, tg = make_batch(B_PER_GPU, NPTS, seed=1000 * rank + s_, regime=regime)
                data.append((pr.to(device), tg.to(device)))

        def fn(i):
            pr, tg = data[i % len(data)]
            x = pr.detach().requires_grad_()
            sh(x, tg).backward()
        k = max(8, min(K, 40))
        ms = timed(fn, k, 3)
        return {"ms_per_step": ms / k, "value": world * B_PER_GPU * k / (ms * 1e-3), "unit": UNIT, "steps": k}
    sharded_api = {
        "autoencoder_loss (EarthMoverDistance, 1 all-reduce per call)": class_leg(synth.autoencoder_batch, pcl.EarthMoverDistance(EPS, ITERS)),
        "segmenter_loss = config 3 (weighted EMD + CE, 2 dependent all-reduces per call)": class_leg(synth.segmenter_batch, pcl.EarthMoverDistance(EPS, ITERS, num_classes=5)),
        "chamfer_loss (ChamferDistance, 1 all-reduce per call)": class_leg(lambda b, n, seed, regime: tuple(x[:, :, :3].contiguous() for x in synth.table_clouds(b, n, seed=seed, regime=regime)), pcl.ChamferDistance()),
        "path": "pointcloud_b200.ShardedLoss(loss class) forward + backward per step, device-resident inputs, python autograd"}

    # ---- BASELINE config 5: Chamfer fwd+bwd, B=64 GLOBAL, N=M in {1k..16k} (strong scaling: 64/N clouds per rank, the ONE all-reduce of
    #      the two batch sums inside the step); config 1: the reference's CPU-runnable case (B=8, N=2048) on the GPU and on the CPU port ----
    def config5_leg():
        Lc, Ac = _lib.lib(), _lib.pts_args
        bg = 64
        bl5 = max(1, bg // world)
        rows = []
        for n5 in (1024, 2048, 4096, 8192, 16384):
            xg, yg = synth.uniform_clouds(bg, n5, seed=0)
            x5, y5 = xg[rank * bl5:(rank + 1) * bl5].to(device), yg[rank * bl5:(rank + 1) * bl5].to(device)
            e5 = lambda *sh, dt=torch.float32: torch.empty(*sh, device=device, dtype=dt)
            dx, dy, ix, iy, lxy = e5(bl5, n5), e5(bl5, n5), e5(bl5, n5, dt=torch.int32), e5(bl5, n5, dt=torch.int32), e5(4)
            gx, gy, ones = e5(bl5, n5, 3), e5(bl5, n5, 3), torch.ones(2, device=device)
            wsb = Lc.pcl_chamfer_workspace_bytes(bl5, n5, n5)
            ws5 = torch.empty(wsb, device=device, dtype=torch.uint8)

            def step5(i):
                rc = Lc.pcl_chamfer_fwd(*Ac(x5), None, *Ac(y5), None, bl5, n5, n5, 3, 0, dx.data_ptr(), ix.data_ptr(), dy.data_ptr(), iy.data_ptr(),
                                        lxy.data_ptr(), ws5.data_ptr(), wsb, st)
                if world > 1:
                    dist.all_reduce(lxy[2:4])
                rc |= Lc.pcl_chamfer_bwd(*Ac(x5), None, *Ac(y5), None, bl5, n5, n5, 3, ix.data_ptr(), iy.data_ptr(), ones.data_ptr(), gx.data_ptr(),
                                         gy.data_ptr(), st)
                if rc:
                    raise RuntimeError(Lc.pcl_last_error().decode())
            k5 = 20 if n5 <= 4096 else 8
            ms5 = timed(step5, k5, 3) / k5
            rows.append({"N": n5, "clouds_per_gpu": bl5, "step_ms": ms5, "clouds_per_s": bg / (ms5 * 1e-3),
                         "algorithmic_fp32_frac": FLOP_PER_CHAMFER_EVAL * 2.0 * bl5 * n5 * n5 / (ms5 * 1e-3) / 1e12 / fp32_peak_tflops})
        return {"B_global": bg, "scaling": "strong", "rows": rows,
                "note": "N >= 6144 takes the spatially pruned forward (most pairs are never evaluated: the algorithmic fraction can exceed 1)"}

    def config1_leg():
        import oracle
        x1c, t1c = synth.table_clouds(8, NPTS, seed=0)
        y1c = t1c[:, :, :3].contiguous()
        xd, yd = x1c.to(device), y1c.to(device)

        def gpu(i):
            xx = xd.detach().requires_grad_()
            loss, _ = pcl.chamfer_distance(xx, yd)
            loss.backward()
        gms = timed(gpu, 20, 3) / 20
        t0 = time.perf_counter()
        for _ in range(3):
            c = oracle.chamfer_forward(x1c, y1c, nthreads=os.cpu_count() or 1)
            oracle.chamfer_backward(x1c, y1c, c["idx_x"], c["idx_y"], 1.0)
        cms = (time.perf_counter() - t0) / 3 * 1e3
        return {"shape": [8, NPTS, NPTS], "gpu_python_api_fwd_bwd_ms": gms, "cpu_oracle_port_fwd_bwd_ms": cms, "cpu_threads": os.cpu_count()}

    config5 = config5_leg()
    config1 = config1_leg() if (rank == 0 and world == 1) else None

    # ---- parity of the timed step against the oracle; the reference's own step on the same GPU; the CPU baseline ----
    reference_gpu, cb, parity_ok, parity = None, None, None, None
    if rank == 0:
        parity_ok, parity = parity_check(torch, np, pcl, pool, device)
        try:
            reference_gpu = reference_gpu_step(torch, pool, ev, emd_ms)
        except Exception as ex:  # the reference build is optional context
            reference_gpu = {"unavailable": repr(ex)}
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_baseline(16, 40, 2)  # ~10 s of CPU work on 16 cores
            cb = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        par = (f"batch-sharded x{world}: {B_PER_GPU} clouds per rank, one NCCL all-reduce (SUM, 4 x fp32 batch sums) per step inside the timed region, "
               "issued asynchronously (the next step's kernels do not queue behind it; nothing but the logged loss depends on it)"
               if world > 1 else "1 rank (the sharded step degenerates to the local call: no collective)")
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "clouds_per_gpu": B_PER_GPU, "points": NPTS, "eps": EPS, "iters": ITERS,
                           "chamfer_mode": "unfused", "parallelism": par,
                           "l2": f"inputs rotate through {n_sets} sets = {n_sets * 2 * B_PER_GPU * NPTS * 12 / 1e6:.0f} MB > 126 MB L2 (no flush needed)"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": KERNELS_PER_STEP * K, "roofline": roofline,
                "roofline_chamfer": roofline_chamfer, "roofline_bwd": roofline_bwd, "parity_checked": parity_ok, "parity": parity,
                "sharded_equals_single_gpu": sharded_equals_single, "strong_scaling": strong, "sharded_api": sharded_api,
                "cpu_baseline": cb, "breakdown_ms": breakdown, "reference_gpu": reference_gpu,
                "other_configs": {"config1_chamfer_B8_N2048": config1, "config3_segmenter_loss": "sharded_api['segmenter_loss = config 3 ...']",
                                  "config5_chamfer_sweep_B64": config5}, "impl": "ours"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
