"""Farthest point sampling time on the GPU: pcl_fps_ragged through the C ABI with preallocated outputs, for the AUTO
cluster size and every forced one, against the torch restatement of pointnet2_utils.py:64-86 on the same GPU.

  python tools/fps_time.py [--out FILE] [--old-lib LIB] [--repeats R]

Each time is the mean over back-to-back launches (CUDA events around the whole window, at least ~0.2 s of work) on
4 rotating input copies, after a warm-up of every shape.  --old-lib loads a second libpcl_b200.so (for instance one built
from a revision before the cluster kernel) and times its pcl_fps on the shapes it supports; for the shapes of PointNet2's
set abstraction the new AUTO, the new CS = 1 and the old library then run R times alternating in the same process,
and the table gives the median and the spread (min..max) of those runs."""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointcloud_b200 import _lib  # noqa: E402

SHAPES = [  # name, B, N, npoint, ragged
    ("SA1", 32, 2048, 512, False), ("SA2", 32, 512, 128, False),
    ("sensor", 1, 4096, 1024, False), ("sensor", 1, 8192, 2048, False), ("sensor", 32, 8192, 2048, False),
    ("sensor", 1, 16384, 2048, False), ("sensor", 4, 16384, 2048, False), ("sensor", 1, 32768, 2048, False),
    ("sensor", 1, 65536, 2048, False), ("sensor", 4, 65536, 2048, False), ("sensor", 16, 65536, 2048, False),
    ("sensor", 64, 65536, 2048, False),
    ("sensor", 1, 262144, 2048, False), ("sensor", 4, 262144, 2048, False), ("sensor", 16, 262144, 2048, False),
    ("sensor", 64, 262144, 2048, False),
    ("ragged", 16, 65536, 2048, True),
]
CLUSTERS = [1, 2, 4, 8, 16]
CTA_POINTS = 16384
R = 4


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, mhz = [s.strip() for s in q.stdout.strip().split(",")]
    return name, float(power), float(mhz)


def timed(fn, min_s=0.2, max_iters=200):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fn(); b.record()
    torch.cuda.synchronize()
    iters = int(min(max_iters, max(3, min_s * 1e3 / max(a.elapsed_time(b), 1e-3))))
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3  # us


def fps_torch(xyz, npoint):  # pointnet2_utils.py:64-86 with the deterministic start index 0 (tests/test_sampling_cpu.py)
    B, N, _ = xyz.shape
    centroids = torch.zeros(B, npoint, dtype=torch.long, device=xyz.device)
    distance = torch.ones(B, N, device=xyz.device) * 1e10
    farthest = torch.zeros(B, dtype=torch.long, device=xyz.device)
    batch = torch.arange(B, device=xyz.device)
    for i in range(npoint):
        centroids[:, i] = farthest
        centroid = xyz[batch, farthest, :].view(B, 1, 3)
        dist = torch.sum((xyz - centroid) ** 2, -1)
        mask = dist < distance
        distance[mask] = dist[mask]
        farthest = torch.max(distance, -1)[1]
    return centroids


def load_old(path):
    L = ctypes.CDLL(os.path.abspath(path))
    L.pcl_fps.restype, L.pcl_fps.argtypes = _lib._SIGNATURES["pcl_fps"]
    L.pcl_fps_max_points.restype = ctypes.c_int
    return L


def fmt(v):
    return f"{v:10.1f}" if v is not None else f"{'-':>10}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--old-lib", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    args = ap.parse_args()
    _lib.require_cuda()
    L = _lib.lib()
    old = load_old(args.old_lib) if args.old_lib else None
    name, power, mhz = device_line()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lines = [f"device: {name}, power limit {power:.0f} W, max SM clock {mhz:.0f} MHz, {sms} SMs",
             f"library: {os.path.basename(_lib.lib_path())}" + (f", old library: {os.path.basename(args.old_lib)}" if old else ""),
             "times in us per launch (fp32 xyz, skip_origin=0); 'us/pt' = AUTO time / samples; '-' = cluster too small for N",
             f"{'shape':<7} {'B':>3} {'N':>7} {'S':>5} | {'AUTO':>10} {'us/pt':>7} | " + " ".join(f"{'CS=' + str(c):>10}" for c in CLUSTERS)
             + f" | {'old fps':>10} | {'torch':>12} | AUTO vs CS=1, old, torch"]
    print("\n".join(lines), flush=True)
    for sname, B, N, S, ragged in SHAPES:
        g = torch.Generator(device="cuda").manual_seed(N + B)
        clouds = [torch.rand(B, N, 3, device="cuda", generator=g) for _ in range(R)]
        lengths = None
        if ragged:
            lengths = torch.linspace(N // 4, N, B, device="cuda").long()
        idx = torch.empty(B, S, device="cuda", dtype=torch.int32)
        it = [0]

        def new(cs):
            def f():
                x = clouds[it[0] % R]; it[0] += 1
                assert L.pcl_fps_ragged(*_lib.pts_args(x), _lib.ptr(lengths), B, N, None, S, None, 0, cs, idx.data_ptr(), None) == 0
            return f

        def old_fn():
            x = clouds[it[0] % R]; it[0] += 1
            assert old.pcl_fps(*_lib.pts_args(x), B, N, S, None, 0, idx.data_ptr(), None) == 0

        has_old = old is not None and not ragged and N <= old.pcl_fps_max_points()
        for f in [new(0)] + [new(c) for c in CLUSTERS if c * CTA_POINTS >= N] + ([old_fn] if has_old else []):
            f()  # warm every configuration of the shape
        torch.cuda.synchronize()
        t_cs = {c: (timed(new(c)) if c * CTA_POINTS >= N else None) for c in CLUSTERS}
        spread = ""
        if has_old and N <= 2048:  # the set-abstraction shapes: alternate AUTO / CS=1 / old in the same process
            runs = {"auto": [], "cs1": [], "old": []}
            for _ in range(args.repeats):
                runs["auto"].append(timed(new(0))); runs["cs1"].append(timed(new(1))); runs["old"].append(timed(old_fn))
            t_auto, t_old = statistics.median(runs["auto"]), statistics.median(runs["old"])
            t_cs[1] = statistics.median(runs["cs1"])
            spread = "  [" + ", ".join(f"{k} {min(v):.1f}..{max(v):.1f}" for k, v in runs.items()) + f" over {args.repeats} alternating runs]"
        else:
            t_auto = timed(new(0))
            t_old = timed(old_fn) if has_old else None
        t_torch = None
        if not ragged:
            x = clouds[0]
            fps_torch(x, 8)
            torch.cuda.synchronize()
            t_torch = timed(lambda: fps_torch(x, S), min_s=0.0, max_iters=1)
        ratio = lambda t: f"{t / t_auto:6.2f}x" if t else f"{'-':>7}"
        lines.append(f"{sname:<7} {B:3d} {N:7d} {S:5d} | {t_auto:10.1f} {t_auto / S:7.3f} | " + " ".join(fmt(t_cs[c]) for c in CLUSTERS)
                     + f" | {fmt(t_old)} | {fmt(t_torch):>12} | {ratio(t_cs[1])} {ratio(t_old)} {ratio(t_torch)}" + spread
                     + (" (lengths spread over [N/4, N])" if ragged else ""))
        print(lines[-1], flush=True)
        del clouds
        torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n"
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
