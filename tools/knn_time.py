"""K-nearest-neighbour kernel time on the GPU: pcl_knn_fwd / pcl_knn_bwd through the C ABI with preallocated outputs,
against the same GPU's dense torch formulation (torch.cdist -> square -> topk(largest=False), backward through autograd).

  python tools/knn_time.py [--out FILE] [--iters N]

Each time is the mean over N back-to-back launches (CUDA events around the whole window) on R rotating input copies,
after a warm-up of every shape.  Pair evaluations per second count B*P1*P2 distances; the share of the FP32 CUDA-core
peak uses 8 FLOP per pair and peak = SMs x 128 lanes x 2 x max SM clock (BASELINE.md / DESIGN.md section 5)."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointcloud_b200 import _lib, synth  # noqa: E402

SHAPES = [  # name, B, P1, P2, K
    ("grouping", 32, 512, 2048, 1), ("grouping", 32, 512, 2048, 16), ("grouping", 32, 512, 2048, 32),
    ("self-kNN", 32, 2048, 2048, 16), ("large", 8, 16384, 16384, 16),
]
L2_BYTES = 126 << 20


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, mhz = [s.strip() for s in q.stdout.strip().split(",")]
    return name, float(power), float(mhz)


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    _lib.require_cuda()
    L = _lib.lib()
    name, power, mhz = device_line()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    peak = sms * 128 * 2 * mhz * 1e6
    lines = [f"device: {name}, power limit {power:.0f} W, max SM clock {mhz:.0f} MHz, {sms} SMs -> FP32 peak {peak / 1e12:.1f} TFLOP/s",
             f"library: {os.path.basename(_lib.lib_path())}",
             "shape            B     P1     P2   K | ours fwd us  bwd us  Gpair/s  peak | torch fwd us  fwd+bwd us | speed-up fwd  fwd+bwd | inputs"]
    for sname, B, P1, P2, K in SHAPES:
        R = 4
        clouds = []
        for r in range(R):
            x, t = synth.table_clouds(B, max(P1, P2), seed=r)
            clouds.append((x[:, :P1].contiguous().cuda(), t[:, :P2, :3].contiguous().cuda()))
        in_bytes = R * B * (P1 + P2) * 3 * 4
        resident = "L2-resident" if in_bytes + B * P1 * K * 8 < L2_BYTES else "exceeds L2"
        dists = torch.empty(B, P1, K, device="cuda"); idx = torch.empty(B, P1, K, device="cuda", dtype=torch.int32)
        gd = torch.randn(B, P1, K, device="cuda")
        g1 = torch.empty(B, P1, 3, device="cuda"); g2 = torch.empty(B, P2, 3, device="cuda")
        A = _lib.pts_args
        it = [0]

        def fwd():
            a, b = clouds[it[0] % R]; it[0] += 1
            assert L.pcl_knn_fwd(*A(a), None, *A(b), None, B, P1, P2, 3, K, 0, dists.data_ptr(), idx.data_ptr(), None) == 0

        def bwd():
            a, b = clouds[it[0] % R]; it[0] += 1
            assert L.pcl_knn_bwd(*A(a), None, *A(b), None, B, P1, P2, 3, K, idx.data_ptr(), gd.data_ptr(), g1.data_ptr(),
                                 g2.data_ptr(), None) == 0

        iters = max(5, args.iters if P1 * P2 <= 2048 * 2048 else args.iters // 5)
        tf, tb = timed(fwd, iters), timed(bwd, iters)
        pairs = B * P1 * P2

        def t_fwd():
            a, b = clouds[it[0] % R]; it[0] += 1
            return torch.cdist(a, b).square().topk(K, dim=-1, largest=False)

        def t_fwd_bwd():
            a, b = clouds[it[0] % R]; it[0] += 1
            a = a.detach().requires_grad_(); b = b.detach().requires_grad_()
            dv, _ = torch.cdist(a, b).square().topk(K, dim=-1, largest=False)
            dv.backward(gd)

        titers = max(3, iters // 2)
        try:
            ttf, ttb = timed(t_fwd, titers), timed(t_fwd_bwd, titers)
            tstr = f"{ttf:12.1f}  {ttb:10.1f} | {ttf / tf:11.2f}x {ttb / (tf + tb):7.2f}x"
        except torch.OutOfMemoryError:
            tstr = f"{'OOM':>12}  {'OOM':>10} | {'-':>12} {'-':>8}"
        torch.cuda.empty_cache()
        lines.append(f"{sname:<12} {B:5d} {P1:6d} {P2:6d} {K:3d} | {tf:11.1f} {tb:7.1f} {pairs / tf / 1e3:8.1f} {8 * pairs / (tf * 1e-6) / peak:5.2f} | "
                     f"{tstr} | {in_bytes / 2**20:.1f} MB in {R} rotating copies, {resident}")
        print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
