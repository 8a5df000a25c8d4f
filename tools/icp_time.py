"""ICP and alignment time on the GPU: (i) iterative_closest_point (one cooperative launch for the whole loop), (ii)
pytorch3d's loop restated in torch with this library's knn_points and fp32 torch.linalg.svd, with its per-iteration
`.all()` host synchronisation -- what a user of this library writes without (i) -- and (iii) the dense torch loop
(cdist + argmin) where it fits in memory.  Also the alignment forward and backward kernels alone.

  python tools/icp_time.py [--out FILE] [--iters N]

Inputs: Table-shaped pairs, Y = X rotated by <= 15 degrees, shifted by <= 0.05, noise sigma = 0.002, shuffled;
max_iterations = 100, relative_rmse_thr = 1e-6.  Each time is the mean over N calls (CUDA events around the whole window,
which ends in a device synchronise) on R rotating input pairs after a warm-up of every shape (tools/knn_time.py's method).
Per-iteration times divide by the iterations that path ran.  The search rate is the algorithmic pair count
(iterations x B x P1 x P2) over path (i)'s whole time, against the FP32 peak at 8 FLOP per pair (tools/knn_time.py)."""
import argparse
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pointcloud_b200 as pcl  # noqa: E402
from pointcloud_b200 import _lib, synth  # noqa: E402
from tools.knn_time import device_line, timed  # noqa: E402

SHAPES = [(32, 2048), (8, 16384), (1, 65536)]
MAX_IT, THR = 100, 1e-6
DENSE_BYTES = 40 << 30  # (iii) runs when its B x P x P fp32 distance matrix fits in this


def make_pair(b, n, seed):
    g = torch.Generator().manual_seed(seed)
    X = synth.table_clouds(b, n, seed=seed)[0]
    axis = torch.randn(b, 3, generator=g)
    axis = axis / axis.norm(dim=1, keepdim=True)
    ang = (torch.rand(b, generator=g) * 2 - 1) * math.radians(15)
    K = torch.zeros(b, 3, 3)
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -axis[:, 2], axis[:, 1], -axis[:, 0]
    K = K - K.transpose(1, 2)
    R = torch.eye(3) + torch.sin(ang)[:, None, None] * K + (1 - torch.cos(ang))[:, None, None] * torch.bmm(K, K)
    T = (torch.rand(b, 1, 3, generator=g) * 2 - 1) * 0.05
    Y = torch.bmm(X, R) + T + 0.002 * torch.randn(b, n, 3, generator=g)
    return X.cuda(), Y[:, torch.randperm(n, generator=g)].contiguous().cuda()


def torch_align(X, Y):
    """pytorch3d's corresponding_points_alignment (no weights, no scale) in fp32 torch."""
    xm, ym = X.mean(1, keepdim=True), Y.mean(1, keepdim=True)
    M = torch.bmm((X - xm).transpose(1, 2), Y - ym) / X.shape[1]
    U, S, Vh = torch.linalg.svd(M)
    E = torch.eye(3, device=X.device).repeat(X.shape[0], 1, 1)
    E[:, 2, 2] = torch.det(torch.bmm(U, Vh))
    R = torch.bmm(torch.bmm(U, E), Vh)
    return R, ym[:, 0] - torch.bmm(xm, R)[:, 0]


def torch_icp(X, Y, nn):
    """pytorch3d's loop: one host synchronisation per iteration.  Returns the iterations run."""
    Xt, prev = X, None
    for it in range(MAX_IT):
        Ynn = nn(Xt, Y)
        R, T = torch_align(X, Ynn)
        Xt = torch.bmm(X, R) + T[:, None]
        rmse = ((Xt - Ynn) ** 2).sum(2).mean(1).sqrt()
        rel = torch.ones_like(rmse) if prev is None else (prev - rmse) / prev
        if bool((rel <= THR).all()):
            return it + 1
        prev = rmse
    return MAX_IT


def nn_lib(Xt, Y):
    return pcl.knn_gather(Y, pcl.knn_points(Xt, Y, K=1).idx)[:, :, 0]


def nn_dense(Xt, Y):
    idx = torch.cdist(Xt, Y).argmin(2)
    return Y.gather(1, idx[..., None].expand(-1, -1, 3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    _lib.require_cuda()
    L = _lib.lib()
    name, power, mhz = device_line()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    peak = sms * 128 * 2 * mhz * 1e6
    lines = [f"device: {name}, power limit {power:.0f} W, max SM clock {mhz:.0f} MHz, {sms} SMs -> FP32 peak {peak / 1e12:.1f} TFLOP/s",
             f"library: {os.path.basename(_lib.lib_path())}; max_iterations={MAX_IT}, relative_rmse_thr={THR}",
             "    B      N | (i) icp us  it  us/it  Gpair/s  peak | (ii) torch+knn us  it  us/it | (iii) dense us  it  us/it | "
             "(ii)/(i) | align fwd us  bwd us"]
    for B, N in SHAPES:
        R_ = 3
        pairs = [make_pair(B, N, 100 * B + r) for r in range(R_)]
        k = [0]

        def nxt():
            p = pairs[k[0] % R_]
            k[0] += 1
            return p

        its = {}

        def run_ours():
            X, Y = nxt()
            its["i"] = len(pcl.iterative_closest_point(X, Y, max_iterations=MAX_IT, relative_rmse_thr=THR).t_history)

        def run_lib():
            X, Y = nxt()
            its["ii"] = torch_icp(X, Y, nn_lib)

        def run_dense():
            X, Y = nxt()
            its["iii"] = torch_icp(X, Y, nn_dense)

        iters = max(2, args.iters if N <= 2048 else args.iters // 5)
        t1 = timed(run_ours, iters)
        t2 = timed(run_lib, max(2, iters // 2))
        if B * N * N * 4 <= DENSE_BYTES:
            try:
                t3 = timed(run_dense, max(2, iters // 2))
                d = f"{t3:13.0f} {its['iii']:3d} {t3 / its['iii']:6.1f}"
            except torch.OutOfMemoryError:
                d = f"{'OOM':>13} {'-':>3} {'-':>6}"
        else:
            d = f"{'does not fit':>13} {'-':>3} {'-':>6}"
        torch.cuda.empty_cache()
        # the alignment kernels alone, on the final correspondences of one pair
        X, Y = pairs[0]
        Ynn = nn_lib(X, Y)
        R, T, s = (torch.empty(B, 3, 3, device="cuda"), torch.empty(B, 3, device="cuda"), torch.empty(B, device="cuda"))
        rec = torch.empty(B, 40, device="cuda", dtype=torch.float64)
        nws = int(L.pcl_points_alignment_workspace_bytes(B, N))
        ws = torch.empty(nws, device="cuda", dtype=torch.uint8)
        gR, gT = torch.randn(B, 3, 3, device="cuda"), torch.randn(B, 3, device="cuda")
        gx, gy = torch.empty(B, N, 3, device="cuda"), torch.empty(B, N, 3, device="cuda")
        A = _lib.pts_args

        def afwd():
            assert L.pcl_points_alignment_fwd(*A(X), *A(Ynn), None, None, B, N, 0, 0, 1e-9, R.data_ptr(), T.data_ptr(),
                                              s.data_ptr(), rec.data_ptr(), ws.data_ptr(), nws, None) == 0

        def abwd():
            assert L.pcl_points_alignment_bwd(*A(X), *A(Ynn), None, None, B, N, 0, 1e-9, rec.data_ptr(), gR.data_ptr(),
                                              gT.data_ptr(), None, gx.data_ptr(), gy.data_ptr(), None, None) == 0

        ta, tb = timed(afwd, 50), timed(abwd, 50)
        gpairs = its["i"] * B * N * N / (t1 * 1e-6) / 1e9
        lines.append(f"{B:5d} {N:6d} | {t1:10.0f} {its['i']:3d} {t1 / its['i']:6.1f} {gpairs:8.0f} {8 * gpairs * 1e9 / peak:5.2f} | "
                     f"{t2:17.0f} {its['ii']:3d} {t2 / its['ii']:6.1f} | {d} | {t2 / t1:7.2f}x | {ta:12.1f} {tb:7.1f}")
        print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
