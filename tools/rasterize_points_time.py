"""Point rasterization and compositing time on the GPU: rasterize_points forward and forward+backward with bin_size=0 (every
pixel block scans its whole cloud), with the automatic bin size and with each fixed bin size; the three compositors'
forward and forward+backward at C=3 and C=16 on the rasterizer's output; and a dense torch restatement on the same GPU
(pixel-chunked d2 -> mask -> topk, backward through autograd).

  python tools/rasterize_points_time.py [--out FILE] [--iters N]

Each time is the mean over N back-to-back calls (CUDA events around the whole window) on R rotating input copies, after a
warm-up of every shape (tools/knn_time.py's method).  Clouds are Table-shaped (synth.table_clouds) with x, y mapped into
[-0.9, 0.9] of the shorter side and z into [0.5, 1.5]; the weights fed to the compositors are 1 - dists / r^2."""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pointcloud_b200 as pcl  # noqa: E402
from pointcloud_b200 import _lib, synth  # noqa: E402
from pointcloud_b200.rasterize_points import auto_bin_size  # noqa: E402
from raster_ref import pixel_centres  # noqa: E402
from tools.knn_time import device_line, timed  # noqa: E402

SHAPES = [  # B, P, (H, W), r, K
    (32, 2048, (128, 128), 0.02, 8),
    (8, 16384, (256, 256), 0.01, 8),
    (8, 16384, (256, 256), 0.01, 1),
    (1, 262144, (512, 512), 0.005, 8),
    (4, 65536, (240, 320), 0.01, 8),
]
BIN_SIZES = (16, 32, 64, 128)


def clouds(B, P, seed):
    x = synth.table_clouds(B, P, seed=seed)[0].clone()
    x[..., :2] = x[..., :2] * 1.8 - 0.9
    x[..., 2] = x[..., 2] + 0.5
    return x.cuda()


def dense_torch(points, H, W, r, K, rows=8):
    """The dense restatement: per chunk of rows a (B, rows, W, P) d2, masked to +inf outside the radius or behind the
    camera, z keyed, topk; dists gathered with autograd."""
    B, P, _ = points.shape
    xs, ys = pixel_centres(H, W, device=points.device)
    idx_out, z_out, d_out = [], [], []
    for r0 in range(0, H, rows):
        yy = ys[r0:r0 + rows]
        dx = xs[None, None, :, None] - points[:, None, None, :, 0]
        dy = yy[None, :, None, None] - points[:, None, None, :, 1]
        d2 = dx * dx + dy * dy
        hit = (d2 <= r * r) & (points[:, None, None, :, 2] >= 0)
        key = torch.where(hit, points[:, None, None, :, 2].expand_as(d2).detach(), torch.full_like(d2, float("inf")))
        kz, ki = torch.topk(key, K, dim=-1, largest=False)
        ok = torch.isfinite(kz)
        idx_out.append(torch.where(ok, ki, -1))
        z_out.append(torch.where(ok, torch.gather(points[..., 2][:, None, None, :].expand_as(d2), -1, ki), -1.0))
        d_out.append(torch.where(ok, torch.gather(d2, -1, ki), -1.0))
    return torch.cat(idx_out, 1), torch.cat(z_out, 1), torch.cat(d_out, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    _lib.require_cuda()
    name, power, mhz = device_line()
    lines = [f"device: {name}, power limit {power:.0f} W, max SM clock {mhz:.0f} MHz",
             f"library: {os.path.basename(_lib.lib_path())}; times in us, mean of {args.iters} calls; "
             "fwd+bwd = forward, sum of zbuf and dists times random upstream gradients, backward"]
    n = args.iters
    for B, P, (H, W), r, K in SHAPES:
        R = 2
        ins = [clouds(B, P, s) for s in range(R)]
        g = torch.Generator().manual_seed(1)
        gz = torch.randn(B, H, W, K, generator=g).cuda()
        gd = torch.randn(B, H, W, K, generator=g).cuda()
        it = [0]

        def nxt():
            x = ins[it[0] % R]
            it[0] += 1
            return x

        auto = auto_bin_size(P)
        row = {}
        for label, bs in [("naive", 0), ("auto", None)] + [(f"bin{b}", b) for b in BIN_SIZES]:
            def fwd():
                return pcl.rasterize_points(nxt(), None, (H, W), r, K, bs)

            def fwd_bwd():
                p = nxt().detach().requires_grad_()
                _, z, d = pcl.rasterize_points(p, None, (H, W), r, K, bs)
                ((z * gz).sum() + (d * gd).sum()).backward()
            row[label] = (timed(fwd, n), timed(fwd_bwd, n))
        want = pcl.rasterize_points(ins[0], None, (H, W), r, K, 0)
        for bs in (None,) + BIN_SIZES:
            got = pcl.rasterize_points(ins[0], None, (H, W), r, K, bs)
            assert all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(got, want)), bs
        hits = float((want[0] >= 0).float().mean())
        try:
            def t_fwd():
                return dense_torch(nxt(), H, W, r, K)

            def t_fwd_bwd():
                p = nxt().detach().requires_grad_()
                _, z, d = dense_torch(p, H, W, r, K)
                ((z * gz).sum() + (d * gd).sum()).backward()
            tt = (timed(t_fwd, max(3, n // 4)), timed(t_fwd_bwd, max(3, n // 4)))
            tstr = f"{tt[0]:.1f} / {tt[1]:.1f}"
        except torch.OutOfMemoryError:
            tt, tstr = None, "OOM"
        torch.cuda.empty_cache()
        lines.append(f"B={B} P={P} {H}x{W} r={r} K={K} (filled slots {100 * hits:.1f} %), auto bin_size={auto}")
        lines.append("  rasterize_points fwd / fwd+bwd: " + "; ".join(f"{k} {v[0]:.1f} / {v[1]:.1f}" for k, v in row.items())
                     + f"; dense torch {tstr}")
        if tt:
            lines.append(f"  auto vs naive: {row['naive'][0] / row['auto'][0]:.2f}x / {row['naive'][1] / row['auto'][1]:.2f}x; "
                         f"auto vs dense torch: {tt[0] / row['auto'][0]:.1f}x / {tt[1] / row['auto'][1]:.1f}x")
        idx, _, dists = want
        ip = idx.permute(0, 3, 1, 2)
        alphas = (1 - dists.permute(0, 3, 1, 2) / r ** 2).contiguous()
        for C in (3, 16):
            feats = torch.rand(B * P, C, device="cuda")
            gimg = torch.randn(B, C, H, W, device="cuda")
            parts = []
            for cname, fn in (("alpha", pcl.alpha_composite), ("norm", pcl.norm_weighted_sum), ("weighted", pcl.weighted_sum)):
                def cf():
                    return fn(ip, alphas, feats.t())

                def cfb():
                    a = alphas.detach().requires_grad_()
                    f = feats.detach().requires_grad_()
                    (fn(ip, a, f.t()) * gimg).sum().backward()
                parts.append(f"{cname} {timed(cf, n):.1f} / {timed(cfb, n):.1f}")
            lines.append(f"  compositors C={C} fwd / fwd+bwd: " + "; ".join(parts))
        for ln in lines[-4:]:
            print(ln, flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
