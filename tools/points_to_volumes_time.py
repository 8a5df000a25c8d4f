"""Points-to-volumes time on the GPU: the public add_points_features_to_volume_densities_features forward and
forward+backward, pcl_points_to_volumes_fwd / _bwd alone through the C ABI with preallocated volumes, and pytorch3d's Python
fallback restated in fp32 torch on the same GPU (per corner one scatter_add_ into the densities and one into the features,
8 corners in trilinear mode and 1 in nearest mode, backward through autograd).

  python tools/points_to_volumes_time.py [--out FILE] [--iters N]

Each time is the mean over N back-to-back calls (CUDA events around the whole window) on R rotating input copies, after a
warm-up of every shape (tools/knn_time.py's method).  Clouds are Table-shaped (synth.table_clouds) scaled from [0, 1] into
[-1, 1], with Gaussian features; initial volumes are random.  The bytes floor of the forward is the padded volume read and
written once, B (C + 1) D H W 4 bytes each way, over 7.7 TB/s (the HGX B200 data sheet's HBM3e bandwidth): a floor that the
public call's clones of the initial volumes alone already meet, not a rate the scatter can reach."""
import argparse
import itertools
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pointcloud_b200 as pcl  # noqa: E402
from pointcloud_b200 import _lib, synth  # noqa: E402
from tools.knn_time import L2_BYTES, device_line, timed  # noqa: E402

HBM = 7.7e12
SHAPES = [  # B, P, grid, C, modes
    (32, 2048, 32, 3, ("trilinear", "nearest")),
    (32, 2048, 64, 32, ("trilinear",)),
    (8, 16384, 64, 16, ("trilinear",)),
    (1, 262144, 128, 3, ("trilinear", "nearest")),
]


def torch_fallback(points, feats, dens0, feat0, mode, min_weight=1e-4, align_corners=True):
    """pytorch3d's Python fallback restated in fp32 torch: lattice coordinates, then per corner a weight, a validity mask, a
    flattened index and two scatter_add_ calls into (B, 1, DHW) and (B, C, DHW); then the rescale."""
    B, P, C = feats.shape
    D, H, W = dens0.shape[2:]
    S = torch.tensor([W, H, D], device=points.device, dtype=torch.float32)
    t = ((points + 1) * 0.5) * (S - 1) if align_corners else ((points + 1) * 0.5) * S - 0.5
    dens = dens0.reshape(B, 1, D * H * W).clone()
    feat = feat0.reshape(B, C, D * H * W).clone()
    ft = feats.permute(0, 2, 1)
    if mode == "trilinear":
        base = t.floor()
        corners = [base + torch.tensor(d, device=t.device, dtype=t.dtype) for d in itertools.product((0, 1), repeat=3)]
    else:
        corners = [t.round()]
    for c in corners:
        w = (1 - (t - c).abs()).prod(-1) if mode == "trilinear" else torch.ones_like(t[..., 0])
        valid = ((c >= 0) & (c < S)).all(-1)
        w = w * valid
        ci = c.long()
        idx = ((ci[..., 2].clamp(0, D - 1) * H + ci[..., 1].clamp(0, H - 1)) * W + ci[..., 0].clamp(0, W - 1))
        dens = dens.scatter_add(2, idx[:, None], w[:, None])
        feat = feat.scatter_add(2, idx[:, None].expand(B, C, P), w[:, None] * ft)
    dens = dens.view(B, 1, D, H, W)
    feat = feat.view(B, C, D, H, W) / dens.clamp(min_weight if mode == "trilinear" else 1.0)
    return feat, dens


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    _lib.require_cuda()
    L = _lib.lib()
    name, power, mhz = device_line()
    lines = [f"device: {name}, power limit {power:.0f} W, max SM clock {mhz:.0f} MHz",
             f"library: {os.path.basename(_lib.lib_path())}; floor = padded volume read + written once at {HBM / 1e12:.1f} TB/s",
             "    B       P grid   C mode      | kernel fwd us  bwd us | public fwd us  fwd+bwd us | torch fwd us  fwd+bwd us | "
             "speed-up fwd  fwd+bwd | floor us | volume"]
    for B, P, G, C, modes in SHAPES:
        R = 2
        ins = []
        for r in range(R):
            g = torch.Generator().manual_seed(r)
            pts = (synth.table_clouds(B, P, seed=r)[0] * 2 - 1).cuda()
            ins.append((pts, torch.randn(B, P, C, generator=g).cuda()))
        dens0 = torch.rand(B, 1, G, G, G, device="cuda")
        feat0 = torch.randn(B, C, G, G, G, device="cuda")
        gd, gf = torch.randn_like(dens0), torch.randn_like(feat0)
        dens, feat = dens0.clone(), feat0.clone()
        gp, gpf = torch.empty(B, P, 3, device="cuda"), torch.empty(B, P, C, device="cuda")
        vol_bytes = B * (C + 1) * G ** 3 * 4
        floor = 2 * vol_bytes / HBM * 1e6
        resident = "L2-resident" if vol_bytes < L2_BYTES else "exceeds L2"
        A = _lib.pts_args
        for mode in modes:
            mi = 0 if mode == "trilinear" else 1
            it = [0]

            def nxt():
                x = ins[it[0] % R]
                it[0] += 1
                return x

            def kfwd():  # accumulates onto the same volumes call after call: the work per call is the same
                p, f = nxt()
                assert L.pcl_points_to_volumes_fwd(*A(p), *A(f), None, None, B, P, C, G, G, G, mi, 1, dens.data_ptr(),
                                                   feat.data_ptr(), None) == 0

            def kbwd():
                p, f = nxt()
                assert L.pcl_points_to_volumes_bwd(*A(p), *A(f), None, None, B, P, C, G, G, G, mi, 1, gd.data_ptr(),
                                                   gf.data_ptr(), gp.data_ptr(), gpf.data_ptr(), None) == 0

            def pub_fwd():
                p, f = nxt()
                return pcl.add_points_features_to_volume_densities_features(p, f, dens0, feat0, mode)

            def pub_fwd_bwd():
                p, f = nxt()
                p, f = p.detach().requires_grad_(), f.detach().requires_grad_()
                vf, vd = pcl.add_points_features_to_volume_densities_features(p, f, dens0, feat0, mode)
                ((vf * gf).sum() + (vd * gd).sum()).backward()

            def t_fwd():
                p, f = nxt()
                return torch_fallback(p, f, dens0, feat0, mode)

            def t_fwd_bwd():
                p, f = nxt()
                p, f = p.detach().requires_grad_(), f.detach().requires_grad_()
                vf, vd = torch_fallback(p, f, dens0, feat0, mode)
                ((vf * gf).sum() + (vd * gd).sum()).backward()

            n = args.iters
            tkf, tkb = timed(kfwd, n), timed(kbwd, n)
            tpf, tpb = timed(pub_fwd, n), timed(pub_fwd_bwd, n)
            try:
                ttf, ttb = timed(t_fwd, max(3, n // 2)), timed(t_fwd_bwd, max(3, n // 2))
                tstr = f"{ttf:12.1f}  {ttb:10.1f} | {ttf / tpf:11.2f}x {ttb / tpb:7.2f}x"
            except torch.OutOfMemoryError:
                tstr = f"{'OOM':>12}  {'OOM':>10} | {'-':>12} {'-':>8}"
            torch.cuda.empty_cache()
            lines.append(f"{B:5d} {P:7d} {G:3d}^3 {C:3d} {mode:<9} | {tkf:13.1f} {tkb:7.1f} | {tpf:13.1f} {tpb:11.1f} | "
                         f"{tstr} | {floor:8.1f} | {vol_bytes / 2**20:.0f} MB, {resident}")
            print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
