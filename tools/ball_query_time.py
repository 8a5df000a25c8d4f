"""Ball-query kernel time on the GPU: pcl_ball_query_fwd / pcl_ball_query_bwd through the C ABI with preallocated
outputs, against the same GPU's dense torch restatement (a query-chunked distance matrix, `< r2`, a cumsum rank and a
scatter of the first K hits; backward through autograd), and at D = 3 the in-library pointnet2 kernel pcl_ball_query
(same scan with `<=`, no lengths, no distances) at the same shapes.

  python tools/ball_query_time.py [--out FILE] [--iters N]

Inputs are uniform unit-cube clouds; for the large sensor clouds the queries are 2048 farthest-point-sampled points of
the cloud.  Each time is the mean over N back-to-back launches (CUDA events around the whole window) on R rotating
input copies, after a warm-up of every shape.  `hits` is the mean number of kept targets per query (capped at K) and
`parts` the number of warps that split the targets of one CTA's 32 queries (the rule of pcl_knn.cu)."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointcloud_b200 import _lib, sample_farthest_points  # noqa: E402
from pointcloud_b200.ball_query import _radius2  # noqa: E402
from tools.knn_time import device_line, timed  # noqa: E402

SHAPES = [  # name, B, P1, P2, K, radius
    ("SA1", 32, 512, 2048, 32, 0.2), ("SA2", 32, 128, 512, 64, 0.4), ("dense", 8, 16384, 16384, 32, 0.05),
    ("sensor", 1, 2048, 65536, 64, 0.02), ("sensor", 1, 2048, 65536, 64, 0.1),
    ("sensor", 1, 2048, 262144, 64, 0.02), ("sensor", 1, 2048, 262144, 64, 0.1),
]


def parts_for(B, P1, P2, K, sms):  # bq_parts_for of pcl_knn.cu, for the report only
    parts = 1
    while parts * 2 <= 16 and B * ((P1 + 31) // 32) * parts < 8 * sms and P2 // (parts * 2) >= 256 and \
            (parts * 2 - 1) * 32 * K * 4 <= 120 * 1024:
        parts *= 2
    return parts


def torch_ball_query(p1, p2, K, r2):
    """Dense restatement: (dists, idx) of the first K targets with d < r2, -1 / 0 pads; differentiable in dists."""
    B, P1, _ = p1.shape
    P2 = p2.shape[1]
    chunk = max(1, (1 << 26) // (B * P2))
    ar = torch.arange(P2, device=p1.device).expand(B, min(chunk, P1), P2)
    ds, ix = [], []
    for s in range(0, P1, chunk):
        q = p1[:, s:s + chunk]
        c = q.shape[1]
        d = (q[:, :, None, :] - p2[:, None, :, :]).square().sum(-1)
        inside = d < r2
        rank = inside.cumsum(-1)
        slot = torch.where(inside & (rank <= K), rank - 1, K)
        ix.append(torch.full((B, c, K + 1), -1, device=p1.device, dtype=torch.int64).scatter_(-1, slot, ar[:, :c])[..., :K])
        ds.append(torch.zeros(B, c, K + 1, device=p1.device).scatter(-1, slot, d)[..., :K])
    return torch.cat(ds, 1), torch.cat(ix, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=40)
    args = ap.parse_args()
    _lib.require_cuda()
    L = _lib.lib()
    name, power, mhz = device_line()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lines = [f"device: {name}, power limit {power:.0f} W, max SM clock {mhz:.0f} MHz, {sms} SMs",
             f"library: {os.path.basename(_lib.lib_path())}",
             "shape     B     P1     P2   K     r parts  hits | ours fwd us  bwd us | pcl_ball_query us | torch fwd us  fwd+bwd us | "
             "speed-up vs torch fwd  fwd+bwd | vs pcl_ball_query"]
    A = _lib.pts_args
    for sname, B, P1, P2, K, radius in SHAPES:
        R = 4 if P2 <= 16384 else 2
        clouds = []
        for r in range(R):
            g = torch.Generator(device="cuda").manual_seed(r)
            t = torch.rand(B, P2, 3, device="cuda", generator=g)
            if sname == "sensor":
                x = sample_farthest_points(t, K=P1)[0].contiguous()
            else:
                x = torch.rand(B, P1, 3, device="cuda", generator=g)
            clouds.append((x, t))
        r2 = _radius2(radius)
        r2_pn2 = float(torch.tensor(radius ** 2, dtype=torch.float32))
        dists = torch.empty(B, P1, K, device="cuda"); idx = torch.empty(B, P1, K, device="cuda", dtype=torch.int32)
        gidx = torch.empty(B, P1, K, device="cuda", dtype=torch.int32)
        gd = torch.randn(B, P1, K, device="cuda")
        g1 = torch.empty(B, P1, 3, device="cuda"); g2 = torch.empty(B, P2, 3, device="cuda")
        it = [0]

        def fwd():
            a, b = clouds[it[0] % R]; it[0] += 1
            assert L.pcl_ball_query_fwd(*A(a), None, *A(b), None, B, P1, P2, 3, K, r2, 0, dists.data_ptr(), idx.data_ptr(), None) == 0

        def bwd():
            a, b = clouds[it[0] % R]; it[0] += 1
            assert L.pcl_ball_query_bwd(*A(a), None, *A(b), None, B, P1, P2, 3, K, idx.data_ptr(), gd.data_ptr(), g1.data_ptr(),
                                        g2.data_ptr(), None) == 0

        def pn2():
            a, b = clouds[it[0] % R]; it[0] += 1
            assert L.pcl_ball_query(*A(b), *A(a), B, P2, P1, r2_pn2, K, gidx.data_ptr(), None) == 0

        iters = args.iters if B * P1 * P2 <= 32 * 512 * 2048 else max(5, args.iters // 4)
        tf = timed(fwd, iters)
        hits = float((idx >= 0).float().sum(-1).mean())
        tb, tp = timed(bwd, iters), timed(pn2, iters)

        def t_fwd():
            a, b = clouds[it[0] % R]; it[0] += 1
            return torch_ball_query(a, b, K, r2)

        def t_fwd_bwd():
            a, b = clouds[it[0] % R]; it[0] += 1
            a = a.detach().requires_grad_(); b = b.detach().requires_grad_()
            dv, _ = torch_ball_query(a, b, K, r2)
            dv.backward(gd)

        titers = max(3, iters // 4)
        try:
            ttf, ttb = timed(t_fwd, titers), timed(t_fwd_bwd, titers)
            tstr = f"{ttf:12.1f}  {ttb:10.1f} | {ttf / tf:20.2f}x {ttb / (tf + tb):7.2f}x"
        except torch.OutOfMemoryError:
            tstr = f"{'OOM':>12}  {'OOM':>10} | {'-':>21} {'-':>8}"
        torch.cuda.empty_cache()
        lines.append(f"{sname:<7} {B:3d} {P1:6d} {P2:6d} {K:3d} {radius:5.2f} {parts_for(B, P1, P2, K, sms):5d} {hits:5.1f} | "
                     f"{tf:11.1f} {tb:7.1f} | {tp:17.1f} | {tstr} | {tp / tf:16.2f}x")
        print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
