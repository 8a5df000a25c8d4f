"""Normal-estimation time on the GPU: pcl_knn_fwd, pcl_frames_fwd and pcl_frames_bwd alone through the C ABI with
preallocated outputs, the public estimate_pointcloud_local_coord_frames forward and forward+backward, and the same GPU's
dense torch restatement (cdist -> topk -> gather -> covariance -> fp32 torch.linalg.eigh -> disambiguation, backward through
autograd).

  python tools/normals_time.py [--out FILE] [--iters N]

Each time is the mean over N back-to-back launches (CUDA events around the whole window) on R rotating input copies, after
a warm-up of every shape (tools/knn_time.py's method).  The frames kernels' algorithmic bytes are what they request: the idx
block (4 K bytes per point), the neighbours' coordinates once per pass over them (3 passes forward, 2 backward, 12 bytes
each; the backward also adds 12 bytes per neighbour with red.add), the point itself and the outputs / upstream gradients
(48 bytes per point).  Most of those are re-reads of an L2-resident cloud, so GB/s is a rate from L2, not from HBM."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pointcloud_b200 as pcl  # noqa: E402
from pointcloud_b200 import _lib, synth  # noqa: E402
from tools.knn_time import L2_BYTES, device_line, timed  # noqa: E402

EIGH_CHUNK = 8192
SHAPES = [("table", 32, 2048, 16), ("table", 32, 2048, 50), ("table", 8, 16384, 32), ("table", 1, 65536, 32)]


def torch_frames(x, K):
    """The dense pipeline a user writes without this library, fp32 throughout."""
    b, n, _ = x.shape
    idx = torch.cdist(x, x).topk(K, dim=-1, largest=False).indices
    nb = x.gather(1, idx.reshape(b, n * K, 1).expand(-1, -1, 3)).view(b, n, K, 3)
    d = nb - nb.mean(2, keepdim=True)
    cov = (d.unsqueeze(4) * d.unsqueeze(3)).mean(2)
    # cusolver's batched fp32 syev refuses the whole batch at these sizes (CUSOLVER_STATUS_INVALID_VALUE on a B200 with
    # torch 2.11 / CUDA 12.8 at 65 536 matrices), so the batch goes in chunks of EIGH_CHUNK matrices
    parts = [torch.linalg.eigh(c) for c in cov.view(-1, 3, 3).split(EIGH_CHUNK)]
    lam = torch.cat([q[0] for q in parts]).view(b, n, 3)
    V = torch.cat([q[1] for q in parts]).view(b, n, 3, 3)
    df = nb - x[:, :, None]

    def flip(v):
        n_pos = ((v[:, :, None] * df).sum(3) > 0).sum(2, keepdim=True)
        return torch.where(2 * n_pos < K, -v, v)
    nrm, z = flip(V[..., 0]), flip(V[..., 2])
    return lam, torch.stack((nrm, torch.cross(nrm, z, dim=2), z), dim=3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    _lib.require_cuda()
    L = _lib.lib()
    name, power, mhz = device_line()
    lines = [f"device: {name}, power limit {power:.0f} W, max SM clock {mhz:.0f} MHz",
             f"library: {os.path.basename(_lib.lib_path())}",
             "shape      B      P   K | knn_fwd us  frames_fwd us  GB/s  frames_bwd us  GB/s | public fwd us  fwd+bwd us | "
             "torch fwd us  fwd+bwd us | speed-up fwd  fwd+bwd | inputs"]
    for sname, B, P, K in SHAPES:
        R = 4
        clouds = [synth.table_clouds(B, P, seed=r)[0].cuda() for r in range(R)]
        in_bytes = R * B * P * 3 * 4 + B * P * (K * 8 + 48 * 2)
        resident = "L2-resident" if in_bytes < L2_BYTES else "exceeds L2"
        dists = torch.empty(B, P, K, device="cuda")
        idx = torch.empty(B, P, K, device="cuda", dtype=torch.int32)
        curv, frames = torch.empty(B, P, 3, device="cuda"), torch.empty(B, P, 3, 3, device="cuda")
        gc, gf = torch.randn(B, P, 3, device="cuda"), torch.randn(B, P, 3, 3, device="cuda")
        gp = torch.empty(B, P, 3, device="cuda")
        A = _lib.pts_args
        it = [0]

        def nxt():
            x = clouds[it[0] % R]
            it[0] += 1
            return x

        def knn():
            x = nxt()
            assert L.pcl_knn_fwd(*A(x), None, *A(x), None, B, P, P, 3, K, 0, dists.data_ptr(), idx.data_ptr(), None) == 0

        knn()  # the kernels below read this idx; the inputs rotate, which changes only what they gather
        torch.cuda.synchronize()

        def ffwd():
            assert L.pcl_frames_fwd(*A(nxt()), None, B, P, K, 1, idx.data_ptr(), curv.data_ptr(), frames.data_ptr(), None) == 0

        def fbwd():
            assert L.pcl_frames_bwd(*A(nxt()), None, B, P, K, idx.data_ptr(), curv.data_ptr(), frames.data_ptr(), gc.data_ptr(),
                                    gf.data_ptr(), gp.data_ptr(), None) == 0

        def pub_fwd():
            return pcl.estimate_pointcloud_local_coord_frames(nxt(), K)

        def pub_fwd_bwd():
            x = nxt().detach().requires_grad_()
            c, f = pcl.estimate_pointcloud_local_coord_frames(x, K)
            ((c * gc).sum() + (f * gf).sum()).backward()

        big = B * P * P > 32 * 2048 * 2048
        iters = max(5, args.iters // 10 if big else args.iters)
        tk, tf, tb = timed(knn, iters), timed(ffwd, iters), timed(fbwd, iters)
        tpf, tpb = timed(pub_fwd, iters), timed(pub_fwd_bwd, iters)
        bytes_f = B * P * (4 * K + 3 * 12 * K + 12 + 48)
        bytes_b = B * P * (4 * K + 2 * 12 * K + 12 * K + 96)

        def t_fwd():
            return torch_frames(nxt(), K)

        def t_fwd_bwd():
            x = nxt().detach().requires_grad_()
            c, f = torch_frames(x, K)
            ((c * gc).sum() + (f * gf).sum()).backward()

        titers = max(3, iters // 5)
        try:
            ttf, ttb = timed(t_fwd, titers), timed(t_fwd_bwd, titers)
            tstr = f"{ttf:12.1f}  {ttb:10.1f} | {ttf / tpf:11.2f}x {ttb / tpb:7.2f}x"
        except torch.OutOfMemoryError:
            tstr = f"{'OOM':>12}  {'OOM':>10} | {'-':>12} {'-':>8}"
        except RuntimeError as e:  # recorded, not hidden: the line says the baseline did not run
            tstr = f"{'failed':>12}  {'failed':>10} | {'-':>12} {'-':>8} ({type(e).__name__}: {str(e)[:60]})"
        torch.cuda.empty_cache()
        lines.append(f"{sname:<6} {B:5d} {P:6d} {K:3d} | {tk:10.1f} {tf:14.1f} {bytes_f / tf / 1e3:5.0f} {tb:14.1f} "
                     f"{bytes_b / tb / 1e3:5.0f} | {tpf:13.1f} {tpb:11.1f} | {tstr} | "
                     f"{R} rotating copies, {in_bytes / 2**20:.1f} MB with idx and outputs, {resident}")
        print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
