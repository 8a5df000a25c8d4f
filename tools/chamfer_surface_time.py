"""chamfer_distance with normals, weights and per-cloud results on the GPU: end-to-end time of the public call, the kernels
alone through the C ABI, the dense torch restatement on the same GPU, and the default path of this library against another
build of it (e.g. the parent commit's), alternated in one process.

  python tools/chamfer_surface_time.py [--out FILE] [--iters N] [--other-lib PATH]

Each time is the mean over N back-to-back calls (CUDA events around the whole window) after a warm-up of every shape.  The
normal kernel's time is the difference between pcl_chamfer_cloud_fwd with and without normals; its algorithmic bytes are, per
valid query, its own normal, its index and the neighbour's normal (12 + 4 + 12 bytes, fp32) and the share is of the HGX B200
data-sheet HBM bandwidth (7.7 TB/s).  The (B, N, 6) clouds the normals are read from (<= 50 MB here) fit the 126 MB L2, so
this is not an HBM measurement."""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pointcloud_b200 as pcl  # noqa: E402
from pointcloud_b200 import _lib  # noqa: E402

SHAPES = [(32, 2048), (64, 8192), (64, 16384)]
HBM = 7.7e12


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


def dense_torch(x, y, xn, yn, w):
    """cdist -> argmin -> gather -> cosine, autograd (full clouds, batch_reduction None)."""
    d2 = torch.cdist(x, y) ** 2
    ix, iy = d2.argmin(2), d2.argmin(1)
    gy = y.gather(1, ix[..., None].expand(-1, -1, 3)); gx = x.gather(1, iy[..., None].expand(-1, -1, 3))
    cx = ((x - gy) ** 2).sum(2).mean(1); cy = ((y - gx) ** 2).sum(2).mean(1)
    nx = yn.gather(1, ix[..., None].expand(-1, -1, 3)); ny = xn.gather(1, iy[..., None].expand(-1, -1, 3))
    tx = (1 - torch.nn.functional.cosine_similarity(xn, nx, dim=2, eps=1e-6).abs()).mean(1)
    ty = (1 - torch.nn.functional.cosine_similarity(yn, ny, dim=2, eps=1e-6).abs()).mean(1)
    return (cx + cy) * w, (tx + ty) * w


def bind(path):
    L = ctypes.CDLL(path)
    for name in ("pcl_chamfer_workspace_bytes", "pcl_chamfer_fwd", "pcl_chamfer_bwd"):
        res, args = _lib._SIGNATURES[name]
        getattr(L, name).restype, getattr(L, name).argtypes = res, args
    return L


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--other-lib", help="another build of libpcl_b200.so whose default path is timed against this one")
    a = ap.parse_args()
    name, power, mhz = device_line()
    lines = [f"# {name}, power limit {power:.0f} W, max SM clock {mhz:.0f} MHz; mean of {a.iters} calls after warm-up (CUDA events)"]
    L = _lib.lib()
    A = _lib.pts_args
    for b, n in SHAPES:
        g = torch.Generator(device="cuda").manual_seed(b + n)
        cx, cy = torch.rand(b, n, 6, device="cuda", generator=g), torch.rand(b, n, 6, device="cuda", generator=g) - 0.5
        x, y = cx[..., :3].contiguous(), cy[..., :3].contiguous()
        xn, yn = cx[..., 3:6], cy[..., 3:6]
        w = torch.rand(b, device="cuda", generator=g) + 0.5
        xg, yg = x.clone().requires_grad_(), y.clone().requires_grad_()
        cxg, cyg = cx.clone().requires_grad_(), cy.clone().requires_grad_()
        variants = {
            "default": lambda: pcl.chamfer_distance(xg, yg),
            "normals": lambda: pcl.chamfer_distance(xg, yg, x_normals=cxg[..., 3:6], y_normals=cyg[..., 3:6]),
            "weights, batch_reduction=None": lambda: pcl.chamfer_distance(xg, yg, weights=w, batch_reduction=None),
        }
        if 4 * b * n * n * 4 < 80e9:
            variants["dense torch (cdist)"] = lambda: dense_torch(xg, yg, cxg[..., 3:6], cyg[..., 3:6], w)
        lines.append(f"\nB={b} N={n}")
        for vname, fn in variants.items():
            with torch.no_grad():
                tf = timed(fn, a.iters)

            def fb():
                l, ln = fn()
                (l.sum() + (ln.sum() if ln is not None else 0)).backward()
            tfb = timed(fb, a.iters)
            lines.append(f"  chamfer_distance {vname:32s} fwd {tf:9.1f} us   fwd+bwd {tfb:9.1f} us")
        # the kernels alone through the C ABI
        e = lambda *s, dt=torch.float32: torch.empty(*s, device="cuda", dtype=dt)
        dx, dy, ix, iy, l4 = e(b, n), e(b, n), e(b, n, dt=torch.int32), e(b, n, dt=torch.int32), e(4)
        sums, nsums, gc, gn = e(2, b), e(2, b), torch.ones(2, b, device="cuda"), torch.ones(2, b, device="cuda")
        gx, gy, gxn, gyn, g2 = e(b, n, 3), e(b, n, 3), e(b, n, 3), e(b, n, 3), torch.ones(2, device="cuda")
        wsb = L.pcl_chamfer_workspace_bytes(b, n, n)
        ws = e(wsb, dt=torch.uint8)
        nul = [None, 0, 0, 0]
        fwd = lambda: L.pcl_chamfer_fwd(*A(x), None, *A(y), None, b, n, n, 3, 0, dx.data_ptr(), ix.data_ptr(), dy.data_ptr(), iy.data_ptr(),
                                        l4.data_ptr(), ws.data_ptr(), wsb, None)
        cfwd = lambda nrm: L.pcl_chamfer_cloud_fwd(*A(x), None, *A(y), None, b, n, n, 3, 0, dx.data_ptr(), ix.data_ptr(), dy.data_ptr(),
                                                   iy.data_ptr(), l4.data_ptr(), sums.data_ptr(), *(A(xn) + A(yn) if nrm else nul + nul),
                                                   nsums.data_ptr() if nrm else None, ws.data_ptr(), wsb, None)
        bwd = lambda: L.pcl_chamfer_bwd(*A(x), None, *A(y), None, b, n, n, 3, ix.data_ptr(), iy.data_ptr(), g2.data_ptr(), gx.data_ptr(),
                                        gy.data_ptr(), None)
        cbwd = lambda: L.pcl_chamfer_cloud_bwd(*A(x), None, *A(y), None, b, n, n, 3, ix.data_ptr(), iy.data_ptr(), gc.data_ptr(), gx.data_ptr(),
                                               gy.data_ptr(), *A(xn), *A(yn), gn.data_ptr(), gxn.data_ptr(), gyn.data_ptr(), None)
        t_f, t_c, t_cn = timed(fwd, a.iters), timed(lambda: cfwd(False), a.iters), timed(lambda: cfwd(True), a.iters)
        t_b, t_cb = timed(bwd, a.iters), timed(cbwd, a.iters)
        t_nk = t_cn - t_c
        nbytes = 2 * b * n * 28
        lines.append(f"  kernels: pcl_chamfer_fwd {t_f:.1f} us, cloud_fwd {t_c:.1f} us, cloud_fwd + normals {t_cn:.1f} us "
                     f"-> normal kernel (+ ticket memset) {t_nk:.1f} us, {nbytes / 1e6:.1f} MB algorithmic, "
                     f"{nbytes / max(t_nk, 1e-3) / 1e3:.0f} GB/s = {nbytes / max(t_nk, 1e-3) * 1e6 / HBM * 100:.0f} % of 7.7 TB/s")
        lines.append(f"  kernels: pcl_chamfer_bwd {t_b:.1f} us, cloud_bwd with normals {t_cb:.1f} us")
        if a.other_lib:
            O = bind(a.other_lib)
            ofwd = lambda: O.pcl_chamfer_fwd(*A(x), None, *A(y), None, b, n, n, 3, 0, dx.data_ptr(), ix.data_ptr(), dy.data_ptr(), iy.data_ptr(),
                                             l4.data_ptr(), ws.data_ptr(), wsb, None)
            obwd = lambda: O.pcl_chamfer_bwd(*A(x), None, *A(y), None, b, n, n, 3, ix.data_ptr(), iy.data_ptr(), g2.data_ptr(), gx.data_ptr(),
                                             gy.data_ptr(), None)
            mine, other = [], []
            for _ in range(5):  # alternated
                other.append(timed(lambda: (ofwd(), obwd()), a.iters))
                mine.append(timed(lambda: (fwd(), bwd()), a.iters))
            lines.append(f"  default path pcl_chamfer_fwd + pcl_chamfer_bwd, 5 alternated rounds: other build "
                         f"{statistics.median(other):.1f} us (range {min(other):.1f}-{max(other):.1f}), this build "
                         f"{statistics.median(mine):.1f} us (range {min(mine):.1f}-{max(mine):.1f})")
        print("\n".join(lines[-8:]), flush=True)
    text = "\n".join(lines) + "\n"
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text)
    print(text)


if __name__ == "__main__":
    main()
