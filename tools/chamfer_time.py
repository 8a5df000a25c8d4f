"""Development aid: Chamfer forward / backward kernel time through the C ABI with preallocated outputs."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pointcloud_b200 as pcl
from pointcloud_b200 import _lib, synth
L = _lib.lib()
b, n = 32, int(os.environ.get("N", 2048))
x1, t = synth.table_clouds(b, n, seed=0); x1, x2 = x1.cuda(), t[:, :, :3].contiguous().cuda()
e = lambda *s, dt=torch.float32: torch.empty(*s, device="cuda", dtype=dt)
dx, dy, ix, iy, lxy = e(b, n), e(b, n), e(b, n, dt=torch.int32), e(b, n, dt=torch.int32), e(2)
gx, gy, ones = e(b, n, 3), e(b, n, 3), torch.ones(2, device="cuda")
wsb = L.pcl_chamfer_workspace_bytes(b, n, n); ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
A = _lib.pts_args
def fwd(mode):
    rc = L.pcl_chamfer_fwd(*A(x1), None, *A(x2), None, b, n, n, 3, mode, dx.data_ptr(), ix.data_ptr(), dy.data_ptr(), iy.data_ptr(), lxy.data_ptr(), ws.data_ptr(), wsb, None)
    assert rc == 0
def bwd():
    rc = L.pcl_chamfer_bwd(*A(x1), None, *A(x2), None, b, n, n, 3, ix.data_ptr(), iy.data_ptr(), ones.data_ptr(), gx.data_ptr(), gy.data_ptr(), None)
    assert rc == 0
def timeit(fn, iters=200):
    for _ in range(10): fn()
    torch.cuda.synchronize(); a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters): fn()
    c.record(); torch.cuda.synchronize(); return a.elapsed_time(c) / iters * 1e3
print(f"N={n}: fwd unfused {timeit(lambda: fwd(0)):.1f} us, fwd fma {timeit(lambda: fwd(1)):.1f} us, bwd {timeit(bwd):.1f} us")
