"""Development aid: Chamfer forward time over N (B = 32 and 64) with the pruned path taken from MIN_POINTS points per cloud on
(pcl_chamfer_set_prune_min: 1 = always, 0 = never, -1 = the library's default of 6144).  Running it with 1 and with 0 shows where
the pruned scan overtakes the brute-force kernel, which is how the default was chosen.

  python tools/chamfer_prune_time.py MIN_POINTS"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pointcloud_b200 as pcl
from pointcloud_b200 import _lib, synth
L = _lib.lib()
prune_min = int(sys.argv[1])
L.pcl_chamfer_set_prune_min(prune_min)
tag = f"prune_min={prune_min}"
for b in (32, 64):
    row = []
    for n in (1024, 2048, 4096, 8192, 16384):
        for kind in ("table", "uniform"):
            if kind == "uniform":
                x1, x2 = synth.uniform_clouds(b, n, seed=0)
            else:
                x1, t = synth.table_clouds(b, n, seed=0); x2 = t[:, :, :3].contiguous()
            x1, x2 = x1.cuda(), x2.cuda()
            e = lambda *s, dt=torch.float32: torch.empty(*s, device="cuda", dtype=dt)
            dx, dy, ix, iy, lxy = e(b, n), e(b, n), e(b, n, dt=torch.int32), e(b, n, dt=torch.int32), e(4)
            wsb = L.pcl_chamfer_workspace_bytes(b, n, n); ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
            A = _lib.pts_args
            def fwd():
                rc = L.pcl_chamfer_fwd(*A(x1), None, *A(x2), None, b, n, n, 3, 0, dx.data_ptr(), ix.data_ptr(), dy.data_ptr(), iy.data_ptr(), lxy.data_ptr(), ws.data_ptr(), wsb, None)
                assert rc == 0
            for _ in range(3): fwd()
            torch.cuda.synchronize(); a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            it = 20 if n <= 4096 else 5
            a.record()
            for _ in range(it): fwd()
            c.record(); torch.cuda.synchronize()
            row.append(f"N={n} {kind[:3]} {a.elapsed_time(c) / it * 1e3:8.1f} us")
    print(f"[{tag}] B={b}: " + " | ".join(row), flush=True)
