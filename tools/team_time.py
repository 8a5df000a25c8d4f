"""Development aid: time the auction on the bench regimes through one path (pcl_emd_set_path; default 2 = team); prints checksums.

  python tools/team_time.py [TAG] [B] [PATH]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import pointcloud_b200 as pcl
from pointcloud_b200 import _lib, synth

tag = sys.argv[1] if len(sys.argv) > 1 else ""
b = int(sys.argv[2]) if len(sys.argv) > 2 else 32
path = int(sys.argv[3]) if len(sys.argv) > 3 else 2
_lib.lib().pcl_emd_set_path(path)
n = 2048
out = []
for kind in ("table", "noisy", "uniform"):
    if kind == "uniform":
        x1, x2 = synth.uniform_clouds(b, n, seed=0)
    else:
        x1, t = synth.table_clouds(b, n, seed=0, regime="independent" if kind == "table" else "noisy")
        x2 = t[:, :, :3].contiguous()
    x1, x2 = x1.cuda(), x2.cuda()
    for _ in range(3):
        d, a, st = pcl.emd_forward_raw(x1, x2, 0.005, 50, want_stats=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        pcl.emd_forward_raw(x1, x2, 0.005, 50)
    e1.record()
    torch.cuda.synchronize()
    chk = (a.long() * torch.arange(1, n + 1, device="cuda")).sum().item() % 1000003
    out.append(f"{kind} {e0.elapsed_time(e1) / 20 * 1e3:7.1f} us chk={chk}")
print(f"[{tag}] B={b} " + " | ".join(out), flush=True)
