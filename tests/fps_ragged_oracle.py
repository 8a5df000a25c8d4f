"""Ragged farthest point sampling restated on top of the FPS oracle (oracle/fps_oracle.c): cloud b is sampled on its
first n_b points with min(k_b, n_b) samples and the start index clamped to [0, n_b - 1]; the remaining slots are -1
(include/pcl.h, pcl_fps_ragged)."""
import numpy as np

import oracle


def fps_ragged(x, npoint, lengths=None, K=None, start=None, skip_origin=False):
    """x (B, N, 3+) float array or tensor; lengths, K, start: None or B integers.  Returns int32 (B, npoint)."""
    if hasattr(x, "detach"):
        x = x.detach().cpu().float().numpy()
    x = np.asarray(x, dtype=np.float32)
    b, n, _ = x.shape
    out = np.full((b, npoint), -1, np.int32)
    for i in range(b):
        nb = n if lengths is None else int(min(max(int(lengths[i]), 0), n))
        kb = npoint if K is None else int(min(max(int(K[i]), 0), npoint))
        s = min(nb, kb)
        if s == 0:
            continue
        st = 0 if start is None else min(max(int(start[i]), 0), nb - 1)
        out[i, :s] = oracle.fps(x[i:i + 1, :nb], s, start=[st], skip_origin=skip_origin)[0]
    return out
