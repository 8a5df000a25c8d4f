"""EMD approximation module (auction algorithm) -- B200 drop-in for
pointcloud_vision/loss/emd/emd_module.py (same names, arguments, outputs and gradient behaviour).

Input:  xyz1, xyz2: [#batch, #points, 3]; xyz1 is the predicted cloud, xyz2 the ground truth.  Any finite
        coordinates give the oracle's results bit for bit as long as pairwise distances stay below 1e9 (the
        reference's initial bid value is -1e9); [0, 1] (emd_module.py:6-9) is only the range for which the
        reference tuned eps.  Any CUDA float dtype / strided view is accepted without a copy (the reference copies
        with .contiguous().float().cuda(), :43-44).
Output: dist [#batch, #points] (squared distance to the match, fp32), assignment [#batch, #points]
        (int32 index into xyz2; not guaranteed to be a bijection, :16-19).
Only xyz1 receives a gradient; xyz2 gets zeros; eps / iters get None (:63-72).
The reference's limits (#points % 1024 == 0, #batch <= 512, :40-41) are accepted but not required;
#points <= pcl_emd_max_points().
"""
import torch
from torch import nn
from torch.autograd import Function

from . import _lib


_WS_BYTES = {}  # (B, N) -> pcl_emd_workspace_bytes: a pure function of the sizes (and the device's SM count), asked once


def emd_workspace(b, n, dev):
    """A workspace for one pcl_emd_* call (torch's caching allocator hands the same block back call after call)."""
    wsb = _WS_BYTES.get((b, n))
    if wsb is None:
        wsb = _WS_BYTES[(b, n)] = _lib.lib().pcl_emd_workspace_bytes(b, n)
    return torch.empty(wsb, device=dev, dtype=torch.uint8), wsb


EMD_PATHS = {"auto": 0, "cluster": 1, "team": 2, "tickets": 3}  # include/pcl.h PCL_EMD_PATH_*


def set_emd_path(path="auto"):
    """Which auction kernel the calls that follow use (process-wide; include/pcl.h pcl_emd_set_path): "auto", "cluster" (one
    thread-block cluster per cloud), "team" (owner CTA per cloud + workers) or "tickets" (cluster kernel whose heavy iterations
    are shared with worker CTAs).  All of them return bit-identical results; the choice is a tuning knob."""
    _lib.check(_lib.lib().pcl_emd_set_path(EMD_PATHS[path] if isinstance(path, str) else int(path)), "pcl_emd_set_path")


def emd_forward_raw(xyz1, xyz2, eps, iters, want_stats=False, want_epilogue=False):
    """One pcl_emd_fwd(_fused) call.  Returns (dist, assignment, stats|None); stats int32 (B,8) =
    [sum_t U_t, iterations run, extra GetMax qualifiers, cluster size, executed evals lo, hi, flags, tiles].
    want_epilogue=True: returns (dist, assignment, stats, unit_grad, sums) with the fused loss epilogue of the same kernel --
    unit_grad (B,N,3) = d(sum sqrt(dist)) / d xyz1 and sums (3,) = [sum sqrt(dist), B*N, mean] (include/pcl.h)."""
    _lib.require_cuda()
    L = _lib.lib()
    xyz1, xyz2 = _lib.as_points(xyz1), _lib.as_points(xyz2)
    b, n, c1 = xyz1.shape
    assert xyz2.shape[0] == b and xyz2.shape[1] == n and c1 >= 3 and xyz2.shape[2] >= 3
    dev = xyz1.device
    with _lib.on_device(dev):
        dist = torch.empty(b, n, device=dev, dtype=torch.float32)
        assignment = torch.empty(b, n, device=dev, dtype=torch.int32)
        stats = torch.empty(b, 8, device=dev, dtype=torch.int32) if want_stats else None
        ws, wsb = emd_workspace(b, n, dev)
        if want_epilogue:
            unit_grad = torch.empty(b, n, 3, device=dev, dtype=torch.float32)
            sums = torch.empty(3, device=dev, dtype=torch.float32)
            rc = L.pcl_emd_fwd_fused(*_lib.pts_args(xyz1), *_lib.pts_args(xyz2), b, n, float(eps), int(iters),
                                     dist.data_ptr(), assignment.data_ptr(), _lib.ptr(stats), 1.0, unit_grad.data_ptr(), sums.data_ptr(),
                                     ws.data_ptr(), wsb, _lib.stream_ptr(dev))
            _lib.check(rc, "pcl_emd_fwd_fused")
            return dist, assignment, stats, unit_grad, sums
        rc = L.pcl_emd_fwd(*_lib.pts_args(xyz1), *_lib.pts_args(xyz2), b, n, float(eps), int(iters),
                           dist.data_ptr(), assignment.data_ptr(), _lib.ptr(stats), ws.data_ptr(), wsb, _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_emd_fwd")
    return dist, assignment, stats


class emdFunction(Function):
    @staticmethod
    def forward(ctx, xyz1, xyz2, eps, iters):
        batchsize, n, _ = xyz1.size()
        _, m, _ = xyz2.size()
        assert (n == m)                                   # emd_module.py:38
        assert (xyz1.size()[0] == xyz2.size()[0])         # :39
        ctx.in_meta = (xyz1.dtype, xyz1.device, xyz2.dtype, xyz2.device)
        xyz1, xyz2 = _lib.as_points(xyz1), _lib.as_points(xyz2)
        dist, assignment, _ = emd_forward_raw(xyz1, xyz2, eps, iters)
        ctx.save_for_backward(xyz1, xyz2, assignment)
        ctx.mark_non_differentiable(assignment)
        return dist, assignment

    @staticmethod
    def backward(ctx, graddist, gradidx):
        xyz1, xyz2, assignment = ctx.saved_tensors
        L = _lib.lib()
        b, n, _ = xyz1.shape
        graddist = graddist.contiguous().float()
        with _lib.on_device(xyz1.device):
            gradxyz1 = torch.empty(b, n, 3, device=xyz1.device, dtype=torch.float32)
            rc = L.pcl_emd_bwd(*_lib.pts_args(xyz1), *_lib.pts_args(xyz2), b, n, assignment.data_ptr(),
                               graddist.data_ptr(), gradxyz1.data_ptr(), _lib.stream_ptr(xyz1.device))
            _lib.check(rc, "pcl_emd_bwd")
        if xyz1.shape[2] != 3:  # caller passed more channels than xyz: only xyz receives gradient
            full = torch.zeros(xyz1.shape, device=xyz1.device, dtype=torch.float32)
            full[:, :, :3] = gradxyz1
            gradxyz1 = full
        dt1, dev1, dt2, dev2 = ctx.in_meta
        gradxyz1 = gradxyz1.to(device=dev1, dtype=dt1)
        gradxyz2 = torch.zeros(xyz2.shape, device=dev2, dtype=dt2) if ctx.needs_input_grad[1] else None  # emd_module.py:69,72
        return gradxyz1, gradxyz2, None, None


class emdModule(nn.Module):
    def __init__(self):
        super(emdModule, self).__init__()

    def forward(self, input1, input2, eps, iters):
        return emdFunction.apply(input1, input2, eps, iters)
