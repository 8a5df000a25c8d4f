"""Points alignment and ICP -- B200 drop-in for `pytorch3d.ops.corresponding_points_alignment` /
`iterative_closest_point`.

The call surface is pytorch3d 0.7.2's as recalled ([3P-memory]; parity with pytorch3d itself is unpinned).  Semantics
(include/pcl.h, "points alignment and ICP"): row vectors, apply(X; R, T, s) = s * (X @ R) + T; the alignment is the weighted
Umeyama / Procrustes fit with pytorch3d's quirk of weighting both centred clouds (so the covariance carries w^2); ICP aligns
the ORIGINAL X to the K=1 nearest neighbours of the current Xt in Y, and stops when every cloud's relative rmse is at most
the threshold in the same iteration.

Differences from pytorch3d: ragged batches take `lengths=` / `x_lengths=` / `y_lengths=` instead of `Pointclouds` objects;
the arithmetic is fp64 (moments, one-sided Jacobi SVD) rounded to fp32 once; the warning pytorch3d issues on ambiguous
rotations is dropped (it needs a host read); the alignment's gradient uses the closed form of the polar factor, which is
finite for repeated singular values, where torch.svd's is not.  Inputs are fp32 / fp16 / bf16 (strided views read in
place); outputs are fp32.
"""
from collections import namedtuple

import torch
from torch.autograd import Function

from . import _lib, cfg
from .chamfer import _MODES

SimilarityTransform = namedtuple("SimilarityTransform", "R T s")
ICPSolution = namedtuple("ICPSolution", "converged rmse Xt RTs t_history")

_ALIGN_RECORD = 40  # PCL_ALIGN_RECORD
_ALIGN_MSG = "Point sets X and Y have to have the same number of batches, points and dimensions."  # pytorch3d's messages
_ICP_MSG = "Point sets X and Y have to have the same number of batches and data dimensions."
_INIT_MSG = ("The initial transformation init_transform has to be a named tuple SimilarityTransform with elements (R, T, s). "
             "R are dim x dim orthonormal matrices of shape (minibatch, dim, dim), T is a batch of dim-dimensional translations "
             "of shape (minibatch, dim) and s is a batch of scalars of shape (minibatch,).")


def _check_d3(d):
    if d != 3:
        raise ValueError(f"point dimension D={d} is not supported (3 only)")


def _lengths(lengths, b, dev, name):
    if lengths is None:
        return None
    if lengths.shape != (b,):
        raise ValueError(f"Expected {name} to be of shape (N,).")
    return lengths.to(device=dev, dtype=torch.int64).contiguous()


def points_alignment_forward_raw(X, Y, weights=None, estimate_scale=False, allow_reflection=False, eps=1e-9, lengths=None):
    """One pcl_points_alignment_fwd call.  Returns dict(R (B,3,3), T (B,3), s (B) fp32, record (B, 40) fp64, and the kernels'
    views of X, Y, weights (fp32) and lengths)."""
    if X.dim() != 3 or Y.dim() != 3 or X.shape != Y.shape:
        raise ValueError(_ALIGN_MSG)
    _check_d3(X.shape[2])
    if weights is not None and tuple(weights.shape) != tuple(X.shape[:2]):
        raise ValueError("weights should have the same first two dimensions as X.")
    _lib.require_cuda()
    L = _lib.lib()
    X = _lib.as_points(X)
    Y = _lib.as_points(Y).to(X.device)
    b, p, _ = X.shape
    dev = X.device
    ln = _lengths(lengths, b, dev, "lengths")
    w = None if weights is None else weights.to(device=dev, dtype=torch.float32).contiguous()
    with _lib.on_device(dev):
        R = torch.empty(b, 3, 3, device=dev, dtype=torch.float32)
        T = torch.empty(b, 3, device=dev, dtype=torch.float32)
        s = torch.empty(b, device=dev, dtype=torch.float32)
        rec = torch.empty(b, _ALIGN_RECORD, device=dev, dtype=torch.float64)
        nws = int(L.pcl_points_alignment_workspace_bytes(b, p))
        ws = torch.empty(max(nws, 1), device=dev, dtype=torch.uint8)
        rc = L.pcl_points_alignment_fwd(*_lib.pts_args(X), *_lib.pts_args(Y), _lib.ptr(ln), _lib.ptr(w), b, p,
                                        int(bool(estimate_scale)), int(bool(allow_reflection)), float(eps), R.data_ptr(),
                                        T.data_ptr(), s.data_ptr(), rec.data_ptr(), ws.data_ptr(), nws, _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_points_alignment_fwd")
    return dict(R=R, T=T, s=s, record=rec, X=X, Y=Y, weights=w, lengths=ln)


class _AlignFunction(Function):
    @staticmethod
    def forward(ctx, X, Y, weights, lengths, estimate_scale, allow_reflection, eps):
        ctx.in_meta = (X.dtype, X.device, Y.dtype, Y.device, None if weights is None else (weights.dtype, weights.device))
        ctx.set_materialize_grads(False)
        r = points_alignment_forward_raw(X, Y, weights, estimate_scale, allow_reflection, eps, lengths)
        ctx.save_for_backward(r["X"], r["Y"], r["record"], r["weights"], r["lengths"])  # weights: the caller's tensor if fp32
        ctx.est, ctx.eps = bool(estimate_scale), float(eps)
        if not estimate_scale:
            ctx.mark_non_differentiable(r["s"])
        return r["R"], r["T"], r["s"]

    @staticmethod
    def backward(ctx, gR, gT, gs):
        X, Y, rec, w, ln = ctx.saved_tensors
        b, p, _ = X.shape
        dev = X.device

        def f32(g):
            return None if g is None else g.to(device=dev, dtype=torch.float32).contiguous()
        gR, gT, gs = f32(gR), f32(gT), f32(gs)
        want_w = w is not None and ctx.needs_input_grad[2]
        L = _lib.lib()
        with _lib.on_device(dev):
            gx = torch.empty(b, p, 3, device=dev, dtype=torch.float32)
            gy = torch.empty(b, p, 3, device=dev, dtype=torch.float32)
            gw = torch.empty(b, p, device=dev, dtype=torch.float32) if want_w else None
            rc = L.pcl_points_alignment_bwd(*_lib.pts_args(X), *_lib.pts_args(Y), _lib.ptr(ln), _lib.ptr(w), b, p,
                                            int(ctx.est), ctx.eps, rec.data_ptr(), _lib.ptr(gR), _lib.ptr(gT), _lib.ptr(gs),
                                            gx.data_ptr(), gy.data_ptr(), _lib.ptr(gw), _lib.stream_ptr(dev))
            _lib.check(rc, "pcl_points_alignment_bwd")
        dx, devx, dy, devy, wm = ctx.in_meta
        gwo = None if gw is None else gw.to(device=wm[1], dtype=wm[0])
        return gx.to(device=devx, dtype=dx), gy.to(device=devy, dtype=dy), gwo, None, None, None, None


def corresponding_points_alignment(X, Y, weights=None, estimate_scale=False, allow_reflection=False, eps=1e-9, *,
                                   lengths=None):
    """pytorch3d.ops.corresponding_points_alignment [3P-memory] for (N, P, 3) tensors X and Y of corresponding points
    (fp32 / fp16 / bf16, strided views read in place), optional weights (N, P) and optional int64 `lengths` (N,) shared by
    X and Y.  Returns SimilarityTransform(R (N,3,3), T (N,3), s (N,)), fp32, such that s * (X @ R) + T best matches Y in the
    weighted least-squares sense.  Differentiable with respect to X, Y and weights (closed form of the polar factor; finite
    for repeated singular values, non-finite only where two signed singular values sum to 0).  Nothing here synchronises
    with the host; pytorch3d's warning on ambiguous rotations is not issued."""
    R, T, s = _AlignFunction.apply(X, Y, weights, lengths, bool(estimate_scale), bool(allow_reflection), float(eps))
    return SimilarityTransform(R, T, s)


def _init_args(init_transform, b, dev):
    if init_transform is None:
        return None
    try:
        R, T, s = init_transform
    except (TypeError, ValueError):
        raise ValueError(_INIT_MSG) from None
    if tuple(R.shape) != (b, 3, 3) or tuple(T.shape) != (b, 3) or tuple(s.shape) != (b,):
        raise ValueError(_INIT_MSG)
    return [t.detach().to(device=dev, dtype=torch.float32).contiguous() for t in (R, T, s)]


def icp_forward_raw(X, Y, init_transform=None, max_iterations=100, relative_rmse_thr=1e-6, estimate_scale=False,
                    allow_reflection=False, x_lengths=None, y_lengths=None, mode=None):
    """One pcl_icp call, without any host synchronisation (CUDA-graph capturable).  Returns dict(Xt (B,P1,3),
    R (max_iterations,B,3,3), T (max_iterations,B,3), s (max_iterations,B), rmse (max_iterations,B) -- slots past the
    iterations run are 0 -- status int32 (2,) = {iterations run, converged}, all fp32 on the device)."""
    if X.dim() != 3 or Y.dim() != 3 or X.shape[0] != Y.shape[0] or X.shape[2] != Y.shape[2]:
        raise ValueError(_ICP_MSG)
    _check_d3(X.shape[2])
    if isinstance(max_iterations, bool) or int(max_iterations) != max_iterations or max_iterations < 0:
        raise ValueError(f"max_iterations={max_iterations} must be a non-negative integer")
    it = int(max_iterations)
    _lib.require_cuda()
    L = _lib.lib()
    X = _lib.as_points(X.detach())
    Y = _lib.as_points(Y.detach()).to(X.device)
    b, p1, _ = X.shape
    p2 = Y.shape[1]
    dev = X.device
    l1, l2 = _lengths(x_lengths, b, dev, "x_lengths"), _lengths(y_lengths, b, dev, "y_lengths")
    init = _init_args(init_transform, b, dev)
    mode = _MODES[cfg.chamfer_mode if mode is None else mode]
    with _lib.on_device(dev):
        Xt = torch.empty(b, p1, 3, device=dev, dtype=torch.float32)
        R = torch.empty(it, b, 3, 3, device=dev, dtype=torch.float32)
        T = torch.empty(it, b, 3, device=dev, dtype=torch.float32)
        s = torch.empty(it, b, device=dev, dtype=torch.float32)
        rmse = torch.empty(it, b, device=dev, dtype=torch.float32)
        status = torch.zeros(2, device=dev, dtype=torch.int32) if b == 0 else torch.empty(2, device=dev, dtype=torch.int32)
        nws = int(L.pcl_icp_workspace_bytes(b, p1, p2, it))
        ws = torch.empty(max(nws, 1), device=dev, dtype=torch.uint8)
        ip = [None] * 3 if init is None else [t.data_ptr() for t in init]
        rc = L.pcl_icp(*_lib.pts_args(X), _lib.ptr(l1), *_lib.pts_args(Y), _lib.ptr(l2), b, p1, p2, *ip, it,
                       float(relative_rmse_thr), int(bool(estimate_scale)), int(bool(allow_reflection)), mode, Xt.data_ptr(),
                       R.data_ptr(), T.data_ptr(), s.data_ptr(), rmse.data_ptr(), status.data_ptr(), ws.data_ptr(), nws,
                       _lib.stream_ptr(dev))
        _lib.check(rc, "pcl_icp")
    return dict(Xt=Xt, R=R, T=T, s=s, rmse=rmse, status=status, init=init)


def iterative_closest_point(X, Y, init_transform=None, max_iterations=100, relative_rmse_thr=1e-6, estimate_scale=False,
                            allow_reflection=False, verbose=False, *, x_lengths=None, y_lengths=None):
    """pytorch3d.ops.iterative_closest_point [3P-memory] for (N, P1, 3) X and (N, P2, 3) Y tensors (fp32 / fp16 / bf16,
    strided views read in place) with optional int64 `x_lengths` / `y_lengths` (N,).  Returns
    ICPSolution(converged: bool, rmse (N,) or None, Xt (N,P1,3), RTs: SimilarityTransform, t_history: list of them).

    The loop runs on the device in one launch and reads its status once at the end (one host synchronisation per call).
    As in pytorch3d, the batch stops only when EVERY cloud's relative rmse is <= relative_rmse_thr in the same iteration,
    so a cloud's result depends on the rest of its batch, and an rmse of exactly 0 twice in a row (an empty X cloud, an
    exact noise-free pair) gives 0/0 = NaN and never converges.  `init_transform` only seeds the first search: every
    iteration aligns the original X.  Rows of Xt past x_lengths are transformed too.

    ICP is not differentiable: its outputs are detached.  For gradients, apply corresponding_points_alignment to the final
    correspondences, e.g. knn_gather(Y, knn_points(Xt, Y, x_lengths, y_lengths).idx, y_lengths)[:, :, 0]."""
    r = icp_forward_raw(X, Y, init_transform, max_iterations, relative_rmse_thr, estimate_scale, allow_reflection, x_lengths,
                        y_lengths)
    b = r["Xt"].shape[0]
    if b == 0:
        iters, converged = min(int(max_iterations), 1), int(max_iterations) > 0  # pytorch3d: .all() of nothing is True
    else:
        iters, converged = (int(v) for v in r["status"].cpu())  # the host synchronisation
        converged = bool(converged)
    t_history = [SimilarityTransform(r["R"][k], r["T"][k], r["s"][k]) for k in range(iters)]
    if iters:
        RTs, rmse = t_history[-1], r["rmse"][iters - 1]
    else:
        dev = r["Xt"].device
        init = r["init"]
        RTs = SimilarityTransform(*init) if init is not None else SimilarityTransform(
            torch.eye(3, device=dev).expand(b, 3, 3).clone(), torch.zeros(b, 3, device=dev), torch.ones(b, device=dev))
        rmse = None
    if verbose:
        h = r["rmse"][:iters].cpu()  # fp32, as pytorch3d computes the relative rmse
        for k in range(iters):
            rel = torch.ones_like(h[k]) if k == 0 else (h[k - 1] - h[k]) / h[k - 1]
            print(f"ICP iteration {k}: mean/max rmse = {h[k].mean():1.2e}/{h[k].max():1.2e} ; "
                  f"mean relative rmse = {rel.mean():1.2e}")
        print(f"ICP has converged in {iters} iterations." if converged else
              f"ICP has not converged in {int(max_iterations)} iterations.")
    return ICPSolution(converged, rmse, r["Xt"], RTs, t_history)
