"""float64 torch restatement of pytorch3d 0.7.2's corresponding_points_alignment and iterative_closest_point, restated from
memory [3P-memory].  Parity with pytorch3d itself is unpinned: THIS FILE IS THE SPECIFICATION the library is tested
against (include/pcl.h, "points alignment and ICP", says the same in C terms).

  apply(X; R, T, s) = s * (X @ R) + T                                   (row vectors)
  alignment: w = mask(lengths) * weights (the mask without weights); xm = sum w x / clamp(sum w, eps), ym likewise;
             a = w (x - xm), b = w (y - ym)  (pytorch3d weights BOTH centred clouds: the covariance carries w^2);
             Wt = clamp(sum w, eps) with weights or lengths, clamp(n, 1) without;  M = a^T b / Wt = U S V^T;
             E = diag(1, 1, det(U V^T)) (I with allow_reflection);  R = U E V^T;
             s = tr(E S) / clamp(sum |a|^2 / Wt, eps) with estimate_scale, else 1;  T = ym - s (xm @ R).
  ICP:       Xt = apply(X; init) or X;  for each iteration: Ynn = nearest Y of every Xt row (lowest index on ties; 0 when
             the Y cloud is empty);  (R, T, s) = alignment(X, Ynn, weights=mask_X);  Xt = apply(X; R, T, s);
             rmse = sqrt(sum_mask |Xt - Ynn|^2 / clamp(n, 1e-9));  rel = 1 first, then (prev - rmse) / prev;
             stop when (rel <= thr).all() -- one decision for the whole batch, and NaN (0 / 0) never passes.

Gradients of the alignment come from autograd through torch.linalg.svd (finite only for distinct singular values)."""
import torch


def mask_of(lengths, b, p, device="cpu"):
    if lengths is None:
        return torch.ones(b, p, dtype=torch.float64, device=device)
    return (torch.arange(p, device=device)[None, :] < lengths.to(device).view(b, 1)).to(torch.float64)


def apply_ref(X, R, T, s):
    return s[:, None, None] * torch.bmm(X, R) + T[:, None, :]


def alignment_parts(X, Y, weights=None, eps=1e-9, lengths=None):
    """(M, Xcov, xm, ym) of the alignment, float64."""
    b, p, _ = X.shape
    w = mask_of(lengths, b, p, X.device)
    if weights is not None:
        w = w * weights.to(torch.float64)
    weighted = weights is not None or lengths is not None
    Wm = w.sum(1).clamp(min=eps)
    xm = (w[..., None] * X).sum(1) / Wm[:, None]
    ym = (w[..., None] * Y).sum(1) / Wm[:, None]
    a = w[..., None] * (X - xm[:, None])
    bb = w[..., None] * (Y - ym[:, None])
    Wt = Wm if weighted else w.sum(1).clamp(min=1.0)
    M = torch.bmm(a.transpose(1, 2), bb) / Wt[:, None, None]
    xcov = (a * a).sum((1, 2)) / Wt
    return M, xcov, xm, ym


def alignment_ref(X, Y, weights=None, estimate_scale=False, allow_reflection=False, eps=1e-9, lengths=None):
    """-> (R, T, s), float64; differentiable through torch.linalg.svd."""
    X, Y = X.to(torch.float64), Y.to(torch.float64)
    M, xcov, xm, ym = alignment_parts(X, Y, weights, eps, lengths)
    U, S, Vh = torch.linalg.svd(M)
    V = Vh.transpose(1, 2)
    e = torch.ones_like(S)
    if not allow_reflection:
        e = torch.cat([e[:, :2], torch.det(torch.bmm(U, Vh)).detach()[:, None]], 1)
    R = torch.bmm(U * e[:, None, :], Vh)
    if estimate_scale:
        s = (e * S).sum(1) / xcov.clamp(min=eps)
    else:
        s = torch.ones(X.shape[0], dtype=torch.float64, device=X.device)
    T = ym - s[:, None] * torch.bmm(xm[:, None], R)[:, 0]
    return R, T, s


def nn_dense(Xt, Y, x_lengths=None, y_lengths=None):
    """Ynn (B, P1, 3) float64: the nearest Y row of every Xt row in float64 squared L2, lowest index on ties; 0 when the Y
    cloud is empty."""
    Xt, Y = Xt.to(torch.float64), Y.to(torch.float64)
    b, p2 = Y.shape[0], Y.shape[1]
    d = ((Xt[:, :, None, :] - Y[:, None, :, :]) ** 2).sum(-1)
    ym = mask_of(y_lengths, b, p2, Y.device).bool()
    d = torch.where(ym[:, None, :], d, torch.full_like(d, float("inf")))
    idx = d.argmin(2) if p2 > 0 else torch.zeros(Xt.shape[:2], dtype=torch.long)
    if p2 == 0:
        return torch.zeros_like(Xt)
    out = Y.gather(1, idx[..., None].expand(-1, -1, 3))
    return torch.where(ym.any(1)[:, None, None], out, torch.zeros_like(out))


def icp_ref(X, Y, init_transform=None, max_iterations=100, relative_rmse_thr=1e-6, estimate_scale=False,
            allow_reflection=False, x_lengths=None, y_lengths=None, nn=nn_dense):
    """pytorch3d's ICP loop in float64.  Returns dict(converged, rmse, Xt, RTs, t_history, rmse_history, rel_history)."""
    X = X.to(torch.float64)
    b, p1, _ = X.shape
    mask = mask_of(x_lengths, b, p1, X.device)
    if init_transform is not None:
        R, T, s = (t.to(torch.float64) for t in init_transform)
        Xt = apply_ref(X, R, T, s)
    else:
        R = torch.eye(3, dtype=torch.float64).expand(b, 3, 3).clone()
        T, s = torch.zeros(b, 3, dtype=torch.float64), torch.ones(b, dtype=torch.float64)
        Xt = X
    prev, rmse, converged = None, None, False
    hist, rmses, rels = [], [], []
    for _ in range(max_iterations):
        Ynn = nn(Xt, Y, x_lengths, y_lengths).to(torch.float64)
        R, T, s = alignment_ref(X, Ynn, weights=mask, estimate_scale=estimate_scale, allow_reflection=allow_reflection)
        Xt = apply_ref(X, R, T, s)
        hist.append((R, T, s))
        rmse = (((Xt - Ynn) ** 2).sum(2) * mask).sum(1).div(mask.sum(1).clamp(min=1e-9)).sqrt()
        rel = torch.ones_like(rmse) if prev is None else (prev - rmse) / prev
        rmses.append(rmse)
        rels.append(rel)
        if bool((rel <= relative_rmse_thr).all()):
            converged = True
            break
        prev = rmse
    return dict(converged=converged, rmse=rmse, Xt=Xt, RTs=(R, T, s), t_history=hist, rmse_history=rmses, rel_history=rels)


def random_rotation(b, generator, max_angle=None):
    """(b, 3, 3) float64 proper rotations: uniform over SO(3), or about a random axis by an angle up to max_angle (rad)."""
    axis = torch.randn(b, 3, generator=generator, dtype=torch.float64)
    axis = axis / axis.norm(dim=1, keepdim=True)
    if max_angle is None:
        q = torch.randn(b, 4, generator=generator, dtype=torch.float64)
        q = q / q.norm(dim=1, keepdim=True)
        w, x, y, z = q.unbind(1)
        return torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                            2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                            2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], 1).view(b, 3, 3)
    ang = (torch.rand(b, generator=generator, dtype=torch.float64) * 2 - 1) * max_angle
    return axis_angle(axis, ang)


def axis_angle(axis, ang):
    """Rodrigues: (b, 3) unit axes, (b,) angles -> (b, 3, 3) rotations (column-vector form; as a row-vector R, X @ R
    rotates by -ang)."""
    K = torch.zeros(axis.shape[0], 3, 3, dtype=torch.float64)
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -axis[:, 2], axis[:, 1], -axis[:, 0]
    K = K - K.transpose(1, 2)
    I = torch.eye(3, dtype=torch.float64).expand_as(K)
    c, s = torch.cos(ang)[:, None, None], torch.sin(ang)[:, None, None]
    return I + s * K + (1 - c) * torch.bmm(K, K)
