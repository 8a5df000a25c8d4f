"""Float64 restatement of pytorch3d 0.7.2's chamfer_distance with normals, weights and every batch_reduction (recalled, parity
unpinned: pytorch3d is not available), for tests.  It follows pytorch3d's structure: gather the nearest neighbour, mask the
padded rows, multiply by the weights, sum over points, divide by the clamped lengths, reduce over the batch.  The normal term is
1 - |F.cosine_similarity(n, n_near, dim=2, eps=1e-6)|, where knn_gather gives a zero normal when the target cloud is empty.
Every gradient comes from torch autograd.  The nearest-neighbour indices come from oracle.chamfer_forward, which is
bit-exact with the kernels; the distances are recomputed in float64 from the points.  TEST INFRASTRUCTURE ONLY."""
import numpy as np
import torch
import torch.nn.functional as F

import oracle


def neighbours(x, y, x_lengths=None, y_lengths=None, mode=0):
    """(idx_x, idx_y) int64 tensors and the oracle's result dict, for float32 copies of x and y."""
    xf = x.detach().float().cpu().numpy()
    yf = y.detach().float().cpu().numpy()
    o = oracle.chamfer_forward(xf, yf, None if x_lengths is None else x_lengths.cpu(), None if y_lengths is None else y_lengths.cpu(),
                               mode=mode, nthreads=8)
    return torch.from_numpy(o["idx_x"]).long(), torch.from_numpy(o["idx_y"]).long(), o


def _gather(t, idx):
    return t.gather(1, idx[..., None].expand(-1, -1, t.shape[2]))


def chamfer_reference(x, y, idx_x, idx_y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None, weights=None,
                      batch_reduction="mean"):
    """-> (loss, loss_normals or None), differentiable in x, y, the normals and the weights (float64 tensors)."""
    n, p1, _ = x.shape
    p2 = y.shape[1]
    xl = torch.full((n,), p1, dtype=torch.int64) if x_lengths is None else x_lengths.cpu().long()
    yl = torch.full((n,), p2, dtype=torch.int64) if y_lengths is None else y_lengths.cpu().long()
    return_normals = x_normals is not None and y_normals is not None
    if weights is not None:
        if weights.size(0) != n or weights.dim() != 1:
            raise ValueError("weights must be of shape (N,).")
        if not (weights >= 0).all():
            raise ValueError("weights cannot be negative.")
        if weights.sum() == 0.0:
            z = x.sum((1, 2)) * weights * 0.0      # zeros attached to the graph, (N,) or summed
            return (z.sum(), z.sum()) if batch_reduction is not None else (z, z.clone())
    x_mask = torch.arange(p1)[None] >= xl[:, None]          # padded query rows
    y_mask = torch.arange(p2)[None] >= yl[:, None]
    # knn_points(K=1): a query whose target cloud is empty has distance 0 and gets no gradient
    cham_x = ((x - _gather(y, idx_x)) ** 2).sum(2)
    cham_y = ((y - _gather(x, idx_y)) ** 2).sum(2)
    cham_x = torch.where(x_mask | (yl[:, None] == 0), torch.zeros_like(cham_x), cham_x)
    cham_y = torch.where(y_mask | (xl[:, None] == 0), torch.zeros_like(cham_y), cham_y)
    if weights is not None:
        cham_x = cham_x * weights.view(n, 1)
        cham_y = cham_y * weights.view(n, 1)
    if return_normals:
        # knn_gather pads slots k >= lengths2 with zeros: K = 1, so a whole empty target cloud gives a zero normal
        near_x = _gather(y_normals, idx_x) * (yl > 0).view(n, 1, 1)
        near_y = _gather(x_normals, idx_y) * (xl > 0).view(n, 1, 1)
        cham_norm_x = 1 - torch.abs(F.cosine_similarity(x_normals, near_x, dim=2, eps=1e-6))
        cham_norm_y = 1 - torch.abs(F.cosine_similarity(y_normals, near_y, dim=2, eps=1e-6))
        cham_norm_x = torch.where(x_mask, torch.zeros_like(cham_norm_x), cham_norm_x)
        cham_norm_y = torch.where(y_mask, torch.zeros_like(cham_norm_y), cham_norm_y)
        if weights is not None:
            cham_norm_x = cham_norm_x * weights.view(n, 1)
            cham_norm_y = cham_norm_y * weights.view(n, 1)
    cham_x, cham_y = cham_x.sum(1), cham_y.sum(1)
    if return_normals:
        cham_norm_x, cham_norm_y = cham_norm_x.sum(1), cham_norm_y.sum(1)
    xlc, ylc = xl.clamp(min=1).double(), yl.clamp(min=1).double()
    cham_x, cham_y = cham_x / xlc, cham_y / ylc
    if return_normals:
        cham_norm_x, cham_norm_y = cham_norm_x / xlc, cham_norm_y / ylc
    if batch_reduction is not None:
        cham_x, cham_y = cham_x.sum(), cham_y.sum()
        if return_normals:
            cham_norm_x, cham_norm_y = cham_norm_x.sum(), cham_norm_y.sum()
        if batch_reduction == "mean":
            div = weights.sum() if weights is not None else max(n, 1)
            cham_x, cham_y = cham_x / div, cham_y / div
            if return_normals:
                cham_norm_x, cham_norm_y = cham_norm_x / div, cham_norm_y / div
    return cham_x + cham_y, (cham_norm_x + cham_norm_y if return_normals else None)


def cloud_sums_reference(x, y, idx_x, idx_y, x_lengths=None, y_lengths=None, x_normals=None, y_normals=None):
    """float64 numpy (2, N) un-normalised per-cloud sums of the distances and, with both normals, of 1 - |cos|: what
    pcl_chamfer_cloud_fwd writes to cloud_sums / normal_sums."""
    n = x.shape[0]
    x, y = torch.as_tensor(np.asarray(x, np.float64)), torch.as_tensor(np.asarray(y, np.float64))
    xl = torch.full((n,), x.shape[1]) if x_lengths is None else x_lengths.cpu().long()
    yl = torch.full((n,), y.shape[1]) if y_lengths is None else y_lengths.cpu().long()
    out = []
    xn = None if x_normals is None else torch.as_tensor(np.asarray(x_normals, np.float64))
    yn = None if y_normals is None else torch.as_tensor(np.asarray(y_normals, np.float64))
    for d in range(2):
        q, t, iq, lq, lt, nq, nt = (x, y, idx_x, xl, yl, xn, yn) if d == 0 else (y, x, idx_y, yl, xl, yn, xn)
        row = []
        for m in range(n):
            k = int(lq[m])
            if k == 0:
                row.append((0.0, 0.0))
                continue
            j = iq[m, :k]
            dist = 0.0 if int(lt[m]) == 0 else float(((q[m, :k] - t[m, j]) ** 2).sum())
            nrm = 0.0
            if nq is not None:
                near = nt[m, j] * (1.0 if int(lt[m]) > 0 else 0.0)
                nrm = float((1 - torch.abs(F.cosine_similarity(nq[m, :k], near, dim=1, eps=1e-6))).sum())
            row.append((dist, nrm))
        out.append(row)
    a = np.array(out)                                               # (2, N, 2)
    return a[..., 0], (a[..., 1] if xn is not None and yn is not None else None)


def cosine_term_grad(a, b, eps=1e-6):
    """The closed form of d(1 - |cos(a, b)|)/da for rows of a and b, as F.cosine_similarity computes the cosine: each vector
    divided by max(|v|, eps); the clamp carries no gradient, and a / |a| is 0 for a = 0."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.linalg.norm(a, axis=-1, keepdims=True), np.linalg.norm(b, axis=-1, keepdims=True)
    ma, mb = np.maximum(na, eps), np.maximum(nb, eps)
    c = ((a / ma) * (b / mb)).sum(-1, keepdims=True)
    ua = np.divide(a, na, out=np.zeros_like(a), where=na > 0)
    return -np.sign(c) * (b / mb - c * ua) / ma
