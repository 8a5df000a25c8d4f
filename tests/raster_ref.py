"""torch restatement of pytorch3d 0.7.2's rasterize_points and of the three point compositors (alpha_composite,
norm_weighted_sum, weighted_sum), restated from memory [3P-memory].  Parity with pytorch3d itself is unpinned: THIS FILE IS
THE SPECIFICATION the library is tested against (include/pcl.h, "rasterize points / compositing", says the same in C terms).

Rasterizer, in float32 with every operation rounded, in this order:
  pixel (row r, column c): xf = ndc(W-1-c, W, H), yf = ndc(H-1-r, H, W),
      ndc(i, S1, S2) = -off + (range*i + off) / S1,  range = S1 > S2 ? (S1*2)/S2 : 2,  off = range/2
  point i of cloud b hits it when i < lengths[b] (clamped to [0, P]), x, y, z, r finite, z >= 0 and
      d2 = dx*dx + dy*dy <= r*r,  dx = xf - x, dy = yf - y   (r = radius, or radius[b, i])
  the pixel keeps the K hits of smallest (z + 0.0, i), ascending:
      idx = offset_b + i (offset_b = sum(lengths[:b])), zbuf = z, dists = d2; unused slots -1 in all three.
Its gradients (rasterize_grads_ref) are autograd of a float64 version on the same idx: zbuf -> z, dists -> 2 g (p_xy - pixel_xy).

Compositors (N, K, H, W) x (C, P_total) -> (N, C, H, W), in float32 in k order, a slot with idx < 0 or >= P_total adding
nothing:
  weighted_sum:       acc += a_k * F[:, idx_k]
  norm_weighted_sum:  acc += (a_k * F[:, idx_k]) / w,  w = clamp(sum of the valid a_k (in k order), min=1e-4)
  alpha_composite:    acc += (T_k * a_k) * F[:, idx_k],  T_0 = 1, T_{k+1} = T_k * (1 - a_k) over every slot
The same functions run in float64 give the gradients by autograd."""
import torch

F32 = torch.float32


def ndc(i, S1, S2, dtype=F32):
    """The pixel centres ndc(i, S1, S2) of the index tensor i, every operation rounded in `dtype`."""
    range_ = torch.tensor(float(S1 * 2), dtype=dtype) / torch.tensor(float(S2), dtype=dtype) if S1 > S2 \
        else torch.tensor(2.0, dtype=dtype)
    off = range_ / 2
    return -off + (range_ * i.to(dtype) + off) / torch.tensor(float(S1), dtype=dtype)


def pixel_centres(H, W, dtype=F32, device="cpu"):
    """-> (xs (W,), ys (H,)): the centre of column c is xs[c], of row r is ys[r]."""
    xs = ndc(W - 1 - torch.arange(W), W, H, dtype)
    ys = ndc(H - 1 - torch.arange(H), H, W, dtype)
    return xs.to(device), ys.to(device)


def clamped_lengths(lengths, B, P):
    if lengths is None:
        return torch.full((B,), P, dtype=torch.int64)
    return lengths.detach().cpu().to(torch.int64).clamp(0, P)


def rasterize_ref(points, lengths=None, image_size=8, radius=0.01, K=8, rows_per_chunk=16):
    """The forward in float32 -> (idx (B,H,W,K) int32, zbuf, dists (B,H,W,K) float32), on points' device."""
    H, W = (image_size, image_size) if isinstance(image_size, int) else image_size
    B, P, _ = points.shape
    dev = points.device
    pts = points.detach().to(F32)
    ln = clamped_lengths(lengths, B, P)
    offs = torch.cumsum(ln, 0) - ln
    xs, ys = pixel_centres(H, W, device=dev)
    idx = torch.full((B, H, W, K), -1, dtype=torch.int32, device=dev)
    zbuf = torch.full((B, H, W, K), -1.0, dtype=F32, device=dev)
    dists = torch.full((B, H, W, K), -1.0, dtype=F32, device=dev)
    for b in range(B):
        n = int(ln[b])
        if n == 0:
            continue
        x, y, z = pts[b, :n, 0], pts[b, :n, 1], pts[b, :n, 2]
        r = (radius[b, :n].detach().to(dev).to(F32) if torch.is_tensor(radius)
             else torch.full((n,), float(radius), dtype=F32, device=dev))
        ok = torch.isfinite(x) & torch.isfinite(y) & torch.isfinite(z) & torch.isfinite(r) & (z >= 0)
        r2 = r * r
        zkey = z + 0.0                                            # -0.0 -> +0.0
        for r0 in range(0, H, rows_per_chunk):
            yy = ys[r0:r0 + rows_per_chunk]
            dx = xs[None, :, None] - x[None, None, :]             # (1, W, n)
            dy = yy[:, None, None] - y[None, None, :]             # (h, 1, n)
            d2 = dx * dx + dy * dy                                # (h, W, n), each product and the sum rounded
            hit = ok & (d2 <= r2)
            key = torch.where(hit, zkey.expand_as(d2), torch.full_like(d2, float("inf")))
            order = torch.sort(key, dim=-1, stable=True).indices[..., :K]   # ties in z: index order
            cnt = hit.sum(-1, keepdim=True)
            kk = torch.arange(order.shape[-1], device=dev)
            used = kk < cnt
            h = yy.shape[0]
            sl = (b, slice(r0, r0 + h), slice(None), slice(0, order.shape[-1]))
            idx[sl] = torch.where(used, (order + offs[b].to(dev)).to(torch.int32), torch.full_like(order, -1, dtype=torch.int32))
            zbuf[sl] = torch.where(used, z[order], torch.full_like(order, -1, dtype=F32))
            dists[sl] = torch.where(used, torch.gather(d2, -1, order), torch.full_like(order, -1, dtype=F32))
    return idx, zbuf, dists


def rasterize_diff_ref(points, idx, lengths=None, image_size=8):
    """(zbuf, dists) of the given idx in float64, differentiable in `points` (B, P, 3) -- the gradient specification.
    Slots with idx -1 are -1 and carry no gradient."""
    H, W = (image_size, image_size) if isinstance(image_size, int) else image_size
    B, P, _ = points.shape
    dev = points.device
    ln = clamped_lengths(lengths, B, P)
    offs = (torch.cumsum(ln, 0) - ln).to(dev)
    xs, ys = pixel_centres(H, W, device=dev)                       # the fp32 centres, as the forward uses them
    K = idx.shape[-1]
    valid = idx >= 0
    local = torch.where(valid, idx.long() - offs[:, None, None, None], torch.zeros_like(idx, dtype=torch.long))
    bb = torch.arange(B, device=dev)[:, None, None, None].expand_as(local)
    p = points.to(torch.float64)[bb, local]                        # (B, H, W, K, 3)
    px = xs.to(torch.float64)[None, None, :, None]
    py = ys.to(torch.float64)[None, :, None, None]
    z = torch.where(valid, p[..., 2], torch.full_like(p[..., 2], -1.0))
    d = torch.where(valid, (px - p[..., 0]) ** 2 + (py - p[..., 1]) ** 2, torch.full_like(p[..., 2], -1.0))
    return z, d


def _valid(idx, P_total):
    return (idx >= 0) & (idx < P_total)


def _gather(features, idx, ok):
    """features (C, P) -> (N, K, H, W, C) of the slots, 0 where not ok."""
    safe = torch.where(ok, idx.long(), torch.zeros_like(idx, dtype=torch.long))
    g = features.t()[safe]
    return torch.where(ok[..., None], g, torch.zeros_like(g))


def composite_ref(mode, pointsidx, alphas, features, dtype=F32):
    """mode 'alpha' | 'norm' | 'weighted' -> (N, C, H, W) in `dtype`, summed in k order as the module docstring says;
    differentiable in alphas and features when dtype is float64."""
    a = alphas.to(dtype)
    F = features.to(dtype)
    N, K, H, W = pointsidx.shape
    ok = _valid(pointsidx, F.shape[1])
    Fk = _gather(F, pointsidx, ok)                                 # (N, K, H, W, C)
    acc = torch.zeros(N, H, W, F.shape[0], dtype=dtype, device=a.device)
    if mode == "norm":
        s = torch.zeros(N, H, W, dtype=dtype, device=a.device)
        for k in range(K):
            s = torch.where(ok[:, k], s + a[:, k], s)
        w = torch.clamp(s, min=1e-4)
    T = torch.ones(N, H, W, dtype=dtype, device=a.device)
    for k in range(K):
        ak = a[:, k]
        if mode == "weighted":
            term = ak[..., None] * Fk[:, k]
        elif mode == "norm":
            term = (ak[..., None] * Fk[:, k]) / w[..., None]
        else:
            term = (T * ak)[..., None] * Fk[:, k]
            T = T * (1 - ak)
        acc = torch.where(ok[:, k, ..., None], acc + term, acc)
    return acc.permute(0, 3, 1, 2)
