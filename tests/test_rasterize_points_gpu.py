"""rasterize_points and the point compositors on the GPU against tests/raster_ref.py: bit-exact forwards, identical bits on
every bin size and bin capacity, gradients against float64 autograd, the end-to-end image loss, stale state, graph capture,
the launch count and host synchronisation.

Let u = 2^-24 and gamma_k = k u / (1 - k u).  A result formed as a sum of M terms, each a product of at most D factors
rounded once per operation, differs from the exact sum by at most gamma_(M+D) times the sum of the terms' magnitudes (the
standard bound for recursive summation plus one rounding per product factor, in any order of summation).

Rasterizer backward.  grad z of point i sums its n slots' grad_zbuf (exact terms): gamma_n scale.  grad x (and y) sums n
terms 2 g (x - xf): 2 g is exact, x - xf and the product are rounded once each, xf is the same fp32 centre as in the float64
restatement: gamma_(n+2) scale, scale = sum |2 g (x - xf)|.  red.add flushes a subnormal to zero, at most 2^-126 per
addition, so the test allows gamma_(n+2) scale + n 2^-126 with n the largest slot count of any point.  Points in no slot
get exactly 0.

Compositor backward, with alphas in [0, 1] (so every T and 1 - a is at most 1 in magnitude):
  weighted:  grad_a_k = sum_c g_c F[c, idx_k]: M = C, D = 1.  grad_F sums n slots' g a: M = n, D = 1.
  norm:      grad_a_k = (e_k - G) / w with e_k (M = C, D = 1) and G = sum_c g_c sum_k a_k F / w (M = C K, D = 3), one
             subtraction and one division: M + D <= C K + C + 6 over the scale (sum_c |g_c F_kc| + sum_c |g_c| sum_k |a_k F_kc| / w) / w.
  alpha:     T_j is a product of j rounded factors (1 - a_t), R_j a recursion of K - j steps of two products and one sum,
             grad_a_j = T_j (e_j - R_j): M + D <= C + 4 K + 4 over sum_c |g_c| (|F_jc| + sum_(k>j) |a_k F_kc|).
The test allows gamma_(2 C K + 4 K + 2 C + 16) of each scale, and n 2^-126 more for grad_F."""
import numpy as np
import pytest
import torch

import pointcloud_b200 as pcl
from helpers import npy, same_bits
from pointcloud_b200 import _lib, synth
from raster_ref import composite_ref, rasterize_diff_ref, rasterize_ref
from test_stale_state_gpu import PATTERNS, Stale, capture_and_replay

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
F64 = torch.float64


def gamma(k):
    return k * U / (1 - k * U)


def cloud(B, P, seed, lo=-1.1, hi=1.1):
    """Table-shaped clouds mapped into the view: x, y in [lo, hi], z in [0.1, 2.1] (uniform noise for tiny P)."""
    if P < 64:
        x = torch.rand(B, P, 3, generator=torch.Generator().manual_seed(seed))
    else:
        x = synth.table_clouds(B, P, seed=seed)[0].clone()
    x[..., :2] = x[..., :2] * (hi - lo) + lo
    x[..., 2] = x[..., 2] * 2 + 0.1
    return x


def lengths_for(B, P, seed):
    n = torch.randint(0, P + 1, (B,), generator=torch.Generator().manual_seed(seed))
    n[0] = P
    if B > 2:
        n[1] = 0
    return n


def check_same(got, want):
    for g, w, name in zip(got, want, ("idx", "zbuf", "dists")):
        assert g.shape == w.shape, name
        assert same_bits(npy(g), npy(w)) if g.dtype == torch.float32 else torch.equal(g, w), name


FWD = [  # B, P, (H, W), K, per-point radius, ragged, radius
    (1, 1, (1, 1), 1, False, False, 0.5),
    (3, 500, (64, 64), 8, False, True, 0.05),
    (2, 2000, (48, 80), 8, True, True, 0.04),
    (2, 2000, (80, 48), 1, False, True, 0.03),
    (4, 1000, (33, 47), 150, True, True, 0.1),
    (2, 3000, (40, 40), 20, False, False, 0.08),
    (2, 3000, (40, 40), 70, True, True, 0.08),
    (8, 2048, (64, 64), 8, False, True, 0.02),
    (1, 20000, (96, 128), 8, False, False, 0.01),
]


@pytest.mark.parametrize("bin_size", [0, None])
@pytest.mark.parametrize("B,P,hw,K,per_point,ragged,r", FWD)
def test_forward_bit_exact(B, P, hw, K, per_point, ragged, r, bin_size):
    pts = cloud(B, P, B * P + K).cuda()
    ln = lengths_for(B, P, K).cuda() if ragged else None
    rad = (torch.rand(B, P, generator=torch.Generator().manual_seed(3)) * 2 * r).cuda() if per_point else r
    got = pcl.rasterize_points_forward_raw(pts, ln, hw, rad, K, bin_size)
    want = rasterize_ref(pts, ln, hw, rad, K)
    check_same((got["idx"], got["zbuf"], got["dists"]), want)
    assert int((want[0] >= 0).sum()) > 0 or P == 1


@pytest.mark.parametrize("form", ["fp16", "bf16", "strided"])
def test_half_and_strided_inputs(form):
    B, P = 3, 3000
    base = cloud(B, P, 4).cuda()
    if form == "strided":
        buf = torch.cat([base, torch.randn(B, P, 3, device="cuda")], 2)
        pts, ref_in = buf[:, :, :3], base
    else:
        pts = base.to(torch.float16 if form == "fp16" else torch.bfloat16)
        ref_in = pts.float()
    ln = lengths_for(B, P, 5).cuda()
    for bs in (0, 16):
        got = pcl.rasterize_points_forward_raw(pts, ln, (50, 70), 0.05, 8, bs)
        check_same((got["idx"], got["zbuf"], got["dists"]), rasterize_ref(ref_in, ln, (50, 70), 0.05, 8))


def test_cloud_on_tile_borders():
    """Points on the pixel lines between 16-pixel blocks, and their radii exactly reaching the next block's centres."""
    H = W = 64
    xs = torch.tensor([1 - 2 * k * 16 / W for k in range(5)])
    g = torch.stack(torch.meshgrid(xs, xs, indexing="ij"), -1).reshape(-1, 2)
    pts = torch.cat([g, torch.rand(g.shape[0], 1) + 0.1], 1)[None].cuda()
    for r in (1.0 / W, 3.0 / W, 0.2):
        want = rasterize_ref(pts, None, (H, W), r, 8)
        for bs in (0, 16, 32, 64):
            got = pcl.rasterize_points_forward_raw(pts, None, (H, W), r, 8, bs)
            check_same((got["idx"], got["zbuf"], got["dists"]), want)


# ---------------------------------------------------------------- paths agree ---------------------------------------------

def all_paths(pts, ln, hw, r, K):
    outs = []
    for bs, cap in ((0, None), (16, None), (32, None), (64, None), (128, None), (16, 1), (32, 1), (None, None), (None, 1)):
        o = pcl.rasterize_points_forward_raw(pts, ln, hw, r, K, bs, cap)
        outs.append((o["idx"], o["zbuf"], o["dists"]))
    for o in outs[1:]:
        check_same(o, outs[0])
    return outs[0]


@pytest.mark.parametrize("K", [1, 8, 40])
def test_every_bin_size_and_capacity_gives_the_same_bits(K):
    B, P = 4, 5000
    pts = cloud(B, P, 6).cuda()
    all_paths(pts, lengths_for(B, P, 7).cuda(), (100, 140), 0.02, K)


def test_one_point_covering_the_image_and_a_crowded_tile():
    pts = cloud(2, 2000, 8).cuda()
    pts[0, 5] = torch.tensor([0.0, 0.0, 0.05])
    rad = torch.full((2, 2000), 0.01, device="cuda")
    rad[0, 5] = 10.0
    out = all_paths(pts, None, (128, 96), rad, 8)
    assert (out[0][0, ..., 0] == 5).all()
    # 100 000 points inside one 16 x 16 pixel block
    g = torch.Generator().manual_seed(9)
    P = 100000
    q = torch.rand(1, P, 3, generator=g)
    q[..., :2] = q[..., :2] * 0.2 + 0.3                                  # x, y in [0.3, 0.5]: one block of a 128 x 128 image
    q[..., 2] += 0.1
    all_paths(q.cuda(), None, 128, 0.01, 8)


def test_a_cloud_alone_equals_its_slice_of_the_batch():
    B, P = 5, 3000
    pts = cloud(B, P, 10).cuda()
    ln = lengths_for(B, P, 11).cuda()
    full = pcl.rasterize_points_forward_raw(pts, ln, 64, 0.03, 8, 16)
    off = int(ln[:3].sum())
    one = pcl.rasterize_points_forward_raw(pts[3:4], ln[3:4], 64, 0.03, 8, 0)
    sub = full["idx"][3:4]
    assert torch.equal(torch.where(sub >= 0, sub - off, sub), one["idx"])
    assert same_bits(npy(full["zbuf"][3:4]), npy(one["zbuf"])) and same_bits(npy(full["dists"][3:4]), npy(one["dists"]))


def test_huge_and_non_finite_points_change_nothing():
    pts = cloud(2, 1000, 12).cuda()
    base = pcl.rasterize_points_forward_raw(pts, None, 64, 0.05, 8, 0)
    bad = torch.tensor([[1e30, 0, 1], [float("nan"), 0, 1], [0, float("inf"), 1], [0, 0, -1], [-3e38, 3e38, 1]],
                       device="cuda").expand(2, 5, 3)
    p2 = torch.cat([pts, bad], 1)
    for bs in (0, 16, 64):
        o = pcl.rasterize_points_forward_raw(p2, None, 64, 0.05, 8, bs)
        shift = torch.where(base["idx"] >= 0, base["idx"] + (base["idx"] >= 1000).int() * 5, base["idx"])
        assert torch.equal(o["idx"], shift) and same_bits(npy(o["zbuf"]), npy(base["zbuf"]))


# ---------------------------------------------------------------- rasterizer backward --------------------------------------

@pytest.mark.parametrize("B,P,hw,K,ragged", [(3, 2000, (48, 64), 8, True), (2, 1500, (40, 40), 1, False),
                                             (2, 800, (32, 24), 30, True)])
def test_rasterizer_backward_against_float64(B, P, hw, K, ragged):
    pts = cloud(B, P, 13 + K).cuda()
    ln = lengths_for(B, P, 14).cuda() if ragged else None
    p = pts.clone().requires_grad_()
    idx, zbuf, dists = pcl.rasterize_points(p, ln, hw, 0.06, K)
    g = torch.Generator().manual_seed(15)
    gz, gd = torch.randn(zbuf.shape, generator=g).cuda(), torch.randn(dists.shape, generator=g).cuda()
    ((zbuf * gz).sum() + (dists * gd).sum()).backward()
    q = pts.double().requires_grad_()
    z, d = rasterize_diff_ref(q, idx, ln, hw)
    ((z * gz.double()).sum() + (d * gd.double()).sum()).backward()
    ref = q.grad
    # scales and slot counts per point
    valid = idx >= 0
    offs = torch.cumsum(torch.tensor([P] * B) if ln is None else ln.cpu(), 0) - (P if ln is None else ln.cpu())
    local = (idx.long() - offs.cuda()[:, None, None, None])[valid]
    bb = torch.arange(B, device="cuda")[:, None, None, None].expand_as(idx)[valid]
    row = bb * P + local
    cnt = torch.zeros(B * P, dtype=F64, device="cuda").index_add_(0, row, torch.ones_like(row, dtype=F64))
    n = int(cnt.max())
    sz = torch.zeros(B * P, dtype=F64, device="cuda").index_add_(0, row, gz.double()[valid].abs())
    zz, dd = rasterize_diff_ref(pts.double(), idx, ln, hw)
    H, W = hw
    from raster_ref import pixel_centres
    xs, ys = pixel_centres(H, W, device="cuda")
    pxy = pts.double()[bb, local]
    ex = (2 * gd.double()[valid] * (pxy[:, 0] - xs.double()[None, None, :, None].expand_as(idx)[valid])).abs()
    ey = (2 * gd.double()[valid] * (pxy[:, 1] - ys.double()[None, :, None, None].expand_as(idx)[valid])).abs()
    sx = torch.zeros(B * P, dtype=F64, device="cuda").index_add_(0, row, ex)
    sy = torch.zeros(B * P, dtype=F64, device="cuda").index_add_(0, row, ey)
    scale = torch.stack([sx, sy, sz], 1).view(B, P, 3)
    err = (p.grad.double() - ref).abs()
    assert not (err > gamma(n + 2) * scale + n * 2.0 ** -126).any(), float((err - gamma(n + 2) * scale).max())
    assert (p.grad.view(B * P, 3)[cnt == 0] == 0).all() and bool((cnt == 0).any())
    assert p.grad.dtype == pts.dtype and float(ref.abs().max()) > 0


def test_rasterizer_backward_in_the_input_dtype():
    p = cloud(2, 1000, 16).cuda().half().requires_grad_()
    _, z, d = pcl.rasterize_points(p, None, 32, 0.1, 4)
    (z.sum() + d.sum()).backward()
    assert p.grad.dtype == torch.float16 and p.grad.shape == p.shape and torch.isfinite(p.grad).all()


# ---------------------------------------------------------------- compositors -----------------------------------------------

MODES = {"alpha": pcl.alpha_composite, "norm": pcl.norm_weighted_sum, "weighted": pcl.weighted_sum}


def comp_case(N, K, H, W, C, P, seed, itype=torch.int64, permuted=True):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(-2, P + 2, (N, H, W, K), generator=g)              # -1, -2 and out-of-range entries
    a = torch.rand(N, H, W, K, generator=g)
    a[0, 0, 0] = 1e-6                                                       # sum below 1e-4
    a[..., 1 % K][torch.rand(N, H, W, generator=g) < 0.3] = 1.0
    a[..., 2 % K][torch.rand(N, H, W, generator=g) < 0.3] = 0.0
    F = torch.randn(P, C, generator=g)
    idx, a, F = idx.to(itype).cuda(), a.cuda(), F.cuda()
    if permuted:
        return idx.permute(0, 3, 1, 2), a.permute(0, 3, 1, 2), F.t()
    return idx.permute(0, 3, 1, 2).contiguous(), a.permute(0, 3, 1, 2).contiguous(), F.t().contiguous()


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("itype", [torch.int32, torch.int64])
@pytest.mark.parametrize("permuted", [True, False])
@pytest.mark.parametrize("N,K,H,W,C,P", [(2, 8, 20, 30, 3, 500), (1, 1, 7, 5, 16, 40), (3, 150, 9, 11, 5, 300)])
def test_compositor_forward_bit_exact(mode, itype, permuted, N, K, H, W, C, P):
    idx, a, F = comp_case(N, K, H, W, C, P, N * K + C, itype, permuted)
    got = MODES[mode](idx, a, F)
    assert got.shape == (N, C, H, W) and got.dtype == torch.float32
    assert same_bits(npy(got), npy(composite_ref(mode, idx, a, F)))


def comp_bound_scales(mode, idx, a, F, g):
    """Per-alpha and per-feature scales of the bound in the module docstring (float64)."""
    a, F, g = a.double(), F.double(), g.double()
    ok = (idx >= 0) & (idx < F.shape[1])
    Fk = F.t()[torch.where(ok, idx.long(), 0)] * ok[..., None]          # (N, K, H, W, C)
    gk = g.permute(0, 2, 3, 1)[:, None]                                  # (N, 1, H, W, C)
    eF = (gk.abs() * Fk.abs()).sum(-1)                                   # (N, K, H, W)
    aF = (a.abs()[..., None] * Fk.abs())                                 # (N, K, H, W, C)
    if mode == "weighted":
        sa = eF
    elif mode == "norm":
        w = torch.clamp((a * ok).sum(1), min=1e-4)[:, None]
        sa = (eF + (gk.abs() * aF.sum(1, keepdim=True)).sum(-1) / w) / w
    else:
        tail = aF.flip(1).cumsum(1).flip(1) - aF                         # sum over k > j
        sa = eF + (gk.abs() * tail).sum(-1)
    return sa


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("N,K,H,W,C,P", [(2, 8, 20, 30, 3, 500), (3, 30, 9, 11, 16, 300)])
def test_compositor_backward_against_float64(mode, N, K, H, W, C, P):
    idx, a, F = comp_case(N, K, H, W, C, P, 17 + K)
    g = torch.randn(N, C, H, W, generator=torch.Generator().manual_seed(18)).cuda()
    aa, ff = a.detach().clone().requires_grad_(), F.detach().clone().requires_grad_()
    (MODES[mode](idx, aa, ff) * g).sum().backward()
    ra, rf = a.double().requires_grad_(), F.double().requires_grad_()
    (composite_ref(mode, idx, ra, rf, F64) * g.double()).sum().backward()
    assert torch.isfinite(aa.grad).all() and torch.isfinite(ff.grad).all()       # alpha = 1 included
    tol = gamma(2 * C * K + 4 * K + 2 * C + 16)
    sa = comp_bound_scales(mode, idx, a, F, g)
    assert not ((aa.grad.double() - ra.grad).abs() > tol * sa + 1e-38).any(), mode
    # grad_F: n slots' g_c * (weight of the slot), weights at most 1 / w
    ok = (idx >= 0) & (idx < P)
    n = int(torch.zeros(P, device="cuda").index_add_(0, idx[ok].long(), torch.ones(int(ok.sum()), device="cuda")).max())
    wmax = 1.0 if mode != "norm" else 1e4
    sf = torch.zeros(C, P, dtype=F64, device="cuda")
    gk = g.double().permute(0, 2, 3, 1)[:, None].expand(N, K, H, W, C)[ok]   # (M, C)
    sf.index_add_(1, idx[ok].long(), gk.abs().t() * wmax)
    assert not ((ff.grad.double() - rf.grad).abs() > gamma(n + 2 * K + 8) * sf + n * 2.0 ** -126).any(), mode


# ---------------------------------------------------------------- end to end ------------------------------------------------

@pytest.mark.parametrize("mode", list(MODES))
def test_end_to_end_image_loss(mode):
    B, P, C, H, W, K, r = 2, 1500, 3, 40, 48, 8, 0.08
    pts = cloud(B, P, 19).cuda()
    ln = lengths_for(B, P, 20).cuda()
    feats = torch.rand(int(ln.sum()), C, generator=torch.Generator().manual_seed(21)).cuda()
    target = torch.rand(B, C, H, W, generator=torch.Generator().manual_seed(22)).cuda()
    p, f = pts.clone().requires_grad_(), feats.clone().requires_grad_()
    idx, zbuf, dists = pcl.rasterize_points(p, ln, (H, W), r, K)
    weights = 1 - dists.permute(0, 3, 1, 2) / r ** 2
    img = MODES[mode](idx.permute(0, 3, 1, 2), weights, f.t())
    ((img - target) ** 2).mean().backward()
    q, fq = pts.double().requires_grad_(), feats.double().requires_grad_()
    _, d = rasterize_diff_ref(q, idx, ln, (H, W))
    w64 = 1 - d.permute(0, 3, 1, 2) / r ** 2
    img64 = composite_ref(mode, idx.permute(0, 3, 1, 2), w64, fq.t(), F64)
    ((img64 - target.double()) ** 2).mean().backward()
    assert float((img.double() - img64).abs().max()) < 1e-4
    for got, ref in ((p.grad, q.grad), (f.grad, fq.grad)):
        s = float(ref.abs().max())
        assert s > 0 and float((got.double() - ref).abs().max()) <= 1e-3 * s


# ---------------------------------------------------------------- stale state, graphs, launches ----------------------------

def test_stale_outputs_workspace_and_shared_memory():
    st = Stale()
    L = st.L
    B, P, H, W = 3, 4000, 40, 56
    pts = cloud(B, P, 23).cuda()
    ln = lengths_for(B, P, 24).cuda()
    A = _lib.pts_args
    for K, bs, cap in ((8, 0, 0), (1, 16, 0), (20, 32, 0), (8, 16, 3)):
        want = rasterize_ref(pts, ln, (H, W), 0.05, K)
        outs = [torch.empty(B, H, W, K, device="cuda", dtype=torch.int32), torch.empty(B, H, W, K, device="cuda"),
                torch.empty(B, H, W, K, device="cuda")]
        nws = int(L.pcl_rasterize_points_workspace_bytes(B, P, H, W, bs, cap))
        ws = torch.empty(max(nws, 4) // 4, device="cuda", dtype=torch.int32)
        st.run(PATTERNS, outs, [ws], lambda q: L.pcl_rasterize_points_fwd(
            *A(pts), ln.data_ptr(), None, 0.05, B, P, H, W, K, bs, cap, outs[0].data_ptr(), outs[1].data_ptr(),
            outs[2].data_ptr(), ws.data_ptr(), nws, q),
            check=lambda o: all(np.array_equal(x.view(np.int32), npy(w).view(np.int32)) for x, w in zip(o, want)))
    K = 8
    idx = pcl.rasterize_points_forward_raw(pts, ln, (H, W), 0.05, K)["idx"]
    gz = torch.ones(B, H, W, K, device="cuda")
    gp = torch.empty(B, P, 3, device="cuda")
    res = st.run(PATTERNS[:2], [gp], [], lambda q: L.pcl_rasterize_points_bwd(
        *A(pts), ln.data_ptr(), B, P, H, W, K, idx.data_ptr(), gz.data_ptr(), None, gp.data_ptr(), q))
    cnt = torch.zeros(B * P, device="cuda").index_add_(
        0, (idx[idx >= 0].long()), torch.ones(int((idx >= 0).sum()), device="cuda"))
    packed = torch.cat([torch.arange(int(ln[b]), device="cuda") + b * P for b in range(B)])
    want = torch.zeros(B * P, device="cuda")
    want[packed] = cnt[:packed.numel()]
    assert np.array_equal(res[0][0][..., 2].reshape(-1), npy(want)) and not res[0][0][..., :2].any()
    # compositors
    idx4, a, F = comp_case(2, 8, 20, 30, 3, 500, 25)
    for mode, m in (("alpha", 0), ("norm", 1), ("weighted", 2)):
        out = torch.empty(2, 3, 20, 30, device="cuda")
        from pointcloud_b200.compositing import _args
        args = _args(m, idx4, a, F)
        st.run(PATTERNS, [out], [], lambda q: L.pcl_composite_fwd(*args, out.data_ptr(), q),
               check=lambda o: same_bits(o[0], npy(composite_ref(mode, idx4, a, F))))


def test_graph_capture_and_replay():
    L = _lib.lib()
    B, P, H, W, K = 3, 3000, 48, 40, 8
    pts, new = cloud(B, P, 26).cuda(), cloud(B, P, 27).cuda()
    ln = lengths_for(B, P, 28).cuda()
    A = _lib.pts_args
    orig = pts.clone()
    for bs, nxt in ((0, new), (16, orig)):                              # each replay sees inputs unlike the captured ones
        outs = [torch.empty(B, H, W, K, device="cuda", dtype=torch.int32), torch.empty(B, H, W, K, device="cuda"),
                torch.empty(B, H, W, K, device="cuda")]
        nws = int(L.pcl_rasterize_points_workspace_bytes(B, P, H, W, bs, 0))
        ws = torch.empty(max(nws, 1), device="cuda", dtype=torch.uint8)
        capture_and_replay([pts], [nxt], outs, lambda q: L.pcl_rasterize_points_fwd(
            *A(pts), ln.data_ptr(), None, 0.05, B, P, H, W, K, bs, 0, outs[0].data_ptr(), outs[1].data_ptr(),
            outs[2].data_ptr(), ws.data_ptr(), nws, q))
    idx = pcl.rasterize_points_forward_raw(pts, ln, (H, W), 0.05, K)["idx"]
    gz, gd = torch.randn(B, H, W, K, device="cuda"), torch.randn(B, H, W, K, device="cuda")
    gp = torch.empty(B, P, 3, device="cuda")
    capture_and_replay([gz], [torch.randn_like(gz)], [gp], lambda q: L.pcl_rasterize_points_bwd(
        *A(pts), ln.data_ptr(), B, P, H, W, K, idx.data_ptr(), gz.data_ptr(), gd.data_ptr(), gp.data_ptr(), q), loose=(0,))
    from pointcloud_b200.compositing import _args
    idx4, a, F = comp_case(2, 8, 20, 30, 3, 500, 29)
    alts = [comp_case(2, 8, 20, 30, 3, 500, s)[1].clone() for s in (30, 31)] + [a.clone()]
    k = 0
    for m in (0, 1, 2):
        out = torch.empty(2, 3, 20, 30, device="cuda")
        capture_and_replay([a], [alts[k % 3]], [out], lambda q: L.pcl_composite_fwd(*_args(m, idx4, a, F), out.data_ptr(), q))
        g = torch.randn(2, 3, 20, 30, device="cuda")
        ga, gf = torch.empty(2, 8, 20, 30, device="cuda"), torch.empty(3, 500, device="cuda")
        capture_and_replay([a], [alts[(k + 1) % 3]], [ga, gf], lambda q: L.pcl_composite_bwd(
            *_args(m, idx4, a, F), g.data_ptr(), ga.data_ptr(), gf.data_ptr(), q), loose=(1,))
        k += 2


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_launches_do_not_depend_on_the_data_and_nothing_syncs():
    B, P, H, W, K = 2, 4000, 64, 64, 8
    p = cloud(B, P, 31).cuda().requires_grad_()
    crowd = p.detach().clone()
    crowd[..., :2] = crowd[..., :2] * 0.01                              # every point in a few bins: bins overflow at cap 8
    feats = torch.rand(B * P, 3, device="cuda", requires_grad=True)
    for bs, cap in ((0, None), (16, None), (16, 8)):
        counts = []
        for src in (p, crowd):
            def fwd():
                return pcl.rasterize_points_forward_raw(src.detach(), None, (H, W), 0.03, K, bs, cap)
            fwd()
            names = _kernels(fwd)
            counts.append((len([n for n in names if "raster_" in n]), len([n for n in names if "emset" in n.lower()])))
        assert counts[0] == counts[1] == ((1, 0) if bs == 0 else (2, 1)), counts
        torch.cuda.set_sync_debug_mode("error")
        try:
            idx, z, d = pcl.rasterize_points(p, None, (H, W), 0.03, K, bs, cap)
            for comp in MODES.values():
                img = comp(idx.permute(0, 3, 1, 2), 1 - d.permute(0, 3, 1, 2) / 0.03 ** 2, feats.t())
                (img.sum() + z.sum()).backward(retain_graph=True)
        finally:
            torch.cuda.set_sync_debug_mode(0)
        torch.cuda.synchronize()
    idx, z, d = pcl.rasterize_points(p, None, (H, W), 0.03, K)
    names = _kernels(lambda: (z.sum() + d.sum()).backward())
    assert len([n for n in names if "raster_bwd_kernel" in n]) == 1
    a = (1 - d.permute(0, 3, 1, 2) / 0.03 ** 2).detach().requires_grad_()
    for comp, kn in ((pcl.alpha_composite, "composite_"),):
        names = _kernels(lambda: comp(idx.permute(0, 3, 1, 2), a, feats.t()))
        assert len([n for n in names if kn in n]) == 1
