"""add_points_features_to_volume_densities_features on the GPU against tests/volumes_ref.py (float64), plus the exact cases,
input forms, non-finite inputs, stale state, graph capture, the launch count and host synchronisation.

Forward bound.  Let u = 2^-24 and n the number of votes a voxel receives (counted by the restatement).  A vote's value is
w * f with w = m * ((wz * wy) * wx): the kernel forms t exactly as the restatement does; on each axis the factor an
in-bounds corner uses is rounded at most once (r = t - floor(t) is exact for t >= 0 and rounded once for t in (-1, 0), where
only the corner that uses r is in bounds; 1 - r is rounded once); then wz * wy, * wx, m * and * f are rounded once each.  So a
feature vote carries a relative error of at most gamma_7 = 7u / (1 - 7u) (a density vote gamma_6; with m = 1, m * is exact).  The voxel's value is v0 plus n such votes added in some order
in fp32: gamma_n (|v0| + sum |w f|) more.  red.global.add flushes a subnormal operand or result to zero, at most 2^-126 per
addition.  So
    |got - ref| <= gamma_(n+7) (|v0| + sum |w f|) + n 2^-126,
with gamma_k = k u / (1 - k u); a voxel with n = 0 is untouched and exact.  Nearest-mode densities under a binary mask with
zero initial values are integer counts below 2^24 and must be exact.  Masks are used as weights: the cases include
fractional masks and integer masks with values above 1.

Backward bound.  grad_point_features[c] = sum_k w_k gf[c, v_k] over at most 8 corners in a fixed order: each term carries
the weight's gamma_6 and the product's u, the sum gamma_8, so gamma_15 sum_k |w_k gf[c, v_k]|.  grad_points[a] sums, per
corner, gd + sum_c f[c] gf[c, v_k] (C + 1 terms, gamma_(C+1)), multiplies by dw_k/dt_a = +-m (wa wb) (four roundings with the
two factors) and sums over 8 corners before the final product with (S - s)/2 (one rounding; the halving is exact):
within gamma_(C+15) (S - s)/2 |m| sum_k (|gd| + sum_c |f gf|).
The test allows gamma_(C+20) of that scale.  The backward uses no atomics, so it is bit-identical run to run and a cloud's
gradients do not depend on the rest of the batch."""
import numpy as np
import pytest
import torch

import pointcloud_b200 as pcl
from helpers import npy, same_bits
from pointcloud_b200 import _lib, synth
from test_stale_state_gpu import PATTERNS, Stale, capture_and_replay
from volumes_ref import splat_ref, votes

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
F64 = torch.float64


def gamma(k):
    return k * U / (1 - k * U)


def cloud(b, p, seed, scale=1.0):
    """Table-shaped clouds scaled from [0, 1] into [-scale, scale] (uniform noise for tiny P)."""
    if p < 64:
        return (torch.rand(b, p, 3, generator=torch.Generator().manual_seed(seed)) * 2 - 1) * scale
    return (synth.table_clouds(b, p, seed=seed)[0] * 2 - 1) * scale


def case(B, P, grid, C, seed, sizes=None, ragged=False, scale=1.1):
    g = torch.Generator().manual_seed(seed)
    pts = cloud(B, P, seed, scale).cuda()
    feats = torch.randn(B, P, C, generator=g).cuda()
    dens0 = torch.rand(B, 1, *grid, generator=g).cuda()
    feat0 = torch.randn(B, C, *grid, generator=g).cuda()
    mask = None
    if ragged:  # True: bool lengths mask; "frac": fractional weights; "int": integer weights 0..3
        n = torch.randint(0, P + 1, (B,), generator=g)
        n[-1] = P
        mask = torch.arange(P)[None] < n[:, None]
        if ragged == "frac":
            mask = mask * torch.rand(B, P, generator=g)
        elif ragged == "int":
            mask = mask * torch.randint(0, 4, (B, P), generator=g)
        mask = mask.cuda()
    gs = None
    if sizes is not None:
        pad = torch.tensor(grid)
        gs = torch.stack([torch.randint(1, int(s) + 3, (B,), generator=g) for s in pad], 1)
        gs[0] = pad
        if B > 2:
            gs[1, 0] = 0
        gs = gs if sizes == "cpu" else gs.cuda()
    return pts, feats, dens0, feat0, mask, gs


def check_forward(out, pts, feats, dens0, feat0, mode, mask, gs, align_corners):
    rf, rd, n, af, ad = splat_ref(pts, feats.float(), dens0, feat0, mode, mask, gs, align_corners, stats=True)
    for got, ref, a in ((out["densities"], rd, ad), (out["features"], rf, af)):
        bound = gamma(n + 7) * a + n * 2.0 ** -126
        err = (got.to(F64) - ref).abs()
        assert got.dtype == torch.float32 and got.shape == ref.shape
        bad = ~(err <= bound)
        assert not bad.any(), f"{int(bad.sum())} voxels off, worst {float((err - bound)[bad].max()):.3g} over the bound"
    return rf, rd


FWD = [  # B, P, grid (D, H, W), C, grid_sizes, ragged mask
    (1, 1, (1, 1, 1), 1, None, False),
    (3, 1000, (8, 9, 10), 4, "cpu", True),
    (3, 5000, (16, 16, 16), 17, "cuda", True),
    (32, 2048, (32, 32, 32), 3, None, True),
    (32, 2048, (20, 24, 28), 64, "cuda", True),
    (3, 4096, (64, 32, 16), 1, "cpu", False),
    (3, 3000, (12, 10, 8), 5, "cuda", "frac"),
    (32, 2048, (32, 32, 32), 4, None, "int"),
    (1, 262144, (128, 128, 128), 3, None, False),
]


@pytest.mark.parametrize("mode", ["trilinear", "nearest"])
@pytest.mark.parametrize("align_corners", [True, False])
@pytest.mark.parametrize("B,P,grid,C,sizes,ragged", FWD)
def test_forward_within_the_bound(B, P, grid, C, sizes, ragged, mode, align_corners):
    pts, feats, dens0, feat0, mask, gs = case(B, P, grid, C, B * P + C, sizes, ragged)
    out = pcl.points_to_volumes_forward_raw(pts, feats, dens0, feat0, mode, mask, gs, align_corners)
    check_forward(out, pts, feats, dens0, feat0, mode, mask, gs, align_corners)


# ---------------------------------------------------------------- exact results ------------------------------------------

def exact_case(B, P, S, C, seed):
    """Points on a quarter-lattice-step grid inside the volume and small integer features: every weight is a multiple of
    1/64 and every voxel sum is exact in fp32, whatever the order of the reductions."""
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, 4 * (S - 1) + 1, (B, P, 3), generator=g).float() / 4
    pts = (2 * t / (S - 1) - 1).cuda()                              # align_corners=True: t = (p + 1) (S - 1) / 2 exactly
    feats = torch.randint(-8, 9, (B, P, C), generator=g).float().cuda()
    return pts, feats


@pytest.mark.parametrize("mode", ["trilinear", "nearest"])
def test_exact_sums_and_the_rescale_bit_for_bit(mode):
    B, P, S, C = 4, 3000, 9, 5
    pts, feats = exact_case(B, P, S, C, 1)
    mask = (torch.rand(B, P, generator=torch.Generator().manual_seed(2)) > 0.2).cuda()
    dens0 = torch.zeros(B, 1, S, S, S, device="cuda")
    raw = pcl.points_to_volumes_forward_raw(pts, feats, dens0, None, mode, mask)
    rf, rd = splat_ref(pts, feats, dens0, None, mode, mask)
    assert torch.equal(raw["densities"].to(F64), rd) and torch.equal(raw["features"].to(F64), rf)
    f, d = pcl.add_points_features_to_volume_densities_features(pts, feats, dens0, None, mode, min_weight=0.01, mask=mask)
    assert same_bits(npy(d), npy(raw["densities"]))
    lo = 0.01 if mode == "trilinear" else 1.0
    assert same_bits(npy(f), npy(raw["features"] / raw["densities"].clamp(lo)))


def test_nearest_densities_are_exact_counts():
    pts, feats, _, _, mask, gs = case(32, 2048, (32, 32, 32), 3, 3, "cuda", True)
    dens0 = torch.zeros(32, 1, 32, 32, 32, device="cuda")
    out = pcl.points_to_volumes_forward_raw(pts, feats, dens0, None, "nearest", mask, gs)
    _, rd = splat_ref(pts, feats, dens0, None, "nearest", mask, gs)
    assert torch.equal(out["densities"].to(F64), rd) and float(rd.sum()) > 1000


# ---------------------------------------------------------------- input forms ---------------------------------------------

@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float64])
def test_half_and_double_inputs(dtype):
    pts, feats, dens0, feat0, mask, gs = case(3, 3000, (12, 10, 8), 4, 4, "cuda", True)
    p, f = pts.to(dtype), feats.to(dtype)
    out = pcl.points_to_volumes_forward_raw(p, f, dens0, feat0, "trilinear", mask, gs)
    check_forward(out, p.float(), f.float(), dens0, feat0, "trilinear", mask, gs, True)


def test_strided_views_noncontiguous_volumes_and_no_features():
    B, P, C = 3, 2000, 3
    buf = torch.cat([cloud(B, P, 5), torch.randn(B, P, C)], 2).cuda()  # (B, P, 6): xyz + rgb
    pts, feats = buf[:, :, :3], buf[:, :, 3:]
    dens_t = torch.rand(B, 1, 10, 12, 14, device="cuda").transpose(2, 4)  # non-contiguous (B, 1, 14, 12, 10)
    feat_t = torch.randn(B, 14, 12, 10, C, device="cuda").permute(0, 4, 1, 2, 3)
    keep = (dens_t.clone(), feat_t.clone())
    out = pcl.points_to_volumes_forward_raw(pts, feats, dens_t, feat_t)
    check_forward(out, pts, feats, dens_t, feat_t, "trilinear", None, None, True)
    assert same_bits(npy(dens_t), npy(keep[0])) and same_bits(npy(feat_t), npy(keep[1]))  # initial volumes untouched
    out = pcl.points_to_volumes_forward_raw(pts, feats, dens_t, None, "nearest")
    check_forward(out, pts, feats, dens_t, None, "nearest", None, None, True)
    f, d = pcl.add_points_features_to_volume_densities_features(pts, feats, dens_t, feat_t)
    assert d.is_contiguous() and f.shape == (B, C, 14, 12, 10) and same_bits(npy(dens_t), npy(keep[0]))


def test_empty_batch_points_and_grid():
    for B, P, grid in ((0, 5, (4, 4, 4)), (2, 0, (4, 4, 4)), (2, 5, (0, 4, 4))):
        d0 = torch.rand(B, 1, *grid, device="cuda")
        out = pcl.points_to_volumes_forward_raw(torch.rand(B, P, 3, device="cuda"), torch.rand(B, P, 2, device="cuda"), d0)
        assert torch.equal(out["densities"], d0) and out["features"].shape == (B, 2, *grid) and not out["features"].any()


# ---------------------------------------------------------------- non-finite inputs ---------------------------------------

def test_nan_points_change_nothing_and_nonfinite_features_reach_their_voxels():
    B, P, S, C = 2, 500, 9, 3
    pts, feats = exact_case(B, P, S, C, 6)
    dens0 = torch.zeros(B, 1, S, S, S, device="cuda")
    base = pcl.points_to_volumes_forward_raw(pts, feats, dens0)
    p2 = torch.cat([pts, torch.tensor([[[float("nan"), 0.0, 0.0]], [[0.0, float("inf"), 0.0]]], device="cuda")], 1)
    f2 = torch.cat([feats, torch.full((B, 1, C), 3.0, device="cuda")], 1)
    for mask in (None, torch.cat([torch.ones(B, P), torch.zeros(B, 1)], 1).cuda()):
        out = pcl.points_to_volumes_forward_raw(p2, f2, dens0, None, "trilinear", mask)
        assert torch.equal(out["densities"], base["densities"]) and torch.equal(out["features"], base["features"])
    # a masked point with NaN features is skipped entirely
    f3 = torch.cat([feats, torch.full((B, 1, C), float("nan"), device="cuda")], 1)
    out = pcl.points_to_volumes_forward_raw(torch.cat([pts, pts[:, :1]], 1), f3, dens0, None, "trilinear",
                                            torch.cat([torch.ones(B, P), torch.zeros(B, 1)], 1).cuda())
    assert torch.equal(out["features"], base["features"])
    # an inf feature on a point with t = (2, 3.5, 4.25): x on a lattice plane, so only 4 of its 8 corners have weight
    t = torch.tensor([2.0, 3.5, 4.25])
    q = (2 * t / (S - 1) - 1).cuda().view(1, 1, 3).expand(B, 1, 3)
    f4 = torch.cat([feats, torch.tensor([float("inf"), 1.0, 1.0], device="cuda").expand(B, 1, C)], 1)
    out = pcl.points_to_volumes_forward_raw(torch.cat([pts, q], 1), f4, dens0)
    alone = pcl.points_to_volumes_forward_raw(q[:, :, :], torch.ones(B, 1, 1, device="cuda"), dens0)["densities"][:, 0]
    assert int((alone > 0).sum()) == 8                             # 4 voxels per cloud
    assert torch.equal(~torch.isfinite(out["features"][:, 0]), alone > 0)
    assert torch.isfinite(out["features"][:, 1:]).all() and torch.isfinite(out["densities"]).all()


# ---------------------------------------------------------------- backward -----------------------------------------------

def grads(pts, feats, dens0, feat0, mode, mask, gs, ac, gd, gf, fn=None):
    """(grad points, grad features, grad dens0, grad feat0) of <vf, gf> + <vd, gd> through the public function (or fn)."""
    p = pts.detach().clone().requires_grad_()
    f = feats.detach().clone().requires_grad_()
    d0 = dens0.detach().clone().requires_grad_()
    f0 = feat0.detach().clone().requires_grad_()
    fn = fn or (lambda *a: pcl.add_points_features_to_volume_densities_features(
        a[0], a[1], a[2], a[3], mode, mask=mask, grid_sizes=gs, rescale_features=False, align_corners=ac))
    vf, vd = fn(p, f, d0, f0)
    loss = 0
    if gf is not None:
        loss = loss + (vf * gf).sum()
    if gd is not None:
        loss = loss + (vd * gd).sum()
    loss.backward()
    return p.grad, f.grad, d0.grad, f0.grad


@pytest.mark.parametrize("mode", ["trilinear", "nearest"])
@pytest.mark.parametrize("use", ["both", "features", "densities"])
@pytest.mark.parametrize("B,P,grid,C,sizes,ac,mk", [(3, 3000, (16, 12, 10), 4, "cuda", True, True),
                                                    (2, 700, (8, 8, 8), 17, "cpu", False, True),
                                                    (32, 2048, (32, 32, 32), 3, None, True, True),
                                                    (3, 3000, (16, 12, 10), 4, "cuda", True, "frac"),
                                                    (2, 700, (8, 8, 8), 6, None, False, "int")])
def test_backward_against_the_restatement(B, P, grid, C, sizes, ac, mk, use, mode):
    pts, feats, dens0, feat0, mask, gs = case(B, P, grid, C, 7 + C, sizes, mk)
    g = torch.Generator().manual_seed(8)
    gd = torch.randn(B, 1, *grid, generator=g).cuda() if use != "features" else None
    gf = torch.randn(B, C, *grid, generator=g).cuda() if use != "densities" else None
    gp, gpf, gd0, gf0 = grads(pts, feats, dens0, feat0, mode, mask, gs, ac, gd, gf)
    rp, rpf, _, _ = grads(pts.double(), feats.double(), dens0.double(), feat0.double(), mode, mask, gs, ac,
                          None if gd is None else gd.double(), None if gf is None else gf.double(),
                          fn=lambda a, b_, c, d: splat_ref(a, b_, c, d, mode, mask, gs, ac))
    rp = torch.zeros(B, P, 3, dtype=F64, device="cuda") if rp is None else rp      # outputs the loss does not depend on
    rpf = torch.zeros(B, P, C, dtype=F64, device="cuda") if rpf is None else rpf
    assert gp.dtype == pts.dtype and gpf.dtype == feats.dtype
    assert (gd0 is None) == (gd is None) and (gd is None or torch.equal(gd0, gd))
    assert (gf0 is None) == (gf is None) and (gf is None or torch.equal(gf0, gf))
    # bound scales from the votes (every in-bounds corner of nonzero weight)
    sizes_t = (torch.tensor(grid).expand(B, 3) if gs is None else gs.cpu()).cuda()
    bb, ii, x, y, z, w, valid = votes(pts, mask, sizes_t, grid, mode, ac)
    bb, ii, x, y, z, w = (a[valid] for a in (bb, ii, x, y, z, w))
    gdv = torch.zeros_like(w) if gd is None else gd.double()[bb, 0, z, y, x].abs()
    gfv = torch.zeros(w.shape[0], C, dtype=F64, device="cuda") if gf is None else gf.double()[bb, :, z, y, x].abs()
    sf = torch.zeros(B, P, C, dtype=F64, device="cuda").index_put_((bb, ii), w.detach().abs()[:, None] * gfv, accumulate=True)
    assert not ((gpf.double() - rpf).abs() > gamma(15) * sf + 1e-40).any()
    if mode == "nearest":
        assert not gp.any()
        return
    m = 1.0 if mask is None else mask.double()[bb, ii]
    acc = (gdv + (feats.double()[bb, ii].abs() * gfv).sum(1)) * abs(m)
    sp = torch.zeros(B, P, dtype=F64, device="cuda").index_put_((bb, ii), acc, accumulate=True)
    half = ((sizes_t.flip(1) - (1 if ac else 0)).double() / 2)[:, None, :]
    bound = gamma(C + 20) * half * sp[..., None] + 1e-40
    err = (gp.double() - rp).abs()
    assert not (err > bound).any(), float((err - bound).max())
    assert float(rp.abs().max()) > 0


def test_backward_is_bit_identical_and_independent_of_the_batch():
    B, P, grid, C = 32, 2048, (32, 32, 32), 5
    pts, feats, dens0, feat0, mask, gs = case(B, P, grid, C, 9, "cuda", True)
    g = torch.Generator().manual_seed(10)
    gd, gf = torch.randn(B, 1, *grid, generator=g).cuda(), torch.randn(B, C, *grid, generator=g).cuda()
    a = grads(pts, feats, dens0, feat0, "trilinear", mask, gs, True, gd, gf)
    b = grads(pts, feats, dens0, feat0, "trilinear", mask, gs, True, gd, gf)
    assert same_bits(npy(a[0]), npy(b[0])) and same_bits(npy(a[1]), npy(b[1]))
    k = B - 1                                                        # the full cloud of the ragged batch
    sl = slice(k, k + 1)
    c = grads(pts[sl], feats[sl], dens0[sl], feat0[sl], "trilinear", mask[sl], gs[sl], True, gd[sl], gf[sl])
    assert same_bits(npy(c[0]), npy(a[0][sl])) and same_bits(npy(c[1]), npy(a[1][sl]))


def test_backward_sees_in_place_changes_of_the_inputs():
    pts, feats, dens0, feat0, _, _ = case(2, 100, (4, 4, 4), 2, 11)
    q = pts.clone().requires_grad_()
    x = q * 1
    f, d = pcl.add_points_features_to_volume_densities_features(x, feats, dens0, feat0)
    with torch.no_grad():
        x.add_(1)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        (f.sum() + d.sum()).backward()


# ---------------------------------------------------------------- stale state and graphs ---------------------------------

def test_stale_outputs_and_shared_memory():
    st = Stale()
    L = st.L
    B, P, grid, C = 3, 5000, (16, 12, 10), 5
    pts, feats, dens0, feat0, mask, gs = case(B, P, grid, C, 12, "cuda", True)
    m = mask.float()
    A = _lib.pts_args
    D, H, W = grid
    for mode in (0, 1):
        name = ("trilinear", "nearest")[mode]
        dens, feat = torch.empty_like(dens0), torch.empty_like(feat0)

        def fwd(q):
            dens.copy_(dens0)
            feat.copy_(feat0)
            return L.pcl_points_to_volumes_fwd(*A(pts), *A(feats), m.data_ptr(), gs.data_ptr(), B, P, C, D, H, W, mode, 1,
                                               dens.data_ptr(), feat.data_ptr(), q)

        def within(o):
            try:
                check_forward(dict(densities=torch.from_numpy(o[0]).cuda(), features=torch.from_numpy(o[1]).cuda()),
                              pts, feats, dens0, feat0, name, mask, gs, True)
                return True
            except AssertionError:
                return False
        st.run(PATTERNS, [dens, feat], [], fwd, loose=(0, 1), check=within)
        g = torch.Generator().manual_seed(13)
        gd, gf = torch.randn(B, 1, *grid, generator=g).cuda(), torch.randn(B, C, *grid, generator=g).cuda()
        gp, gpf = torch.empty(B, P, 3, device="cuda"), torch.empty(B, P, C, device="cuda")
        eager = grads(pts, feats, dens0, feat0, name, mask, gs, True, gd, gf)
        st.run(PATTERNS, [gp, gpf], [], lambda q: L.pcl_points_to_volumes_bwd(
            *A(pts), *A(feats), m.data_ptr(), gs.data_ptr(), B, P, C, D, H, W, mode, 1, gd.data_ptr(), gf.data_ptr(),
            gp.data_ptr(), gpf.data_ptr(), q),
            check=lambda o: same_bits(o[0], npy(eager[0])) and same_bits(o[1], npy(eager[1])))


def test_graph_capture_and_replay():
    L = _lib.lib()
    B, P, grid, C = 4, 3000, (16, 16, 16), 3
    pts, feats, dens0, feat0, mask, gs = case(B, P, grid, C, 14, "cuda", True)
    new = case(B, P, grid, C, 15, "cuda", True)
    m = mask.float()
    A = _lib.pts_args
    D, H, W = grid
    dens, feat = torch.empty_like(dens0), torch.empty_like(feat0)

    def fwd(q):
        dens.copy_(dens0)
        feat.copy_(feat0)
        return L.pcl_points_to_volumes_fwd(*A(pts), *A(feats), m.data_ptr(), gs.data_ptr(), B, P, C, D, H, W, 0, 1,
                                           dens.data_ptr(), feat.data_ptr(), q)
    capture_and_replay([pts, feats], [new[0], new[1]], [dens, feat], fwd, loose=(0, 1))
    gd, gf = torch.randn(B, 1, *grid, device="cuda"), torch.randn(B, C, *grid, device="cuda")
    gp, gpf = torch.empty(B, P, 3, device="cuda"), torch.empty(B, P, C, device="cuda")
    capture_and_replay([pts, feats, gd], [new[0], new[1], torch.randn(B, 1, *grid, device="cuda")], [gp, gpf],
                       lambda q: L.pcl_points_to_volumes_bwd(*A(pts), *A(feats), m.data_ptr(), gs.data_ptr(), B, P, C, D, H,
                                                             W, 0, 1, gd.data_ptr(), gf.data_ptr(), gp.data_ptr(),
                                                             gpf.data_ptr(), q))
    # the public forward + rescale as one graph, on inputs whose every voxel sum is exact in fp32 (dyadic weights times
    # small integers, so the order of the reductions cannot matter): the replay must equal an eager call bit for bit
    S = 9
    pts, feats = exact_case(B, P, S, C, 17)
    new_pts, _ = exact_case(B, P, S, C, 18)
    dens0, feat0 = torch.zeros(B, 1, S, S, S, device="cuda"), torch.zeros(B, C, S, S, S, device="cuda")
    mask = torch.randint(0, 3, (B, P), generator=torch.Generator().manual_seed(19)).cuda()
    gs = torch.tensor([[9, 9, 9], [5, 9, 5], [9, 5, 9], [5, 5, 5]]).cuda()  # S - 1 in {8, 4}: weights stay multiples of 2^-9
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    fn = pcl.add_points_features_to_volume_densities_features
    with torch.cuda.stream(s):
        fn(pts, feats, dens0, feat0, mask=mask, grid_sizes=gs)
    s.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        f, d = fn(pts, feats, dens0, feat0, mask=mask, grid_sizes=gs)
    pts.copy_(new_pts)
    graph.replay()
    torch.cuda.synchronize()
    ef, ed = fn(new_pts, feats, dens0, feat0, mask=mask, grid_sizes=gs)
    assert same_bits(npy(d), npy(ed)) and same_bits(npy(f), npy(ef))
    _, rd = splat_ref(new_pts, feats, dens0, feat0, "trilinear", mask, gs, True)
    assert torch.equal(d.to(F64), rd) and float(rd.sum()) > 0


def test_one_library_kernel_each_way_and_no_host_synchronisation():
    from torch.profiler import ProfilerActivity, profile
    B, P, grid, C = 4, 3000, (16, 16, 16), 3
    pts, feats, dens0, feat0, mask, gs = case(B, P, grid, C, 16, "cuda", True)
    p = pts.clone().requires_grad_()
    fn = pcl.add_points_features_to_volume_densities_features
    for gsz in (None, gs):
        f, d = fn(p, feats, dens0, feat0, mask=mask, grid_sizes=gsz)       # warm-up
        (f.sum() + d.sum()).backward()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            f, d = fn(p, feats, dens0, feat0, mask=mask, grid_sizes=gsz)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        assert len([n for n in names if "p2v_" in n]) == 1 and any("p2v_fwd_kernel" in n for n in names), names
        loss = f.sum() + d.sum()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            loss.backward()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        assert len([n for n in names if "p2v_" in n]) == 1 and any("p2v_bwd_kernel" in n for n in names), names
        torch.cuda.set_sync_debug_mode("error")
        try:
            f, d = fn(p, feats, dens0, feat0, mask=mask, grid_sizes=gsz)
            (f.sum() + d.sum()).backward()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        torch.cuda.synchronize()
