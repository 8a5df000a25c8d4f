"""add_points_features_to_volume_densities_features without a GPU: the float64 restatement (tests/volumes_ref.py) against
hand-computed cases, an independent per-point, per-corner loop, conservation and shifts, the ragged and non-finite rules
and central differences; the argument checks of the public function and of the C ABI."""
import ctypes
import math

import numpy as np
import pytest
import torch

from pointcloud_b200 import _lib
from volumes_ref import add_points_features_ref, lattice, splat_ref

_PCL_E_SHAPE, _PCL_E_ARG = -1, -2
F64 = torch.float64


def zeros(b, d, h, w, c=None):
    dens = torch.zeros(b, 1, d, h, w, dtype=F64)
    return dens if c is None else (dens, torch.zeros(b, c, d, h, w, dtype=F64))


def one_point(p, grid=(4, 4, 4), mode="trilinear", align_corners=True, feat=1.0):
    pts = torch.tensor([[p]], dtype=torch.float32)
    f, d = splat_ref(pts, torch.tensor([[[feat]]], dtype=F64), zeros(1, *grid), None, mode, align_corners=align_corners)
    return f[0, 0], d[0, 0]


def coord(i, S, align_corners=True):
    """The local coordinate of lattice position i."""
    return 2.0 * i / (S - 1) - 1.0 if align_corners else (2.0 * i + 1.0) / S - 1.0


# ---------------------------------------------------------------- hand-computed cases -------------------------------------

def test_centre_of_eight_voxels_gives_an_eighth_to_each():
    x = coord(1.5, 4)
    _, d = one_point([x, x, x])
    assert d[1:3, 1:3, 1:3].eq(0.125).all() and d.sum() == 1.0


def test_lattice_node_gives_weight_one_to_one_voxel():
    f, d = one_point([coord(1, 5), coord(2, 5), coord(3, 5)], grid=(5, 5, 5), feat=2.5)
    assert d[3, 2, 1] == 1.0 and d.sum() == 1.0                   # [z, y, x]
    assert f[3, 2, 1] == 2.5 and f.sum() == 2.5


@pytest.mark.parametrize("S", [1, 2, 5, 64])
def test_ends_of_the_range(S):
    sizes = torch.tensor([[S, S, S]])
    t = lattice(torch.tensor([[[-1.0, 1.0, 0.0]]]), sizes, True)[0, 0]
    assert t[0] == 0 and t[1] == S - 1
    t = lattice(torch.tensor([[[-1.0, 1.0, 0.0]]]), sizes, False)[0, 0]
    assert t[0] == -0.5 and t[1] == S - 0.5


def test_ends_of_the_range_vote_into_the_end_voxels():
    _, d = one_point([-1.0, 1.0, 1.0], grid=(3, 5, 7))
    assert d[2, 4, 0] == 1.0 and d.sum() == 1.0
    _, d = one_point([-1.0, 1.0, 1.0], grid=(3, 5, 7), align_corners=False)  # t = -0.5 / S - 0.5: half of each weight
    assert d[2, 4, 0] == 0.125 and d.sum() == 0.125


def test_nearest_ties_round_away_from_zero():
    # align_corners=False, S = 4: t = ((p + 1) * 4 - 1) * 0.5; the y and z coordinates -0.75 give t = 0
    for p, t, want in [(-0.5, 0.5, 1), (0.0, 1.5, 2), (0.5, 2.5, 3), (0.25, 2.0, 2), (-0.75, 0.0, 0)]:
        assert lattice(torch.tensor([[[p, 0.0, 0.0]]]), torch.tensor([[4, 4, 4]]), False)[0, 0, 0] == t
        _, d = one_point([p, -0.75, -0.75], mode="nearest", align_corners=False)
        assert d[0, 0, want] == 1.0 and d.sum() == 1.0, (p, want)       # 0.5 -> 1 and 2.5 -> 3, where half to even gives 0, 2
    # t = -0.5 rounds to -1 (away from zero) and is dropped, where torch.round would give voxel 0
    _, d = one_point([-1.0, 0.0, 0.0], mode="nearest", align_corners=False)
    assert d.sum() == 0


# ---------------------------------------------------------------- an independent loop --------------------------------------

def loop_ref(pts, feats, dens0, feat0, mode, mask, sizes, align_corners):
    B, P, C = feats.shape
    D, H, W = dens0.shape[2:]
    dens, feat = dens0.clone().numpy(), feat0.clone().numpy()
    s, o = (1, 0) if align_corners else (0, 1)
    f32 = np.float32
    for b in range(B):
        Sz = [int(sizes[b, 2]), int(sizes[b, 1]), int(sizes[b, 0])]  # W, H, D
        lim = [min(Sz[0], W), min(Sz[1], H), min(Sz[2], D)]
        for i in range(P):
            m = 1.0 if mask is None else float(mask[b, i])
            if m == 0:
                continue
            t = [float((((f32(pts[b, i, a]) + f32(1)) * f32(Sz[a] - s)) - f32(o)) * f32(0.5)) for a in range(3)]
            if mode == "nearest":
                corners = [([int(math.copysign(math.floor(abs(v) + 0.5), v)) for v in t], m)]
            else:
                fl = [math.floor(v) for v in t]
                r = [v - q for v, q in zip(t, fl)]
                corners = []
                for k in range(8):
                    d = [k & 1, (k >> 1) & 1, k >> 2]
                    wa = [r[a] if d[a] else 1 - r[a] for a in range(3)]
                    corners.append(([fl[a] + d[a] for a in range(3)], m * ((wa[2] * wa[1]) * wa[0])))
            for (x, y, z), w in corners:
                if not (0 <= x < lim[0] and 0 <= y < lim[1] and 0 <= z < lim[2]) or w == 0:
                    continue
                dens[b, 0, z, y, x] += w
                for c in range(C):
                    feat[b, c, z, y, x] += w * float(feats[b, i, c])
    return feat, dens


@pytest.mark.parametrize("mode", ["trilinear", "nearest"])
@pytest.mark.parametrize("align_corners", [True, False])
@pytest.mark.parametrize("seed", range(3))
def test_restatement_equals_an_independent_loop(mode, align_corners, seed):
    g = torch.Generator().manual_seed(seed)
    B, P, C, D, H, W = 2, 9, 3, 3, 4, 5
    pts = (torch.rand(B, P, 3, generator=g) * 2.4 - 1.2)
    feats = torch.randn(B, P, C, generator=g, dtype=F64)
    dens0, feat0 = torch.randn(B, 1, D, H, W, generator=g, dtype=F64), torch.randn(B, C, D, H, W, generator=g, dtype=F64)
    mask = (torch.rand(B, P, generator=g) > 0.3).to(F64) * torch.rand(B, P, generator=g, dtype=F64)
    sizes = torch.tensor([[3, 4, 5], [2, 5, 3]])
    f, d = splat_ref(pts, feats, dens0, feat0, mode, mask, sizes, align_corners)
    lf, ld = loop_ref(pts, feats, dens0, feat0, mode, mask, sizes, align_corners)
    assert np.array_equal(d.numpy(), ld) and np.array_equal(f.numpy(), lf)


# ---------------------------------------------------------------- conservation and shifts ----------------------------------

def test_votes_of_interior_points_sum_to_the_mask():
    g = torch.Generator().manual_seed(5)
    pts = torch.rand(3, 200, 3, generator=g) * 1.8 - 0.9           # every corner inside with align_corners
    m = torch.rand(3, 200, generator=g, dtype=F64)
    _, d = splat_ref(pts, torch.ones(3, 200, 1, dtype=F64), zeros(3, 6, 7, 8), None, mask=m)
    np.testing.assert_allclose(d.sum((1, 2, 3, 4)).numpy(), m.sum(1).numpy(), rtol=1e-13)


def test_shift_by_one_voxel_shifts_the_volume():
    g = torch.Generator().manual_seed(6)
    S = 9
    # coordinates on a 1/64 lattice in [-0.75, 0.25]: p + 2 / (S - 1) and t stay exact in fp32
    pts = torch.randint(0, 65, (1, 50, 3), generator=g).float() / 64 - 0.75
    feats = torch.rand(1, 50, 2, generator=g, dtype=F64)
    sh = pts.clone()
    sh[..., 0] += 2.0 / (S - 1)                                    # x by one voxel
    f1, d1 = splat_ref(pts, feats, zeros(1, S, S, S), None)
    f2, d2 = splat_ref(sh, feats, zeros(1, S, S, S), None)
    assert torch.equal(d2[..., 1:], d1[..., :-1]) and torch.equal(f2[..., 1:], f1[..., :-1])
    assert d2[..., 0].abs().max() == 0 and d1[..., -1].abs().max() == 0


# ---------------------------------------------------------------- ragged and edge cases ------------------------------------

def test_smaller_grid_sizes_leave_the_other_voxels_alone():
    g = torch.Generator().manual_seed(7)
    pts = torch.rand(2, 300, 3, generator=g) * 2 - 1
    dens0, feat0 = torch.randn(2, 1, 6, 6, 6, generator=g, dtype=F64), torch.randn(2, 2, 6, 6, 6, generator=g, dtype=F64)
    sizes = torch.tensor([[3, 4, 5], [6, 6, 6]])
    f, d = splat_ref(pts, torch.rand(2, 300, 2, dtype=F64), dens0, feat0, grid_sizes=sizes)
    outside = torch.ones(6, 6, 6, dtype=torch.bool)
    outside[:3, :4, :5] = False
    assert torch.equal(d[0, 0][outside], dens0[0, 0][outside]) and torch.equal(f[0][:, outside], feat0[0][:, outside])
    assert not torch.equal(d[0, 0][~outside], dens0[0, 0][~outside])
    assert d[0, 0, :3, :4, :5].sum() - dens0[0, 0, :3, :4, :5].sum() == pytest.approx(300, rel=1e-12)  # all votes inside


def test_oversize_and_zero_grid_sizes_drop_votes():
    pts = torch.tensor([[[1.0, 1.0, 1.0], [0.0, 0.0, 0.0]]] * 3)
    sizes = torch.tensor([[100, 100, 100], [0, 4, 4], [-3, 4, 4]])
    _, d = splat_ref(pts, torch.ones(3, 2, 1, dtype=F64), zeros(3, 4, 4, 4), None, grid_sizes=sizes)
    # cloud 0: t = 99 and 49.5 on every axis, beyond the padded 4 -> nothing; clouds 1, 2: D_b <= 0 -> nothing
    assert d.abs().sum() == 0


def test_masked_nan_points_are_skipped_and_unmasked_ones_add_nothing():
    pts = torch.tensor([[[float("nan"), 0.0, 0.0], [0.1, 0.2, 0.3], [float("inf"), 0.0, 0.0], [0.0, 1e30, 0.0]]])
    feats = torch.tensor([[[float("nan")], [1.0], [float("inf")], [2.0]]], dtype=F64)
    for mask in (None, torch.tensor([[0.0, 1.0, 0.0, 1.0]])):
        f, d = splat_ref(pts, feats, zeros(1, 4, 4, 4), None, mask=mask)
        _, d1 = splat_ref(pts[:, 1:2], feats[:, 1:2], zeros(1, 4, 4, 4), None)
        assert torch.isfinite(f).all() and torch.equal(d, d1)
    pg = pts.clone().requires_grad_()
    fg = feats.clone().requires_grad_()
    f, d = splat_ref(pg, fg, zeros(1, 4, 4, 4), None)
    (f.sum() + d.sum()).backward()
    assert torch.isfinite(pg.grad).all() and (pg.grad[0, [0, 2, 3]] == 0).all() and (fg.grad[0, [0, 2, 3]] == 0).all()


def test_fractional_mask_is_a_weight():
    g = torch.Generator().manual_seed(8)
    pts, feats = torch.rand(1, 40, 3, generator=g) * 2 - 1, torch.randn(1, 40, 2, generator=g, dtype=F64)
    f1, d1 = splat_ref(pts, feats, zeros(1, 5, 5, 5), None, mask=torch.full((1, 40), 0.25, dtype=F64))
    f2, d2 = splat_ref(pts, feats, zeros(1, 5, 5, 5), None)
    np.testing.assert_allclose(d1.numpy(), 0.25 * d2.numpy(), rtol=1e-14, atol=1e-16)
    np.testing.assert_allclose(f1.numpy(), 0.25 * f2.numpy(), rtol=1e-14, atol=1e-16)


def test_rescale_divides_by_the_clamped_densities():
    g = torch.Generator().manual_seed(9)
    pts, feats = torch.rand(2, 30, 3, generator=g) * 2 - 1, torch.randn(2, 30, 3, generator=g, dtype=F64)
    for mode, lo in (("trilinear", 1e-4), ("nearest", 1.0)):
        f, d = add_points_features_ref(pts, feats, zeros(2, 4, 4, 4), None, mode, rescale_features=True)
        fu, du = splat_ref(pts, feats, zeros(2, 4, 4, 4), None, mode)
        assert torch.equal(d, du) and torch.equal(f, fu / du.clamp(lo))


# ---------------------------------------------------------------- gradients ------------------------------------------------

@pytest.mark.parametrize("align_corners", [True, False])
def test_gradients_match_central_differences(align_corners):
    g = torch.Generator().manual_seed(10)
    B, P, C, S = 2, 12, 2, 5
    # keep every coordinate at least 0.1 lattice steps from a lattice plane, so that the floor is locally constant
    t = torch.randint(0, S - 1, (B, P, 3), generator=g).to(F64) + 0.1 + 0.8 * torch.rand(B, P, 3, generator=g, dtype=F64)
    s, o = (1, 0) if align_corners else (0, 1)
    pts64 = (2 * t + o) / (S - s) - 1
    feats = torch.randn(B, P, C, generator=g, dtype=F64)
    gd, gf = torch.randn(B, 1, S, S, S, generator=g, dtype=F64), torch.randn(B, C, S, S, S, generator=g, dtype=F64)

    def loss(p, f):
        vf, vd = splat_ref(p, f, zeros(B, S, S, S), None, align_corners=align_corners)
        return (vf * gf).sum() + (vd * gd).sum()

    p = pts64.float().requires_grad_()   # the restatement reads fp32 coordinates; its derivative is (S - s) / 2 exactly
    f = feats.clone().requires_grad_()
    loss(p, f).backward()
    h = 1e-3
    num = torch.zeros(B, P, 3, dtype=F64)
    for b in range(B):
        for i in range(P):
            for a in range(3):
                e = torch.zeros(B, P, 3)
                e[b, i, a] = h
                num[b, i, a] = (loss(p.detach() + e, feats) - loss(p.detach() - e, feats)) / (2 * h)
    # fp32 coordinates: the step is h up to one fp32 rounding of p +- h
    np.testing.assert_allclose(p.grad.numpy(), num.numpy(), rtol=1e-3, atol=1e-3 * float(num.abs().max()))
    numf = torch.zeros(B, P, C, dtype=F64)
    for b in range(B):
        for i in range(P):
            for c in range(C):
                e = torch.zeros(B, P, C, dtype=F64)
                e[b, i, c] = 1e-6
                numf[b, i, c] = (loss(p.detach(), feats + e) - loss(p.detach(), feats - e)) / 2e-6
    np.testing.assert_allclose(f.grad.numpy(), numf.numpy(), rtol=1e-7, atol=1e-9)


def test_nearest_mode_gives_the_points_no_gradient():
    p = (torch.rand(1, 20, 3) * 2 - 1).requires_grad_()
    f = torch.randn(1, 20, 2, dtype=F64).requires_grad_()
    vf, vd = splat_ref(p, f, zeros(1, 4, 4, 4), None, "nearest")
    (vf.sum() + vd.sum()).backward()
    assert (p.grad == 0).all() and (f.grad != 0).any()


# ---------------------------------------------------------------- argument checks ------------------------------------------

def test_public_function_raises_like_pytorch3d():
    import pointcloud_b200 as pcl
    fn = pcl.add_points_features_to_volume_densities_features
    p, f = torch.rand(2, 10, 3), torch.rand(2, 10, 4)
    dens, feat = torch.zeros(2, 1, 4, 4, 4), torch.zeros(2, 4, 4, 4, 4)
    with pytest.raises(ValueError):
        fn(torch.rand(2, 10, 2), f, dens, feat)
    with pytest.raises(ValueError, match="^Only one-dimensional densities are allowed.$"):
        fn(p, f, torch.zeros(2, 2, 4, 4, 4), feat)
    with pytest.raises(ValueError, match='^No such interpolation mode "cubic"$'):
        fn(p, f, dens, feat, mode="cubic")
    with pytest.raises(ValueError, match="Batch sizes"):
        fn(p, f, torch.zeros(3, 1, 4, 4, 4), None)
    with pytest.raises(ValueError, match="Batch sizes"):
        fn(torch.rand(3, 10, 3), f, dens, feat)
    with pytest.raises(ValueError, match="channels"):
        fn(p, f, dens, torch.zeros(2, 3, 4, 4, 4))
    with pytest.raises(ValueError, match="grid"):
        fn(p, f, dens, torch.zeros(2, 4, 4, 4, 5))
    with pytest.raises(ValueError, match="mask"):
        fn(p, f, dens, feat, mask=torch.ones(2, 9))
    with pytest.raises(ValueError, match="grid_sizes"):
        fn(p, f, dens, feat, grid_sizes=torch.ones(2, 2, dtype=torch.int64))


def _buf(n):
    b = (ctypes.c_float * n)()
    return ctypes.addressof(b), b


def test_abi_refuses_bad_arguments_without_a_device():
    L = _lib.lib()
    (p, kp), (f, kf), (o, ko) = _buf(64), _buf(64), _buf(64)
    ok = dict(B=1, P=4, C=2, D=2, H=2, W=2, mode=0, ac=1, dt=0, pp=p, fp=f)
    cases = [(dict(B=-1), _PCL_E_SHAPE), (dict(P=-1), _PCL_E_SHAPE), (dict(C=0), _PCL_E_SHAPE), (dict(D=-2), _PCL_E_SHAPE),
             (dict(B=70000), _PCL_E_SHAPE), (dict(W=(1 << 24) + 1), _PCL_E_SHAPE), (dict(mode=2), _PCL_E_ARG),
             (dict(mode=-1), _PCL_E_ARG), (dict(ac=2), _PCL_E_ARG), (dict(dt=7), _PCL_E_ARG), (dict(pp=None), _PCL_E_ARG),
             (dict(fp=None), _PCL_E_ARG)]
    for change, want in cases:
        a = dict(ok, **change)
        head = [a["pp"], a["dt"], 12, 3, a["fp"], 0, 8, 2, None, None, a["B"], a["P"], a["C"], a["D"], a["H"], a["W"],
                a["mode"], a["ac"]]
        assert L.pcl_points_to_volumes_fwd(*head, o, o, None) == want, change
        assert L.pcl_last_error()
        assert L.pcl_points_to_volumes_bwd(*head, o, o, o, o, None) == want, change
    head = [p, 0, 12, 3, f, 0, 8, 2, None, None, 1, 4, 2, 2, 2, 2, 0, 1]
    assert L.pcl_points_to_volumes_fwd(*head, None, o, None) == _PCL_E_ARG
    L.pcl_points_to_volumes_fwd(*head[:17], 5, o, o, None)
    assert b"align_corners" in L.pcl_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback_for_points_to_volumes():
    import pointcloud_b200 as pcl
    from pointcloud_b200._lib import PclError
    with pytest.raises(PclError):
        pcl.add_points_features_to_volume_densities_features(torch.rand(1, 8, 3), torch.rand(1, 8, 2),
                                                             torch.zeros(1, 1, 4, 4, 4))
    L = _lib.lib()
    (p, kp), (o, ko) = _buf(64), _buf(64)
    head = [p, 0, 12, 3, p, 0, 12, 3, None, None, 1, 4, 3, 2, 2, 2, 0, 1]
    assert L.pcl_points_to_volumes_fwd(*head, o, o, None) < 0 and L.pcl_last_error()
    assert L.pcl_points_to_volumes_bwd(*head, o, o, o, o, None) < 0 and L.pcl_last_error()
