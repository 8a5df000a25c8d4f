"""tests/icp_ref.py (the float64 restatement that specifies corresponding_points_alignment and iterative_closest_point)
against known transforms, brute force, hand-computed moments and the ICP loop's rules; the argument checks of the Python
functions and the C ABI (no launch)."""
import ctypes
import math

import numpy as np
import pytest
import torch

import pointcloud_b200 as pcl
from icp_ref import alignment_parts, alignment_ref, apply_ref, axis_angle, icp_ref, nn_dense, random_rotation
from pointcloud_b200 import _lib, synth

_PCL_E_SHAPE, _PCL_E_ARG = -1, -2


def table(b, n, seed):
    return synth.table_clouds(b, n, seed=seed)[0].double()


def uniform(b, n, seed):
    return torch.rand(b, n, 3, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


def planar(b, n, seed):
    """Table tops: z = 0.2 exactly, so M has rank 2."""
    x = uniform(b, n, seed)
    x[..., 2] = 0.2
    return x


@pytest.mark.parametrize("cloud", [table, uniform, planar])
@pytest.mark.parametrize("estimate_scale", [False, True])
def test_known_similarity_transforms_are_recovered(cloud, estimate_scale):
    g = torch.Generator().manual_seed(1)
    b = 6
    X = cloud(b, 500, 2)
    R = random_rotation(b, g)
    # rotations near 180 degrees about random axes
    axis = torch.randn(2, 3, generator=g, dtype=torch.float64)
    R[:2] = axis_angle(axis / axis.norm(dim=1, keepdim=True), torch.tensor([math.pi - 1e-7, -math.pi + 1e-4], dtype=torch.float64))
    T = torch.randn(b, 3, generator=g, dtype=torch.float64)
    s = (0.5 + torch.rand(b, generator=g, dtype=torch.float64)) if estimate_scale else torch.ones(b, dtype=torch.float64)
    Y = apply_ref(X, R, T, s)
    Rr, Tr, sr = alignment_ref(X, Y, estimate_scale=estimate_scale)
    assert (Rr - R).abs().max() < 1e-12 and (Tr - T).abs().max() < 1e-12 and (sr - s).abs().max() < 1e-12
    assert torch.allclose(torch.det(Rr), torch.ones(b, dtype=torch.float64), atol=1e-13)


def test_mirror_gives_a_reflection_only_when_allowed_and_otherwise_the_best_rotation():
    g = torch.Generator().manual_seed(3)
    X = uniform(1, 7, 4) - 0.5
    F = torch.diag(torch.tensor([1.0, 1.0, -1.0], dtype=torch.float64))[None]
    Y = torch.bmm(X, F) + 0.01 * torch.randn(1, 7, 3, generator=g, dtype=torch.float64)
    Rr, _, _ = alignment_ref(X, Y, allow_reflection=True)
    assert abs(float(torch.det(Rr)) + 1) < 1e-12
    Rp, _, _ = alignment_ref(X, Y)
    assert abs(float(torch.det(Rp)) - 1) < 1e-12
    # brute force: tr(R^T M) over a fine grid of ZYZ Euler angles never beats the proper rotation found
    M = alignment_parts(X, Y)[0][0]
    n = 72
    a = torch.linspace(-math.pi, math.pi, n, dtype=torch.float64)
    bb = torch.linspace(0, math.pi, n // 2, dtype=torch.float64)
    A, B_, C = torch.meshgrid(a, bb, a, indexing="ij")
    A, B_, C = A.reshape(-1), B_.reshape(-1), C.reshape(-1)
    ez = torch.tensor([0.0, 0.0, 1.0], dtype=torch.float64).expand(A.numel(), 3)
    ey = torch.tensor([0.0, 1.0, 0.0], dtype=torch.float64).expand(A.numel(), 3)
    Rg = torch.bmm(torch.bmm(axis_angle(ez, A), axis_angle(ey, B_)), axis_angle(ez, C))
    grid_best = float((Rg * M).sum((1, 2)).max())
    best = float((Rp[0] * M).sum())
    assert best >= grid_best - 1e-12
    assert best - grid_best < 0.02 * float(M.norm())  # the grid is fine enough to come close


def test_weights_enter_the_covariance_squared_hand_computed():
    X = torch.tensor([[[1.0, 0, 0], [0, 1, 0], [-1, 0, 0], [0, -1, 0]]], dtype=torch.float64)
    w = torch.tensor([[1.0, 1.0, 2.0, 0.0]], dtype=torch.float64)
    M, xcov, xm, ym = alignment_parts(X, X, w)
    # sum w = 4, xm = (-1/4, 1/4, 0); M = sum w^2 xc xc^T / 4 = [[62, 10], [10, 14]] / 64 (sum w xc xc^T would give 44, 4, 12)
    want = torch.tensor([[62.0, 10, 0], [10, 14, 0], [0, 0, 0]], dtype=torch.float64) / 64
    assert torch.equal(xm[0], torch.tensor([-0.25, 0.25, 0.0], dtype=torch.float64))
    assert torch.allclose(M[0], want, rtol=0, atol=1e-15) and abs(float(xcov[0]) - 76 / 64) < 1e-15


def test_constant_weights_change_nothing_and_zero_weights_remove_outliers():
    g = torch.Generator().manual_seed(5)
    b, n = 3, 200
    X = table(b, n, 6)
    Y = apply_ref(X, random_rotation(b, g, 0.3), torch.randn(b, 3, generator=g, dtype=torch.float64),
                  torch.ones(b, dtype=torch.float64)) + 0.01 * torch.randn(b, n, 3, generator=g, dtype=torch.float64)
    for est in (False, True):
        ref = alignment_ref(X, Y, estimate_scale=est)
        got = alignment_ref(X, Y, weights=torch.full((b, n), 0.37, dtype=torch.float64), estimate_scale=est)
        for r, q in zip(ref, got):
            assert torch.allclose(r, q, rtol=0, atol=1e-12)
        # 20 wild outliers with weight 0 change nothing
        Xo = torch.cat([X, 100 * torch.randn(b, 20, 3, generator=g, dtype=torch.float64)], 1)
        Yo = torch.cat([Y, 100 * torch.randn(b, 20, 3, generator=g, dtype=torch.float64)], 1)
        w = torch.cat([torch.ones(b, n), torch.zeros(b, 20)], 1).double()
        for r, q in zip(ref, alignment_ref(Xo, Yo, weights=w, estimate_scale=est)):
            assert torch.allclose(r, q, rtol=0, atol=1e-12)
        # lengths act as 0/1 weights
        for r, q in zip(alignment_ref(Xo, Yo, weights=w, estimate_scale=est),
                        alignment_ref(Xo, Yo, estimate_scale=est, lengths=torch.full((b,), n))):
            assert torch.allclose(r, q, rtol=0, atol=1e-12)


def pair(b, n, seed, angle=15, shift=0.05, noise=0.002):
    g = torch.Generator().manual_seed(seed)
    X = table(b, n, seed)
    R = random_rotation(b, g, math.radians(angle))
    T = (torch.rand(b, 3, generator=g, dtype=torch.float64) * 2 - 1) * shift
    Y = apply_ref(X, R, T, torch.ones(b, dtype=torch.float64)) + noise * torch.randn(b, n, 3, generator=g, dtype=torch.float64)
    return X, Y[:, torch.randperm(n, generator=g)], R, T


def test_init_transform_only_seeds_the_first_search():
    X, Y, R, T = pair(2, 300, 7)
    init = (R.transpose(1, 2).contiguous() * 0 + torch.eye(3, dtype=torch.float64), T * 0.5, torch.ones(2, dtype=torch.float64))
    r1 = icp_ref(X, Y, init, max_iterations=1)
    want = alignment_ref(X, nn_dense(apply_ref(X, *init), Y), weights=torch.ones(2, 300, dtype=torch.float64))
    for a, b in zip(r1["RTs"], want):
        assert torch.equal(a, b)
    r2 = icp_ref(X, Y, init, max_iterations=2)
    want2 = alignment_ref(X, nn_dense(r1["Xt"], Y), weights=torch.ones(2, 300, dtype=torch.float64))
    for a, b in zip(r2["RTs"], want2):
        assert torch.equal(a, b)          # iteration 1 aligns the original X to the neighbours of Xt, not Xt itself
    assert not torch.equal(r1["RTs"][1], icp_ref(X, Y, None, max_iterations=1)["RTs"][1])


def test_zero_iterations():
    X, Y, R, T = pair(2, 50, 8)
    r = icp_ref(X, Y, None, max_iterations=0)
    assert r["converged"] is False and r["rmse"] is None and r["t_history"] == [] and torch.equal(r["Xt"], X)
    assert torch.equal(r["RTs"][0], torch.eye(3, dtype=torch.float64).expand(2, 3, 3))
    init = (R, T, torch.full((2,), 1.5, dtype=torch.float64))
    r = icp_ref(X, Y, init, max_iterations=0)
    assert torch.equal(r["Xt"], apply_ref(X, *init)) and all(torch.equal(a, b) for a, b in zip(r["RTs"], init))


def test_exact_pairs_and_empty_clouds_never_converge():
    # symmetric axis-aligned points: M is diagonal, so the SVD, R = I and T = 0 are exact and rmse is exactly 0
    X = torch.tensor([[[1.0, 0, 0], [-1, 0, 0], [0, 2, 0], [0, -2, 0], [0, 0, 3], [0, 0, -3]]], dtype=torch.float64)
    r = icp_ref(X, X.clone(), max_iterations=7)
    assert not r["converged"] and len(r["t_history"]) == 7
    assert float(r["rmse_history"][0][0]) == 0.0 and math.isnan(float(r["rel_history"][1][0]))
    # an empty X cloud next to a converging one
    X2, Y2, _, _ = pair(2, 100, 9)
    r = icp_ref(X2, Y2, max_iterations=9, x_lengths=torch.tensor([100, 0]))
    assert not r["converged"] and len(r["t_history"]) == 9


def test_batch_stops_when_the_last_cloud_does():
    X, Y, _, _ = pair(2, 400, 10, angle=25)
    Y[1] = apply_ref(X[1:2], axis_angle(torch.tensor([[0.0, 0, 1]], dtype=torch.float64), torch.tensor([0.02], dtype=torch.float64)),
                     torch.zeros(1, 3, dtype=torch.float64), torch.ones(1, dtype=torch.float64))[0] + 0.002 * torch.randn(
        400, 3, generator=torch.Generator().manual_seed(11), dtype=torch.float64)
    alone = [len(icp_ref(X[k:k + 1], Y[k:k + 1], relative_rmse_thr=1e-4)["t_history"]) for k in range(2)]
    assert alone[0] != alone[1]
    both = icp_ref(X, Y, relative_rmse_thr=1e-4)
    assert both["converged"] and len(both["t_history"]) == max(alone)


def test_python_argument_errors_need_no_device():
    x = torch.zeros(2, 5, 3)
    with pytest.raises(ValueError, match="same number of batches, points and dimensions"):
        pcl.corresponding_points_alignment(x, torch.zeros(2, 6, 3))
    with pytest.raises(ValueError, match="weights should have the same first two dimensions"):
        pcl.corresponding_points_alignment(x, x, weights=torch.ones(2, 4))
    with pytest.raises(ValueError, match="D=2 is not supported"):
        pcl.corresponding_points_alignment(torch.zeros(2, 5, 2), torch.zeros(2, 5, 2))
    with pytest.raises(ValueError, match="same number of batches and data dimensions"):
        pcl.iterative_closest_point(x, torch.zeros(3, 5, 3))
    with pytest.raises(ValueError, match="D=4 is not supported"):
        pcl.iterative_closest_point(torch.zeros(2, 5, 4), torch.zeros(2, 7, 4))
    with pytest.raises(ValueError, match="max_iterations"):
        pcl.iterative_closest_point(x, x, max_iterations=-1)


def test_library_symbols_and_signatures():
    L = _lib.lib()
    for name in ("pcl_points_alignment_workspace_bytes", "pcl_points_alignment_fwd", "pcl_points_alignment_bwd",
                 "pcl_icp_workspace_bytes", "pcl_icp"):
        fn = getattr(L, name)
        assert fn.argtypes == _lib._SIGNATURES[name][1]
    assert len(_lib._SIGNATURES["pcl_points_alignment_fwd"][1]) == 22
    assert len(_lib._SIGNATURES["pcl_points_alignment_bwd"][1]) == 22
    assert len(_lib._SIGNATURES["pcl_icp"][1]) == 30
    assert L.pcl_points_alignment_workspace_bytes(4, 100) == 4 * 4 * 24 * 8
    assert L.pcl_icp_workspace_bytes(32, 2048, 2048, 100) >= 32 * 2048 * 4 + 32 * 64 * 24 * 8
    assert L.pcl_icp_workspace_bytes(0, 10, 10, 10) == 0


def test_abi_refuses_bad_arguments_without_a_device():
    L = _lib.lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    # negative sizes, a bad dtype, a null input
    assert L.pcl_points_alignment_fwd(p, 0, 9, 3, p, 0, 9, 3, None, None, -1, 3, 0, 0, 1e-9, p, p, p, None, None, 0, None) == _PCL_E_SHAPE
    assert L.pcl_points_alignment_fwd(p, 7, 9, 3, p, 0, 9, 3, None, None, 1, 3, 0, 0, 1e-9, p, p, p, None, None, 0, None) == _PCL_E_ARG
    assert L.pcl_points_alignment_bwd(p, 0, 9, 3, None, 0, 9, 3, None, None, 1, 3, 0, 1e-9, p, None, None, None, p, p, None, None) == _PCL_E_ARG
    # too small a workspace
    assert L.pcl_points_alignment_fwd(p, 0, 9, 3, p, 0, 9, 3, None, None, 1, 3, 0, 0, 1e-9, p, p, p, None, None, 0, None) == _PCL_E_ARG
    assert b"workspace" in L.pcl_last_error()
    icp = [p, 0, 9, 3, None, p, 0, 9, 3, None, 1, 3, 3, None, None, None, 5, 1e-6, 0, 0, 0, p, p, p, p, p, p, None, 0, None]
    for k, v, want in [(16, -1, _PCL_E_ARG), (20, 9, _PCL_E_ARG), (13, p, _PCL_E_ARG), (10, -1, _PCL_E_SHAPE), (1, 7, _PCL_E_ARG)]:
        a = list(icp)
        a[k] = v
        assert L.pcl_icp(*a) == want and L.pcl_last_error()
