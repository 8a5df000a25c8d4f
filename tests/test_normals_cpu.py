"""Normals and local frames without a GPU: the float64 restatement (tests/normals_ref.py) against geometry, numpy and
finite differences; the argument checks of the public functions and of the C ABI; the no-fallback behaviour."""
import ctypes
import math

import numpy as np
import pytest
import torch

from normals_ref import frames_ref, knn_idx
from pointcloud_b200 import _lib

_PCL_E_SHAPE, _PCL_E_ARG, _PCL_E_UNSUPPORTED = -1, -2, -5


def _unit(v):
    return v / np.linalg.norm(v)


def test_tilted_plane_gives_the_plane_normal():
    g = torch.Generator().manual_seed(0)
    nrm = torch.tensor(_unit(np.array([0.3, -0.5, 0.8])))
    a = torch.tensor(_unit(np.cross(nrm.numpy(), [1.0, 0.0, 0.0])))
    c = torch.cross(nrm, a, dim=0)
    uv = torch.rand(1, 400, 2, generator=g, dtype=torch.float64)
    pts = uv[..., :1] * a + uv[..., 1:] * c + 1e-4 * torch.randn(1, 400, 1, generator=g, dtype=torch.float64) * nrm + 0.7
    for K in (8, 30):
        curv, frames = frames_ref(pts, knn_idx(pts, K), disambiguate=False)
        assert ((frames[0, :, :, 0] @ nrm).abs() > 1 - 1e-4).all()
        assert (curv[0, :, 0] < 1e-3 * curv[0, :, 1]).all()


@pytest.mark.parametrize("K", [20, 40, 64])
def test_sphere_normals_point_inwards_after_disambiguation(K):
    g = torch.Generator().manual_seed(1)
    d = torch.randn(1, 3000, 3, generator=g, dtype=torch.float64)
    radial = d / d.norm(dim=2, keepdim=True)
    pts = 0.5 * radial + torch.tensor([0.1, 0.2, 0.3], dtype=torch.float64)
    _, frames = frames_ref(pts, knn_idx(pts, K))
    # Every neighbour lies on the sphere, so it projects <= 0 on the outward radius at p_i, and the normal is flipped to
    # -radial.  The normal is the radius at the neighbourhood's mean, not at p_i; with few neighbours (K = 12 here) an
    # off-centre p_i can see more than half of them above that plane, and K = 3 is exactly planar.
    cos = (frames[0, :, :, 0] * radial[0]).sum(1)
    assert (cos < -0.99).all()


def test_eigenvalues_match_numpy_cov():
    g = np.random.default_rng(2)
    pts = torch.tensor(g.random((2, 90, 3)))
    K = 12
    idx = knn_idx(pts, K)
    curv, frames = frames_ref(pts, idx, disambiguate=False)
    for b in range(2):
        for i in range(0, 90, 7):
            c = np.cov(pts[b, idx[b, i]].numpy().T, bias=True)
            np.testing.assert_allclose(curv[b, i].numpy(), np.linalg.eigvalsh(c), rtol=1e-10, atol=1e-15)
            v = frames[b, i].numpy()
            np.testing.assert_allclose(c @ v, v * curv[b, i].numpy(), atol=1e-13)


def test_rotation_equivariance_and_translation_invariance():
    g = np.random.default_rng(3)
    pts = torch.tensor(g.random((2, 120, 3)) * [1.0, 0.5, 0.2])
    K = 10
    idx = knn_idx(pts, K)
    q, _ = np.linalg.qr(g.standard_normal((3, 3)))
    q *= np.sign(np.linalg.det(q))                       # a proper rotation: the cross product keeps its sign
    R = torch.tensor(q)
    curv, frames = frames_ref(pts, idx)
    curv_r, frames_r = frames_ref(pts @ R.T, idx)
    np.testing.assert_allclose(curv_r.numpy(), curv.numpy(), rtol=1e-9, atol=1e-15)
    np.testing.assert_allclose(frames_r.numpy(), (R @ frames).numpy(), atol=1e-9)
    curv_t, frames_t = frames_ref(pts + torch.tensor([3.0, -2.0, 0.5], dtype=torch.float64), idx)
    np.testing.assert_allclose(curv_t.numpy(), curv.numpy(), rtol=1e-6, atol=1e-14)
    np.testing.assert_allclose(frames_t.numpy(), frames.numpy(), atol=1e-7)


@pytest.mark.parametrize("disambiguate", [False, True])
def test_gradients_match_central_differences(disambiguate):
    g = torch.Generator().manual_seed(4)
    pts = torch.rand(2, 24, 3, generator=g, dtype=torch.float64) * torch.tensor([1.0, 0.6, 0.3], dtype=torch.float64)
    K = 6
    lengths = torch.tensor([24, 17])
    idx = knn_idx(pts, K, lengths)
    wc = torch.randn(2, 24, 3, generator=g, dtype=torch.float64)
    wf = torch.randn(2, 24, 3, 3, generator=g, dtype=torch.float64)

    def f(x):
        c, fr = frames_ref(x, idx, lengths, disambiguate)
        return (c * wc).sum() + (fr * wf).sum()

    x = pts.clone().requires_grad_()
    (grad,) = torch.autograd.grad(f(x), x)
    num = torch.zeros_like(pts)
    h = 1e-6
    for b in range(2):
        for i in range(24):
            for c in range(3):
                e = torch.zeros_like(pts)
                e[b, i, c] = h
                num[b, i, c] = (f(pts + e) - f(pts - e)) / (2 * h)
    np.testing.assert_allclose(grad.numpy(), num.numpy(), rtol=1e-5, atol=1e-6 * float(num.abs().max()))
    assert (grad[1, 17:] == 0).all()                     # padded rows are nobody's neighbour


def test_public_functions_raise_like_pytorch3d():
    import pointcloud_b200 as pcl
    kmax = _lib.lib().pcl_knn_max_k()
    x = torch.rand(2, 80, 3)
    for fn in (pcl.estimate_pointcloud_normals, pcl.estimate_pointcloud_local_coord_frames):
        with pytest.raises(ValueError, match="shape \\(minibatch, N, 3\\)"):
            fn(torch.rand(2, 80, 2))
        with pytest.raises(ValueError, match="shape \\(minibatch, N, 3\\)"):
            fn(torch.rand(80, 3))
        for K in (0, kmax + 1, 2.5, True):
            with pytest.raises(ValueError, match="neighborhood_size"):
                fn(x, K)
        with pytest.raises(ValueError, match="has to be >= size"):
            fn(torch.rand(2, 50, 3), 50)                 # P == K: no room for K neighbours besides the point
        with pytest.raises(ValueError, match="has to be >= size"):
            fn(x, 16, lengths=torch.tensor([80, 16]))
        with pytest.raises(ValueError, match="has to be >= size"):
            fn(x, 16, lengths=torch.tensor([0, 80]))
        with pytest.raises(ValueError, match="lengths"):
            fn(x, 16, lengths=torch.tensor([80]))


def _pts():
    buf = (ctypes.c_float * 64)()
    return [ctypes.addressof(buf), 0, 3 * 4, 3], buf


def test_abi_refuses_bad_arguments_without_a_device():
    L = _lib.lib()
    (p, dt, bs, rs), keep = _pts()
    idx = (ctypes.c_int * 64)(); out = (ctypes.c_float * 64)(); fr = (ctypes.c_float * 64)()
    ai, ao, af = ctypes.addressof(idx), ctypes.addressof(out), ctypes.addressof(fr)
    for (B, P, K, dtype, pp, ii), want in [((1, 4, 0, dt, p, ai), _PCL_E_SHAPE), ((1, 4, L.pcl_knn_max_k() + 1, dt, p, ai), _PCL_E_UNSUPPORTED),
                                           ((-1, 4, 2, dt, p, ai), _PCL_E_SHAPE), ((1, -4, 2, dt, p, ai), _PCL_E_SHAPE),
                                           ((70000, 4, 2, dt, p, ai), _PCL_E_SHAPE), ((1, 4, 2, 7, p, ai), _PCL_E_ARG),
                                           ((1, 4, 2, dt, None, ai), _PCL_E_ARG), ((1, 4, 2, dt, p, None), _PCL_E_ARG)]:
        rc = L.pcl_frames_fwd(pp, dtype, bs, rs, None, B, P, K, 1, ii, ao, af, None)
        assert rc == want and L.pcl_last_error()
        rc = L.pcl_frames_bwd(pp, dtype, bs, rs, None, B, P, K, ii, ao, af, ao, af, ao, None)
        assert rc == want and L.pcl_last_error()
    assert L.pcl_frames_fwd(p, dt, bs, rs, None, 1, 4, 2, 1, ai, None, af, None) == _PCL_E_ARG
    assert L.pcl_frames_bwd(p, dt, bs, rs, None, 1, 4, 2, ai, ao, af, None, None, None, None) == _PCL_E_ARG
    L.pcl_frames_fwd(p, dt, bs, rs, None, 1, 4, 0, 1, ai, ao, af, None)
    assert b"K=0" in L.pcl_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback_for_normals():
    import pointcloud_b200 as pcl
    from pointcloud_b200._lib import PclError
    with pytest.raises(PclError):
        pcl.estimate_pointcloud_normals(torch.rand(1, 64, 3), 8)
    with pytest.raises(PclError):
        pcl.estimate_pointcloud_local_coord_frames(torch.rand(1, 64, 3), 8, lengths=torch.tensor([40]))
    L = _lib.lib()
    (p, dt, bs, rs), keep = _pts()
    idx = (ctypes.c_int * 64)(); out = (ctypes.c_float * 64)()
    rc = L.pcl_frames_fwd(p, dt, bs, rs, None, 1, 4, 2, 1, ctypes.addressof(idx), ctypes.addressof(out), ctypes.addressof(out), None)
    assert rc < 0 and L.pcl_last_error()
    rc = L.pcl_frames_bwd(p, dt, bs, rs, None, 1, 4, 2, ctypes.addressof(idx), ctypes.addressof(out), ctypes.addressof(out),
                          None, ctypes.addressof(out), ctypes.addressof(out), None)
    assert rc < 0 and L.pcl_last_error()
