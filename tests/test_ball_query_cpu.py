"""Ball query without a GPU: the CPU oracle (tests/ball_query_oracle.c) against a numpy restatement and against the kNN
oracle, the argument checks of the C ABI and of pointcloud_b200.ball_query, and the no-fallback behaviour."""
import ctypes

import numpy as np
import pytest
import torch

import ball_query_oracle as bo
from pointcloud_b200 import _lib

_PCL_E_SHAPE, _PCL_E_ARG, _PCL_E_UNSUPPORTED = -1, -2, -5


def _same(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


def _check_oracle(p1, p2, K, r2, l1=None, l2=None):
    d, i = bo.ball_query_forward(p1, p2, K, r2, l1, l2)
    dn, inn = bo.ball_query_numpy(p1, p2, K, r2, l1, l2)
    assert _same(d, dn) and np.array_equal(i, inn)
    for mode in (0, 1):
        dm, im = bo.ball_query_forward(p1, p2, K, r2, l1, l2, mode=mode)
        dk, ik = bo.ball_query_from_knn(p1, p2, K, r2, l1, l2, mode=mode)
        assert _same(dm, dk) and np.array_equal(im, ik)
    return d, i


def test_oracle_random_ragged_and_k_above_p2():
    g = np.random.default_rng(0)
    for b, n1, n2, dd, K, r in [(2, 50, 80, 3, 8, 0.3), (3, 33, 70, 3, 16, 0.5), (2, 20, 64, 1, 5, 0.05),
                                (2, 17, 40, 8, 7, 0.9), (1, 9, 5, 2, 12, 2.0)]:
        p1, p2 = g.random((b, n1, dd), np.float32), g.random((b, n2, dd), np.float32)
        r2 = bo.radius2(r)
        d, i = _check_oracle(p1, p2, K, r2)
        assert (d[i < 0] == 0).all()
        assert (d[i >= 0] < r2).all()
        for n in range(b):
            for q in range(n1):
                row = i[n, q][i[n, q] >= 0]
                assert (np.diff(row) > 0).all()                           # ascending indices
                assert (i[n, q, len(row):] == -1).all()                    # pads after the hits
        l1 = g.integers(0, n1 + 1, b); l2 = g.integers(0, n2 + 1, b)
        l1[0] = 0
        d, i = _check_oracle(p1, p2, K, r2, l1, l2)
        for n in range(b):
            assert (i[n, l1[n]:] == -1).all() and (d[n, l1[n]:] == 0).all()  # rows past len1: (0, -1)
            assert (i[n] < max(l2[n], 1)).all()
    # K > P2 with every target inside: all P2 targets in order, then pads
    p1, p2 = g.random((2, 10, 3), np.float32), g.random((2, 6, 3), np.float32)
    d, i = _check_oracle(p1, p2, 9, bo.radius2(10.0))
    assert np.array_equal(i[..., :6], np.broadcast_to(np.arange(6), (2, 10, 6))) and (i[..., 6:] == -1).all()


def test_oracle_fewer_hits_than_k_and_empty_clouds():
    g = np.random.default_rng(1)
    p1, p2 = g.random((3, 40, 3), np.float32), g.random((3, 200, 3), np.float32)
    l1, l2 = np.array([40, 0, 17]), np.array([0, 200, 3])
    d, i = _check_oracle(p1, p2, 32, bo.radius2(0.1), l1, l2)
    assert (i[0] == -1).all() and (i[1] == -1).all()
    cnt = (i[2, :17] >= 0).sum(-1)
    assert (cnt <= 3).all() and (cnt < 32).all()


def test_oracle_lattice_excludes_the_radius_exactly():
    ax = np.arange(6, dtype=np.float32) * 0.25
    lat = np.stack(np.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(1, -1, 3)
    r2 = np.float32(0.0625)                                               # 0.25**2 exactly: the 6 face neighbours sit on it
    assert bo.radius2(0.25) == r2
    d, i = _check_oracle(lat, lat, 27, r2)
    assert (i[..., 1:] == -1).all() and np.array_equal(i[0, :, 0], np.arange(lat.shape[1]))  # only the point itself
    d, i = _check_oracle(lat, lat, 27, np.nextafter(r2, np.float32(1)))
    inner = 1 * 36 + 1 * 6 + 1                                            # (1, 1, 1): all 6 face neighbours are kept
    assert (i[0, inner] >= 0).sum() == 7 and (d[0, inner][i[0, inner] >= 0] <= r2).all()


def test_oracle_duplicates_and_non_finite_coordinates():
    g = np.random.default_rng(2)
    base = g.random((1, 30, 3), np.float32)
    p2 = np.concatenate([base, base], axis=1)
    p1 = g.random((1, 20, 3), np.float32)
    d, i = _check_oracle(p1, p2, 64, bo.radius2(0.4))
    for q in range(20):                                                   # a kept point's copy 30 later is kept too
        row = set(i[0, q][i[0, q] >= 0].tolist())
        assert all((j + 30 in row) for j in row if j < 30)
    p1, p2 = g.random((2, 30, 3), np.float32), g.random((2, 60, 3), np.float32)
    p2[0, 3, 1] = np.nan; p2[0, 10, 0] = np.inf; p2[1, 7, 2] = -np.inf; p2[1, 8] = np.nan
    p1[0, 4, 0] = np.nan; p1[1, 5, 2] = np.inf
    d, i = _check_oracle(p1, p2, 64, np.float32(np.inf))                  # even an infinite radius keeps no inf / NaN
    assert (i[0, 4] == -1).all() and (i[1, 5] == -1).all()
    kept = set(i[0, 0][i[0, 0] >= 0].tolist())
    assert 3 not in kept and 10 not in kept and len(kept) == 58
    assert np.isfinite(d).all()


def _pts():
    buf = (ctypes.c_float * 64)()
    return [ctypes.addressof(buf), 0, 3 * 4, 3], buf


def test_abi_refuses_bad_arguments_without_a_device():
    L = _lib.lib()
    (p, dt, bs, rs), keep = _pts()
    out = (ctypes.c_float * 64)(); oi = (ctypes.c_int * 64)()
    o, i = ctypes.addressof(out), ctypes.addressof(oi)
    for K, D, code in [(0, 3, _PCL_E_SHAPE), (1, 9, _PCL_E_UNSUPPORTED), (1, 0, _PCL_E_UNSUPPORTED)]:
        assert L.pcl_ball_query_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, D, K, 0.1, 0, o, i, None) == code
        assert L.pcl_last_error()
        assert L.pcl_ball_query_bwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, D, K, i, o, o, o, None) == code
    L.pcl_ball_query_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 0, 0.1, 0, o, i, None)
    assert b"K=0" in L.pcl_last_error()
    assert L.pcl_ball_query_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 65536, 4, 4, 3, 2, 0.1, 0, o, i, None) == _PCL_E_SHAPE
    assert L.pcl_ball_query_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, -1, 4, 4, 3, 2, 0.1, 0, o, i, None) == _PCL_E_SHAPE
    assert L.pcl_ball_query_fwd(p, 7, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, 0.1, 0, o, i, None) == _PCL_E_ARG
    assert L.pcl_ball_query_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, 0.1, 2, o, i, None) == _PCL_E_ARG
    assert b"mode" in L.pcl_last_error()
    assert L.pcl_ball_query_fwd(None, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, 0.1, 0, o, i, None) == _PCL_E_ARG
    assert L.pcl_ball_query_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, 0.1, 0, o, None, None) == _PCL_E_ARG
    assert L.pcl_ball_query_bwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, None, o, o, o, None) == _PCL_E_ARG


def test_python_argument_errors():
    import pointcloud_b200 as pcl
    x = torch.rand(2, 8, 3)
    for K in (0, -3, 2.5, True):
        with pytest.raises(ValueError, match="K="):
            pcl.ball_query(x, x, K=K)
    with pytest.raises(ValueError):
        pcl.ball_query(torch.rand(2, 8, 9), torch.rand(2, 8, 9))
    with pytest.raises(ValueError, match="Expected points"):
        pcl.ball_query(torch.rand(8, 3), x)
    with pytest.raises(ValueError, match="batch dimension"):
        pcl.ball_query(x, torch.rand(3, 8, 3))
    with pytest.raises(ValueError, match="point dimension"):
        pcl.ball_query(x, torch.rand(2, 8, 2))
    with pytest.raises(ValueError, match="lengths2"):
        pcl.ball_query(x, x, lengths2=torch.tensor([8]))


def test_radius2_is_the_fp32_square_of_the_fp32_radius():
    from pointcloud_b200.ball_query import _radius2
    for r in (0.2, 0.1, 0.05, 0.02, 0.4, 1e-3, 0.3):
        assert np.float32(_radius2(r)) == bo.radius2(r)
        assert _radius2(r) == float(np.float32(np.float32(r) * np.float32(r)))
    assert any(bo.radius2(r) != np.float32(r ** 2) for r in (0.2, 0.1, 0.05, 0.02, 0.4, 0.3, 0.7))  # differs from query_ball_point's


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback_for_ball_query():
    import pointcloud_b200 as pcl
    from pointcloud_b200._lib import PclError
    with pytest.raises(PclError):
        pcl.ball_query(torch.rand(1, 16, 3), torch.rand(1, 16, 3), K=4)
    L = _lib.lib()
    (p, dt, bs, rs), keep = _pts()
    out = (ctypes.c_float * 64)(); oi = (ctypes.c_int * 64)()
    o, i = ctypes.addressof(out), ctypes.addressof(oi)
    assert L.pcl_ball_query_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, 0.1, 0, o, i, None) < 0
    assert L.pcl_last_error()
    assert L.pcl_ball_query_bwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, i, o, o, o, None) < 0
