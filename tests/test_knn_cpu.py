"""K nearest neighbours without a GPU: the CPU oracle (tests/knn_oracle.c) against an independent numpy restatement,
the argument checks of the C ABI and of pointcloud_b200.knn_points, and the no-fallback behaviour."""
import ctypes

import numpy as np
import pytest
import torch

import knn_oracle as ko
import oracle
from pointcloud_b200 import _lib


def _same(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))  # bit patterns: NaN == NaN


def _check_oracle(p1, p2, K, l1=None, l2=None):
    d, i = ko.knn_forward(p1, p2, K, l1, l2)
    dn, inn = ko.knn_numpy(p1, p2, K, l1, l2)
    assert _same(d, dn) and np.array_equal(i, inn)
    return d, i


def test_oracle_matches_numpy_random_and_ragged():
    g = np.random.default_rng(0)
    for b, n1, n2, dd, K in [(2, 50, 80, 3, 1), (3, 33, 70, 3, 16), (2, 20, 64, 1, 64), (2, 17, 40, 8, 7), (1, 9, 5, 2, 12)]:
        p1, p2 = g.random((b, n1, dd), np.float32), g.random((b, n2, dd), np.float32)
        d, i = _check_oracle(p1, p2, K)
        kv = min(K, n2)
        assert (np.diff(d[..., :kv], axis=-1) >= 0).all()
        assert (d[..., kv:] == 0).all() and (i[..., kv:] == 0).all()          # K > P2: padded slots are 0 / 0
        l1 = g.integers(0, n1 + 1, b); l2 = g.integers(0, n2 + 1, b)
        l1[0], l2[-1] = 0, min(K, n2) - 1 if min(K, n2) > 1 else 0           # an empty query cloud, fewer targets than K
        d, i = _check_oracle(p1, p2, K, l1, l2)
        for n in range(b):
            assert (d[n, l1[n]:] == 0).all() and (i[n, l1[n]:] == 0).all()
            assert (i[n, :, min(K, l2[n]):] == 0).all()
            assert (i[n, :l1[n], :min(K, l2[n])] < l2[n]).all()


def test_oracle_ties_go_to_the_lowest_index():
    g = np.random.default_rng(1)
    base = g.random((1, 10, 3), np.float32)
    p2 = np.concatenate([base, base, base[:, :5]], axis=1)              # every target duplicated (some three times)
    p1 = g.random((1, 40, 3), np.float32)
    d, i = _check_oracle(p1, p2, 6)
    for q in range(40):
        for k in range(5):
            if d[0, q, k] == d[0, q, k + 1]:
                assert i[0, q, k] < i[0, q, k + 1]
    # a lattice: many exactly equal distances
    ax = np.arange(5, dtype=np.float32) * 0.25
    lat = np.stack(np.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(1, -1, 3)
    d, i = _check_oracle(lat[:, ::7], lat, 32)
    assert np.array_equal(i[0, :, 0], np.arange(0, 125, 7))              # a point's own copy comes first
    d, i = _check_oracle(lat, lat, 27)


def test_oracle_non_finite_coordinates():
    g = np.random.default_rng(2)
    p1, p2 = g.random((2, 30, 3), np.float32), g.random((2, 60, 3), np.float32)
    p2[0, 3, 1] = np.nan; p2[0, 10, 0] = np.inf; p2[1, 7, 2] = -np.inf; p2[1, 8] = np.nan
    p1[0, 4, 0] = np.nan; p1[1, 5, 2] = np.inf
    d, i = _check_oracle(p1, p2, 64)
    # order: finite distances, then +inf, then NaN (reported as 0x7fffffff), each group by index
    row = d[0, 0]
    assert np.isposinf(row[58]) and np.isnan(row[59]) and i[0, 0, 58] == 10 and i[0, 0, 59] == 3
    assert row[59:].view(np.uint32)[0] == 0x7FFFFFFF
    assert np.isnan(d[0, 4, :60]).all() and np.array_equal(i[0, 4, :60], np.arange(60))  # a NaN query: all keys tie on NaN
    assert np.isposinf(d[1, 5, :59]).all() and np.array_equal(i[1, 5, :59], np.r_[0:8, 9:60])  # an infinite query
    assert np.isnan(d[1, 5, 59]) and i[1, 5, 59] == 8


def test_oracle_k1_equals_the_chamfer_oracle_in_both_modes():
    g = np.random.default_rng(3)
    for dd in (1, 3, 5, 8):
        x, y = g.random((3, 70, dd), np.float32), g.random((3, 90, dd), np.float32)
        xl, yl = np.array([70, 0, 31]), np.array([90, 45, 1])
        for mode in (0, 1):
            oc = oracle.chamfer_forward(x, y, xl, yl, mode=mode)
            d, i = ko.knn_forward(x, y, 1, xl, yl, mode=mode)
            assert _same(d[..., 0], oc["dist_x"]) and np.array_equal(i[..., 0], oc["idx_x"])


def test_oracle_backward_matches_numpy():
    g = np.random.default_rng(4)
    b, n1, n2, dd, K = 3, 40, 55, 3, 9
    p1, p2 = g.random((b, n1, dd), np.float32), g.random((b, n2, dd), np.float32)
    l1, l2 = np.array([40, 12, 0]), np.array([55, 5, 30])
    d, i = ko.knn_forward(p1, p2, K, l1, l2)
    gd = g.standard_normal((b, n1, K)).astype(np.float32)
    g1, g2 = ko.knn_backward(p1, p2, i, gd, l1, l2)
    e1, e2 = np.zeros_like(g1, dtype=np.float64), np.zeros_like(g2, dtype=np.float64)
    for n in range(b):
        for q in range(l1[n]):
            for k in range(min(K, l2[n])):
                diff = 2.0 * gd[n, q, k] * (p1[n, q].astype(np.float64) - p2[n, i[n, q, k]])
                e1[n, q] += diff; e2[n, i[n, q, k]] -= diff
    np.testing.assert_allclose(g1, e1, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(g2, e2, rtol=1e-5, atol=1e-6)
    assert (g1[1, 12:] == 0).all() and (g1[2] == 0).all()               # padded rows: no gradient
    assert (g2[1, 5:] == 0).all()                                         # targets beyond len2 are never chosen


def _pts():
    buf = (ctypes.c_float * 64)()
    return [ctypes.addressof(buf), 0, 3 * 4, 3], buf


def test_abi_refuses_bad_k_and_d_without_a_device():
    L = _lib.lib()
    assert L.pcl_knn_max_k() >= 32
    (p, dt, bs, rs), keep = _pts()
    out = (ctypes.c_float * 64)(); oi = (ctypes.c_int * 64)()
    for K, D in [(0, 3), (L.pcl_knn_max_k() + 1, 3), (1, 9), (1, 0)]:
        rc = L.pcl_knn_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, D, K, 0, ctypes.addressof(out), ctypes.addressof(oi), None)
        assert rc in (_PCL_E_SHAPE, _PCL_E_UNSUPPORTED) and L.pcl_last_error()
        rc = L.pcl_knn_bwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, D, K, ctypes.addressof(oi), ctypes.addressof(out),
                           ctypes.addressof(out), ctypes.addressof(out), None)
        assert rc in (_PCL_E_SHAPE, _PCL_E_UNSUPPORTED) and L.pcl_last_error()
    L.pcl_knn_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 0, 0, ctypes.addressof(out), ctypes.addressof(oi), None)
    assert b"K=0" in L.pcl_last_error()
    import pointcloud_b200 as pcl
    x = torch.rand(2, 8, 3)
    for kw in [dict(K=0), dict(K=L.pcl_knn_max_k() + 1), dict(K=2, norm=1)]:
        with pytest.raises(NotImplementedError if "norm" in kw else ValueError):
            pcl.knn_points(x, x, **kw)
    with pytest.raises(ValueError):
        pcl.knn_points(torch.rand(2, 8, 9), torch.rand(2, 8, 9))
    with pytest.raises(ValueError, match="batch dimension"):
        pcl.knn_points(x, torch.rand(3, 8, 3))
    with pytest.raises(ValueError, match="point dimension"):
        pcl.knn_points(x, torch.rand(2, 8, 2))
    with pytest.raises(ValueError, match="lengths1"):
        pcl.knn_points(x, x, lengths1=torch.tensor([8]))


_PCL_E_SHAPE, _PCL_E_UNSUPPORTED = -1, -5


def test_knn_gather_pads_and_indexes_on_cpu():
    import pointcloud_b200 as pcl
    x = torch.arange(2 * 5 * 2, dtype=torch.float32).view(2, 5, 2)
    idx = torch.tensor([[[4, 0, 1]], [[2, 3, 0]]])
    out = pcl.knn_gather(x, idx, lengths=torch.tensor([5, 2]))
    assert out.shape == (2, 1, 3, 2)
    assert torch.equal(out[0, 0], x[0, [4, 0, 1]])
    assert torch.equal(out[1, 0, :2], x[1, [2, 3]]) and (out[1, 0, 2] == 0).all()
    with pytest.raises(ValueError):
        pcl.knn_gather(x, idx[:1].expand(3, -1, -1))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback_for_knn():
    import pointcloud_b200 as pcl
    from pointcloud_b200._lib import PclError
    with pytest.raises(PclError):
        pcl.knn_points(torch.rand(1, 16, 3), torch.rand(1, 16, 3), K=4)
    L = _lib.lib()
    (p, dt, bs, rs), keep = _pts()
    out = (ctypes.c_float * 64)(); oi = (ctypes.c_int * 64)()
    rc = L.pcl_knn_fwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, 0, ctypes.addressof(out), ctypes.addressof(oi), None)
    assert rc < 0 and L.pcl_last_error()
    rc = L.pcl_knn_bwd(p, dt, bs, rs, None, p, dt, bs, rs, None, 1, 4, 4, 3, 2, ctypes.addressof(oi), ctypes.addressof(out),
                       ctypes.addressof(out), ctypes.addressof(out), None)
    assert rc < 0 and L.pcl_last_error()
