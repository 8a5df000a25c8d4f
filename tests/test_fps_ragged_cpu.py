"""Ragged farthest point sampling without a GPU: the test-side ragged oracle pinned against the FPS oracle, the
argument checks of pcl_fps_ragged and of sample_farthest_points, and the no-fallback behaviour."""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from fps_ragged_oracle import fps_ragged
from pointcloud_b200 import _lib, synth

_PCL_E_SHAPE, _PCL_E_ARG, _PCL_E_UNSUPPORTED = -1, -2, -5


def test_ragged_oracle_with_full_lengths_is_the_fps_oracle():
    x, _ = synth.uniform_clouds(3, 300, seed=0)
    assert np.array_equal(fps_ragged(x, 64, lengths=[300] * 3), oracle.fps(x, 64))
    assert np.array_equal(fps_ragged(x, 64, lengths=[300] * 3, K=[64] * 3), oracle.fps(x, 64))
    start = [5, 299, 17]
    assert np.array_equal(fps_ragged(x, 40, start=start), oracle.fps(x, 40, start=start))
    _, t = synth.table_clouds(2, 512, seed=1)
    assert np.array_equal(fps_ragged(t, 100), oracle.fps(t[:, :, :3], 100))          # extra channels are ignored


def test_ragged_oracle_ignores_points_beyond_the_length():
    x, _ = synth.uniform_clouds(3, 400, seed=2)
    lengths = [400, 123, 7]
    a = fps_ragged(x, 50, lengths=lengths)
    y = x.clone()
    y[1, 123:] = 10.0                                                                   # far away: would be chosen first
    y[2, 7:] = torch.rand(393, 3)
    assert np.array_equal(a, fps_ragged(y, 50, lengths=lengths))
    assert (a[1] < 123).all() and np.array_equal(a[1], oracle.fps(x[1:2, :123], 50)[0])


def test_ragged_oracle_padding():
    x, _ = synth.uniform_clouds(4, 64, seed=3)
    got = fps_ragged(x, 20, lengths=[0, 64, 5, 64], K=[20, 0, 20, 9], start=[3, 3, 9, 100])
    assert (got[0] == -1).all() and (got[1] == -1).all()                               # n_b = 0, k_b = 0
    assert (got[2, 5:] == -1).all() and sorted(got[2, :5].tolist()) == [0, 1, 2, 3, 4]  # k_b > n_b: every point once
    assert got[2, 0] == 4 and got[3, 0] == 63                                           # start clamped to n_b - 1
    assert (got[3, 9:] == -1).all() and (got[3, :9] >= 0).all()


def _pts():
    buf = (ctypes.c_float * 64)()
    return [ctypes.addressof(buf), 0, 3 * 4, 3], buf


def test_abi_refuses_bad_arguments_without_a_device():
    L = _lib.lib()
    mx = L.pcl_fps_max_points()
    assert mx >= 262144
    (p, dt, bs, rs), keep = _pts()
    oi = (ctypes.c_int * 64)()
    out = ctypes.addressof(oi)
    cases = [  # (B, N, npoint, cluster) -> code
        ((1, mx + 1, 4, 0), _PCL_E_UNSUPPORTED), ((-1, 4, 4, 0), _PCL_E_SHAPE), ((1, 0, 4, 0), _PCL_E_SHAPE),
        ((1, 4, -1, 0), _PCL_E_SHAPE), ((1, 4, 4, 3), _PCL_E_ARG), ((1, 4, 4, 32), _PCL_E_ARG), ((1, 4, 4, -1), _PCL_E_ARG),
        ((1, 16385, 4, 1), _PCL_E_UNSUPPORTED), ((1, mx, 4, 8), _PCL_E_UNSUPPORTED),
    ]
    for (B, N, npoint, cluster), code in cases:
        rc = L.pcl_fps_ragged(p, dt, bs, rs, None, B, N, None, npoint, None, 0, cluster, out, None)
        assert rc == code and L.pcl_last_error(), (B, N, npoint, cluster, rc)
    L.pcl_fps_ragged(p, dt, bs, rs, None, 1, 4, None, 4, None, 0, 5, out, None)
    assert b"cluster=5" in L.pcl_last_error()
    assert L.pcl_fps(p, dt, bs, rs, 1, mx + 1, 4, None, 0, out, None) == _PCL_E_UNSUPPORTED
    assert L.pcl_fps(p, dt, bs, rs, 1, 4, -1, None, 0, out, None) == _PCL_E_SHAPE
    assert L.pcl_fps_ragged(p, 7, bs, rs, None, 1, 4, None, 4, None, 0, 0, out, None) == _PCL_E_ARG   # dtype
    assert L.pcl_fps_ragged(p, dt, bs, rs, None, 0, 4, None, 4, None, 0, 0, out, None) == 0           # nothing to do
    assert L.pcl_fps_ragged(p, dt, bs, rs, None, 2, 4, None, 0, None, 0, 0, out, None) == 0


def test_sample_farthest_points_argument_errors():
    import pointcloud_b200 as pcl
    x = torch.rand(2, 8, 3)
    with pytest.raises(ValueError, match="lengths"):
        pcl.sample_farthest_points(x, lengths=torch.tensor([8]))
    with pytest.raises(ValueError, match="lengths"):
        pcl.sample_farthest_points(x, lengths=torch.tensor([[8, 8]]))
    with pytest.raises(ValueError, match="K"):
        pcl.sample_farthest_points(x, K=[4, 4, 4])
    with pytest.raises(ValueError, match="K"):
        pcl.sample_farthest_points(x, K=torch.tensor([[4, 4]]))
    with pytest.raises(ValueError, match="K"):
        pcl.sample_farthest_points(x, K=-1)
    with pytest.raises(ValueError, match="K"):
        pcl.sample_farthest_points(x, K=[4, -2])
    with pytest.raises(ValueError):
        pcl.sample_farthest_points(torch.rand(8, 3), K=4)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback_for_ragged_fps():
    import pointcloud_b200 as pcl
    from pointcloud_b200._lib import PclError
    x = torch.rand(2, 16, 3)
    with pytest.raises(PclError):
        pcl.sample_farthest_points(x, lengths=torch.tensor([16, 9]), K=4)
    with pytest.raises(PclError):
        pcl.sample_farthest_points(x, K=[4, 2])
    with pytest.raises(PclError):
        pcl.fps_forward_raw(x, K=4)
    L = _lib.lib()
    (p, dt, bs, rs), keep = _pts()
    oi = (ctypes.c_int * 64)()
    rc = L.pcl_fps_ragged(p, dt, bs, rs, None, 1, 4, None, 4, None, 0, 0, ctypes.addressof(oi), None)
    assert rc < 0 and L.pcl_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_scalar_k_forms_reach_the_device_path():
    import pointcloud_b200 as pcl
    from pointcloud_b200._lib import PclError
    x = torch.rand(2, 16, 3)
    for K in (np.int64(4), torch.tensor(4), np.int32(3)):           # scalars, not (N,) tensors: no ValueError
        with pytest.raises(PclError):
            pcl.sample_farthest_points(x, K=K)
        with pytest.raises(PclError):
            pcl.sample_farthest_points(x, lengths=torch.tensor([16, 9]), K=K)
    with pytest.raises(ValueError, match="K"):
        pcl.sample_farthest_points(x, K=torch.tensor([1.5, 2.0]))
