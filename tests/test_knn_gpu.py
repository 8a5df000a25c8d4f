"""GPU tests of K-nearest-neighbour search: bit-exact distances and indices against the CPU oracle
(tests/knn_oracle.c), K = 1 against the Chamfer kernels, gradients within 1e-5 relative of the oracle, and
size-independent properties at full size."""
import numpy as np
import pytest
import torch

import knn_oracle as ko
import pointcloud_b200 as pcl
from pointcloud_b200 import _lib, synth
from helpers import npy

pytestmark = pytest.mark.gpu
REL = 1e-5
MODES = {"unfused": 0, "fma": 1}


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def run_case(p1, p2, K, l1=None, l2=None, mode="unfused"):
    r = pcl.knn_forward_raw(p1.cuda(), p2.cuda(), l1, l2, K=K, mode=mode)
    od, oi = ko.knn_forward(p1, p2, K, l1, l2, mode=MODES[mode])
    assert np.array_equal(_bits(npy(r["dists"])), _bits(od))   # bit-exact fp32 distances (NaN bit patterns included)
    assert np.array_equal(npy(r["idx"]), oi)
    return od, oi


def _rand(shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("mode", ["unfused", "fma"])
@pytest.mark.parametrize("b,p1,p2,K", [(4, 2048, 2048, 16), (32, 512, 2048, 32), (3, 700, 1300, 5), (2, 21, 2048, 1),
                                       (5, 1024, 33, 64), (1, 1, 1, 1), (2, 300, 40, 64), (8, 512, 4096, 16)])
def test_forward_bit_exact_vs_oracle_d3(b, p1, p2, K, mode):
    run_case(_rand((b, p1, 3), p1), _rand((b, p2, 3), p2 + K), K, mode=mode)


@pytest.mark.parametrize("mode", ["unfused", "fma"])
@pytest.mark.parametrize("d", [1, 2, 4, 5, 6, 7, 8])
def test_forward_bit_exact_vs_oracle_generic_d(d, mode):
    run_case(_rand((3, 700, d), d), _rand((3, 1300, d), 10 + d), 16, mode=mode)
    run_case(_rand((2, 96, d), d), _rand((2, 512, d), 20 + d), pcl.knn.knn_max_k(), mode=mode)


def test_max_k_and_table_clouds():
    kmax = _lib.lib().pcl_knn_max_k()
    assert kmax == 64
    x, t = synth.table_clouds(4, 2048, seed=2)
    for mode in MODES:
        run_case(x, t[:, :, :3].contiguous(), kmax, mode=mode)


def test_ties_duplicates_and_lattice():
    g = torch.Generator().manual_seed(5)
    y = torch.rand(2, 512, 3, generator=g)
    y = torch.cat([y, y, y[:, :100]], dim=1)             # every target at least twice: exact ties everywhere
    run_case(torch.rand(2, 900, 3, generator=g), y, 24)
    ax = torch.arange(12, dtype=torch.float32) * 0.125
    lat = torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(1, -1, 3)  # 1728 lattice points
    d, i = run_case(lat, lat, 27)
    assert np.array_equal(i[0, :, 0], np.arange(lat.shape[1]))


def test_ragged_and_empty_clouds():
    g = torch.Generator().manual_seed(7)
    p1, p2 = torch.rand(6, 1000, 3, generator=g), torch.rand(6, 1500, 3, generator=g)
    l1 = torch.tensor([1000, 0, 517, 33, 1000, 1])
    l2 = torch.tensor([1500, 700, 0, 5, 16, 1499])         # empty target cloud, fewer targets than K, exactly K
    for mode in MODES:
        d, i = run_case(p1, p2, 16, l1, l2, mode=mode)
    assert (d[1] == 0).all() and (d[2] == 0).all() and (i[3, :33, 5:] == 0).all()
    run_case(p1[:, :, :2].contiguous(), p2[:, :, :2].contiguous(), 16, l1, l2)


def test_half_bf16_and_strided_inputs():
    pred, target = synth.autoencoder_batch(3, 1024, seed=1)
    for dt in (torch.float16, torch.bfloat16):
        p1, p2 = pred.to(dt).cuda()[:, :, :3], target.to(dt).cuda()[:, :, :3]
        assert p1.stride(-1) == 1 and not p1.is_contiguous()
        assert _lib.as_points(p1).data_ptr() == p1.data_ptr()          # no copy
        r = pcl.knn_forward_raw(p1, p2, K=8)
        od, oi = ko.knn_forward(p1.float().cpu(), p2.float().cpu(), 8)
        assert np.array_equal(_bits(npy(r["dists"])), _bits(od)) and np.array_equal(npy(r["idx"]), oi)
    run_case(pred[:, :, :3], target[:, :, :3], 12)         # fp32 strided view (oracle reads the same strides)


def test_non_finite_points():
    g = torch.Generator().manual_seed(9)
    p1, p2 = torch.rand(2, 300, 3, generator=g), torch.rand(2, 700, 3, generator=g)
    p2[0, 3, 1] = float("nan"); p2[0, 10, 0] = float("inf"); p2[1, 7, 2] = -float("inf"); p2[1, 8] = float("nan")
    p1[0, 4, 0] = float("nan"); p1[1, 5, 2] = float("inf")
    for mode in MODES:
        d, i = run_case(p1, p2, 64, mode=mode)
    assert np.isnan(d[0, 4]).all() and np.array_equal(i[0, 4], np.arange(64))
    q = torch.full((1, 40, 3), 3e38)                         # finite coordinates whose distances overflow to +inf
    run_case(q, -q[:, :35], 8)


@pytest.mark.parametrize("mode", ["unfused", "fma"])
@pytest.mark.parametrize("d", [3, 2, 6])
def test_k1_identical_to_chamfer(d, mode):
    g = torch.Generator().manual_seed(11 + d)
    x, y = torch.rand(4, 2048, d, generator=g), torch.rand(4, 1500, d, generator=g)
    xl, yl = torch.tensor([2048, 100, 0, 777]), torch.tensor([1500, 1, 300, 0])
    for lens in ((None, None), (xl, yl)):
        c = pcl.chamfer_forward_raw(x.cuda(), y.cuda(), *lens, mode=mode)
        r = pcl.knn_forward_raw(x.cuda(), y.cuda(), *lens, K=1, mode=mode)
        assert torch.equal(r["dists"][..., 0].view(torch.int32), c["dist_x"].view(torch.int32))
        assert torch.equal(r["idx"][..., 0], c["idx_x"])


def _grad_case(p1, p2, K, l1=None, l2=None):
    a, b = p1.cuda().requires_grad_(), p2.cuda().requires_grad_()
    out = pcl.knn_points(a, b, l1, l2, K=K)
    g = torch.randn(out.dists.shape, generator=torch.Generator().manual_seed(K)).cuda()
    (out.dists * g).sum().backward()
    assert out.idx.dtype == torch.int64 and not out.idx.requires_grad
    od, oi = ko.knn_forward(p1, p2, K, l1, l2)
    assert np.array_equal(npy(out.idx), oi)
    g1, g2 = ko.knn_backward(p1, p2, oi, npy(g), l1, l2)
    np.testing.assert_allclose(npy(a.grad), g1, rtol=REL, atol=1e-6 * np.abs(g1).max())
    np.testing.assert_allclose(npy(b.grad), g2, rtol=REL, atol=1e-6 * np.abs(g2).max())
    return npy(a.grad), npy(b.grad)


def test_gradients_vs_oracle():
    _grad_case(_rand((4, 2048, 3), 1), _rand((4, 2048, 3), 2), 16)
    _grad_case(_rand((3, 500, 5), 3), _rand((3, 900, 5), 4), 7)
    l1, l2 = torch.tensor([500, 0, 123]), torch.tensor([900, 50, 3])
    ga, gb = _grad_case(_rand((3, 500, 3), 5), _rand((3, 900, 3), 6), 32, l1, l2)
    assert (ga[1] == 0).all() and (ga[2, 123:] == 0).all() and (ga[0] != 0).any()      # padded rows: zero gradient
    assert (gb[1, 50:] == 0).all() and (gb[2, 3:] == 0).all()


def test_fp16_gradient_dtype_and_return_nn():
    p1 = torch.rand(2, 256, 3, dtype=torch.float16, device="cuda", requires_grad=True)
    p2 = torch.rand(2, 400, 3, device="cuda", requires_grad=True)
    l2 = torch.tensor([400, 10])
    out = pcl.knn_points(p1, p2, lengths2=l2, K=12, return_nn=True)
    assert out.knn.shape == (2, 256, 12, 3)
    ref = pcl.knn_gather(p2, out.idx, l2)
    assert torch.equal(out.knn, ref) and (out.knn[1, :, 10:] == 0).all()
    assert torch.equal(out.knn[0], p2[0][out.idx[0]])
    out.knn.sum().backward()                                # gradient to p2 through knn_gather only
    assert p1.grad is None
    cnt = torch.zeros(2, 400, device="cuda")
    valid = torch.arange(12, device="cuda")[None, None, :] < l2.cuda()[:, None, None]
    cnt.scatter_add_(1, out.idx.reshape(2, -1), valid.expand(-1, 256, -1).reshape(2, -1).float())
    assert torch.equal(p2.grad, cnt[..., None].expand(-1, -1, 3))
    p2.grad = None
    out = pcl.knn_points(p1, p2, K=4)
    out.dists.sum().backward()
    assert p1.grad.dtype == torch.float16 and p2.grad.dtype == torch.float32


def test_full_size_properties():
    b, n, K = 32, 2048, 16
    x, t = synth.table_clouds(b, n, seed=4)
    p1, p2 = x.cuda(), t[:, :, :3].contiguous().cuda()
    r1 = pcl.knn_forward_raw(p1, p2, K=K)
    r2 = pcl.knn_forward_raw(p1, p2, K=K)
    assert torch.equal(r1["dists"], r2["dists"]) and torch.equal(r1["idx"], r2["idx"])   # two runs are identical
    d, i = r1["dists"], r1["idx"].long()
    # every distance is the recomputed distance of its index (unfused order)
    nb = torch.gather(p2, 1, i.view(b, -1, 1).expand(-1, -1, 3)).view(b, n, K, 3)
    df = p1[:, :, None, :] - nb
    rd = (df[..., 0] * df[..., 0] + df[..., 1] * df[..., 1]) + df[..., 2] * df[..., 2]
    assert torch.equal(rd, d)
    # rows are sorted by (distance, index)
    dd, di = d[..., 1:] - d[..., :-1], i[..., 1:] - i[..., :-1]
    assert bool(((dd > 0) | ((dd == 0) & (di > 0))).all())
    # no sampled target beats the K-th distance (exhaustive over 256 queries of every cloud)
    q = p1[:, ::8]
    full = (q[:, :, None, :] - p2[:, None, :, :]).square().sum(-1)          # (b, 256, n), any rounding
    kth = d[:, ::8, K - 1:K]
    below = (full < kth * (1 - 1e-5)).sum(-1)
    assert bool((below <= K - 1).all())
