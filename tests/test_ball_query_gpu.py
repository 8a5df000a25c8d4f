"""GPU tests of ball query: bit-exact distances and indices against the CPU oracle (tests/ball_query_oracle.c) on both
sides of the target-split rule, agreement with knn_points, gradients against torch autograd on the gathered
formulation, the -1 rule of pcl_knn_bwd, and a 262 144-point cloud around FPS centroids."""
import numpy as np
import pytest
import torch

import ball_query_oracle as bo
import pointcloud_b200 as pcl
from pointcloud_b200 import _lib, synth
from helpers import npy

pytestmark = pytest.mark.gpu
MODES = {"unfused": 0, "fma": 1}


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


def run_case(p1, p2, K, radius, l1=None, l2=None, mode="unfused"):
    r = pcl.ball_query_forward_raw(p1.cuda(), p2.cuda(), l1, l2, K=K, radius=radius, mode=mode)
    od, oi = bo.ball_query_forward(p1, p2, K, bo.radius2(radius), l1, l2, mode=MODES[mode])
    assert np.array_equal(_bits(npy(r["dists"])), _bits(od))
    assert np.array_equal(npy(r["idx"]), oi)
    return od, oi


def _rand(shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("mode", ["unfused", "fma"])
@pytest.mark.parametrize("b,p1,p2,K,r", [
    (32, 512, 2048, 32, 0.2),      # PointNet++ SA1: split in two
    (32, 128, 512, 64, 0.4),       # SA2
    (1, 64, 8192, 16, 0.3),        # 2 query warps: sixteen parts
    (1, 100, 4096, 64, 0.05),      # sixteen parts at the largest buffered K
    (2, 300, 5000, 500, 0.3),      # pytorch3d's default K: split in two
    (1, 40, 3000, 1000, 0.5),      # K too large to buffer: one part
    (64, 2048, 1024, 8, 0.1),      # enough query warps: one part
    (3, 700, 1300, 5, 0.15), (1, 1, 1, 1, 1.0), (2, 33, 40, 64, 2.0)])
def test_forward_bit_exact_vs_oracle_d3(b, p1, p2, K, r, mode):
    run_case(_rand((b, p1, 3), p1), _rand((b, p2, 3), p2 + K), K, r, mode=mode)


@pytest.mark.parametrize("mode", ["unfused", "fma"])
@pytest.mark.parametrize("d", [1, 2, 4, 5, 6, 7, 8])
def test_forward_bit_exact_vs_oracle_generic_d(d, mode):
    run_case(_rand((3, 700, d), d), _rand((3, 1300, d), 10 + d), 16, 0.3 + 0.05 * d, mode=mode)
    run_case(_rand((1, 96, d), d), _rand((1, 6000, d), 20 + d), 64, 0.2 + 0.08 * d, mode=mode)


def test_ragged_and_empty_clouds():
    g = torch.Generator().manual_seed(7)
    p1, p2 = torch.rand(6, 1000, 3, generator=g), torch.rand(6, 1500, 3, generator=g)
    l1 = torch.tensor([1000, 0, 517, 33, 1000, 1])
    l2 = torch.tensor([1500, 700, 0, 5, 16, 1499])
    for mode in MODES:
        d, i = run_case(p1, p2, 16, 0.2, l1, l2, mode=mode)
    assert (i[1] == -1).all() and (i[2] == -1).all() and (i[3, :33] < 5).all() and (i[0, 1000:] == -1).all()
    run_case(p1[:1, :40], p2[:1], 32, 0.2, l1[:1] * 0 + 40, torch.tensor([1200]))   # split, ragged targets
    run_case(p1[:, :, :2].contiguous(), p2[:, :, :2].contiguous(), 16, 0.1, l1, l2)


def test_half_bf16_and_strided_inputs():
    pred, target = synth.autoencoder_batch(3, 1024, seed=1)
    for dt in (torch.float16, torch.bfloat16):
        p1, p2 = pred.to(dt).cuda()[:, :, :3], target.to(dt).cuda()[:, :, :3]
        assert p1.stride(-1) == 1 and not p1.is_contiguous()
        assert _lib.as_points(p1).data_ptr() == p1.data_ptr()
        r = pcl.ball_query_forward_raw(p1, p2, K=24, radius=0.1)
        od, oi = bo.ball_query_forward(p1.float().cpu(), p2.float().cpu(), 24, bo.radius2(0.1))
        assert np.array_equal(_bits(npy(r["dists"])), _bits(od)) and np.array_equal(npy(r["idx"]), oi)
    run_case(pred[:, :, :3], target[:, :, :3], 12, 0.1)


def test_lattice_duplicates_and_non_finite_points():
    ax = torch.arange(12, dtype=torch.float32) * 0.25
    lat = torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(1, -1, 3)
    d, i = run_case(lat, lat, 27, 0.25)                                   # face neighbours sit exactly on radius2
    assert (i[..., 1:] == -1).all()
    y = _rand((2, 512, 3), 5)
    run_case(_rand((2, 900, 3), 6), torch.cat([y, y, y[:, :100]], dim=1), 48, 0.2)
    g = torch.Generator().manual_seed(9)
    p1, p2 = torch.rand(2, 300, 3, generator=g), torch.rand(2, 700, 3, generator=g)
    p2[0, 3, 1] = float("nan"); p2[0, 10, 0] = float("inf"); p2[1, 7, 2] = -float("inf"); p2[1, 8] = float("nan")
    p1[0, 4, 0] = float("nan"); p1[1, 5, 2] = float("inf")
    for mode in MODES:
        d, i = run_case(p1, p2, 64, 0.3, mode=mode)
    assert (i[0, 4] == -1).all() and (i[1, 5] == -1).all()


def test_split_and_unsplit_rows_are_identical():
    x, t = _rand((1, 256, 3), 1), _rand((1, 16384, 3), 2)
    alone = pcl.ball_query_forward_raw(x.cuda(), t.cuda(), K=48, radius=0.15)               # 8 query warps: split
    many = pcl.ball_query_forward_raw(x.expand(64, -1, -1).cuda(), t.expand(64, -1, -1).cuda(), K=48, radius=0.15)
    assert torch.equal(many["idx"], alone["idx"].expand(64, -1, -1))
    assert torch.equal(many["dists"].view(torch.int32), alone["dists"].view(torch.int32).expand(64, -1, -1))
    run_case(x, t, 48, 0.15)


@pytest.mark.parametrize("mode", ["unfused", "fma"])
def test_kept_distances_equal_knn(mode):
    x, t = _rand((4, 512, 3), 3), _rand((4, 2048, 3), 4)
    K, r = 64, 0.12                                                       # ~14 points per ball: mostly fewer than K
    bq = pcl.ball_query(x.cuda(), t.cuda(), K=K, radius=r, return_nn=False, mode=mode)
    kn = pcl.knn_points(x.cuda(), t.cuda(), K=K, mode=mode)
    r2 = float(bo.radius2(r))
    kd, ki, bd, bi = npy(kn.dists), npy(kn.idx), npy(bq.dists), npy(bq.idx)
    full = 0
    for n in range(4):
        for q in range(512):
            kept = bi[n, q] >= 0
            m = dict(zip(ki[n, q].tolist(), kd[n, q].tolist()))
            for j, dv in zip(bi[n, q][kept].tolist(), bd[n, q][kept].tolist()):
                if j in m:
                    assert np.float32(m[j]).view(np.uint32) == np.float32(dv).view(np.uint32)
            if kd[n, q, K - 1] >= r2:                                     # the ball holds <= K points: same index set
                assert set(bi[n, q][kept].tolist()) == set(ki[n, q][kd[n, q] < r2].tolist())
                full += 1
    assert full > 1000


def _gathered_reference(p1, p2, idx, g):
    a, b = p1.detach().float().clone().requires_grad_(), p2.detach().float().clone().requires_grad_()
    n, l, k = idx.shape
    nb = b.gather(1, idx.clamp(min=0).reshape(n, l * k, 1).expand(-1, -1, b.shape[2])).view(n, l, k, -1)
    d = (a[:, :, None, :] - nb).square().sum(-1) * (idx >= 0)
    (d * g).sum().backward()
    return a.grad, b.grad


@pytest.mark.parametrize("b,n1,n2,dd,K,r", [(4, 2048, 2048, 3, 16, 0.1), (3, 500, 900, 5, 500, 0.5),
                                            (1, 64, 8192, 3, 64, 0.06)])
def test_gradients_vs_torch_autograd(b, n1, n2, dd, K, r):
    p1 = _rand((b, n1, dd), n1).cuda().requires_grad_()
    p2 = _rand((b, n2, dd), n2).cuda().requires_grad_()
    l1 = torch.tensor([n1] + [n1 // 3] * (b - 1)); l2 = torch.tensor([n2] + [n2 // 7] * (b - 1))
    out = pcl.ball_query(p1, p2, l1, l2, K=K, radius=r, return_nn=False)
    g = torch.randn(out.dists.shape, generator=torch.Generator().manual_seed(K)).cuda()
    (out.dists * g).sum().backward()
    assert out.idx.dtype == torch.int64 and not out.idx.requires_grad and (out.idx == -1).any()
    e1, e2 = _gathered_reference(p1, p2, out.idx, g)
    for got, ref in ((p1.grad, e1), (p2.grad, e2)):
        np.testing.assert_allclose(npy(got), npy(ref), rtol=1e-5, atol=1e-6 * float(ref.abs().max()))
    for n in range(1, b):
        assert (p1.grad[n, n1 // 3:] == 0).all() and (p2.grad[n, n2 // 7:] == 0).all()   # pads: zero gradient


def test_return_nn_zeros_and_gradient():
    p1 = torch.rand(2, 256, 3, dtype=torch.float16, device="cuda", requires_grad=True)
    p2 = torch.rand(2, 400, 3, device="cuda", requires_grad=True)
    out = pcl.ball_query(p1, p2, lengths2=torch.tensor([400, 10]), K=12, radius=0.2)
    assert out.knn.shape == (2, 256, 12, 3)
    pad = out.idx < 0
    assert pad.any() and (out.knn[pad] == 0).all()
    assert torch.equal(out.knn[0][~pad[0]], p2.detach()[0][out.idx[0][~pad[0]]])
    out.knn.sum().backward()                                               # gradient to p2 through the gather only
    assert p1.grad is None
    cnt = torch.zeros(2, 400, device="cuda")
    cnt.scatter_add_(1, out.idx.clamp(min=0).reshape(2, -1), (~pad).reshape(2, -1).float())
    assert torch.equal(p2.grad, cnt[..., None].expand(-1, -1, 3))
    p2.grad = None
    out = pcl.ball_query(p1, p2, K=4, radius=0.3)
    out.dists.sum().backward()
    assert p1.grad.dtype == torch.float16 and p2.grad.dtype == torch.float32


def test_knn_bwd_skips_minus_one_slots():
    L = _lib.lib()
    b, n1, n2, K = 2, 300, 500, 16
    p1, p2 = _rand((b, n1, 3), 1).cuda(), _rand((b, n2, 3), 2).cuda()
    idx = pcl.knn_forward_raw(p1, p2, K=K)["idx"]
    g = torch.randn(b, n1, K, generator=torch.Generator().manual_seed(3)).cuda()
    drop = torch.rand(b, n1, K, generator=torch.Generator().manual_seed(4)).cuda() < 0.3

    def bwd(ix, gd):
        g1, g2 = torch.empty(b, n1, 3, device="cuda"), torch.empty(b, n2, 3, device="cuda")
        rc = L.pcl_knn_bwd(*_lib.pts_args(p1), None, *_lib.pts_args(p2), None, b, n1, n2, 3, K, ix.data_ptr(),
                           gd.contiguous().data_ptr(), g1.data_ptr(), g2.data_ptr(), _lib.stream_ptr())
        assert rc == 0
        return g1, g2

    a1, a2 = bwd(torch.where(drop, -1, idx).int().contiguous(), g)       # -1 slots with a nonzero gradient
    b1, b2 = bwd(idx, torch.where(drop, 0.0, g))                          # the same slots with a zero gradient
    assert torch.equal(a1, b1)
    np.testing.assert_allclose(npy(a2), npy(b2), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("radius", [0.02, 0.1])
def test_large_cloud_around_fps_centroids(radius):
    cloud = _rand((1, 262144, 3), 12)
    c, _ = pcl.sample_farthest_points(cloud.cuda(), K=2048)
    od, oi = run_case(c.cpu(), cloud, 64, radius)
    hits = (oi >= 0).sum(-1)
    assert (hits >= 1).all()                                               # every centroid is a point of the cloud
    if radius == 0.1:
        assert (hits == 64).mean() > 0.9
