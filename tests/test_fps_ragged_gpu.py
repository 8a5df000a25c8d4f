"""GPU tests of farthest point sampling on ragged batches and large clouds (pcl_fps_ragged, sample_farthest_points):
bit-exact against the ragged oracle for every cluster size, agreement with pcl_fps, and the pytorch3d call surface."""
import numpy as np
import pytest
import torch

import oracle
import pointcloud_b200 as pcl
from fps_ragged_oracle import fps_ragged
from helpers import npy
from pointcloud_b200 import _lib, synth

pytestmark = pytest.mark.gpu

CLUSTERS = [0, 1, 2, 4, 8, 16]  # 0 = AUTO


def raw(x, npoint, lengths=None, K=None, start=None, skip_origin=False, cluster=0):
    t = lambda v: None if v is None else torch.as_tensor(v)
    return npy(pcl.fps_forward_raw(x, t(lengths), t(K), npoint, start_idx=t(start), skip_origin=skip_origin, cluster=cluster))


@pytest.mark.parametrize("cluster", CLUSTERS)
def test_ragged_bit_exact_vs_oracle(cluster):
    x, _ = synth.uniform_clouds(8, 3000, seed=cluster)
    lengths = [3000, 0, 1, 2999, 1500, 17, 512, 3000]
    K = [200, 200, 0, 5000, 64, 200, 512, 1]                 # 0, more than n_b, more than npoint
    start = [0, 4, 9, 2998, 1499, 40, 7, 3001]               # some >= n_b: clamped
    want = fps_ragged(x, 200, lengths, K, start)
    assert np.array_equal(raw(x.cuda(), 200, lengths, K, start, cluster=cluster), want)
    assert np.array_equal(raw(x.cuda(), 200, lengths, None, None, cluster=cluster), fps_ragged(x, 200, lengths))
    assert np.array_equal(raw(x.cuda(), 200, None, K, None, cluster=cluster), fps_ragged(x, 200, None, K))


@pytest.mark.parametrize("cluster", CLUSTERS)
def test_ragged_special_inputs(cluster):
    # skip_origin with every point at the origin: index 0 repeats, like the oracle
    z = torch.zeros(2, 700, 3)
    assert np.array_equal(raw(z.cuda(), 30, [700, 300], [30, 10], skip_origin=True, cluster=cluster),
                          fps_ragged(z, 30, [700, 300], [30, 10], skip_origin=True))
    # some points at the origin
    g = torch.Generator().manual_seed(5)
    zo = torch.cat([torch.zeros(3, 50, 3), torch.rand(3, 900, 3, generator=g) + 0.05], dim=1)
    assert np.array_equal(raw(zo.cuda(), 64, [950, 60, 40], skip_origin=True, cluster=cluster),
                          fps_ragged(zo, 64, [950, 60, 40], skip_origin=True))
    # duplicate points: once every distinct location is taken, the lowest index with running minimum 0 repeats
    base = torch.rand(2, 40, 3, generator=g)
    d = torch.cat([base] * 25, dim=1)
    assert np.array_equal(raw(d.cuda(), 100, [1000, 333], cluster=cluster), fps_ragged(d, 100, [1000, 333]))
    # fp16 / bf16 and strided views, read in place
    pred, target = synth.autoencoder_batch(3, 2048, seed=cluster)
    lengths, K = [2048, 1000, 3], [256, 256, 256]
    for dt in (torch.float16, torch.bfloat16):
        v = target.cuda().to(dt)[:, :, :3]
        assert np.array_equal(raw(v, 256, lengths, K, cluster=cluster), fps_ragged(v.float().cpu(), 256, lengths, K))
    assert np.array_equal(raw(target.cuda()[:, :, :3], 256, lengths, K, cluster=cluster), fps_ragged(target, 256, lengths, K))


@pytest.mark.parametrize("n", [2048, 16384])
def test_ragged_without_lengths_equals_pcl_fps(n):
    x, _ = synth.uniform_clouds(4, n, seed=n)
    for skip in (False, True):
        a = pcl.farthest_point_sample(x.cuda(), 512, skip_origin=skip).int()
        for cluster in CLUSTERS:
            assert torch.equal(pcl.fps_forward_raw(x.cuda(), npoint=512, skip_origin=skip, cluster=cluster), a)
    # npoint > N: pcl_fps continues (index 0 repeats), pcl_fps_ragged pads -1
    y, _ = synth.uniform_clouds(2, 100, seed=1)
    assert np.array_equal(npy(pcl.farthest_point_sample(y.cuda(), 150, skip_origin=False)), oracle.fps(y, 150))
    assert np.array_equal(raw(y.cuda(), 150), fps_ragged(y, 150))


def test_large_clouds_vs_oracle():
    mx = _lib.lib().pcl_fps_max_points()
    x, _ = synth.uniform_clouds(2, 16385, seed=11)
    want = oracle.fps(x, 2048)
    assert np.array_equal(npy(pcl.farthest_point_sample(x.cuda(), 2048, skip_origin=False)), want)
    for cluster in (2, 4, 16):
        assert np.array_equal(raw(x.cuda(), 2048, cluster=cluster), want)
    y, _ = synth.uniform_clouds(1, mx, seed=12)
    got = npy(pcl.farthest_point_sample(y.cuda(), 2048, skip_origin=False))
    assert np.array_equal(got, oracle.fps(y, 2048))
    assert np.array_equal(raw(y.cuda(), 2048, [mx - 1000]), fps_ragged(y, 2048, [mx - 1000]))


def test_many_waves_and_cluster_independence_at_65536():
    # 64 clouds of 65536 points need clusters of >= 4 CTAs of 128 KB shared memory each: more than one wave
    B, N = 64, 65536
    x, _ = synth.uniform_clouds(B, N, seed=13)
    lengths = torch.randint(N // 4, N + 1, (B,), generator=torch.Generator().manual_seed(3))
    got = {c: raw(x.cuda(), 128, lengths, cluster=c) for c in (0, 4, 8, 16)}
    want = fps_ragged(x, 128, lengths)
    for c, v in got.items():
        assert np.array_equal(v, want), c


def test_results_do_not_depend_on_cluster_size_and_prefix_property():
    x, _ = synth.uniform_clouds(3, 65536, seed=14)
    lengths = [65536, 40000, 20000]
    runs = [raw(x.cuda(), 1024, lengths, cluster=c) for c in (0, 4, 8, 16)]
    assert all(np.array_equal(r, runs[0]) for r in runs[1:])
    assert all(len(np.unique(r)) == 1024 and (r < n).all() for r, n in zip(runs[0], lengths))
    short = raw(x.cuda(), 300, lengths)
    assert np.array_equal(runs[0][:, :300], short)                       # the first m samples of a longer run
    small, _ = synth.uniform_clouds(5, 4096, seed=15)
    runs = [raw(small.cuda(), 700, [4096, 3000, 100, 1, 0], cluster=c) for c in CLUSTERS]
    assert all(np.array_equal(r, runs[0]) for r in runs[1:])


def test_sample_farthest_points_ragged_surface():
    pts = torch.rand(4, 1000, 6, generator=torch.Generator().manual_seed(6)).cuda()
    lengths = torch.tensor([1000, 500, 3, 0]).cuda()

    def check(points, idx, K):
        assert idx.dtype == torch.int64 and idx.shape == (4, max(K)) and points.shape == (4, max(K), 6)
        want = fps_ragged(pts[:, :, :3].cpu(), max(K), lengths.cpu(), K)
        assert np.array_equal(npy(idx), want)
        pad = idx < 0
        assert (points[pad] == 0).all()
        gathered = torch.gather(pts, 1, idx.clamp(min=0).unsqueeze(-1).expand(-1, -1, 6))
        assert torch.equal(points[~pad], gathered[~pad])

    for K in ([64, 10, 8, 5], (7, 7, 7, 7)):
        check(*pcl.sample_farthest_points(pts, lengths=lengths, K=K), list(K))
    Kt = torch.tensor([64, 100, 2, 5]).cuda()
    check(*pcl.sample_farthest_points(pts, lengths=lengths, K=Kt), Kt.tolist())
    check(*pcl.sample_farthest_points(pts, lengths=lengths, K=50), [50] * 4)
    p, i = pcl.sample_farthest_points(pts, lengths=lengths, K=20, random_start_point=True)
    for b, n in enumerate(lengths.tolist()):
        assert (i[b, 0] == -1) if n == 0 else (0 <= int(i[b, 0]) < n)
    # the lengths-free int-K form is unchanged: K > P repeats index 0
    p, i = pcl.sample_farthest_points(pts[:, :10], K=12)
    assert np.array_equal(npy(i), oracle.fps(pts[:, :10, :3].cpu(), 12))


def test_scalar_k_forms_and_random_start_with_long_lengths():
    pts = torch.rand(3, 300, 3, generator=torch.Generator().manual_seed(8)).cuda()
    _, want = pcl.sample_farthest_points(pts, K=40)
    for K in (np.int64(40), torch.tensor(40)):
        assert torch.equal(pcl.sample_farthest_points(pts, K=K)[1], want)
    lengths = torch.tensor([300, 1000, 5]).cuda()                          # 1000 > P: the cloud is all 300 points
    _, ref = pcl.sample_farthest_points(pts, lengths=lengths, K=np.int32(40))
    assert np.array_equal(npy(ref), fps_ragged(pts.cpu(), 40, lengths.cpu()))
    firsts = torch.stack([pcl.sample_farthest_points(pts, lengths=lengths, K=8, random_start_point=True)[1][:, 0]
                          for _ in range(200)])
    assert (firsts >= 0).all() and (firsts[:, 1] < 300).all() and (firsts[:, 2] < 5).all()
    assert (firsts[:, 1] == 299).float().mean() < 0.05                     # drawn from [0, 300), not piled up at P - 1
