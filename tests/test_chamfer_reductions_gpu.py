"""GPU tests of Chamfer's reductions and backward against float64 references built from the kernel's own nearest neighbours:
  loss_xy[0..3] (finish_block, pcl_chamfer.cu: one lane per cloud, clouds 32 apart in one lane) at batch sizes above 32
  with ragged lengths that include 0, 1 and P, both arithmetic modes, the brute-force and the pruned path;
  the gradient of pcl.chamfer_distance (chamfer_bwd_kernel: fp32 atomics, g / B / len) against an fp64 scatter, for every
  D, fp16 / bf16 inputs and an upstream gradient other than 1.
Distances and indices are checked bit for bit against the CPU oracle at every shape (the oracle costs seconds even at
2 x 20000 points)."""
import math

import numpy as np
import pytest
import torch

import oracle
import pointcloud_b200 as pcl
from helpers import npy

pytestmark = pytest.mark.gpu
REL = 1e-5  # north star tolerance for fp32 scalars and gradients


@pytest.fixture
def prune_min():
    """Sets the pruned path's switch-over (pcl_chamfer_set_prune_min) for one test and restores the default afterwards."""
    L = pcl._lib.lib()
    yield L.pcl_chamfer_set_prune_min
    L.pcl_chamfer_set_prune_min(-1)


def ragged_lengths(g, b, p, special):
    """int64 lengths in [0, p] with the values 0, 1 and p at the positions `special` (the last one past the first 32 clouds)."""
    ln = torch.randint(0, p + 1, (b,), generator=g)
    for pos, v in zip(special, (0, 1, p)):
        ln[pos] = v
    return ln


def make_case(b, p1, p2, d, ragged, seed):
    g = torch.Generator().manual_seed(seed)
    x, y = torch.rand(b, p1, d, generator=g), torch.rand(b, p2, d, generator=g)
    if not ragged:
        return x, y, None, None
    if b == 2:
        return x, y, torch.tensor([p1, p1 - 1]), torch.tensor([p2 - 3, p2])
    # x: 0, 1, P1 at clouds 0, 1, b-1; y: 0, 1, P2 at clouds 2, 0, 1 -- an empty cloud against a full one and both ways round
    return x, y, ragged_lengths(g, b, p1, (0, 1, b - 1)), ragged_lengths(g, b, p2, (2, 0, 1))


def loss_reference(dist, lengths, p):
    """(batch mean, batch sum) of sum_i dist[b, i < len_b] / max(len_b, 1) in float64 (math.fsum per cloud and over clouds)."""
    b = dist.shape[0]
    per = []
    for n in range(b):
        ln = p if lengths is None else int(lengths[n])
        per.append(math.fsum(dist[n, :ln].astype(np.float64).tolist()) / max(ln, 1))
    total = math.fsum(per)
    return total / max(b, 1), total


def close(got, want):
    return abs(float(got) - want) <= REL * abs(want) + 1e-30


# (B, P1, P2, ragged): above 32 clouds (the second and later trips of finish_block's cloud loop), then the full sizes
LOSS_CASES = [(33, 700, 1000, True), (64, 500, 300, True), (100, 300, 700, True), (1000, 300, 257, True),
              (32, 2048, 2048, True), (4, 16384, 16384, False), (2, 20000, 20000, True)]


@pytest.mark.parametrize("prune", ["never", "forced", "default"])
@pytest.mark.parametrize("mode", ["unfused", "fma"])
@pytest.mark.parametrize("b,p1,p2,ragged", LOSS_CASES)
def test_loss_xy_against_float64_of_the_kernels_distances(prune_min, b, p1, p2, ragged, mode, prune):
    """loss_xy[0..1] = (sum_b fsum(dist[b, :len_b]) / max(len_b, 1)) / max(B, 1) and loss_xy[2..3] the un-normalised sums.
    "forced" prunes every size up to the pruned path's 16384-point limit (2 x 20000 stays brute-force); "default" prunes
    from 6144 points on."""
    if prune == "default" and min(p1, p2) < 6144:
        pytest.skip("below 6144 points the default is the brute-force path, run as 'never'")
    prune_min({"never": 0, "forced": 1, "default": -1}[prune])
    x, y, xl, yl = make_case(b, p1, p2, 3, ragged, seed=b + p1 + p2)
    o = oracle.chamfer_forward(x, y, xl, yl, mode=0 if mode == "unfused" else 1, nthreads=16)
    r = pcl.chamfer_forward_raw(x.cuda(), y.cuda(), xl, yl, mode=mode)
    for k in ("dist_x", "idx_x", "dist_y", "idx_y"):
        assert np.array_equal(npy(r[k]), o[k]), k
    loss = npy(torch.cat([r["loss_xy"], r["loss_sums"]]))
    for d, (dist, ln, p) in enumerate(((npy(r["dist_x"]), xl, p1), (npy(r["dist_y"]), yl, p2))):
        mean, total = loss_reference(dist, None if ln is None else ln.numpy(), p)
        assert close(loss[d], mean) and close(loss[2 + d], total), (d, loss, mean, total)
    assert close(loss[0], float(o["loss_x"])) and close(loss[1], float(o["loss_y"]))


def grad_reference(x, y, idx_x, idx_y, xl, yl, g):
    """fp64 d(g * (loss_x + loss_y)) / d(x, y) through the given nearest neighbours: np.add.at scatters onto the targets."""
    x, y = x.astype(np.float64), y.astype(np.float64)
    b, p1, _ = x.shape
    p2 = y.shape[1]
    gx, gy = np.zeros_like(x), np.zeros_like(y)
    for n in range(b):
        lx = p1 if xl is None else int(xl[n])
        ly = p2 if yl is None else int(yl[n])
        if lx == 0 or ly == 0:
            continue
        for q, t, gq, gt, lq, idx in ((x, y, gx, gy, lx, idx_x), (y, x, gy, gx, ly, idx_y)):
            j = idx[n, :lq].astype(np.int64)
            diff = (2.0 * g / max(b, 1) / lq) * (q[n, :lq] - t[n, j])
            gq[n, :lq] += diff
            np.add.at(gt[n], j, -diff)
    return gx, gy


def dtype_ulp(r, dt):
    """Spacing of `dt` (fp16 / bf16) at |r|, subnormals included."""
    man, tiny = {torch.float16: (10, 2.0 ** -24), torch.bfloat16: (7, 2.0 ** -133)}[dt]
    e = np.floor(np.log2(np.maximum(np.abs(r), 1e-300)))
    return np.maximum(2.0 ** (e - man), tiny)


def check_grad(got, want, dt=torch.float32):
    got = got.astype(np.float64)
    tol = REL * np.abs(want) + 1e-6 * max(np.abs(want).max(), 1e-30)
    if dt != torch.float32:                 # the gradient is returned in the input's dtype: one rounding to it
        tol = tol + dtype_ulp(want, dt)
    bad = np.abs(got - want) > tol
    assert not bad.any(), (int(bad.sum()), got[bad][:5], want[bad][:5])


GRAD_CASES = [(b, p1, p2, 3, ragged, torch.float32) for b, p1, p2, ragged in LOSS_CASES] + \
             [(40, 300, 257, d, True, torch.float32) for d in (1, 2, 4, 5, 7, 8)] + \
             [(40, 700, 600, 3, True, dt) for dt in (torch.float16, torch.bfloat16)] + [(2, 333, 444, 5, True, torch.float16)]


@pytest.mark.parametrize("b,p1,p2,d,ragged,dt", GRAD_CASES)
def test_chamfer_gradient_against_float64_scatter(b, p1, p2, d, ragged, dt):
    """pcl.chamfer_distance autograd with upstream gradient 0.37 against the fp64 scatter over the kernel's own indices;
    padded rows get exactly 0; the gradient comes back in each input's dtype."""
    x, y, xl, yl = make_case(b, p1, p2, d, ragged, seed=7 * b + p1 + d)
    xg = x.to(dt).cuda().requires_grad_()
    yg = y.cuda().requires_grad_()
    loss, _ = pcl.chamfer_distance(xg, yg, x_lengths=None if xl is None else xl.cuda(), y_lengths=None if yl is None else yl.cuda())
    (loss * 0.37).backward()
    assert xg.grad.dtype == dt and yg.grad.dtype == torch.float32
    r = pcl.chamfer_forward_raw(xg.detach(), yg.detach(), xl, yl)
    xv = xg.detach().float().cpu().numpy()                       # the values the kernel read
    o = oracle.chamfer_forward(xv, y, xl, yl, nthreads=16)
    assert np.array_equal(npy(r["idx_x"]), o["idx_x"]) and np.array_equal(npy(r["idx_y"]), o["idx_y"])
    assert abs(float(loss) - float(o["loss"])) <= REL * float(o["loss"])
    gx, gy = grad_reference(xv, y.numpy(), npy(r["idx_x"]), npy(r["idx_y"]), None if xl is None else xl.numpy(),
                            None if yl is None else yl.numpy(), 0.37)
    check_grad(npy(xg.grad.float()), gx, dt)
    check_grad(npy(yg.grad), gy)
    for n in range(b):                                            # padded rows: exactly 0
        if xl is not None:
            assert not xg.grad[n, int(xl[n]):].any()
        if yl is not None:
            assert not yg.grad[n, int(yl[n]):].any()
