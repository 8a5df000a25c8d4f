"""The auction EMD outside the unit cube, on every path, against the CPU oracle bit for bit.

The reference tuned eps for clouds in [0,1]^3, but nothing in the kernels assumes that range: the skip filter of the Bid scan
rounds in the safe direction at any magnitude (DESIGN.md "Why skipping is exact", tests/test_emd_filter_cpu.py).  Here the
kernels run on tiny, large, far-from-origin and per-axis mixed-scale clouds, lattice ties and duplicate targets at scale 100
(near-ties at the ulp level are where an unsound skip would change a bid), and fp16 predictions at scale 100.

The kernel's Morton key quantises [0,1]^3, so outside it the internal order of a cloud is mostly its input order.  The clouds
are therefore handed over sorted along a Morton curve of their own bounding box: tiles of 32 targets are compact, and whole
tiles are skipped at every scale (checked through stats[:, 4:6]) -- otherwise the tile test would not be exercised.  The order
changes no result (every tie rule works on original indices), and the oracle runs on the same clouds."""
import numpy as np
import pytest
import torch

import oracle
import pointcloud_b200 as pcl
from emd_epilogue_ref import epilogue_grad, epilogue_sum, float32_neighbours
from helpers import npy, same_bits

pytestmark = pytest.mark.gpu
B, N, EPS, ITERS = 3, 2048, 0.005, 50
F_COLD = 4                                # launch flag in stats[:, 6] (pcl_emd_core.cuh EMD_F_COLD)
PATHS = ["cluster", "team", "tickets"]
CASES = ["scale 1e-3", "scale 16", "scale 100", "scale 1e3", "offset 1e3", "mixed axes", "grid ties x100",
         "duplicate targets x100", "fp16 x100"]


@pytest.fixture
def emd_path():
    """Selects an auction kernel for one test and restores the automatic choice afterwards."""
    yield pcl.set_emd_path
    pcl.set_emd_path("auto")


def morton_sorted(x):
    """(B, N, 3) float32: every cloud re-ordered along a 30-bit Morton curve over its own bounding box."""
    out = []
    for c in x.numpy():
        lo, hi = c.min(0).astype(np.float64), c.max(0).astype(np.float64)
        q = ((c - lo) / np.where(hi > lo, hi - lo, 1.0) * 1023).astype(np.int64)
        key = np.zeros(len(c), np.int64)
        for bit in range(10):
            for axis in range(3):
                key |= ((q[:, axis] >> bit) & 1) << (3 * bit + axis)
        out.append(c[np.argsort(key, kind="stable")])
    return torch.from_numpy(np.stack(out))


def clouds(case, b=B, n=N, seed=0):
    """(prediction, target) on the CPU; the prediction is fp16 for "fp16 x100", every other tensor fp32."""
    g = torch.Generator().manual_seed(seed)
    x1, x2 = torch.rand(b, n, 3, generator=g), torch.rand(b, n, 3, generator=g)
    if case.startswith("scale"):
        s = float(case.split()[1])
        x1, x2 = x1 * s, x2 * s
    elif case == "offset 1e3":                 # unit spread 1000 away from the origin: ulp(1000) = 6.1e-5
        x1, x2 = x1 + 1000.0, x2 + 1000.0
    elif case == "mixed axes":                 # x in [0, 0.01], y in [0, 1], z in [0, 100]
        axes = torch.tensor([0.01, 1.0, 100.0])
        x1, x2 = x1 * axes, x2 * axes
    elif case == "grid ties x100":             # a coarse lattice: thousands of equal distances and equal values
        x1 = torch.randint(0, 6, (b, n, 3), generator=g).float() / 6 * 100
        x2 = torch.randint(0, 6, (b, n, 3), generator=g).float() / 6 * 100
    elif case == "duplicate targets x100":     # every target eight times
        x1, x2 = x1 * 100, (x2[:, : n // 8] * 100).repeat(1, 8, 1)
    elif case == "fp16 x100":
        x1, x2 = x1 * 100, x2 * 100
    x1, x2 = morton_sorted(x1.float()), morton_sorted(x2.float())
    return (x1.half() if case.startswith("fp16") else x1), x2


_ORACLE = {}


def oracle_of(case, b=B, n=N):
    """(prediction, target, oracle result) per case; the oracle sees the fp32 values the kernel reads (fp16 up-cast)."""
    if (case, b, n) not in _ORACLE:
        x1, x2 = clouds(case, b, n)
        _ORACLE[(case, b, n)] = (x1, x2, oracle.emd_forward(x1.float(), x2, EPS, ITERS, nthreads=b))
    return _ORACLE[(case, b, n)]


def check_skipping(st, n):
    """Whole tiles were skipped on every cloud: the executed pair evaluations (stats[4:6]) stay below N per bidder turn."""
    evals = st[:, 4].astype(np.uint32).astype(np.uint64) + (st[:, 5].astype(np.uint32).astype(np.uint64) << np.uint64(32))
    assert (evals < np.uint64(n) * st[:, 0].astype(np.uint64)).all(), (evals, st[:, 0])


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("path", PATHS)
def test_every_path_is_bit_exact_vs_oracle_at_every_scale(emd_path, path, case):
    x1, x2, o = oracle_of(case)
    emd_path(path)
    d, a, st = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), EPS, ITERS, want_stats=True)
    assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
    st = npy(st)
    assert np.array_equal(st[:, 0], o["sum_unass"]) and np.array_equal(st[:, 1], o["iters_run"])
    assert (st[:, 3] == 0).all() if path == "team" else (st[:, 3] > 0).all(), st[:, 3]
    check_skipping(st, N)


def test_cluster_path_with_the_auction_state_in_l2_at_scale_100(emd_path):
    """N = 5000 > 3584: the cold half of the auction state lives in global memory (L2)."""
    x1, x2, o = oracle_of("scale 100", b=2, n=5000)
    emd_path("cluster")
    d, a, st = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), EPS, ITERS, want_stats=True)
    assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
    st = npy(st)
    assert np.array_equal(st[:, 0], o["sum_unass"]) and np.array_equal(st[:, 1], o["iters_run"])
    assert ((st[:, 6] & F_COLD) != 0).all(), st[:, 6]
    check_skipping(st, 5000)


@pytest.mark.parametrize("path", PATHS)
def test_fused_loss_epilogue_at_scale_100(emd_path, path):
    """pcl_emd_fwd_fused: the gradient of sum sqrt(dist) bit for bit against the float32 restatement, the sum to within one
    float32 ulp of the exactly rounded sum."""
    x1, x2, o = oracle_of("scale 100")
    emd_path(path)
    d, a, st, grad, sums = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), EPS, ITERS, want_stats=True, want_epilogue=True)
    assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
    assert same_bits(npy(grad), epilogue_grad(x1.numpy(), x2.numpy(), o["dist"], o["assignment"], 1.0))
    s, count, _ = epilogue_sum(o["dist"])
    sums = npy(sums)
    assert sums[1] == np.float32(count) and sums[0] in float32_neighbours(s), (sums, s)
    assert sums[2] == np.float32(sums[0]) / np.float32(sums[1])
    check_skipping(npy(st), N)
