"""Pins the float32 restatement of the fused EMD loss epilogue (tests/emd_epilogue_ref.py) to the reference: the golden
gradient of dist.sqrt().mean() went through the reference's own emd_module.py (tests/golden/make_golden.py, raw_*), and
the special values (unassigned points, dist == 0) follow torch's sqrt backward and the reference's backward kernel."""
import numpy as np
import torch

import oracle
from emd_epilogue_ref import epilogue_grad, epilogue_sum, float32_neighbours


def ulp_distance(a, b):
    """Distance in float32 ulps (sign-magnitude bit patterns mapped onto a monotonic integer line)."""
    def line(x):
        i = np.asarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7fffffff), i)
    return np.abs(line(a) - line(b))


def test_restatement_reproduces_the_golden_gradient_through_the_reference_module(golden):
    x1, x2, dist, asg = golden["raw_xyz1"], golden["raw_xyz2"], golden["raw_dist"], golden["raw_assignment"]
    b, n = dist.shape
    grad_scale = np.float32(1.0 / (b * n))            # mean backward: 1/numel, a power of two here
    mine = epilogue_grad(x1, x2, dist, asg, grad_scale)
    ref = golden["raw_grad"]
    assert mine.shape == ref.shape and np.isfinite(ref).all()
    # Not bit for bit: torch's CPU sqrt (vectorised) is not correctly rounded -- it is one ulp off IEEE sqrt on a few
    # elements -- and the golden gradient went through it, while the restatement (like the kernel's __fsqrt_rn) rounds
    # sqrt exactly.  One ulp in sqrt(dist) becomes at most two ulps after the two float32 products that follow.  The
    # recorded golden differs on 29 of 6144 elements, by at most 2 ulps.
    dist_ulp = ulp_distance(mine, ref)
    assert dist_ulp.max() <= 2, dist_ulp.max()
    assert (dist_ulp == 0).mean() >= 0.99


def test_restatement_special_values_follow_torch_and_the_reference_backward():
    """Where sqrt is exact (perfect squares, 0) torch's chain -- sqrt backward, then (2*g) * (x1 - x2[a]) of the reference's
    backward (oracle.emd_backward) -- is reproduced bit for bit, including inf and NaN at dist == 0."""
    x2 = np.array([[[0.0, 0.0, 0.0], [0.5, 0.25, 1.0], [0.3, 0.3, 0.0], [1.0, 1.0, 1.0]]], np.float32)
    x1 = np.array([[[0.5, 0.0, 0.0], [0.5, 0.25, 1.0], [0.3, 0.3, 1e-30], [0.0, 0.0, 1.0]]], np.float32)
    asg = np.array([[0, 1, 2, 3]], np.int32)
    d = ((x1.astype(np.float32) - x2) ** 2).sum(-1).astype(np.float32)  # 0.25, 0, 0 (underflow), 2
    d[0, 3] = np.float32(4.0)                                           # any dist works; keep sqrt exact
    for gs in (np.float32(1.0), np.float32(0.37), np.float32(1.0 / 4)):
        t = torch.from_numpy(d).requires_grad_()
        t.sqrt().backward(torch.full_like(t, float(gs)))
        g_ref, _ = oracle.emd_backward(x1, x2, asg, t.grad.numpy())
        mine = epilogue_grad(x1, x2, d, asg, gs)
        assert np.array_equal(mine, g_ref, equal_nan=True), (mine, g_ref)
        assert np.isnan(mine[0, 1]).all()                 # inf * 0
        assert np.isinf(mine[0, 2, 2]) and np.isnan(mine[0, 2, :2]).all()   # dist underflowed to 0, dz != 0
    # unassigned points (assignment == -1) get exactly 0, like emd_bwd_kernel and the unfused path
    asg_u = np.array([[0, -1, 2, -1]], np.int32)
    g = epilogue_grad(x1, x2, d, asg_u, np.float32(1.0))
    assert not g[0, 1].any() and not g[0, 3].any() and np.array_equal(g[0, 0], epilogue_grad(x1, x2, d, asg, 1.0)[0, 0])


def test_restatement_sum_is_the_exactly_rounded_sum():
    g = np.random.default_rng(3)
    d = (g.random((5, 777)) ** 4).astype(np.float32)
    s, count, mean = epilogue_sum(d)
    assert count == 5 * 777 and mean == s / count
    r = np.sqrt(d).astype(np.float64)
    assert abs(s - r.sum()) <= 1e-12 * s
    lo, mid, hi = float32_neighbours(s)
    assert lo < mid < hi and mid == np.float32(s)
    assert epilogue_sum(np.zeros((2, 3), np.float32))[0] == 0.0
