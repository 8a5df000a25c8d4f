"""float32 restatement of the auction kernel's fused loss epilogue (pcl_emd_fwd_fused, include/pcl.h).

Given the predictions, the targets and the auction's (dist, assignment), the epilogue writes
  grad = 2 * (grad_scale / (2 * sqrt(dist))) * (xyz1 - xyz2[assignment])
in the operation order of torch's sqrt backward (grad / (2 * result)) followed by the reference's
NmDistanceGradKernel ((2 * g) * (x1 - x2)), and sum sqrt(dist) in fp64.  Every step below is one IEEE-rounded
float32 operation, so `epilogue_grad` is a bit-exact expectation of the kernel's gradient; `epilogue_sum` is the
exactly rounded sum the kernel's fixed-order fp64 reduction approximates.
"""
import math

import numpy as np


def epilogue_grad(xyz1, xyz2, dist, assignment, grad_scale):
    """(B, N, 3) float32.  Unassigned points (assignment == -1) get 0, like emd_bwd_kernel; an assigned point with
    dist == 0 gets inf or NaN, like dists.sqrt() in the reference."""
    x1 = np.asarray(xyz1, dtype=np.float32)
    x2 = np.asarray(xyz2, dtype=np.float32)
    d = np.asarray(dist, dtype=np.float32)
    a = np.asarray(assignment).astype(np.int64)
    two = np.float32(2.0)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        g2 = (np.float32(grad_scale) / (two * np.sqrt(d))) * two
        matched = np.take_along_axis(x2, np.maximum(a, 0)[..., None], 1)
        grad = g2[..., None] * (x1 - matched)
    grad[a < 0] = 0.0
    return grad.astype(np.float32, copy=False)


def epilogue_sum(dist):
    """(sum, count, mean) of float32 sqrt(dist) over the whole batch: the sum exactly rounded from the float64 values
    (math.fsum), count = B*N, mean = sum / count in float64."""
    d = np.asarray(dist, dtype=np.float32)
    s = math.fsum(np.sqrt(d).astype(np.float64).ravel().tolist())
    count = d.size
    return s, count, s / count if count else float("nan")


def float32_neighbours(v):
    """float32(v) and its two float32 neighbours: the values a fixed-order fp64 sum of many terms may round to."""
    f = np.float32(v)
    return (np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf)))
