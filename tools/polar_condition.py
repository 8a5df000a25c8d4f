"""Why pcl_icp.cu solves the alignment with a one-sided Jacobi SVD of M rather than an eigen-decomposition of M^T M
(DESIGN.md, "alignment / ICP exactness").  CPU only, numpy float64.

For random 3 x 3 matrices M = Q1 diag(sigma) Q2^T with det Q1 = det Q2 = +1, it forms R = U V^T the way the kernel would
with eigh(M^T M): V and sigma^2 from the eigen-decomposition (v3 negated if det V < 0), u1 = M v1 / sigma1, u2 = M v2
orthogonalised against u1, u3 = u1 x u2; and compares it with R from numpy's SVD of M itself, whose error is about
2^-52 sigma1 / (sigma_i + sigma_j).  The eigen route squares the condition: its error grows like
2^-52 sigma1^2 / (sigma2 (sigma2 + sigma3)).

  python tools/polar_condition.py [--cases N] [--sigma 1 1e-6 0.3e-6]
"""
import argparse

import numpy as np


def proper_q(rng):
    q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
    if np.linalg.det(q) < 0:
        q[:, 0] *= -1
    return q


def r_from_eigh(M):
    lam, V = np.linalg.eigh(M.T @ M)
    V = V[:, ::-1]
    if np.linalg.det(V) < 0:
        V[:, 2] *= -1
    s1 = np.sqrt(max(lam[-1], 0.0))
    u1 = M @ V[:, 0] / s1
    u2 = M @ V[:, 1]
    u2 -= u1 * (u1 @ u2)
    u2 /= np.linalg.norm(u2)
    return np.stack([u1, u2, np.cross(u1, u2)], 1) @ V.T


def r_from_svd(M):
    U, _, Vt = np.linalg.svd(M)
    return U @ np.diag([1.0, 1.0, np.linalg.det(U @ Vt)]) @ Vt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", type=int, default=200)
    ap.add_argument("--sigma", type=float, nargs=3, default=[1.0, 1e-6, 0.3e-6])
    args = ap.parse_args()
    rng = np.random.default_rng(0)
    errs = []
    for _ in range(args.cases):
        M = proper_q(rng) @ np.diag(args.sigma) @ proper_q(rng).T
        errs.append(np.abs(r_from_eigh(M) - r_from_svd(M)).max())
    print(f"sigma = {args.sigma}, {args.cases} cases: max |R_eigh - R_svd| median {np.median(errs):.2e}, worst {np.max(errs):.2e}"
          f" (fp32 ulp at 1: {2.0 ** -23:.2e})")


if __name__ == "__main__":
    main()
