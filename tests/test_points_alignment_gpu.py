"""corresponding_points_alignment and iterative_closest_point on the GPU against tests/icp_ref.py (float64) and against
the loop of the library's own public parts.

Alignment accuracy bound.  The kernels and the reference both start from the fp32 inputs up-cast to fp64, so their
covariances M agree to a few units of 2^-52 ||M|| (the sums differ in order only).  R = U V^T is the polar factor of M;
for a perturbation dM it moves by at most 2 ||dM|| / min_{i<j} (sig'_i + sig'_j), with sig' the singular values with the
sign of det(U V^T) on the last one (this is the H_ij denominator of the backward).  Where min (sig'_i + sig'_j) >= 1e-6
sig_1 (with allow_reflection also 2 |sig'_3| >= 1e-6 sig_1: the sign of u3 is free where sig_3 = 0), the fp64 R of both sides therefore agree to 2 * 2^-50 * 1e6 < 2e-9, and what is left is the one rounding of each
entry (|R_ij| <= 1) to fp32: 2^-25.  The test allows 2^-23.  T = ym - s (xm R) is rounded once from an fp64 value that
carries the same relative error times |xm|: the test allows 2 fp32 ulps of |T| + 1e-7 (1 + |xm|); s: 2 ulps.
Degenerate clouds (all points equal, collinear, P <= 3) have no unique R: they must give finite proper rotations, the same
bits on every run, and tr(R^T M) within 1e-6 ||M|| of the maximum sig'_1 + sig'_2 + sig'_3.

Backward.  Distinct singular values: against autograd through the float64 torch.linalg.svd restatement, within 1e-4
relative + 1e-4 of the largest entry.  Repeated singular values (cube vertices): torch's SVD backward divides by
sig_i^2 - sig_j^2 = 0 there; the closed form must stay finite and match central differences of the restatement."""
import math

import numpy as np
import pytest
import torch

import pointcloud_b200 as pcl
from helpers import npy, same_bits
from icp_ref import alignment_parts, alignment_ref, apply_ref, axis_angle, icp_ref, nn_dense, random_rotation
from pointcloud_b200 import _lib, synth
from test_stale_state_gpu import PATTERNS, Stale, capture_and_replay

pytestmark = pytest.mark.gpu

F32 = torch.float32


def table(b, n, seed):
    return synth.table_clouds(b, n, seed=seed)[0]


def pair(b, n, seed, angle=15.0, shift=0.05, noise=0.002, n2=None):
    """Table-shaped X and Y = X rotated by <= angle degrees, shifted by <= shift, noisy and shuffled; also the truth."""
    g = torch.Generator().manual_seed(seed)
    X = table(b, n, seed).double()
    R = random_rotation(b, g, math.radians(angle))
    T = (torch.rand(b, 3, generator=g, dtype=torch.float64) * 2 - 1) * shift
    src = X if n2 is None else table(b, n2, seed + 1000).double()
    Y = apply_ref(src, R, T, torch.ones(b, dtype=torch.float64)) + noise * torch.randn(*src.shape, generator=g, dtype=torch.float64)
    Y = Y[:, torch.randperm(src.shape[1], generator=g)]
    return X.float(), Y.float(), R, T


def signed_sigmas(M):
    U, S, Vh = torch.linalg.svd(M)
    d = torch.det(torch.bmm(U, Vh))
    return torch.cat([S[:, :2], (S[:, 2] * d)[:, None]], 1)


def ulp(x):
    return np.spacing(np.abs(np.asarray(x, np.float32))).astype(np.float64)


# ---------------------------------------------------------------- alignment forward ------------------------------------

def alignment_case(b, p, seed, weighted, ragged, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    X = torch.rand(b, p, 3, generator=g) if p < 64 else table(b, p, seed)
    R = random_rotation(b, g).float()
    Y = (scale * torch.bmm(X, R) + torch.randn(b, 1, 3, generator=g) + 0.01 * torch.randn(b, p, 3, generator=g)).float()
    w = torch.rand(b, p, generator=g) + 0.1 if weighted else None
    lengths = torch.randint(0, p + 1, (b,), generator=g) if ragged else None
    if ragged:
        lengths[0] = 0
        lengths[-1] = p
    return X, Y, w, lengths


def check_alignment(X, Y, w, lengths, est, refl):
    r = pcl.points_alignment_forward_raw(X.cuda(), Y.cuda(), None if w is None else w.cuda(), est, refl, 1e-9,
                                         None if lengths is None else lengths.cuda())
    R, T, s = npy(r["R"]).astype(np.float64), npy(r["T"]).astype(np.float64), npy(r["s"]).astype(np.float64)
    x64, y64 = X.double(), Y.double()
    Rr, Tr, sr = (t.numpy() for t in alignment_ref(x64, y64, w, est, refl, 1e-9, lengths))
    M, _, xm, _ = alignment_parts(x64, y64, w, 1e-9, lengths)
    sg = signed_sigmas(M)
    if refl:
        sg = sg.abs()
    b = X.shape[0]
    assert np.isfinite(R).all()
    assert (np.abs(np.einsum("bji,bjk->bik", R, R) - np.eye(3)) <= 2.0 ** -21).all()
    if not refl:
        assert (np.abs(np.linalg.det(R) - 1) <= 2.0 ** -20).all()
    sums = [sg[:, 0] + sg[:, 1], sg[:, 0] + sg[:, 2], sg[:, 1] + sg[:, 2]] + ([2 * sg[:, 2]] if refl else [])
    pair_min = torch.stack(sums, 1).min(1).values.numpy()
    ok = pair_min > 1e-6 * sg[:, 0].abs().numpy()
    assert (np.abs(R - Rr)[ok] <= 2.0 ** -23).all()
    tol_t = 2 * ulp(Tr) + 1e-7 * (1 + np.abs(xm.numpy()).max(1, keepdims=True))
    assert (np.abs(T - Tr)[ok] <= tol_t[ok]).all()
    assert (np.abs(s - sr)[ok] <= 2 * ulp(sr)[ok]).all()
    # where R is not unique, it still attains the maximum of tr(R^T M)
    Mn = M.numpy()
    got = np.einsum("bij,bij->b", R, Mn)
    best = sg.sum(1).numpy()
    assert (np.abs(got - best) <= 1e-6 * np.linalg.norm(Mn, axis=(1, 2)) + 1e-30).all()
    return r, ok.sum(), b


@pytest.mark.parametrize("p", [1, 2, 3, 4, 333, 2048, 65536])
@pytest.mark.parametrize("weighted,ragged", [(False, False), (True, False), (True, True), (False, True)])
@pytest.mark.parametrize("est,refl", [(False, False), (True, False), (False, True), (True, True)])
def test_alignment_forward(p, weighted, ragged, est, refl):
    b = 64 if p <= 2048 else 3
    X, Y, w, lengths = alignment_case(b, p, p + 7 * weighted + 3 * ragged, weighted, ragged, scale=1.7 if est else 1.0)
    _, n_ok, _ = check_alignment(X, Y, w, lengths, est, refl)
    if p >= 4 and not ragged:
        assert n_ok == b  # random clouds of 4 or more points are well conditioned


def test_alignment_degenerate_clouds():
    g = torch.Generator().manual_seed(21)
    b, p = 4, 50
    X = torch.rand(b, p, 3, generator=g)
    Y = torch.rand(b, p, 3, generator=g)
    X[0] = X[0, :1]                                             # all points equal
    t = torch.rand(p, 1, generator=g)
    X[1] = t * torch.tensor([1.0, 2.0, -0.5])                  # collinear
    Y[1] = t * torch.tensor([0.3, -1.0, 0.2]) + 0.1
    Y[2] = Y[2, :1]                                             # Y all equal: M = 0, R = I
    runs = [check_alignment(X, Y, None, None, est, False)[0] for est in (False, True)]
    for r in runs:
        again = pcl.points_alignment_forward_raw(X.cuda(), Y.cuda(), estimate_scale=r is runs[1])
        assert same_bits(npy(again["R"]), npy(r["R"])) and same_bits(npy(again["T"]), npy(r["T"]))
    assert np.array_equal(npy(runs[0]["R"])[2], np.eye(3, dtype=np.float32)) and np.array_equal(npy(runs[0]["R"])[0], np.eye(3, dtype=np.float32))
    for p_small in (1, 2, 3):
        check_alignment(X[:, :p_small], Y[:, :p_small], None, None, False, False)


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("est", [False, True])
def test_alignment_of_clouds_without_rows(weighted, est):
    """P = 0 (a zero-size tensor may have a NULL data pointer): M = 0, so R = I, T = 0 and s = 0 / max(0, eps) = 0 with
    estimate_scale (1 without), as the float64 restatement gives; the backward gives empty gradients."""
    b = 3
    X = torch.empty(b, 0, 3, device="cuda").requires_grad_()
    Y = torch.empty(b, 0, 3, device="cuda").requires_grad_()
    w = torch.empty(b, 0, device="cuda").requires_grad_() if weighted else None
    R, T, s = pcl.corresponding_points_alignment(X, Y, w, est)
    assert np.array_equal(npy(R), np.broadcast_to(np.eye(3, dtype=np.float32), (b, 3, 3)))
    assert not npy(T).any() and np.array_equal(npy(s), np.full(b, 0.0 if est else 1.0, np.float32))
    Rr, Tr, sr = alignment_ref(torch.zeros(b, 0, 3, dtype=torch.float64), torch.zeros(b, 0, 3, dtype=torch.float64),
                               None if w is None else torch.zeros(b, 0, dtype=torch.float64), est)
    assert not Tr.any() and torch.equal(sr, torch.full((b,), 0.0 if est else 1.0, dtype=torch.float64))
    (R.sum() + T.sum() + (s.sum() if est else 0)).backward()
    assert X.grad.shape == (b, 0, 3) and Y.grad.shape == (b, 0, 3)


def test_icp_of_clouds_without_rows():
    """P1 = 0: every cloud is empty, rmse is 0 every iteration, 0 / 0 never passes, so the loop runs max_iterations with
    R = I, T = 0, s = 1; P2 = 0 as well: Ynn = 0 wherever X has rows."""
    b = 2
    X0, Y = torch.empty(b, 0, 3, device="cuda"), pair(b, 50, 98)[1].cuda()
    r = pcl.iterative_closest_point(X0, Y, max_iterations=4)
    assert r.converged is False and len(r.t_history) == 4 and r.Xt.shape == (b, 0, 3)
    assert not npy(r.rmse).any() and not npy(r.RTs.T).any() and np.array_equal(npy(r.RTs.s), np.ones(b, np.float32))
    assert np.array_equal(npy(r.RTs.R), np.broadcast_to(np.eye(3, dtype=np.float32), (b, 3, 3)))
    X = pair(b, 40, 99)[0].cuda()
    r = pcl.iterative_closest_point(X, torch.empty(b, 0, 3, device="cuda"), max_iterations=3)
    ref = icp_ref(X.cpu().double(), torch.zeros(b, 0, 3, dtype=torch.float64), max_iterations=3)
    assert r.converged == ref["converged"] and len(r.t_history) == len(ref["t_history"])
    np.testing.assert_allclose(npy(r.rmse), ref["rmse"].numpy(), rtol=1e-6)
    xc = X.double() - X.double().mean(1, keepdim=True)          # R = I and T = -xm: every Ynn is 0
    np.testing.assert_allclose(npy(r.Xt), xc.cpu().numpy(), rtol=0, atol=1e-6)


def test_backward_sees_in_place_changes_of_the_weights():
    X, Y = torch.rand(2, 30, 3, device="cuda").requires_grad_(), torch.rand(2, 30, 3, device="cuda")
    w = torch.rand(2, 30, device="cuda").requires_grad_()
    R, T, s = pcl.corresponding_points_alignment(X, Y, w)
    with torch.no_grad():
        w.mul_(2)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        (R.sum() + T.sum()).backward()


# ---------------------------------------------------------------- alignment backward -----------------------------------

def grads_gpu(X, Y, w, lengths, est, refl, gR, gT, gs):
    xg, yg = X.cuda().requires_grad_(), Y.cuda().requires_grad_()
    wg = None if w is None else w.cuda().requires_grad_()
    R, T, s = pcl.corresponding_points_alignment(xg, yg, wg, est, refl, lengths=None if lengths is None else lengths.cuda())
    loss = (R * gR.cuda()).sum() + (T * gT.cuda()).sum() + ((s * gs.cuda()).sum() if est else 0)
    loss.backward()
    return npy(xg.grad), npy(yg.grad), None if w is None else npy(wg.grad)


def ref_loss(X, Y, w, lengths, est, refl, gR, gT, gs):
    R, T, s = alignment_ref(X, Y, w, est, refl, 1e-9, lengths)
    return (R * gR.double()).sum() + (T * gT.double()).sum() + ((s * gs.double()).sum() if est else 0)


@pytest.mark.parametrize("weighted,ragged,est,refl", [(False, False, False, False), (True, False, True, False),
                                                      (True, True, True, True), (False, True, True, False)])
def test_alignment_backward_distinct_singular_values(weighted, ragged, est, refl):
    g = torch.Generator().manual_seed(31)
    b, p = 6, 300
    X = torch.rand(b, p, 3, generator=g) * torch.tensor([1.0, 0.6, 0.3])    # distinct extents: relative gaps >= 1e-3
    Y = torch.bmm(X, random_rotation(b, g).float()) * 1.3 + 0.5 + 0.05 * torch.randn(b, p, 3, generator=g)
    w = torch.rand(b, p, generator=g) + 0.2 if weighted else None
    lengths = torch.tensor([p, 150, 60, p, 40, 299]) if ragged else None
    gR, gT, gs = torch.randn(b, 3, 3, generator=g), torch.randn(b, 3, generator=g), torch.randn(b, generator=g)
    M = alignment_parts(X.double(), Y.double(), w, 1e-9, lengths)[0]
    S = torch.linalg.svdvals(M)
    assert ((S[:, :2] - S[:, 1:]) >= 1e-3 * S[:, :1]).all()
    gx, gy, gw = grads_gpu(X, Y, w, lengths, est, refl, gR, gT, gs)
    xr, yr = X.double().requires_grad_(), Y.double().requires_grad_()
    wr = None if w is None else w.double().requires_grad_()
    ref_loss(xr, yr, wr, lengths, est, refl, gR, gT, gs).backward()
    for got, want in [(gx, xr.grad), (gy, yr.grad)] + ([(gw, wr.grad)] if weighted else []):
        want = want.numpy()
        np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * np.abs(want).max())
    if ragged:
        for k, n in enumerate(lengths.tolist()):
            assert not gx[k, n:].any() and not gy[k, n:].any() and (gw is None or not gw[k, n:].any())


def test_alignment_backward_repeated_singular_values():
    cube = torch.tensor([[x, y, z] for x in (-1.0, 1.0) for y in (-1.0, 1.0) for z in (-1.0, 1.0)])
    R0 = axis_angle(torch.tensor([[0.0, 0.6, 0.8]], dtype=torch.float64), torch.tensor([0.7], dtype=torch.float64)).float()
    X = (cube * 0.5 + 0.2)[None]
    Y = torch.bmm(X, R0) + torch.tensor([0.1, -0.2, 0.3])
    w = torch.linspace(0.5, 1.5, 8)[None]
    M = alignment_parts(X.double(), Y.double())[0]
    S = torch.linalg.svdvals(M)[0]
    assert float(S.max() - S.min()) < 1e-6 * float(S.max())        # sig_1 = sig_2 = sig_3
    g = torch.Generator().manual_seed(41)
    gR, gT, gs = torch.randn(1, 3, 3, generator=g), torch.randn(1, 3, generator=g), torch.randn(1, generator=g)
    for wt in (None, w):
        gx, gy, gw = grads_gpu(X, Y, wt, None, True, False, gR, gT, gs)
        assert np.isfinite(gx).all() and np.isfinite(gy).all()
        h, scale = 1e-6, 0.0
        for which, base, got in [("x", X, gx), ("y", Y, gy)] + ([("w", wt, gw)] if wt is not None else []):
            fd = np.zeros(base.numel())
            flat = base.double().reshape(-1)
            for k in range(flat.numel()):
                vals = []
                for sgn in (1, -1):
                    q = flat.clone()
                    q[k] += sgn * h
                    q = q.view(base.shape)
                    args = dict(x=X.double(), y=Y.double(), w=None if wt is None else wt.double())
                    args[which] = q
                    vals.append(float(ref_loss(args["x"], args["y"], args["w"], None, True, False, gR, gT, gs)))
                fd[k] = (vals[0] - vals[1]) / (2 * h)
            scale = max(scale, np.abs(fd).max())  # the weights' gradient of an exact fit is ~0: judged on the points' scale
            np.testing.assert_allclose(got.reshape(-1), fd, rtol=1e-4, atol=1e-4 * scale)


# ---------------------------------------------------------------- ICP: the loop of its own public parts ----------------

def replay_check(X, Y, xl, yl, init=None, est=False, K=6, thr=1e-6):
    """icp(max_iterations=k) against alignment(X, Ynn of icp(k-1).Xt) for k = 1..K, bit for bit; rmse within 1 ulp of the
    float64 replay; the stopping iteration from the returned fp32 rmse history."""
    Xc, Yc = X.cuda(), Y.cuda()
    xlc, ylc = (None if t is None else t.cuda() for t in (xl, yl))
    b, p1, _ = X.shape
    mask = (torch.arange(p1)[None] < (xl if xl is not None else torch.full((b,), p1))[:, None]).float().cuda()
    full = pcl.iterative_closest_point(Xc, Yc, init, K, thr, est, x_lengths=xlc, y_lengths=ylc)
    raw = pcl.icp_forward_raw(Xc, Yc, init, K, thr, est, x_lengths=xlc, y_lengths=ylc)
    prev = pcl.iterative_closest_point(Xc, Yc, init, 0, thr, est, x_lengths=xlc, y_lengths=ylc)
    hist = []
    for k in range(1, len(full.t_history) + 1):
        cur = pcl.iterative_closest_point(Xc, Yc, init, k, thr, est, x_lengths=xlc, y_lengths=ylc)
        idx = pcl.knn_points(prev.Xt, Yc, xlc, ylc, K=1).idx
        ynn = pcl.knn_gather(Yc, idx, ylc)[:, :, 0]
        want = pcl.corresponding_points_alignment(Xc, ynn, weights=mask, estimate_scale=est)
        for a, w_ in zip(cur.RTs, want):
            assert same_bits(npy(a), npy(w_)), f"iteration {k}"
        for a, w_ in zip(full.t_history[k - 1], want):
            assert same_bits(npy(a), npy(w_))
        d = ((cur.Xt.double() - ynn.double()) ** 2).sum(2) * mask.double()
        r64 = (d.sum(1) / mask.double().sum(1).clamp(min=1e-9)).sqrt().cpu().numpy()
        got = npy(cur.rmse).astype(np.float64)
        assert (np.abs(got - r64) <= ulp(r64)).all()
        assert same_bits(npy(cur.rmse), npy(raw["rmse"][k - 1]))
        hist.append(cur.rmse.cpu())
        prev = cur
    stop = None
    for k, r in enumerate(hist):
        rel = torch.ones_like(r) if k == 0 else (hist[k - 1] - r) / hist[k - 1]
        if bool((rel <= thr).all()):
            stop = k + 1
            break
    assert full.converged == (stop is not None)
    assert len(full.t_history) == (stop if stop is not None else K)
    return full


def test_icp_replay_ragged_empty_init_scale():
    X, Y, R, T = pair(4, 500, 51, n2=700)
    xl, yl = torch.tensor([500, 400, 37, 0]), torch.tensor([700, 650, 0, 200])
    init = pcl.SimilarityTransform(torch.eye(3).expand(4, 3, 3).cuda().contiguous(), torch.full((4, 3), 0.01).cuda(),
                                   torch.ones(4).cuda())
    full = replay_check(X, Y, xl, yl, init=init, est=True, K=6)
    assert not full.converged and npy(full.rmse)[3] == 0       # the empty X cloud: rmse 0, 0 / 0, never converges
    full = replay_check(X, Y, xl, yl, K=5)
    assert not full.converged and len(full.t_history) == 5


def test_icp_replay_two_clouds_that_stop_at_different_iterations():
    X, Y, _, _ = pair(2, 600, 52, angle=25)
    g = torch.Generator().manual_seed(53)
    Y[1] = (X[1] + 0.001 + 0.002 * torch.randn(600, 3, generator=g))[torch.randperm(600, generator=g)]
    alone = [len(pcl.iterative_closest_point(X[k:k + 1].cuda(), Y[k:k + 1].cuda(), relative_rmse_thr=1e-4).t_history)
             for k in range(2)]
    assert alone[0] != alone[1]
    full = replay_check(X, Y, None, None, K=60, thr=1e-4)
    assert full.converged and len(full.t_history) == max(alone)


# ---------------------------------------------------------------- ICP against the float64 pytorch3d loop --------------

def test_icp_against_float64_loop():
    thr = 1e-6
    X, Y, Rgt, Tgt = pair(8, 1024, 63)  # a seed whose reference decisions all stay a factor 2 away from the threshold
    ref = icp_ref(X.double(), Y.double(), relative_rmse_thr=thr)
    rel = torch.stack(ref["rel_history"]).abs()
    assert not ((rel > thr / 2) & (rel < 2 * thr)).any()        # no decision of the reference is close to the threshold
    got = pcl.iterative_closest_point(X.cuda(), Y.cuda(), relative_rmse_thr=thr)
    assert got.converged == ref["converged"] and len(got.t_history) == len(ref["t_history"])
    assert np.abs(npy(got.RTs.R) - ref["RTs"][0].numpy()).max() <= 1e-5
    assert np.abs(npy(got.RTs.T) - ref["RTs"][1].numpy()).max() <= 1e-5
    assert np.abs(npy(got.RTs.R) - Rgt.numpy()).max() <= 0.02 and np.abs(npy(got.RTs.T) - Tgt.numpy()).max() <= 0.01
    assert (npy(got.rmse) <= 0.005).all()                      # the noise level: 0.002 per coordinate


# ---------------------------------------------------------------- inputs and runs ---------------------------------------

def test_input_forms_repeat_and_nan():
    X, Y, _, _ = pair(3, 700, 71, n2=900)
    w = torch.rand(3, 700, generator=torch.Generator().manual_seed(72))
    X6 = torch.cat([X, torch.randn(3, 700, 3)], 2).cuda()
    for form in ("fp16", "bf16", "strided"):
        if form == "strided":
            xa, ya, xb, yb = X6[:, :, :3], Y.cuda(), X6[:, :, :3].contiguous(), Y.cuda()
        else:
            dt = torch.float16 if form == "fp16" else torch.bfloat16
            xa, ya = X.cuda().to(dt), Y.cuda().to(dt)
            xb, yb = xa.float(), ya.float()
        a = pcl.corresponding_points_alignment(xa, ya[:, :700], w.cuda(), True)
        bq = pcl.corresponding_points_alignment(xb, yb[:, :700], w.cuda(), True)
        assert all(same_bits(npy(p), npy(q)) for p, q in zip(a, bq))
        ia, ib = pcl.icp_forward_raw(xa, ya, None, 8), pcl.icp_forward_raw(xb, yb, None, 8)
        for k in ("Xt", "R", "T", "s", "rmse", "status"):
            assert np.array_equal(npy(ia[k]), npy(ib[k])), (form, k)
    r1, r2 = pcl.icp_forward_raw(X.cuda(), Y.cuda(), None, 20), pcl.icp_forward_raw(X.cuda(), Y.cuda(), None, 20)
    for k in ("Xt", "R", "T", "s", "rmse", "status"):
        assert np.array_equal(npy(r1[k]), npy(r2[k]))
    Xn = X.clone()
    Xn[1, 5, 0] = float("nan")
    n_it = 12
    bad = pcl.icp_forward_raw(Xn.cuda(), Y.cuda(), None, n_it)
    clean = pcl.icp_forward_raw(X.cuda(), Y.cuda(), None, n_it, relative_rmse_thr=-1.0)  # never stops either
    assert npy(bad["status"]).tolist() == [n_it, 0]
    for k in ("R", "T", "s", "rmse"):
        assert same_bits(npy(bad[k])[:, [0, 2]], npy(clean[k])[:, [0, 2]])
    assert same_bits(npy(bad["Xt"])[[0, 2]], npy(clean["Xt"])[[0, 2]])


def test_zero_iterations_and_empty_batch():
    X, Y, R, T = pair(2, 100, 81)
    r = pcl.iterative_closest_point(X.cuda(), Y.cuda(), max_iterations=0)
    assert r.converged is False and r.rmse is None and r.t_history == [] and torch.equal(r.Xt.cpu(), X)
    init = pcl.SimilarityTransform(R.float().cuda(), T.float().cuda(), torch.full((2,), 1.25).cuda())
    r = pcl.iterative_closest_point(X.cuda(), Y.cuda(), init, max_iterations=0)
    want = apply_ref(X.double(), R.float().double(), T.float().double(), torch.full((2,), 1.25, dtype=torch.float64))
    assert np.abs(npy(r.Xt) - want.numpy()).max() < 1e-5 and all(torch.equal(a, b) for a, b in zip(r.RTs, init))
    e = pcl.iterative_closest_point(torch.zeros(0, 5, 3).cuda(), torch.zeros(0, 6, 3).cuda())
    assert e.converged and len(e.t_history) == 1 and e.Xt.shape == (0, 5, 3)


# ---------------------------------------------------------------- stale state and graphs --------------------------------

def test_stale_outputs_workspace_and_shared_memory():
    st = Stale()
    L = st.L
    X, Y, _, _ = pair(5, 777, 91, n2=1000)
    Xc, Yc = X.cuda(), Y.cuda()
    xl, yl = torch.tensor([777, 500, 33, 0, 700]).cuda(), torch.tensor([1000, 999, 0, 50, 600]).cuda()
    b, p1, p2 = 5, 777, 1000
    A = _lib.pts_args
    # alignment forward and backward
    w = torch.rand(b, p1, generator=torch.Generator().manual_seed(92)).cuda()
    Yp = Yc[:, :p1].contiguous()
    eager = pcl.points_alignment_forward_raw(Xc, Yp, w, True, False, 1e-9, xl)
    R, T, s = torch.empty(b, 3, 3, device="cuda"), torch.empty(b, 3, device="cuda"), torch.empty(b, device="cuda")
    rec = torch.empty(b, 40, device="cuda", dtype=torch.float64)
    nws = int(L.pcl_points_alignment_workspace_bytes(b, p1))
    ws = torch.empty(nws, device="cuda", dtype=torch.uint8)
    st.run(PATTERNS, [R, T, s], [ws, rec], lambda q: L.pcl_points_alignment_fwd(
        *A(Xc), *A(Yp), xl.data_ptr(), w.data_ptr(), b, p1, 1, 0, 1e-9, R.data_ptr(), T.data_ptr(), s.data_ptr(),
        rec.data_ptr(), ws.data_ptr(), nws, q),
        check=lambda o: all(same_bits(o[k], npy(eager[n])) for k, n in enumerate("RTs")))
    gR, gT, gs = torch.randn(b, 3, 3, device="cuda"), torch.randn(b, 3, device="cuda"), torch.randn(b, device="cuda")
    rec = eager["record"]
    gx, gy, gw = torch.empty(b, p1, 3, device="cuda"), torch.empty(b, p1, 3, device="cuda"), torch.empty(b, p1, device="cuda")
    res = st.run(PATTERNS, [gx, gy, gw], [], lambda q: L.pcl_points_alignment_bwd(
        *A(Xc), *A(Yp), xl.data_ptr(), w.data_ptr(), b, p1, 1, 1e-9, rec.data_ptr(), gR.data_ptr(), gT.data_ptr(),
        gs.data_ptr(), gx.data_ptr(), gy.data_ptr(), gw.data_ptr(), q))
    assert not res[0][0][1, 500:].any() and not res[0][2][3].any()
    # ICP (the workspace includes the barrier words)
    it = 9
    eager = pcl.icp_forward_raw(Xc, Yc, None, it, 1e-6, False, False, xl, yl)
    outs = [torch.empty(b, p1, 3, device="cuda"), torch.empty(it, b, 3, 3, device="cuda"), torch.empty(it, b, 3, device="cuda"),
            torch.empty(it, b, device="cuda"), torch.empty(it, b, device="cuda"), torch.empty(2, device="cuda", dtype=torch.int32)]
    nws = int(L.pcl_icp_workspace_bytes(b, p1, p2, it))
    ws = torch.empty(nws, device="cuda", dtype=torch.uint8)
    st.run(PATTERNS, outs, [ws], lambda q: L.pcl_icp(
        *A(Xc), xl.data_ptr(), *A(Yc), yl.data_ptr(), b, p1, p2, None, None, None, it, 1e-6, 0, 0, 0,
        *[o.data_ptr() for o in outs], ws.data_ptr(), nws, q),
        check=lambda o: all(np.array_equal(o[k], npy(eager[n])) for k, n in enumerate(["Xt", "R", "T", "s", "rmse", "status"])))


def test_graph_capture_and_replay_of_icp():
    X, Y, _, _ = pair(3, 500, 95)
    X2, Y2, _, _ = pair(3, 500, 96)
    xs, ys = X.cuda(), Y.cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        pcl.icp_forward_raw(xs, ys, None, 30, 1e-5)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out = pcl.icp_forward_raw(xs, ys, None, 30, 1e-5)
    xs.copy_(X2.cuda())
    ys.copy_(Y2.cuda())
    g.replay()
    torch.cuda.synchronize()
    eager = pcl.icp_forward_raw(X2.cuda(), Y2.cuda(), None, 30, 1e-5)
    for k in ("Xt", "R", "T", "s", "rmse", "status"):
        assert np.array_equal(npy(out[k]), npy(eager[k])), k
    assert not np.array_equal(npy(out["Xt"]), npy(pcl.icp_forward_raw(X.cuda(), Y.cuda(), None, 30, 1e-5)["Xt"]))
    # the C entry point through the shared helper as well
    L = _lib.lib()
    b, p = 3, 500
    o = [torch.empty(b, p, 3, device="cuda"), torch.empty(30, b, 3, 3, device="cuda"), torch.empty(30, b, 3, device="cuda"),
         torch.empty(30, b, device="cuda"), torch.empty(30, b, device="cuda"), torch.empty(2, device="cuda", dtype=torch.int32)]
    nws = int(L.pcl_icp_workspace_bytes(b, p, p, 30))
    ws = torch.empty(nws, device="cuda", dtype=torch.uint8)
    capture_and_replay([xs, ys], [X.cuda(), Y.cuda()], o, lambda q: L.pcl_icp(
        *_lib.pts_args(xs), None, *_lib.pts_args(ys), None, b, p, p, None, None, None, 30, 1e-5, 0, 0, 0,
        *[t.data_ptr() for t in o], ws.data_ptr(), nws, q))


def test_launch_count_does_not_depend_on_max_iterations():
    from torch.profiler import ProfilerActivity, profile
    X, Y, _, _ = pair(4, 1000, 97, angle=1, shift=0.003)  # the float64 loop stops after 7 iterations at 1e-4
    Xc, Yc = X.cuda(), Y.cuda()
    counts, iters = [], []
    for m in (10, 1000):
        r = pcl.iterative_closest_point(Xc, Yc, max_iterations=m, relative_rmse_thr=1e-4)  # warm-up
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            r = pcl.iterative_closest_point(Xc, Yc, max_iterations=m, relative_rmse_thr=1e-4)
            torch.cuda.synchronize()
        dev = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        kernels = [n for n in dev if not n.startswith(("Memset", "Memcpy"))]
        assert len(kernels) == 1 and "icp_kernel" in kernels[0], dev
        counts.append(len(dev))
        iters.append(len(r.t_history))
        assert r.converged and 2 <= len(r.t_history) < 10
    assert counts[0] == counts[1] and iters[0] == iters[1]
