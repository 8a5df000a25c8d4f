"""chamfer_distance's normals, weights and batch reductions without a GPU: the float64 restatement (tests/chamfer_surface_ref.py)
against an independent numpy one and hand cases, the cosine-gradient formula against torch autograd, and the argument checks of
pcl_chamfer_cloud_fwd / pcl_chamfer_cloud_bwd and of pointcloud_b200.chamfer_distance."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from chamfer_surface_ref import chamfer_reference, cloud_sums_reference, cosine_term_grad, neighbours
from pointcloud_b200 import _lib

_PCL_E_ARG, _PCL_E_UNSUPPORTED = -2, -5


def make(n, p1, p2, d, seed, lengths=True):
    g = torch.Generator().manual_seed(seed)
    x, y = torch.rand(n, p1, d, generator=g), torch.rand(n, p2, d, generator=g)
    xn, yn = torch.randn(n, p1, 3, generator=g), torch.randn(n, p2, 3, generator=g)
    xl = yl = None
    if lengths:
        xl, yl = torch.randint(0, p1 + 1, (n,), generator=g), torch.randint(0, p2 + 1, (n,), generator=g)
        xl[0], xl[1], xl[-1] = 0, 1, p1       # 0, 1 and P on both sides, an empty cloud against a full one
        yl[0], yl[1], yl[2] = p2, 0, 1
    w = torch.rand(n, generator=g, dtype=torch.float64)
    return x, y, xn, yn, xl, yl, w


def numpy_chamfer(x, y, xn, yn, xl, yl, w, batch_reduction):
    """Dense float32 distance matrices (the oracle's unfused arithmetic), lowest-index argmin and per-point loops in float64."""
    x, y, xn, yn = (np.asarray(t, np.float64 if k >= 2 else np.float32) for k, t in enumerate((x, y, xn, yn)))
    n, p1, d = x.shape
    p2 = y.shape[1]
    xl = np.full(n, p1) if xl is None else np.asarray(xl)
    yl = np.full(n, p2) if yl is None else np.asarray(yl)
    per, per_n, idx = np.zeros(n), np.zeros(n), []
    for m in range(n):
        for q, t, nq, nt, lq, lt in ((x, y, xn, yn, xl, yl), (y, x, yn, xn, yl, xl)):
            k, kt = int(lq[m]), int(lt[m])
            dm = np.zeros((k, kt), np.float32)
            for c in range(d):
                df = q[m, :k, c][:, None] - t[m, :kt, c][None, :]
                dm = dm + df * df
            j = dm.argmin(1) if kt > 0 else np.zeros(k, np.int64)
            idx.append(j)
            s = sn = 0.0
            for i in range(k):
                if kt > 0:
                    s += float(((q[m, i].astype(np.float64) - t[m, j[i]]) ** 2).sum())
                    a, b = nq[m, i], nt[m, j[i]]
                    c = np.dot(a / max(np.linalg.norm(a), 1e-6), b / max(np.linalg.norm(b), 1e-6))
                    sn += 1.0 - abs(c)
                else:
                    sn += 1.0                   # the neighbour's normal is the zero vector: cos = 0
            wm = 1.0 if w is None else float(w[m])
            per[m] += wm * s / max(k, 1)
            per_n[m] += wm * sn / max(k, 1)
    if batch_reduction is None:
        return per, per_n, idx
    div = 1.0 if batch_reduction == "sum" else (float(w.sum()) if w is not None else max(n, 1))
    return per.sum() / div, per_n.sum() / div, idx


@pytest.mark.parametrize("d", [3, 6])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("batch_reduction", [None, "sum", "mean"])
def test_reference_matches_numpy(d, weighted, batch_reduction):
    x, y, xn, yn, xl, yl, w = make(5, 23, 31, d, seed=d + 10 * weighted)
    w = w if weighted else None
    ix, iy, _ = neighbours(x, y, xl, yl)
    loss, lossn = chamfer_reference(x.double(), y.double(), ix, iy, xl, yl, xn.double(), yn.double(), w, batch_reduction)
    want, wantn, idx = numpy_chamfer(x, y, xn, yn, xl, yl, w, batch_reduction)
    np.testing.assert_allclose(loss.numpy(), want, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(lossn.numpy(), wantn, rtol=1e-12, atol=1e-15)
    for m in range(5):                                           # the oracle's indices are numpy's lowest-index argmin
        assert np.array_equal(ix[m, :int(xl[m])].numpy(), idx[2 * m]) and np.array_equal(iy[m, :int(yl[m])].numpy(), idx[2 * m + 1])
    sums, nsums = cloud_sums_reference(x, y, ix, iy, xl, yl, xn, yn)
    if batch_reduction == "sum" and not weighted:
        den = np.stack([xl.clamp(min=1).numpy(), yl.clamp(min=1).numpy()])
        np.testing.assert_allclose((sums / den).sum(), float(loss), rtol=1e-12)
        np.testing.assert_allclose((nsums / den).sum(), float(lossn), rtol=1e-12)


def test_empty_target_cloud_adds_one_per_query_to_the_normal_term():
    x, y, xn, yn, _, _, _ = make(3, 7, 9, 3, seed=1, lengths=False)
    xl, yl = torch.tensor([7, 5, 0]), torch.tensor([0, 9, 0])    # cloud 0: x against nothing; cloud 2: both empty
    ix, iy, _ = neighbours(x, y, xl, yl)
    sums, nsums = cloud_sums_reference(x, y, ix, iy, xl, yl, xn, yn)
    assert sums[0, 0] == 0 and nsums[0, 0] == 7 and nsums[1, 0] == 0
    assert (sums[:, 2] == 0).all() and (nsums[:, 2] == 0).all()
    xg, xng = x.double().requires_grad_(), xn.double().requires_grad_()
    yng = yn.double().requires_grad_()
    loss, lossn = chamfer_reference(xg, y.double(), ix, iy, xl, yl, xng, yng, batch_reduction=None)
    assert float(lossn[0].detach()) == 1.0 and float(loss[0].detach()) == 0.0   # point mean: 7 / 7
    lossn[0].backward(retain_graph=True)
    assert not xng.grad.any() and not yng.grad.any()            # c = 0 and the target term is masked: no gradient
    loss[0].backward()
    assert not xg.grad.any()


def test_one_normal_only_gives_none_and_weights_of_ones_equal_no_weights():
    x, y, xn, yn, xl, yl, _ = make(4, 12, 10, 3, seed=2)
    ix, iy, _ = neighbours(x, y, xl, yl)
    X, Y = x.double(), y.double()
    assert chamfer_reference(X, Y, ix, iy, xl, yl, xn.double(), None)[1] is None
    assert chamfer_reference(X, Y, ix, iy, xl, yl, None, yn.double())[1] is None
    for br in (None, "sum", "mean"):
        a = chamfer_reference(X, Y, ix, iy, xl, yl, xn.double(), yn.double(), torch.ones(4, dtype=torch.float64), br)
        b = chamfer_reference(X, Y, ix, iy, xl, yl, xn.double(), yn.double(), None, br)
        torch.testing.assert_close(a[0], b[0], rtol=1e-14, atol=0)
        torch.testing.assert_close(a[1], b[1], rtol=1e-14, atol=0)
    s = chamfer_reference(X, Y, ix, iy, xl, yl, xn.double(), yn.double(), None, "sum")
    m = chamfer_reference(X, Y, ix, iy, xl, yl, xn.double(), yn.double(), None, "mean")
    torch.testing.assert_close(s[0], 4 * m[0], rtol=1e-14, atol=0)
    torch.testing.assert_close(s[1], 4 * m[1], rtol=1e-14, atol=0)


def test_all_zero_weights_return_zeros_attached_to_the_graph():
    x, y, xn, yn, xl, yl, _ = make(3, 8, 8, 3, seed=3)
    ix, iy, _ = neighbours(x, y, xl, yl)
    w = torch.zeros(3, dtype=torch.float64, requires_grad=True)
    for br, shape in ((None, (3,)), ("sum", ()), ("mean", ())):
        xg = x.double().requires_grad_()
        a, b = chamfer_reference(xg, y.double(), ix, iy, xl, yl, None, None, w, br)
        assert a.shape == shape and b.shape == shape and not a.any() and not b.any()
        a.sum().backward()
        assert xg.grad is not None and not xg.grad.any()


def test_cosine_gradient_formula_matches_autograd():
    """d(1 - |cos|)/da of F.cosine_similarity(eps=1e-6) = -sign(c) (b^ - c u_a) / max(|a|, eps), u_a = a/|a| (0 at a = 0),
    including a normal shorter than eps, a zero normal and both signs of c."""
    g = torch.Generator().manual_seed(4)
    a = torch.randn(64, 3, generator=g, dtype=torch.float64)
    b = torch.randn(64, 3, generator=g, dtype=torch.float64)
    a[0] *= 1e-7 / a[0].norm()                               # shorter than eps
    b[1] *= 3e-7 / b[1].norm()
    a[2] = 0.0                                               # zero normal: c = 0, no gradient
    b[3] = 0.0
    a[4] = -b[4] * 2.5                                       # anti-parallel
    a.requires_grad_(), b.requires_grad_()
    (1 - torch.abs(F.cosine_similarity(a[None], b[None], dim=2, eps=1e-6))).sum().backward()
    np.testing.assert_allclose(cosine_term_grad(a.detach(), b.detach()), a.grad.numpy(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(cosine_term_grad(b.detach(), a.detach()), b.grad.numpy(), rtol=1e-9, atol=1e-12)
    assert not a.grad[2].any() and not b.grad[2].any() and not a.grad[3].any()
    assert a.grad[0].abs().max() > 1e5                        # the clamped norm: 1 / eps scale


def _pts():
    buf = (ctypes.c_float * 64)()
    return [ctypes.addressof(buf), 0, 3 * 4, 3], buf


def test_abi_refuses_bad_arguments_without_a_device():
    L = _lib.lib()
    pts, keep = _pts()
    out = (ctypes.c_float * 64)(); oi = (ctypes.c_int * 64)()
    o, i = ctypes.addressof(out), ctypes.addressof(oi)
    none = [None, 0, 0, 0]
    ws = (ctypes.c_ubyte * 4096)()

    def fwd(D=3, xn=pts, yn=pts, nsums=o, xdt=0):
        return L.pcl_chamfer_cloud_fwd(*pts, None, *pts, None, 1, 4, 4, D, 0, o, i, o, i, o, o, xn[0], xdt, xn[2], xn[3], *yn, nsums,
                                       ctypes.addressof(ws), 4096, None)
    for kw, code in [(dict(D=9), _PCL_E_UNSUPPORTED), (dict(xn=none), _PCL_E_ARG), (dict(yn=none), _PCL_E_ARG), (dict(xdt=7), _PCL_E_ARG)]:
        assert fwd(**kw) == code and L.pcl_last_error()
    assert b"normal" in L.pcl_last_error()

    def bwd(gc=o, gn=o, xn=pts, gxn=o, D=3):
        return L.pcl_chamfer_cloud_bwd(*pts, None, *pts, None, 1, 4, 4, D, i, i, gc, o, o, *xn, *pts, gn, gxn, o, None)
    for kw, code in [(dict(gc=None), _PCL_E_ARG), (dict(xn=none), _PCL_E_ARG), (dict(gxn=None), _PCL_E_ARG), (dict(D=0), _PCL_E_UNSUPPORTED)]:
        assert bwd(**kw) == code and L.pcl_last_error()
    assert L.pcl_chamfer_workspace_bytes(33, 100, 200) == L.pcl_chamfer_workspace_bytes(33, 100, 200)  # unchanged sizing call


def test_python_argument_checks():
    import pointcloud_b200 as pcl
    x = torch.rand(2, 8, 3)
    n8 = torch.rand(2, 8, 3)
    with pytest.raises(ValueError, match="weights must be of shape"):
        pcl.chamfer_distance(x, x, weights=torch.ones(3))
    with pytest.raises(ValueError, match="weights must be of shape"):
        pcl.chamfer_distance(x, x, weights=torch.ones(2, 1))
    with pytest.raises(ValueError, match="weights cannot be negative"):
        pcl.chamfer_distance(x, x, weights=torch.tensor([1.0, -0.5]))
    with pytest.raises(ValueError, match="batch_reduction"):
        pcl.chamfer_distance(x, x, batch_reduction="max")
    with pytest.raises(ValueError, match="normals"):
        pcl.chamfer_distance(x, x, x_normals=torch.rand(2, 7, 3), y_normals=n8)
    with pytest.raises(ValueError, match="normals"):
        pcl.chamfer_distance(x, x, x_normals=n8, y_normals=torch.rand(2, 8, 2))
    with pytest.raises(NotImplementedError):
        pcl.chamfer_distance(x, x, weights=torch.ones(2), point_reduction="sum")
    # all-zero weights return before any kernel runs (as in pytorch3d): zeros of the reduced shape, attached to the graph
    xg = x.clone().requires_grad_()
    for br, shape in ((None, (2,)), ("sum", ()), ("mean", ())):
        a, b = pcl.chamfer_distance(xg, x, weights=torch.zeros(2), batch_reduction=br)
        assert a.shape == shape and b.shape == shape and not a.any() and not b.any() and a.requires_grad


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback_with_normals_or_weights():
    import pointcloud_b200 as pcl
    from pointcloud_b200._lib import PclError
    x, n = torch.rand(2, 16, 3), torch.rand(2, 16, 3)
    for kw in (dict(x_normals=n, y_normals=n), dict(weights=torch.ones(2)), dict(batch_reduction=None), dict(batch_reduction="sum")):
        with pytest.raises(PclError):
            pcl.chamfer_distance(x, x, **kw)
