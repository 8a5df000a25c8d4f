"""GPU tests of chamfer_distance's normals, weights and batch reductions (pcl_chamfer_cloud_fwd / pcl_chamfer_cloud_bwd) against
the float64 restatement of pytorch3d 0.7.2 (tests/chamfer_surface_ref.py, indices from the CPU oracle).

dist / idx are bit-exact with the oracle; cloud_sums, normal_sums, both return values and the gradients of x, y, both normals and
the weights are within 1e-5 relative of float64, and what float64 makes exactly 0 (pads, empty clouds) is exactly 0.  The
default call is unchanged: its loss equals the call with normals bit for bit, and pcl_chamfer_fwd equals pcl_chamfer_cloud_fwd
with every new pointer NULL.  Gradients are fp32 atomics, so they are compared within tolerance, never bit for bit."""
import numpy as np
import pytest
import torch

import pointcloud_b200 as pcl
import smem_poison
from chamfer_surface_ref import chamfer_reference, cloud_sums_reference, neighbours
from helpers import npy, same_bits
from pointcloud_b200 import _lib

pytestmark = pytest.mark.gpu
REL = 1e-5


@pytest.fixture
def prune_min():
    """Sets the pruned path's switch-over (pcl_chamfer_set_prune_min) for one test and restores the default afterwards."""
    L = _lib.lib()
    yield L.pcl_chamfer_set_prune_min
    L.pcl_chamfer_set_prune_min(-1)


def make(b, p1, p2, d, seed, ragged=True):
    """Points, (B, P, 6) xyz+normal clouds whose [..., 3:6] slices are the normals, lengths with 0, 1 and P on both sides
    (the last of them past the first 32 clouds), random weights."""
    g = torch.Generator().manual_seed(seed)
    x, y = torch.rand(b, p1, d, generator=g), torch.rand(b, p2, d, generator=g)
    cx, cy = torch.randn(b, p1, 6, generator=g), torch.randn(b, p2, 6, generator=g)
    xl = yl = None
    if ragged:
        xl, yl = torch.randint(0, p1 + 1, (b,), generator=g), torch.randint(0, p2 + 1, (b,), generator=g)
        xl[0], xl[1], xl[b - 1] = 0, 1, p1
        yl[2], yl[0], yl[b - 1 if b > 33 else 1] = 0, 1, p2
    w = torch.rand(b, generator=g, dtype=torch.float64) + 0.1
    return x, y, cx, cy, xl, yl, w


def close(got, want, what=""):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = max(float(np.abs(want).max(initial=0.0)), 1e-30)
    np.testing.assert_allclose(got, want, rtol=REL, atol=1e-6 * scale, err_msg=what)
    assert not got[want == 0].any(), f"{what}: exact zeros of the reference are not zero"


def dtype_tol(want, dt):
    """One rounding to fp16 / bf16 (the gradient comes back in the input's dtype), subnormals included."""
    if dt == torch.float32:
        return 0.0
    man, tiny = {torch.float16: (10, 2.0 ** -24), torch.bfloat16: (7, 2.0 ** -133)}[dt]
    return np.maximum(2.0 ** (np.floor(np.log2(np.maximum(np.abs(want), 1e-300))) - man), tiny)


def run_case(x, y, cx, cy, xl, yl, w, batch_reduction, normals, dt=torch.float32, mode=None, weights="random"):
    """chamfer_distance on the GPU and the float64 reference, forward and backward; returns the GPU results."""
    dev = "cuda"
    xg, yg = x.to(dt).to(dev).requires_grad_(), y.to(dt).to(dev).requires_grad_()
    cxg, cyg = cx.to(dt).to(dev).requires_grad_(), cy.to(dt).to(dev).requires_grad_()
    xn, yn = cxg[..., 3:6], cyg[..., 3:6]                       # strided views, read in place
    wt = {"none": None, "random": w, "some_zero": w * (torch.arange(len(w)) % 3 != 0), "all_zero": w * 0}[weights]
    wg = None if wt is None else wt.to(dev).requires_grad_()
    kw = dict(x_lengths=None if xl is None else xl.to(dev), y_lengths=None if yl is None else yl.to(dev), weights=wg,
              batch_reduction=batch_reduction, mode=mode)
    if normals in ("one", "both"):
        kw["x_normals"] = xn
    if normals == "both":
        kw["y_normals"] = yn
    loss, lossn = pcl.chamfer_distance(xg, yg, **kw)
    assert (lossn is None) == (normals != "both") or weights == "all_zero"
    # reference, on the values the kernels read
    X, Y = xg.detach().double().cpu().requires_grad_(), yg.detach().double().cpu().requires_grad_()
    CX, CY = cxg.detach().double().cpu().requires_grad_(), cyg.detach().double().cpu().requires_grad_()
    W = None if wt is None else wt.clone().requires_grad_()
    ix, iy, o = neighbours(X, Y, xl, yl, mode=0 if mode in (None, "unfused") else 1)
    rl, rn = chamfer_reference(X, Y, ix, iy, xl, yl, CX[..., 3:6] if normals != "none" else None,
                               CY[..., 3:6] if normals == "both" else None, W, batch_reduction)
    close(npy(loss), npy(rl), "loss")
    g = torch.Generator().manual_seed(5)
    up = torch.rand(tuple(rl.shape), generator=g, dtype=torch.float64) + 0.5     # upstream gradients other than 1
    tot, rtot = (loss * up.to(dev)).sum(), (rl * up).sum()
    if lossn is not None and rn is not None:
        close(npy(lossn), npy(rn), "loss_normals")
        upn = torch.rand(tuple(rn.shape), generator=g, dtype=torch.float64) + 0.5
        tot, rtot = tot + (lossn * upn.to(dev)).sum(), rtot + (rn * upn).sum()
    rtot.backward()
    tot.backward()
    for name, got, ref in (("grad x", xg.grad, X.grad), ("grad y", yg.grad, Y.grad), ("grad x normals", cxg.grad, CX.grad),
                           ("grad y normals", cyg.grad, CY.grad)):
        if got is None:
            assert ref is None or not ref.any(), name
            continue
        want = np.zeros(tuple(got.shape)) if ref is None else npy(ref)
        assert got.dtype == dt
        gotv = npy(got.float()).astype(np.float64)
        tol = REL * np.abs(want) + 1e-6 * max(float(np.abs(want).max(initial=0.0)), 1e-30) + dtype_tol(want, dt)
        bad = np.abs(gotv - want) > tol
        assert not bad.any(), (name, int(bad.sum()), gotv[bad][:4], want[bad][:4])
        assert not gotv[want == 0].any(), f"{name}: exact zeros of the reference are not zero"
    if wg is not None:
        close(npy(wg.grad), npy(W.grad), "grad weights")
    return o


@pytest.mark.parametrize("normals", ["none", "one", "both"])
@pytest.mark.parametrize("weights", ["none", "random", "some_zero", "all_zero"])
@pytest.mark.parametrize("batch_reduction", [None, "sum", "mean"])
def test_reductions_weights_and_normals(batch_reduction, weights, normals):
    """B = 40 > 32 with ragged lengths 0, 1 and P on both sides."""
    x, y, cx, cy, xl, yl, w = make(40, 300, 257, 3, seed=1)
    run_case(x, y, cx, cy, xl, yl, w, batch_reduction, normals, weights=weights)


@pytest.mark.parametrize("path", ["brute", "pruned"])
@pytest.mark.parametrize("mode", ["unfused", "fma"])
@pytest.mark.parametrize("dt", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("d", [3, 6])
def test_widths_dtypes_modes_and_paths(prune_min, d, dt, mode, path):
    if path == "pruned" and d != 3:
        pytest.skip("the pruned path is D = 3 only")
    prune_min(1 if path == "pruned" else 0)
    x, y, cx, cy, xl, yl, w = make(35, 700, 650, d, seed=d + 2)
    run_case(x, y, cx, cy, xl, yl, w, None, "both", dt=dt, mode=mode)
    run_case(x, y, cx, cy, xl, yl, w, "mean", "both", dt=dt, mode=mode, weights="none")


@pytest.mark.parametrize("path", ["brute", "pruned"])
def test_raw_outputs_against_oracle_and_default_path_unchanged(prune_min, path):
    """dist / idx bit-exact; cloud_sums, normal_sums within 1e-5 of float64; pcl_chamfer_fwd == pcl_chamfer_cloud_fwd with NULL
    pointers == with every output; the Chamfer loss with normals is the loss without them, bit for bit."""
    prune_min(1 if path == "pruned" else 0)
    x, y, cx, cy, xl, yl, w = make(37, 1000, 900, 3, seed=3)
    xc, yc, cxc, cyc = x.cuda(), y.cuda(), cx.cuda(), cy.cuda()
    xlc, ylc = xl.cuda(), yl.cuda()
    ix, iy, o = neighbours(x, y, xl, yl)
    plain = pcl.chamfer_forward_raw(xc, yc, xlc, ylc)
    cloud = pcl.chamfer_forward_raw(xc, yc, xlc, ylc, cloud_sums=True)
    full = pcl.chamfer_forward_raw(xc, yc, xlc, ylc, x_normals=cxc[..., 3:6], y_normals=cyc[..., 3:6])
    for r in (plain, cloud, full):
        for k in ("dist_x", "idx_x", "dist_y", "idx_y"):
            assert np.array_equal(npy(r[k]), o[k]), k
        assert same_bits(npy(r["loss_xy"]), npy(plain["loss_xy"])) and same_bits(npy(r["loss_sums"]), npy(plain["loss_sums"]))
    assert cloud["normal_sums"] is None and full["normal_sums"] is not None
    sums, nsums = cloud_sums_reference(x, y, ix, iy, xl, yl, cx[..., 3:6], cy[..., 3:6])
    close(npy(cloud["cloud_sums"]), sums, "cloud_sums")
    assert same_bits(npy(cloud["cloud_sums"]), npy(full["cloud_sums"]))
    close(npy(full["normal_sums"]), nsums, "normal_sums")
    a, _ = pcl.chamfer_distance(xc, yc, x_lengths=xlc, y_lengths=ylc)
    b, bn = pcl.chamfer_distance(xc, yc, x_lengths=xlc, y_lengths=ylc, x_normals=cxc[..., 3:6], y_normals=cyc[..., 3:6])
    assert bn is not None and same_bits(npy(a), npy(b))


def test_cloud_backward_matches_pcl_chamfer_bwd():
    """grad_cloud = g / B / len (as the Python layer forms it) gives pcl_chamfer_bwd's gradients; with normals the point
    gradients stay the same."""
    L = _lib.lib()
    x, y, cx, cy, xl, yl, w = make(34, 500, 400, 3, seed=4)
    b, p1, p2 = 34, 500, 400
    xc, yc, xlc, ylc = x.cuda(), y.cuda(), xl.cuda(), yl.cuda()
    r = pcl.chamfer_forward_raw(xc, yc, xlc, ylc)
    gout = torch.tensor([1.0, 0.37], device="cuda")
    den = torch.stack([xlc.clamp(min=1).float(), ylc.clamp(min=1).float()])
    gc = (gout[:, None] / torch.full((1, 1), float(b), device="cuda") / den).contiguous()
    A = lambda t: _lib.pts_args(t)
    outs = []
    for variant in ("bwd", "cloud", "cloud+normals"):
        gx, gy = torch.empty(b, p1, 3, device="cuda"), torch.empty(b, p2, 3, device="cuda")
        if variant == "bwd":
            rc = L.pcl_chamfer_bwd(*A(xc), xlc.data_ptr(), *A(yc), ylc.data_ptr(), b, p1, p2, 3, r["idx_x"].data_ptr(), r["idx_y"].data_ptr(),
                                   gout.data_ptr(), gx.data_ptr(), gy.data_ptr(), None)
        else:
            nrm = variant == "cloud+normals"
            cxc, cyc = cx.cuda()[..., 3:6], cy.cuda()[..., 3:6]
            gn = torch.ones(2, b, device="cuda")
            gxn, gyn = torch.empty(b, p1, 3, device="cuda"), torch.empty(b, p2, 3, device="cuda")
            na = A(cxc) + A(cyc) if nrm else [None, 0, 0, 0] * 2
            rc = L.pcl_chamfer_cloud_bwd(*A(xc), xlc.data_ptr(), *A(yc), ylc.data_ptr(), b, p1, p2, 3, r["idx_x"].data_ptr(),
                                         r["idx_y"].data_ptr(), gc.data_ptr(), gx.data_ptr(), gy.data_ptr(), *na,
                                         gn.data_ptr() if nrm else None, gxn.data_ptr() if nrm else None, gyn.data_ptr() if nrm else None, None)
        assert rc == 0, L.pcl_last_error()
        outs.append((npy(gx), npy(gy)))
    for gx, gy in outs[1:]:
        close(gx, outs[0][0].astype(np.float64), "grad x")
        close(gy, outs[0][1].astype(np.float64), "grad y")


def test_empty_batch_and_empty_clouds():
    for b, p1, p2 in ((0, 5, 7), (3, 0, 6), (3, 6, 0), (2, 0, 0)):
        x, y = torch.rand(b, p1, 3, device="cuda", requires_grad=True), torch.rand(b, p2, 3, device="cuda", requires_grad=True)
        xn, yn = torch.randn(b, p1, 3, device="cuda", requires_grad=True), torch.randn(b, p2, 3, device="cuda", requires_grad=True)
        for br in (None, "sum", "mean"):
            loss, lossn = pcl.chamfer_distance(x, y, x_normals=xn, y_normals=yn, batch_reduction=br,
                                               weights=torch.ones(b, device="cuda") if b else None)
            assert loss.shape == ((b,) if br is None else ())
            assert not loss.any()
            # a query against an empty cloud adds 1: the normal term is 1 per direction with queries
            per = float(p1 > 0 and p2 == 0) + float(p2 > 0 and p1 == 0)
            want = np.full(b, per) if br is None else (per * b if br == "sum" else (per if b else 0.0))
            close(npy(lossn), want, "loss_normals")
            (loss.sum() + lossn.sum()).backward()
            for t in (x, y, xn, yn):
                assert t.grad is None or not t.grad.any()


PATTERNS = (0x00000000, 0xFFFFFFFF, 0x7F7FFFFF, 0xFF7FFFFF, 0x3F000000, 0xBF000000)


def _i32(p):
    return p - (1 << 32) if p >= 1 << 31 else p


@pytest.mark.parametrize("path", ["brute", "pruned"])
def test_stale_outputs_workspace_and_shared_memory(prune_min, path):
    """Outputs and workspace filled with each pattern and every SM's shared memory poisoned before the call: the forward is
    bit-identical across patterns and equals the oracle and float64, the backward gradients agree within tolerance (their
    float64 check is test_reductions_weights_and_normals) and rows that get nothing are exactly 0 under every pattern."""
    prune_min(1 if path == "pruned" else 0)
    L = _lib.lib()
    x, y, cx, cy, xl, yl, w = make(36, 600, 640, 3, seed=6)
    b, p1, p2 = 36, 600, 640
    xc, yc, xlc, ylc = x.cuda(), y.cuda(), xl.cuda(), yl.cuda()
    cxc, cyc = cx.cuda(), cy.cuda()
    xn, yn = cxc[..., 3:6], cyc[..., 3:6]
    ix, iy, o = neighbours(x, y, xl, yl)
    sums_ref, nsums_ref = cloud_sums_reference(x, y, ix, iy, xl, yl, cx[..., 3:6], cy[..., 3:6])
    A = lambda t: _lib.pts_args(t)
    dx, idx_x = torch.empty(b, p1, device="cuda"), torch.empty(b, p1, device="cuda", dtype=torch.int32)
    dy, idx_y = torch.empty(b, p2, device="cuda"), torch.empty(b, p2, device="cuda", dtype=torch.int32)
    loss, sums, nsums = torch.empty(4, device="cuda"), torch.empty(2, b, device="cuda"), torch.empty(2, b, device="cuda")
    gx, gy = torch.empty(b, p1, 3, device="cuda"), torch.empty(b, p2, 3, device="cuda")
    gxn, gyn = torch.empty(b, p1, 3, device="cuda"), torch.empty(b, p2, 3, device="cuda")
    gc, gn = torch.rand(2, b, device="cuda") + 0.5, torch.rand(2, b, device="cuda") + 0.5
    ws = torch.empty(L.pcl_chamfer_workspace_bytes(b, p1, p2), device="cuda", dtype=torch.uint8)
    fwd_outs = [dx, idx_x, dy, idx_y, loss, sums, nsums]
    s = torch.cuda.Stream()
    hits = torch.zeros(smem_poison.MAX_SMID, dtype=torch.int32, device="cuda")
    s.wait_stream(torch.cuda.current_stream())
    res = []
    for k, pat in enumerate(PATTERNS):
        with torch.cuda.stream(s):
            hits.zero_()
            for t in fwd_outs + [gx, gy, gxn, gyn]:
                if t.dtype == torch.float32:
                    t.view(torch.int32).fill_(_i32(pat))
                else:
                    t.fill_(0x7FFFFFFF if k % 2 == 0 else -2)
            ws.view(torch.int32).fill_(_i32(pat))
            smem_poison.poison(pat, s, hits)
            rc = L.pcl_chamfer_cloud_fwd(*A(xc), xlc.data_ptr(), *A(yc), ylc.data_ptr(), b, p1, p2, 3, 0, dx.data_ptr(), idx_x.data_ptr(),
                                         dy.data_ptr(), idx_y.data_ptr(), loss.data_ptr(), sums.data_ptr(), *A(xn), *A(yn), nsums.data_ptr(),
                                         ws.data_ptr(), ws.numel(), s.cuda_stream)
            assert rc == 0, L.pcl_last_error()
            smem_poison.poison(pat, s, hits)
            rc = L.pcl_chamfer_cloud_bwd(*A(xc), xlc.data_ptr(), *A(yc), ylc.data_ptr(), b, p1, p2, 3, idx_x.data_ptr(), idx_y.data_ptr(),
                                         gc.data_ptr(), gx.data_ptr(), gy.data_ptr(), *A(xn), *A(yn), gn.data_ptr(), gxn.data_ptr(),
                                         gyn.data_ptr(), s.cuda_stream)
            assert rc == 0, L.pcl_last_error()
        s.synchronize()
        res.append([npy(t).copy() for t in fwd_outs + [gx, gy, gxn, gyn]])
    for r in res:
        for got, want in zip(r[:4], (o["dist_x"], o["idx_x"], o["dist_y"], o["idx_y"])):
            assert np.array_equal(got, want)
        for i in range(4, 7):
            assert same_bits(r[i], res[0][i])
        close(r[5], sums_ref, "cloud_sums")
        close(r[6], nsums_ref, "normal_sums")
        for i in range(7, 11):
            close(r[i], res[0][i].astype(np.float64), f"gradient {i - 7}")   # fp32 atomics: not bit-reproducible


def test_graph_capture_and_replay():
    """pcl_chamfer_cloud_fwd with normals and pcl_chamfer_cloud_bwd captured on a side stream, replayed on new inputs: the
    replay equals a direct call (forward bit for bit, gradients within tolerance)."""
    L = _lib.lib()
    b, p1, p2 = 33, 513, 470
    x, y, cx, cy, xl, yl, w = make(b, p1, p2, 3, seed=8)
    x2, y2, cx2, cy2, _, _, _ = make(b, p1, p2, 3, seed=9)
    xc, yc, cxc, cyc, xlc, ylc = x.cuda(), y.cuda(), cx.cuda(), cy.cuda(), xl.cuda(), yl.cuda()
    A = lambda t: _lib.pts_args(t)
    dx, idx_x = torch.empty(b, p1, device="cuda"), torch.empty(b, p1, device="cuda", dtype=torch.int32)
    dy, idx_y = torch.empty(b, p2, device="cuda"), torch.empty(b, p2, device="cuda", dtype=torch.int32)
    loss, sums, nsums = torch.empty(4, device="cuda"), torch.empty(2, b, device="cuda"), torch.empty(2, b, device="cuda")
    gx, gy, gxn, gyn = (torch.empty(b, p, 3, device="cuda") for p in (p1, p2, p1, p2))
    gc, gn = torch.rand(2, b, device="cuda") + 0.5, torch.rand(2, b, device="cuda") + 0.5
    ws = torch.empty(L.pcl_chamfer_workspace_bytes(b, p1, p2), device="cuda", dtype=torch.uint8)
    outs = [dx, idx_x, dy, idx_y, loss, sums, nsums, gx, gy, gxn, gyn]

    def call(st):
        rc = L.pcl_chamfer_cloud_fwd(*A(xc), xlc.data_ptr(), *A(yc), ylc.data_ptr(), b, p1, p2, 3, 0, dx.data_ptr(), idx_x.data_ptr(),
                                     dy.data_ptr(), idx_y.data_ptr(), loss.data_ptr(), sums.data_ptr(), *A(cxc[..., 3:6]), *A(cyc[..., 3:6]),
                                     nsums.data_ptr(), ws.data_ptr(), ws.numel(), st)
        return rc or L.pcl_chamfer_cloud_bwd(*A(xc), xlc.data_ptr(), *A(yc), ylc.data_ptr(), b, p1, p2, 3, idx_x.data_ptr(), idx_y.data_ptr(),
                                             gc.data_ptr(), gx.data_ptr(), gy.data_ptr(), *A(cxc[..., 3:6]), *A(cyc[..., 3:6]), gn.data_ptr(),
                                             gxn.data_ptr(), gyn.data_ptr(), st)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        assert call(s.cuda_stream) == 0, L.pcl_last_error()
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    rc = []
    with torch.cuda.graph(g, stream=s):
        rc.append(call(torch.cuda.current_stream().cuda_stream))
    assert rc == [0], L.pcl_last_error()
    before = [npy(t).copy() for t in outs]
    for t, v in ((xc, x2), (yc, y2), (cxc, cx2), (cyc, cy2)):
        t.copy_(v)
    g.replay()
    torch.cuda.synchronize()
    replay = [npy(t).copy() for t in outs]
    with torch.cuda.stream(s):
        assert call(s.cuda_stream) == 0
    s.synchronize()
    direct = [npy(t) for t in outs]
    for i, (a, d) in enumerate(zip(replay, direct)):
        if i < 7:
            assert same_bits(a, d) if a.dtype == np.float32 else np.array_equal(a, d), i
        else:
            close(a, d.astype(np.float64), f"gradient {i}")
    assert any(not np.array_equal(a, c) for a, c in zip(replay, before))      # the replay computed on the new inputs
