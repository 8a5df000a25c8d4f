"""GPU tests of the auction kernel's fused loss epilogue (pcl_emd_fwd_fused, include/pcl.h) on every path that writes it:
the plain cluster kernel, the team kernel, the ticket path (the cluster kernel's EXPORT instantiation) and the cold state of
clouds above 3584 points -- each with predictions read from the shared-memory cache (flag X1) and from global memory
(strided, fp16, bf16).  Expectations:
  dist / assignment: the CPU oracle, bit for bit;
  gradient: the float32 restatement of tests/emd_epilogue_ref.py, bit for bit (NaN compared as NaN);
  sum sqrt(dist): the exactly rounded sum (math.fsum) to within one float32 ulp -- the kernel's fp64 order depends on
  how the points are split over CTAs, so the sum may differ between paths, but not between two calls.
Then the loss surfaces built on the epilogue (EarthMoverDistance, chamfer_emd_loss, pcl_chamfer_emd_step) at the shapes
where AUTO takes the team, ticket and cold paths, and where B exceeds the SM count."""
import numpy as np
import pytest
import torch

import oracle
import pointcloud_b200 as pcl
from oracle import loss_oracle
from pointcloud_b200 import _lib, synth
from emd_epilogue_ref import epilogue_grad, epilogue_sum, float32_neighbours
from helpers import npy, reference_structure, same_bits

pytestmark = pytest.mark.gpu
EPS = 0.005
F_X1, F_COLD = 2, 4          # launch flags in stats[:, 6] (pcl_emd_core.cuh EMD_F_*)
REL = 1e-5

# (B, N, iterations) -> the paths forced on it ("auto" where only the cluster kernel can run: the cold state above 3584 points)
MATRIX = {
    (4, 2048, 50): ("cluster", "team", "tickets"),
    (8, 3072, 50): ("cluster", "team"),
    (48, 2048, 50): ("cluster", "team", "tickets"),
    (3, 3584, 50): ("cluster", "team", "tickets"),
    (300, 256, 50): ("cluster",),            # B > 256: the per-CTA partials of the sum outgrow their 256-entry minimum
    (1, 1, 50): ("cluster",),
    (2, 37, 1): ("cluster",),
    (2, 37, 0): ("cluster", "team", "tickets"),  # no iteration: every point stays unassigned (assignment -1, gradient 0)
    (64, 2048, 50): ("tickets",),
    (2, 3585, 50): ("auto",),
    (2, 5000, 50): ("auto",),
    (1, 8192, 50): ("auto",),
}
FORMS = ("fp32", "strided", "fp16", "bf16")
_DT = {"fp16": torch.float16, "bf16": torch.bfloat16}


@pytest.fixture
def emd_path():
    """Selects an auction kernel for one test and restores the automatic choice afterwards."""
    yield pcl.set_emd_path
    pcl.set_emd_path("auto")


def make_inputs(b, n, form, seed):
    """(prediction, target) on the GPU in one of the four input forms; the target is fp32 (strided in the strided form)."""
    pred, target = synth.autoencoder_batch(b, n, seed=seed)
    pc, tc = pred.cuda(), target.cuda()
    if form == "strided":                                   # row stride 6 (utils.py:254)
        return pc[:, :, :3], tc[:, :, :3]
    x1 = pc[:, :, :3].contiguous()
    return (x1 if form == "fp32" else x1.to(_DT[form])), tc[:, :, :3].contiguous()


_ORACLE = {}


def oracle_of(x1, x2, iters):
    """oracle.emd_forward on the fp32 values the kernel reads (fp16 / bf16 up-cast like .float()), memoised per input."""
    a, t = x1.float().cpu(), x2.float().cpu()
    key = (a.numpy().tobytes(), t.numpy().tobytes(), iters)
    if key not in _ORACLE:
        _ORACLE.clear()
        _ORACLE[key] = (a.numpy(), t.numpy(), oracle.emd_forward(a, t, EPS, iters, nthreads=16))
    return _ORACLE[key]


def fused_call(x1, x2, iters, grad_scale):
    """pcl_emd_fwd_fused through the C ABI -> (dist, assignment, stats, grad, sums) as numpy arrays.  The outputs start as
    NaN so that an element the kernel does not write cannot pass for one it wrote."""
    L = _lib.lib()
    b, n = x1.shape[0], x1.shape[1]
    dist = torch.empty(b, n, device="cuda")
    asg = torch.empty(b, n, device="cuda", dtype=torch.int32)
    stats = torch.empty(b, 8, device="cuda", dtype=torch.int32)
    grad = torch.full((b, n, 3), float("nan"), device="cuda")
    sums = torch.full((3,), float("nan"), device="cuda")
    wsb = L.pcl_emd_workspace_bytes(b, n)
    ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
    rc = L.pcl_emd_fwd_fused(*_lib.pts_args(x1), *_lib.pts_args(x2), b, n, EPS, iters, dist.data_ptr(), asg.data_ptr(),
                             stats.data_ptr(), float(grad_scale), grad.data_ptr(), sums.data_ptr(), ws.data_ptr(), wsb,
                             torch.cuda.current_stream().cuda_stream)
    assert rc == 0, L.pcl_last_error()
    torch.cuda.synchronize()
    return npy(dist), npy(asg), npy(stats), npy(grad), npy(sums)


def check_sums(sums, dist):
    s, count, _ = epilogue_sum(dist)
    assert sums[1] == np.float32(count)                                          # B*N, exactly
    assert sums[0] in float32_neighbours(s), (sums[0], s)                        # fp64 in a partition-dependent order: <= 1 ulp
    assert sums[2] == np.float32(sums[0]) / np.float32(sums[1])                  # the mean is the float32 ratio of the two


def check_stats(st, path, n):
    st = np.asarray(st)
    assert (st[:, 6] == st[0, 6]).all()                                          # launch flags are uniform over the grid
    if path == "team":
        assert (st[:, 3] == 0).all(), st[:, 3]                                   # stats[3] = 0: the team kernel ran
    else:
        assert (st[:, 3] > 0).all(), st[:, 3]                                    # a cluster kernel ran (plain or ticket path)
    assert (((st[:, 6] & F_COLD) != 0) == (n > 3584)).all(), st[:, 6]           # the cold state exactly above 3584 points


def run_matrix_case(b, n, iters, form):
    x1, x2 = make_inputs(b, n, form, seed=10007 * b + n)
    a1, a2, o = oracle_of(x1, x2, iters)
    scales = (1.0, np.float32(1.0 / (b * n)), 0.37)
    first = None
    for path in MATRIX[(b, n, iters)]:
        pcl.set_emd_path(path)
        outs = []
        for gs in scales:
            d, a, st, g, s = fused_call(x1, x2, iters, gs)
            assert np.array_equal(a, o["assignment"]) and np.array_equal(d, o["dist"]), (path, gs)
            assert same_bits(g, epilogue_grad(a1, a2, o["dist"], o["assignment"], gs)), (path, gs)
            check_sums(s, o["dist"])
            check_stats(st, path, n)
            outs.append((d, a, g, s))
        d, a, st, g, s = fused_call(x1, x2, iters, scales[-1])                   # again: the ticket and partials are reused
        assert np.array_equal(s.view(np.int32), outs[-1][3].view(np.int32)) and same_bits(g, outs[-1][2])
        print(f"[{path} B={b} N={n} {form}] stats[:,3]={sorted(set(st[:, 3].tolist()))} stats[:,6]={sorted(set(st[:, 6].tolist()))}"
              f" X1={'on' if st[0, 6] & F_X1 else 'off'} COLD={'on' if st[0, 6] & F_COLD else 'off'}")
        if first is None:
            first = outs
        for (d0, a0, g0, _), (d1, a1_, g1, _) in zip(first, outs):                # every path: the same dist, assignment, grad
            assert np.array_equal(d0, d1) and np.array_equal(a0, a1_) and same_bits(g0, g1), path
    # the plain entry point right after launches that left their partials in shared memory: the padding targets of the last
    # tile (N not a multiple of 32) must be priced by the kernel, not by what an earlier kernel left there
    d, a, _ = pcl.emd_forward_raw(x1, x2, EPS, iters)
    assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
    if iters == 0:
        assert (o["assignment"] == -1).all()                                     # (the last iteration assigns every bidder)


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("b,n,iters", list(MATRIX))
def test_fused_epilogue_every_path_and_input_form(emd_path, b, n, iters, form):
    run_matrix_case(b, n, iters, form)


@pytest.mark.parametrize("form", ["strided", "fp16"])
def test_matrix_reads_predictions_from_shared_and_global_memory(form):
    """The matrix runs the strided and fp16 forms both with the shared-memory prediction cache (X1: 4 x 2048) and without it
    (global loads with strides / conversion: 8 x 3072, where the cache no longer fits next to the auction state)."""
    for (b, n), x1_on in (((4, 2048), True), ((8, 3072), False)):
        assert (b, n, 50) in MATRIX
        x1, x2 = make_inputs(b, n, form, seed=10007 * b + n)
        _, _, st, _, _ = fused_call(x1, x2, 1, 1.0)
        assert (((st[:, 6] & F_X1) != 0) == x1_on).all(), st[:, 6]


def degenerate_clouds(case, b=3, n=2048):
    g = torch.Generator().manual_seed(7)
    if case == "identical_clouds":
        x2 = torch.rand(b, n, 3, generator=g)
        return x2.clone(), x2
    # grid_ties (test_emd_gpu.py): coordinates on a coarse lattice -- thousands of equal distances, and points that
    # coincide with a target (dist == 0)
    return (torch.randint(0, 6, (b, n, 3), generator=g).float() / 6, torch.randint(0, 6, (b, n, 3), generator=g).float() / 6)


@pytest.mark.parametrize("path", ["cluster", "team", "tickets", "auto"])
@pytest.mark.parametrize("case", ["identical_clouds", "grid_ties"])
def test_fused_epilogue_degenerate_clouds(emd_path, path, case):
    """dist == 0 on an assigned point: the gradient is NaN (inf * 0), like dists.sqrt() in the reference; every other point
    is finite and equals the restatement.  Not every point finds itself after 50 iterations, so neither an all-NaN
    gradient nor a zero sum is asserted."""
    emd_path(path)
    x1, x2 = degenerate_clouds(case)
    o = oracle.emd_forward(x1, x2, EPS, 50, nthreads=3)
    gs = np.float32(1.0 / x1[:, :, 0].numel())
    d, a, st, g, s = fused_call(x1.cuda(), x2.cuda(), 50, gs)
    assert np.array_equal(a, o["assignment"]) and np.array_equal(d, o["dist"])
    ref = epilogue_grad(x1.numpy(), x2.numpy(), o["dist"], o["assignment"], gs)
    assert same_bits(g, ref)
    zero = (o["dist"] == 0) & (o["assignment"] >= 0)
    assert zero.any() and np.isnan(g[zero]).all() and np.isfinite(g[~zero]).all()
    check_sums(s, o["dist"])
    if path == "team":
        assert (st[:, 3] == 0).all()


# ---- the loss surfaces built on the epilogue, at the shapes where AUTO leaves the plain cluster path --------------------
# (8, 3072): team path; (48, 2048): ticket path (clusters of <= 2 CTAs); (2, 5000): cold state; (160, 1024): B above the
# SM count -> clusters of one CTA in more than one wave
SURFACE_SHAPES = [(8, 3072), (48, 2048), (2, 5000), (160, 1024)]


def auto_path_stats(x1, x2):
    _, _, st = pcl.emd_forward_raw(x1, x2, EPS, 50, want_stats=True)
    return npy(st)


@pytest.mark.parametrize("b,n", SURFACE_SHAPES)
def test_earth_mover_distance_fused_at_auto_path_shapes(b, n):
    """pcl.EarthMoverDistance (Autoencoder form: epilogue value and gradient) against the unfused reference structure, the
    float64 mean of sqrt(dist) and, at the team-path shape, the CPU loss oracle."""
    pred, target = synth.autoencoder_batch(b, n, seed=b + n, regime="noisy")
    pc, tc = pred.cuda(), target.cuda()
    st = auto_path_stats(pc[:, :, :3], tc[:, :, :3])
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    expect = {(8, 3072): lambda s: (s[:, 3] == 0).all(), (48, 2048): lambda s: (s[:, 3] <= 2).all() and (s[:, 3] > 0).all(),
              (2, 5000): lambda s: ((s[:, 6] & F_COLD) != 0).all(), (160, 1024): lambda s: b < sm or (s[:, 3] == 1).all()}
    assert expect[(b, n)](st), st[:, [3, 6]]
    out = []
    for fused in (True, False):
        p = pc.clone().requires_grad_()
        fn = pcl.EarthMoverDistance(EPS, 50) if fused else reference_structure(EPS, 50)
        logged = {}
        fn.log = lambda k, v: logged.__setitem__(k, float(v.detach()))
        loss = fn(p, tc)
        loss.backward()
        out.append((float(loss), npy(p.grad), logged["train_loss/EMD"]))
    assert out[0][0] == pytest.approx(out[1][0], rel=REL)
    np.testing.assert_allclose(out[0][1], out[1][1], rtol=REL, atol=1e-10)
    assert np.isfinite(out[0][1]).all()
    d, _, _ = pcl.emd_forward_raw(pc[:, :, :3], tc[:, :, :3], EPS, 50)
    mean64 = epilogue_sum(npy(d))[2]
    assert abs(out[0][2] - mean64) <= 1e-6 * mean64, (out[0][2], mean64)     # the fused point term: float32 of the fp64 mean
    if (b, n) == (8, 3072):
        po = pred.clone().requires_grad_()
        lo = loss_oracle.EarthMoverDistance(EPS, 50)(po, target)
        lo.backward()
        assert out[0][0] == pytest.approx(float(lo), rel=REL)
        np.testing.assert_allclose(out[0][1], po.grad.numpy(), rtol=REL, atol=1e-10)


@pytest.mark.parametrize("chamfer_mode", [0, 1])
@pytest.mark.parametrize("b,n", SURFACE_SHAPES)
def test_chamfer_emd_step_at_auto_path_shapes(b, n, chamfer_mode):
    """pcl.chamfer_emd_loss (autograd, upstream gradients other than 1) and pcl_chamfer_emd_step (C ABI: Chamfer on the side
    stream next to the auction) against chamfer_distance + emdModule().sqrt().mean() in the same Chamfer arithmetic mode."""
    L = _lib.lib()
    pred, target = synth.autoencoder_batch(b, n, seed=3 * b + n, regime="noisy")
    pc, tc = pred.cuda(), target.cuda()
    px, tx = pc[:, :, :3], tc[:, :, :3]
    # the separate calls
    xg = px.detach().clone().requires_grad_()
    cl, _ = pcl.chamfer_distance(xg, tx, mode=chamfer_mode)
    cl.backward()
    xe = px.detach().clone().requires_grad_()
    dist, _ = pcl.emdModule()(xe, tx, EPS, 50)
    el = dist.sqrt().mean()
    el.backward()
    # the composite C call
    losses = torch.zeros(8, device="cuda")
    gch, gem = torch.empty(b, n, 3, device="cuda"), torch.empty(b, n, 3, device="cuda")
    nbytes = L.pcl_chamfer_emd_step_scratch_bytes(b, n)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    rc = L.pcl_chamfer_emd_step(*_lib.pts_args(px), *_lib.pts_args(tx), b, n, EPS, 50, chamfer_mode, losses.data_ptr(), gch.data_ptr(),
                                gem.data_ptr(), scratch.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, L.pcl_last_error()
    torch.cuda.synchronize()
    lz = npy(losses)
    assert float(lz[0] + lz[1]) == pytest.approx(float(cl), rel=1e-6) and float(lz[2] + lz[3]) == pytest.approx(b * float(cl), rel=1e-6)
    assert lz[5] == np.float32(b * n) and lz[4] in float32_neighbours(epilogue_sum(npy(dist))[0])
    assert float(lz[6]) == pytest.approx(float(el), rel=1e-6)
    np.testing.assert_allclose(npy(gch), npy(xg.grad), rtol=REL, atol=1e-9)
    np.testing.assert_allclose(npy(gem), npy(xe.grad), rtol=REL, atol=1e-10)
    # the autograd surface over the same call, 6 channels in, upstream gradients 2 and 0.5
    pa = pc.clone().requires_grad_()
    c, e = pcl.chamfer_emd_loss(pa, tc, EPS, 50, chamfer_mode=chamfer_mode)
    (2.0 * c + 0.5 * e).backward()
    assert abs(float(c) - float(cl)) <= 1e-6 * abs(float(cl)) and abs(float(e) - float(el)) <= 1e-6 * abs(float(el))
    want = 2.0 * npy(xg.grad) + 0.5 * npy(xe.grad)
    np.testing.assert_allclose(npy(pa.grad[:, :, :3]), want, rtol=REL, atol=1e-9)
    assert not pa.grad[:, :, 3:].any()
