"""GPU tests of the loss callables (the drop-in surface of pointcloud_vision/utils.py:207-309): fused path
vs the reference-structure path vs the golden vectors of the real reference Python, the `.log` protocol,
mixed precision, SegmentingChamferDistance, the host-buffer C entry point and the sharded wrapper on one rank."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import pointcloud_b200 as pcl
from oracle import loss_oracle
from pointcloud_b200 import synth
from helpers import npy, reference_structure

pytestmark = pytest.mark.gpu
REL = 1e-5


def _t(a):
    return torch.from_numpy(np.asarray(a))


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("tag,C", [("ae", None), ("seg", 5)])
def test_earth_mover_distance_matches_reference_python_golden(golden, tag, C, fused):
    pred = _t(golden[f"{tag}_pred"]).cuda().requires_grad_()
    fn = pcl.EarthMoverDistance(eps=0.005, its=50, num_classes=C) if fused else reference_structure(0.005, 50, C)
    logged = {}
    fn.log = lambda k, v: logged.__setitem__(k, float(v.detach()))     # train.py:161
    loss = fn(pred, _t(golden[f"{tag}_target"]).cuda())
    assert loss.dim() == 0 and loss.device.type == "cuda"
    loss.backward()
    assert float(loss) == pytest.approx(float(golden[f"{tag}_loss"]), rel=REL)
    keys = ["EMD", "feature"] + (["cross_entropy", "kl_divergence"] if C else [])
    assert set(logged) == {f"train_loss/{k}" for k in keys}
    for k in keys:
        assert logged[f"train_loss/{k}"] == pytest.approx(float(golden[f"{tag}_log_{k}"]), rel=REL)
    np.testing.assert_allclose(npy(pred.grad), golden[f"{tag}_grad"], rtol=REL, atol=1e-10)


@pytest.mark.parametrize("C", [None, 5])
def test_fused_and_reference_structure_agree_at_full_size(C):
    """BASELINE configs 2/3: B=32, N=2048, train settings."""
    pred, target = (synth.segmenter_batch if C else synth.autoencoder_batch)(32, 2048, seed=4, regime="noisy")
    out = []
    for fused in (True, False):
        p = pred.cuda().requires_grad_()
        fn = pcl.EarthMoverDistance(0.005, 50, num_classes=C) if fused else reference_structure(0.005, 50, C)
        loss = fn(p, target.cuda())
        loss.backward()
        out.append((float(loss), npy(p.grad)))
    assert out[0][0] == pytest.approx(out[1][0], rel=REL)
    np.testing.assert_allclose(out[0][1], out[1][1], rtol=REL, atol=1e-10)
    assert np.isfinite(out[0][1]).all()


def test_earth_mover_distance_vs_loss_oracle_small_segmenter():
    pred, target = synth.segmenter_batch(3, 1024, seed=8)
    po = pred.clone().requires_grad_()
    lo = loss_oracle.EarthMoverDistance(0.005, 50, num_classes=5)(po, target)
    lo.backward()
    pg = pred.cuda().requires_grad_()
    lg = pcl.EarthMoverDistance(0.005, 50, num_classes=5)(pg, target.cuda())
    lg.backward()
    assert float(lg) == pytest.approx(float(lo), rel=REL)
    np.testing.assert_allclose(npy(pg.grad), po.grad.numpy(), rtol=REL, atol=1e-10)


def test_mixed_precision_prediction():
    """cfg.precision = '16-mixed': the model output may arrive as fp16/bf16; the kernels up-cast like .float()."""
    pred, target = synth.autoencoder_batch(2, 1024, seed=9)
    for dt in (torch.float16, torch.bfloat16):
        ph = pred.cuda().to(dt).requires_grad_()
        loss = pcl.EarthMoverDistance(0.005, 50)(ph, target.cuda())
        loss.backward()
        pf = ph.detach().float().requires_grad_()
        lf = pcl.EarthMoverDistance(0.005, 50)(pf, target.cuda())
        lf.backward()
        assert ph.grad.dtype == dt
        assert float(loss) == pytest.approx(float(lf), rel=2e-3)
        np.testing.assert_allclose(npy(ph.grad.float()[:, :, :3]), npy(pf.grad[:, :, :3]), rtol=2e-2, atol=1e-6)


def test_segmenting_chamfer_distance_golden_and_oracle(golden):
    labels = {nm: i for i, nm in enumerate(["env", "cube", "arm", "base", "gripper"])}
    pred = {k: _t(golden[f"mseg_pred_{k}"]).cuda().requires_grad_() for k in labels}
    loss = pcl.SegmentingChamferDistance(labels)(pred, _t(golden["mseg_target"]).cuda())
    loss.backward()
    assert float(loss) == pytest.approx(float(golden["mseg_loss"]), rel=REL)
    for k in labels:
        np.testing.assert_allclose(npy(pred[k].grad), golden[f"mseg_grad_{k}"], rtol=REL, atol=1e-9)
    # full-size MultiSegmenter batch (P_c = 21/820/103... of 2048, variable-length targets) vs the oracle
    pd, target, labels = synth.multisegmenter_batch(8, 2048, seed=6)
    po = {k: v.clone().requires_grad_() for k, v in pd.items()}
    lo = loss_oracle.SegmentingChamferDistance(labels)(po, target)
    lo.backward()
    pg = {k: v.cuda().requires_grad_() for k, v in pd.items()}
    lg = pcl.SegmentingChamferDistance(labels)(pg, target.cuda())
    lg.backward()
    assert float(lg) == pytest.approx(float(lo), rel=REL)
    for k in labels:
        np.testing.assert_allclose(npy(pg[k].grad), po[k].grad.numpy(), rtol=REL, atol=1e-9)
    # a custom (non-FilterClasses) filter takes the reference's per-cloud loop and must agree with the batched one
    f = pcl.FilterClasses([2], label_dim=3)
    a = pcl.FilteringChamferDistance(f)(pg["arm"].detach(), target.cuda())
    b = pcl.FilteringChamferDistance(lambda p: f(p))(pg["arm"].detach(), target.cuda())
    assert float(a) == pytest.approx(float(b), rel=1e-6)


def test_sqrt_at_zero_distance_behaves_like_the_reference():
    """utils.py:304: dists.sqrt() has an infinite derivative at 0 -- the reference yields non-finite grads when a
    prediction coincides with its match; the fused path must not silently hide that."""
    _, target = synth.autoencoder_batch(1, 1024, seed=3)
    for fused in (True, False):
        p = target.clone().cuda().requires_grad_()
        loss = (pcl.EarthMoverDistance(0.005, 50) if fused else reference_structure(0.005, 50))(p, target.cuda())
        loss.backward()
        assert float(loss) == pytest.approx(0.0, abs=1e-6)
        assert not torch.isfinite(p.grad[:, :, :3]).all()


def test_host_buffer_step_entry_point_matches_device_path():
    """pcl_chamfer_emd_step_host: pinned host buffers in, losses + gradients out (what a non-torch caller binds)."""
    from pointcloud_b200 import _lib
    L = _lib.lib()
    b, n = 4, 1024
    x1, x2 = synth.uniform_clouds(b, n, seed=12)
    ph, th = x1.pin_memory(), x2.pin_memory()
    loss_h = torch.zeros(8).pin_memory()      # {chamfer x, y means; chamfer x, y batch sums; sum sqrt(dist), B*N, EMD mean, -}
    gch, geh = torch.zeros(b, n, 3).pin_memory(), torch.zeros(b, n, 3).pin_memory()
    nbytes = L.pcl_loss_host_scratch_bytes(b, n)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    rc = L.pcl_chamfer_emd_step_host(ph.data_ptr(), th.data_ptr(), b, n, 0.005, 50, 0, loss_h.data_ptr(), gch.data_ptr(),
                                     geh.data_ptr(), scratch.data_ptr(), nbytes, st)
    assert rc == 0, L.pcl_last_error()
    torch.cuda.synchronize()
    xg = x1.cuda().requires_grad_()
    cl, _ = pcl.chamfer_distance(xg, x2.cuda())
    cl.backward()
    assert float(loss_h[0] + loss_h[1]) == pytest.approx(float(cl), rel=1e-6)
    np.testing.assert_allclose(gch.numpy(), npy(xg.grad), rtol=REL, atol=1e-9)
    xe = x1.cuda().requires_grad_()
    dist, _ = pcl.emdModule()(xe, x2.cuda(), 0.005, 50)
    el = dist.sqrt().mean()
    el.backward()
    assert float(loss_h[6]) == pytest.approx(float(el), rel=1e-6) and float(loss_h[5]) == b * n
    assert float(loss_h[4]) == pytest.approx(float(dist.detach().sqrt().sum()), rel=1e-6)
    assert float(loss_h[2] + loss_h[3]) == pytest.approx(b * float(cl), rel=1e-6)
    np.testing.assert_allclose(geh.numpy(), npy(xe.grad), rtol=REL, atol=1e-10)
    rc = L.pcl_chamfer_emd_step_host(ph.data_ptr(), th.data_ptr(), b, n, 0.005, 50, 0, loss_h.data_ptr(), None, None,
                                     scratch.data_ptr(), 16, st)
    assert rc == -4 and b"scratch" in L.pcl_last_error()


def test_composite_device_step_matches_separate_calls():
    """pcl_chamfer_emd_step (Chamfer forked onto the library's side stream) == the separate entry points."""
    from pointcloud_b200 import _lib
    L = _lib.lib()
    b, n = 6, 2048
    pred, target = synth.autoencoder_batch(b, n, seed=21)
    pc, tc = pred.cuda(), target.cuda()
    px, tx = pc[:, :, :3], tc[:, :, :3]                         # strided views straight into the composite call
    losses = torch.zeros(8, device="cuda")
    gch, gem = torch.empty(b, n, 3, device="cuda"), torch.empty(b, n, 3, device="cuda")
    nbytes = L.pcl_chamfer_emd_step_scratch_bytes(b, n)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    for _ in range(3):                                         # repeated calls reuse the side stream / events
        rc = L.pcl_chamfer_emd_step(*_lib.pts_args(px), *_lib.pts_args(tx), b, n, 0.005, 50, 0, losses.data_ptr(), gch.data_ptr(),
                                    gem.data_ptr(), scratch.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
        assert rc == 0, L.pcl_last_error()
    torch.cuda.synchronize()
    xg = px.detach().clone().requires_grad_()
    cl, _ = pcl.chamfer_distance(xg, tx)
    cl.backward()
    xe = px.detach().clone().requires_grad_()
    dist, _ = pcl.emdModule()(xe, tx, 0.005, 50)
    el = dist.sqrt().mean()
    el.backward()
    assert float(losses[0] + losses[1]) == pytest.approx(float(cl), rel=1e-6) and float(losses[6]) == pytest.approx(float(el), rel=1e-6)
    np.testing.assert_allclose(npy(gch), npy(xg.grad), rtol=REL, atol=1e-9)
    np.testing.assert_allclose(npy(gem), npy(xe.grad), rtol=REL, atol=1e-10)


def test_composite_step_can_be_captured_in_a_cuda_graph():
    """The whole step (two streams, fork/join events, cluster launch) is capturable: replaying the graph on new inputs
    copied into the captured buffers gives the same losses as a direct call."""
    from pointcloud_b200 import _lib
    L = _lib.lib()
    b, n = 4, 2048
    x1, x2 = synth.uniform_clouds(b, n, seed=40)
    y1, y2 = synth.uniform_clouds(b, n, seed=41)
    pin, tin = x1.cuda(), x2.cuda()
    losses = torch.zeros(8, device="cuda")
    gch, gem = torch.empty(b, n, 3, device="cuda"), torch.empty(b, n, 3, device="cuda")
    nbytes = L.pcl_chamfer_emd_step_scratch_bytes(b, n)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")

    def call(stream):
        rc = L.pcl_chamfer_emd_step(*_lib.pts_args(pin), *_lib.pts_args(tin), b, n, 0.005, 50, 0, losses.data_ptr(), gch.data_ptr(),
                                    gem.data_ptr(), scratch.data_ptr(), nbytes, stream.cuda_stream)
        assert rc == 0, L.pcl_last_error()

    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        call(s)                                   # warm-up outside capture (creates the side stream, sets attributes)
    s.synchronize()
    direct_a = losses.clone()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        call(torch.cuda.current_stream())
    pin.copy_(y1.cuda()); tin.copy_(y2.cuda())
    graph.replay()
    torch.cuda.synchronize()
    replay_b = losses.clone()
    call(torch.cuda.current_stream())
    torch.cuda.synchronize()
    assert torch.equal(replay_b, losses) and not torch.equal(direct_a, replay_b)
    pin.copy_(x1.cuda()); tin.copy_(x2.cuda())
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(losses, direct_a)


def test_sharded_wrapper_single_rank_is_identity():
    pred, target = synth.segmenter_batch(4, 1024, seed=2)
    p1, p2 = pred.cuda().requires_grad_(), pred.cuda().requires_grad_()
    a = pcl.EarthMoverDistance(0.005, 50, num_classes=5)(p1, target.cuda())
    b = pcl.ShardedLoss(pcl.EarthMoverDistance(0.005, 50, num_classes=5))(p2, target.cuda())
    a.backward(); b.backward()
    assert float(a) == pytest.approx(float(b), rel=1e-6)
    np.testing.assert_allclose(npy(p1.grad), npy(p2.grad), rtol=1e-6, atol=1e-12)


def test_fused_feature_term_entry_points():
    """pcl_emd_seg_ce_fwd/bwd and pcl_emd_feat_mse_fwd/bwd against plain torch on strided fp32 / bf16 views
    (utils.py:278-279,293-301): sums and gradients within 1e-5 relative, argmax histogram exact."""
    from pointcloud_b200.losses import _MatchedFeatureMSESums, _SegCrossEntropySums
    g = torch.Generator().manual_seed(31)
    b, n, c = 3, 777, 5
    pred = torch.randn(b, n, 3 + c, generator=g).cuda()
    matched = torch.randint(0, c, (b, n), generator=g).int().cuda()
    cw = torch.rand(c, generator=g).cuda() + 0.1
    for dt in (torch.float32, torch.bfloat16):
        p = pred.detach().to(dt).clone().requires_grad_()
        sums, hist = _SegCrossEntropySums.apply(p[:, :, 3:], matched, cw)
        (sums[0] / sums[1] * 0.7).backward()
        q = pred.detach().to(dt).float().clone().requires_grad_()
        ref = F.cross_entropy(q[:, :, 3:].permute(0, 2, 1), matched.long(), weight=cw)
        (ref * 0.7).backward()
        assert float(sums[0] / sums[1]) == pytest.approx(float(ref), rel=REL)
        assert torch.equal(hist, torch.bincount(q[:, :, 3:].argmax(2).view(-1), minlength=c))
        tol = REL if dt == torch.float32 else 1e-2   # bf16: the gradient itself is rounded to bf16
        np.testing.assert_allclose(npy(p.grad.float()), npy(q.grad), rtol=tol, atol=1e-9 if dt == torch.float32 else 1e-7)
    # matched-feature MSE (Autoencoder): pred (B,N,6), target (B,N,6) permuted by a non-bijective assignment
    predf = torch.rand(b, n, 6, generator=g).cuda().requires_grad_()
    target = torch.rand(b, n, 6, generator=g).cuda()
    asg = torch.randint(0, n, (b, n), generator=g).int().cuda()
    s2 = _MatchedFeatureMSESums.apply(predf[:, :, 3:], target[:, :, 3:], asg)
    (s2[0] / s2[1]).backward()
    q = predf.detach().clone().requires_grad_()
    ref = F.mse_loss(q[:, :, 3:], target.take_along_dim(asg.long().unsqueeze(-1), 1)[:, :, 3:])
    ref.backward()
    assert float(s2[0] / s2[1]) == pytest.approx(float(ref), rel=REL) and float(s2[1]) == b * n * 3
    np.testing.assert_allclose(npy(predf.grad), npy(q.grad), rtol=REL, atol=1e-10)


def _seg_ce(L, logits, matched, cw, grad_sum):
    """pcl_emd_seg_ce_fwd + _bwd through the C ABI -> (rc of the forward, sums, argmax histogram, fp32 gradient)."""
    b, n, c = logits.shape
    sums = torch.full((2,), float("nan"), device="cuda")
    hist = torch.empty(c, device="cuda", dtype=torch.int64)
    grad = torch.full((b, n, c), float("nan"), device="cuda")
    g = torch.tensor([grad_sum], device="cuda")
    wsb = L.pcl_emd_feature_workspace_bytes()
    ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
    st = torch.cuda.current_stream().cuda_stream
    rc = L.pcl_emd_seg_ce_fwd(*pcl._lib.pts_args(logits), matched.data_ptr(), cw.data_ptr(), b, n, c, sums.data_ptr(), hist.data_ptr(),
                              ws.data_ptr(), wsb, st)
    if rc:
        return rc, None, None, None
    assert L.pcl_emd_seg_ce_bwd(*pcl._lib.pts_args(logits), matched.data_ptr(), cw.data_ptr(), b, n, c, g.data_ptr(), grad.data_ptr(), st) == 0
    torch.cuda.synchronize()
    return rc, npy(sums), npy(hist), npy(grad)


@pytest.mark.parametrize("dt", [torch.float32, torch.float16])
@pytest.mark.parametrize("C", [1, 2, 33, 64])
def test_seg_cross_entropy_kernels_at_their_limits(C, dt):
    """pcl_emd_seg_ce_fwd / _bwd against float64 torch up to EP_MAX_C = 64 classes, logits spread over +-50, fp16 logits,
    matched labels outside [0, C) (no weight, no gradient), and rows whose maximum is tied: the argmax histogram counts the
    FIRST maximum, like torch.argmax."""
    L = pcl._lib.lib()
    g = torch.Generator().manual_seed(60 + C)
    b, n = 4, 1000
    z = (torch.rand(b, n, 3 + C, generator=g) * 100 - 50).to(dt)
    ties = torch.rand(b, n, generator=g) < 0.3
    if C > 1:                                            # copy each tied row's maximum to another, random class
        zf = z.float()
        am = zf[:, :, 3:].argmax(2, keepdim=True)
        other = torch.randint(0, C, (b, n, 1), generator=g)
        row_max = zf[:, :, 3:].gather(2, am)
        z[:, :, 3:].scatter_(2, other, torch.where(ties[..., None], row_max, zf[:, :, 3:].gather(2, other)).to(dt))
    logits = z.cuda()[:, :, 3:]                          # strided view, row stride 3 + C
    matched = torch.randint(0, C, (b, n), generator=g, dtype=torch.int32)
    matched[:, ::97] = -1
    matched[:, 5::89] = C
    cw = torch.rand(C, generator=g) + 0.1
    rc, sums, hist, grad = _seg_ce(L, logits, matched.cuda(), cw.cuda(), 0.7)
    assert rc == 0, L.pcl_last_error()
    q = logits.cpu().double()
    lab = matched.long()
    ok = (lab >= 0) & (lab < C)
    lse = torch.logsumexp(q, 2)
    w = torch.where(ok, cw.double()[lab.clamp(0, C - 1)], torch.zeros((), dtype=torch.float64))
    nll = lse - q.gather(2, lab.clamp(0, C - 1)[..., None])[..., 0]
    num, den = float((w * nll).sum()), float(w.sum())
    assert abs(float(sums[0]) - num) <= REL * abs(num) + 1e-6 and float(sums[1]) == pytest.approx(den, rel=1e-6)
    first_max = q.argmax(2)                              # torch.argmax: the first maximal index
    if C > 1:
        last_max = C - 1 - q.flip(2).argmax(2)
        assert (first_max != last_max).sum() > 100       # the tie rule decides the histogram
    assert np.array_equal(hist, np.bincount(first_max.view(-1).numpy(), minlength=C))
    want = 0.7 * w[..., None] * (torch.softmax(q, 2) - F.one_hot(lab.clamp(0, C - 1), C).double() * ok[..., None])
    np.testing.assert_allclose(grad, want.numpy(), rtol=REL, atol=1e-6 * max(float(want.abs().max()), 1e-30))
    assert not grad[~ok.numpy()].any()
    if C == 64:                                          # one class more than the kernels hold
        z65 = torch.rand(b, n, 65, generator=g).cuda()
        from pointcloud_b200._lib import PclError
        from pointcloud_b200.losses import _SegCrossEntropySums
        with pytest.raises(PclError):
            _SegCrossEntropySums.apply(z65, matched.cuda(), torch.rand(65).cuda())
        gbuf, one = torch.empty(b, n, 65, device="cuda"), torch.ones(1, device="cuda")
        assert L.pcl_emd_seg_ce_bwd(*pcl._lib.pts_args(z65), matched.cuda().data_ptr(), torch.rand(65).cuda().data_ptr(), b, n, 65,
                                    one.data_ptr(), gbuf.data_ptr(), torch.cuda.current_stream().cuda_stream) != 0


@pytest.mark.parametrize("F_", [1, 5, 13])
def test_matched_feature_mse_kernels_feature_widths(F_):
    """pcl_emd_feat_mse_fwd / _bwd against float64 torch for F = 1, 5, 13 feature channels (strided views, a non-bijective
    assignment): sums[0] within 1e-5, sums[1] = B*N*F exactly, gradient 2 * g * (feat - tfeat[assignment])."""
    from pointcloud_b200.losses import _MatchedFeatureMSESums
    g = torch.Generator().manual_seed(70 + F_)
    b, n = 3, 1500
    pred = torch.rand(b, n, 3 + F_, generator=g).cuda().requires_grad_()
    target = torch.rand(b, n, 3 + F_, generator=g).cuda()
    asg = torch.randint(0, n, (b, n), generator=g).int().cuda()
    s = _MatchedFeatureMSESums.apply(pred[:, :, 3:], target[:, :, 3:], asg)
    (s[0] * 0.37).backward()
    diff = pred.detach().double()[:, :, 3:] - target.double().take_along_dim(asg.long().unsqueeze(-1), 1)[:, :, 3:]
    num = float((diff ** 2).sum())
    assert abs(float(s[0]) - num) <= REL * num and float(s[1]) == b * n * F_
    np.testing.assert_allclose(npy(pred.grad[:, :, 3:]), npy(0.37 * 2 * diff), rtol=REL, atol=1e-12)
    assert not pred.grad[:, :, :3].any()


@pytest.mark.parametrize("dt", [torch.float32, torch.float16])
def test_match_hist_truncates_labels_like_long(dt):
    """pcl_emd_match_hist at C = 64 with labels that are negative, fractional (-0.5 truncates to 0) or >= C, and unassigned
    points: hist = torch.bincount of the matched targets' labels .long(), restricted to [0, C); matched = those labels."""
    L = pcl._lib.lib()
    g = torch.Generator().manual_seed(80)
    b, n, c = 5, 900, 64
    values = torch.tensor([-3.0, -1.0, -0.5, 0.0, 0.7, 1.0, 5.5, 31.0, 62.9, 63.0, 64.0, 65.0, 100.0])
    lab = torch.where(torch.rand(b, n, generator=g) < 0.5, values[torch.randint(0, len(values), (b, n), generator=g)],
                      torch.randint(0, c, (b, n), generator=g).float())
    target = torch.rand(b, n, 4, generator=g)
    target[:, :, 3] = lab
    tl = target.to(dt).cuda()[:, :, 3:4]
    asg = torch.randint(0, n, (b, n), generator=g, dtype=torch.int32)
    asg[:, ::50] = -1
    hist = torch.empty(c, device="cuda", dtype=torch.int64)
    matched = torch.empty(b, n, device="cuda", dtype=torch.int32)
    rc = L.pcl_emd_match_hist(*pcl._lib.pts_args(tl), asg.cuda().data_ptr(), b, n, c, hist.data_ptr(), matched.data_ptr(),
                              torch.cuda.current_stream().cuda_stream)
    assert rc == 0, L.pcl_last_error()
    lab_long = tl[..., 0].cpu().float().long()
    want = torch.where(asg >= 0, lab_long.gather(1, asg.long().clamp(min=0)), torch.full((), -1, dtype=torch.long))
    assert torch.equal(matched.cpu().long(), want)
    inside = want[(want >= 0) & (want < c)]
    assert torch.equal(hist.cpu(), torch.bincount(inside, minlength=c)[:c])
    assert (lab.gather(1, asg.long().clamp(min=0))[asg >= 0] == -0.5).any()   # some matched label truncates from -0.5 to class 0


def test_class_filter_kernel_matches_the_reference_loop():
    """pcl_class_filter (through FilteringChamferDistance._filter_pad) against the reference's per-cloud loop
    (utils.py:110-124,222-226): kept points in order, zero padding, counts; several labels; fp16 target; a cloud without the class."""
    from pointcloud_b200.losses import FilterClasses, FilteringChamferDistance
    g = torch.Generator().manual_seed(41)
    b, n = 5, 1000
    target = torch.rand(b, n, 4, generator=g)
    target[:, :, 3] = torch.randint(0, 5, (b, n), generator=g).float()
    target[2, :, 3] = 4.0                                   # cloud 2 holds only class 4
    for whitelist, dt in (([1], torch.float32), ([0, 3], torch.float32), ([2], torch.float16)):
        t = target.to(dt).cuda()
        fcd = FilteringChamferDistance(FilterClasses(whitelist, label_dim=3))
        xyz, num = fcd._filter_pad(t, torch.float32)
        assert xyz.shape == (b, n, 3) and num.dtype == torch.int64
        for i in range(b):
            lab = t[i, :, 3].long()
            mask = torch.zeros(n, dtype=torch.bool, device="cuda")
            for v in whitelist:
                mask |= lab == v
            ref = t[i][mask][:, :3].float()
            k = int(num[i])
            assert k == ref.shape[0]
            assert torch.equal(xyz[i, :k], ref) and not xyz[i, k:].any()
    # the loss through the kernel equals the loss through the reference-structure loop (any other callable falls back to it)
    pred = torch.rand(b, 37, 3, generator=g).cuda().requires_grad_()
    tc = target.cuda()
    l1 = FilteringChamferDistance(FilterClasses([1], label_dim=3))(pred, tc)
    l2 = FilteringChamferDistance(lambda p: FilterClasses([1], label_dim=3)(p))(pred, tc)
    assert float(l1) == pytest.approx(float(l2), rel=REL)


def test_chamfer_emd_loss_equals_the_separate_calls():
    """pcl.chamfer_emd_loss (one fused C-ABI call, both gradients from the forward) == chamfer_distance + emdModule().sqrt().mean()
    with autograd, value and gradient, including extra channels and upstream gradients other than 1."""
    x1, t = synth.table_clouds(6, 1024, seed=77, regime="noisy")
    pred6 = torch.cat([x1, torch.rand(6, 1024, 3)], dim=2).cuda()
    target = t.cuda()
    for p0, tg in ((x1.cuda(), target[:, :, :3].contiguous()), (pred6, target)):
        pa = p0.clone().requires_grad_()
        c, e = pcl.chamfer_emd_loss(pa, tg, 0.005, 50)
        (2.0 * c + 0.5 * e).backward()
        pb = p0.clone().requires_grad_()
        c2, _ = pcl.chamfer_distance(pb[:, :, :3], tg[:, :, :3])
        d, _ = pcl.emdModule()(pb[:, :, :3], tg[:, :, :3], 0.005, 50)
        e2 = d.sqrt().mean()
        (2.0 * c2 + 0.5 * e2).backward()
        assert abs(float(c) - float(c2)) <= 1e-6 * abs(float(c2)) and abs(float(e) - float(e2)) <= 1e-6 * abs(float(e2))
        assert pa.grad.shape == pb.grad.shape
        assert torch.allclose(pa.grad, pb.grad, rtol=1e-5, atol=1e-9)


def test_ticket_path_is_capturable_in_a_cuda_graph():
    """The ticket path launches its worker kernel on a library-owned stream (forked / joined with events): the pair must record into a CUDA
    graph like the composite step does, and replaying the graph on new inputs must give the oracle's assignment."""
    import oracle
    b, n = 48, 2048                       # clusters of 2 + 52 worker CTAs
    xa, ta = synth.table_clouds(b, n, seed=5, regime="independent")
    xb, tb = synth.table_clouds(b, n, seed=6, regime="noisy")
    x1, x2 = xa.cuda(), ta[:, :, :3].contiguous().cuda()
    pcl.set_emd_path("tickets")
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            pcl.emd_forward_raw(x1, x2, 0.005, 50)   # warm-up outside the capture (attributes, streams, events exist)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            d, a, _ = pcl.emd_forward_raw(x1, x2, 0.005, 50)
        for xs, ts in ((xb, tb), (xa, ta)):
            x1.copy_(xs.cuda()); x2.copy_(ts[:, :, :3].contiguous().cuda())
            g.replay()
            torch.cuda.synchronize()
            o = oracle.emd_forward(xs, ts[:, :, :3].contiguous(), 0.005, 50, nthreads=16)
            assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
    finally:
        pcl.set_emd_path("auto")
