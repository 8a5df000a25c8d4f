"""Every entry point's result depends only on its inputs: not on what earlier kernels left in shared memory, nor on the
contents of the workspace or of the outputs it is handed.

Before each call, on the call's stream and in this order: the outputs are filled with a poison (fp32: the pattern's bits,
int32: 0x7fffffff or -2, int64: 0x5a bytes), the workspace with the pattern's bytes, and every SM's shared memory with the
pattern (tests/smem_poison.cu).  The results of one call under every pattern must be bit-identical (NaN equal to NaN), equal
the oracle, and hold their documented pad values.  Outputs accumulated with fp32 atomics (kNN / ball query grad_p2, the
Chamfer gradients) are checked against a float64 np.add.at reference instead, with rows that get nothing exactly 0.
The canary test first establishes that the poison reaches every SM and survives until the next kernel.
The graph tests capture every entry point on a side stream and replay it on new inputs.

Mutation runs may select the forward tests alone (-k forward): those compare kernel outputs on the host only and never
feed a kernel-made index to another kernel."""
import numpy as np
import pytest
import torch

import ball_query_oracle as bqo
import knn_oracle as ko
import oracle
import pointcloud_b200 as pcl
import smem_poison
from emd_epilogue_ref import epilogue_grad, epilogue_sum, float32_neighbours
from fps_ragged_oracle import fps_ragged
from helpers import npy, reference_structure, same_bits
from pointcloud_b200 import _lib, synth

pytestmark = pytest.mark.gpu

PATTERNS = (0x00000000, 0xFFFFFFFF, 0x7F7FFFFF, 0xFF7FFFFF, 0x3F000000, 0xBF000000)
LARGE = (0x00000000, 0xFF7FFFFF)          # two patterns where the inputs are large
EPS, ITERS = 0.005, 50
REL = 1e-5


def _i32(p):
    return p - (1 << 32) if p >= 1 << 31 else p


def _pats(elements):
    return PATTERNS if elements <= 40000 else LARGE


def _rand(shape, seed, scale=1.0):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed)) * scale


class Stale:
    """Runs one call under each pattern on a side stream; see the module docstring."""

    def __init__(self):
        self.L = _lib.lib()
        self.stream = torch.cuda.Stream()
        self.hits = torch.zeros(smem_poison.MAX_SMID, dtype=torch.int32, device="cuda")
        self.sms = torch.cuda.get_device_properties(0).multi_processor_count

    def prepare(self, pattern, k, outs, scratch):
        with torch.cuda.stream(self.stream):
            self.hits.zero_()
            for t in outs:
                if t.dtype == torch.float32:
                    t.view(torch.int32).fill_(_i32(pattern))
                elif t.dtype == torch.int32:
                    t.fill_(0x7FFFFFFF if k % 2 == 0 else -2)
                else:
                    assert t.dtype == torch.int64
                    t.view(torch.uint8).fill_(0x5A)
            for w in scratch:
                w.view(torch.int32).fill_(_i32(pattern))
            smem_poison.poison(pattern, self.stream, self.hits)

    def run(self, patterns, outs, scratch, call, loose=(), check=None):
        """-> one list of host arrays per pattern.  Outputs whose position is in `loose` are not compared across patterns.
        check(arrays) -> bool, when given, is the oracle comparison of every pattern's result; the failure names the patterns."""
        self.stream.wait_stream(torch.cuda.current_stream())
        res = []
        for k, p in enumerate(patterns):
            self.prepare(p, k, outs, scratch)
            with torch.cuda.stream(self.stream):
                rc = call(self.stream.cuda_stream)
            assert rc == 0, self.L.pcl_last_error()
            self.stream.synchronize()
            assert int((self.hits > 0).sum()) == self.sms
            res.append([npy(t).copy() for t in outs])
        if check is not None:
            wrong = [f"{p:#010x}" for p, r in zip(patterns, res) if not check(r)]
            assert not wrong, f"patterns {wrong} differ from the oracle"
        for i in range(len(outs)):
            if i not in loose:
                eq = [same_bits(res[0][i], r[i]) if r[i].dtype == np.float32 else np.array_equal(res[0][i], r[i]) for r in res]
                assert all(eq), f"output {i}: patterns {[f'{p:#010x}' for p, e in zip(patterns, eq) if not e]} differ from {patterns[0]:#010x}"
        return res


@pytest.fixture(scope="module")
def stale():
    return Stale()


@pytest.fixture
def emd_path():
    yield pcl.set_emd_path
    pcl.set_emd_path("auto")


def close(got, want, scale=None):
    """got (fp32) within 1e-5 relative of the float64 reference; rows the reference leaves at 0 exactly 0."""
    want = np.asarray(want, np.float64)
    s = scale if scale is not None else max(float(np.abs(want).max(initial=0.0)), 1e-30)
    np.testing.assert_allclose(got, want, rtol=REL, atol=1e-6 * s)


# ---------------------------------------------------------------- the canary ----------------------------------------------

def test_canary_every_sm_keeps_the_poison_until_the_next_kernel(stale):
    """Poison with two patterns in turn; after each, a kernel that only reads its shared memory finds the pattern on every SM.
    Without this the poison tests below would prove nothing."""
    bad = torch.zeros(smem_poison.MAX_SMID, dtype=torch.int32, device="cuda")
    peek_hits = torch.zeros_like(bad)
    for p in (0x3F000000, 0xFF7FFFFF):
        with torch.cuda.stream(stale.stream):
            stale.hits.zero_(); bad.zero_(); peek_hits.zero_()
            smem_poison.poison(p, stale.stream, stale.hits)
            smem_poison.peek(p, stale.stream, peek_hits, bad)
        stale.stream.synchronize()
        assert int((stale.hits > 0).sum()) == stale.sms and int((peek_hits > 0).sum()) == stale.sms
        assert not bad.any(), f"pattern {p:#x}: {int((bad > 0).sum())} SMs lost it"


# ---------------------------------------------------------------- EMD -----------------------------------------------------

EMD_CASES = [(path, b, n, "fp32") for path in ("cluster", "team", "tickets") for b, n in ((2, 37), (1, 1), (3, 1000), (4, 2047))]
EMD_CASES += [("auto", 48, 2047, "fp32"), ("auto", 2, 3585, "fp32"), ("auto", 1, 5000, "fp32"), ("cluster", 3, 1000, "fp16")]
_ORACLE = {}


def emd_inputs(b, n, form="fp32"):
    pred, target = synth.autoencoder_batch(b, n, seed=7919 * b + n)
    x1, x2 = pred[:, :, :3].contiguous(), target[:, :, :3].contiguous()
    if form == "fp16":
        x1 = x1.half()
    key = (b, n, form)
    if key not in _ORACLE:
        a1, a2 = x1.float().numpy(), x2.numpy()
        _ORACLE[key] = (a1, a2, oracle.emd_forward(a1, a2, EPS, ITERS, nthreads=16))
    return x1.cuda(), x2.cuda(), _ORACLE[key]


@pytest.mark.parametrize("path,b,n,form", EMD_CASES)
def test_emd_forward_and_fused_epilogue(stale, emd_path, path, b, n, form):
    emd_path(path)
    L = stale.L
    x1, x2, (a1, a2, o) = emd_inputs(b, n, form)
    pats = _pats(b * n * 8)
    dist, asg = torch.empty(b, n, device="cuda"), torch.empty(b, n, device="cuda", dtype=torch.int32)
    grad, sums = torch.empty(b, n, 3, device="cuda"), torch.empty(3, device="cuda")
    wsb = L.pcl_emd_workspace_bytes(b, n)
    ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
    args = (*_lib.pts_args(x1), *_lib.pts_args(x2), b, n, EPS, ITERS, dist.data_ptr(), asg.data_ptr(), None)
    d, a = stale.run(pats, [dist, asg], [ws], lambda s: L.pcl_emd_fwd(*args, ws.data_ptr(), wsb, s))[0]
    assert np.array_equal(d, o["dist"]) and np.array_equal(a, o["assignment"])
    gs = np.float32(1.0 / (b * n))
    d, a, g, sm = stale.run(pats, [dist, asg, grad, sums], [ws],
                            lambda s: L.pcl_emd_fwd_fused(*args, float(gs), grad.data_ptr(), sums.data_ptr(), ws.data_ptr(), wsb, s))[0]
    assert np.array_equal(d, o["dist"]) and np.array_equal(a, o["assignment"])
    assert same_bits(g, epilogue_grad(a1, a2, o["dist"], o["assignment"], gs))
    s, count, _ = epilogue_sum(o["dist"])
    assert sm[1] == np.float32(count) and sm[0] in float32_neighbours(s) and sm[2] == np.float32(sm[0]) / np.float32(sm[1])


def emd_side_inputs(b, n, C, seed):
    """Prediction, target with an integer label in channel 3, a permutation assignment and its squared distances."""
    g = torch.Generator().manual_seed(seed)
    x1, t = torch.rand(b, n, 3, generator=g), torch.rand(b, n, 4, generator=g)
    t[:, :, 3] = torch.randint(0, C, (b, n), generator=g).float()
    asg = torch.stack([torch.randperm(n, generator=g) for _ in range(b)]).int()
    m = t[:, :, :3].gather(1, asg.long()[..., None].expand(-1, -1, 3))
    dist = ((x1 - m) ** 2).sum(-1) + 1e-4
    return x1, t, asg, dist


@pytest.mark.parametrize("n", [37, 2047])
@pytest.mark.parametrize("C", [1, 7, 64])
def test_emd_backward_match_hist_and_weighted_reduce(stale, n, C):
    L = stale.L
    b = 3
    x1, t, asg, dist = emd_side_inputs(b, n, C, seed=n + C)
    xc, tc, ac, dc = x1.cuda(), t.cuda(), asg.cuda(), dist.cuda()
    pats = _pats(b * n * 3)
    # pcl_emd_bwd: the oracle, bit for bit
    gd = _rand((b, n), 5 + n).cuda()
    grad = torch.empty(b, n, 3, device="cuda")
    (g,) = stale.run(pats, [grad], [], lambda s: L.pcl_emd_bwd(*_lib.pts_args(xc), *_lib.pts_args(tc), b, n, ac.data_ptr(),
                                                                gd.data_ptr(), grad.data_ptr(), s))[0]
    assert same_bits(g, oracle.emd_backward(x1, t[:, :, :3], asg, gd.cpu())[0])
    # pcl_emd_match_hist: the histogram of the permuted target's labels, and those labels
    hist, matched = torch.empty(C, device="cuda", dtype=torch.int64), torch.empty(b, n, device="cuda", dtype=torch.int32)
    lab = tc[:, :, 3:4]
    h, m = stale.run(pats, [hist, matched], [], lambda s: L.pcl_emd_match_hist(*_lib.pts_args(lab), ac.data_ptr(), b, n, C,
                                                                               hist.data_ptr(), matched.data_ptr(), s))[0]
    want = t[:, :, 3].long().gather(1, asg.long()).numpy()
    assert np.array_equal(m, want) and np.array_equal(h, np.bincount(want.ravel(), minlength=C))
    # pcl_emd_weighted_reduce and pcl_emd_weighted_bwd with class weights
    cw = (_rand((C,), C) + 0.1).cuda()
    sums = torch.empty(2, device="cuda")
    wsb = L.pcl_emd_workspace_bytes(b, n)
    ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
    (sm,) = stale.run(pats, [sums], [ws], lambda s: L.pcl_emd_weighted_reduce(dc.data_ptr(), matched.data_ptr(), cw.data_ptr(), b, n, C,
                                                                               sums.data_ptr(), ws.data_ptr(), wsb, s))[0]
    w = cw.cpu().double().numpy()[want]
    d64 = dist.double().numpy()
    num, den = float((w * np.sqrt(d64)).sum()), float(w.sum())
    assert abs(float(sm[0]) - num) <= 1e-6 * num and abs(float(sm[1]) - den) <= 1e-6 * den
    gout = torch.tensor([0.37], device="cuda")
    (g,) = stale.run(pats, [grad], [], lambda s: L.pcl_emd_weighted_bwd(*_lib.pts_args(xc), *_lib.pts_args(tc), b, n, ac.data_ptr(),
                                                                         dc.data_ptr(), matched.data_ptr(), cw.data_ptr(), C,
                                                                         sums.data_ptr(), gout.data_ptr(), grad.data_ptr(), s))[0]
    mt = t[:, :, :3].double().gather(1, asg.long()[..., None].expand(-1, -1, 3)).numpy()
    want_g = 2 * (0.37 * w / (2 * np.sqrt(d64)) / float(sm[1]))[..., None] * (x1.double().numpy() - mt)
    close(g, want_g)


# ---------------------------------------------------------------- loss feature terms and the class filter ------------------

@pytest.mark.parametrize("C", [1, 33, 64])
def test_seg_cross_entropy(stale, C):
    L = stale.L
    b, n = 3, 1000
    g = torch.Generator().manual_seed(90 + C)
    logits = (torch.rand(b, n, C, generator=g) * 20 - 10)
    matched = torch.randint(0, C, (b, n), generator=g, dtype=torch.int32)
    matched[:, ::97] = -1                                     # labels outside [0, C): no weight, no gradient
    matched[:, 5::89] = C
    cw = torch.rand(C, generator=g) + 0.1
    lc, mc, cwc = logits.cuda(), matched.cuda(), cw.cuda()
    sums, hist = torch.empty(2, device="cuda"), torch.empty(C, device="cuda", dtype=torch.int64)
    grad = torch.empty(b, n, C, device="cuda")
    wsb = L.pcl_emd_feature_workspace_bytes()
    ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
    sm, h = stale.run(PATTERNS, [sums, hist], [ws], lambda s: L.pcl_emd_seg_ce_fwd(*_lib.pts_args(lc), mc.data_ptr(), cwc.data_ptr(), b, n, C,
                                                                                    sums.data_ptr(), hist.data_ptr(), ws.data_ptr(), wsb, s))[0]
    gsum = torch.tensor([0.7], device="cuda")
    (gr,) = stale.run(PATTERNS, [grad], [], lambda s: L.pcl_emd_seg_ce_bwd(*_lib.pts_args(lc), mc.data_ptr(), cwc.data_ptr(), b, n, C,
                                                                            gsum.data_ptr(), grad.data_ptr(), s))[0]
    q, lab = logits.double(), matched.long()
    ok = (lab >= 0) & (lab < C)
    w = torch.where(ok, cw.double()[lab.clamp(0, C - 1)], torch.zeros((), dtype=torch.float64))
    nll = torch.logsumexp(q, 2) - q.gather(2, lab.clamp(0, C - 1)[..., None])[..., 0]
    num, den = float((w * nll).sum()), float(w.sum())
    assert abs(float(sm[0]) - num) <= REL * abs(num) + 1e-6 and abs(float(sm[1]) - den) <= 1e-6 * den
    assert np.array_equal(h, np.bincount(q.argmax(2).view(-1).numpy(), minlength=C))
    onehot = torch.nn.functional.one_hot(lab.clamp(0, C - 1), C).double() * ok[..., None]
    close(gr, (0.7 * w[..., None] * (torch.softmax(q, 2) - onehot)).numpy())
    assert not gr[~ok.numpy()].any()


@pytest.mark.parametrize("F", [1, 5, 13])
def test_feature_mse(stale, F):
    L = stale.L
    b, n = 3, 1000
    g = torch.Generator().manual_seed(100 + F)
    pred, target = torch.rand(b, n, 3 + F, generator=g), torch.rand(b, n, 3 + F, generator=g)
    asg = torch.randint(0, n, (b, n), generator=g, dtype=torch.int32)   # not a bijection
    fc, tc, ac = pred.cuda()[:, :, 3:], target.cuda()[:, :, 3:], asg.cuda()
    sums, grad = torch.empty(2, device="cuda"), torch.empty(b, n, F, device="cuda")
    wsb = L.pcl_emd_feature_workspace_bytes()
    ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
    (sm,) = stale.run(PATTERNS, [sums], [ws], lambda s: L.pcl_emd_feat_mse_fwd(*_lib.pts_args(fc), *_lib.pts_args(tc), ac.data_ptr(), b, n, F,
                                                                                sums.data_ptr(), ws.data_ptr(), wsb, s))[0]
    gsum = torch.tensor([0.37], device="cuda")
    (gr,) = stale.run(PATTERNS, [grad], [], lambda s: L.pcl_emd_feat_mse_bwd(*_lib.pts_args(fc), *_lib.pts_args(tc), ac.data_ptr(), b, n, F,
                                                                              gsum.data_ptr(), grad.data_ptr(), s))[0]
    diff = pred.double()[:, :, 3:] - target.double().take_along_dim(asg.long()[..., None], 1)[:, :, 3:]
    num = float((diff ** 2).sum())
    assert abs(float(sm[0]) - num) <= REL * num and float(sm[1]) == b * n * F
    close(gr, (0.37 * 2 * diff).numpy())


@pytest.mark.parametrize("labels", [[3], list(range(2, 18))])
def test_class_filter(stale, labels):
    L = stale.L
    b, n = 4, 1000
    g = torch.Generator().manual_seed(len(labels))
    target = torch.rand(b, n, 5, generator=g)
    target[:, :, 4] = torch.randint(0, 20, (b, n), generator=g).float()
    target[2, :, 4] = 19.0                                    # a cloud without any kept class
    target[3, :, 4] = float(labels[0])                        # a cloud that is kept whole
    tc = target.cuda()
    out, lengths = torch.empty(b, n, 3, device="cuda"), torch.empty(b, device="cuda", dtype=torch.int64)
    lab = (_lib.c_int64 * len(labels))(*labels)
    o, ln = stale.run(PATTERNS, [out, lengths], [], lambda s: L.pcl_class_filter(*_lib.pts_args(tc), b, n, 4, lab, len(labels),
                                                                                 out.data_ptr(), lengths.data_ptr(), s))[0]
    for c in range(b):
        keep = np.isin(target[c, :, 4].long().numpy(), labels)
        k = int(keep.sum())
        assert ln[c] == k and np.array_equal(o[c, :k], target[c, keep, :3].numpy()) and not o[c, k:].any()
    assert ln[2] == 0 and ln[3] == n


# ---------------------------------------------------------------- Chamfer -------------------------------------------------

# (D, B, P1, P2, lengths): brute force at D = 3 and every generic width, the pruned path at 6145 points
CHAMFER_CASES = {
    "d3": (3, 4, 1000, 1025, ([1000, 0, 1, 257], [1, 0, 1025, 300])),
    "d1": (1, 4, 300, 513, ([300, 0, 1, 77], [513, 0, 1, 40])),
    "d2": (2, 4, 300, 513, ([300, 0, 1, 77], [1, 0, 513, 40])),
    "d5": (5, 4, 300, 513, ([300, 0, 1, 77], [513, 0, 1, 40])),
    "d8": (8, 4, 300, 513, ([1, 0, 300, 77], [513, 0, 1, 40])),
    "pruned": (3, 3, 6145, 6145, ([6145, 0, 6000], [6145, 0, 6144])),
}
_CH = {}


@pytest.fixture
def prune_min():
    L = _lib.lib()
    yield L.pcl_chamfer_set_prune_min
    L.pcl_chamfer_set_prune_min(-1)


def chamfer_case(name, mode, ragged):
    d, b, p1, p2, lens = CHAMFER_CASES[name]
    x, y = _rand((b, p1, d), p1 + d), _rand((b, p2, d), p2 + 10 * d)
    xl, yl = (torch.tensor(lens[0]), torch.tensor(lens[1])) if ragged else (None, None)
    key = (name, mode, ragged)
    if key not in _CH:
        _CH[key] = oracle.chamfer_forward(x, y, xl, yl, mode=mode, nthreads=8)
    return x, y, xl, yl, _CH[key]


def chamfer_fwd_call(L, xc, yc, xl, yl, b, p1, p2, d, mode, outs, ws):
    dx, ix, dy, iy, loss = outs
    return lambda s: L.pcl_chamfer_fwd(*_lib.pts_args(xc), _lib.ptr(xl), *_lib.pts_args(yc), _lib.ptr(yl), b, p1, p2, d, mode,
                                       dx.data_ptr(), ix.data_ptr(), dy.data_ptr(), iy.data_ptr(), loss.data_ptr(), ws.data_ptr(),
                                       ws.numel(), s)


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("name", list(CHAMFER_CASES))
def test_chamfer_forward(stale, prune_min, name, mode, ragged):
    L = stale.L
    prune_min(6144 if name == "pruned" else 0)
    x, y, xl, yl, o = chamfer_case(name, mode, ragged)
    b, p1, d = x.shape
    p2 = y.shape[1]
    xc, yc = x.cuda(), y.cuda()
    xlc, ylc = (xl.cuda(), yl.cuda()) if ragged else (None, None)
    outs = [torch.empty(b, p1, device="cuda"), torch.empty(b, p1, device="cuda", dtype=torch.int32),
            torch.empty(b, p2, device="cuda"), torch.empty(b, p2, device="cuda", dtype=torch.int32), torch.empty(4, device="cuda")]
    ws = torch.empty(L.pcl_chamfer_workspace_bytes(b, p1, p2), device="cuda", dtype=torch.uint8)
    want = (o["dist_x"], o["idx_x"], o["dist_y"], o["idx_y"])              # padded rows: 0 / 0
    dx, ix, dy, iy, loss = stale.run(_pats(b * max(p1, p2)), outs, [ws], chamfer_fwd_call(L, xc, yc, xlc, ylc, b, p1, p2, d, mode, outs, ws),
                                     check=lambda r: all(np.array_equal(g, w) for g, w in zip(r, want)))[0]
    for k, ref in ((0, o["loss_x"]), (1, o["loss_y"])):
        assert abs(float(loss[k]) - float(ref)) <= 1e-6 * abs(float(ref)) + 1e-30
        assert abs(float(loss[k + 2]) - b * float(ref)) <= 1e-6 * b * abs(float(ref)) + 1e-30


def chamfer_grad_ref(x, y, xl, yl, ix, iy, g):
    """float64 np.add.at restatement of pcl_chamfer_bwd (include/pcl.h) -> (grad_x, grad_y, rows of grad_x / grad_y that get
    a contribution)."""
    x, y = x.double().numpy(), y.double().numpy()
    b, p1, _ = x.shape
    p2 = y.shape[1]
    gx, gy = np.zeros_like(x), np.zeros_like(y)
    hx, hy = np.zeros((b, p1), bool), np.zeros((b, p2), bool)
    for n in range(b):
        lx = p1 if xl is None else int(xl[n])
        ly = p2 if yl is None else int(yl[n])
        if lx == 0 or ly == 0:
            continue
        for q, t, lq, idx, gq, gt, hq, ht, gg in ((x, y, lx, ix, gx, gy, hx, hy, g[0]), (y, x, ly, iy, gy, gx, hy, hx, g[1])):
            j = idx[n, :lq].astype(np.int64)
            diff = 2 * (gg / max(b, 1) / max(lq, 1)) * (q[n, :lq] - t[n, j])
            gq[n, :lq] += diff
            np.add.at(gt[n], j, -diff)
            hq[n, :lq] = True
            ht[n, j] = True
    return gx, gy, hx, hy


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("name", ["d3", "d5", "pruned"])
def test_chamfer_backward(stale, name, ragged):
    """The gradients are fp32 atomics: each pattern's against the float64 scatter of the oracle's indices."""
    L = stale.L
    x, y, xl, yl, o = chamfer_case(name, 0, ragged)
    b, p1, d = x.shape
    p2 = y.shape[1]
    xc, yc = x.cuda(), y.cuda()
    xlc, ylc = (xl.cuda(), yl.cuda()) if ragged else (None, None)
    ixc, iyc = torch.from_numpy(o["idx_x"]).cuda(), torch.from_numpy(o["idx_y"]).cuda()
    gout = torch.tensor([1.0, 0.37], device="cuda")
    gx, gy = torch.empty(b, p1, d, device="cuda"), torch.empty(b, p2, d, device="cuda")
    res = stale.run(_pats(b * max(p1, p2)), [gx, gy], [], loose=(0, 1),
                    call=lambda s: L.pcl_chamfer_bwd(*_lib.pts_args(xc), _lib.ptr(xlc), *_lib.pts_args(yc), _lib.ptr(ylc), b, p1, p2, d,
                                                     ixc.data_ptr(), iyc.data_ptr(), gout.data_ptr(), gx.data_ptr(), gy.data_ptr(), s))
    rx, ry, hx, hy = chamfer_grad_ref(x, y, xl, yl, o["idx_x"], o["idx_y"], (1.0, 0.37))
    for gxa, gya in res:
        close(gxa, rx); close(gya, ry)
        assert not gxa[~hx].any() and not gya[~hy].any()


# ---------------------------------------------------------------- kNN -----------------------------------------------------

KNN_CASES = [(d, K) for d in (1, 3, 8) for K in (1, 17, 64)]
KNN_LENS = (torch.tensor([300, 0, 77]), torch.tensor([513, 1, 40]))    # fewer targets than K: pad slots 0 / 0


def knn_inputs(d, K, split):
    if split:                                              # B = 1, one query warp: parts_for splits the targets over warps
        return _rand((1, 32, d), d), _rand((1, 40000, d), 40000 + d), None, None
    return _rand((3, 300, d), d + K), _rand((3, 513, d), 513 + d + K), *KNN_LENS


@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("d,K", KNN_CASES)
def test_knn_forward(stale, d, K, split):
    L = stale.L
    p1, p2, l1, l2 = knn_inputs(d, K, split)
    b, n1, _ = p1.shape
    n2 = p2.shape[1]
    a, c = p1.cuda(), p2.cuda()
    l1c, l2c = (l1.cuda(), l2.cuda()) if l1 is not None else (None, None)
    dists, idx = torch.empty(b, n1, K, device="cuda"), torch.empty(b, n1, K, device="cuda", dtype=torch.int32)
    mode = d % 2                                           # both arithmetic modes over the widths
    od, oi = ko.knn_forward(p1, p2, K, l1, l2, mode=mode)
    dd, ii = stale.run(_pats(b * n2), [dists, idx], [], lambda s: L.pcl_knn_fwd(*_lib.pts_args(a), _lib.ptr(l1c), *_lib.pts_args(c),
                                                                                   _lib.ptr(l2c), b, n1, n2, d, K, mode, dists.data_ptr(),
                                                                                   idx.data_ptr(), s),
                       check=lambda r: same_bits(r[0], od) and np.array_equal(r[1], oi))[0]
    if l1 is not None:                                     # the pads themselves: rows past len1, slots past len2
        assert not dd[1].any() and not ii[1].any() and not dd[2, 77:].any() and not ii[2, 77:].any()
        assert not dd[2, :, 40:].any() and not ii[2, :, 40:].any()


def _scatter_ref(p1, p2, idx, gd, l1, l2, K):
    """float64 restatement of the kNN / ball-query backward (include/pcl.h) -> (grad_p1, grad_p2, rows of grad_p2 that get
    a contribution); slots with idx -1 contribute nothing."""
    a, c = p1.double().numpy(), p2.double().numpy()
    b, n1, _ = a.shape
    n2 = c.shape[1]
    g1, g2 = np.zeros_like(a), np.zeros_like(c)
    hit = np.zeros((b, n2), bool)
    for n in range(b):
        lq = n1 if l1 is None else int(l1[n])
        lt = n2 if l2 is None else int(l2[n])
        for k in range(min(K, lt)):
            j = idx[n, :lq, k].astype(np.int64)
            ok = j >= 0
            diff = 2 * gd[n, :lq, k, None].astype(np.float64) * (a[n, :lq] - c[n, np.maximum(j, 0)]) * ok[:, None]
            g1[n, :lq] += diff
            np.add.at(g2[n], j[ok], -diff[ok])
            hit[n, j[ok]] = True
    return g1, g2, hit


@pytest.mark.parametrize("d,K", [(1, 17), (3, 64), (8, 1)])
def test_knn_backward(stale, d, K):
    """grad_p1 (one thread per row, fixed order) is bit-identical under every pattern; grad_p2 is fp32 atomics."""
    L = stale.L
    p1, p2, l1, l2 = knn_inputs(d, K, False)
    b, n1, _ = p1.shape
    n2 = p2.shape[1]
    _, oi = ko.knn_forward(p1, p2, K, l1, l2)
    gd = _rand((b, n1, K), 3 * K) - 0.5
    a, c, ic, gdc, l1c, l2c = p1.cuda(), p2.cuda(), torch.from_numpy(oi).cuda(), gd.cuda(), l1.cuda(), l2.cuda()
    g1, g2 = torch.empty(b, n1, d, device="cuda"), torch.empty(b, n2, d, device="cuda")
    res = stale.run(PATTERNS, [g1, g2], [], loose=(1,),
                    call=lambda s: L.pcl_knn_bwd(*_lib.pts_args(a), _lib.ptr(l1c), *_lib.pts_args(c), _lib.ptr(l2c), b, n1, n2, d, K,
                                                 ic.data_ptr(), gdc.data_ptr(), g1.data_ptr(), g2.data_ptr(), s))
    r1, r2, hit = _scatter_ref(p1, p2, oi, gd.numpy(), l1, l2, K)
    for ga, gb in res:
        close(ga, r1); close(gb, r2)
        assert not gb[~hit].any() and not ga[1].any() and not ga[2, 77:].any()


# ---------------------------------------------------------------- ball query ----------------------------------------------

# (K, D, split): P2 = 129 never splits; the split cases give one query warp 1300 targets (bq_parts_for: 4 parts at K = 5,
# 2 at K = 500; K = 961 is above the split bound and runs unsplit)
BQ_CASES = [(K, d, False) for K in (1, 5, 500, 961) for d in (3, 8)] + [(5, 3, True), (500, 3, True), (961, 3, True), (500, 8, True)]


def bq_inputs(K, d, split):
    r = 0.35 if d == 3 else 0.8
    if split:
        return _rand((1, 32, d), K + d), _rand((1, 1300, d), 1300 + d), None, torch.tensor([1299]), r
    return _rand((3, 100, d), K + d), _rand((3, 129, d), 129 + K + d), torch.tensor([100, 0, 31]), torch.tensor([129, 5, 1]), r


@pytest.mark.parametrize("K,d,split", BQ_CASES)
def test_ball_query_forward(stale, K, d, split):
    L = stale.L
    p1, p2, l1, l2, r = bq_inputs(K, d, split)
    b, n1, _ = p1.shape
    n2 = p2.shape[1]
    r2 = bqo.radius2(r)
    a, c = p1.cuda(), p2.cuda()
    l1c, l2c = (l1.cuda() if l1 is not None else None), l2.cuda()
    dists, idx = torch.empty(b, n1, K, device="cuda"), torch.empty(b, n1, K, device="cuda", dtype=torch.int32)
    od, oi = bqo.ball_query_forward(p1, p2, K, r2, l1, l2)
    dd, ii = stale.run(_pats(b * n1 * K), [dists, idx], [],
                       lambda s: L.pcl_ball_query_fwd(*_lib.pts_args(a), _lib.ptr(l1c), *_lib.pts_args(c), _lib.ptr(l2c), b, n1, n2, d, K,
                                                      r2, 0, dists.data_ptr(), idx.data_ptr(), s),
                       check=lambda r: same_bits(r[0], od) and np.array_equal(r[1], oi))[0]
    assert not dd[ii < 0].any() and ((ii >= 0).sum(-1) > 0).any()           # pads 0 / -1, and some hits
    if K == 961:
        assert (ii[..., -1] == -1).all()


@pytest.mark.parametrize("K,d,split", [(5, 3, False), (961, 8, False), (500, 3, True)])
def test_ball_query_backward(stale, K, d, split):
    L = stale.L
    p1, p2, l1, l2, r = bq_inputs(K, d, split)
    b, n1, _ = p1.shape
    n2 = p2.shape[1]
    _, oi = bqo.ball_query_forward(p1, p2, K, bqo.radius2(r), l1, l2)
    gd = _rand((b, n1, K), K) - 0.5
    a, c, ic, gdc = p1.cuda(), p2.cuda(), torch.from_numpy(oi).cuda(), gd.cuda()
    l1c, l2c = (l1.cuda() if l1 is not None else None), l2.cuda()
    g1, g2 = torch.empty(b, n1, d, device="cuda"), torch.empty(b, n2, d, device="cuda")
    res = stale.run(_pats(b * n1 * K), [g1, g2], [], loose=(1,),
                    call=lambda s: L.pcl_ball_query_bwd(*_lib.pts_args(a), _lib.ptr(l1c), *_lib.pts_args(c), _lib.ptr(l2c), b, n1, n2, d,
                                                        K, ic.data_ptr(), gdc.data_ptr(), g1.data_ptr(), g2.data_ptr(), s))
    r1, r2_, hit = _scatter_ref(p1, p2, oi, gd.numpy(), l1, l2, K)
    for ga, gb in res:
        close(ga, r1); close(gb, r2_)
        assert not gb[~hit].any()


# ---------------------------------------------------------------- sampling: pointnet2 ball query, FPS -------------------

def test_pointnet2_ball_query_forward(stale):
    L = stale.L
    b, n, s_, ns, r = 2, 513, 100, 32, 0.2
    xyz, new = _rand((b, n, 3), 1), _rand((b, s_, 3), 2)
    xc, nc = xyz.cuda(), new.cuda()
    out = torch.empty(b, s_, ns, device="cuda", dtype=torch.int32)
    r2 = float(torch.tensor(r ** 2, dtype=torch.float32))
    (o,) = stale.run(PATTERNS, [out], [], lambda s: L.pcl_ball_query(*_lib.pts_args(xc), *_lib.pts_args(nc), b, n, s_, r2, ns,
                                                                      out.data_ptr(), s))[0]
    assert np.array_equal(o, oracle.ball_query(r, ns, xyz, new))


FPS_CASES = [(513, c) for c in (1, 2, 4, 8, 16)] + [(16385, c) for c in (2, 4, 8, 16)]


@pytest.mark.parametrize("n,cluster", FPS_CASES)
def test_fps_forward(stale, n, cluster):
    """pcl_fps_ragged at every forced cluster size (ragged lengths, per-cloud K, -1 pads) and pcl_fps at the automatic one."""
    L = stale.L
    b, npoint = 3, 64
    xyz = _rand((b, n, 3), n + cluster)
    lengths, K = torch.tensor([n, n // 2 + 1, 1]), torch.tensor([64, 17, 5])
    xc, lc, kc = xyz.cuda(), lengths.cuda(), K.cuda()
    out = torch.empty(b, npoint, device="cuda", dtype=torch.int32)
    (o,) = stale.run(_pats(n), [out], [], lambda s: L.pcl_fps_ragged(*_lib.pts_args(xc), lc.data_ptr(), b, n, kc.data_ptr(), npoint, None, 0,
                                                                      cluster, out.data_ptr(), s))[0]
    assert np.array_equal(o, fps_ragged(xyz, npoint, lengths.tolist(), K.tolist()))
    assert (o[1, 17:] == -1).all() and (o[2, 1:] == -1).all()
    if cluster == 2:
        (o,) = stale.run(_pats(n), [out], [], lambda s: L.pcl_fps(*_lib.pts_args(xc), b, n, npoint, None, 0, out.data_ptr(), s))[0]
        assert np.array_equal(o, oracle.fps(xyz, npoint))


# ---------------------------------------------------------------- the composite step --------------------------------------

@pytest.mark.parametrize("b,n", [(2, 37), (8, 2047)])
def test_composite_step_device_and_host(stale, b, n):
    """pcl_chamfer_emd_step (Chamfer gradient: atomics) and pcl_chamfer_emd_step_host against each other and against the
    separate calls; losses[7] is unused."""
    L = stale.L
    pred, target = synth.autoencoder_batch(b, n, seed=b * n + 3, regime="noisy")
    px, tx = pred[:, :, :3].contiguous(), target[:, :, :3].contiguous()
    pc, tc = px.cuda(), tx.cuda()
    pats = _pats(b * n * 4)
    losses, gch, gem = torch.empty(8, device="cuda"), torch.empty(b, n, 3, device="cuda"), torch.empty(b, n, 3, device="cuda")
    nbytes = L.pcl_chamfer_emd_step_scratch_bytes(b, n)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    res = stale.run(pats, [losses[:7], gch, gem], [scratch], loose=(1,),
                    call=lambda s: L.pcl_chamfer_emd_step(*_lib.pts_args(pc), *_lib.pts_args(tc), b, n, EPS, ITERS, 0, losses.data_ptr(),
                                                          gch.data_ptr(), gem.data_ptr(), scratch.data_ptr(), nbytes, s))
    lz, _, ge = res[0]
    # the separate calls
    xg = pc.clone().requires_grad_()
    cl, _ = pcl.chamfer_distance(xg, tc, mode=0)
    cl.backward()
    d, a, _, ug, sums = pcl.emd_forward_raw(pc, tc, EPS, ITERS, want_epilogue=True)
    assert float(lz[0] + lz[1]) == pytest.approx(float(cl.detach()), rel=1e-6)
    assert lz[4] in float32_neighbours(epilogue_sum(npy(d))[0]) and lz[5] == np.float32(b * n)
    assert float(lz[6]) == pytest.approx(float(npy(sums)[2]), rel=1e-6)
    np.testing.assert_allclose(ge, npy(ug) / (b * n), rtol=REL, atol=1e-10)
    for _, gc, _ in res:
        np.testing.assert_allclose(gc, npy(xg.grad), rtol=REL, atol=1e-9)
    # the host-buffer entry point: pinned host outputs poisoned like device ones
    hs = L.pcl_loss_host_scratch_bytes(b, n)
    dev = torch.empty(hs, dtype=torch.uint8, device="cuda")
    ph, th = px.pin_memory(), tx.pin_memory()
    lh = torch.empty(8).pin_memory()
    gch_h, gem_h = torch.empty(b, n, 3).pin_memory(), torch.empty(b, n, 3).pin_memory()
    for k, p in enumerate(pats):
        for t in (lh, gch_h, gem_h):
            t.view(torch.int32).fill_(_i32(p))
        stale.prepare(p, k, [], [dev])
        rc = L.pcl_chamfer_emd_step_host(ph.data_ptr(), th.data_ptr(), b, n, EPS, ITERS, 0, lh.data_ptr(), gch_h.data_ptr(),
                                         gem_h.data_ptr(), dev.data_ptr(), hs, stale.stream.cuda_stream)
        assert rc == 0, L.pcl_last_error()
        stale.stream.synchronize()
        assert same_bits(lh.numpy()[:7], lz) and same_bits(gem_h.numpy(), ge)
        np.testing.assert_allclose(gch_h.numpy(), npy(xg.grad), rtol=REL, atol=1e-9)


# ---------------------------------------------------------------- the Python surface --------------------------------------

def dirty(pattern):
    """Leave the pattern in blocks of torch's caching allocator (the wrappers' torch.empty buffers) and in shared memory."""
    junk = torch.empty(64 << 20, dtype=torch.int32, device="cuda")
    junk.fill_(_i32(pattern))
    del junk
    hits = torch.zeros(smem_poison.MAX_SMID, dtype=torch.int32, device="cuda")
    smem_poison.poison(pattern, torch.cuda.current_stream(), hits)


@pytest.mark.parametrize("pattern", LARGE)
def test_python_surface_after_poison(pattern):
    p1, p2 = _rand((2, 300, 3), 1), _rand((2, 513, 3), 2)
    dirty(pattern)
    out = pcl.knn_points(p1.cuda(), p2.cuda(), K=17)
    od, oi = ko.knn_forward(p1, p2, 17)
    assert same_bits(npy(out.dists), od) and np.array_equal(npy(out.idx), oi)
    dirty(pattern)
    d, i, _ = pcl.ball_query(p1.cuda(), p2.cuda(), K=50, radius=0.3)
    od, oi = bqo.ball_query_forward(p1, p2, 50, bqo.radius2(0.3))
    assert same_bits(npy(d), od) and np.array_equal(npy(i), oi)
    dirty(pattern)
    _, idx = pcl.sample_farthest_points(p2.cuda(), lengths=torch.tensor([513, 200]), K=40)
    assert np.array_equal(npy(idx), fps_ragged(p2, 40, [513, 200]))
    dirty(pattern)
    x, y, _, _, o = chamfer_case("d3", 0, False)
    loss, _ = pcl.chamfer_distance(x.cuda(), y.cuda(), mode=0)
    assert float(loss) == pytest.approx(float(o["loss"]), rel=1e-6)
    x1, x2, (_, _, oe) = emd_inputs(3, 1000)
    dirty(pattern)
    dist, asg = pcl.emdModule()(x1, x2, EPS, ITERS)
    assert np.array_equal(npy(dist), oe["dist"]) and np.array_equal(npy(asg), oe["assignment"])
    pred, target = synth.autoencoder_batch(3, 1000, seed=5)
    losses = []
    for fn in (reference_structure(EPS, ITERS), pcl.EarthMoverDistance(EPS, ITERS)):
        fn.log = lambda k, v: None
        dirty(pattern)
        losses.append(float(fn(pred.cuda(), target.cuda())))
    assert losses[1] == pytest.approx(losses[0], rel=REL)


# ---------------------------------------------------------------- CUDA graph capture --------------------------------------

def capture_and_replay(inputs, new_inputs, outputs, call, loose=()):
    """Warm up outside the capture, capture one call on a side stream, replay it on new inputs copied into the captured
    buffers, and require the replay to equal a direct call on those inputs.  A launch or memset on the legacy stream, a
    host synchronisation or an unjoined fork inside the call makes the capture fail."""
    L = _lib.lib()
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
    before = [npy(o).copy() for o in outputs]
    for t, v in zip(inputs, new_inputs):
        t.copy_(v)
    g.replay()
    torch.cuda.synchronize()
    replay = [npy(o).copy() for o in outputs]
    with torch.cuda.stream(s):
        assert call(s.cuda_stream) == 0
    s.synchronize()
    changed = False
    for i, (a, b, c) in enumerate(zip(replay, [npy(o) for o in outputs], before)):
        if i in loose:
            np.testing.assert_allclose(a, b, rtol=REL, atol=1e-6 * max(float(np.abs(b).max(initial=0)), 1e-30))
        else:
            assert same_bits(a, b) if a.dtype == np.float32 else np.array_equal(a, b)
        changed |= not np.array_equal(a, c)
    assert changed                                         # the replay computed on the new inputs


@pytest.mark.parametrize("path,b,n", [("cluster", 3, 1000), ("team", 4, 2047), ("tickets", 4, 2047), ("auto", 1, 5000)])
def test_graph_emd_fused(emd_path, path, b, n):
    emd_path(path)
    L = _lib.lib()
    x1, x2, _ = emd_inputs(b, n)
    y1, y2 = _rand((b, n, 3), 1), _rand((b, n, 3), 2)
    dist, asg = torch.empty(b, n, device="cuda"), torch.empty(b, n, device="cuda", dtype=torch.int32)
    grad, sums = torch.empty(b, n, 3, device="cuda"), torch.empty(3, device="cuda")
    wsb = L.pcl_emd_workspace_bytes(b, n)
    ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
    capture_and_replay([x1, x2], [y1, y2], [dist, asg, grad, sums],
                       lambda s: L.pcl_emd_fwd_fused(*_lib.pts_args(x1), *_lib.pts_args(x2), b, n, EPS, ITERS, dist.data_ptr(), asg.data_ptr(),
                                                     None, 0.37, grad.data_ptr(), sums.data_ptr(), ws.data_ptr(), wsb, s))


def test_graph_emd_side_calls():
    L = _lib.lib()
    b, n, C = 3, 2047, 7
    x1, t, asg, dist = emd_side_inputs(b, n, C, 1)
    y1, u, asg2, dist2 = emd_side_inputs(b, n, C, 2)
    xc, tc, ac, dc = x1.cuda(), t.cuda(), asg.cuda(), dist.cuda()
    gd = _rand((b, n), 3).cuda()
    grad, grad2 = torch.empty(b, n, 3, device="cuda"), torch.empty(b, n, 3, device="cuda")
    hist, matched = torch.empty(C, device="cuda", dtype=torch.int64), torch.empty(b, n, device="cuda", dtype=torch.int32)
    cw, sums, gout = (_rand((C,), 4) + 0.1).cuda(), torch.empty(2, device="cuda"), torch.tensor([0.37], device="cuda")
    wsb = L.pcl_emd_workspace_bytes(b, n)
    ws = torch.empty(wsb, device="cuda", dtype=torch.uint8)
    lab = tc[:, :, 3:4]

    def call(s):
        rc = L.pcl_emd_bwd(*_lib.pts_args(xc), *_lib.pts_args(tc), b, n, ac.data_ptr(), gd.data_ptr(), grad.data_ptr(), s)
        rc = rc or L.pcl_emd_match_hist(*_lib.pts_args(lab), ac.data_ptr(), b, n, C, hist.data_ptr(), matched.data_ptr(), s)
        rc = rc or L.pcl_emd_weighted_reduce(dc.data_ptr(), matched.data_ptr(), cw.data_ptr(), b, n, C, sums.data_ptr(), ws.data_ptr(), wsb, s)
        return rc or L.pcl_emd_weighted_bwd(*_lib.pts_args(xc), *_lib.pts_args(tc), b, n, ac.data_ptr(), dc.data_ptr(), matched.data_ptr(),
                                            cw.data_ptr(), C, sums.data_ptr(), gout.data_ptr(), grad2.data_ptr(), s)
    capture_and_replay([xc, tc, ac, dc], [y1, u, asg2, dist2], [grad, hist, matched, sums, grad2], call)


def test_graph_feature_terms_and_class_filter():
    L = _lib.lib()
    b, n, C, F = 3, 1000, 33, 5
    z, z2 = _rand((b, n, C), 1, 10), _rand((b, n, C), 2, 10)
    matched = torch.randint(0, C, (b, n), generator=torch.Generator().manual_seed(3), dtype=torch.int32).cuda()
    feat, tfeat = _rand((b, n, F), 4).cuda(), _rand((b, n, F), 5).cuda()
    asg = torch.randint(0, n, (b, n), generator=torch.Generator().manual_seed(6), dtype=torch.int32).cuda()
    target = _rand((b, n, 4), 7)
    target[:, :, 3] = torch.randint(0, 5, (b, n), generator=torch.Generator().manual_seed(8)).float()
    target2 = target.clone()
    target2[:, :, 3] = (target[:, :, 3] + 1) % 5
    lc, tc, cw, gs = z.cuda(), target.cuda(), (_rand((C,), 9) + 0.1).cuda(), torch.tensor([0.7], device="cuda")
    s1, s2, hist = torch.empty(2, device="cuda"), torch.empty(2, device="cuda"), torch.empty(C, device="cuda", dtype=torch.int64)
    gl, gf = torch.empty(b, n, C, device="cuda"), torch.empty(b, n, F, device="cuda")
    out, lengths = torch.empty(b, n, 3, device="cuda"), torch.empty(b, device="cuda", dtype=torch.int64)
    wsb = L.pcl_emd_feature_workspace_bytes()
    w1, w2 = torch.empty(wsb, device="cuda", dtype=torch.uint8), torch.empty(wsb, device="cuda", dtype=torch.uint8)
    labels = (_lib.c_int64 * 2)(1, 3)

    def call(s):
        rc = L.pcl_emd_seg_ce_fwd(*_lib.pts_args(lc), matched.data_ptr(), cw.data_ptr(), b, n, C, s1.data_ptr(), hist.data_ptr(), w1.data_ptr(), wsb, s)
        rc = rc or L.pcl_emd_seg_ce_bwd(*_lib.pts_args(lc), matched.data_ptr(), cw.data_ptr(), b, n, C, gs.data_ptr(), gl.data_ptr(), s)
        rc = rc or L.pcl_emd_feat_mse_fwd(*_lib.pts_args(lc[:, :, :F]), *_lib.pts_args(tfeat), asg.data_ptr(), b, n, F, s2.data_ptr(), w2.data_ptr(), wsb, s)
        rc = rc or L.pcl_emd_feat_mse_bwd(*_lib.pts_args(lc[:, :, :F]), *_lib.pts_args(tfeat), asg.data_ptr(), b, n, F, gs.data_ptr(), gf.data_ptr(), s)
        return rc or L.pcl_class_filter(*_lib.pts_args(tc), b, n, 3, labels, 2, out.data_ptr(), lengths.data_ptr(), s)
    capture_and_replay([lc, tc], [z2, target2], [s1, hist, gl, s2, gf, out, lengths], call)


def test_graph_chamfer_pruned_and_brute_force(prune_min):
    L = _lib.lib()
    prune_min(6144)
    for name in ("pruned", "d5"):
        x, y, xl, yl, _ = chamfer_case(name, 0, True)
        b, p1, d = x.shape
        p2 = y.shape[1]
        xc, yc, xlc, ylc = x.cuda(), y.cuda(), xl.cuda(), yl.cuda()
        outs = [torch.empty(b, p1, device="cuda"), torch.empty(b, p1, device="cuda", dtype=torch.int32),
                torch.empty(b, p2, device="cuda"), torch.empty(b, p2, device="cuda", dtype=torch.int32), torch.empty(4, device="cuda")]
        ws = torch.empty(L.pcl_chamfer_workspace_bytes(b, p1, p2), device="cuda", dtype=torch.uint8)
        gx, gy, gout = torch.empty(b, p1, d, device="cuda"), torch.empty(b, p2, d, device="cuda"), torch.tensor([1.0, 0.37], device="cuda")
        fwd = chamfer_fwd_call(L, xc, yc, xlc, ylc, b, p1, p2, d, 0, outs, ws)

        def call(s):
            return fwd(s) or L.pcl_chamfer_bwd(*_lib.pts_args(xc), xlc.data_ptr(), *_lib.pts_args(yc), ylc.data_ptr(), b, p1, p2, d,
                                               outs[1].data_ptr(), outs[3].data_ptr(), gout.data_ptr(), gx.data_ptr(), gy.data_ptr(), s)
        capture_and_replay([xc, yc], [_rand((b, p1, d), 11), _rand((b, p2, d), 12)], outs + [gx, gy], call, loose=(5, 6))


def test_graph_knn_and_ball_query_split():
    L = _lib.lib()
    K = 17
    p1, p2, _, _ = knn_inputs(3, K, True)
    a, c = p1.cuda(), p2.cuda()
    n1, n2 = p1.shape[1], p2.shape[1]
    dists, idx = torch.empty(1, n1, K, device="cuda"), torch.empty(1, n1, K, device="cuda", dtype=torch.int32)
    gd = _rand((1, n1, K), 1).cuda()
    g1, g2 = torch.empty(1, n1, 3, device="cuda"), torch.empty(1, n2, 3, device="cuda")
    bd, bi = torch.empty(1, n1, 500, device="cuda"), torch.empty(1, n1, 500, device="cuda", dtype=torch.int32)
    bgd = _rand((1, n1, 500), 2).cuda()
    h1, h2 = torch.empty(1, n1, 3, device="cuda"), torch.empty(1, n2, 3, device="cuda")
    r2 = bqo.radius2(0.05)

    def call(s):
        rc = L.pcl_knn_fwd(*_lib.pts_args(a), None, *_lib.pts_args(c), None, 1, n1, n2, 3, K, 0, dists.data_ptr(), idx.data_ptr(), s)
        rc = rc or L.pcl_knn_bwd(*_lib.pts_args(a), None, *_lib.pts_args(c), None, 1, n1, n2, 3, K, idx.data_ptr(), gd.data_ptr(),
                                 g1.data_ptr(), g2.data_ptr(), s)
        rc = rc or L.pcl_ball_query_fwd(*_lib.pts_args(a), None, *_lib.pts_args(c), None, 1, n1, n2, 3, 500, r2, 0, bd.data_ptr(), bi.data_ptr(), s)
        return rc or L.pcl_ball_query_bwd(*_lib.pts_args(a), None, *_lib.pts_args(c), None, 1, n1, n2, 3, 500, bi.data_ptr(), bgd.data_ptr(),
                                          h1.data_ptr(), h2.data_ptr(), s)
    capture_and_replay([a, c], [_rand((1, n1, 3), 3), _rand((1, n2, 3), 4)], [dists, idx, g1, g2, bd, bi, h1, h2], call, loose=(2, 3, 6, 7))


def test_graph_sampling():
    """pcl_fps_ragged with a cluster of 4, pcl_fps and pointnet2's pcl_ball_query."""
    L = _lib.lib()
    b, n, npoint = 3, 16385, 64
    xyz = _rand((b, n, 3), 1).cuda()
    lc, kc = torch.tensor([n, 9000, 1]).cuda(), torch.tensor([64, 17, 5]).cuda()
    o1, o2 = torch.empty(b, npoint, device="cuda", dtype=torch.int32), torch.empty(b, npoint, device="cuda", dtype=torch.int32)
    new = _rand((b, 100, 3), 2).cuda()
    o3 = torch.empty(b, 100, 32, device="cuda", dtype=torch.int32)
    r2 = float(torch.tensor(0.2 ** 2, dtype=torch.float32))

    def call(s):
        rc = L.pcl_fps_ragged(*_lib.pts_args(xyz), lc.data_ptr(), b, n, kc.data_ptr(), npoint, None, 0, 4, o1.data_ptr(), s)
        rc = rc or L.pcl_fps(*_lib.pts_args(xyz), b, n, npoint, None, 0, o2.data_ptr(), s)
        return rc or L.pcl_ball_query(*_lib.pts_args(xyz), *_lib.pts_args(new), b, n, 100, r2, 32, o3.data_ptr(), s)
    capture_and_replay([xyz], [_rand((b, n, 3), 3)], [o1, o2, o3], call)
