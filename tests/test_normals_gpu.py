"""estimate_pointcloud_normals / estimate_pointcloud_local_coord_frames on the GPU against the float64 restatement
(tests/normals_ref.py) on the same neighbours.

Bounds (DESIGN.md, "normal estimation exactness"): the kernels compute in fp64 and round once, so
  - eigenvalues are within 2 fp32 ulps + 1e-12 * lam2 of the reference;
  - frame components are within 2^-23 absolute where the column is conditioned (lam2 / gap <= 1e6);
  - |V^T V - I| <= 2^-22 on every row;
  - the disambiguation signs equal the reference's wherever no projection is close enough to 0 to move n_pos across K/2.
Gradients: the backward reads the fp32 frames and curvatures, so each point's contribution carries a relative error of about
2^-24 * lam2 / gap (<= 1.2e-6 on the rows given an upstream gradient here, whose relative gap is >= 0.05), and the fp32
atomics add about (terms per point) * 2^-24 relative to the sum of magnitudes.  The tolerance is 1e-4 relative plus 1e-4 of
the largest reference entry, about 50 times that."""
import numpy as np
import pytest
import torch

import pointcloud_b200 as pcl
from helpers import npy, same_bits
from normals_ref import frames_ref
from pointcloud_b200 import _lib, synth
from test_stale_state_gpu import PATTERNS, Stale, capture_and_replay

pytestmark = pytest.mark.gpu

COND = 1e6


def _rand(shape, seed, scale=1.0):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed)) * scale


def table(b, n, seed=0):
    return synth.table_clouds(b, n, seed=seed)[0]


def check_forward(points, K, lengths=None, disambiguate=True):
    """Run frames_forward_raw and compare with the reference on the same idx; returns the raw result."""
    r = pcl.frames_forward_raw(points.cuda(), K, disambiguate, None if lengths is None else lengths.cuda())
    assert torch.equal(r["idx"].long(), pcl.knn_points(points.cuda(), points.cuda(), lengths, lengths, K=K).idx)
    curv, frames = npy(r["curvatures"]).astype(np.float64), npy(r["frames"]).astype(np.float64)
    p64 = points.float().double()
    rc, rf = frames_ref(p64, r["idx"].cpu(), lengths, disambiguate)
    rc, rf = rc.numpy(), rf.numpy()
    b, n, _ = points.shape
    lens = np.full(b, n) if lengths is None else np.minimum(lengths.numpy(), n)
    valid = (np.arange(n)[None, :] < lens[:, None]) & (lens[:, None] > K)
    assert not curv[~valid].any() and not frames[~valid].any()          # padded rows and small clouds: exactly 0
    c, f, rc, rf = curv[valid], frames[valid], rc[valid], rf[valid]
    # eigenvalues
    ulp = np.spacing(np.abs(rc).astype(np.float32)).astype(np.float64)
    assert (np.abs(c - rc) <= 2 * ulp + 1e-12 * np.abs(rc[:, 2:3])).all()
    # orthonormality on every row, degenerate ones included
    assert (np.abs(np.einsum("nij,nik->njk", f, f) - np.eye(3)) <= 2.0 ** -22).all()
    # conditioned columns
    l0, l1, l2 = rc[:, 0], rc[:, 1], rc[:, 2]
    tiny = np.finfo(np.float64).tiny
    ok0 = np.abs(l2) <= COND * np.maximum(l1 - l0, tiny)
    ok2 = np.abs(l2) <= COND * np.maximum(l2 - l1, tiny)
    oks = [ok0, ok0 & ok2, ok2]
    if disambiguate:
        # rows where n_pos of the reference's v0 / v2 cannot cross K / 2 under a perturbation of the projections
        nb = p64[:, :, None].expand(-1, -1, K, -1).numpy()
        idx = r["idx"].cpu().long()
        nbr = p64.gather(1, idx.reshape(b, n * K, 1).expand(-1, -1, 3)).view(b, n, K, 3).numpy()
        df = (nbr - nb)[valid]
        dn = np.linalg.norm(df, axis=2)
        for col in (0, 2):
            proj = np.einsum("nkc,nc->nk", df, rf[:, :, col])
            tol = 1e-8 * dn + 1e-300
            lo, hi = (proj > tol).sum(1), (proj > -tol).sum(1)
            oks[col] = oks[col] & ((2 * lo < K) == (2 * hi < K))
        oks[1] = oks[0] & oks[2]
        for col in range(3):
            assert (np.abs(f[:, :, col] - rf[:, :, col])[oks[col]] <= 2.0 ** -23).all(), f"column {col}"
    else:
        for col in range(3):  # eigenvector signs are arbitrary without disambiguation
            s = np.sign(np.einsum("nc,nc->n", f[:, :, col], rf[:, :, col]))[:, None]
            assert (np.abs(s * f[:, :, col] - rf[:, :, col])[oks[col]] <= 2.0 ** -23).all(), f"column {col}"
    return r


@pytest.mark.parametrize("K", [3, 16, 50, 64])
def test_table_clouds(K):
    check_forward(table(32, 2048, seed=K), K)


@pytest.mark.parametrize("disambiguate", [True, False])
@pytest.mark.parametrize("b,n,K", [(4, 1000, 8), (3, 333, 50), (2, 4099, 20)])
def test_uniform_clouds_and_p_not_a_multiple_of_32(b, n, K, disambiguate):
    x, _ = synth.uniform_clouds(b, n, seed=n + K)
    check_forward(x * torch.tensor([1.0, 0.5, 0.25]), K, disambiguate=disambiguate)


def test_one_large_cloud():
    check_forward(table(1, 65536, seed=5), 32)


def test_degenerate_neighbourhoods_are_finite_orthonormal_and_repeatable():
    g = torch.Generator().manual_seed(6)
    base = torch.rand(2, 40, 3, generator=g)
    dup = torch.cat([base, base, base[:, :20]], dim=1)                  # every point two or three times
    line = torch.linspace(0, 1, 90)[None, :, None] * torch.tensor([0.3, -0.2, 0.9])  # collinear
    same = torch.full((2, 90, 3), 0.25)                                 # an all-equal cloud
    for pts in (dup, line.expand(2, -1, -1).contiguous(), same):
        for K in (1, 2, 16):
            a = pcl.frames_forward_raw(pts.cuda(), K)
            b = pcl.frames_forward_raw(pts.cuda(), K)
            f = npy(a["frames"]).astype(np.float64)
            assert np.isfinite(f).all() and np.isfinite(npy(a["curvatures"])).all()
            assert (np.abs(np.einsum("bnij,bnik->bnjk", f, f) - np.eye(3)) <= 2.0 ** -22).all()
            assert same_bits(npy(a["frames"]), npy(b["frames"])) and same_bits(npy(a["curvatures"]), npy(b["curvatures"]))
    c = npy(pcl.frames_forward_raw(same.cuda(), 16)["curvatures"])
    assert not c.any()


def test_ragged_rows_equal_clouds_run_alone():
    K = 16
    x = table(4, 1500, seed=7)
    lengths = torch.tensor([1500, 17, 900, 1200])                       # n_b = K + 1 included
    r = pcl.frames_forward_raw(x.cuda(), K, True, lengths.cuda())
    for bi in range(4):
        m = int(lengths[bi])
        alone = pcl.frames_forward_raw(x[bi:bi + 1, :m].contiguous().cuda(), K)
        assert same_bits(npy(r["frames"])[bi, :m], npy(alone["frames"])[0])
        assert same_bits(npy(r["curvatures"])[bi, :m], npy(alone["curvatures"])[0])
        assert not npy(r["frames"])[bi, m:].any() and not npy(r["curvatures"])[bi, m:].any()
    check_forward(x, K, lengths)


def test_clouds_of_at_most_k_points_give_zero_rows_at_the_c_level():
    """The Python layer raises for n_b <= K (pytorch3d's check); the C entry point writes zero rows for those clouds."""
    L = _lib.lib()
    K = 16
    x = table(3, 300, seed=17).cuda()
    lengths = torch.tensor([300, 16, 3], device="cuda")
    idx = pcl.knn_forward_raw(x, x, lengths, lengths, K)["idx"]
    curv = torch.full((3, 300, 3), float("nan"), device="cuda")
    frames = torch.full((3, 300, 3, 3), float("nan"), device="cuda")
    assert L.pcl_frames_fwd(*_lib.pts_args(x), lengths.data_ptr(), 3, 300, K, 1, idx.data_ptr(), curv.data_ptr(), frames.data_ptr(),
                            _lib.stream_ptr()) == 0
    alone = pcl.frames_forward_raw(x[:1], K)
    assert same_bits(npy(frames)[0], npy(alone["frames"])[0]) and not npy(frames)[1:].any() and not npy(curv)[1:].any()
    gp = torch.full((3, 300, 3), float("nan"), device="cuda")
    g = torch.ones(3, 300, 3, 3, device="cuda")
    assert L.pcl_frames_bwd(*_lib.pts_args(x), lengths.data_ptr(), 3, 300, K, idx.data_ptr(), curv.data_ptr(), frames.data_ptr(),
                            None, g.data_ptr(), gp.data_ptr(), _lib.stream_ptr()) == 0
    assert not npy(gp)[1:].any()


def test_input_forms_equal_the_fp32_copy():
    K = 16
    x6 = _rand((3, 1024, 6), 8).cuda()
    views = [x6[..., :3], x6[..., :3].half(), x6[..., :3].bfloat16()]
    for v in views:
        a = pcl.frames_forward_raw(v, K)
        b = pcl.frames_forward_raw(v.float().contiguous(), K)
        for key in ("curvatures", "frames"):
            assert same_bits(npy(a[key]), npy(b[key]))
        assert torch.equal(a["idx"], b["idx"])
    check_forward(x6[..., :3].half().cpu(), K)


def test_two_runs_are_bit_identical():
    x = table(8, 2048, seed=9).cuda()
    a, b = pcl.frames_forward_raw(x, 50), pcl.frames_forward_raw(x, 50)
    assert same_bits(npy(a["frames"]), npy(b["frames"])) and same_bits(npy(a["curvatures"]), npy(b["curvatures"]))


# ---------------------------------------------------------------- gradients ------------------------------------------------

def _grad_case(seed, b=4, n=600, K=16):
    x = _rand((b, n, 3), seed) * torch.tensor([1.0, 0.6, 0.3])
    lengths = torch.tensor([n, n - 111, n, 300][:b])
    return x, lengths, K


def _upstream_mask(x, lengths, K, r):
    """Rows whose relative spectral gap is >= 0.05 and whose signs agree with the reference: the only rows given an
    upstream gradient (the others get 0, which contributes exactly 0 on both sides)."""
    rc, rf = frames_ref(x.double(), r["idx"].cpu(), lengths)
    lam = rc.numpy()
    gap = np.minimum(lam[..., 1] - lam[..., 0], lam[..., 2] - lam[..., 1]) >= 0.05 * lam[..., 2]
    agree = (np.einsum("bnic,bnic->bnc", npy(r["frames"]).astype(np.float64), rf.numpy()) > 0).all(-1)
    return torch.from_numpy(gap & agree)


@pytest.mark.parametrize("through", ["curvatures", "frames", "normals", "middle", "all"])
def test_gradients_against_autograd_of_the_reference(through):
    x, lengths, K = _grad_case(10)
    r = pcl.frames_forward_raw(x.cuda(), K, True, lengths.cuda())
    mask = _upstream_mask(x, lengths, K, r)
    g = torch.Generator().manual_seed(11)
    wc = torch.randn(*x.shape, generator=g, dtype=torch.float64) * mask[..., None]
    wf = torch.randn(*x.shape, 3, generator=g, dtype=torch.float64) * mask[..., None, None]
    if through == "middle":
        wf[..., 0] = 0; wf[..., 2] = 0                                   # only the cross-product column

    def loss(c, f, nrm):
        if through == "curvatures":
            return (c * wc.to(c)).sum()
        if through in ("frames", "middle"):
            return (f * wf.to(f)).sum()
        if through == "normals":
            return (nrm * wf[..., 0].to(nrm)).sum()
        return (c * wc.to(c)).sum() + (f * wf.to(f)).sum() + (nrm * wf[..., 1].to(nrm)).sum()

    xg = x.cuda().requires_grad_()
    c, f = pcl.estimate_pointcloud_local_coord_frames(xg, K, lengths=lengths.cuda())
    nrm = pcl.estimate_pointcloud_normals(xg, K, lengths=lengths.cuda())
    loss(c, f, nrm).backward()
    xr = x.double().requires_grad_()
    rc, rf = frames_ref(xr, r["idx"].cpu(), lengths)
    loss(rc, rf, rf[..., 0]).backward()
    want = xr.grad.numpy()
    got = npy(xg.grad).astype(np.float64)
    assert np.abs(want).max() > 0
    np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * np.abs(want).max())
    assert not got[1, int(lengths[1]):].any()


def test_gradient_dtype_and_device_follow_the_input():
    x, _, K = _grad_case(12, b=2, n=256)
    for dt in (torch.float16, torch.bfloat16):
        xg = x.to(dt).cuda().requires_grad_()
        pcl.estimate_pointcloud_normals(xg, K).sum().backward()
        assert xg.grad.dtype == dt and xg.grad.is_cuda
    xg = x.clone().requires_grad_()                                     # a CPU input: gradient back on the CPU
    pcl.estimate_pointcloud_local_coord_frames(xg, K)[0].sum().backward()
    assert xg.grad.device.type == "cpu"


def surface(b, seed):
    """(b, 1024, 3) jittered height fields sampled on a 64 x 16 grid over the unit square: every 16-neighbourhood is
    elongated along x and thin along the normal, so its three eigenvalues are well apart and the gradient through the
    eigenvectors is well conditioned."""
    g = torch.Generator().manual_seed(seed)
    u, v = torch.meshgrid(torch.linspace(0, 1, 64), torch.linspace(0, 1, 16), indexing="ij")
    uv = torch.stack([u, v], -1).reshape(1, -1, 2) + 0.002 * torch.randn(b, 1024, 2, generator=g)
    ph = torch.rand(b, 1, 2, generator=g) * 6
    h = 0.1 * torch.sin(3 * uv[..., 0] + ph[..., 0]) * torch.cos(2 * uv[..., 1] + ph[..., 1])
    return torch.cat([uv, h[..., None]], -1).contiguous()


def test_chamfer_with_estimated_normals_end_to_end():
    from chamfer_surface_ref import chamfer_reference, neighbours
    K = 16
    pred, gt = surface(4, 13), surface(4, 14)
    pg = pred.cuda().requires_grad_()
    nx = pcl.estimate_pointcloud_normals(pg, K)
    ny = pcl.estimate_pointcloud_normals(gt.cuda(), K)
    loss, loss_n = pcl.chamfer_distance(pg, gt.cuda(), x_normals=nx, y_normals=ny)
    (loss + loss_n).backward()
    # float64 restatement of the whole composition on the same neighbours
    ix, iy, _ = neighbours(pred, gt)
    kx = pcl.knn_points(pred.cuda(), pred.cuda(), K=K).idx.cpu()
    ky = pcl.knn_points(gt.cuda(), gt.cuda(), K=K).idx.cpu()
    pr = pred.double().requires_grad_()
    rnx = frames_ref(pr, kx)[1][..., 0]
    rny = frames_ref(gt.double(), ky)[1][..., 0]
    rl, rln = chamfer_reference(pr, gt.double(), ix, iy, x_normals=rnx, y_normals=rny)
    assert abs(float(loss) - float(rl)) <= 1e-5 * abs(float(rl))
    assert abs(float(loss_n) - float(rln)) <= 1e-5 * abs(float(rln))
    (rl + rln).backward()
    want = pr.grad.numpy()
    np.testing.assert_allclose(npy(pg.grad), want, rtol=1e-3, atol=1e-3 * np.abs(want).max())
    # the normal path contributes: the gradient differs from the distance-only one
    pd = pred.cuda().requires_grad_()
    pcl.chamfer_distance(pd, gt.cuda())[0].backward()
    assert not torch.allclose(pd.grad, pg.grad)


# ---------------------------------------------------------------- stale state and graphs --------------------------------

def test_stale_outputs_and_shared_memory():
    st = Stale()
    L = st.L
    K = 50
    x = table(3, 2000, seed=14).cuda()
    lengths = torch.tensor([2000, 51, 777]).cuda()
    b, n, _ = x.shape
    r = pcl.frames_forward_raw(x, K, True, lengths)
    idx = r["idx"]
    curv, frames = torch.empty(b, n, 3, device="cuda"), torch.empty(b, n, 3, 3, device="cuda")
    res = st.run(PATTERNS, [curv, frames], [], lambda s: L.pcl_frames_fwd(*_lib.pts_args(x), lengths.data_ptr(), b, n, K, 1,
                                                                          idx.data_ptr(), curv.data_ptr(), frames.data_ptr(), s),
                 check=lambda o: same_bits(o[0], npy(r["curvatures"])) and same_bits(o[1], npy(r["frames"])))
    gc, gf = torch.randn(b, n, 3, device="cuda"), torch.randn(b, n, 3, 3, device="cuda")
    gp = torch.empty(b, n, 3, device="cuda")
    res = st.run(PATTERNS, [gp], [], loose=(0,),
                 call=lambda s: L.pcl_frames_bwd(*_lib.pts_args(x), lengths.data_ptr(), b, n, K, idx.data_ptr(), r["curvatures"].data_ptr(),
                                                 r["frames"].data_ptr(), gc.data_ptr(), gf.data_ptr(), gp.data_ptr(), s))
    for o in res[1:]:
        np.testing.assert_allclose(o[0], res[0][0], rtol=1e-5, atol=1e-5 * np.abs(res[0][0]).max())
    assert not res[0][0][1, 51:].any() and not res[0][0][2, 777:].any()


def test_graph_capture_of_both_entry_points():
    L = _lib.lib()
    K = 16
    b, n = 4, 1000
    x = table(b, n, seed=15).cuda()
    idx = torch.empty(b, n, K, device="cuda", dtype=torch.int32)
    dists = torch.empty(b, n, K, device="cuda")
    curv, frames = torch.empty(b, n, 3, device="cuda"), torch.empty(b, n, 3, 3, device="cuda")
    gc, gf = torch.randn(b, n, 3, device="cuda"), torch.randn(b, n, 3, 3, device="cuda")
    gp = torch.empty(b, n, 3, device="cuda")

    def call(s):
        rc = L.pcl_knn_fwd(*_lib.pts_args(x), None, *_lib.pts_args(x), None, b, n, n, 3, K, 0, dists.data_ptr(), idx.data_ptr(), s)
        rc = rc or L.pcl_frames_fwd(*_lib.pts_args(x), None, b, n, K, 1, idx.data_ptr(), curv.data_ptr(), frames.data_ptr(), s)
        return rc or L.pcl_frames_bwd(*_lib.pts_args(x), None, b, n, K, idx.data_ptr(), curv.data_ptr(), frames.data_ptr(),
                                      gc.data_ptr(), gf.data_ptr(), gp.data_ptr(), s)
    capture_and_replay([x], [table(b, n, seed=16).cuda()], [idx, curv, frames, gp], call, loose=(3,))
