"""rasterize_points and the point compositors without a GPU: the torch restatement (tests/raster_ref.py) against an
independent numpy brute force and hand-computed cases, the compositor restatements against a direct loop, and the argument
checks of the public functions and of the C ABI."""
import ctypes

import numpy as np
import pytest
import torch

import pointcloud_b200 as pcl
from pointcloud_b200 import _lib
from raster_ref import composite_ref, pixel_centres, rasterize_ref

_PCL_E_SHAPE, _PCL_E_ARG, _PCL_E_WORKSPACE = -1, -2, -4
F32 = np.float32


# ---------------------------------------------------------------- pixel centres --------------------------------------------

@pytest.mark.parametrize("S", [1, 2, 5, 64, 255])
def test_square_centres(S):
    xs, ys = pixel_centres(S, S)
    # -1 + (2i + 1) / S with each operation rounded in fp32; column 0 (and row 0) is the largest index i
    want = np.array([F32(-1) + F32(2 * i + 1) / F32(S) for i in range(S)], F32)[::-1]
    assert np.array_equal(xs.numpy(), want) and np.array_equal(ys.numpy(), want)


def test_non_square_centres_pinned_by_hand():
    xs, ys = pixel_centres(2, 4)
    assert xs.tolist() == [1.5, 0.5, -0.5, -1.5] and ys.tolist() == [0.5, -0.5]
    xs, ys = pixel_centres(4, 2)                                     # the shorter side spans [-1, 1]
    assert xs.tolist() == [0.5, -0.5] and ys.tolist() == [1.5, 0.5, -0.5, -1.5]


# ---------------------------------------------------------------- numpy brute force ----------------------------------------

def brute(points, lengths, H, W, radius, K):
    """A dense (pixel, point) d2 matrix in float32 numpy and np.lexsort on (z, i)."""
    B, P, _ = points.shape
    ln = np.clip(lengths, 0, P) if lengths is not None else np.full(B, P)
    S1, S2 = W, H
    rx = np.float32(S1 * 2) / np.float32(S2) if S1 > S2 else np.float32(2)
    ry = np.float32(S2 * 2) / np.float32(S1) if S2 > S1 else np.float32(2)
    ix = (W - 1 - np.arange(W)).astype(F32)
    iy = (H - 1 - np.arange(H)).astype(F32)
    xs = -(rx / 2) + (rx * ix + rx / 2) / np.float32(W)
    ys = -(ry / 2) + (ry * iy + ry / 2) / np.float32(H)
    idx = -np.ones((B, H, W, K), np.int32)
    zb = -np.ones((B, H, W, K), F32)
    ds = -np.ones((B, H, W, K), F32)
    off = 0
    for b in range(B):
        n = int(ln[b])
        p = points[b, :n].astype(F32)
        r = (radius[b, :n] if isinstance(radius, np.ndarray) else np.full(n, radius)).astype(F32)
        ok = np.isfinite(p).all(1) & np.isfinite(r) & (p[:, 2] >= 0)
        dx = xs[None, :, None] - p[None, None, :, 0]
        dy = ys[:, None, None] - p[None, None, :, 1]
        with np.errstate(invalid="ignore", over="ignore"):
            d2 = (dx * dx).astype(F32) + (dy * dy).astype(F32)
            hit = ok & (d2 <= (r * r).astype(F32))
        for row in range(H):
            for col in range(W):
                js = np.nonzero(hit[row, col])[0]
                zs = p[js, 2] + F32(0)
                o = js[np.lexsort((js, zs))][:K]
                idx[b, row, col, :len(o)] = o + off
                zb[b, row, col, :len(o)] = p[o, 2]
                ds[b, row, col, :len(o)] = d2[row, col, o]
        off += n
    return idx, zb, ds


def same(a, b):
    return np.array_equal(np.asarray(a).view(np.int32), np.asarray(b).view(np.int32))


@pytest.mark.parametrize("seed,B,P,H,W,K,per_point", [(0, 3, 40, 9, 9, 4, False), (1, 2, 60, 6, 11, 8, True),
                                                     (2, 4, 25, 13, 7, 1, False), (3, 2, 80, 8, 8, 20, True)])
def test_restatement_matches_a_numpy_brute_force(seed, B, P, H, W, K, per_point):
    g = torch.Generator().manual_seed(seed)
    pts = torch.rand(B, P, 3, generator=g) * 2.4 - 1.2
    pts[..., 2] = torch.rand(B, P, generator=g) * 2 - 0.2                  # some z < 0
    pts[..., 2][torch.rand(B, P, generator=g) < 0.3] = 0.5                 # ties in z
    lengths = torch.randint(0, P + 1, (B,), generator=g)
    lengths[0] = P
    radius = torch.rand(B, P, generator=g) * 0.4 if per_point else 0.3
    got = rasterize_ref(pts, lengths, (H, W), radius, K)
    want = brute(pts.numpy(), lengths.numpy(), H, W, radius.numpy() if per_point else radius, K)
    for a, b in zip(got, want):
        assert same(a.numpy(), b)
    assert (got[0] >= 0).sum() > 10


def one(points, radius=0.5, H=4, W=4, K=4, lengths=None):
    return rasterize_ref(torch.tensor([points], dtype=torch.float32), lengths, (H, W), radius, K)


def test_a_point_exactly_on_the_circle_hits():
    # square 4: column 1 is x = 0.25, row 1 is y = 0.25; the point at x = -0.25 is 0.5 away, radius 0.5
    idx, _, d = one([[-0.25, 0.25, 1.0]], radius=0.5)
    assert idx[0, 1, 1, 0] == 0 and d[0, 1, 1, 0] == 0.25
    idx, _, _ = one([[-0.25, 0.25, 1.0]], radius=float(np.nextafter(F32(0.5), F32(0))))
    assert idx[0, 1, 1, 0] == -1


def test_minus_zero_and_plus_zero_tie_so_the_index_decides():
    idx, z, _ = one([[0.0, 0.0, 0.0], [0.0, 0.0, -0.0]], radius=2.0, K=2)
    assert idx[0, 0, 0].tolist() == [0, 1]
    assert z[0, 0, 0, 1].item() == 0 and np.signbit(z[0, 0, 0, 1].item())   # zbuf keeps the stored -0.0
    idx, _, _ = one([[0.0, 0.0, -0.0], [0.0, 0.0, 0.0]], radius=2.0, K=2)
    assert idx[0, 0, 0].tolist() == [0, 1]


def test_negative_z_never_hits_and_a_negative_radius_acts_as_its_magnitude():
    idx, _, _ = one([[0.0, 0.0, -1e-30]], radius=2.0)
    assert (idx == -1).all()
    a = one([[0.1, -0.2, 0.5]], radius=-0.6)
    b = one([[0.1, -0.2, 0.5]], radius=0.6)
    assert all(same(x.numpy(), y.numpy()) for x, y in zip(a, b)) and (a[0] >= 0).any()


@pytest.mark.parametrize("bad", [[float("nan"), 0, 1], [0, float("inf"), 1], [0, 0, float("nan")], [0, 0, float("inf")]])
def test_non_finite_coordinates_never_hit(bad):
    idx, _, _ = one([bad, [0.0, 0.0, 2.0]], radius=10.0, K=2)
    assert (idx[..., 0] == 1).all() and (idx[..., 1] == -1).all()


def test_nan_radius_never_hits():
    r = torch.tensor([[float("nan"), 10.0]])
    idx, _, _ = rasterize_ref(torch.tensor([[[0.0, 0.0, 1.0], [0.0, 0.0, 2.0]]]), None, 4, r, 2)
    assert (idx[..., 0] == 1).all() and (idx[..., 1] == -1).all()


def test_empty_cloud_and_packed_offsets():
    pts = torch.tensor([[[0.0, 0.0, 1.0]], [[0.0, 0.0, 1.0]], [[0.0, 0.0, 1.0]]])
    idx, z, d = rasterize_ref(pts, torch.tensor([1, 0, 1]), 2, 5.0, 2)
    assert (idx[0, ..., 0] == 0).all() and (idx[1] == -1).all() and (z[1] == -1).all() and (d[1] == -1).all()
    assert (idx[2, ..., 0] == 1).all()                                         # offset_2 = 1 + 0
    idx, _, _ = rasterize_ref(pts, None, 2, 5.0, 1)
    assert idx[:, 0, 0, 0].tolist() == [0, 1, 2]                               # b * P without lengths


def test_k_larger_than_the_hits():
    idx, z, d = one([[0.0, 0.0, 3.0], [0.0, 0.0, 1.0], [0.0, 0.0, 2.0]], radius=5.0, K=7)
    assert idx[0, 0, 0].tolist() == [1, 2, 0, -1, -1, -1, -1] and z[0, 0, 0, 3:].eq(-1).all() and d[0, 0, 0, 3:].eq(-1).all()


# ---------------------------------------------------------------- compositors -----------------------------------------------

def loop_composite(mode, idx, a, F):
    N, K, H, W = idx.shape
    C, P = F.shape
    out = np.zeros((N, C, H, W), F32)
    for n in range(N):
        for h in range(H):
            for w in range(W):
                s = F32(0)
                for k in range(K):
                    if 0 <= idx[n, k, h, w] < P:
                        s = F32(s + a[n, k, h, w])
                wn = max(s, F32(1e-4))
                T = F32(1)
                for k in range(K):
                    j, ak = idx[n, k, h, w], a[n, k, h, w]
                    if 0 <= j < P:
                        for c in range(C):
                            if mode == "weighted":
                                t = F32(ak * F[c, j])
                            elif mode == "norm":
                                t = F32(F32(ak * F[c, j]) / wn)
                            else:
                                t = F32(F32(T * ak) * F[c, j])
                            out[n, c, h, w] = F32(out[n, c, h, w] + t)
                    T = F32(T * F32(1 - ak))
    return out


@pytest.mark.parametrize("mode", ["alpha", "norm", "weighted"])
def test_compositor_restatements_match_a_direct_loop(mode):
    g = torch.Generator().manual_seed(5)
    N, K, H, W, C, P = 2, 5, 3, 4, 3, 17
    idx = torch.randint(-3, P + 3, (N, K, H, W), generator=g)                    # -1s and out-of-range entries
    a = torch.rand(N, K, H, W, generator=g)
    a[0, :, 0, 0] = 1e-6                                                        # sum below 1e-4
    a[1, 1] = 1.0
    a[1, 2] = 0.0
    F = torch.randn(C, P, generator=g)
    got = composite_ref(mode, idx, a, F).numpy()
    want = loop_composite(mode, idx.numpy(), a.numpy(), F.numpy())
    assert same(got, want)


# ---------------------------------------------------------------- argument checks ------------------------------------------

def test_argument_errors_raise_before_any_kernel():
    p = torch.rand(2, 10, 3)
    with pytest.raises(ValueError):
        pcl.rasterize_points(torch.rand(2, 10, 2))
    with pytest.raises(ValueError):
        pcl.rasterize_points(p, points_per_pixel=151)
    with pytest.raises(ValueError):
        pcl.rasterize_points(p, radius=torch.rand(2, 9))
    with pytest.raises(ValueError):
        pcl.rasterize_points(p, bin_size=10)
    with pytest.raises(ValueError):
        pcl.rasterize_points(p, image_size=(0, 4))
    with pytest.raises(ValueError):
        pcl.rasterize_points(p, lengths=torch.tensor([1, 2, 3]))
    with pytest.raises(ValueError):
        pcl.alpha_composite(torch.zeros(1, 2, 3, 4, dtype=torch.int64), torch.rand(1, 2, 3, 3), torch.rand(3, 5))
    with pytest.raises(ValueError):
        pcl.weighted_sum(torch.zeros(1, 2, 3, 4), torch.rand(1, 2, 3, 4), torch.rand(3, 5))
    with pytest.raises(ValueError):
        pcl.norm_weighted_sum(torch.zeros(1, 2, 3, 4, dtype=torch.int32), torch.rand(1, 2, 3, 4), torch.rand(3, 5, 1))


def test_c_abi_limits():
    L = _lib.lib()
    assert L.pcl_raster_max_k() == 150
    assert L.pcl_rasterize_points_workspace_bytes(2, 100, 64, 64, 0, 0) == 0
    assert L.pcl_rasterize_points_workspace_bytes(2, 100, 64, 64, 32, 0) == 2 * 4 * (1 + 100) * 4      # cap = min(P, 10000)
    assert L.pcl_rasterize_points_workspace_bytes(2, 100, 64, 64, 32, 7) == 2 * 4 * (1 + 7) * 4
    buf = (ctypes.c_float * 64)()
    ptr = ctypes.addressof(buf)

    def fwd(B=1, P=4, H=4, W=4, K=2, bs=0, ws=0):
        return L.pcl_rasterize_points_fwd(ptr, 0, 12, 3, None, None, 0.1, B, P, H, W, K, bs, 0, ptr, ptr, ptr, ptr, ws, None)
    assert fwd(K=0) == _PCL_E_SHAPE and fwd(K=151) == _PCL_E_SHAPE
    assert fwd(H=0) == _PCL_E_SHAPE and fwd(W=16385) == _PCL_E_SHAPE
    assert fwd(B=1 << 16, P=1 << 15) == _PCL_E_SHAPE                              # B * P >= 2^31
    assert fwd(bs=8) == _PCL_E_ARG
    assert fwd(bs=16, ws=4) == _PCL_E_WORKSPACE
    assert b"workspace" in L.pcl_last_error()
    st = (ctypes.c_int64 * 4)(1, 1, 1, 1)
    assert L.pcl_composite_fwd(7, ptr, 0, st, ptr, st, ptr, st, 1, 1, 1, 1, 1, 1, ptr, None) == _PCL_E_ARG
    assert L.pcl_composite_fwd(0, ptr, 2, st, ptr, st, ptr, st, 1, 1, 1, 1, 1, 1, ptr, None) == _PCL_E_ARG
