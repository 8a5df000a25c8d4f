"""Proof check of the auction's skip rules at every coordinate scale (DESIGN.md "Why skipping is exact").

The Bid scan of the auction EMD evaluates a target exactly only when an fp32 filter cannot prove that the target's value
v = bid_value_exact(s, price) = fl32((3 - sqrt_rn(s)) - price) lies below T, a proven lower bound of the bidder's final
second-best value.  Three rules decide what is skipped (pcl_emd_core.cuh):
  candidate (scan_tile, the warp-per-bidder scans): u = filter_u(c, T_m) = RU(c - T_m), skip when fma(u, u, -s) < 0;
  tile      (tile_skippable): u from the tile's maximum of c, s replaced by 0.999999 x the squared distance to the tile's
            box; skip when u < 0 or fma(u, u, -d2) < 0;
  threshold T_m = filter_threshold(T) = RD(T - FILTER_MARGIN), with T the second largest exact value of up to four seed
            objects (seed_threshold) and raised to the running second best after every exact evaluation (top2_exact);
where c = RU(3 - price) and s = fma(dz,dz, fma(dx,dx, dy*dy)).  Each rule is restated here operation by operation with the
kernel's rounding (exactly: fp32 results are rounded from error-free fp64 pairs) and checked for the one property the proof
needs: a skipped target has v < T.  Inputs: coordinate scales 2^-10 .. 10^4, offsets of +-10^3 and -2.5*10^4 with unit
spread, prices up to the size of the value range, thresholds a few ulp from v on both sides, exact ties, lattice ties.

Rounding both subtractions to nearest instead (NEAREST below, the kernel's rule before directed rounding) makes the error of
T_m and u grow with |T|, |c| and sqrt(s); once it outgrows the 2e-6 margin, candidates whose value reaches T are skipped.
Restated with that rule, these checks fail at every scale >= 16 (the candidate check from 16, the tile and scan checks from
100; test_nearest_rounding_is_unsound_beyond_the_unit_cube keeps that demonstration), and test_restated_rule_is_the_kernels
fails on a kernel that rounds to nearest.
"""
import os
import re
import zlib
from fractions import Fraction

import numpy as np
import pytest

F, D = np.float32, np.float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pointcloud_b200", "csrc")
MARGIN = F(2e-6)                       # FILTER_MARGIN
SHRINK = F(0.999999)                   # tile_skippable's relative shrink of the box distance
KERNEL = ("down", "up")                # rounding of (T - margin, c - T_m): filter_threshold, filter_u
NEAREST = ("nearest", "nearest")


# ---- exact fp32 rounding from fp64 -------------------------------------------------------------------------------
def two_sum(a, b):
    """a + b == s + e exactly, s = fl64(a + b) (Knuth)."""
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def round32(s, e, mode):
    """The exact real s + e (an fp64 pair with |e| <= ulp(s)/2) rounded to fp32: "down", "up" or "nearest" (ties to even)."""
    f = s.astype(F)
    d = f.astype(D) - s                                   # exact (Sterbenz): f = RN32(s) is within half an ulp of s
    above, below = d > e, d < e                           # f > s + e, f < s + e
    lo = np.where(above, np.nextafter(f, F(-np.inf)), f)
    hi = np.where(below, np.nextafter(f, F(np.inf)), f)
    if mode == "down":
        return lo
    if mode == "up":
        return hi
    mid = (lo.astype(D) + hi.astype(D)) * 0.5             # exact: the midpoint of two fp32 neighbours
    dm = s - mid                                          # exact (Sterbenz); compare s + e with mid
    even = np.where(lo.view(np.int32) & 1, hi, lo)
    near = np.where(dm > -e, hi, np.where(dm < -e, lo, even))
    return np.where(lo == hi, lo, near)


def sub(a, b, mode="nearest"):
    """fp32 a - b rounded as __fsub_rn / __fsub_rd / __fsub_ru."""
    a, b = np.asarray(a, F), np.asarray(b, F)
    return round32(*two_sum(a.astype(D), -b.astype(D)), mode)


def mul(a, b):
    """__fmul_rn: the fp64 product of two fp32 numbers is exact, so one rounding."""
    return (np.asarray(a, F).astype(D) * np.asarray(b, F).astype(D)).astype(F)


def fma(a, b, c):
    """__fmaf_rn"""
    p = np.asarray(a, F).astype(D) * np.asarray(b, F).astype(D)
    return round32(*two_sum(p, np.asarray(c, F).astype(D)), "nearest")


def sq3(dx, dy, dz):
    """sq3_ref: fma(dz,dz, fma(dx,dx, dy*dy))"""
    return fma(dz, dz, fma(dx, dx, mul(dy, dy)))


def sqdist(t, a):
    """(..., 3) target and bidder -> the kernel's squared distance (target minus bidder per axis)"""
    return sq3(sub(t[..., 0], a[..., 0]), sub(t[..., 1], a[..., 1]), sub(t[..., 2], a[..., 2]))


def value(s, p):
    """bid_value_exact: fl32((3.0 - (double)sqrt_rn(s)) - (double)p), each fp64 operation rounded to nearest."""
    r = np.sqrt(np.asarray(s, F))                          # IEEE fp32 square root
    return ((3.0 - r.astype(D)) - np.asarray(p, F).astype(D)).astype(F)


def c_of(p):
    """c = RU(3 - price), the target's upper bound of the price term"""
    return sub(F(3), p, "up")


# ---- the three rules ---------------------------------------------------------------------------------------------
def threshold(T, rule):
    return sub(T, MARGIN, rule[0])


def candidate_skipped(c, tm, s, rule):
    u = sub(c, tm, rule[1]).astype(D)
    return u * u < np.asarray(s, F).astype(D)              # the sign of fma(u, u, -s) (exact; -0 counts as "not skipped")


def tile_skipped(lo, hi, a, cmax, tm, rule):
    """tile_skippable; lo / hi (..., 3) box corners, a (..., 3) bidder, cmax the tile maximum of c"""
    dd = [np.maximum(np.maximum(sub(lo[..., i], a[..., i]), sub(a[..., i], hi[..., i])), F(0)) for i in range(3)]
    d2 = mul(sq3(*dd), SHRINK)
    u = sub(cmax, tm, rule[1])
    return (u < 0) | (u.astype(D) * u.astype(D) < d2.astype(D))


# ---- inputs ------------------------------------------------------------------------------------------------------
SCALES = [2.0 ** -10, 2.0 ** -4, 1.0, 2.0, 4.0, 8.0, 16.0, 100.0, 1000.0, 1e4]
OFFSETS = [1e3, -1e3, -2.5e4]
CASES = [(f"scale {s:g}", s, 0.0) for s in SCALES] + [(f"offset {o:g}", 1.0, o) for o in OFFSETS]


def points(g, n, scale, offset):
    return (g.random((n, 3)) * scale + offset).astype(F)


def steps(x, k):
    """x moved by k fp32 ulps (k an integer array, |k| <= 8)"""
    x = x.copy()
    for i in range(8):
        x = np.where(k > i, np.nextafter(x, F(np.inf)), x)
        x = np.where(k < -i, np.nextafter(x, F(-np.inf)), x)
    return x


def candidates(scale, offset, n, seed):
    """(s, p, c, v, T) for n (bidder, target) pairs: prices up to twice the largest distance, thresholds a few ulp from v
    (ties included), around v within a few margins, and far above v (the common case of a scan)."""
    g = np.random.default_rng(seed)
    s = sqdist(points(g, n, scale, offset), points(g, n, scale, offset))
    span = 2.0 * np.sqrt(3.0) * scale
    p = np.where(g.random(n) < 0.2, 0.0, g.random(n) * span).astype(F)
    v = value(s, p)
    kind = g.integers(0, 4, n)
    T = np.where(kind == 0, steps(v, g.integers(-4, 5, n)), v)                                   # ulp neighbours
    T = np.where(kind == 1, v, T)                                                                # exact ties
    T = np.where(kind == 2, (v.astype(D) + (g.random(n) * 16 - 8) * float(MARGIN)).astype(F), T)  # a few margins
    T = np.where(kind == 3, (v.astype(D) + g.random(n) * span).astype(F), T)                    # far above v
    return s, p, c_of(p), v, T


@pytest.mark.parametrize("name,scale,offset", CASES)
def test_candidate_filter_skips_only_values_below_the_threshold(name, scale, offset):
    s, p, c, v, T = candidates(scale, offset, 400_000, seed=zlib.crc32(name.encode()))
    skipped = candidate_skipped(c, threshold(T, KERNEL), s, KERNEL)
    bad = skipped & (v >= T)
    assert not bad.any(), (name, int(bad.sum()), s[bad][:3], p[bad][:3], T[bad][:3])
    assert skipped.mean() > 0.1, name                     # not vacuous: thresholds far above v are skipped


def tiles(scale, offset, seed, ntiles=3000):
    """ntiles tiles of 32 targets with prices, a bidder per tile, and the tile's exact maximum value for that bidder.
    Tile shapes: a compact random cluster, 32 copies of one point (box == point), and a coarse lattice (tied distances)."""
    g = np.random.default_rng(seed)
    kind = g.integers(0, 3, ntiles)
    centre = points(g, ntiles, scale, offset)
    spread = np.where(kind == 0, 0.05, 0.0)[:, None, None] * scale
    t = (centre[:, None, :].astype(D) + (g.random((ntiles, 32, 3)) - 0.5) * spread).astype(F)
    lat = (centre[:, None, :].astype(D) + g.integers(0, 3, (ntiles, 32, 3)) * (0.01 * scale)).astype(F)
    t = np.where((kind == 2)[:, None, None], lat, t)
    a = (centre.astype(D) + (g.random((ntiles, 3)) - 0.5) * (0.3 * scale)).astype(F)
    span = 2.0 * np.sqrt(3.0) * scale
    p = np.where(g.random((ntiles, 32)) < 0.2, 0.0, g.random((ntiles, 32)) * span).astype(F)
    same = (g.random(ntiles) < 0.5)[:, None]               # half the tiles: one price for all targets
    p = np.where(same, p[:, :1], p)
    s = sqdist(t, a[:, None, :])
    vmax = value(s, p).max(1)
    return t, a, p, vmax


@pytest.mark.parametrize("name,scale,offset", CASES)
def test_tile_test_skips_only_tiles_below_the_threshold(name, scale, offset):
    g = np.random.default_rng(zlib.crc32(name.encode()) + 1)
    t, a, p, vmax = tiles(scale, offset, seed=zlib.crc32(name.encode()))
    n = len(vmax)
    T = np.where(g.random(n) < 0.5, steps(vmax, g.integers(-4, 5, n)),
                 (vmax.astype(D) + (g.random(n) * 16 - 8) * float(MARGIN)).astype(F))
    cmax = c_of(p).max(1)
    skipped = tile_skipped(t.min(1), t.max(1), a, cmax, threshold(T, KERNEL), KERNEL)
    bad = skipped & (vmax >= T)
    assert not bad.any(), (name, int(bad.sum()))


def scan(t, a, p, seeds, rule):
    """A bidder's Bid scan as the kernel runs it, vectorised over bidders: threshold from the seeds (seed_threshold), then the
    targets tile by tile (tile_skippable), candidate by candidate (scan_tile), raising the threshold after every exact
    evaluation (top2_exact).  t (N,3) targets, a (M,3) bidders, p (N,) prices, seeds (M,4) distinct target indices.
    Returns best, better, argmax (lowest index among equal maxima) and whether a skipped target had v >= its T."""
    M, N = len(a), len(t)
    c = c_of(p)
    s = sqdist(t[None, :, :], a[:, None, :])               # (M, N)
    v = value(s, p[None, :])
    sv = np.take_along_axis(v, seeds, 1)
    T = np.sort(sv, 1)[:, -2]                              # second largest of the four seed values
    tm = threshold(T, rule)
    best = np.full(M, -1e9, F)
    better = np.full(M, -1e9, F)
    bi = np.full(M, -1)
    unsound = np.zeros(M, bool)
    for k0 in range(0, N, 32):
        box = t[k0:k0 + 32]
        skip_tile = tile_skipped(box.min(0)[None], box.max(0)[None], a, c[k0:k0 + 32].max()[None], tm, rule)
        for k in range(k0, min(k0 + 32, N)):
            Tk = np.maximum(T, better)
            skip = skip_tile | candidate_skipped(c[k], tm, s[:, k], rule)
            unsound |= skip & (v[:, k] >= Tk)
            vk = v[:, k]
            up1 = ~skip & (vk > best)                      # ascending k: strict > keeps the lowest index among equal maxima
            up2 = ~skip & ~up1 & (vk > better)
            better = np.where(up1, best, np.where(up2, vk, better))
            bi = np.where(up1, k, bi)
            best = np.where(up1, vk, best)
            tm = np.where(~skip, np.maximum(tm, threshold(better, rule)), tm)
    return best, better, bi, unsound


def scan_inputs(scale, offset, prices, seed, M=512, N=256):
    """Targets in a spatially coherent order (tiles of 32 are compact), bidders among them, four distinct seeds per bidder.
    prices: "random" (up to twice the largest distance), "ties" (values of all targets within a few ulp for one bidder)
    or "lattice" (coarse lattice, zero prices: exact ties everywhere)."""
    g = np.random.default_rng(seed)
    t = points(g, N, scale, offset)
    if prices == "lattice":
        t = (g.integers(0, 6, (N, 3)) * (scale / 6) + offset).astype(F)
    t = t[np.lexsort((t[:, 2], t[:, 1], np.floor((t[:, 0] - offset) / scale * 8)))]
    a = points(g, M, scale, offset)
    if prices == "lattice":
        a = (g.integers(0, 6, (M, 3)) * (scale / 6) + offset).astype(F)
    p = np.zeros(N, F)
    if prices == "random":
        p = (g.random(N) * 2.0 * np.sqrt(3.0) * scale).astype(F)
    elif prices == "ties":   # v_k ~ V0 for bidder 0 and its neighbours: p_k = 3 - r_k - V0 (>= 0), then jittered by ulps
        r = np.sqrt(sqdist(t, np.broadcast_to(a[0], t.shape))).astype(D)
        V0 = 3.0 - r.max() - 1.0
        p = steps((3.0 - r - V0).astype(F), g.integers(-2, 3, N))
        a[1:] = (a[0].astype(D) + (g.random((M - 1, 3)) - 0.5) * 1e-3 * scale).astype(F)
    seeds = np.argsort(g.random((M, N)), 1)[:, :4]
    return t, a, p, seeds


@pytest.mark.parametrize("prices", ["random", "ties", "lattice"])
@pytest.mark.parametrize("name,scale,offset", CASES)
def test_seeded_scan_equals_the_exhaustive_scan(name, scale, offset, prices):
    t, a, p, seeds = scan_inputs(scale, offset, prices, seed=zlib.crc32(f"{name} {prices}".encode()))
    best, better, bi, unsound = scan(t, a, p, seeds, KERNEL)
    assert not unsound.any(), (name, prices, int(unsound.sum()))
    v = value(sqdist(t[None], a[:, None]), p[None])
    top = -np.sort(-v, 1)
    assert np.array_equal(best, top[:, 0]) and np.array_equal(better, top[:, 1]), (name, prices)
    assert np.array_equal(bi, v.argmax(1)), (name, prices)  # argmax: the first index among equal maxima


@pytest.mark.parametrize("scale", [16.0, 100.0, 1000.0, 1e4])
def test_nearest_rounding_is_unsound_beyond_the_unit_cube(scale):
    """The checks above catch the rule they replace: rounded to nearest, T - margin and c - T_m lose the margin to
    rounding once ulp(T) approaches it, and targets whose value reaches T are skipped."""
    s, p, c, v, T = candidates(scale, 0.0, 400_000, seed=3)
    bad = candidate_skipped(c, threshold(T, NEAREST), s, NEAREST) & (v >= T)
    assert bad.any(), scale
    assert not (candidate_skipped(c, threshold(T, KERNEL), s, KERNEL) & (v >= T)).any()


def test_rounding_emulation_is_exact():
    """sub / fma against exact rational arithmetic, including exponent gaps beyond fp64's 53 bits and fp32 midpoints."""
    g = np.random.default_rng(11)
    n = 3000
    a = (g.standard_normal(n) * np.exp2(g.integers(-30, 30, n))).astype(F)
    b = (g.standard_normal(n) * np.exp2(g.integers(-30, 30, n))).astype(F)
    b[:200] = a[:200] * F(1 + 2 ** -23) ** 2                       # cancellation
    a[200:400], b[200:400] = (1 + np.arange(1, 201) * 2.0 ** -23).astype(F), F(2 ** -24)  # exact midpoints: ties to even
    up, down, near = sub(a, b, "up"), sub(a, b, "down"), sub(a, b, "nearest")
    assert np.array_equal(near, a - b)                              # numpy's fp32 subtraction is IEEE round-to-nearest
    c = (g.standard_normal(n) * np.exp2(g.integers(-40, 40, n))).astype(F)
    f = fma(a, b, c)
    for i in range(n):
        x = Fraction(float(a[i])) - Fraction(float(b[i]))
        assert Fraction(float(down[i])) <= x <= Fraction(float(up[i]))
        assert down[i] == up[i] if Fraction(float(down[i])) == x else np.nextafter(down[i], F(np.inf)) == up[i]
        y = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        lo, hi = np.nextafter(f[i], F(-np.inf)), np.nextafter(f[i], F(np.inf))
        assert abs(Fraction(float(f[i])) - y) <= min(abs(Fraction(float(lo)) - y), abs(Fraction(float(hi)) - y))


def test_restated_rule_is_the_kernels():
    """The restatement above is the kernel's rule: the margin, the rounding of both helpers, and every site of the Bid scans
    goes through them (no threshold or u formed with another rounding)."""
    core = open(os.path.join(CSRC, "pcl_emd_core.cuh")).read()
    m = re.search(r"constexpr float FILTER_MARGIN = ([0-9.e+-]+)f;", core)
    assert m and F(float(m.group(1))) == MARGIN
    assert re.search(r"float filter_threshold\(float T\) \{ return __fsub_rd\(T, FILTER_MARGIN\); \}", core)
    assert re.search(r"float filter_u\(float c, float tm\) \{ return __fsub_ru\(c, tm\); \}", core)
    assert "__fmul_rn(__fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy))), 0.999999f)" in core
    for f in ("pcl_emd_core.cuh", "pcl_emd.cu", "pcl_emd_team.cu", "pcl_emd_tasks.cuh"):
        src = open(os.path.join(CSRC, f)).read()
        body = src.replace("{ return __fsub_rd(T, FILTER_MARGIN); }", "").replace("{ return __fsub_ru(c, tm); }", "")
        assert "FILTER_MARGIN)" not in body, f                     # T - margin only inside filter_threshold
        assert not re.search(r"__f(sub|add)_r[nzdu]\([^;]*\btm\)", body), f   # c - T_m only inside filter_u
