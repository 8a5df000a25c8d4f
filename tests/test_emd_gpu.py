"""GPU parity tests of the auction EMD kernels (through the C ABI) against
  (1) the CPU oracle (bit-exact, always),
  (2) the UNMODIFIED reference extension (oracle/_ref/emd.so, see oracle/build_ref.py) -- exact on clouds
      where the reference's GetMax race cannot fire (oracle race_events == 0), statistical otherwise; where that
      extension cannot be built, against its recorded runs (tests/golden/reference_envelope.npz),
  (3) golden vectors that went through the reference's own emd_module.py,
  (4) size-independent properties at BASELINE.json's full size (B=32, N=2048)."""
import os

import numpy as np
import pytest
import torch

import oracle
import pointcloud_b200 as pcl
from pointcloud_b200 import synth
from pointcloud_b200._lib import PclError
from helpers import npy, ref_emd_backward, ref_emd_forward, sqdist_to_match

pytestmark = pytest.mark.gpu


def clouds(kind, b, n, seed):
    if kind == "uniform":
        return synth.uniform_clouds(b, n, seed=seed)
    x1, t = synth.table_clouds(b, n, seed=seed, regime="independent" if kind == "table" else "noisy")
    return x1, t[:, :, :3].contiguous()


@pytest.mark.parametrize("kind,b,n,eps,iters", [
    ("uniform", 2, 1024, 0.005, 50), ("uniform", 3, 2048, 0.005, 50), ("table", 3, 2048, 0.005, 50),
    ("noisy", 3, 2048, 0.005, 50), ("uniform", 1, 4096, 0.005, 50), ("uniform", 5, 1000, 0.005, 50),
    ("uniform", 2, 333, 0.002, 400), ("uniform", 40, 1024, 0.005, 20), ("uniform", 1, 1, 0.005, 3),
    ("uniform", 2, 37, 0.005, 1), ("table", 2, 1024, 0.002, 3000),
    ("uniform", 2, 8192, 0.005, 50), ("uniform", 3, 5000, 0.005, 30), ("table", 1, 6144, 0.005, 50),  # > 4096: cold state in L2
])
def test_emd_forward_bit_exact_vs_oracle(kind, b, n, eps, iters):
    x1, x2 = clouds(kind, b, n, seed=100 + n)
    o = oracle.emd_forward(x1, x2, eps, iters, nthreads=8)
    d, a, st = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), eps, iters, want_stats=True)
    assert np.array_equal(npy(a), o["assignment"])
    assert np.array_equal(npy(d), o["dist"])          # bit-exact fp32
    st = npy(st)
    assert np.array_equal(st[:, 0], o["sum_unass"]) and np.array_equal(st[:, 1], o["iters_run"])


@pytest.mark.parametrize("case", ["grid_ties", "all_pred_identical", "duplicate_targets", "out_of_range", "identical_clouds", "tiny_eps"])
def test_emd_degenerate_inputs_bit_exact_vs_oracle(case, ref_ext):
    """Exact ties everywhere: the order-independent tie rules (lowest original target index among equal values, largest
    bidder index inside the GetMax window) must reproduce the oracle's sequential scan regardless of the internal
    Morton order, the tile skipping and the scan mode."""
    g = torch.Generator().manual_seed(7)
    b, n, eps, iters = 3, 2048, 0.005, 50
    x1, x2 = torch.rand(b, n, 3, generator=g), torch.rand(b, n, 3, generator=g)
    if case == "grid_ties":            # coordinates on a coarse lattice: thousands of equal distances and equal values
        x1 = torch.randint(0, 6, (b, n, 3), generator=g).float() / 6
        x2 = torch.randint(0, 6, (b, n, 3), generator=g).float() / 6
    elif case == "all_pred_identical":
        x1 = torch.full((b, n, 3), 0.5)
    elif case == "duplicate_targets":
        x2 = x2[:, : n // 8].repeat(1, 8, 1)
    elif case == "out_of_range":       # the reference assumes [0,1]^3 (emd_module.py:9); values may go negative outside
        x1, x2 = x1 * 3 - 1, x2 * 4 - 2
    elif case == "identical_clouds":
        x1 = x2.clone()
    elif case == "tiny_eps":
        eps, iters = 1e-7, 30
    o = oracle.emd_forward(x1, x2, eps, iters, nthreads=3)
    d, a, st = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), eps, iters, want_stats=True)
    assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
    assert np.array_equal(npy(st)[:, 0], o["sum_unass"])
    if ref_ext is not None:            # and the unmodified reference agrees wherever it is deterministic
        rd, ra = ref_emd_forward(ref_ext, x1, x2, eps, iters)
        for i in range(b):
            if o["race_events"][i] == 0:
                assert np.array_equal(npy(ra[i]), npy(a[i]))


def test_emd_matches_unmodified_reference_extension(ref_ext):
    if ref_ext is None:
        pytest.skip("oracle/_ref/emd.so not built (needs /root/reference at build time)")
    checked = 0
    for kind, seed in [("uniform", 1), ("noisy", 2), ("uniform", 3), ("table", 4)]:
        x1, x2 = clouds(kind, 8, 2048, seed)
        o = oracle.emd_forward(x1, x2, 0.005, 50, nthreads=8)
        d, a, _ = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.005, 50)
        rd, ra = ref_emd_forward(ref_ext, x1, x2, 0.005, 50)
        for i in range(8):
            if o["race_events"][i] == 0:  # the reference is deterministic on this cloud -> exact
                assert np.array_equal(npy(ra[i]), npy(a[i])) and np.array_equal(npy(rd[i]), npy(d[i]))
                checked += 1
        # coarse sanity bound on every cloud, racy or not (the sharp statement is the envelope test below): mean
        # sqrt(dist) within 2 %
        ours, theirs = npy(d).astype(np.float64), npy(rd).astype(np.float64)
        assert abs(np.sqrt(ours).mean() - np.sqrt(theirs).mean()) <= 0.02 * np.sqrt(theirs).mean()
    assert checked >= 12


@pytest.fixture
def emd_path():
    """Selects an auction kernel for one test and restores the automatic choice afterwards."""
    yield pcl.set_emd_path
    pcl.set_emd_path("auto")


@pytest.mark.parametrize("path", ["cluster", "team", "tickets"])
@pytest.mark.parametrize("kind,b,n,eps,iters", [
    ("table", 32, 2048, 0.005, 50), ("noisy", 32, 2048, 0.005, 50), ("uniform", 3, 2048, 0.005, 50), ("table", 4, 2048, 0.005, 50),
    ("uniform", 5, 1000, 0.005, 50), ("uniform", 2, 333, 0.002, 400), ("uniform", 40, 1024, 0.005, 20), ("uniform", 1, 1, 0.005, 3),
    ("uniform", 2, 37, 0.005, 1), ("table", 2, 1024, 0.002, 3000), ("table", 100, 2048, 0.005, 50), ("uniform", 8, 3584, 0.005, 30),
])
def test_every_auction_kernel_is_bit_exact_vs_oracle(emd_path, path, kind, b, n, eps, iters):
    """The three kernels behind pcl_emd_fwd (include/pcl.h pcl_emd_set_path) distribute the same auction differently -- fixed
    clusters, owner + workers pulling tasks from an L2 mirror, clusters that export part of their heavy iterations to workers
    and steal items from each other -- and must all reproduce the oracle bit for bit, whoever ran which task."""
    emd_path(path)
    x1, x2 = clouds(kind, b, n, seed=0 if n == 2048 and b in (4, 32) else 100 + n)
    o = oracle.emd_forward(x1, x2, eps, iters, nthreads=16)
    for _ in range(2):  # twice: the task protocol's control block is re-zeroed by every call
        d, a, st = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), eps, iters, want_stats=True)
        assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
        st = npy(st)
        assert np.array_equal(st[:, 0], o["sum_unass"]) and np.array_equal(st[:, 1], o["iters_run"])
        if path == "team":
            assert (st[:, 3] == 0).all()  # stats[3]: cluster size, 0 = team kernel


def test_team_and_ticket_paths_refuse_what_they_cannot_do(emd_path):
    x1, x2 = clouds("uniform", 1, 5000, seed=5)  # > 3584 points: only the cluster kernel keeps part of the state in L2
    for path in ("team", "tickets"):
        emd_path(path)
        with pytest.raises(PclError):
            pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.005, 5)
    emd_path("auto")
    pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.005, 5)


# pick_cluster (csrc/pcl_emd.cu): the largest power of two <= 16 such that all b clusters are resident at once (a cluster lives
# inside one GPC: 8 clusters of 16 or 16 clusters of 8 do not fit a B200 although 128 <= 148 SMs).  Measured on B200:
# (which of two sizes fits can depend on how the part's GPCs are populated)
CLUSTER_SIZE_ON_B200 = {4: (16,), 8: (8, 16), 12: (8,), 16: (4, 8), 32: (4,), 40: (2,), 80: (1,)}


@pytest.mark.parametrize("b", [4, 8, 12, 16, 32, 40, 80])
@pytest.mark.parametrize("regime", ["independent", "noisy"])
def test_emd_bit_exact_at_every_cluster_size_on_the_bench_workload(emd_path, b, regime):
    """The launch bench.py times is B=32, N=2048 -> clusters of 4 CTAs; the dealing of the bidders to the CTAs of a
    cluster depends on the cluster size, so every size (16, 8, 4, 2, 1) is checked against the oracle at N=2048 on
    the bench's own clouds (bench.py make_pool: synth.table_clouds(32, 2048, seed=1000*rank+s, regime))."""
    import ctypes
    sm = ctypes.c_int(0)
    pcl._lib.lib().pcl_device_info(ctypes.byref(sm), None, None, None)
    emd_path("cluster")
    for seed in ((0, 1, 2, 3) if b == 32 else (0,)):       # B=32: all four base batches of the bench pool
        x1, t = synth.table_clouds(b, 2048, seed=seed, regime=regime)
        x2 = t[:, :, :3].contiguous()
        o = oracle.emd_forward(x1, x2, 0.005, 50, nthreads=16)
        d, a, st = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.005, 50, want_stats=True)
        st = npy(st)
        assert (st[:, 3] == st[0, 3]).all() and b * int(st[0, 3]) <= sm.value, st[:, 3]
        if sm.value == 148:  # every cluster size 16, 8, 4, 2, 1 is exercised on the machine this is built for
            assert int(st[0, 3]) in CLUSTER_SIZE_ON_B200[b], st[:, 3]
        assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
        assert np.array_equal(st[:, 0], o["sum_unass"]) and np.array_equal(st[:, 1], o["iters_run"])


def test_emd_deviation_lies_inside_the_reference_nondeterminism_envelope(ref_ext):
    """The reference's GetMax lets the LAST writer inside a +-1e-6 window win (emd_cuda.cu:181-194): which bidder that is
    depends on the thread schedule, so the unmodified reference is not reproducible -- on the bench's early-training batch
    every cloud has 8-37 such events and four IDENTICAL launches differ by up to 2 % in a cloud's mean sqrt(dist)
    (measured: tools/envelope_probe.py).  Every cloud without an event must equal the reference bit for bit; on the others
    our fixed rule (largest bidder index) must be one more draw from the reference's own distribution: per cloud and for
    the batch value the trainer sees, our result lies within 5 sigma of the reference's runs (4 repeats + 8 re-orderings
    of the predictions -- the same point sets, rows permuted back), sigma floored by the pooled per-cloud value."""
    if ref_ext is None:
        pytest.skip("oracle/_ref/emd.so not built (needs /root/reference at build time)")
    b, n = 32, 2048
    for regime in ("independent", "noisy"):                              # pool[0] and pool[1] of bench.py
        x1, t = synth.table_clouds(b, n, seed=0, regime=regime)
        x2 = t[:, :, :3].contiguous()
        o = oracle.emd_forward(x1, x2, 0.005, 50, nthreads=16)
        d, a, _ = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.005, 50)
        ours = np.sqrt(npy(d).astype(np.float64)).mean(1)                # per-cloud mean sqrt(dist)
        racy = o["race_events"] > 0
        g = torch.Generator().manual_seed(5)
        runs = []
        for r in range(12):
            perm = torch.arange(n) if r < 4 else torch.randperm(n, generator=g)
            rd, ra = ref_emd_forward(ref_ext, x1[:, perm], x2, 0.005, 50)
            inv = torch.empty_like(perm)
            inv[perm] = torch.arange(n)
            rd, ra = npy(rd)[:, inv.numpy()], npy(ra)[:, inv.numpy()]
            if r < 4:
                for i in np.nonzero(~racy)[0]:                           # deterministic clouds: exact
                    assert np.array_equal(ra[i], npy(a[i])) and np.array_equal(rd[i], npy(d[i]))
            runs.append(np.sqrt(rd.astype(np.float64)).mean(1))
        runs = np.stack(runs)                                            # (12, B)
        sigma = runs.std(0, ddof=1)
        pooled = float(np.sqrt((sigma[racy] ** 2).mean())) if racy.any() else 0.0
        dev = np.abs(ours - runs.mean(0))
        print(f"[{regime}] race-free clouds {int((~racy).sum())}/{b} (bit-exact vs the reference); racy clouds: reference sigma "
              f"pooled {pooled:.2e} (max {sigma.max():.2e}, identical-launch spread max {(runs[:4].max(0) - runs[:4].min(0)).max():.2e}), "
              f"ours - reference mean: max {dev.max():.2e} = {np.max(dev / np.maximum(np.maximum(sigma, pooled), 1e-12)):.2f} sigma")
        assert (dev[~racy] <= 1e-12).all()
        assert (dev <= 5.0 * np.maximum(sigma, pooled) + 1e-12).all(), (dev, sigma, pooled)
        batch = runs.mean(1)                                             # the loss value of the batch, per reference run
        assert abs(ours.mean() - batch.mean()) <= 5.0 * batch.std(ddof=1) + 1e-12


def test_emd_deviation_lies_inside_the_recorded_reference_envelope():
    """The per-cloud statements of the test above against the reference's recorded runs instead of live ones:
    tests/golden/reference_envelope.npz holds, per cloud of the same two batches, the mean and the spread (ddof=1) of the
    reference's 12 runs, restored by tests/golden/make_envelope_golden.py from profiles/r2_s1_envelope.txt.  Every cloud
    without a race event must equal the reference; the others must lie within 5 sigma of its runs.  (The batch-level
    statement needs each run's batch value, which the recording does not keep.)"""
    env = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_envelope.npz"))
    b, n = 32, 2048
    for regime in ("independent", "noisy"):
        x1, t = synth.table_clouds(b, n, seed=0, regime=regime)
        d, _, _ = pcl.emd_forward_raw(x1.cuda(), t[:, :, :3].contiguous().cuda(), 0.005, 50)
        ours = np.sqrt(npy(d).astype(np.float64)).mean(1)
        racy = env[f"{regime}_race_events"] > 0
        sigma = env[f"{regime}_ref_std"]
        pooled = float(np.sqrt((sigma[racy] ** 2).mean())) if racy.any() else 0.0
        dev = np.abs(ours - env[f"{regime}_ref_mean"])
        assert (dev[~racy] <= 1e-12).all(), regime
        assert (dev <= 5.0 * np.maximum(sigma, pooled) + 1e-12).all(), (regime, dev, sigma, pooled)


def test_emd_backward_matches_reference_and_oracle(ref_ext):
    x1, x2 = clouds("uniform", 4, 1024, 9)
    d, a, _ = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.005, 50)
    gd = torch.rand(4, 1024, generator=torch.Generator().manual_seed(1))
    g1, _ = oracle.emd_backward(x1, x2, npy(a), gd)
    xg = x1.cuda().requires_grad_()
    x2g = x2.cuda().requires_grad_()
    dist, asg = pcl.emdModule()(xg, x2g, 0.005, 50)
    assert dist.dtype == torch.float32 and asg.dtype == torch.int32 and not asg.requires_grad  # emd_module.py:74-79
    (dist * gd.cuda()).sum().backward()
    assert np.array_equal(npy(xg.grad), g1)                 # same fp32 op order as NmDistanceGradKernel
    assert x2g.grad is not None and not x2g.grad.any()      # target gets zeros (emd_module.py:69,72)
    if ref_ext is not None:
        rg = ref_emd_backward(ref_ext, x1, x2, gd.cuda(), a)
        assert np.array_equal(npy(rg), g1)


def test_emd_matches_golden_through_reference_module(golden):
    d, a, _ = pcl.emd_forward_raw(torch.from_numpy(golden["raw_xyz1"]).cuda(), torch.from_numpy(golden["raw_xyz2"]).cuda(), 0.005, 50)
    assert np.array_equal(npy(a), golden["raw_assignment"]) and np.array_equal(npy(d), golden["raw_dist"])
    x1 = torch.from_numpy(golden["raw_xyz1"]).cuda().requires_grad_()
    dist, _ = pcl.emdModule()(x1, torch.from_numpy(golden["raw_xyz2"]).cuda(), 0.005, 50)
    dist.sqrt().mean().backward()
    np.testing.assert_allclose(npy(x1.grad), golden["raw_grad"], rtol=1e-5, atol=1e-12)  # north star: 1e-5 relative


def test_emd_strided_views_and_half_inputs_need_no_copy():
    pred, target = synth.autoencoder_batch(3, 1024, seed=5)
    o = oracle.emd_forward(pred[:, :, :3], target[:, :, :3], 0.005, 50)
    pc, tc = pred.cuda(), target.cuda()
    d, a, _ = pcl.emd_forward_raw(pc[:, :, :3], tc[:, :, :3], 0.005, 50)   # row stride 6 (utils.py:254)
    assert np.array_equal(npy(a), o["assignment"]) and np.array_equal(npy(d), o["dist"])
    for dt in (torch.float16, torch.bfloat16):                             # cfg.precision = '16-mixed'
        ph = pc.to(dt)
        oh = oracle.emd_forward(ph[:, :, :3].float().cpu(), target[:, :, :3], 0.005, 50)  # == .float() up-cast
        dh, ah, _ = pcl.emd_forward_raw(ph[:, :, :3], tc[:, :, :3], 0.005, 50)
        assert np.array_equal(npy(ah), oh["assignment"]) and np.array_equal(npy(dh), oh["dist"])
        xg = ph.clone().requires_grad_()
        dist, _ = pcl.emdModule()(xg[:, :, :3], tc[:, :, :3], 0.005, 50)
        dist.sum().backward()
        assert xg.grad.dtype == dt and not xg.grad[:, :, 3:].any() and xg.grad[:, :, :3].any()


def test_emd_full_size_properties_and_determinism():
    """BASELINE config 2 size: B=32, N=2048, eps=0.005, 50 iterations (cfg.py:36-37)."""
    for kind in ("uniform", "table"):
        x1, x2 = clouds(kind, 32, 2048, 0)
        d, a, st = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.005, 50, want_stats=True)
        d2, a2, _ = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.005, 50)
        assert torch.equal(a, a2) and torch.equal(d, d2)                      # run-to-run deterministic
        an, dn = npy(a), npy(d)
        assert an.min() >= 0 and an.max() < 2048
        np.testing.assert_allclose(dn, sqdist_to_match(x1.numpy(), x2.numpy(), an), rtol=1e-5, atol=1e-10)  # "Verified EMD"
        uniq = np.array([len(np.unique(r)) for r in an])
        assert (uniq >= (0.93 if kind == "uniform" else 0.55) * 2048).all()     # near-bijection (emd_module.py:90); table-shaped
        # clouds are far from converged after 50 iterations (SURVEY App. C: 1713-1934 unique; this generator: 1300-1900)
        # permuting the target permutes the assignment but keeps every distance: the auction is index-covariant
        # only up to tie-breaks, so check the value-level invariant instead: EMD is within 3 % after a shuffle
        perm = torch.randperm(2048, generator=torch.Generator().manual_seed(1))
        dp, _, _ = pcl.emd_forward_raw(x1.cuda(), x2[:, perm].cuda(), 0.005, 50)
        assert abs(float(dp.sqrt().mean()) - float(d.sqrt().mean())) <= 0.03 * float(d.sqrt().mean())
        # identical clouds: every point is its own best match
        dz, az, _ = pcl.emd_forward_raw(x2.cuda(), x2.cuda(), 0.005, 50)
        assert float(dz.sqrt().mean()) < 1e-3


def test_emd_converges_with_test_settings():
    x1, x2 = clouds("uniform", 2, 1024, 3)
    o = oracle.emd_forward(x1, x2, 0.002, 10000, nthreads=2)      # cfg.py:40-41
    d, a, st = pcl.emd_forward_raw(x1.cuda(), x2.cuda(), 0.002, 10000, want_stats=True)
    assert np.array_equal(npy(a), o["assignment"]) and (npy(st)[:, 1] < 10000).all()
    assert all(len(np.unique(r)) == 1024 for r in npy(a))         # early exit on a bijection


def test_emd_error_behaviour():
    x = torch.rand(1, 1024, 3).cuda()
    with pytest.raises(AssertionError):
        pcl.emdModule()(x, torch.rand(1, 2048, 3).cuda(), 0.005, 50)          # n != m (emd_module.py:38)
    with pytest.raises(AssertionError):
        pcl.emdModule()(x, torch.rand(2, 1024, 3).cuda(), 0.005, 50)          # batch mismatch (:39)
    nmax = pcl._lib.lib().pcl_emd_max_points()
    big = torch.rand(1, nmax + 1024, 3).cuda()
    with pytest.raises(PclError, match="not supported"):
        pcl.emdModule()(big, big, 0.005, 50)
    d, a, _ = pcl.emd_forward_raw(torch.rand(0, 1024, 3).cuda(), torch.rand(0, 1024, 3).cuda(), 0.005, 50)  # empty batch
    assert d.shape == (0, 1024)
