"""The device simulator with LogGaussianCox curves (csrc/cont_rand.cu: generation 0 cell by cell of the grid, Poisson counts of the
trapezoid areas and times by the inverse CDF of the linear rate).  Its samples must be those of the curve model: time rescaling
(tests/cont_compensator.py) with negative controls, per-cell Poisson counts, agreement with the host thinning sampler, determinism, the
homogeneous path untouched, the handle usable by the sweeps, the refusals, and a device chain that recovers the curves."""
import ctypes

import numpy as np
import pytest

import cont_compensator as cc
import nhp_b200 as nhp
import synth
from nhp_b200.core import ContinuousData, Context, _ptr
from test_rand_lgcp_host_cpu import skewed_curves

pytestmark = pytest.mark.gpu

INVALID = -1


def model(x, lam, kind="ln", wmax=0.2, net=False, seed=3, m=0.0, eta=None):
    K = lam.shape[0]
    base = nhp.LogGaussianCoxProcess(x, lam.copy(), m=m, sigma=1.0, eta=eta or (x[-1] - x[0]) / 8.0)
    if kind == "ln":
        _, W, mu, tau, A = synth.ln_params(K, seed, wmax=max(wmax, 1e-3), density=0.6)
        imp, law = nhp.LogitNormalImpulseResponse(mu, tau, 1.0), dict(kind="ln", p1=mu, p2=tau, dtmax=1.0)
    else:  # the simulators draw untruncated Exponential lags
        _, W, theta, A = synth.exp_params(K, seed, wmax=max(wmax, 1e-3), density=0.6)
        imp, law = nhp.ExponentialImpulseResponse(theta, dtmax=np.inf), dict(kind="exp", p1=theta)
    W = W * (wmax > 0)
    if net:
        A[0, 1] = 1.0  # at least one link
        proc = nhp.ContinuousNetworkHawkesProcess(base, imp, nhp.DenseWeightModel(W), A, nhp.BernoulliNetworkModel(0.5, K))
        return proc, dict(law, W=W, A=A)
    return nhp.ContinuousStandardHawkesProcess(base, imp, nhp.DenseWeightModel(W)), dict(law, W=W)


def raw_rand(proc, T, seed, max_events):
    """nhp_cont_rand on the process's context as it stands: (code, handle or None)."""
    ctx = proc._ctx()
    h = ctypes.c_void_p()
    rc = ctx.lib.nhp_cont_rand(ctx.h, float(T), int(seed), int(max_events), ctypes.byref(h))
    return rc, (ContinuousData.from_handle(ctx, h, proc.ndims()) if rc == 0 else h.value)


def device_curves(proc):
    ctx = proc._ctx()
    v = np.empty(proc.baseline.lam_grid.size)
    ctx.check(ctx.lib.nhp_cont_baseline_get(ctx.h, _ptr(v)))
    return v.reshape(proc.baseline.lam_grid.shape)


@pytest.mark.parametrize("kind,net,G", [("ln", False, 17), ("exp", False, 9), ("ln", True, 41)])
def test_device_sample_rescales_to_a_unit_poisson_process(kind, net, G):
    K, T = 4, 4000.0
    x, lam = skewed_curves(K, T, G, 11 + G)
    proc, law = model(x, lam, kind, net=net)
    t, nodes, dur = nhp.rand_device(proc, T, seed=12).download()
    assert dur == T and np.all(np.diff(t) >= 0) and t[0] >= 0.0 and t[-1] <= T
    assert np.all(np.bincount(nodes - 1, minlength=K) > 3000)
    ok, p = cc.rescaling_holds(t, nodes, x, lam, **law)
    assert ok, p
    for control in (cc.time_averaged(x, lam, T), cc.reversed_in_time(x, lam)):  # negative controls
        assert not np.allclose(control, lam)
        assert cc.rescaling_pvalues(t, nodes, x, control, **law).min() < 1e-6


def clipped_cells(x, lam, T):
    """Edges of the grid intervals clipped to [0, T] and the trapezoid area of every (node, cell)."""
    e = np.concatenate([[0.0], x[(x > 0.0) & (x < T)], [T]])
    y = np.stack([np.interp(e, x, v) for v in lam])
    return e, 0.5 * (y[:, 1:] + y[:, :-1]) * np.diff(e), (y[:, 1:] == 0) & (y[:, :-1] == 0)


def test_counts_per_cell_are_poisson_of_the_trapezoid():
    """W = 0: over replicates the count of every (node, clipped cell) has the Poisson(area) mean and variance; a grid reaching past
    [0, T] on both sides is clipped, and a segment where the curve is 0 at both ends never holds an event."""
    K, T, reps = 2, 100.0, 300
    x = np.linspace(-10.0, 115.0, 11)  # cells of 12.5; [0, T] cuts the first and the last
    lam = np.array([[0.5, 1.0, 2.0, 3.0, 2.5, 1.5, 1.0, 0.5, 0.2, 0.1, 0.3],
                    [1.0, 2.0, 0.0, 0.0, 0.0, 1.5, 3.0, 3.0, 0.5, 1.0, 2.0]])
    proc, _ = model(x, lam, "ln", wmax=0.0)
    e, area, zero = clipped_cells(x, lam, T)
    assert zero.sum() == 2 and e[1] == 2.5 and e[-2] == 90.0
    counts = np.empty((reps, K, e.size - 1))
    for r in range(reps):
        t, nodes, _ = nhp.rand_device(proc, T, seed=1000 + r).download()
        for k in range(K):
            counts[r, k] = np.histogram(t[nodes == k + 1], bins=e)[0]
    assert np.all(counts[:, zero] == 0) and counts[:, 1].sum() > 0  # node 2 is zero on [15, 40]
    pos = area > 0
    mean, var = counts.mean(axis=0), counts.var(axis=0, ddof=1)
    z_mean = (mean - area)[pos] / np.sqrt(area[pos] / reps)
    z_var = (var - area)[pos] / np.sqrt((area[pos] + 2 * area[pos] ** 2) / reps)
    assert np.all(np.abs(z_mean) < 5), (mean, area)
    assert np.all(np.abs(z_var) < 6), (var, area)


def test_device_sample_matches_host_simulator_in_distribution():
    """Inversion on the device against thinning on the host, with children: per-(node, cell) counts over many short samples."""
    K, T, G, reps = 2, 30.0, 7, 300
    x, lam = skewed_curves(K, T, G, 21)
    proc, _ = model(x, lam, "ln", wmax=0.4, seed=22)
    e = x
    host = np.empty((reps, K, G - 1))
    dev = np.empty((reps, K, G - 1))
    for r in range(reps):
        for out, (t, nodes, _) in ((host, nhp.rand(proc, T, np.random.default_rng(2000 + r))), (dev, nhp.rand_device(proc, T, seed=3000 + r).download())):
            for k in range(K):
                out[r, k] = np.histogram(t[nodes == k + 1], bins=e)[0]
    se = np.sqrt(host.var(axis=0, ddof=1) / reps + dev.var(axis=0, ddof=1) / reps)
    z = (dev.mean(axis=0) - host.mean(axis=0)) / se
    assert np.all(np.abs(z) < 4.5), z
    assert 0.6 < dev.sum(axis=(1, 2)).var() / host.sum(axis=(1, 2)).var() < 1.6


def test_seed_determines_the_sample_and_clearing_the_curves_restores_the_homogeneous_path():
    K, T = 3, 300.0
    x, lam = skewed_curves(K, T, 13, 31)
    proc, _ = model(x, lam, "ln", wmax=0.3, net=True, seed=32)
    a, b, c = (nhp.rand_device(proc, T, seed=s).download() for s in (33, 33, 34))
    assert all(np.array_equal(p, q) for p, q in zip(a[:2], b[:2]))
    assert a[0].size != c[0].size or not np.array_equal(a[0], c[0])
    # curves set, then cleared: bit for bit the homogeneous sample of a fresh context
    ctx = proc._ctx()
    proc._push(ctx)
    ctx.check(ctx.lib.nhp_cont_baseline_grid(ctx.h, 0, None, None))
    rc, d = raw_rand(proc, T, 35, 100000)
    assert rc == 0
    hom = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(proc.baseline.lam), proc.impulses, proc.weights, proc.adjacency_matrix, proc.network)
    hom.ctx = Context()
    ref = nhp.rand_device(hom, T, seed=35, max_events=100000).download()
    got = d.download()
    assert got[0].size > 500
    np.testing.assert_array_equal(got[0], ref[0])
    np.testing.assert_array_equal(got[1], ref[1])


def test_constant_curves_give_the_homogeneous_law():
    K, T, G = 3, 4000.0, 9
    lam0 = np.array([0.7, 1.0, 1.4])
    x = np.linspace(0.0, T, G)
    proc, law = model(x, np.repeat(lam0[:, None], G, axis=1), "exp", wmax=0.3, seed=41)
    t, nodes, _ = nhp.rand_device(proc, T, seed=42).download()
    ok, p = cc.rescaling_holds(t, nodes, np.array([0.0, T]), np.repeat(lam0[:, None], 2, axis=1), **law)
    assert ok, p
    hom = nhp.ContinuousStandardHawkesProcess(nhp.HomogeneousProcess(lam0), proc.impulses, proc.weights)
    n_c = np.array([nhp.rand_device(proc, 200.0, seed=100 + r).n_own for r in range(150)], float)
    n_h = np.array([nhp.rand_device(hom, 200.0, seed=400 + r).n_own for r in range(150)], float)
    assert abs(n_c.mean() - n_h.mean()) < 4.5 * np.sqrt((n_c.var() + n_h.var()) / 150)


def test_the_sample_is_ordinary_data_for_the_sweeps():
    K, T, G = 4, 500.0, 21
    x, lam = skewed_curves(K, T, G, 51)
    proc, _ = model(x, lam, "ln", wmax=0.3, seed=52)
    d = nhp.rand_device(proc, T, seed=53)
    # the handle from nhp_events_from_device against a fresh nhp_events_upload of its copy: the parity bar, 1e-10 relative
    ll_dev = nhp.loglikelihood(proc, d)
    ll_up = nhp.loglikelihood(proc, d.download())
    assert ll_dev == pytest.approx(ll_up, rel=1e-10)
    # the Gibbs sweep with the curves' prior (the elliptical-slice update) runs on it
    res = nhp.mcmc_device_(proc, d, nsteps=3, seed=54, baseline_on_device=True)
    curves = np.array(res.samples)[:, :K * G]
    assert np.all(np.isfinite(curves)) and np.all(curves > 0) and not np.allclose(curves[-1], lam.ravel())


def test_refusals_leave_no_handle_and_the_curves_unchanged():
    K, T, G = 3, 100.0, 9
    for x in (np.linspace(0.5, T, G), np.linspace(0.0, T - 1.0, G)):
        lam = np.ones((K, G)) + np.arange(G) / G
        proc, _ = model(x, lam, "ln", seed=61)
        proc._push(proc._ctx())
        rc, h = raw_rand(proc, T, 1, 100000)
        assert rc == INVALID and h is None
        assert b"does not cover" in proc._ctx().lib.nhp_last_error(proc._ctx().h)
        np.testing.assert_array_equal(device_curves(proc), lam)
        with pytest.raises(ValueError):
            nhp.rand_device(proc, T, seed=1)  # the default max_events integrates the curves over [0, T] first
    x = np.linspace(0.0, T, G)
    lam = 2.0 + np.arange(G) / G
    lam = np.repeat(lam[None, :], K, axis=0)
    proc, _ = model(x, lam, "ln", wmax=0.0, seed=62)
    proc._push(proc._ctx())
    rc, h = raw_rand(proc, T, 1, 100)  # generation 0 alone has ~750 events
    assert rc == INVALID and h is None
    assert b"generation 0" in proc._ctx().lib.nhp_last_error(proc._ctx().h)
    np.testing.assert_array_equal(device_curves(proc), lam)


# Posterior-mean curves of a 400-sweep device chain (burn-in 100) on a sample drawn from the curves, K = 3, 9 grid points, T = 2000
# (about 1800 events per node): the largest relative error over the 27 grid values was 0.273 on the B200 (NVIDIA B200, 1000 W power
# limit; chain seed 72), and 1.340 for the control chain on data from the time averages.  The tolerance sits between the two.
RECOVERY_TOL = 0.4


def _chain_mean_curves(lam_gen, x, T, seed):
    K, G = lam_gen.shape
    gen, _ = model(x, lam_gen, "ln", wmax=0.2, seed=71)
    d = nhp.rand_device(gen, T, seed=seed)
    fit, _ = model(x, np.ones((K, G)), "ln", wmax=0.2, seed=71, eta=T / 8.0)
    res = nhp.mcmc_device_(fit, d, nsteps=400, seed=72, baseline_on_device=True)
    return np.array(res.samples)[100:, :K * G].mean(axis=0).reshape(K, G)


def test_device_chain_recovers_the_curves_of_the_sample():
    K, G, T = 3, 9, 2000.0
    x = np.linspace(0.0, T, G)
    lam_true = 0.9 + 0.45 * np.sin(2 * np.pi * x[None, :] / T + 2.0 * np.arange(K)[:, None])
    err = np.abs(_chain_mean_curves(lam_true, x, T, 73) / lam_true - 1.0)
    ctrl = np.abs(_chain_mean_curves(cc.time_averaged(x, lam_true, T), x, T, 73) / lam_true - 1.0)
    print(f"recovery: max relative error {err.max():.4f} (mean {err.mean():.4f}), control {ctrl.max():.4f}")
    assert err.max() < RECOVERY_TOL, err
    assert ctrl.max() > 2 * RECOVERY_TOL, ctrl  # a chain on data from the time averages ends far from the true curves
