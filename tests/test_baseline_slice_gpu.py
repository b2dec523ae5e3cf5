"""The elliptical-slice update of LogGaussianCoxProcess curves on the device (csrc/cont_slice.cu, nhp_cont_resample_baseline) and the
device chains that use it.  Given z and u the curves must be those of tests/slice_reference.py (which the CPU tests pin to the host
mirror) computed from the parents the device drew, with the same attempt counts; with Philox the chain must sample the posterior."""
import ctypes

import numpy as np
import pytest

import nhp_b200 as nhp
import slice_reference as sr
import synth
from nhp_b200.continuous import _hyper, _resample_parents
from nhp_b200.core import _f64, _ptr

pytestmark = pytest.mark.gpu

STATE, NUMERIC, INVALID = -4, -5, -1


def curves(K, T, seed, G, spread=0.3):
    rng = np.random.default_rng(seed)
    x = np.linspace(0.0, T, G)
    return x, 1.0 + spread * np.sin(2 * np.pi * rng.uniform(0.5, 3.0, (K, 1)) * x[None, :] / T + rng.uniform(0, 6, (K, 1)))


def model(net, kind, K, x, lam, seed, m=0.0, wmax=None, eta=None):
    wmax = 1.5 / K if wmax is None else wmax
    if kind == "ln":
        _, W, p1, p2, A = synth.ln_params(K, seed, wmax=wmax, density=0.5)
        imp = nhp.LogitNormalImpulseResponse(p1, p2, 1.0)
    else:
        _, W, p1, A = synth.exp_params(K, seed, wmax=wmax, density=0.5)
        imp = nhp.ExponentialImpulseResponse(p1, dtmax=1.0)
    base = nhp.LogGaussianCoxProcess(x, lam.copy(), m=m, sigma=1.0, eta=eta or (x[-1] - x[0]) / 10.0)
    if net:
        return nhp.ContinuousNetworkHawkesProcess(base, imp, nhp.DenseWeightModel(W), A, nhp.BernoulliNetworkModel(0.5, K))
    return nhp.ContinuousStandardHawkesProcess(base, imp, nhp.DenseWeightModel(W))


def parents_of(ctx, d):
    par = np.empty(d.n_own, dtype=np.int64)
    ctx.check(ctx.lib.nhp_cont_parents_get(ctx.h, d.h, _ptr(par), None))
    return par


def draws(K, G, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((K, G)), rng.random((K, sr.NU))


def check_against_statement(proc, data, seed, zu_seed):
    t, nodes, T = data
    K, G = proc.baseline.lam_grid.shape
    ctx = proc._ctx()
    d = proc.upload(data)
    proc._push(ctx)
    _resample_parents(ctx, d, seed, 0, None, False)
    tb = sr.baseline_events(t, nodes, parents_of(ctx, d), K)
    z, u = draws(K, G, zu_seed)
    before = proc.baseline.lam_grid.copy()
    got = proc.baseline.resample_device_(ctx, d, z=z, u=u)
    ref, att = sr.slice_update(proc.baseline.x, before, proc.baseline._chol, proc.baseline.m, tb, z, u)
    np.testing.assert_allclose(got, ref, rtol=1e-12)
    np.testing.assert_array_equal(proc.baseline.last_attempts, att)
    d.free()
    return tb, att


@pytest.mark.parametrize("net,kind,G", [(False, "ln", 2), (False, "exp", 37), (True, "ln", 37), (True, "exp", 2), (True, "ln", 600), (False, "exp", 600)])
def test_given_draws_the_curves_are_the_statement(net, kind, G):
    K = 6
    t, nodes, T = synth.poisson_stream(3000, K, 40.0, 11 + G)
    keep = nodes != K  # the last node has no events, so none attributed to the baseline
    t, nodes = t[keep], nodes[keep]
    x, lam = curves(K, T, 12, G)
    proc = model(net, kind, K, x, lam, 13, m=0.1)
    tb, att = check_against_statement(proc, (t, nodes, T), 14, 15 + G)
    assert tb[K - 1].size == 0 and all(tb[k].size > 0 for k in range(K - 1))
    assert att.min() >= 1


def test_thousand_skewed_nodes_are_the_statement():
    """K = 1000 with config 4-like skew: a few nodes hold many events (several work items), most hold few."""
    K, n = 1000, 300000
    rng = np.random.default_rng(21)
    w = 1.0 / np.arange(1, K + 1) ** 0.9
    nodes = rng.choice(np.arange(1, K + 1), n, p=w / w.sum()).astype(np.int64)
    t = np.sort(rng.uniform(0.0, 2000.0, n))
    T = 2000.0
    x, lam = curves(K, T, 22, 41)
    proc = model(True, "ln", K, x, lam * 0.5, 23, wmax=0.3 / K)
    tb, att = check_against_statement(proc, (t, nodes, T), 24, 25)
    assert max(b.size for b in tb) > 4 * 512 and att.max() >= 2


def test_philox_is_reproducible_and_keyed_by_the_counter():
    K, G = 8, 21
    t, nodes, T = synth.poisson_stream(4000, K, 50.0, 31)
    x, lam = curves(K, T, 32, G)
    proc = model(True, "ln", K, x, lam, 33)
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    outs = []
    for counter in (1, 1, 2):
        proc.baseline.lam_grid = lam.copy()
        proc._push(ctx)
        _resample_parents(ctx, d, 34, 0, None, False)
        outs.append(proc.baseline.resample_device_(ctx, d, seed=35, counter=counter))
    assert np.array_equal(outs[0], outs[1])
    assert not np.array_equal(outs[0], outs[2])
    assert not np.array_equal(outs[0], lam)
    d.free()


def _posterior_mean_quadrature(x, tk, m, Sigma, n=801, span=6.0):
    g = np.linspace(-span, span, n)
    y0, y1 = np.meshgrid(g, g, indexing="ij")
    P = np.linalg.inv(Sigma)
    logp = -0.5 * (P[0, 0] * y0 * y0 + 2 * P[0, 1] * y0 * y1 + P[1, 1] * y1 * y1)
    v0, v1 = np.exp(m + y0), np.exp(m + y1)
    logp += -0.5 * (v0 + v1) * (x[1] - x[0])
    for ti in tk:
        logp += np.log((v1 * (ti - x[0]) + v0 * (x[1] - ti)) / (x[1] - x[0]))
    p = np.exp(logp - logp.max())
    p /= p.sum()
    return np.array([np.sum(p * y0), np.sum(p * y1)])


def test_chains_with_fixed_parents_sample_the_posterior():
    """G = 2 and 64 identical nodes with fixed (baseline) parents: 64 independent chains of the update.  Their mean of y must match
    a 2-D quadrature of the posterior within 5 standard errors (the chains' means are the batch means)."""
    K, G, T, m, nb = 64, 2, 10.0, 0.5, 20
    tk = np.sort(np.random.default_rng(41).uniform(0.0, T, nb))
    t = np.repeat(tk, K)
    nodes = np.tile(np.arange(1, K + 1, dtype=np.int64), nb)
    x = np.array([0.0, T])
    proc = model(False, "exp", K, x, np.full((K, G), 1.5), 42, m=m, wmax=1e-3, eta=T / 2.0)
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    proc._push(ctx)
    proc.baseline.push_prior(ctx)
    par = np.zeros(t.size, dtype=np.int64)
    nsteps, burn = 1500, 100
    ys = np.empty((nsteps, K, G))
    for s in range(nsteps):
        ctx.check(ctx.lib.nhp_cont_parents_set(ctx.h, d.h, _ptr(par)))
        ctx.check(ctx.lib.nhp_cont_resample_baseline(ctx.h, d.h, 43, s, None, None, None))
        v = np.empty(K * G)
        ctx.check(ctx.lib.nhp_cont_baseline_get(ctx.h, _ptr(v)))
        ys[s] = np.log(v.reshape(K, G)) - m
    chain_means = ys[burn:].mean(axis=0)  # [K, G]
    est, se = chain_means.mean(axis=0), chain_means.std(axis=0, ddof=1) / np.sqrt(K)
    ref = _posterior_mean_quadrature(x, tk, m, proc.baseline.Sigma)
    assert np.all(np.abs(est - ref) < 5 * se), (est, ref, se)
    assert np.all(se < 0.1)
    d.free()


def _sweep_explicit(ctx, d, seed, counter, T, hy, alpha, beta):
    lib = ctx.lib
    ctx.check(lib.nhp_cont_resample_parents(ctx.h, d.h, seed, counter, None, None, None))
    ctx.check(lib.nhp_cont_resample_params(ctx.h, d.h, seed, counter, float(T), _ptr(hy), hy.size, 1))
    ctx.check(lib.nhp_cont_resample_baseline(ctx.h, d.h, seed, counter, None, None, None))
    ctx.check(lib.nhp_cont_resample_adjacency_dev(ctx.h, d.h, -1.0, seed, counter + (1 << 40), 0, 1, 1))
    rho = ctypes.c_double()
    ctx.check(lib.nhp_cont_resample_network(ctx.h, seed, counter, alpha, beta, ctypes.byref(rho)))


def _state(ctx, K, G):
    out = [np.empty(K)] + [np.empty(K * K) for _ in range(4)] + [np.empty(K * G)]
    ctx.check(ctx.lib.nhp_cont_params_get(ctx.h, *[_ptr(a) for a in out[:5]]))
    ctx.check(ctx.lib.nhp_cont_baseline_get(ctx.h, _ptr(out[5])))
    rho = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_network_get(ctx.h, ctypes.byref(rho)))
    return out + [np.array([rho.value])]


def test_gibbs_sweep_with_a_prior_is_the_explicit_sequence():
    K, G = 6, 31
    t, nodes, T = synth.poisson_stream(5000, K, 40.0, 51)
    x, lam = curves(K, T, 52, G)
    proc = model(True, "ln", K, x, lam, 53, wmax=0.3)
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    states = []
    try:
        for explicit in (False, True):  # both chains start from the pushed model on the same handle
            proc._push(ctx)
            proc.baseline.push_prior(ctx)
            ctx.check(ctx.lib.nhp_cont_network_set(ctx.h, 0.5))
            hy = _hyper(proc)
            for counter in range(3):
                if explicit:
                    _sweep_explicit(ctx, d, 54, counter, T, hy, 1.0, 1.0)
                else:
                    ctx.check(ctx.lib.nhp_cont_gibbs_sweep(ctx.h, d.h, d.h, 54, counter, float(T), _ptr(hy), hy.size, 1.0, 1.0))
                    info = np.zeros(8)
                    ctx.check(ctx.lib.nhp_cont_sweep_info(ctx.h, info.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
                    assert info[3] > 0.0 and info[4] >= 2
            states.append(_state(ctx, K, G))
    finally:
        d.free()
    for a, b in zip(*states):  # the float statistics are accumulated with atomics: equal up to the summation order
        np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-12)
    assert not np.allclose(states[0][5], lam.ravel())


@pytest.mark.parametrize("net", [False, True])
def test_device_trace_holds_the_curves_of_the_chain(net):
    K, G, nsteps = 5, 17, 6
    t, nodes, T = synth.poisson_stream(4000, K, 30.0, 61)
    x, lam = curves(K, T, 62, G)
    a, b = model(net, "ln", K, x, lam, 63, wmax=0.3), model(net, "ln", K, x, lam, 63, wmax=0.3)
    ref = nhp.mcmc_(a, (t, nodes, T), nsteps=nsteps, seed=64, device_draws=True, baseline_on_device=True)
    got = nhp.mcmc_device_(b, (t, nodes, T), nsteps=nsteps, seed=64, baseline_on_device=True)
    assert len(got.samples) == nsteps
    for p, q in zip(ref.samples, got.samples):
        np.testing.assert_allclose(p, q, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(a.params(), b.params(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(b.baseline.lam_grid.ravel(), got.samples[-1][(1 if net else 0):(1 if net else 0) + K * G], rtol=0)
    assert not np.array_equal(got.samples[0], got.samples[-1])
    # a trace without curves
    ctx = b._ctx()
    b._push(ctx)  # no prior: the trace keeps no curves
    ctx.check(ctx.lib.nhp_cont_trace_begin(ctx.h, 2))
    ctx.check(ctx.lib.nhp_cont_trace_push(ctx.h))
    v = np.empty(K * G)
    assert ctx.lib.nhp_cont_trace_read_curves(ctx.h, 0, 1, _ptr(v)) == STATE
    ctx.check(ctx.lib.nhp_cont_trace_free(ctx.h))
    # a trace with curves refuses a grid of another size
    b._push(ctx)
    b.baseline.push_prior(ctx)
    ctx.check(ctx.lib.nhp_cont_trace_begin(ctx.h, 2))
    x2 = np.linspace(0.0, T, G + 1)
    ctx.check(ctx.lib.nhp_cont_baseline_grid(ctx.h, x2.size, _ptr(x2), _ptr(_f64(np.ones(K * x2.size)))))
    assert ctx.lib.nhp_cont_trace_push(ctx.h) == STATE
    ctx.check(ctx.lib.nhp_cont_trace_free(ctx.h))


def test_posterior_means_agree_with_the_host_update():
    """Curves and W from the device-update chain against the host-update chain (mcmc_(device_draws=True)) on a small model."""
    K, G, nsteps, burn = 3, 9, 600, 100
    x = np.linspace(0.0, 200.0, G)
    lam_true = 0.8 + 0.4 * np.sin(x[None, :] / 40.0 + np.arange(K)[:, None])
    _, W, mu, tau, _ = synth.ln_params(K, 71, wmax=0.2)
    gen = nhp.ContinuousStandardHawkesProcess(nhp.HomogeneousProcess(np.full(K, 1.0)), nhp.LogitNormalImpulseResponse(mu, tau, 1.0), nhp.DenseWeightModel(W))
    t, nodes, T = nhp.rand(gen, 200.0, np.random.default_rng(72))
    res = []
    for dev in (False, True):
        proc = nhp.ContinuousStandardHawkesProcess(nhp.LogGaussianCoxProcess(x, np.ones((K, G)), sigma=1.0, eta=40.0),
                                                   nhp.LogitNormalImpulseResponse(mu.copy(), tau.copy(), 1.0), nhp.DenseWeightModel(W.copy()))
        r = nhp.mcmc_(proc, (t, nodes, T), nsteps=nsteps, seed=73 + dev, device_draws=True, baseline_on_device=dev)
        res.append(np.array(r.samples[burn:]))
    nb = K * G
    for sl in (slice(0, nb), slice(nb + 2 * K * K, nb + 3 * K * K)):  # curves; W (params: baseline, mu, tau, W)
        a, b = res[0][:, sl], res[1][:, sl]
        # batch means over 10 batches per chain: a generous Monte-Carlo error of the difference
        sa = a.reshape(10, -1, a.shape[1]).mean(axis=1).std(axis=0, ddof=1) / np.sqrt(10)
        sb = b.reshape(10, -1, b.shape[1]).mean(axis=1).std(axis=0, ddof=1) / np.sqrt(10)
        diff = np.abs(a.mean(axis=0) - b.mean(axis=0))
        assert np.all(diff < 5 * np.sqrt(sa ** 2 + sb ** 2) + 0.02 * np.abs(a.mean(axis=0))), (diff, sa, sb)


def test_error_paths_leave_the_curves_unchanged():
    K, G = 4, 9
    t, nodes, T = synth.poisson_stream(2000, K, 30.0, 81)
    x, lam = curves(K, T, 82, G)
    proc = model(True, "ln", K, x, lam, 83)
    ctx = proc._ctx()
    lib = ctx.lib
    d = proc.upload((t, nodes, T))
    get = lambda: (lambda v: (ctx.check(lib.nhp_cont_baseline_get(ctx.h, _ptr(v))), v)[1])(np.empty(K * G))
    run = lambda z=None, u=None: lib.nhp_cont_resample_baseline(ctx.h, d.h, 1, 0, _ptr(z), _ptr(u), None)
    L = _f64(proc.baseline._chol.ravel(order="F"))
    # missing curves
    ctx.check(lib.nhp_cont_params_set(ctx.h, 1, K, _ptr(_f64(np.ones(K))), _ptr(_f64(np.ones(K * K) * 0.01)), None,
                                      _ptr(_f64(np.zeros(K * K))), _ptr(_f64(np.ones(K * K))), 1.0))
    assert run() == STATE
    assert lib.nhp_cont_baseline_get(ctx.h, _ptr(np.empty(K * G))) == STATE
    assert lib.nhp_cont_baseline_prior(ctx.h, G, _ptr(L), 0.0) == STATE
    # missing prior (the curves' _push does not send it), missing parents
    proc._push(ctx)
    assert run() == STATE
    proc.baseline.push_prior(ctx)
    assert run() == STATE  # no parent sweep yet
    np.testing.assert_array_equal(get(), lam.ravel())
    # mismatched grid, invalid L
    assert lib.nhp_cont_baseline_prior(ctx.h, G + 1, _ptr(_f64(np.eye(G + 1).ravel())), 0.0) == INVALID
    for bad in (np.nan, -1.0, 0.0):
        L2 = L.copy()
        L2[G + 1] = bad  # the diagonal entry (1, 1)
        assert lib.nhp_cont_baseline_prior(ctx.h, G, _ptr(L2), 0.0) == INVALID
    L3 = L.copy()
    L3[G] = np.inf  # strictly upper (0, 1): ignored
    ctx.check(lib.nhp_cont_baseline_prior(ctx.h, G, _ptr(L3), 0.0))
    # a new grid size drops the prior
    x2 = np.linspace(0.0, T, G + 2)
    ctx.check(lib.nhp_cont_baseline_grid(ctx.h, x2.size, _ptr(x2), _ptr(_f64(np.ones(K * x2.size)))))
    _resample_parents(ctx, d, 2, 0, None, False)
    assert run() == STATE
    # the attempt limit: angle uniforms of 0 keep theta at the rejected end of the bracket
    proc._push(ctx)
    proc.baseline.push_prior(ctx)
    _resample_parents(ctx, d, 2, 0, None, False)
    z, u = np.full(K * G, 30.0), np.random.default_rng(84).random(K * sr.NU)
    u.reshape(K, sr.NU)[:, 1] = 0.25
    u.reshape(K, sr.NU)[:, 2:] = 0.0
    assert run(z, u) == NUMERIC
    assert b"maximum attempts" in lib.nhp_last_error(ctx.h)
    np.testing.assert_array_equal(get(), lam.ravel())
    # the context is unchanged: the same parents still serve a successful update
    z, u = draws(K, G, 85)
    ctx.check(run(_f64(z), _f64(u)))
    assert not np.array_equal(get(), lam.ravel())
    # a zero curve value
    lam0 = lam.copy()
    lam0[1, 3] = 0.0
    proc.baseline.lam_grid = lam0
    proc._push(ctx)
    proc.baseline.push_prior(ctx)
    _resample_parents(ctx, d, 2, 0, None, False)
    assert run() == NUMERIC
    np.testing.assert_array_equal(get(), lam0.ravel())
    # the Gibbs sweep without a prior still refuses the network process up front
    proc.baseline.lam_grid = lam.copy()
    proc._push(ctx)
    hy = _hyper(proc)
    assert lib.nhp_cont_gibbs_sweep(ctx.h, d.h, d.h, 1, 0, float(T), _ptr(hy), hy.size, 1.0, 1.0) == -6
    d.free()
