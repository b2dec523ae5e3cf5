"""The discrete Gibbs chain on the device (nhp_disc_gibbs_sweep + nhp_disc_trace_*), checked stage by stage against the oracle.

A sweep is: parent counts (Philox: SEED, uniform index, counter), conjugate draws from the counts left on the device, table refresh
(bump table, compact parent lists) on the device, and for a network process the in-place adjacency sweep (counter + 2^40), another
refresh and the Beta draw of rho.  The conjugate and Beta draws are not reproducible on the host; everything else is, given the
values read back: the counts and the adjacency sweep use Philox uniforms (synth.philox_uniform)."""
import ctypes

import numpy as np
import pytest
from scipy import stats

import nhp_b200 as nhp
import oracle_ffi as orc
import synth
from nhp_b200 import _lib
from nhp_b200 import discrete as D
from nhp_b200.core import Context, _fmat, _ptr

pytestmark = pytest.mark.gpu

SEED, STEPS, RHO0 = 777, 6, 0.15


def make(N, T, B, L, seed, network=True, density=RHO0, rho=RHO0, wscale=0.6, rate=0.1):
    rng = np.random.default_rng(seed)
    lam0 = rng.uniform(0.5, 1.5, N) * rate
    W = rng.uniform(0.1, 1.0, (N, N)) * wscale / N
    theta = rng.dirichlet(np.ones(B), (N, N))
    data = rng.poisson(rate, (N, T)).astype(np.int64)
    base, imp, wts = D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W)
    if not network:
        return D.DiscreteStandardHawkesProcess(base, imp, wts), data
    A = (rng.random((N, N)) < density).astype(np.float64)
    return D.DiscreteNetworkHawkesProcess(base, imp, wts, A, nhp.BernoulliNetworkModel(rho, N)), data


def hyper(proc):
    b, w, imp = proc.baseline, proc.weights, proc.impulses
    return np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)


def read_params(ctx, N, B, net=True):
    """nhp_disc_params_get + nhp_disc_network_get: ([p, c] matrices, theta [p, c, b]), rho."""
    l0, W, th = np.empty(N), np.empty(N * N), np.empty(N * N * B)
    A = np.empty(N * N) if net else None
    ctx.check(ctx.lib.nhp_disc_params_get(ctx.h, _ptr(l0), _ptr(W), _ptr(A), _ptr(th)))
    rho = ctypes.c_double()
    ctx.check(ctx.lib.nhp_disc_network_get(ctx.h, ctypes.byref(rho)))
    unf = lambda v: None if v is None else v.reshape(N, N).T.copy()
    return dict(lambda0=l0, W=unf(W), A=unf(A), theta=th.reshape(B, N, N).transpose(2, 1, 0).copy()), rho.value


def assert_params_equal(P, Q, keys=("lambda0", "W", "A", "theta"), msg=""):
    for k in keys:
        if P[k] is not None or Q[k] is not None:
            np.testing.assert_array_equal(P[k], Q[k], err_msg=f"{k} {msg}")


def device_counts(ctx, d, N, B, seed=0, counter=0, u=None):
    """nhp_disc_gibbs_counts with the context's current tables -> counts[c, k]."""
    counts = np.empty(N * (1 + N * B))
    ctx.check(ctx.lib.nhp_disc_gibbs_counts(ctx.h, d.h, int(seed), int(counter), _ptr(u), 0 if u is None else u.size, _ptr(counts)))
    return counts.reshape(1 + N * B, N).T.copy()


def push(ctx, P, B, dt=1.0):
    N = P["lambda0"].size
    th = np.ascontiguousarray(P["theta"].transpose(2, 1, 0)).ravel()
    A = None if P["A"] is None else _fmat(P["A"])
    ctx.check(ctx.lib.nhp_disc_params_set(ctx.h, N, B, _ptr(P["lambda0"]), _ptr(_fmat(P["W"])), _ptr(A), _ptr(th), dt))


@pytest.mark.parametrize("env", [{}, {"NHP_DISC_ADJ_STREAM": "0"}, {"NHP_DISC_WARP": "0"}], ids=["default", "adj_per_column", "gibbs_block"])
def test_chained_disc_sweeps_match_oracle_stage_by_stage(monkeypatch, env):
    """Six chained sweeps on one handle.  Before step s the device holds P_s, rho_s (read back); then
    - the parent counts with the tables the previous sweep left == oracle's given philox_uniform(SEED, event, s);
    - after the sweep, A_{s+1} == oracle's adjacency sweep with the freshly drawn lambda0, W, theta, the old A_s and rho_s, given
      philox_uniform(SEED, p + N c, s + 2^40);
    - the trace holds every P_{s+1} and rho_{s+1} bit for bit."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    N, T, B, L = 12, 3000, 3, 5
    proc, data = make(N, T, B, L, 5)
    ctx = proc._ctx()
    lib = ctx.lib
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    conv = orc.disc_convolve(data, orc.disc_basis(L, B))
    proc._push(ctx)
    ctx.check(lib.nhp_disc_network_set(ctx.h, RHO0))
    hy = hyper(proc)
    kk = (np.arange(N)[:, None] + N * np.arange(N)[None, :]).astype(np.uint64)
    nev = int(data.sum())
    samples, sparse_steps = [], 0
    ctx.check(lib.nhp_disc_trace_begin(ctx.h, STEPS))
    try:
        for s in range(STEPS):
            P, rho = read_params(ctx, N, B)
            if s == 0:
                assert rho == RHO0
            sparse_steps += s > 0 and np.count_nonzero(P["A"] * P["W"]) <= 0.5 * N * N  # lists built on the device
            om = orc.Disc(P["lambda0"], P["W"], P["theta"], dt=1.0, A=P["A"])
            u = synth.philox_uniform(SEED, np.arange(nev, dtype=np.uint64), s)
            assert np.count_nonzero(device_counts(ctx, d, N, B, SEED, s) != om.gibbs_counts(data, conv, u)) == 0, s
            ctx.check(lib.nhp_disc_gibbs_sweep(ctx.h, d.h, SEED, s, _ptr(hy), 5, 1.0, 1.0))
            P1, rho1 = read_params(ctx, N, B)
            A_ref = orc.Disc(P1["lambda0"], P1["W"], P1["theta"], dt=1.0, A=P["A"]).resample_adjacency(
                P["A"], np.full((N, N), rho), data, conv, synth.philox_uniform(SEED, kk, s + 2 ** 40))
            np.testing.assert_array_equal(P1["A"], A_ref, err_msg=f"step {s}")
            np.testing.assert_allclose(P1["theta"].sum(axis=2), 1.0, rtol=1e-12)
            assert 0.0 < rho1 < 1.0 and rho1 != rho
            samples.append((P1, rho1))
        assert sparse_steps >= 1  # device-built compact lists served a parent sweep
        cnt, cap = ctypes.c_int64(), ctypes.c_int64()
        ctx.check(lib.nhp_disc_trace_count(ctx.h, ctypes.byref(cnt), ctypes.byref(cap)))
        assert cnt.value == cap.value == STEPS
        trho, tl0, tW, tA, tth = np.empty(STEPS), np.empty((STEPS, N)), np.empty((STEPS, N * N)), np.empty((STEPS, N * N)), np.empty((STEPS, N * N * B))
        ctx.check(lib.nhp_disc_trace_read(ctx.h, 0, STEPS, _ptr(trho), _ptr(tl0), _ptr(tW), _ptr(tA), _ptr(tth)))
        for s, (P1, rho1) in enumerate(samples):
            assert trho[s] == rho1
            unf = lambda v: v.reshape(N, N).T
            assert_params_equal(P1, dict(lambda0=tl0[s], W=unf(tW[s]), A=unf(tA[s]), theta=tth[s].reshape(B, N, N).transpose(2, 1, 0)), msg=f"sample {s}")
    finally:
        ctx.check(lib.nhp_disc_trace_free(ctx.h))
        d.free()


def test_device_built_tables_equal_host_pushed_ones():
    """After an in-place adjacency sweep the tables are rebuilt on the device.  The parent counts given u must equal those after an
    nhp_disc_params_set of the same values read back, and the oracle's.  The two sweeps cross the 0.5 density limit in both
    directions: a dense A (no lists) thins out under a small link probability, a sparse A (lists) fills up under one near 1."""
    N, T, B, L = 16, 2500, 4, 6
    proc, data = make(N, T, B, L, 9, wscale=0.05)  # weak evidence: the link probability decides
    ctx = proc._ctx()
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    conv = orc.disc_convolve(data, orc.disc_basis(L, B))
    u = np.random.default_rng(3).random(int(data.sum()))
    rng = np.random.default_rng(4)
    for density, rho in ((0.6, 0.02), (0.3, 0.98)):
        proc.adjacency_matrix = (rng.random((N, N)) < density).astype(np.float64)
        proc._push(ctx)
        ctx.check(ctx.lib.nhp_disc_network_set(ctx.h, rho))
        ctx.check(ctx.lib.nhp_disc_resample_adjacency_dev(ctx.h, d.h, -1.0, SEED, int(density * 10)))
        P, _ = read_params(ctx, N, B)
        assert (np.count_nonzero(P["A"]) > 0.5 * N * N) != (density > 0.5), density  # the sweep crossed the density limit
        c_dev = device_counts(ctx, d, N, B, u=u)
        push(ctx, P, B)
        c_host = device_counts(ctx, d, N, B, u=u)
        ref = orc.Disc(P["lambda0"], P["W"], P["theta"], dt=1.0, A=P["A"]).gibbs_counts(data, conv, u)
        assert np.count_nonzero(c_dev != c_host) == 0 and np.count_nonzero(c_dev != ref) == 0, density
    d.free()


@pytest.mark.parametrize("network", [True, False])
@pytest.mark.parametrize("counter", [0, 5])
def test_one_sweep_equals_resample_on_device(network, counter):
    """From the same state and (seed, counter), nhp_disc_gibbs_sweep and discrete.resample_on_device_ (counts, device draws with
    the host's Mn, host round trip of the parameters, adjacency sweep with the N x N link probability) give the same lambda0, W,
    theta and A bit for bit; rho is drawn differently by design."""
    N, T, B, L = 20, 3000, 4, 8
    ref, data = make(N, T, B, L, 21, network=network, density=0.3, rho=0.3)
    ctx = ref._ctx()
    d = ref.upload(data)
    D.convolve(ref, d, export=False)
    ref._push(ctx)
    P0, _ = read_params(ctx, N, B, network)
    D.resample_on_device_(ref, d, seed=SEED, counter=counter)
    push(ctx, P0, B)
    ctx.check(ctx.lib.nhp_disc_network_set(ctx.h, 0.3))
    hy = hyper(ref)
    ctx.check(ctx.lib.nhp_disc_gibbs_sweep(ctx.h, d.h, SEED, counter, _ptr(hy), 5, 1.0 if network else 0.0, 1.0 if network else 0.0))
    P1, _ = read_params(ctx, N, B, network)
    Q = dict(lambda0=ref.baseline.lam, W=ref.weights.W, A=ref.adjacency_matrix, theta=ref.impulses.theta)
    assert_params_equal(P1, Q)
    if network:
        assert not np.array_equal(P1["A"], P0["A"])
    d.free()


def test_rho_draw_is_the_beta_posterior():
    """Rewound to the same pushed state before every sweep (different counters), rho given the A' of that sweep is
    Beta(alpha + sum A', beta + N^2 - sum A'): its CDF values are uniform (Kolmogorov-Smirnov)."""
    N, T, B, L = 6, 800, 2, 4
    proc, data = make(N, T, B, L, 33, density=0.4, rho=0.4, wscale=0.3)
    ctx = proc._ctx()
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    proc._push(ctx)
    P0, _ = read_params(ctx, N, B)
    hy = hyper(proc)
    alpha, beta = 2.0, 3.0
    R = 400
    pit, sums = np.empty(R), np.empty(R)
    for r in range(R):
        push(ctx, P0, B)
        ctx.check(ctx.lib.nhp_disc_network_set(ctx.h, 0.4))
        ctx.check(ctx.lib.nhp_disc_gibbs_sweep(ctx.h, d.h, SEED, 1000 + r, _ptr(hy), 5, alpha, beta))
        P, rho = read_params(ctx, N, B)
        sums[r] = P["A"].sum()
        pit[r] = stats.beta.cdf(rho, alpha + sums[r], beta + N * N - sums[r])
    assert np.unique(sums).size > 3  # the sweeps produced different A'
    assert stats.kstest(pit, "uniform").pvalue > 1e-3
    d.free()


def test_standard_process_chain_matches_the_host_chain():
    """mcmc_device_ of a standard process: its posterior means of lambda0 and W agree with the host chain (mcmc_, NumPy draws)
    within Monte Carlo error; theta rows sum to one; the process holds the last sample."""
    N, T, B, L = 4, 6000, 3, 5
    dev, data = make(N, T, B, L, 41, network=False, wscale=0.8, rate=0.15)
    host, _ = make(N, T, B, L, 41, network=False, wscale=0.8, rate=0.15)
    d = dev.upload(data)
    steps, burn = 400, 100
    res = D.mcmc_device_(dev, d, nsteps=steps, seed=3)
    assert len(res.samples) == steps and all(np.all(np.isfinite(x)) for x in res.samples)
    np.testing.assert_array_equal(res.samples[-1], dev.params())
    np.testing.assert_allclose(dev.impulses.theta.sum(axis=2), 1.0, rtol=1e-12)
    hres = D.mcmc_(host, d, nsteps=steps, seed=4)
    xd, xh = np.array(res.samples[burn:]), np.array(hres.samples[burn:])
    # lambda0 and W (sum over b of W .* theta) from the samples
    fd = np.concatenate([xd[:, :N], xd[:, N:].reshape(-1, B, N * N).sum(axis=1)], axis=1)
    fh = np.concatenate([xh[:, :N], xh[:, N:].reshape(-1, B, N * N).sum(axis=1)], axis=1)
    n_eff = (steps - burn) / 10.0  # conservative: neighbouring Gibbs samples are correlated
    se = np.sqrt((fd.var(axis=0) + fh.var(axis=0)) / n_eff)
    assert np.all(np.abs(fd.mean(axis=0) - fh.mean(axis=0)) < 5 * se + 1e-9)


def rc_of(fn, *args):
    return int(fn(*args))


def test_trace_and_sweep_contracts():
    """The trace stops at its capacity, _push refuses a changed model, _read rejects samples it does not hold; the sweep refuses a
    time-sharded handle (UNSUPPORTED), a wrong hyper-parameter count (INVALID), a context without parameters or data without its
    convolution (STATE), each before changing anything."""
    N, T, B, L = 8, 1500, 3, 5
    proc, data = make(N, T, B, L, 51)
    ctx = Context()
    proc.ctx = ctx
    lib = ctx.lib
    d = proc.upload(data)
    hy = hyper(proc)
    # no parameters yet, then no convolution
    assert rc_of(lib.nhp_disc_gibbs_sweep, ctx.h, d.h, SEED, 0, _ptr(hy), 5, 1.0, 1.0) == _lib.NHP_ERR_STATE
    proc._push(ctx)
    ctx.check(lib.nhp_disc_network_set(ctx.h, RHO0))
    P0, rho0 = read_params(ctx, N, B)
    assert rc_of(lib.nhp_disc_gibbs_sweep, ctx.h, d.h, SEED, 0, _ptr(hy), 5, 1.0, 1.0) == _lib.NHP_ERR_STATE
    D.convolve(proc, d, export=False)
    assert rc_of(lib.nhp_disc_gibbs_sweep, ctx.h, d.h, SEED, 0, _ptr(hy), 4, 1.0, 1.0) == _lib.NHP_ERR_INVALID
    sh = D.DiscreteData(ctx, data[:, 100:], t_halo=L)
    D.convolve(proc, sh, export=False)
    assert rc_of(lib.nhp_disc_gibbs_sweep, ctx.h, sh.h, SEED, 0, _ptr(hy), 5, 1.0, 1.0) == _lib.NHP_ERR_UNSUPPORTED
    assert rc_of(lib.nhp_disc_resample_adjacency_dev, ctx.h, sh.h, -1.0, SEED, 0) == _lib.NHP_ERR_UNSUPPORTED
    P, rho = read_params(ctx, N, B)
    assert_params_equal(P, P0)
    assert rho == rho0
    # trace: capacity 2, three sweeps
    ctx.check(lib.nhp_disc_trace_begin(ctx.h, 2))
    for s in range(3):
        ctx.check(lib.nhp_disc_gibbs_sweep(ctx.h, d.h, SEED, s, _ptr(hy), 5, 1.0, 1.0))
    cnt, cap = ctypes.c_int64(), ctypes.c_int64()
    ctx.check(lib.nhp_disc_trace_count(ctx.h, ctypes.byref(cnt), ctypes.byref(cap)))
    assert (cnt.value, cap.value) == (2, 2)
    assert rc_of(lib.nhp_disc_trace_push, ctx.h) == _lib.NHP_ERR_STATE
    buf = np.empty(N * N * B * 4)
    assert rc_of(lib.nhp_disc_trace_read, ctx.h, 1, 2, None, _ptr(buf), None, None, None) == _lib.NHP_ERR_INVALID
    assert rc_of(lib.nhp_disc_trace_read, ctx.h, -1, 1, None, _ptr(buf), None, None, None) == _lib.NHP_ERR_INVALID
    ctx.check(lib.nhp_disc_trace_read(ctx.h, 1, 1, None, _ptr(buf), None, None, None))
    # a model without A, or with another B, since _begin
    ctx.check(lib.nhp_disc_trace_begin(ctx.h, 4))
    ctx.check(lib.nhp_disc_trace_push(ctx.h))
    Q, _ = read_params(ctx, N, B)
    push(ctx, dict(Q, A=None), B)
    assert rc_of(lib.nhp_disc_trace_push, ctx.h) == _lib.NHP_ERR_STATE
    push(ctx, dict(Q, theta=np.full((N, N, B + 1), 1.0 / (B + 1))), B + 1)
    assert rc_of(lib.nhp_disc_trace_push, ctx.h) == _lib.NHP_ERR_STATE
    push(ctx, Q, B)
    ctx.check(lib.nhp_disc_trace_push(ctx.h))
    ctx.check(lib.nhp_disc_trace_count(ctx.h, ctypes.byref(cnt), None))
    assert cnt.value == 2
    ctx.check(lib.nhp_disc_trace_free(ctx.h))
    sh.free()
    d.free()


def test_network_chain_runs_and_keeps_the_last_sample():
    """mcmc_device_ of a Bernoulli network process: samples in the order of params(process), the process holds the last one."""
    N, T, B, L = 10, 2000, 3, 5
    proc, data = make(N, T, B, L, 61)
    res = D.mcmc_device_(proc, data, nsteps=5, seed=2)
    assert len(res.samples) == 5 and res.samples[0].size == 1 + N + N * N * (2 + B)
    np.testing.assert_array_equal(res.samples[-1], proc.params())
    assert 0.0 < proc.network.rho < 1.0
