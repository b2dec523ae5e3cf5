"""The adjacency sampler and the structure log-likelihood of network processes with LogGaussianCoxProcess baselines
(csrc/cont_adjacency.cu, csrc/cont_baseline.cu; continuous.jl:444-519 with total_intensity reading lambda0_c(t_i)).  The decisions
given u must be those of the sequential sweep of tests/grid_reference.py, for every form of the sweep."""
import ctypes

import numpy as np
import pytest

import grid_reference as gr
import nhp_b200 as nhp
import oracle_ffi as orc
import synth
from nhp_b200.core import _f64, _ptr

pytestmark = pytest.mark.gpu


def curves(K, T, seed, G=41, spread=0.3, dip=None, mean=1.0, width=1):
    """Curves with the given mean, +-spread variation, and optionally a dip to `dip` times the mean over `width` grid points inside
    [0, T]."""
    rng = np.random.default_rng(seed)
    x = np.linspace(0.0, T, G)
    lam = mean * (1.0 + spread * np.sin(2 * np.pi * rng.uniform(0.5, 3.0, (K, 1)) * x[None, :] / T + rng.uniform(0, 6, (K, 1))))
    if dip is not None:
        for k in range(K):
            g = rng.integers(2, G - 1 - width)
            lam[k, g:g + width] = mean * dip
    return x, lam


def network(kind, K, seed, rho, x, lam, dtmax=1.0, wmax=None):
    wmax = 1.5 / K if wmax is None else wmax
    if kind == "ln":
        lam0, W, p1, p2, A = synth.ln_params(K, seed, wmax=wmax, density=0.5)
        imp = nhp.LogitNormalImpulseResponse(p1, p2, dtmax)
    else:
        lam0, W, p1, A = synth.exp_params(K, seed, wmax=wmax, density=0.5)
        p2 = None
        imp = nhp.ExponentialImpulseResponse(p1, dtmax=dtmax)
    base = nhp.HomogeneousProcess(lam0) if x is None else nhp.LogGaussianCoxProcess(x, lam)
    proc = nhp.ContinuousNetworkHawkesProcess(base, imp, nhp.DenseWeightModel(W), A, nhp.BernoulliNetworkModel(rho, K))
    ref = gr.Model(1 if kind == "ln" else 0, lam0, W, p1, p2, A=A, dtmax=dtmax, x=x, lam=lam)
    return proc, ref


def run_both(proc, ref, data, rho, u, A0, **kw):
    t, nodes, T = data
    proc.adjacency_matrix = A0.copy()
    A_gpu = nhp.resample_adjacency_matrix_(proc, data, u=u, **kw).copy()
    A_ref = ref.resample_adjacency(A0, rho, t, nodes, T, u, kw.get("col_begin", 0), kw.get("col_stride", 1))
    return A_gpu, A_ref


@pytest.mark.parametrize("kind,dtmax,env", [
    ("ln", 1.0, {}),                                              # 18-byte LogitNormal payload
    ("ln", 1.0, {"NHP_ADJ_PRE": "0"}),                            # lag payload
    ("ln", 1.0, {"NHP_ADJ_CHUNK": "64"}),                         # thread-block clusters
    ("ln", 1.0, {"NHP_ADJ_CHUNK": "7", "NHP_ADJ_CLUSTER": "0"}),  # single-CTA streaming form
    ("ln", 1.0, {"NHP_ADJ_CACHE": "0"}),                          # uncached fallback
    ("exp", 1.0, {}),
    ("exp", np.inf, {}),                                          # cut-off horizon from the curves' minimum
    ("exp", 1.0, {"NHP_ADJ_CHUNK": "64"}),
    ("exp", 1.0, {"NHP_ADJ_CHUNK": "7", "NHP_ADJ_CLUSTER": "0"}),
    ("exp", 1.0, {"NHP_ADJ_CACHE": "0"}),
    ("exp", np.inf, {"NHP_ADJ_CHUNK": "64"}),
    ("ln", 1.0, {"NHP_ADJ_PRE": "0", "NHP_ADJ_CHUNK": "64"}),     # lag payload across a cluster
    ("ln", 1.0, {"NHP_ADJ_S0": "1"}),                             # batches grow from one bucket with the observed flip rate
    ("ln", 1.0, {"NHP_ADJ_S0": "4", "NHP_ADJ_CHUNK": "64"}),
])
def test_sweep_with_curves_matches_reference(monkeypatch, kind, dtmax, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    K, rho = 13, 0.4
    n, rate = (1500, 20.0) if dtmax == np.inf else (4000, 60.0)
    t, nodes, T = synth.poisson_stream(n, K, rate, 31)
    x, lam = curves(K, T, 32, spread=0.3)
    proc, ref = network(kind, K, 33, rho, x, lam, dtmax=dtmax)
    A0 = proc.adjacency_matrix.copy()
    bad = 0
    for rep in range(2):
        u = np.random.default_rng(40 + rep).random((K, K))
        A_gpu, A_ref = run_both(proc, ref, (t, nodes, T), rho, u, A0)
        bad += int(np.count_nonzero(A_gpu != A_ref))
    assert bad == 0
    if env.get("NHP_ADJ_CACHE") != "0":
        info = nhp.adjacency_info()
        assert info["steps"] == K * K and info["pairs"] > 0
        if "NHP_ADJ_CHUNK" in env:
            assert info["virtual_columns"] > K
        if "NHP_ADJ_CLUSTER" in env:
            assert info["cluster"] == 0


@pytest.mark.parametrize("chunk", [None, 64])
def test_deep_dips_below_the_flips_restart_but_stay_exact(monkeypatch, chunk):
    """Curves that fall to 1e-3 of their mean inside every column, with single contributions far above that minimum: the
    certification bound (taken from the column minimum) is loose, batches restart, and the decisions are still the sequential ones."""
    if chunk is not None:
        monkeypatch.setenv("NHP_ADJ_CHUNK", str(chunk))
    K, n, rho = 60, 9000, 0.5
    t, nodes, T = synth.poisson_stream(n, K, 12.0, 77)
    x, lam = curves(K, T, 78, G=61, spread=0.3, dip=1e-3, width=3)
    proc, ref = network("ln", K, 79, rho, x, lam, wmax=0.4)
    A0 = proc.adjacency_matrix.copy()
    rates = np.array([np.interp(t[nodes == c + 1], x, lam[c]).min() for c in range(K)])
    assert np.median(rates) < 2e-3  # the columns do see the dips
    u = np.random.default_rng(80).random((K, K))
    A_gpu, A_ref = run_both(proc, ref, (t, nodes, T), rho, u, A0)
    assert int(np.count_nonzero(A_gpu != A_ref)) == 0
    assert int(np.count_nonzero(A_ref != A0)) > 5 * K
    info = nhp.adjacency_info()
    assert info["batches"] > 0 and info["recomputed_steps"] > 0


def test_column_partition_and_config4_shape():
    """cfg4's shape (K = 1000, rho = 0.05, mean window 64) with curves, on every 50th column through the column-partition entry
    point, and a small partition (col_begin = 1, col_stride = 3)."""
    K, n, rho = 1000, 40000, 0.05
    t, nodes, T = synth.poisson_stream(n, K, 64.0, 4)
    x, lam = curves(K, T, 5, G=17)
    lam0, W, mu, tau, A0 = synth.ln_params(K, 2, wmax=0.5 / (K * rho), density=rho)
    proc = nhp.ContinuousNetworkHawkesProcess(nhp.LogGaussianCoxProcess(x, lam), nhp.LogitNormalImpulseResponse(mu, tau, 1.0), nhp.DenseWeightModel(W),
                                              A0.copy(), nhp.BernoulliNetworkModel(rho, K))
    ref = gr.Model(1, lam0, W, mu, tau, A=A0, dtmax=1.0, x=x, lam=lam)
    u = np.random.default_rng(6).random((K, K))
    A_gpu, A_ref = run_both(proc, ref, (t, nodes, T), rho, u, A0, col_begin=3, col_stride=50)
    np.testing.assert_array_equal(A_gpu, A_ref)
    other = [c for c in range(K) if c % 50 != 3]
    np.testing.assert_array_equal(A_gpu[:, other], A0[:, other])
    K, rho = 11, 0.3
    t, nodes, T = synth.poisson_stream(3000, K, 50.0, 7)
    x, lam = curves(K, T, 8)
    proc, ref = network("ln", K, 9, rho, x, lam)
    A0 = proc.adjacency_matrix.copy()
    u = np.random.default_rng(10).random((K, K))
    A_gpu, A_ref = run_both(proc, ref, (t, nodes, T), rho, u, A0, col_begin=1, col_stride=3)
    np.testing.assert_array_equal(A_gpu, A_ref)


def test_constant_curves_are_the_homogeneous_sweep():
    K, rho = 12, 0.4
    t, nodes, T = synth.poisson_stream(3000, K, 50.0, 12)
    lam0, W, mu, tau, A0 = synth.ln_params(K, 13, wmax=1.5 / K, density=0.5)
    lam0 = np.random.default_rng(14).uniform(0.5, 1.5, K)
    x = np.linspace(0.0, T, 9)
    mk = lambda base: nhp.ContinuousNetworkHawkesProcess(base, nhp.LogitNormalImpulseResponse(mu, tau, 1.0), nhp.DenseWeightModel(W), A0.copy(),
                                                         nhp.BernoulliNetworkModel(rho, K))
    pg, ph = mk(nhp.LogGaussianCoxProcess(x, np.repeat(lam0[:, None], x.size, axis=1))), mk(nhp.HomogeneousProcess(lam0))
    om = orc.Cont(1, lam0, W, mu, tau, A=A0, dtmax=1.0)
    for rep in range(3):
        u = np.random.default_rng(15 + rep).random((K, K))
        Ag = nhp.resample_adjacency_matrix_(pg, (t, nodes, T), u=u).copy()
        Ah = nhp.resample_adjacency_matrix_(ph, (t, nodes, T), u=u).copy()
        pg.adjacency_matrix, ph.adjacency_matrix = A0.copy(), A0.copy()
        np.testing.assert_array_equal(Ag, Ah)
        np.testing.assert_array_equal(Ag, om.resample_adjacency(A0, np.full((K, K), rho), t, nodes, T, u))


@pytest.mark.parametrize("kind,pre,chunk", [("ln", "1", None), ("ln", "0", 64), ("exp", "1", 7), ("ln", "1", 64)])
def test_structure_loglikelihood_with_curves(monkeypatch, kind, pre, chunk):
    """Once the handle carries the pair structure, the log-likelihood with curves streams the active buckets (k_adj_loglik) from
    the per-event rates: equal to the window sweep and to the reference, for every payload; nhp_cont_loglik_dist at one rank too."""
    monkeypatch.setenv("NHP_ADJ_PRE", pre)
    if chunk is not None:
        monkeypatch.setenv("NHP_ADJ_CHUNK", str(chunk))
    K, n, rho = 23, 5000, 0.15
    t, nodes, T = synth.poisson_stream(n, K, 70.0, 21)
    x, lam = curves(K, T, 22, spread=0.3)
    proc, ref = network(kind, K, 5, rho, x, lam, wmax=2.0 / (K * rho))
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    proc._push(ctx)
    ctx.check(ctx.lib.nhp_cont_resample_adjacency_dev(ctx.h, d.h, rho, 5, 1, 0, 1, 1))  # builds the structure, changes A
    nhp.pull_params_(proc, ctx)
    A1 = proc.adjacency_matrix.copy()
    assert 0 < np.count_nonzero(A1 * proc.weights.W) <= 0.25 * K * K
    ll = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll)))          # structure path
    ll_struct = ll.value
    ctx.check(ctx.lib.nhp_cont_loglik_dist(ctx.h, d.h, d.h, 0, ctypes.byref(ll)))
    ll_dist = ll.value
    monkeypatch.setenv("NHP_ADJ_LOGLIK", "0")
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll)))          # window sweep
    ll_window = ll.value
    ref.A = A1
    want = ref.loglik(t, nodes, T)
    assert ll_struct == pytest.approx(ll_window, rel=1e-12)
    assert ll_struct == pytest.approx(want, rel=1e-10)
    assert ll_dist == pytest.approx(ll_struct, rel=1e-12)
    d.free()


def test_device_resident_sweep_equals_host_argument_sweep():
    K, n, rho, seed, counter = 12, 3000, 0.3, 77, 5
    t, nodes, T = synth.poisson_stream(n, K, 50.0, 12)
    x, lam = curves(K, T, 13)
    proc, ref = network("ln", K, 3, rho, x, lam)
    A0 = proc.adjacency_matrix.copy()
    kk = (np.arange(K)[:, None] + K * np.arange(K)[None, :]).astype(np.uint64)
    u = synth.philox_uniform(seed, kk, counter)
    A_host = nhp.resample_adjacency_matrix_(proc, (t, nodes, T), u=u).copy()
    np.testing.assert_array_equal(A_host, ref.resample_adjacency(A0, rho, t, nodes, T, u))
    proc.adjacency_matrix = A0.copy()
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    proc._push(ctx)
    ctx.check(ctx.lib.nhp_cont_resample_adjacency_dev(ctx.h, d.h, rho, seed, counter, 0, 1, 1))
    nhp.pull_params_(proc, ctx)
    np.testing.assert_array_equal(proc.adjacency_matrix, A_host)
    np.testing.assert_array_equal(proc.baseline.lam_grid, lam)  # the host keeps its curves
    d.free()


def test_curve_versions_on_one_handle():
    """Curves 1, then curves 2, then a homogeneous lambda0, on one events handle: every sweep reads the rates and minima of the
    baseline it was given."""
    K, n, rho = 10, 3000, 0.45
    t, nodes, T = synth.poisson_stream(n, K, 40.0, 41)
    x, lam1 = curves(K, T, 42, spread=0.3, dip=0.01)
    _, lam2 = curves(K, T, 43, spread=0.6, mean=2.0)
    proc, ref = network("ln", K, 44, rho, x, lam1)
    d = proc.upload((t, nodes, T))
    A0 = proc.adjacency_matrix.copy()
    lam0 = ref.lambda0.copy()
    for step, base in enumerate([(x, lam1), (x, lam2), None, (x, lam1)]):
        if base is None:
            proc.baseline = nhp.HomogeneousProcess(lam0)
            ref.x = ref.lam = None
        else:
            proc.baseline = nhp.LogGaussianCoxProcess(*base)
            ref.x, ref.lam = base
        u = np.random.default_rng(50 + step).random((K, K))
        proc.adjacency_matrix = A0.copy()
        A_gpu = nhp.resample_adjacency_matrix_(proc, d, u=u).copy()
        np.testing.assert_array_equal(A_gpu, ref.resample_adjacency(A0, rho, t, nodes, T, u))
    d.free()


def test_cutoff_horizon_after_conjugate_draws_keeps_the_curves_minimum():
    K, n = 6, 2000
    t, nodes, T = synth.poisson_stream(n, K, 20.0, 61)
    x, lam = curves(K, T, 62, dip=0.02)
    proc, _ = network("exp", K, 63, 0.5, x, lam, dtmax=np.inf)
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    proc._push(ctx)
    nhp.resample_parents(proc, d, seed=1, counter=0, export=False)
    hy = nhp.continuous._hyper(proc)
    ctx.check(ctx.lib.nhp_cont_resample_params(ctx.h, d.h, 1, 0, float(T), _ptr(hy), hy.size, 1))
    h = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_horizon(ctx.h, n, 0, ctypes.byref(h)))
    nhp.pull_params_(proc, ctx)
    W, th, A = proc.weights.W, proc.impulses.theta, proc.adjacency_matrix
    act = A * W != 0.0
    want = np.log(n * np.max(np.abs(A * W * th)[act]) / (1e-14 * lam.min())) / th[act].min()
    assert h.value == pytest.approx(want, rel=1e-12)
    d.free()


def test_zero_rate_at_an_event_is_refused_before_anything_changes():
    K, rho = 5, 0.4
    t, nodes, T = synth.poisson_stream(1500, K, 30.0, 71)
    x, lam = curves(K, T, 72, G=21)
    lam[2, 5:8] = 0.0  # node 3 has no baseline over two grid cells that hold its events
    sel = (nodes == 3) & (t > x[5]) & (t < x[7])
    assert sel.any()
    proc, _ = network("ln", K, 73, rho, x, lam)
    A0 = proc.adjacency_matrix.copy()
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    with pytest.raises(nhp.NHPError):
        nhp.resample_adjacency_matrix_(proc, d, u=np.random.default_rng(1).random((K, K)))
    with pytest.raises(nhp.NHPError):
        ctx.check(ctx.lib.nhp_cont_resample_adjacency_dev(ctx.h, d.h, rho, 1, 1, 0, 1, 1))
    np.testing.assert_array_equal(proc.adjacency_matrix, A0)
    nhp.pull_params_(proc, ctx)
    np.testing.assert_array_equal(proc.adjacency_matrix, A0)
    # columns that do not hold those events can still be swept
    u = np.random.default_rng(2).random((K, K))
    A1 = nhp.resample_adjacency_matrix_(proc, d, u=u, col_begin=1, col_stride=2).copy()
    np.testing.assert_array_equal(A1[:, 0::2], A0[:, 0::2])
    d.free()


def test_device_gibbs_sweep_refuses_a_network_with_curves_up_front():
    K, rho = 6, 0.4
    t, nodes, T = synth.poisson_stream(2000, K, 30.0, 81)
    x, lam = curves(K, T, 82)
    proc, _ = network("ln", K, 83, rho, x, lam)
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    proc._push(ctx)
    ctx.check(ctx.lib.nhp_cont_network_set(ctx.h, rho))
    get = lambda: [np.empty(K)] + [np.empty(K * K) for _ in range(4)]
    before = get()
    ctx.check(ctx.lib.nhp_cont_params_get(ctx.h, *[_ptr(a) for a in before]))
    hy = nhp.continuous._hyper(proc)
    rc = ctx.lib.nhp_cont_gibbs_sweep(ctx.h, d.h, d.h, 1, 0, float(T), _ptr(hy), hy.size, 1.0, 1.0)
    assert rc == -6  # NHP_ERR_UNSUPPORTED
    after = get()
    ctx.check(ctx.lib.nhp_cont_params_get(ctx.h, *[_ptr(a) for a in after]))
    for a, b in zip(before, after):
        np.testing.assert_array_equal(a, b)
    # no parent sweep ran: the slice likelihood still finds no parent assignment on the device
    ll = np.empty(K)
    assert ctx.lib.nhp_cont_baseline_loglik(ctx.h, d.h, x.size, _ptr(_f64(x)), _ptr(_f64(lam.ravel())), _ptr(ll)) == -4  # NHP_ERR_STATE
    d.free()


def test_gibbs_steps_of_a_network_with_curves():
    """resample_ (host draws) and mcmc_(device_draws=True) on a network LogGaussianCoxProcess model; mcmc_device_ refuses it."""
    K = 5
    x0 = np.linspace(0.0, 300.0, 31)
    base_lam = np.exp(0.3 * np.sin(x0[None, :] / 40.0 + np.arange(K)[:, None]))
    lam0, W, mu, tau, A = synth.ln_params(K, 91, wmax=0.3, density=0.6)
    gen = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(np.full(K, 1.0)), nhp.LogitNormalImpulseResponse(mu, tau, 1.0),
                                             nhp.DenseWeightModel(W), A.copy(), nhp.BernoulliNetworkModel(0.6, K))
    t, nodes, T = nhp.rand(gen, 300.0, np.random.default_rng(2))
    mk = lambda: nhp.ContinuousNetworkHawkesProcess(nhp.LogGaussianCoxProcess(x0, base_lam.copy()), nhp.LogitNormalImpulseResponse(mu.copy(), tau.copy(), 1.0),
                                                    nhp.DenseWeightModel(W.copy()), A.copy(), nhp.BernoulliNetworkModel(0.6, K))
    proc = mk()
    rng = np.random.default_rng(3)
    d = proc.upload((t, nodes, T))
    for s in range(3):
        x = nhp.resample_(proc, d, rng, seed=4, counter=s)
        assert np.all(np.isfinite(x))
    assert set(np.unique(proc.adjacency_matrix)) <= {0.0, 1.0}
    assert np.all(proc.baseline.lam_grid > 0) and not np.array_equal(proc.baseline.lam_grid, base_lam)
    proc = mk()
    res = nhp.mcmc_(proc, d, nsteps=4, seed=5, device_draws=True)
    assert len(res.samples) == 4 and all(np.all(np.isfinite(s)) for s in res.samples)
    assert set(np.unique(proc.adjacency_matrix)) <= {0.0, 1.0}
    assert np.all(proc.baseline.lam_grid > 0) and not np.array_equal(proc.baseline.lam_grid, base_lam)
    assert 0.0 < proc.network.rho < 1.0
    with pytest.raises(ValueError):
        nhp.mcmc_device_(mk(), d, nsteps=2)
    d.free()
