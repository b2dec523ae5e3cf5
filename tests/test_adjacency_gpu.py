"""GPU parity tests of the cached adjacency sampler (csrc/cont_adjacency.cu; continuous.jl:444-519): the virtual-column
structure, shared-memory intensities and speculative batches must give exactly the oracle's sequential sweep."""
import numpy as np
import pytest

import nhp_b200 as nhp
import oracle_ffi as orc
import synth
from test_cont_gpu import make_exp, make_ln

pytestmark = pytest.mark.gpu


def run_both(proc, om, data, rho, u, A0, **kw):
    t, nodes, T = data
    K = A0.shape[0]
    proc.adjacency_matrix = A0.copy()
    A_gpu = nhp.resample_adjacency_matrix_(proc, (t, nodes, T), u=u, **kw).copy()
    A_ref = om.resample_adjacency(A0, np.full((K, K), rho), t, nodes, T, u, kw.get("col_begin", 0), kw.get("col_stride", 1))
    return A_gpu, A_ref


@pytest.mark.parametrize("chunk", [None, 7, 64])   # 64: thread-block clusters of 4 (8) CTAs per column; 7: too many chunks for a cluster -> streaming form
@pytest.mark.parametrize("s0", [None, 1])
@pytest.mark.parametrize("kind,K,n,rate,rho", [("ln", 4, 900, 14.0, 0.5), ("ln", 37, 6000, 80.0, 0.2), ("exp", 6, 1500, 20.0, 0.4)])
def test_chunked_speculative_sweep_matches_oracle(monkeypatch, kind, K, n, rate, rho, chunk, s0):
    """Small chunks force several chunks per column (intensities streamed through global memory between batches); few nodes and
    long windows make most (event, parent) pairs repeat, so runs straddle 32-entry groups; rho near 1/2 makes links flip often."""
    if chunk is not None:
        monkeypatch.setenv("NHP_ADJ_CHUNK", str(chunk))
    if s0 is not None:
        monkeypatch.setenv("NHP_ADJ_S0", str(s0))
    t, nodes, T = synth.poisson_stream(n, K, rate, 50 + K)
    proc, om = (make_ln(K, 7, density=0.5, wmax=1.5 / K) if kind == "ln" else make_exp(K, 7, density=0.5, wmax=1.5 / K, dtmax=1.0))
    proc.network = nhp.BernoulliNetworkModel(rho, K)
    A0 = proc.adjacency_matrix.copy()
    bad = 0
    for rep in range(2):
        u = np.random.default_rng(300 + rep).random((K, K))
        A_gpu, A_ref = run_both(proc, om, (t, nodes, T), rho, u, A0)
        bad += int(np.count_nonzero(A_gpu != A_ref))
    assert bad == 0
    info = nhp.adjacency_info()
    assert info["steps"] == K * K and info["pairs"] > 0
    if chunk is not None:
        assert info["virtual_columns"] > K


@pytest.mark.parametrize("chunk", [None, 64])
def test_flips_larger_than_the_baseline_rate_are_certified_one_sidedly(monkeypatch, chunk):
    """lambda0 far below a single pair's contribution: every accepted flip moves intensities by more than lambda0 / 2, the case the
    first certification rule could only handle by ending the batch.  The one-sided bounds (S / (1 + on / lambda0) <= S' <= S (1 + off / lambda0))
    must still give exactly the sequential sweep (tests/test_certification_bound.py checks the bound itself)."""
    if chunk is not None:
        monkeypatch.setenv("NHP_ADJ_CHUNK", str(chunk))
    K, n, rho = 70, 9000, 0.5
    rng = np.random.default_rng(11)
    lam0 = np.full(K, 0.02)
    W, mu, tau = rng.uniform(0.0, 0.4, (K, K)), rng.uniform(-1.0, 1.0, (K, K)), rng.uniform(0.5, 2.0, (K, K))
    A0 = (rng.random((K, K)) < 0.5).astype(np.float64)
    t, nodes, T = synth.poisson_stream(n, K, 12.0, 77)
    proc = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.LogitNormalImpulseResponse(mu, tau, 1.0), nhp.DenseWeightModel(W), A0.copy(),
                                              nhp.BernoulliNetworkModel(rho, K))
    om = orc.Cont(1, lam0, W, mu, tau, A=A0, dtmax=1.0)
    bad = flips = 0
    for rep in range(2):
        u = np.random.default_rng(500 + rep).random((K, K))
        A_gpu, A_ref = run_both(proc, om, (t, nodes, T), rho, u, A0)
        bad += int(np.count_nonzero(A_gpu != A_ref))
        flips += int(np.count_nonzero(A_ref != A0))
    assert bad == 0
    assert flips > 10 * K  # the sweep really flips many links per column


@pytest.mark.parametrize("chunk,cluster", [(None, None), (64, None), (64, "0")])
def test_lag_payload_and_forced_streaming_form_match_oracle(monkeypatch, chunk, cluster):
    """LogitNormal with the 10-byte lag payload (what a tight memory budget selects) and the single-CTA streaming form forced on
    data that would fit a cluster."""
    monkeypatch.setenv("NHP_ADJ_PRE", "0")
    if chunk is not None:
        monkeypatch.setenv("NHP_ADJ_CHUNK", str(chunk))
    if cluster is not None:
        monkeypatch.setenv("NHP_ADJ_CLUSTER", cluster)
    K, n, rho = 11, 4000, 0.3
    t, nodes, T = synth.poisson_stream(n, K, 60.0, 77)
    proc, om = make_ln(K, 7, density=0.5, wmax=1.5 / K)
    proc.network = nhp.BernoulliNetworkModel(rho, K)
    A0 = proc.adjacency_matrix.copy()
    u = np.random.default_rng(5).random((K, K))
    A_gpu, A_ref = run_both(proc, om, (t, nodes, T), rho, u, A0)
    np.testing.assert_array_equal(A_gpu, A_ref)
    info = nhp.adjacency_info()
    assert info["bytes_per_pair"] == 10
    if cluster == "0":
        assert info["cluster"] == 0
    elif chunk is None:
        assert info["cluster"] == 1
    else:  # the smallest cluster whose chunks hold the largest column (~364 events at 64 per chunk)
        max_col = int(np.bincount(nodes, minlength=K).max())
        assert info["cluster"] == -(-max_col // 64) and 2 <= info["cluster"] <= 8


def test_uncached_fallback_matches_oracle(monkeypatch):
    monkeypatch.setenv("NHP_ADJ_CACHE", "0")
    K, n, rho = 9, 1500, 0.3
    t, nodes, T = synth.poisson_stream(n, K, 40.0, 30)
    proc, om = make_ln(K, 7, density=0.5, wmax=1.5 / K)
    proc.network = nhp.BernoulliNetworkModel(rho, K)
    A0 = proc.adjacency_matrix.copy()
    u = np.random.default_rng(1).random((K, K))
    A_gpu, A_ref = run_both(proc, om, (t, nodes, T), rho, u, A0)
    np.testing.assert_array_equal(A_gpu, A_ref)


def test_exponential_sampler_starting_from_an_empty_network():
    """ADVICE r1 (high): with A = 0 the sweeps' cut-off horizon collapses (no active link), but the sampler evaluates W h for
    links that are off: its horizon comes from all K^2 entries, so the data can switch links on."""
    K, rho = 5, 0.5
    proc, _ = make_exp(K, 7, density=0.5, wmax=1.0 / K)  # dtmax = Inf; branching ratio ~ 0.5 with every link on
    proc.adjacency_matrix = np.ones((K, K))
    t, nodes, T = nhp.rand(proc, 120.0, np.random.default_rng(3))  # excitation present in the data
    assert 300 < t.size < 5000
    proc.network = nhp.BernoulliNetworkModel(rho, K)
    A0 = np.zeros((K, K))
    om = orc.Cont(0, proc.baseline.lam, proc.weights.W, proc.impulses.theta, A=A0, dtmax=np.inf)
    u = np.random.default_rng(4).random((K, K))
    A_gpu, A_ref = run_both(proc, om, (t, nodes, T), rho, u, A0)
    np.testing.assert_array_equal(A_gpu, A_ref)
    assert A_ref.sum() > 0  # the reference does switch links on from the empty network


def test_exponential_sampler_inactive_link_with_the_smallest_theta():
    """ADVICE r1 (high): an inactive link whose theta is below every active theta must not have its tail cut."""
    K, n, rho = 4, 1000, 0.5
    lam0, W, theta, A = synth.exp_params(K, 11, wmax=2.0 / K, density=0.6)
    A[:] = 1.0
    A[2, 1] = 0.0
    theta[2, 1] = 0.02  # far slower than every active link (0.5 .. 2): look-back 25x longer
    W[2, 1] = 0.6
    t, nodes, T = synth.poisson_stream(n, K, 6.0, 9)
    proc = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.ExponentialImpulseResponse(theta), nhp.DenseWeightModel(W), A,
                                              nhp.BernoulliNetworkModel(rho, K))
    om = orc.Cont(0, lam0, W, theta, A=A, dtmax=np.inf)
    mism = 0
    for rep in range(4):
        u = np.random.default_rng(20 + rep).random((K, K))
        A_gpu, A_ref = run_both(proc, om, (t, nodes, T), rho, u, A)
        mism += int(np.count_nonzero(A_gpu != A_ref))
    assert mism == 0


def test_config4_shape_columns_match_oracle():
    """cfg4's shape (K = 1000, rho = 0.05, mean window 64) at an oracle-sized N, on every 50th column (the columns are
    independent: continuous.jl:462-464), through the column-partition entry point."""
    K, n, rho = 1000, 40000, 0.05
    t, nodes, T = synth.poisson_stream(n, K, 64.0, 4)
    proc, om = make_ln(K, 2, density=rho, wmax=0.5 / (K * rho))
    A0 = proc.adjacency_matrix.copy()
    u = np.random.default_rng(6).random((K, K))
    A_gpu, A_ref = run_both(proc, om, (t, nodes, T), rho, u, A0, col_begin=3, col_stride=50)
    np.testing.assert_array_equal(A_gpu, A_ref)
    other = [c for c in range(K) if c % 50 != 3]
    np.testing.assert_array_equal(A_gpu[:, other], A0[:, other])


def test_device_resident_sweep_equals_host_argument_sweep():
    """nhp_cont_resample_adjacency_dev (in place on the context's matrix, scalar rho, Philox) == the host-argument entry point
    fed the same Philox uniforms."""
    K, n, rho, seed, counter = 12, 3000, 0.3, 77, 5
    t, nodes, T = synth.poisson_stream(n, K, 50.0, 12)
    proc, om = make_ln(K, 3, density=0.5, wmax=1.5 / K)
    proc.network = nhp.BernoulliNetworkModel(rho, K)
    A0 = proc.adjacency_matrix.copy()
    kk = (np.arange(K)[:, None] + K * np.arange(K)[None, :]).astype(np.uint64)  # u[p, c] is keyed by p + K c
    u = synth.philox_uniform(seed, kk, counter)
    A_ref = om.resample_adjacency(A0, np.full((K, K), rho), t, nodes, T, u)
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    proc._push(ctx)
    ctx.check(ctx.lib.nhp_cont_resample_adjacency_dev(ctx.h, d.h, rho, seed, counter, 0, 1, 1))
    nhp.pull_params_(proc, ctx)
    np.testing.assert_array_equal(proc.adjacency_matrix, A_ref)
    # the masked tables were rebuilt: the log-likelihood is the one of the new matrix
    om2 = orc.Cont(1, proc.baseline.lam, proc.weights.W, proc.impulses.mu, proc.impulses.tau, A=A_ref, dtmax=1.0)
    ll = __import__("ctypes").c_double()
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, __import__("ctypes").byref(ll)))
    assert ll.value == pytest.approx(om2.loglik(t, nodes, T), rel=1e-10)


def test_network_draw_moments():
    """rho ~ Beta(alpha + sum A, beta + K^2 - sum A) (networks.jl:72-78) on the device."""
    K = 8
    proc, _ = make_ln(K, 3, density=0.4, wmax=0.1)
    ctx = proc._ctx()
    proc._push(ctx)
    import ctypes
    nA = float(proc.adjacency_matrix.sum())
    a, b = 1.0 + nA, 1.0 + K * K - nA
    xs = []
    for r in range(4000):
        rho = ctypes.c_double()
        ctx.check(ctx.lib.nhp_cont_resample_network(ctx.h, 5, r, 1.0, 1.0, ctypes.byref(rho)))
        xs.append(rho.value)
    xs = np.array(xs)
    mean, var = a / (a + b), a * b / ((a + b) ** 2 * (a + b + 1))
    assert abs(xs.mean() - mean) < 5 * np.sqrt(var / xs.size)
    assert abs(xs.var() - var) < 0.15 * var


def test_device_chain_network_process_runs_and_stays_finite():
    K = 6
    proc, _ = make_ln(K, 12, density=0.6, wmax=0.5)
    t, nodes, T = nhp.rand(proc, 400.0, np.random.default_rng(2))
    res = nhp.mcmc_(proc, (t, nodes, T), nsteps=6, seed=3, device_draws=True)
    assert len(res.samples) == 6 and all(np.all(np.isfinite(s)) for s in res.samples)
    assert set(np.unique(proc.adjacency_matrix)) <= {0.0, 1.0}
    assert 0.0 < proc.network.rho < 1.0


@pytest.mark.parametrize("kind,pre,chunk", [("ln", "1", None), ("ln", "0", 64), ("exp", "1", 7), ("ln", "1", 64)])
def test_loglikelihood_through_the_cached_structure_matches_oracle(monkeypatch, kind, pre, chunk):
    """Once a handle carries the pair structure, the log-likelihood of a sparse network streams the buckets of the active links only
    (k_adj_loglik): same value as the oracle and as the window sweep, with all payload / chunking variants."""
    import ctypes
    monkeypatch.setenv("NHP_ADJ_PRE", pre)
    if chunk is not None:
        monkeypatch.setenv("NHP_ADJ_CHUNK", str(chunk))
    K, n, rho = 23, 5000, 0.15
    t, nodes, T = synth.poisson_stream(n, K, 70.0, 21)
    proc, om = make_ln(K, 5, density=rho, wmax=2.0 / (K * rho)) if kind == "ln" else make_exp(K, 5, density=rho, wmax=2.0 / (K * rho), dtmax=1.0)
    proc.network = nhp.BernoulliNetworkModel(rho, K)
    ctx = proc._ctx()
    d = proc.upload((t, nodes, T))
    proc._push(ctx)
    ll = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll)))          # window sweep: no structure yet
    ll_window = ll.value
    ctx.check(ctx.lib.nhp_cont_resample_adjacency_dev(ctx.h, d.h, rho, 5, 1, 0, 1, 1))  # builds the structure, changes A
    nhp.pull_params_(proc, ctx)
    A1 = proc.adjacency_matrix.copy()
    assert 0 < np.count_nonzero(A1 * proc.weights.W) <= 0.25 * K * K
    launches = ctx.launches
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll)))          # structure path
    ll_struct = ll.value
    monkeypatch.setenv("NHP_ADJ_LOGLIK", "0")
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll)))          # window sweep, new A
    ll_window1 = ll.value
    if kind == "ln":
        om1 = orc.Cont(1, proc.baseline.lam, proc.weights.W, proc.impulses.mu, proc.impulses.tau, A=A1, dtmax=1.0)
    else:
        om1 = orc.Cont(0, proc.baseline.lam, proc.weights.W, proc.impulses.theta, A=A1, dtmax=1.0)
    ref = om1.loglik(t, nodes, T, recursive=False)
    assert ll_struct == pytest.approx(ref, rel=1e-10)
    assert ll_struct == pytest.approx(ll_window1, rel=1e-12)
    assert ll_window != ll_window1 or np.array_equal(A1, proc.adjacency_matrix)
    d.free()
