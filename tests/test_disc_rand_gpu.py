"""GPU tests of the discrete device simulator (csrc/disc_rand.cu; rand(process::DiscreteHawkesProcess, T), discrete.jl:20-38).

The specification is the law the likelihood assumes: given the earlier bins, data[c, t] ~ Poisson(lambda[t, c]) with lambda from
nhp_disc_intensity.  The main check computes that lambda on the returned handle (a path independent of the simulator) and tests the
randomised PIT of every bin; negative controls show the test has power.  The rest: agreement in distribution with the host simulator,
the stationary mean, the lag shape, equality with an uploaded handle, determinism, parameter recovery by the device VB and Gibbs
chains on true samples, and the refusals.  Seeds are fixed, so every statistical check is deterministic; the measured statistic is
written next to each threshold (NVIDIA B200)."""
import ctypes

import numpy as np
import pytest

import nhp_b200 as nhp
import oracle_ffi as orc
from disc_rand_law import law_holds
from nhp_b200 import _lib
from nhp_b200 import discrete as D
from nhp_b200.core import _fmat, _ptr

pytestmark = pytest.mark.gpu


def make(N, B, L, seed, theta=None, network=True, rates=(0.2, 0.4), radius=0.85, density=0.6, kappa=1.0, alpha=1.0, beta=1.0):
    """A stable process: W scaled to the given spectral radius of [A]W, a self-link on every node."""
    rng = np.random.default_rng(seed)
    lam0 = rng.uniform(*rates, N)
    A = (rng.random((N, N)) < density).astype(np.float64)
    np.fill_diagonal(A, 1.0)
    W = rng.uniform(0.5, 1.0, (N, N)) * (A if network else 1.0)
    W *= radius / np.max(np.abs(np.linalg.eigvals(W)))
    th = rng.dirichlet(np.ones(B), (N, N)) if theta is None else np.broadcast_to(theta, (N, N, B)).copy()
    b, i, w = D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(th, L), nhp.DenseWeightModel(W, kappa=kappa)
    if not network:
        return D.DiscreteStandardHawkesProcess(b, i, w)
    return D.DiscreteNetworkHawkesProcess(b, i, w, A, nhp.BernoulliNetworkModel(0.5, N, alpha, beta))


def variant(proc, W=None, theta=None):
    """The same model with W and / or theta replaced (negative controls)."""
    b, imp = proc.baseline, proc.impulses
    i = D.DiscreteGaussianImpulseResponse(imp.theta if theta is None else theta, imp.nlags)
    w = nhp.DenseWeightModel(proc.weights.W if W is None else W)
    if proc.adjacency_matrix is None:
        return D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(b.lam), i, w)
    return D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(b.lam), i, w, proc.adjacency_matrix, proc.network)


# ---- 1. the conditional law -------------------------------------------------------------------------------------------------------
def test_sample_has_the_conditional_law_of_the_likelihood():
    """N = 5, T = 2e5, network process with mixed theta: the PIT of every bin against intensity() on the handle is U(0, 1)
    (measured: KS p 0.29, z -0.66, per-node |z| <= 1.2); with the intensity of W x 1.1 it is not (z -115)."""
    proc = make(5, 3, 20, 1)
    d = D.rand_device(proc, 200000, seed=21)
    data = d.download()
    assert data.sum() == d.events_count() > 1_000_000
    ok, st = law_holds(data, D.intensity(proc, d))
    assert ok, st
    bad, st = law_holds(data, D.intensity(variant(proc, W=proc.weights.W * 1.1), d))
    assert not bad and st[1] < -20, st


def test_lag_law_has_power_against_reversed_theta():
    """theta concentrated on the first basis: the sample passes (measured KS p 0.25) and the intensity with theta reversed along b
    fails the same test (measured KS p 2.8e-7; z stays at -1.1, only the timing of the children is wrong)."""
    proc = make(5, 3, 20, 1, theta=np.array([0.96, 0.03, 0.01]))
    d = D.rand_device(proc, 200000, seed=22)
    data = d.download()
    ok, st = law_holds(data, D.intensity(proc, d))
    assert ok, st
    bad, st = law_holds(data, D.intensity(variant(proc, theta=proc.impulses.theta[:, :, ::-1].copy()), d))
    assert not bad, st


# ---- 3. device against host in distribution ---------------------------------------------------------------------------------------
def test_device_sample_matches_host_simulator_in_distribution():
    """100 short samples each (N = 3, T = 2000): total counts (mean within 4.5 standard errors, variance ratio in (0.6, 1.6)) and the
    lag-1 cross-covariance of the excited pair (0 -> 1) agree."""
    N, T, reps = 3, 2000, 100
    proc = make(N, 2, 4, 5, rates=(0.05, 0.1), radius=0.6, density=1.0)
    proc.weights.W[0, 1] = 0.5  # one clearly excited pair
    host = [D.rand(proc, T, np.random.default_rng(100 + r)) for r in range(reps)]
    dev = [D.rand_device(proc, T, seed=500 + r).download() for r in range(reps)]

    def stat(xs):
        tot = np.array([x.sum() for x in xs], dtype=float)
        cov = np.array([np.mean((x[0, :-1] - x[0].mean()) * (x[1, 1:] - x[1].mean())) for x in xs])
        return tot, cov

    (th, ch), (td, cd) = stat(host), stat(dev)
    se = np.sqrt(th.var() / reps + td.var() / reps)
    assert abs(th.mean() - td.mean()) < 4.5 * se, (th.mean(), td.mean(), se)
    assert 0.6 < td.var() / th.var() < 1.6, (td.var(), th.var())
    sec = np.sqrt(ch.var() / reps + cd.var() / reps)
    assert abs(ch.mean() - cd.mean()) < 4.5 * sec, (ch.mean(), cd.mean(), sec)
    assert cd.mean() > 5 * cd.std() / np.sqrt(reps)  # the pair is visibly excited


# ---- 4. stationary mean -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("network", [True, False])
def test_counts_have_the_stationary_mean(network):
    """E[counts] = ((I - e^T)^-1 lambda0 dt) T with e the expected children per event (effective_weights); over-dispersed error bar
    6 sqrt(mean) / (1 - radius)."""
    proc = make(6, 3, 8, 7, network=network, rates=(0.02, 0.05), radius=0.6)
    T = 400000
    counts = D.rand_device(proc, T, seed=3).download().sum(axis=1).astype(float)
    e = proc.effective_weights()
    mean = np.linalg.solve(np.eye(6) - e.T, proc.baseline.lam * proc.dt) * T
    assert np.all(np.abs(counts - mean) < 6.0 * np.sqrt(mean) / (1 - 0.6)), (counts, mean)


# ---- 5. lag shape -----------------------------------------------------------------------------------------------------------------
def test_children_follow_the_lag_distribution():
    """Node 0 (sparse baseline) excites node 1 only, node 1 has no baseline: the counts of node 1 l bins after an isolated event of node
    0 average W q_l, q_l = sum_b theta_b phi_b[l] dt, for l = 1..L, and are exactly zero at lag 0 and at lags L+1..2L."""
    L, B = 10, 3
    lam0 = np.array([0.002, 0.0])
    W = np.array([[0.0, 0.9], [0.0, 0.0]])
    th = np.zeros((2, 2, B))
    th[:, :] = [0.5, 0.2, 0.3]
    proc = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(th, L), nhp.DenseWeightModel(W))
    data = D.rand_device(proc, 3_000_000, seed=9).download()
    tp = np.nonzero(data[0])[0]
    gap = np.diff(tp)
    iso = tp[1:-1][(gap[:-1] > 2 * L) & (gap[1:] > 2 * L) & (data[0, tp[1:-1]] == 1)]
    iso = iso[iso + 2 * L < data.shape[1]]
    assert iso.size > 3500
    win = data[1, iso[:, None] + np.arange(0, 2 * L + 1)]  # lags 0..2L
    q = proc.impulses.basis() @ th[0, 1] * proc.dt
    m = win.mean(axis=0)
    assert np.all(win[:, 0] == 0) and np.all(win[:, L + 1:] == 0)
    se = np.sqrt(0.9 * q / iso.size)
    assert np.all(np.abs(m[1:L + 1] - 0.9 * q) < 5 * se + 1e-3), (m[1:L + 1], 0.9 * q)


# ---- 6. the handle equals an uploaded one -----------------------------------------------------------------------------------------
def _sweep_params(ctx, d, proc, hy, n=3):
    proc._push(ctx)
    ctx.check(ctx.lib.nhp_disc_network_set(ctx.h, 0.5))
    for s in range(n):
        ctx.check(ctx.lib.nhp_disc_gibbs_sweep(ctx.h, d.h, 17, s, _ptr(hy), 5, 1.0, 1.0))
    N, B = proc.ndims(), proc.impulses.nbasis()
    out = [np.empty(N), np.empty(N * N), np.empty(N * N), np.empty(N * N * B)]
    ctx.check(ctx.lib.nhp_disc_params_get(ctx.h, *[_ptr(a) for a in out]))
    return out


def test_simulated_handle_equals_uploaded_handle():
    proc = make(6, 3, 7, 11, rates=(0.05, 0.1), radius=0.7)
    ctx = proc._ctx()
    d1 = D.rand_device(proc, 30000, seed=4)
    data = d1.download()
    d2 = D.DiscreteData(ctx, data)
    assert d1.events_count() == d2.events_count() == int(data.sum())
    assert np.array_equal(d2.download(), data)
    c1, c2 = D.convolve(proc, d1), D.convolve(proc, d2)
    assert np.array_equal(c1, c2)
    l1, l2 = D.loglikelihood(proc, d1), D.loglikelihood(proc, d2)
    assert l1 == l2
    oconv = orc.disc_convolve(data, orc.disc_basis(7, 3))
    ref = orc.Disc(proc.baseline.lam, proc.weights.W, proc.impulses.theta, A=proc.adjacency_matrix).loglik(data, oconv)
    assert l1 == pytest.approx(ref, rel=1e-10)
    assert np.array_equal(D.resample_parents(proc, d1, seed=5, counter=2), D.resample_parents(proc, d2, seed=5, counter=2))
    hy = np.array([1.0, 1.0, 1.0, 1.0, 1.0])
    p1, p2 = _sweep_params(ctx, d1, proc, hy), _sweep_params(ctx, d2, proc, hy)
    for a, b in zip(p1, p2):
        assert np.array_equal(a, b)


def test_upload_download_round_trip_is_exact():
    rng = np.random.default_rng(2)
    data = rng.poisson(0.7, (7, 5001)).astype(np.int64)
    data[3, 17] = 2**31 - 1
    d = D.DiscreteData(nhp.default_context(), data, t_halo=40)
    assert np.array_equal(d.download(), data)
    assert d.events_count() == int(data[:, 40:].sum())


# ---- 7. determinism ---------------------------------------------------------------------------------------------------------------
def test_sample_is_a_function_of_the_seed():
    proc = make(4, 3, 6, 13)
    a, b, c = (D.rand_device(proc, 20000, seed=s).download() for s in (8, 8, 9))
    assert np.array_equal(a, b) and not np.array_equal(a, c)
    std = make(4, 3, 6, 13, network=False)
    net = D.DiscreteNetworkHawkesProcess(std.baseline, std.impulses, std.weights, np.ones((4, 4)), nhp.BernoulliNetworkModel(0.5, 4))
    assert np.array_equal(D.rand_device(std, 20000, seed=8).download(), D.rand_device(net, 20000, seed=8).download())


def test_theta_need_not_sum_to_one_exactly():
    """The context takes theta that sums to 1 within allclose; e is computed from theta as written, so a theta scaled by (1 + 1e-9)
    gives a sample whose law is still the likelihood's (same checks as the main test at a smaller size; measured KS p 0.29, z 1.2)."""
    proc = make(3, 2, 5, 15)
    proc.impulses.theta *= 1.0 + 1e-9
    d = D.rand_device(proc, 100000, seed=1)
    ok, st = law_holds(d.download(), D.intensity(proc, d))
    assert ok, st


# ---- 8. recovery on true samples --------------------------------------------------------------------------------------------------
def test_vb_recovers_the_parameters_of_a_true_sample():
    """vb_device_ on a standard-process sample (N = 4, T = 2e5): E[W] = kappav / nuv and E[lambda0] = alphav / betav lie within 8
    mean-field posterior standard deviations of the truth (measured: largest |error| / sd 6.2 for W, 4.6 for lambda0; the
    mean-field sd understates the posterior spread of W, whose entries trade off against each other) and within 10 % of it (measured: 8.6 % for W, 4.2 % for lambda0)."""
    N, T = 4, 200000
    proc = make(N, 3, 6, 17, network=False, rates=(0.05, 0.1), radius=0.6)
    W0, l0 = proc.weights.W.copy(), proc.baseline.lam.copy()
    d = D.rand_device(proc, T, seed=5)
    D.vb_device_(proc, d, max_steps=100, rtol=1e-10)
    b, w = proc.baseline, proc.weights
    EW, sW = w.kappav / w.nuv, np.sqrt(w.kappav) / w.nuv
    El, sl = b.alphav / b.betav, np.sqrt(b.alphav) / b.betav
    assert np.all(np.abs(EW - W0) < 8 * sW) and np.all(np.abs(EW - W0) < 0.1 * W0), ((EW - W0) / sW)
    assert np.all(np.abs(El - l0) < 8 * sl) and np.all(np.abs(El - l0) < 0.1 * l0), ((El - l0) / sl)


def test_gibbs_recovers_the_links_of_a_true_sample():
    """mcmc_device_ on a network sample with clearly separated links (weights 0.4 or more on the links, none elsewhere), started from
    the full graph: the posterior mean of A is above 0.9 on the true links and below 0.1 elsewhere (measured: 1.0 on every link,
    0.053 at most elsewhere, mean rho 0.039).  A link of near-zero weight explains the data as well as no link, so off the true links the
    posterior of A follows the link probability; a sparse Beta(1, 200) prior on rho keeps that low."""
    N, T = 5, 200000
    proc = make(N, 3, 6, 19, rates=(0.05, 0.1), radius=0.6, density=0.3, alpha=1.0, beta=200.0)
    A0 = proc.adjacency_matrix.copy()
    assert 0 < A0.sum() < N * N and np.min(proc.weights.W[A0 == 1]) > 0.4
    d = D.rand_device(proc, T, seed=6)
    proc.adjacency_matrix = np.ones((N, N))
    proc.weights.W = np.full((N, N), 0.1)
    res = D.mcmc_device_(proc, d, nsteps=400, seed=3)
    S = np.array(res.samples[100:])
    Abar = S[:, -N * N:].mean(axis=0).reshape(N, N).T  # vec(A) -> [p, c]
    assert np.min(Abar[A0 == 1]) > 0.9, Abar
    assert np.max(Abar[A0 == 0]) < 0.1, Abar


# ---- 9. refusals ------------------------------------------------------------------------------------------------------------------
def _rand(ctx, T, L, max_events=10**6):
    h = ctypes.c_void_p()
    rc = ctx.lib.nhp_disc_rand(ctx.h, T, L, 1, max_events, ctypes.byref(h))
    return rc, h.value


def test_refusals_leave_no_handle():
    ctx = nhp.Context(0)  # a fresh context: no discrete parameters yet
    assert _rand(ctx, 100, 3) == (_lib.NHP_ERR_STATE, None)
    N, B = 3, 2
    lam0, W, th = np.full(N, 0.1), np.full((N, N), 0.1), np.full((N, N, B), 0.5)
    A = np.ones((N, N))

    def push(W=W, th=th, A=A):
        thf = np.ascontiguousarray(th.transpose(2, 1, 0)).ravel()
        ctx.check(ctx.lib.nhp_disc_params_set(ctx.h, N, B, _ptr(lam0), _ptr(_fmat(W)), _ptr(None if A is None else _fmat(A)), _ptr(thf), 1.0))

    push()
    for T, L in ((0, 3), (-5, 3), (2**31 // N, 3), (100, 0), (100, 2049)):
        assert _rand(ctx, T, L) == (_lib.NHP_ERR_INVALID, None), (T, L)
    for kw in (dict(W=-W), dict(W=W * np.inf), dict(th=-th), dict(th=th * np.nan), dict(A=-A)):
        push(**kw)
        assert _rand(ctx, 100, 3) == (_lib.NHP_ERR_INVALID, None), kw
    push(W=np.full((N, N), 0.6))  # unstable: every event has 1.8 children on average
    rc, h = _rand(ctx, 100000, 3, max_events=200000)
    assert (rc, h) == (_lib.NHP_ERR_INVALID, None) and "is the process stable?" in ctx.lib.nhp_last_error(ctx.h).decode()
    push()
    assert _rand(ctx, 100000, 3, max_events=10)[0] == _lib.NHP_ERR_INVALID  # generation 0 alone
    rc, h = _rand(ctx, 1000, 3)
    assert rc == 0 and h
    assert ctx.lib.nhp_disc_free(ctx.h, ctypes.c_void_p(h)) == 0

