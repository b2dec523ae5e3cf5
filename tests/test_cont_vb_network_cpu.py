"""Network VB of continuous processes on the host: the NumPy twin of tests/cont_vb_network_reference.py and the Python layer's layout
helpers and refusals (continuous.network_*), without a GPU."""
import numpy as np
import pytest
from scipy import integrate
from scipy.special import digamma, expit, gammaln

import cont_vb_network_reference as RN
import cont_vb_reference as R
import nhp_b200 as nhp
from nhp_b200 import continuous as C

EXP, LN = R.EXP, R.LN
HYPER = {EXP: [1.5, 0.5, 2.0, 3.0, 2.0, 1.0, 0.1, 10.0, 1.0, 1.0], LN: [1.5, 0.5, 2.0, 3.0, 0.2, 1.5, 2.0, 0.7, 0.1, 10.0, 1.0, 1.0]}


def stream(counts, T, seed):
    rng = np.random.default_rng(seed)
    c = rng.permutation(np.repeat(np.arange(len(counts)), counts))
    return np.sort(rng.uniform(0.0, T, c.size)), c


def random_state(K, kind, seed):
    rng = np.random.default_rng(seed)
    mats = [rng.uniform(0.5, 3.0, (K, K)), rng.uniform(3.0, 30.0, (K, K))]
    if kind == EXP:
        mats += [rng.uniform(2.0, 10.0, (K, K)), rng.uniform(0.5, 3.0, (K, K))]
    else:
        mats += [rng.normal(0.0, 1.0, (K, K)), rng.uniform(0.5, 5.0, (K, K)), rng.uniform(1.0, 6.0, (K, K)), rng.uniform(0.5, 3.0, (K, K))]
    qs = R.pack(rng.uniform(2.0, 10.0, K), rng.uniform(1.0, 5.0, K), mats)
    return RN.join(qs, rng.uniform(0.05, 0.5, (K, K)), rng.uniform(2.0, 20.0, (K, K)), rng.uniform(0.0, 1.0, (K, K)), rng.uniform(1.0, 4.0),
                   rng.uniform(1.0, 4.0))


@pytest.mark.parametrize("seed", [0, 1])
def test_mixture_log_weight_against_quadrature(seed):
    """E[ln W] under pv Gamma(kappav, nuv) + (1 - pv) Gamma(kappa0v, nu0v) by quadrature, to 1e-9."""
    K, kind = 2, EXP
    q = random_state(K, kind, seed)
    lw = RN.mixture_lw(q, K, kind)
    qs, k0v, n0v, pv, _, _ = RN.split(q, K, kind)
    _, _, P = R.planes(qs, K, kind)
    for p in range(K):
        for c in range(K):
            def f(x, a, b):  # over x = ln w, where the density of a small-shape spike is smooth: Gamma(a, b) density of w times w
                return x * np.exp(a * np.log(b) - gammaln(a) + a * x - b * np.exp(x))
            parts = [integrate.quad(f, -60.0 / a, np.log((a + 60.0) / b), args=(a, b), limit=400, epsabs=1e-13, epsrel=1e-12)[0] for a, b in
                     ((P[0][p, c], P[1][p, c]), (k0v[p, c], n0v[p, c]))]
            want = pv[p, c] * parts[0] + (1.0 - pv[p, c]) * parts[1]
            assert abs(lw[p, c] - want) <= 1e-9 * max(1.0, abs(want)), (p, c, lw[p, c], want)


@pytest.mark.parametrize("kind,dtmax", [(EXP, np.inf), (LN, 1.0)])
def test_elbo_never_decreases(kind, dtmax):
    """30 twin steps at K = 3 from the all-links start: the bound of successive states never decreases (beyond 1e-12 relative: the
    Exponential look-back horizon depends on the state)."""
    K, T = 3, 60.0
    t, c = stream([60, 50, 70], T, 3 + kind)
    q = RN.prior_state(K, kind, HYPER[kind])
    prev = RN.elbo(t, c, K, kind, q, HYPER[kind], T, dtmax)
    for k in range(30):
        q, _, _ = RN.vb_step(t, c, K, kind, q, HYPER[kind], T, dtmax)
        cur = RN.elbo(t, c, K, kind, q, HYPER[kind], T, dtmax)
        assert cur >= prev - 1e-12 * abs(prev), (k, prev, cur)
        prev = cur


@pytest.mark.parametrize("kind,dtmax", [(EXP, 3.0), (LN, 1.0)])
def test_spike_equal_to_slab_is_the_standard_step(kind, dtmax):
    """With kappa0 = kappa, nu0 = nu, kappa0v = kappav and nu0v = nuv the standard part of a network step is cont_vb_reference.vb_step
    and pv = sigmoid(psi(alpharhov) - psi(betarhov)) (the old q(rho))."""
    K, T = 3, 50.0
    t, c = stream([40, 50, 45], T, 9 + kind)
    h = list(HYPER[kind])
    ns = RN.nstd(kind)
    h[ns], h[ns + 1] = h[2], h[3]
    q = random_state(K, kind, 4)
    qs, _, _, pv, ar, br = RN.split(q, K, kind)
    _, _, P = R.planes(qs, K, kind)
    q = RN.join(qs, P[0], P[1], pv, ar, br)
    qn, _, _ = RN.vb_step(t, c, K, kind, q, h, T, dtmax)
    qsr, _, _ = R.vb_step(t, c, K, kind, qs, h[:ns], T, dtmax)
    qsn, k0n, n0n, pvn, _, _ = RN.split(qn, K, kind)
    np.testing.assert_allclose(qsn, qsr, rtol=1e-12, atol=1e-12)
    _, _, Pn = R.planes(qsn, K, kind)
    assert np.array_equal(k0n, Pn[0]) and np.array_equal(n0n, Pn[1])
    np.testing.assert_allclose(pvn, expit(digamma(ar) - digamma(br)), rtol=1e-12)


def proc(kind, K=3, network=None, baseline=None):
    rng = np.random.default_rng(1)
    W = rng.uniform(0.05, 0.2, (K, K))
    imp = nhp.ExponentialImpulseResponse(np.full((K, K), 2.0), 2.0, 1.0) if kind == EXP else \
        nhp.LogitNormalImpulseResponse(np.zeros((K, K)), np.ones((K, K)), 1.0, 0.2, 1.5, 2.0, 0.7)
    base = baseline or nhp.HomogeneousProcess(np.ones(K), 1.5, 0.5)
    return nhp.ContinuousNetworkHawkesProcess(base, imp, nhp.DenseWeightModel(W, 2.0, 3.0), np.ones((K, K)),
                                              network or nhp.BernoulliNetworkModel(0.3, K, 1.0, 1.0))


@pytest.mark.parametrize("kind", [EXP, LN])
def test_layout_and_hyper_helpers(kind):
    """network_hyper, network_vb_size and network_prior_variational_params match the twin's layout; network_posterior_means reads it
    back (A = pv, the mixture and slab means of W, lambda0, p1, p2, rho)."""
    K = 3
    p = proc(kind, K)
    hy = C.network_hyper(p)
    assert np.array_equal(hy, HYPER[kind])
    q0 = C.network_prior_variational_params(p)
    assert q0.size == C.network_vb_size(p) == 2 * K + (7 if kind == EXP else 9) * K * K + 2
    assert np.array_equal(q0, RN.prior_state(K, kind, hy))
    assert np.array_equal(C.network_prior_variational_params(p, pv=0.3, kappa0=0.2, nu0=5.0),
                          RN.prior_state(K, kind, np.concatenate([hy[:-4], [0.2, 5.0], hy[-2:]]), pv=0.3))
    q = random_state(K, kind, 7)
    m = C.network_posterior_means(p, q)
    qs, k0v, n0v, pv, ar, br = RN.split(q, K, kind)
    l0, Ws, p1, p2 = R.posterior_means(qs, K, kind)
    assert np.array_equal(m["A"], pv) and np.array_equal(m["W_slab"], Ws) and np.array_equal(m["lambda0"], l0)
    assert np.array_equal(m["p1"], p1) and ((m["p2"] is None) if kind == EXP else np.array_equal(m["p2"], p2))
    np.testing.assert_allclose(m["W"], pv * Ws + (1.0 - pv) * k0v / n0v, rtol=1e-15)
    assert m["rho"] == ar / (ar + br)
    assert np.array_equal(RN.join(*RN.split(q, K, kind)), q)
    with pytest.raises(ValueError):
        C.network_posterior_means(p, q[:-1])
    with pytest.raises(ValueError):
        C.network_prior_variational_params(p, pv=1.5)


def test_refusals_come_before_any_device_call(monkeypatch):
    """A standard process, a DenseNetworkModel, a LogGaussianCox baseline, a kappa0 / nu0 that is not positive and finite and a q0 of the
    wrong size raise ValueError without a context; the standard VB functions still refuse a network process."""
    import nhp_b200
    from nhp_b200 import core

    def no_device(*a, **k):
        raise AssertionError("a device context was requested")

    monkeypatch.setattr(core, "default_context", no_device)
    monkeypatch.setattr(C, "default_context", no_device)
    monkeypatch.setattr(nhp_b200, "default_context", no_device, raising=False)
    K = 3
    net = proc(EXP, K)
    std = nhp.ContinuousStandardHawkesProcess(net.baseline, net.impulses, net.weights)
    dense = proc(EXP, K, network=nhp.DenseNetworkModel(K))
    lg = proc(EXP, K, baseline=nhp.LogGaussianCoxProcess([0.0, 2.0], np.ones((K, 2))))
    data = (np.array([0.5, 1.0]), np.array([1, 2]), 2.0)
    q = C.network_prior_variational_params(net)
    for p, kw in ((std, {}), (dense, {}), (lg, {}), (net, dict(kappa0=0.0)), (net, dict(nu0=-1.0)), (net, dict(kappa0=float("nan"))),
                  (net, dict(nu0=float("inf"))), (net, dict(q0=q[:-1])), (net, dict(q0=np.ones(C.vb_size(net))))):
        with pytest.raises(ValueError):
            C.network_vb_device_(p, data, **kw)
    for p in (std, dense, lg):
        with pytest.raises(ValueError):
            C.network_vb_statistics(p, data, q)
        with pytest.raises(ValueError):
            C.network_prior_variational_params(p)
    with pytest.raises(ValueError):
        C.network_vb_statistics(net, data, q[:-1])
    for f in (lambda: C.vb_device_(net, data), lambda: C.vb_statistics(net, data, np.ones(C.vb_size(net))), lambda: C.prior_variational_params(net)):
        with pytest.raises(ValueError):
            f()
    assert not hasattr(net.network, "pv")
