"""The NumPy twin of continuous mean-field VB (tests/cont_vb_reference.py) checked on its own, without a GPU: the responsibilities,
the shifted one-pass M-step against a direct two-pass one, the effective-parameter identities against quadrature, a hand-derived
single-pair update and the prior for pairs without statistics; and the Python layer's layout helpers and refusals."""
import numpy as np
import pytest
from scipy import integrate, stats
from scipy.special import roots_hermite

import cont_vb_reference as R
import nhp_b200 as nhp
from nhp_b200 import continuous as C

EXP, LN = R.EXP, R.LN


def stream(K, n, T, seed, ties=0):
    rng = np.random.default_rng(seed)
    t = np.sort(rng.uniform(0.0, T, n))
    if ties:
        t[1:1 + ties] = t[0]
    return t, rng.integers(0, K, n)


def random_state(K, kind, seed):
    rng = np.random.default_rng(seed)
    mats = [rng.uniform(0.5, 5.0, (K, K)), rng.uniform(2.0, 20.0, (K, K))]
    if kind == EXP:
        mats += [rng.uniform(2.0, 10.0, (K, K)), rng.uniform(0.5, 3.0, (K, K))]
    else:
        mats += [rng.normal(0.0, 1.0, (K, K)), rng.uniform(0.5, 5.0, (K, K)), rng.uniform(1.0, 6.0, (K, K)), rng.uniform(0.5, 3.0, (K, K))]
    return R.pack(rng.uniform(2.0, 10.0, K), rng.uniform(1.0, 5.0, K), mats)


@pytest.mark.parametrize("kind,dtmax", [(EXP, np.inf), (EXP, 0.7), (LN, 1.0)])
def test_responsibilities_sum_to_one(kind, dtmax):
    K = 4
    t, c = stream(K, 400, 40.0, 1, ties=3)
    q = random_state(K, kind, 2)
    st = R.expected_stats(t, c, K, kind, q, dtmax)
    for u0, js, u in st["resp"]:
        assert 0.0 < u0 <= 1.0 and np.all(u >= 0.0)
        assert abs(u0 + u.sum() - 1.0) <= 1e-14
    # every event is somebody's child once: the expected counts add up to the events
    assert abs(st["M0"].sum() + st["Mnm"].sum() - t.size) <= 1e-10 * t.size


def test_shifted_m_step_equals_two_pass():
    """The one-pass statistics about the current mv give the same Normal-Gamma update as the weighted mean and the weighted sum of
    squares about it computed in two passes over the (u, y) of every pair."""
    K, dtmax = 3, 1.0
    t, c = stream(K, 300, 30.0, 3)
    q = random_state(K, LN, 4)
    hyper = [1.5, 0.5, 2.0, 3.0, 0.3, 1.7, 2.5, 0.8]
    st = R.expected_stats(t, c, K, LN, q, dtmax)
    qn, _ = R.m_step(q, K, LN, hyper, 30.0, st)
    w = [[[] for _ in range(K)] for _ in range(K)]
    for i, (u0, js, u) in enumerate(st["resp"]):
        for j, uj in zip(js, u):
            if uj > 0:
                dt = t[i] - t[j]
                w[c[j]][c[i]].append((uj, np.log(dt / (dtmax - dt))))
    mumu, kmu, a0, b0 = hyper[4:]
    _, _, P = R.planes(qn, K, LN)
    for p in range(K):
        for cc in range(K):
            uy = np.array(w[p][cc])
            n = uy[:, 0].sum()
            ybar = np.sum(uy[:, 0] * uy[:, 1]) / n
            S = np.sum(uy[:, 0] * (uy[:, 1] - ybar) ** 2)
            lv = kmu + n
            assert P[3][p, cc] == pytest.approx(lv, rel=1e-14)
            assert P[2][p, cc] == pytest.approx((kmu * mumu + n * ybar) / lv, rel=1e-12, abs=1e-12)
            assert P[4][p, cc] == pytest.approx(a0 + n / 2, rel=1e-14)
            assert P[5][p, cc] == pytest.approx(b0 + S / 2 + kmu * n * (ybar - mumu) ** 2 / (2 * lv), rel=1e-11)


@pytest.mark.parametrize("seed", range(4))
def test_effective_identity_exponential(seed):
    """ln W_eff + ln h(dt; theta_eff) = E_q[ln W] + E_q[ln theta - theta dt], the right side by quadrature over the Gamma factors."""
    rng = np.random.default_rng(seed)
    kv, nv, a, b = rng.uniform(0.5, 8.0), rng.uniform(0.5, 8.0), rng.uniform(0.5, 8.0), rng.uniform(0.5, 8.0)
    q = R.pack([1.0], [1.0], [np.array([[x]]) for x in (kv, nv, a, b)])
    _, W, th, _ = R.effective_params(q, 1, EXP)
    gw, gt = stats.gamma(kv, scale=1 / nv), stats.gamma(a, scale=1 / b)
    Elw = integrate.quad(lambda x: np.log(x) * gw.pdf(x), 0, np.inf, epsabs=1e-13, epsrel=1e-13, limit=200)[0]
    for dt in rng.uniform(0.0, 3.0, 4):
        Elh = integrate.quad(lambda x: (np.log(x) - x * dt) * gt.pdf(x), 0, np.inf, epsabs=1e-13, epsrel=1e-13, limit=200)[0]
        lhs = np.log(W[0, 0]) + np.log(R.impulse(EXP, np.array(dt), th[0, 0], None, np.inf))
        assert lhs == pytest.approx(Elw + Elh, abs=1e-9)


@pytest.mark.parametrize("seed", range(3))
def test_effective_identity_logitnormal(seed):
    """ln W_eff + ln h(dt; mv, av / bv) = E_q[ln W] + E_q[ln h(dt; mu, tau)] under q(mu, tau) = NormalGamma(mv, lambdav, av, bv), the
    right side by nested quadrature: adaptive over tau outside, Gauss-Hermite over mu | tau inside (40 nodes)."""
    rng = np.random.default_rng(10 + seed)
    kv, nv = rng.uniform(0.5, 8.0), rng.uniform(0.5, 8.0)
    mv, lv, a, b = rng.normal(), rng.uniform(0.5, 5.0), rng.uniform(1.0, 6.0), rng.uniform(0.5, 3.0)
    D = 1.3
    q = R.pack([1.0], [1.0], [np.array([[x]]) for x in (kv, nv, mv, lv, a, b)])
    _, W, mu_e, tau_e = R.effective_params(q, 1, LN)
    Elw = integrate.quad(lambda x: np.log(x) * stats.gamma(kv, scale=1 / nv).pdf(x), 0, np.inf, epsabs=1e-13, epsrel=1e-13, limit=200)[0]
    gt = stats.gamma(a, scale=1 / b)
    gh_x, gh_w = roots_hermite(40)
    for dt in rng.uniform(0.05, D - 0.05, 3):
        y = np.log(dt / (D - dt))
        c0 = np.log(D * D / (dt * (D - dt))) - 0.5 * np.log(2 * np.pi)

        def inner(tau):
            m = mv + np.sqrt(2.0 / (lv * tau)) * gh_x
            return np.sum(gh_w * (0.5 * np.log(tau) - 0.5 * tau * (y - m) ** 2)) / np.sqrt(np.pi) * gt.pdf(tau)

        Elh = c0 + integrate.quad(inner, 0, np.inf, epsabs=1e-12, epsrel=1e-12, limit=200)[0]
        lhs = np.log(W[0, 0]) + np.log(R.impulse(LN, np.array(dt), mu_e[0, 0], tau_e[0, 0], D))
        assert lhs == pytest.approx(Elw + Elh, abs=1e-8)


def test_single_pair_update_by_hand():
    """K = 1, statistics written down by hand: M0 = 3, Mn = 5, Mnm = 2, S1 = 0.5, S2 = 1.25 about mv = 0.4, with hyper-parameters
    (alpha0, beta0, kappa, nu) = (1, 2, 3, 4), (mumu, kappamu, a0, b0) = (0.1, 2, 1.5, 0.5) and T = 10:
      alphav = 4, betav = 12, kappav = 5, nuv = 9; n = 2, d = 0.25, ybar = 0.65, S = 1.25 - 2 * 0.0625 = 1.125;
      lambdav = 4, mv = (0.2 + 1.3) / 4 = 0.375, av = 2.5, bv = 0.5 + 0.5625 + 2 * 2 * 0.3025 / 8 = 1.21375.
    Exponential (alpha, beta) = (2, 3) with S1 = 0.5: atheta = 4, btheta = 3.5."""
    st = dict(M0=np.array([3.0]), Mn=np.array([5.0]), Mnm=np.array([[2.0]]), S1=np.array([[0.5]]), S2=np.array([[1.25]]))
    q = R.pack([1.0], [1.0], [np.array([[x]]) for x in (1.0, 1.0, 0.4, 1.0, 1.0, 1.0)])
    qn, _ = R.m_step(q, 1, LN, [1, 2, 3, 4, 0.1, 2, 1.5, 0.5], 10.0, st)
    assert np.allclose(qn, [4, 12, 5, 9, 0.375, 4, 2.5, 1.21375], rtol=1e-15, atol=0)
    qe = R.pack([1.0], [1.0], [np.ones((1, 1))] * 4)
    qn, _ = R.m_step(qe, 1, EXP, [1, 2, 3, 4, 2, 3], 10.0, st)
    assert np.allclose(qn, [4, 12, 5, 9, 4, 3.5], rtol=1e-15, atol=0)


@pytest.mark.parametrize("kind", [EXP, LN])
def test_empty_pair_gets_prior(kind):
    """A pair with no expected parent (n = 0) comes out at its prior, finite, whatever the state was."""
    K = 2
    hyper = [1.0, 2.0, 3.0, 4.0, 2.0, 3.0] if kind == EXP else [1.0, 2.0, 3.0, 4.0, -0.2, 2.0, 1.5, 0.5]
    q = random_state(K, kind, 7)
    z = np.zeros((K, K))
    st = dict(M0=np.zeros(K), Mn=np.zeros(K), Mnm=z, S1=z, S2=z)
    qn, _ = R.m_step(q, K, kind, hyper, 5.0, st)
    assert np.all(np.isfinite(qn))
    assert np.array_equal(qn, R.prior_state(K, kind, hyper) + np.concatenate([np.zeros(K), np.full(K, 5.0), np.zeros(qn.size - 2 * K)]))


def proc(kind, K=3):
    W = np.full((K, K), 0.1)
    imp = nhp.ExponentialImpulseResponse(np.ones((K, K)), alpha=2.0, beta=3.0) if kind == EXP else \
        nhp.LogitNormalImpulseResponse(np.zeros((K, K)), np.ones((K, K)), 1.0, mumu=0.3, kappamu=2.0, alpha0=1.5, beta0=0.5)
    return nhp.ContinuousStandardHawkesProcess(nhp.HomogeneousProcess(np.ones(K), 1.5, 2.5), imp, nhp.DenseWeightModel(W, 3.0, 4.0))


@pytest.mark.parametrize("kind", [EXP, LN])
def test_python_layout_helpers(kind):
    p = proc(kind)
    hyper = C._hyper(p)
    q0 = C.prior_variational_params(p)
    assert q0.size == C.vb_size(p) and np.array_equal(q0, R.prior_state(3, kind, hyper))
    q = random_state(3, kind, 5)
    m = C.posterior_means(p, q)
    l0, W, p1, p2 = R.posterior_means(q, 3, kind)
    assert np.array_equal(m["lambda0"], l0) and np.array_equal(m["W"], W) and np.array_equal(m["p1"], p1)
    assert (m["p2"] is None) if kind == EXP else np.array_equal(m["p2"], p2)
    with pytest.raises(ValueError):
        C.posterior_means(p, q[:-1])


def test_python_refusals_before_any_device_call():
    p = proc(EXP)
    net = nhp.ContinuousNetworkHawkesProcess(p.baseline, p.impulses, p.weights, np.ones((3, 3)), nhp.DenseNetworkModel(3))
    data = (np.array([0.5, 1.0]), np.array([1, 2]), 2.0)
    for f in (lambda: C.vb_device_(net, data), lambda: C.vb_statistics(net, data, np.ones(C.vb_size(p))), lambda: C.prior_variational_params(net)):
        with pytest.raises(ValueError):
            f()
    lg = nhp.ContinuousStandardHawkesProcess(nhp.LogGaussianCoxProcess([0.0, 2.0], np.ones((3, 2))), p.impulses, p.weights)
    with pytest.raises(ValueError):
        C.vb_device_(lg, data)
