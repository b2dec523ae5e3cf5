"""NumPy twin of the continuous network VB step (nhp_cont_vb_stats / nhp_cont_vb_step on a state of nhp_cont_vb_network_set), built on
cont_vb_reference.py, for the tests.

The model: A[p,c] ~ Bernoulli(rho), rho ~ Beta(alpha_rho, beta_rho), W | A=1 ~ Gamma(kappa, nu), W | A=0 ~ Gamma(kappa0, nu0), lambda0 and
the impulse as for the standard VB.  q = [standard q; kappa0v; nu0v; pv; alpharhov; betarhov], every K^2 plane flat as X[p + K c];
hyper = [standard hyper; kappa0, nu0, alpha_rho, beta_rho].  The E-step is the standard one with the mixture
lW = pv (psi(kappav) - ln nuv) + (1 - pv) (psi(kappa0v) - ln nu0v).

`elbo` is the bound the step ascends, with the responsibilities at their optimum for q (so their expected complete-data log-likelihood
plus their entropy is sum_i ln Z_i at the effective parameters) and every parent event's whole impulse in the compensator (the W term
is -Mn[p] E[W]).  Each part of the step maximises it over one factor with the others fixed, so it never decreases from step to step."""
import numpy as np
from scipy.special import betaln, digamma, expit, gammaln, xlogy

import cont_vb_reference as R

EXP, LN = R.EXP, R.LN


def nstd(kind):
    """Hyper-parameters of the standard state."""
    return 6 if kind == EXP else 8


def split(q, K, kind):
    """q -> (the standard state, kappa0v, nu0v, pv as [p, c] matrices, alpharhov, betarhov)."""
    q = np.asarray(q, dtype=np.float64)
    KK, n = K * K, 2 * K + R.nplanes(kind) * K * K
    assert q.size == n + 3 * KK + 2
    m = [q[n + j * KK:n + (j + 1) * KK].reshape(K, K).T.copy() for j in range(3)]
    return q[:n].copy(), m[0], m[1], m[2], float(q[-2]), float(q[-1])


def join(qs, k0v, n0v, pv, ar, br):
    return np.concatenate([np.asarray(qs, float)] + [np.asarray(x, float).T.ravel() for x in (k0v, n0v, pv)] + [[ar, br]])


def mixture_lw(q, K, kind):
    """E[ln W] under q(A, W): pv (psi(kappav) - ln nuv) + (1 - pv) (psi(kappa0v) - ln nu0v), [p, c]."""
    qs, k0v, n0v, pv, _, _ = split(q, K, kind)
    _, _, P = R.planes(qs, K, kind)
    return pv * (digamma(P[0]) - np.log(P[1])) + (1.0 - pv) * (digamma(k0v) - np.log(n0v))


def effective_params(q, K, kind):
    """(lambda0_eff, W_eff, p1, p2) of a network state: those of the standard part with its lW replaced by the mixture's."""
    qs = split(q, K, kind)[0]
    lam0, W, p1, p2 = R.effective_params(qs, K, kind)
    _, _, P = R.planes(qs, K, kind)
    return lam0, W * np.exp(mixture_lw(q, K, kind) - (digamma(P[0]) - np.log(P[1]))), p1, p2


def expected_stats(t, c, K, kind, q, dtmax):
    """The statistics of nhp_cont_vb_stats on a network state (the dict of R.expected_stats)."""
    t = np.asarray(t, float)
    c = np.asarray(c, int)
    lam0, W, p1, p2 = effective_params(q, K, kind)
    hz = R.horizon(kind, dtmax, lam0, W, p1, t.size)
    resp = R.responsibilities(t, c, K, kind, lam0, W, p1, p2, dtmax, hz)
    st = R.expected_stats(t, c, K, kind, split(q, K, kind)[0], dtmax, resp=resp)
    st["hz"] = hz
    return st


def m_step(q, K, kind, hyper, T, st):
    """The update of nhp_cont_vb_step on a network state from the statistics `st` of the same q: (q_new, change)."""
    h = np.asarray(hyper, float)
    ns = nstd(kind)
    kap, nu, kap0, nu0, ar0, br0 = h[2], h[3], h[ns], h[ns + 1], h[ns + 2], h[ns + 3]
    qs, k0v, n0v, pv, ar, br = split(q, K, kind)
    qs_new, change = R.m_step(qs, K, kind, h[:ns], T, st)
    _, _, P = R.planes(qs_new, K, kind)
    kv, nv = P[0], P[1]
    k0 = kap0 + st["Mnm"]
    n0 = nu0 + st["Mn"][:, None] * np.ones((1, K))
    cprior = (kap * np.log(nu) - gammaln(kap)) - (kap0 * np.log(nu0) - gammaln(kap0))
    logit = (digamma(ar) - digamma(br)) + (gammaln(kv) - kv * np.log(nv)) - (gammaln(k0) - k0 * np.log(n0)) + cprior
    p = expit(logit)
    S = float(np.sum(p))
    arn, brn = ar0 + S, (br0 + K * K) - S
    change = max(change, float(np.max(np.abs(k0 - k0v) / k0v)), float(np.max(np.abs(n0 - n0v) / n0v)), float(np.max(np.abs(p - pv))),
                 abs(arn - ar) / ar, abs(brn - br) / br)
    return join(qs_new, k0, n0, p, arn, brn), float(change)


def vb_step(t, c, K, kind, q, hyper, T, dtmax):
    st = expected_stats(t, c, K, kind, q, dtmax)
    return m_step(q, K, kind, hyper, T, st) + (st,)


def gamma_kl(a, b, a0, b0):
    """KL(Gamma(a, rate b) || Gamma(a0, rate b0))."""
    return (a - a0) * digamma(a) - gammaln(a) + gammaln(a0) + a0 * (np.log(b) - np.log(b0)) + a * (b0 - b) / b


def elbo(t, c, K, kind, q, hyper, T, dtmax):
    """The bound of the module docstring at state q."""
    t = np.asarray(t, float)
    c = np.asarray(c, int)
    h = np.asarray(hyper, float)
    ns = nstd(kind)
    kap, nu, kap0, nu0, ar0, br0 = h[2], h[3], h[ns], h[ns + 1], h[ns + 2], h[ns + 3]
    qs, k0v, n0v, pv, ar, br = split(q, K, kind)
    av, bv, P = R.planes(qs, K, kind)
    lam0, W, p1, p2 = effective_params(q, K, kind)
    hz = R.horizon(kind, dtmax, lam0, W, p1, t.size)
    lnZ = 0.0
    for i in range(t.size):  # sum_i ln Z_i: the responsibilities' expected log-likelihood plus their entropy at their optimum
        lo = np.searchsorted(t, t[i] - hz, side="right")
        js = np.arange(lo, i)
        val = W[c[js], c[i]] * R.impulse(kind, t[i] - t[js], p1[c[js], c[i]], None if p2 is None else p2[c[js], c[i]], dtmax)
        lnZ += np.log(lam0[c[i]] + np.sum(val))
    Mn = np.bincount(c, minlength=K).astype(float)
    EW = pv * P[0] / P[1] + (1.0 - pv) * k0v / n0v
    val = lnZ - T * np.sum(av / bv) - np.sum(Mn[:, None] * EW)
    val -= np.sum(gamma_kl(av, bv, h[0], h[1]))
    if kind == EXP:
        val -= np.sum(gamma_kl(P[2], P[3], h[4], h[5]))
    else:
        mumu, kmu, a0, b0 = h[4], h[5], h[6], h[7]
        mv, lv, a, b = P[2], P[3], P[4], P[5]
        val -= np.sum(gamma_kl(a, b, a0, b0) + 0.5 * (kmu / lv + kmu * (a / b) * (mv - mumu) ** 2 - 1.0 - np.log(kmu / lv)))
    val -= np.sum(pv * gamma_kl(P[0], P[1], kap, nu) + (1.0 - pv) * gamma_kl(k0v, n0v, kap0, nu0))
    eln1, eln0 = digamma(ar) - digamma(ar + br), digamma(br) - digamma(ar + br)
    val += np.sum(pv * eln1 + (1.0 - pv) * eln0 - xlogy(pv, pv) - xlogy(1.0 - pv, 1.0 - pv))
    val -= betaln(ar0, br0) - betaln(ar, br) + (ar - ar0) * digamma(ar) + (br - br0) * digamma(br) + (ar0 - ar + br0 - br) * digamma(ar + br)
    return float(val)


def prior_state(K, kind, hyper, pv=1.0):
    """The default start: the standard prior state, kappa0v = kappa0, nu0v = nu0, every pv equal, q(rho) = Beta(alpha_rho, beta_rho)."""
    h = np.asarray(hyper, float)
    ns = nstd(kind)
    return join(R.prior_state(K, kind, h[:ns]), np.full((K, K), h[ns]), np.full((K, K), h[ns + 1]), np.full((K, K), float(pv)), h[ns + 2], h[ns + 3])
