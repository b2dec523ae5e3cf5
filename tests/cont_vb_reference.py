"""NumPy twin of the continuous mean-field VB step (nhp_cont_vb_stats / nhp_cont_vb_step), for the tests.

Brute force: every event's window of predecessors is evaluated on its own, with the parent probabilities at the effective parameters
of the state q, and the expected statistics and the conjugate update are formed from them in plain double precision.

Layouts are the device's: q = [alphav(K); betav(K); kappav; nuv; atheta; btheta] (Exponential) or [...; kappav; nuv; mv; lambdav; av;
bv] (LogitNormal), every K^2 plane flat as X[p + K c].  Matrices returned here are indexed [parent, child]; `planes` and `pack`
convert.  Nodes are 0-based; kind 0 = Exponential, 1 = LogitNormal.  hyper = [alpha0, beta0, kappa, nu, alpha, beta] or
[alpha0, beta0, kappa, nu, mumu, kappamu, a0, b0]."""
import numpy as np
from scipy.special import digamma

EXP, LN = 0, 1


def nplanes(kind):
    return 4 if kind == EXP else 6


def planes(q, K, kind):
    """q -> (alphav[K], betav[K], [K^2 planes as [p, c] matrices])."""
    q = np.asarray(q, dtype=np.float64)
    KK = K * K
    assert q.size == 2 * K + nplanes(kind) * KK
    return q[:K].copy(), q[K:2 * K].copy(), [q[2 * K + j * KK:2 * K + (j + 1) * KK].reshape(K, K).T.copy() for j in range(nplanes(kind))]


def pack(alphav, betav, mats):
    return np.concatenate([np.asarray(alphav, float), np.asarray(betav, float)] + [np.asarray(m, float).T.ravel() for m in mats])


def effective_params(q, K, kind):
    """(lambda0_eff[K], W_eff[p, c], p1, p2) at which the parent probabilities are the VB responsibilities."""
    av, bv, P = planes(q, K, kind)
    lam0 = np.exp(digamma(av) - np.log(bv))
    lw = digamma(P[0]) - np.log(P[1])
    if kind == EXP:
        th = P[2] / P[3]
        return lam0, np.exp(lw + digamma(P[2]) - np.log(P[3])) / th, th, None
    mv, lv, a, b = P[2], P[3], P[4], P[5]
    return lam0, np.exp(lw + 0.5 * (digamma(a) - np.log(a)) - 0.5 / lv), mv.copy(), a / b


def posterior_means(q, K, kind):
    av, bv, P = planes(q, K, kind)
    if kind == EXP:
        return av / bv, P[0] / P[1], P[2] / P[3], None
    return av / bv, P[0] / P[1], P[2].copy(), P[4] / P[5]


def horizon(kind, dtmax, lam0, W, p1, n_total):
    """The look-back window of the sweeps (nhp_cont_horizon, non-recursive): dtmax for LogitNormal; for Exponential min(dtmax, cut),
    the cut-off beyond which the omitted tail is < 1e-14 of the smallest baseline rate."""
    if kind == LN:
        return float(dtmax)
    act = W != 0.0
    if not act.any():
        return min(float(dtmax), 1e-300)
    th_min, wt_max = float(np.min(p1[act])), float(np.max(np.abs(W[act] * p1[act])))
    h = float(dtmax)
    lmin = float(np.min(lam0))
    if th_min > 0 and np.isfinite(th_min) and lmin > 0 and n_total > 0:
        cut = np.log(n_total * wt_max / (1e-14 * lmin)) / th_min
        if 0 < cut < h:
            h = cut
    return h


def impulse(kind, dt, p1, p2, dtmax):
    """h(dt) per pair (arrays of matching shape); zero outside the support."""
    if kind == EXP:
        return np.where(dt >= 0, p1 * np.exp(-p1 * dt), 0.0)
    D = dtmax
    inside = (dt > 0) & (dt < D)
    dts = np.where(inside, dt, 0.5 * D)
    y = np.log(dts / (D - dts))
    v = D * D * np.sqrt(p2 / (2 * np.pi)) / (dts * (D - dts)) * np.exp(-0.5 * p2 * (y - p1) ** 2)
    return np.where(inside, v, 0.0)


def responsibilities(t, c, K, kind, lam0, W, p1, p2, dtmax, hz):
    """Per event i: (u0, js, u) with u0 the baseline probability and u[m] that of the predecessor js[m] (window t_j > t_i - hz)."""
    t = np.asarray(t, float)
    c = np.asarray(c, int)
    out = []
    for i in range(t.size):
        lo = np.searchsorted(t, t[i] - hz, side="right")
        js = np.arange(lo, i)
        ps = c[js]
        ci = c[i]
        dt = t[i] - t[js]
        val = W[ps, ci] * impulse(kind, dt, p1[ps, ci], None if p2 is None else p2[ps, ci], dtmax)
        Z = lam0[ci] + np.sum(val)
        out.append((lam0[ci] / Z, js, val / Z))
    return out


def expected_stats(t, c, K, kind, q, dtmax, resp=None):
    """dict(M0, Mn, Mnm, S1, S2, resp, hz) of nhp_cont_vb_stats from state q: Mnm = sum u, S1 = sum u dt (Exponential) or
    sum u (y - mv) (LogitNormal), S2 = sum u (y - mv)^2 (LogitNormal), M0[k] = expected baseline events of node k."""
    t = np.asarray(t, float)
    c = np.asarray(c, int)
    lam0, W, p1, p2 = effective_params(q, K, kind)
    hz = horizon(kind, dtmax, lam0, W, p1, t.size)
    if resp is None:
        resp = responsibilities(t, c, K, kind, lam0, W, p1, p2, dtmax, hz)
    M0, Mn = np.zeros(K), np.bincount(c, minlength=K).astype(float)
    Mnm, S1, S2 = np.zeros((K, K)), np.zeros((K, K)), np.zeros((K, K))
    for i, (u0, js, u) in enumerate(resp):
        M0[c[i]] += u0
        if js.size == 0:
            continue
        ps = c[js]
        dt = t[i] - t[js]
        np.add.at(Mnm, (ps, c[i]), u)
        if kind == EXP:
            np.add.at(S1, (ps, c[i]), u * dt)
        else:
            ok = u > 0
            y = np.log(dt[ok] / (dtmax - dt[ok]))
            dz = y - p1[ps[ok], c[i]]
            np.add.at(S1, (ps[ok], c[i]), u[ok] * dz)
            np.add.at(S2, (ps[ok], c[i]), u[ok] * dz * dz)
    return dict(M0=M0, Mn=Mn, Mnm=Mnm, S1=S1, S2=S2, resp=resp, hz=hz)


def m_step(q, K, kind, hyper, T, st):
    """The update of nhp_cont_vb_step from the expected statistics `st` (those of the same q): (q_new, change)."""
    av, bv, P = planes(q, K, kind)
    h = np.asarray(hyper, float)
    n = st["Mnm"]
    a_new, b_new = h[0] + st["M0"], np.full(K, h[1] + T)
    kv, nv = h[2] + n, h[3] + st["Mn"][:, None] * np.ones((1, K))
    if kind == EXP:
        mats = [kv, nv, h[4] + n, h[5] + st["S1"]]
        pos_old, pos_new, mv_old, mv_new = P, mats, None, None
    else:
        mumu, kmu, a0, b0 = h[4], h[5], h[6], h[7]
        with np.errstate(invalid="ignore", divide="ignore"):
            d = np.where(n > 0, st["S1"] / np.where(n > 0, n, 1.0), 0.0)
        ybar = P[2] + d
        S = np.maximum(st["S2"] - n * d * d, 0.0)
        lv = kmu + n
        mv = (kmu * mumu + n * ybar) / lv
        avn = a0 + 0.5 * n
        bvn = b0 + 0.5 * S + kmu * n * (ybar - mumu) ** 2 / (2.0 * lv)
        mats = [kv, nv, mv, lv, avn, bvn]
        pos_old, pos_new, mv_old, mv_new = [P[0], P[1], P[3], P[4], P[5]], [kv, nv, lv, avn, bvn], P[2], mv
    change = max(np.max(np.abs(a_new - av) / av), np.max(np.abs(b_new - bv) / bv))
    for o, w in zip(pos_old, pos_new):
        change = max(change, float(np.max(np.abs(w - o) / o)))
    if mv_old is not None:
        change = max(change, float(np.max(np.abs(mv_new - mv_old))))
    return pack(a_new, b_new, mats), float(change)


def vb_step(t, c, K, kind, q, hyper, T, dtmax):
    st = expected_stats(t, c, K, kind, q, dtmax)
    return m_step(q, K, kind, hyper, T, st) + (st,)


def prior_state(K, kind, hyper):
    h = np.asarray(hyper, float)
    mats = [np.full((K, K), x) for x in (h[2:6] if kind == EXP else h[2:8])]
    return pack(np.full(K, h[0]), np.full(K, h[1]), mats)
