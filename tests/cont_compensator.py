"""The law of a continuous Hawkes sample with LogGaussianCox curves, as a test: the time-rescaling theorem.

The compensator of node c, Lambda_c(t) = int_0^t lambda0_c + sum over earlier events j with A[c_j, c] set of W[c_j, c] G(t - t_j), with
lambda0_c the piecewise-linear curve and G the integrated impulse response, maps the events of node c to a unit-rate Poisson process:
its increments between consecutive events of c (from 0 to the first) are i.i.d. Exp(1) (Brown et al. 2002).  A wrong baseline shows in
the Kolmogorov-Smirnov test of the increments.  Integrated impulses: Exponential W (1 - e^{-theta d}) (no truncation, as the
simulators draw it); LogitNormal W Phi((logit(d / dtmax) - mu) sqrt(tau)) below dtmax and W beyond (with dtmax = 1 the impulse
integrates to 1, the simulators' Poisson(W) children per event)."""
import numpy as np
from scipy import stats

KS_P_MIN = 1e-3


def baseline_integral(x, y, t):
    """int_0^t of the piecewise-linear curve (x, y) at the times t (the grid covers [0, max t])."""
    x, y, t = np.asarray(x, float), np.asarray(y, float), np.asarray(t, float)
    cum = np.concatenate([[0.0], np.cumsum(0.5 * (y[1:] + y[:-1]) * np.diff(x))])

    def F(s):  # int_{x[0]}^s
        g = np.clip(np.searchsorted(x, s, side="right") - 1, 0, x.size - 2)
        return cum[g] + 0.5 * (s - x[g]) * (y[g] + np.interp(s, x, y))

    return F(t) - F(np.zeros(1))[0]


def compensator(t, nodes, x, values, W, A=None, kind="ln", p1=None, p2=None, dtmax=1.0):
    """Lambda_{c_i}(t_i) at every event i of a sorted sample (nodes 1-based); values[k] is node k's curve on grid x."""
    t, c = np.asarray(t, float), np.asarray(nodes, np.int64) - 1
    K = values.shape[0]
    AW = W if A is None else W * A
    out = np.empty(t.size)
    for k in range(K):
        on = c == k
        out[on] = baseline_integral(x, values[k], t[on])
    if not np.any(AW):
        return out
    if kind == "exp":  # S[p, c] = sum over events j on p of e^{-theta (t - t_j)}, decayed event by event
        N, S, tp = np.zeros(K), np.zeros((K, K)), 0.0
        for i in range(t.size):
            S *= np.exp(-p1 * (t[i] - tp))
            tp = t[i]
            out[i] += np.sum(AW[:, c[i]] * (N - S[:, c[i]]))
            N[c[i]] += 1.0
            S[c[i], :] += 1.0
        return out
    # LogitNormal: parents older than dtmax count fully, the ones inside the window through the LogitNormal CDF
    for p in range(K):
        tp = t[c == p]
        out += AW[p, c] * np.searchsorted(tp, t - dtmax, side="right")
    lo = np.searchsorted(t, t - dtmax, side="right")
    n_in = np.arange(t.size) - lo
    i = np.repeat(np.arange(t.size), n_in)
    j = np.repeat(lo - np.cumsum(np.concatenate([[0], n_in[:-1]])), n_in) + np.arange(i.size)
    d = (t[i] - t[j]) / dtmax
    keep = (d > 0.0) & (d < 1.0)
    i, j, d = i[keep], j[keep], d[keep]
    z = (np.log(d / (1.0 - d)) - p1[c[j], c[i]]) * np.sqrt(p2[c[j], c[i]])
    np.add.at(out, i, AW[c[j], c[i]] * stats.norm.cdf(z))
    return out


def rescaling_pvalues(t, nodes, x, values, **model):
    """[K, 2] per node: the KS p-values of (0) the compensator's increments against Exp(1) and (1) the rescaled times
    Lambda(t_i) / Lambda(t_n), i < n, against U(0, 1) (given the n-th point of a unit Poisson process, the earlier ones are uniform
    order statistics on [0, Lambda(t_n)]).  The increments' marginal law is blind to a rate that is wrong slowly, up here and down
    there; the uniformity of the rescaled times is not."""
    lam = compensator(t, nodes, x, values, **model)
    c = np.asarray(nodes, np.int64) - 1
    out = np.empty((values.shape[0], 2))
    for k in range(values.shape[0]):
        lk = lam[c == k]
        out[k, 0] = stats.kstest(np.diff(np.concatenate([[0.0], lk])), "expon").pvalue
        out[k, 1] = stats.kstest(lk[:-1] / lk[-1], "uniform").pvalue
    return out


def rescaling_holds(t, nodes, x, values, **model):
    """The pass condition: every p-value above 1e-3 / (2 K) (Bonferroni across the nodes and the two tests)."""
    p = rescaling_pvalues(t, nodes, x, values, **model)
    return bool(np.all(p > KS_P_MIN / p.size)), p


def time_averaged(x, values, T):
    """The negative control of the time averages: constant curves at each curve's mean over [0, T], on the same grid."""
    avg = np.array([baseline_integral(x, v, [T])[0] for v in values]) / T
    return np.repeat(avg[:, None], x.size, axis=1)


def reversed_in_time(x, values):
    """The negative control of the reversed curves: lambda(x[0] + x[-1] - t) on a grid symmetric about its midpoint."""
    return values[:, ::-1].copy()
