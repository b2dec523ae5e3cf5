"""The conditional law of a discrete Hawkes sample, as a test: given the earlier bins, data[c, t] ~ Poisson(lambda[t, c]) independently.

The randomised probability integral transform F(x - 1; lambda) + V (F(x; lambda) - F(x - 1; lambda)), V ~ U(0, 1), of every bin is then
i.i.d. U(0, 1) (Brockwell 2007); a wrong lambda shows in its Kolmogorov-Smirnov test or in the standardised excess sum(x - lambda) /
sqrt(sum lambda), overall and per node."""
import numpy as np
from scipy import stats

KS_P_MIN, Z_MAX = 1e-3, 5.0


def law_statistics(data, lam, seed=0):
    """data [N, T] counts, lam [T, N] intensities -> (KS p-value of the PIT, overall z, per-node z [N])."""
    x = np.asarray(data, dtype=np.float64).T  # [T, N]
    lo, hi = stats.poisson.cdf(x - 1, lam), stats.poisson.cdf(x, lam)
    u = lo + np.random.default_rng(seed).random(x.shape) * (hi - lo)
    ks = stats.kstest(u.ravel(), "uniform").pvalue
    z = np.sum(x - lam) / np.sqrt(np.sum(lam))
    zn = np.sum(x - lam, axis=0) / np.sqrt(np.sum(lam, axis=0))
    return ks, z, zn


def law_holds(data, lam, seed=0):
    """The pass condition: KS p-value above 1e-3, |z| < 5 overall and per node (for a handful of nodes, 5 sigma each is the
    Bonferroni margin with room to spare)."""
    ks, z, zn = law_statistics(data, lam, seed)
    return bool(ks > KS_P_MIN and abs(z) < Z_MAX and np.all(np.abs(zn) < Z_MAX)), (ks, z, zn)
