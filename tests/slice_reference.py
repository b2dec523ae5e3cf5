"""NumPy restatement of the elliptical-slice update of LogGaussianCoxProcess curves (baselines.jl:214-326), node by node, driven by
explicit random numbers in the layout of nhp_cont_resample_baseline: z[k, g] standard normals (the prior draw is L z_k) and u[k, j]
uniforms, j = 0 the slice height and j = 1 + a the angle uniform of attempt a."""
import ctypes

import numpy as np

MAX_ATTEMPTS = 100
NU = 1 + MAX_ATTEMPTS
TWO_PI = 2.0 * np.pi


def trapezoid(y, x):
    return float(np.sum(0.5 * (y[1:] + y[:-1]) * np.diff(x)))


def node_loglik(x, f, t_k):
    """ll_k(f) = -trapezoid(f) + sum of log f(t_i) over the baseline events t_k of the node."""
    return float(np.sum(np.log(np.interp(t_k, x, f)))) - trapezoid(f, x)


def baseline_events(t, nodes, parents, K):
    """Times of the events whose parent is the baseline (parents 0), per node (nodes 1-based)."""
    t, nodes, parents = np.asarray(t), np.asarray(nodes), np.asarray(parents)
    return [t[(nodes == k + 1) & (parents == 0)] for k in range(K)]


def slice_update(x, lam, L, m, tb, z, u):
    """New curves and the candidates each node evaluated; RuntimeError when a node reaches the attempt limit."""
    K, G = lam.shape
    out, att = lam.copy(), np.zeros(K, dtype=np.int64)
    for k in range(K):
        y = np.log(lam[k]) - m
        nu = L @ z[k]
        lly = node_loglik(x, lam[k], tb[k]) + np.log(u[k, 0])
        theta = 0.0 + (TWO_PI - 0.0) * u[k, 1]
        lo, hi = theta - TWO_PI, theta
        for a in range(MAX_ATTEMPTS):
            f = np.exp(m + (y * np.cos(theta) + nu * np.sin(theta)))
            if node_loglik(x, f, tb[k]) >= lly:
                out[k], att[k] = f, a + 1
                break
            if theta < 0.0:
                lo = theta
            else:
                hi = theta
            if a + 1 == MAX_ATTEMPTS:
                raise RuntimeError("Elliptical slice sampling reached maximum attempts.")
            theta = lo + (hi - lo) * u[k, 2 + a]
    return out, att


class ScriptedRng:
    """Stands in for the numpy Generator that LogGaussianCoxProcess.resample_ consumes: standard_normal((G, K)) returns z, random(K) the
    slice heights, and the n-th call of uniform the angle uniforms u[:, 1 + n] mapped to [lo, hi) as numpy does (lo + (hi - lo) u)."""

    def __init__(self, z, u):
        self.z, self.u, self.col = np.asarray(z), np.asarray(u), 1

    def standard_normal(self, shape):
        assert shape == self.z.T.shape
        return self.z.T.copy()

    def random(self, n):
        return self.u[:n, 0].copy()

    def uniform(self, lo, hi, size=None):
        v = self.u[:, self.col] if self.col < self.u.shape[1] else np.full(self.u.shape[0], 0.5)
        self.col += 1
        lo, hi = np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)
        return lo + (hi - lo) * v


class NumpyLoglikContext:
    """A context whose nhp_cont_baseline_loglik is ll_k(f) of the given baseline events, evaluated in NumPy."""

    def __init__(self, x, tb):
        ctx = self
        self.h, self.tb, self.x, self.calls = None, tb, np.asarray(x), 0

        class Lib:
            @staticmethod
            def nhp_cont_baseline_loglik(h, dh, G, xp, vp, llp):
                K = len(ctx.tb)
                as_arr = lambda p, n: np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_double)), shape=(n,))
                vals = as_arr(vp, K * G).reshape(K, G)
                ll = as_arr(llp, K)
                for k in range(K):
                    ll[k] = node_loglik(ctx.x, vals[k], ctx.tb[k])
                ctx.calls += 1
                return 0
        self.lib = Lib()

    def check(self, rc):
        assert rc == 0
