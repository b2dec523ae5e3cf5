"""Host-side mirror of the reference's continuous-time API (Julia absent in this image, so the
host layer above the C ABI is Python; julia/NHPB200.jl holds the ccall shim a maintainer adds).

Same names, argument meaning and error behaviour as the reference:
  components  HomogeneousProcess (baselines.jl:27-39), ExponentialImpulseResponse (impulses.jl:30-37),
              LogitNormalImpulseResponse (impulses.jl:138-148), DenseWeightModel (weights.jl:47-55),
              DenseNetworkModel / BernoulliNetworkModel (networks.jl:20-54)
  processes   ContinuousStandardHawkesProcess (continuous.jl:108-112),
              ContinuousNetworkHawkesProcess (continuous.jl:315-321)
  functions   loglikelihood, intensity, resample_parents, sufficient_statistics, resample_ ("resample!"),
              resample_adjacency_matrix_, mcmc_ ("mcmc!"), mle_ ("mle!"), rand, params / params_; vb_device_ (mean-field VB
              of a standard process on the device, which the reference does not have for continuous processes) and
              network_vb_device_ (the same for a network process, with a variational adjacency matrix)
Matrices are numpy arrays indexed X[parent, child] like the Julia ones; nodes are 1-based.
Everything that touches the event history runs in libnhp on the GPU; the conjugate draws
(O(K^2) host math) stay here, as they stay in Julia.
"""
import ctypes
import time

import numpy as np

from ._lib import NHP_EXPONENTIAL, NHP_LOGITNORMAL
from .core import ContinuousData, Context, _f64, _fmat, _i64, _ptr, default_context


# ------------------------------------------------------------------------------------------
# components
# ------------------------------------------------------------------------------------------
class HomogeneousProcess:
    """baselines.jl:27-39: constant intensity lam ~ Gamma(alpha0, beta0)."""

    def __init__(self, lam, alpha0=1.0, beta0=1.0):
        lam = np.array(lam, dtype=np.float64).reshape(-1)
        if np.any(lam < 0):
            raise ValueError("HomogeneousProcess: intensity parameter λ must be non-negative")  # DomainError baselines.jl:32
        if not alpha0 > 0:
            raise ValueError("HomogeneousProcess: shape parameter α0 must be positive")
        if not beta0 > 0:
            raise ValueError("HomogeneousProcess: rate parameter β0 must be positive")
        self.lam, self.alpha0, self.beta0 = lam, float(alpha0), float(beta0)

    def ndims(self):
        return self.lam.size

    def params(self):
        return self.lam.copy()

    def params_(self, x):
        x = np.asarray(x, dtype=np.float64).reshape(-1)
        if x.size != self.lam.size:
            raise ValueError("Parameter vector length does not match model parameter length.")  # baselines.jl:45
        self.lam = x.copy()

    def resample_(self, M0, duration, rng):
        """baselines.jl:72-77: lam_k ~ Gamma(alpha0 + M0[k], 1/(beta0 + T))."""
        self.lam = rng.gamma(self.alpha0 + M0, 1.0 / (self.beta0 + duration))

    def logprior(self):
        from scipy.stats import gamma
        return float(np.sum(gamma(self.alpha0, scale=1.0 / self.beta0).logpdf(self.lam)))


class LogGaussianCoxProcess:
    """baselines.jl:187-336: lambda_k(t) = exp(m + y_k(t)), y_k ~ GP(0, SquaredExponentialKernel(sigma, eta)) on the grid `x`, linearly
    interpolated in between (utils/interpolation.jl).  `lam[k, g]` are the curve values at the grid points.  On the device the curves
    live inside the sweeps (nhp_cont_baseline_grid); the elliptical-slice update evaluates its likelihood for all nodes at once from the
    device-resident parent assignment (nhp_cont_baseline_loglik), or runs on the device as a whole (resample_device_)."""

    def __init__(self, x, lam, m=0.0, sigma=1.0, eta=1.0):
        self.x = np.array(x, dtype=np.float64).reshape(-1)
        self.lam_grid = np.array(lam, dtype=np.float64)
        if self.lam_grid.ndim != 2 or self.lam_grid.shape[1] != self.x.size:
            raise ValueError("LogGaussianCoxProcess: lam must be [nodes, len(x)]")
        if np.any(self.lam_grid < 0):
            raise ValueError("LogGaussianCoxProcess: intensities must be non-negative")
        self.m, self.sigma, self.eta = float(m), float(sigma), float(eta)
        d = self.x[:, None] - self.x[None, :]
        self.Sigma = self.sigma ** 2 * np.exp(-0.5 * (d / self.eta) ** 2) + 1e-8 * np.eye(self.x.size)
        self._chol = np.linalg.cholesky(self.Sigma)

    @property
    def lam(self):
        """What nhp_cont_params_set takes as lambda0 (the curves replace it on the device): the time averages."""
        return self.integrated_intensity() / (self.x[-1] - self.x[0])

    def ndims(self):
        return self.lam_grid.shape[0]

    def params(self):
        return self.lam_grid.ravel().copy()

    def intensity(self, node, time):
        if time < self.x[0] or time > self.x[-1]:
            raise ValueError("Value is outside interpolation support")  # DomainError interpolation.jl:29
        return float(np.interp(time, self.x, self.lam_grid[node]))

    def integrated_intensity(self):
        return np.trapezoid(self.lam_grid, self.x, axis=1) if hasattr(np, "trapezoid") else np.trapz(self.lam_grid, self.x, axis=1)

    def _clipped(self, duration):
        """The grid clipped to [0, duration] (which it must cover) and the curves' values on it, exact for the piecewise-linear rate."""
        if not (self.x[0] <= 0.0 and self.x[-1] >= duration):
            raise ValueError(f"LogGaussianCoxProcess: the grid [{self.x[0]}, {self.x[-1]}] does not cover [0, {duration}]")
        xs = np.concatenate([[0.0], self.x[(self.x > 0.0) & (self.x < duration)], [float(duration)]])
        return xs, np.stack([np.interp(xs, self.x, y) for y in self.lam_grid])

    def integrated_intensity_on(self, duration):
        """Per node: the integral of the curve over [0, duration] (trapezoid on the clipped grid)."""
        xs, ys = self._clipped(duration)
        return np.sum(0.5 * (ys[:, 1:] + ys[:, :-1]) * np.diff(xs), axis=1)

    def sample(self, node, duration, rng):
        """The baseline events of `node` on [0, duration], sorted: Poisson(max * duration) uniform candidates, each kept with
        probability lambda(t) / max, where max is the curve's maximum on [0, duration] (thinning, as the reference's rejection_sample)."""
        xs, ys = self._clipped(duration)
        top = float(np.max(ys[node]))
        n = rng.poisson(top * duration)
        ts = rng.uniform(0.0, duration, n)
        keep = rng.random(n) * top < np.interp(ts, self.x, self.lam_grid[node])
        return np.sort(ts[keep])

    def logprior(self):
        y = np.log(self.lam_grid) - self.m
        z = np.linalg.solve(self._chol, y.T)
        return float(-0.5 * np.sum(z * z) - self.ndims() * (np.sum(np.log(np.diag(self._chol))) + 0.5 * self.x.size * np.log(2 * np.pi)))

    def resample_(self, ctx, d, rng, max_attempts=100):
        """resample!(process::LogGaussianCoxProcess, data, parents) (baselines.jl:214-254): one elliptical-slice update per node
        [Murray, Adams & MacKay 2010]; all nodes advance together, every attempt is one device evaluation of the K likelihoods."""
        K, G = self.lam_grid.shape
        xs = _f64(self.x)

        def loglik(vals):
            ll = np.empty(K)
            ctx.check(ctx.lib.nhp_cont_baseline_loglik(ctx.h, d.h, G, _ptr(xs), _ptr(_f64(vals.ravel())), _ptr(ll)))
            return ll

        y = np.log(self.lam_grid) - self.m
        nu = (self._chol @ rng.standard_normal((G, K))).T
        lly = loglik(self.lam_grid) + np.log(rng.random(K))
        theta = rng.uniform(0.0, 2.0 * np.pi, K)
        lo, hi = theta - 2.0 * np.pi, theta.copy()
        done = np.zeros(K, dtype=bool)
        ynew = y.copy()
        for _ in range(max_attempts):
            cand = y * np.cos(theta)[:, None] + nu * np.sin(theta)[:, None]
            vals = np.where(done[:, None], np.exp(self.m + ynew), np.exp(self.m + cand))
            ok = (loglik(vals) >= lly) & ~done
            ynew[ok] = cand[ok]
            done |= ok
            if done.all():
                break
            neg = theta < 0.0
            lo = np.where(~done & neg, theta, lo)
            hi = np.where(~done & ~neg, theta, hi)
            theta = np.where(done, theta, rng.uniform(lo, hi))
        else:
            raise RuntimeError("Elliptical slice sampling reached maximum attempts.")  # baselines.jl:316
        self.lam_grid = np.exp(self.m + ynew)
        return self.lam_grid.copy()

    def push_prior(self, ctx):
        """Send the GP prior of the log-curves to the device (nhp_cont_baseline_prior): the Cholesky factor of Sigma and m.  The
        context must hold the curves; setting them again with another grid size, or new parameters, drops the prior."""
        ctx.check(ctx.lib.nhp_cont_baseline_prior(ctx.h, self.x.size, _ptr(_f64(self._chol.ravel(order="F"))), self.m))

    def pull_(self, ctx):
        """Read the device's curves into `lam_grid` (nhp_cont_baseline_get)."""
        v = np.empty(self.lam_grid.size)
        ctx.check(ctx.lib.nhp_cont_baseline_get(ctx.h, _ptr(v)))
        self.lam_grid = v.reshape(self.lam_grid.shape)
        return self.lam_grid

    def resample_device_(self, ctx, d, seed=0, counter=0, z=None, u=None):
        """The update of `resample_` on the device (nhp_cont_resample_baseline), from the parents of the last parent sweep on `d`,
        which must hold the current curves.  Random numbers: Philox keyed by (seed, counter), or the explicit `z[k, g]` standard
        normals and `u[k, j]` uniforms (j = 0 slice height, j = 1 + a angle of attempt a; 101 per node) in the order `resample_`
        consumes them.  Returns the new curves; `last_attempts` holds the candidates each node evaluated."""
        K, G = self.lam_grid.shape
        self.push_prior(ctx)
        zz = uu = None
        if z is not None or u is not None:
            zz, uu = _f64(z).reshape(-1), _f64(u).reshape(-1)
            if zz.size != K * G or uu.size != K * 101:
                raise ValueError("z must hold K x len(x) normals and u K x 101 uniforms")
        att = np.zeros(K, dtype=np.int64)
        ctx.check(ctx.lib.nhp_cont_resample_baseline(ctx.h, d.h, int(seed), int(counter), _ptr(zz), _ptr(uu), _ptr(att)))
        self.last_attempts = att
        return self.pull_(ctx).copy()


class ExponentialImpulseResponse:
    """impulses.jl:30-37: theta[parent, child]; dtmax defaults to Inf."""
    kind = NHP_EXPONENTIAL

    def __init__(self, theta, alpha=1.0, beta=1.0, dtmax=np.inf):
        self.theta = np.array(theta, dtype=np.float64)
        self.alpha, self.beta, self.dtmax = float(alpha), float(beta), float(dtmax)

    def size(self):
        return self.theta.shape[0]

    def params(self):
        return self.theta.T.ravel().copy()  # vec(theta)

    def params_(self, x):
        x = np.asarray(x, dtype=np.float64).reshape(-1)
        if x.size != self.theta.size:
            raise ValueError("Parameter vector length does not match model parameter length.")  # impulses.jl:44-45
        K = self.size()
        self.theta = x.reshape(K, K).T.copy()

    def p1(self):
        return self.theta

    def p2(self):
        return None

    def resample_(self, Mnm, S1, S2, rng):
        """impulses.jl:68-73 with Xnm = duration_mean (0 where Mnm == 0)."""
        with np.errstate(invalid="ignore", divide="ignore"):
            Xnm = np.where(Mnm > 0, S1 / Mnm, 0.0)
        self.theta = rng.gamma(self.alpha + Mnm, 1.0 / (self.beta + Mnm * Xnm))

    def logprior(self):
        from scipy.stats import gamma
        return float(np.sum(gamma(self.alpha, scale=1.0 / self.beta).logpdf(self.theta)))

    def sample(self, p, c, n, rng):
        return np.sort(rng.exponential(1.0 / self.theta[p, c], n))  # impulses.jl:63-66


class LogitNormalImpulseResponse:
    """impulses.jl:138-148: mu, tau [parent, child], support [0, dtmax]."""
    kind = NHP_LOGITNORMAL

    def __init__(self, mu, tau, dtmax, mumu=1.0, kappamu=1.0, alpha0=1.0, beta0=1.0):
        self.mu = np.array(mu, dtype=np.float64)
        self.tau = np.array(tau, dtype=np.float64)
        self.mumu, self.kappamu, self.alpha0, self.beta0, self.dtmax = float(mumu), float(kappamu), float(alpha0), float(beta0), float(dtmax)

    def size(self):
        return self.mu.shape[0]

    def params(self):
        return np.concatenate([self.mu.T.ravel(), self.tau.T.ravel()])

    def params_(self, x):
        x = np.asarray(x, dtype=np.float64).reshape(-1)
        if x.size != self.mu.size + self.tau.size:
            raise ValueError("Parameter vector length does not match model parameter length.")  # impulses.jl:155-156
        K = self.size()
        self.mu = x[: K * K].reshape(K, K).T.copy()
        self.tau = x[K * K:].reshape(K, K).T.copy()

    def p1(self):
        return self.mu

    def p2(self):
        return self.tau

    def resample_(self, Mnm, S1, S2, rng):
        """impulses.jl:204-214 (incl. quirk Q5: beta0 only enters where the statistic is NaN)."""
        with np.errstate(invalid="ignore", divide="ignore"):
            Xnm = S1 / Mnm
            alpha = self.alpha0 + Mnm / 2.0
            beta = S2 / 2.0 + Mnm * self.kappamu / (Mnm + self.kappamu) * (Xnm - self.mumu) ** 2 / 2.0
            beta = np.where(np.isnan(beta), self.beta0, beta)
            self.tau = rng.gamma(alpha, 1.0 / beta)
            kappa = self.kappamu + Mnm
            mun = (self.kappamu * self.mumu + Mnm * Xnm) / (self.kappamu + Mnm)
            mun = np.where(np.isnan(mun), self.mumu, mun)
            sigma = (1.0 / (kappa * self.tau)) ** 0.5
        self.mu = rng.normal(mun, sigma)

    def logprior(self):
        from scipy.stats import gamma, norm
        lp = np.sum(gamma(self.alpha0, scale=1.0 / self.beta0).logpdf(self.tau))
        sigma = 1.0 / np.sqrt(self.kappamu * self.tau)
        return float(lp + np.sum(norm(self.mumu, sigma).logpdf(self.mu)))

    def sample(self, p, c, n, rng):
        z = rng.normal(self.mu[p, c], 1.0 / np.sqrt(self.tau[p, c]), n)  # impulses.jl:196-202
        return np.sort(self.dtmax / (1.0 + np.exp(-z)))


class DenseWeightModel:
    """weights.jl:47-55: W[parent, child] ~ Gamma(kappa, nu)."""

    def __init__(self, W, kappa=1.0, nu=1.0):
        self.W = np.array(W, dtype=np.float64)
        self.kappa, self.nu = float(kappa), float(nu)

    def size(self):
        return self.W.shape[0]

    def params(self):
        return self.W.T.ravel().copy()

    def params_(self, x):
        x = np.asarray(x, dtype=np.float64).reshape(-1)
        if x.size != self.W.size:
            raise ValueError("Parameter vector length does not match model parameter length.")  # weights.jl:10-11
        K = self.size()
        self.W = x.reshape(K, K).T.copy()

    def resample_(self, Mn, Mnm, rng):
        """weights.jl:59-64: W[p,c] ~ Gamma(kappa + Mnm[p,c], 1/(nu + Mn[p])) (also where A == 0, quirk Q14)."""
        self.W = rng.gamma(self.kappa + Mnm, 1.0 / (self.nu + Mn)[:, None] * np.ones_like(Mnm))

    def logprior(self):
        from scipy.stats import gamma
        return float(np.sum(gamma(self.kappa, scale=1.0 / self.nu).logpdf(self.W)))


SparseWeightModel = DenseWeightModel  # weights.jl:105-139: same Gibbs update (kappa1, nu1)


class DenseNetworkModel:
    """networks.jl:20-32"""

    def __init__(self, nnodes):
        self.nnodes = int(nnodes)

    def params(self):
        return np.zeros(0)

    def link_probability(self):
        return np.ones((self.nnodes, self.nnodes))

    def resample_(self, A, rng):
        pass


class BernoulliNetworkModel:
    """networks.jl:45-54: rho ~ Beta(alpha, beta)."""

    def __init__(self, rho, nnodes, alpha=1.0, beta=1.0):
        self.rho, self.nnodes, self.alpha, self.beta = float(rho), int(nnodes), float(alpha), float(beta)

    def params(self):
        return np.array([self.rho])

    def link_probability(self):
        return self.rho * np.ones((self.nnodes, self.nnodes))  # networks.jl:65-68

    def resample_(self, A, rng):
        nlinks = float(np.sum(A))  # networks.jl:72-78
        self.rho = float(rng.beta(self.alpha + nlinks, self.beta + A.size - nlinks))


# ------------------------------------------------------------------------------------------
# processes
# ------------------------------------------------------------------------------------------
class ContinuousHawkesProcess:
    adjacency_matrix = None

    def ndims(self):
        return self.baseline.ndims()

    # ---- device plumbing
    def _ctx(self):
        if getattr(self, "ctx", None) is None:
            self.ctx = default_context()
        return self.ctx

    def _push(self, ctx):
        """Send the current parameters to the device (nhp_cont_params_set)."""
        K = self.ndims()
        imp = self.impulses
        for name, M in (("weights", self.weights.W), ("impulse", imp.p1())):
            if M.shape != (K, K):
                raise ValueError(f"{name} parameter shape {M.shape} does not match the {K} nodes of the baseline")
        A = None if self.adjacency_matrix is None else _fmat(self.adjacency_matrix)
        lam = _f64(self.baseline.lam)
        W = _fmat(self.weights.W)
        p1 = _fmat(imp.p1())
        p2 = None if imp.p2() is None else _fmat(imp.p2())
        ctx.check(ctx.lib.nhp_cont_params_set(ctx.h, imp.kind, K, _ptr(lam), _ptr(W), _ptr(A), _ptr(p1), _ptr(p2), float(imp.dtmax)))
        if isinstance(self.baseline, LogGaussianCoxProcess):  # the curves replace the homogeneous lambda0 inside the sweeps
            b = self.baseline
            ctx.check(ctx.lib.nhp_cont_baseline_grid(ctx.h, b.x.size, _ptr(_f64(b.x)), _ptr(_f64(b.lam_grid.ravel()))))

    def upload(self, data, ctx=None):
        """Make `data = (events, nodes, duration)` device resident; pass the result wherever `data` is accepted."""
        ctx = ctx or self._ctx()
        if isinstance(data, ContinuousData):
            return data
        events, nodes, duration = data
        return ContinuousData(ctx, events, nodes, duration, self.ndims())

    def _data(self, data):
        if isinstance(data, ContinuousData):
            return data, False
        return self.upload(data), True


class ContinuousStandardHawkesProcess(ContinuousHawkesProcess):
    """continuous.jl:108-112"""

    def __init__(self, baseline, impulses, weights):
        self.baseline, self.impulses, self.weights = baseline, impulses, weights

    def params(self):
        return np.concatenate([self.baseline.params(), self.impulses.params(), self.weights.params()])  # continuous.jl:116-119

    def params_(self, x):
        x = np.asarray(x, dtype=np.float64)
        nb, nw, ni = self.baseline.params().size, self.weights.params().size, self.impulses.params().size
        self.baseline.params_(x[:nb])
        self.impulses.params_(x[nb:nb + ni])
        self.weights.params_(x[nb + ni:nb + ni + nw])  # continuous.jl:121-129

    def isstable(self):
        return float(np.max(np.abs(np.linalg.eigvals(self.weights.W)))) < 1.0

    def logprior(self):
        return self.baseline.logprior() + self.weights.logprior() + self.impulses.logprior()  # continuous.jl:278-284


class ContinuousNetworkHawkesProcess(ContinuousHawkesProcess):
    """continuous.jl:315-321"""

    def __init__(self, baseline, impulses, weights, adjacency_matrix, network):
        self.baseline, self.impulses, self.weights, self.network = baseline, impulses, weights, network
        self.adjacency_matrix = np.array(adjacency_matrix, dtype=np.float64)  # Bool / Int64 / Float64 in Julia

    def params(self):
        return np.concatenate([self.network.params(), self.baseline.params(), self.weights.params(), self.impulses.params(),
                               self.adjacency_matrix.T.ravel()])  # continuous.jl:325-333

    def isstable(self):
        return float(np.max(np.abs(np.linalg.eigvals(self.adjacency_matrix * self.weights.W)))) < 1.0


# ------------------------------------------------------------------------------------------
# hot-path functions (all on the GPU through libnhp)
# ------------------------------------------------------------------------------------------
def loglikelihood(process, data, recursive=True):
    """continuous.jl:210-239 / 360-389."""
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        process._push(ctx)
        ll = ctypes.c_double()
        ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, int(bool(recursive)), ctypes.byref(ll)))
        return ll.value
    finally:
        if tmp:
            d.free()


def loglikelihood_gradient(process, data, recursive=True):
    """Extension for `mle!` (the reference differentiates numerically, continuous.jl:185-190): the log-likelihood and its
    analytic gradient from two sweeps (nhp_cont_loglik_grad).  Returns `(ll, grads)` with `grads` a dict of
    `lambda0 [K]`, `W`, `p1`, `p2` as `[parent, child]` matrices (Exponential: p1 = theta; LogitNormal: p1 = mu, p2 = tau)."""
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        process._push(ctx)
        K = process.ndims()
        ll = ctypes.c_double()
        g0, gW, g1 = np.zeros(K), np.zeros(K * K), np.zeros(K * K)
        g2 = np.zeros(K * K) if process.impulses.p2() is not None else None
        ctx.check(ctx.lib.nhp_cont_loglik_grad(ctx.h, d.h, int(bool(recursive)), ctypes.byref(ll), _ptr(g0), _ptr(gW), _ptr(g1), _ptr(g2)))
        unf = lambda v: None if v is None else v.reshape(K, K).T.copy()
        return ll.value, dict(lambda0=g0, W=unf(gW), p1=unf(g1), p2=unf(g2))
    finally:
        if tmp:
            d.free()


def gradient_vector(process, grads):
    """Flatten `loglikelihood_gradient` output in the order of `params(process)` (continuous.jl:116-119)."""
    parts = [grads["lambda0"], grads["p1"].T.ravel()]
    if grads["p2"] is not None:
        parts.append(grads["p2"].T.ravel())
    parts.append(grads["W"].T.ravel())
    return np.concatenate(parts)


def event_intensity(process, data):
    """total_intensity at every event (continuous.jl:286-300 / 391-405)."""
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        process._push(ctx)
        out = np.empty(d.n_own, dtype=np.float64)
        ctx.check(ctx.lib.nhp_cont_event_intensity(ctx.h, d.h, _ptr(out)))
        return out
    finally:
        if tmp:
            d.free()


def intensity(process, data, times):
    """continuous.jl:76-96: `times` Vector -> (len(times), K) matrix; scalar -> (K,) vector."""
    ctx = process._ctx()
    scalar = np.ndim(times) == 0
    tq = _f64(np.atleast_1d(times))
    if np.any(tq < 0):
        raise ValueError("time must be non-negative")  # DomainError baselines.jl:111
    d, tmp = process._data(data)
    try:
        process._push(ctx)
        K = process.ndims()
        out = np.empty(tq.size * K, dtype=np.float64)
        ctx.check(ctx.lib.nhp_cont_intensity(ctx.h, d.h, _ptr(tq), tq.size, _ptr(out)))
        lam = out.reshape(K, tq.size).T.copy()
        return lam[0] if scalar else lam
    finally:
        if tmp:
            d.free()


def resample_parents(process, data, seed=0, counter=0, u=None, export=True, with_loglik=False):
    """parents.jl:1-23 -> (parents, parentnodes), 1-based, 0 = baseline.  with_loglik: the sweep also accumulates the
    log-likelihood terms (read them with sweep_loglikelihood)."""
    ctx = process._ctx()
    ctx.check(ctx.lib.nhp_set_option(ctx.h, 1, int(bool(with_loglik))))
    d, tmp = process._data(data)
    try:
        process._push(ctx)
        return _resample_parents(ctx, d, seed, counter, u, export)
    finally:
        if tmp:
            d.free()


def _resample_parents(ctx, d, seed, counter, u, export):
    par = np.empty(d.n_own, dtype=np.int64) if export else None
    pn = np.empty(d.n_own, dtype=np.int64) if export else None
    uu = None if u is None else _f64(u)
    if uu is not None and uu.size != d.n_own:
        raise ValueError("u must hold one uniform per event")
    ctx.check(ctx.lib.nhp_cont_resample_parents(ctx.h, d.h, int(seed), int(counter), _ptr(uu), _ptr(par), _ptr(pn)))
    return par, pn


def sweep_loglikelihood(process, data):
    """Log-likelihood of the parameters the most recent `resample_parents` sweep on `data` ran with; the sweep
    accumulates the terms while it evaluates the intensities, so no second pass over the events is needed."""
    ctx = process._ctx()
    ll = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_sweep_loglik(ctx.h, data.h, ctypes.byref(ll)))
    return ll.value


def sufficient_statistics(process, data, parents=None):
    """All Gibbs statistics of the current (or given) parent assignment in one call:
    dict(M0, Mn, Mnm, S1, S2) with K x K matrices indexed [parent, child]
    (baselines.jl:79-96, weights.jl:29-43, impulses.jl:75-96, 216-252)."""
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        process._push(ctx)
        if parents is not None:
            par = _i64(parents[0] if isinstance(parents, tuple) else parents)
            ctx.check(ctx.lib.nhp_cont_parents_set(ctx.h, d.h, _ptr(par)))
        return _read_stats(ctx, d, process.ndims())
    finally:
        if tmp:
            d.free()


def _read_stats(ctx, d, K):
    M0, Mn = np.empty(K), np.empty(K)
    Mnm, S1, S2 = np.empty(K * K), np.empty(K * K), np.empty(K * K)
    ctx.check(ctx.lib.nhp_cont_suffstats(ctx.h, d.h, _ptr(M0), _ptr(Mn), _ptr(Mnm), _ptr(S1), _ptr(S2)))
    f = lambda v: v.reshape(K, K).T.copy()
    return dict(M0=M0, Mn=Mn, Mnm=f(Mnm), S1=f(S1), S2=f(S2))


def resample_adjacency_matrix_(process, data, seed=0, counter=0, u=None, col_begin=0, col_stride=1):
    """continuous.jl:444-487; mutates process.adjacency_matrix.  col_begin/col_stride: resample only the columns
    c with c % col_stride == col_begin (multi-GPU column partition; the caller exchanges the owned columns)."""
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        process._push(ctx)
        K = process.ndims()
        rho = _fmat(process.network.link_probability())
        A = _fmat(process.adjacency_matrix).copy()
        uu = None if u is None else _fmat(u)
        ctx.check(ctx.lib.nhp_cont_resample_adjacency_cols(ctx.h, d.h, _ptr(rho), int(seed), int(counter), _ptr(uu), _ptr(A), int(col_begin), int(col_stride)))
        process.adjacency_matrix = A.reshape(K, K).T.copy()
        return process.adjacency_matrix
    finally:
        if tmp:
            d.free()


def resample_(process, data, rng, seed=0, counter=0):
    """One Gibbs sweep, `resample!` (continuous.jl:202-208 / 350-358).  Parent sampling, the
    counters and the impulse statistics run on the GPU in one fused sweep; the conjugate draws
    use `rng` (numpy Generator) on the host."""
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        process._push(ctx)
        _resample_parents(ctx, d, seed, counter, None, False)
        st = _read_stats(ctx, d, process.ndims())
        if isinstance(process.baseline, LogGaussianCoxProcess):
            process.baseline.resample_(ctx, d, rng)
        else:
            process.baseline.resample_(st["M0"], d.duration, rng)
        process.weights.resample_(st["Mn"], st["Mnm"], rng)
        process.impulses.resample_(st["Mnm"], st["S1"], st["S2"], rng)
        if process.adjacency_matrix is not None:
            resample_adjacency_matrix_(process, d, seed=seed, counter=counter + (1 << 40))
            process.network.resample_(process.adjacency_matrix, rng)
        return process.params()
    finally:
        if tmp:
            d.free()


class MarkovChainMonteCarlo:  # inference.jl:22-31
    def __init__(self, samples, elapsed):
        self.samples, self.elapsed = samples, elapsed


def _hyper(process):
    """Hyper-parameters in the order nhp_cont_resample_params expects."""
    b, w, imp = process.baseline, process.weights, process.impulses
    # a LogGaussianCoxProcess baseline has no Gamma prior: the homogeneous draw these two feed is not used while the curves are on the device
    a0, b0 = (1.0, 1.0) if isinstance(b, LogGaussianCoxProcess) else (b.alpha0, b.beta0)
    if imp.kind == NHP_EXPONENTIAL:
        return _f64([a0, b0, w.kappa, w.nu, imp.alpha, imp.beta])
    return _f64([a0, b0, w.kappa, w.nu, imp.mumu, imp.kappamu, imp.alpha0, imp.beta0])


def pull_params_(process, ctx=None):
    """Copy the device-resident parameters (nhp_cont_params_get) into the host-side component objects."""
    ctx = ctx or process._ctx()
    K = process.ndims()
    lam, W, p1 = np.empty(K), np.empty(K * K), np.empty(K * K)
    p2 = np.empty(K * K) if process.impulses.p2() is not None else None
    A = np.empty(K * K) if process.adjacency_matrix is not None else None
    ctx.check(ctx.lib.nhp_cont_params_get(ctx.h, _ptr(lam), _ptr(W), _ptr(A), _ptr(p1), _ptr(p2)))
    unf = lambda v: v.reshape(K, K).T.copy()
    if A is not None:
        process.adjacency_matrix = unf(A)
    if not isinstance(process.baseline, LogGaussianCoxProcess):  # the host holds the curves (the device's lambda0 stands in for them)
        process.baseline.lam = lam
    process.weights.W = unf(W)
    if process.impulses.kind == NHP_EXPONENTIAL:
        process.impulses.theta = unf(p1)
    else:
        process.impulses.mu, process.impulses.tau = unf(p1), unf(p2)
    return process.params()


def resample_on_device_(process, data, rng=None, seed=0, counter=0, push=True, pull=True, baseline_on_device=False):
    """One Gibbs sweep that never leaves the GPU: parent sweep + fused statistics, second pass, the conjugate draws of
    baseline / weights / impulses (nhp_cont_resample_params), and for a network process the adjacency sweep on the
    device-resident matrix (nhp_cont_resample_adjacency_dev) and the Beta draw of rho (nhp_cont_resample_network), with
    every table rebuilt in place.  `push=False` continues from the parameters already on the device (a chain);
    `pull=False` leaves the host objects untouched.
    A LogGaussianCoxProcess baseline takes its elliptical-slice update (with `rng`, or a generator seeded by (seed, counter)) from the
    device-resident parents after the conjugate draws, and its new curves go to the device before the adjacency sweep.  Weights and
    impulses are then drawn before the curves; given the parents they do not depend on them, so the sweep samples the same
    conditionals.  `baseline_on_device=True` runs that update on the device instead (nhp_cont_resample_baseline, Philox keyed by
    (seed, counter)): the curves do not cross PCIe unless `pull`."""
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        net = process.adjacency_matrix is not None
        if push:
            process._push(ctx)
            if net and isinstance(process.network, BernoulliNetworkModel):
                ctx.check(ctx.lib.nhp_cont_network_set(ctx.h, float(process.network.rho)))
        _resample_parents(ctx, d, seed, counter, None, False)
        hy = _hyper(process)
        ctx.check(ctx.lib.nhp_cont_resample_params(ctx.h, d.h, int(seed), int(counter), float(d.duration), _ptr(hy), hy.size, 1))
        b = process.baseline
        if isinstance(b, LogGaussianCoxProcess) and baseline_on_device:
            b.push_prior(ctx)
            ctx.check(ctx.lib.nhp_cont_resample_baseline(ctx.h, d.h, int(seed), int(counter), None, None, None))
            if pull:
                b.pull_(ctx)
        elif isinstance(b, LogGaussianCoxProcess):
            b.resample_(ctx, d, rng if rng is not None else np.random.default_rng([int(seed), int(counter)]))
            # after the slice update: the new curves invalidate the parent assignment it reads
            ctx.check(ctx.lib.nhp_cont_baseline_grid(ctx.h, b.x.size, _ptr(_f64(b.x)), _ptr(_f64(b.lam_grid.ravel()))))
        if net:
            bern = isinstance(process.network, BernoulliNetworkModel)
            ctx.check(ctx.lib.nhp_cont_resample_adjacency_dev(ctx.h, d.h, -1.0 if bern else 1.0, int(seed), int(counter + (1 << 40)), 0, 1, 1))
            if bern:
                rho = ctypes.c_double()
                ctx.check(ctx.lib.nhp_cont_resample_network(ctx.h, int(seed), int(counter), process.network.alpha, process.network.beta, ctypes.byref(rho)))
                process.network.rho = rho.value
        return pull_params_(process, ctx) if pull else None
    finally:
        if tmp:
            d.free()


def mcmc_device_(process, data, nsteps=1000, seed=0, baseline_on_device=False):
    """`mcmc!` (inference.jl:49-70) with the chain AND its sample trace on the device: parameters go up once, every sweep is one
    nhp_cont_gibbs_sweep (which appends its sample to the trace: device-to-device, adjacency bit-packed), and the trace comes back
    in one read at the end.  Returns MarkovChainMonteCarlo with the samples in the order of `params(process)`
    ([rho;] lambda0; theta | mu, tau; W [; vec(A)], continuous.jl:116-119, 325-333); the process holds the last sample.
    A LogGaussianCoxProcess baseline needs `baseline_on_device=True`: its prior goes up with the parameters, every sweep runs the
    elliptical-slice update of the curves on the device, and the samples hold `lam_grid.ravel()` in the baseline's place."""
    lgcp = isinstance(process.baseline, LogGaussianCoxProcess)
    if lgcp and not baseline_on_device:  # the device's draws would leave the curves where they are
        raise ValueError("mcmc_device_: a LogGaussianCoxProcess baseline takes its elliptical-slice update on the host unless "
                         "baseline_on_device=True: pass it, or use mcmc_(device_draws=True)")
    ctx = process._ctx()
    d, tmp = process._data(data)
    t0 = time.time()
    try:
        K = process.ndims()
        net = process.adjacency_matrix is not None
        bern = net and isinstance(process.network, BernoulliNetworkModel)
        process._push(ctx)
        if lgcp:
            process.baseline.push_prior(ctx)
        if bern:
            ctx.check(ctx.lib.nhp_cont_network_set(ctx.h, float(process.network.rho)))
        ctx.check(ctx.lib.nhp_cont_trace_begin(ctx.h, int(nsteps)))
        hy = _hyper(process)
        for step in range(nsteps):
            ctx.check(ctx.lib.nhp_cont_gibbs_sweep(ctx.h, d.h, d.h, int(seed), int(step), float(d.duration), _ptr(hy), hy.size,
                                                   float(process.network.alpha) if bern else 0.0, float(process.network.beta) if bern else 0.0))
        ln = process.impulses.p2() is not None
        rho, l0, W, p1 = np.empty(nsteps), np.empty((nsteps, K)), np.empty((nsteps, K * K)), np.empty((nsteps, K * K))
        p2 = np.empty((nsteps, K * K)) if ln else None
        A = np.empty((nsteps, K * K)) if net else None
        ctx.check(ctx.lib.nhp_cont_trace_read(ctx.h, 0, int(nsteps), _ptr(rho), _ptr(l0), _ptr(W), _ptr(A), _ptr(p1), _ptr(p2)))
        if lgcp:  # the curves take the baseline's place in the samples
            l0 = np.empty((nsteps, process.baseline.lam_grid.size))
            ctx.check(ctx.lib.nhp_cont_trace_read_curves(ctx.h, 0, int(nsteps), _ptr(l0)))
            process.baseline.lam_grid = l0[-1].reshape(process.baseline.lam_grid.shape).copy()
        ctx.check(ctx.lib.nhp_cont_trace_free(ctx.h))
        pull_params_(process, ctx)
        if bern:
            process.network.rho = float(rho[-1])
        samples = []
        for k in range(nsteps):
            imp = [p1[k]] + ([p2[k]] if ln else [])
            if net:  # continuous.jl:325-333: [network; baseline; weights; impulses; vec(A)]
                parts = ([np.array([rho[k]])] if bern else [process.network.params()]) + [l0[k], W[k]] + imp + [A[k]]
            else:    # continuous.jl:116-119: [baseline; impulses; weights]
                parts = [l0[k]] + imp + [W[k]]
            samples.append(np.concatenate(parts))
        return MarkovChainMonteCarlo(samples, time.time() - t0)
    finally:
        if tmp:
            d.free()


# ------------------------------------------------------------------------------------------
# mean-field VB of a standard process (the reference's vb! is discrete only); the state q lives on the device
# ------------------------------------------------------------------------------------------
def _vb_checks(process, name):
    """ValueError, before any device call, for what the device VB does not run."""
    if not isinstance(process, ContinuousStandardHawkesProcess):
        raise ValueError(f"{name}: VB runs a ContinuousStandardHawkesProcess (a network process has no variational adjacency matrix here)")
    if isinstance(process.baseline, LogGaussianCoxProcess):
        raise ValueError(f"{name}: VB takes a HomogeneousProcess baseline (LogGaussianCox curves have no variational factor)")


def vb_size(process):
    """Doubles in the variational state q: 2 K + 4 K^2 (Exponential) or 2 K + 6 K^2 (LogitNormal)."""
    K = process.ndims()
    return 2 * K + (4 if process.impulses.kind == NHP_EXPONENTIAL else 6) * K * K


def prior_variational_params(process):
    """The default start of VB: q set to the priors.  q = [alphav(K); betav(K); kappav; nuv; then atheta; btheta (Exponential) |
    mv; lambdav; av; bv (LogitNormal)], each K^2 plane flat as X[p + K c] (the layout of nhp_cont_vb_set)."""
    _vb_checks(process, "prior_variational_params")
    K = process.ndims()
    b, w, imp = process.baseline, process.weights, process.impulses
    planes = [w.kappa, w.nu] + ([imp.alpha, imp.beta] if imp.kind == NHP_EXPONENTIAL else [imp.mumu, imp.kappamu, imp.alpha0, imp.beta0])
    return np.concatenate([np.full(K, b.alpha0), np.full(K, b.beta0)] + [np.full(K * K, float(x)) for x in planes])


def posterior_means(process, q):
    """Posterior means of the state q: dict(lambda0 = alphav / betav, W = kappav / nuv, p1 = atheta / btheta | mv, p2 = None | av / bv),
    matrices [parent, child] -- what the device holds as parameters after a VB call."""
    K = process.ndims()
    q = _f64(q).reshape(-1)
    if q.size != vb_size(process):
        raise ValueError(f"variational state of {q.size} entries; this process needs {vb_size(process)}")
    KK = K * K
    pl = [q[2 * K + j * KK:2 * K + (j + 1) * KK].reshape(K, K).T for j in range((q.size - 2 * K) // KK)]  # [p + K c] -> [p, c]
    out = dict(lambda0=q[:K] / q[K:2 * K], W=pl[0] / pl[1])
    if process.impulses.kind == NHP_EXPONENTIAL:
        out.update(p1=pl[2] / pl[3], p2=None)
    else:
        out.update(p1=pl[2].copy(), p2=pl[4] / pl[5])
    return out


def _vb_set(ctx, process, q):
    q = _f64(q).reshape(-1)
    if q.size != vb_size(process):
        raise ValueError(f"variational state of {q.size} entries; this process needs {vb_size(process)}")
    hy = _hyper(process)
    process._push(ctx)  # kind, K and dtmax of the state come from the device's parameters
    ctx.check(ctx.lib.nhp_cont_vb_set(ctx.h, _ptr(hy), hy.size, _ptr(q)))
    return q


def vb_statistics(process, data, q):
    """The E-step of VB from state q (nhp_cont_vb_stats): the expected Gibbs statistics dict(M0, Mnm, S1, S2), matrices [parent, child].
    Mnm is the expected parent count, S1 the expected sum of lags (Exponential) or of y - mv with y = logit(lag / dtmax) (LogitNormal),
    S2 the expected sum of (y - mv)^2 (LogitNormal; zeros for Exponential), M0 the expected baseline count per node.  The host objects
    do not change; the device's parameters become the posterior means of q."""
    _vb_checks(process, "vb_statistics")
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        K = process.ndims()
        _vb_set(ctx, process, q)
        M0, Mnm, S1, S2 = np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
        ctx.check(ctx.lib.nhp_cont_vb_stats(ctx.h, d.h, _ptr(M0), _ptr(Mnm), _ptr(S1), _ptr(S2)))
        f = lambda v: v.reshape(K, K).T.copy()
        return dict(M0=M0, Mnm=f(Mnm), S1=f(S1), S2=f(S2))
    finally:
        if tmp:
            d.free()


def vb_device_(process, data, max_steps=100, rtol=None, q0=None, trace=True):
    """Mean-field VB of a ContinuousStandardHawkesProcess with the loop and the state on the device.  The state q0 (default
    prior_variational_params) and the hyper-parameters go up once (nhp_cont_vb_set); each step is one nhp_cont_vb_step: the expected
    parent statistics from two sweeps over the events at the effective parameters, then the conjugate update of q in place.  Without
    `rtol` it runs max_steps steps; with it, it stops after the first step whose change (the largest |new - old| / old over the positive
    entries, |new - old| over mv) is <= rtol.  Returns the list of states q, one per step (`trace=True`: they are kept in a device-side
    trace and come back in one read), or a list holding only the last state (`trace=False`: no trace is kept, which matters at large K:
    one state of K = 5000 is 800 MB).  The process then holds the posterior means of the last state (and the device does too)."""
    _vb_checks(process, "vb_device_")
    if max_steps < 1:
        return []
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        q = _vb_set(ctx, process, prior_variational_params(process) if q0 is None else q0)
        states = _vb_device_loop(ctx, d, q.size, max_steps, rtol, trace)
        pull_params_(process, ctx)
        return states
    finally:
        if tmp:
            d.free()


def _vb_device_loop(ctx, d, size, max_steps, rtol, trace):
    """The step loop of vb_device_ and network_vb_device_ on the state the context keeps (`size` doubles): the states of the steps from
    the device-side trace, or the last state alone."""
    change = ctypes.c_double()
    if trace:
        ctx.check(ctx.lib.nhp_cont_vb_trace_begin(ctx.h, int(max_steps)))
    try:
        steps = 0
        for _ in range(max_steps):
            ctx.check(ctx.lib.nhp_cont_vb_step(ctx.h, d.h, ctypes.byref(change)))
            steps += 1
            if rtol is not None and change.value <= rtol:
                break
        if trace:
            out = np.empty((steps, size))
            ctx.check(ctx.lib.nhp_cont_vb_trace_read(ctx.h, 0, steps, _ptr(out)))
            return list(out)
        last = np.empty(size)
        ctx.check(ctx.lib.nhp_cont_vb_get(ctx.h, _ptr(last)))
        return [last]
    finally:
        if trace:
            ctx.check(ctx.lib.nhp_cont_vb_trace_free(ctx.h))


# ------------------------------------------------------------------------------------------
# mean-field VB of a network process (BernoulliNetworkModel), the model of the discrete network VB: A[p,c] ~ Bernoulli(rho),
# rho ~ Beta(alpha, beta) of the network model, W | A=1 ~ Gamma(kappa, nu) (the slab: the weights model's prior), W | A=0 ~
# Gamma(kappa0, nu0) (the spike), W entering the intensity directly; lambda0 and the impulse as for vb_device_.  The state is the
# standard one followed by kappa0v; nu0v; pv; alpharhov; betarhov, with pv[p + K c] = q(A[p,c] = 1).
# ------------------------------------------------------------------------------------------
def _network_vb_checks(process, name, kappa0=0.1, nu0=10.0):
    """ValueError, before any device call, for what the device network VB does not run."""
    if not isinstance(process, ContinuousNetworkHawkesProcess):
        raise ValueError(f"{name}: network VB runs a ContinuousNetworkHawkesProcess (vb_device_ runs a standard process)")
    if not isinstance(process.network, BernoulliNetworkModel):
        raise ValueError(f"{name}: network VB needs a BernoulliNetworkModel, got {type(process.network).__name__}")
    if isinstance(process.baseline, LogGaussianCoxProcess):
        raise ValueError(f"{name}: VB takes a HomogeneousProcess baseline (LogGaussianCox curves have no variational factor)")
    for nm, v in (("kappa0", kappa0), ("nu0", nu0)):
        if isinstance(v, (bool, np.bool_)) or not (float(v) > 0.0 and np.isfinite(float(v))):
            raise ValueError(f"{name}: {nm} = {v!r} must be positive and finite")


def network_vb_size(process):
    """Doubles in the network VB state: 2 K + 7 K^2 + 2 (Exponential) or 2 K + 9 K^2 + 2 (LogitNormal)."""
    K = process.ndims()
    return 2 * K + (7 if process.impulses.kind == NHP_EXPONENTIAL else 9) * K * K + 2


def network_hyper(process, kappa0=0.1, nu0=10.0):
    """The hyper-parameters of nhp_cont_vb_network_set: those of nhp_cont_vb_set, then kappa0, nu0 and the network model's alpha, beta."""
    _network_vb_checks(process, "network_hyper", kappa0, nu0)
    return np.concatenate([_hyper(process), [float(kappa0), float(nu0), process.network.alpha, process.network.beta]])


def network_prior_variational_params(process, pv=1.0, kappa0=0.1, nu0=10.0):
    """The default start of network VB: the standard factors at their priors (prior_variational_params), kappa0v = kappa0, nu0v = nu0,
    every link probability pv (default 1: every link on) and q(rho) = Beta(alpha, beta) of the network model."""
    _network_vb_checks(process, "network_prior_variational_params", kappa0, nu0)
    pv = float(pv)
    if not 0.0 <= pv <= 1.0:
        raise ValueError(f"network_prior_variational_params: pv = {pv!r} is not a probability")
    K = process.ndims()
    b, w, imp = process.baseline, process.weights, process.impulses
    planes = [w.kappa, w.nu] + ([imp.alpha, imp.beta] if imp.kind == NHP_EXPONENTIAL else [imp.mumu, imp.kappamu, imp.alpha0, imp.beta0])
    planes += [kappa0, nu0, pv]
    return np.concatenate([np.full(K, b.alpha0), np.full(K, b.beta0)] + [np.full(K * K, float(x)) for x in planes] +
                          [[process.network.alpha, process.network.beta]])


def network_posterior_means(process, q):
    """Posterior means of a network state: dict(A = pv, W = pv kappav / nuv + (1 - pv) kappa0v / nu0v (the mixture mean), W_slab =
    kappav / nuv, lambda0, p1, p2 as posterior_means, rho = alpharhov / (alpharhov + betarhov)), matrices [parent, child].  The device
    holds W_slab as W and [A > 1/2] as the adjacency matrix after a network VB call."""
    K = process.ndims()
    q = _f64(q).reshape(-1)
    if q.size != network_vb_size(process):
        raise ValueError(f"network variational state of {q.size} entries; this process needs {network_vb_size(process)}")
    KK, n = K * K, vb_size(process)
    pl = [q[n + j * KK:n + (j + 1) * KK].reshape(K, K).T for j in range(3)]  # kappa0v, nu0v, pv as [p, c]
    kv, nv = q[2 * K:2 * K + KK].reshape(K, K).T, q[2 * K + KK:2 * K + 2 * KK].reshape(K, K).T
    out = dict(lambda0=q[:K] / q[K:2 * K], A=pl[2].copy(), W=pl[2] * kv / nv + (1.0 - pl[2]) * pl[0] / pl[1], W_slab=kv / nv,
               rho=float(q[-2] / (q[-2] + q[-1])))
    pl = [q[2 * K + j * KK:2 * K + (j + 1) * KK].reshape(K, K).T for j in range(2, (n - 2 * K) // KK)]
    if process.impulses.kind == NHP_EXPONENTIAL:
        out.update(p1=pl[0] / pl[1], p2=None)
    else:
        out.update(p1=pl[0].copy(), p2=pl[2] / pl[3])
    return out


def _network_vb_set(ctx, process, q, kappa0, nu0):
    q = _f64(q).reshape(-1)
    if q.size != network_vb_size(process):
        raise ValueError(f"network variational state of {q.size} entries; this process needs {network_vb_size(process)}")
    hy = network_hyper(process, kappa0, nu0)
    process._push(ctx)  # kind, K and dtmax of the state come from the device's parameters; the adjacency matrix makes it a network process
    ctx.check(ctx.lib.nhp_cont_vb_network_set(ctx.h, _ptr(hy), hy.size, _ptr(q)))
    return q


def network_vb_statistics(process, data, q):
    """The E-step of network VB from state q (nhp_cont_vb_stats on a network state): dict(M0, Mnm, S1, S2) as vb_statistics, with the
    effective weights of the mixture.  The host objects do not change; the device then holds the point estimate of q (the slab means
    as W, A = [pv > 1/2], rho)."""
    _network_vb_checks(process, "network_vb_statistics")
    q = _f64(q).reshape(-1)
    if q.size != network_vb_size(process):
        raise ValueError(f"network variational state of {q.size} entries; this process needs {network_vb_size(process)}")
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        K = process.ndims()
        _network_vb_set(ctx, process, q, 0.1, 10.0)  # the spike's hyper-parameters do not enter the E-step
        M0, Mnm, S1, S2 = np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
        ctx.check(ctx.lib.nhp_cont_vb_stats(ctx.h, d.h, _ptr(M0), _ptr(Mnm), _ptr(S1), _ptr(S2)))
        f = lambda v: v.reshape(K, K).T.copy()
        return dict(M0=M0, Mnm=f(Mnm), S1=f(S1), S2=f(S2))
    finally:
        if tmp:
            d.free()


def network_vb_device_(process, data, max_steps=100, rtol=None, q0=None, trace=True, kappa0=0.1, nu0=10.0):
    """Mean-field VB of a ContinuousNetworkHawkesProcess with a BernoulliNetworkModel, shaped like vb_device_: the state q0 (default
    network_prior_variational_params, every link on) and network_hyper go up once (nhp_cont_vb_network_set); each step is one
    nhp_cont_vb_step on the network state.  Returns the states as vb_device_ does.  The process then holds the device's point estimate
    (lambda0, the slab means of W, [pv > 1/2] as its adjacency matrix, the impulse's means), network.rho = alpharhov / (alpharhov +
    betarhov) and network.pv, the link probabilities [parent, child].  A standard process, another network model, a LogGaussianCox
    baseline, a kappa0 / nu0 that is not positive and finite, or a q0 of the wrong size raise ValueError before any device call."""
    _network_vb_checks(process, "network_vb_device_", kappa0, nu0)
    q = network_prior_variational_params(process, 1.0, kappa0, nu0) if q0 is None else _f64(q0).reshape(-1)
    if q.size != network_vb_size(process):
        raise ValueError(f"network_vb_device_: variational state of {q.size} entries; this process needs {network_vb_size(process)}")
    if max_steps < 1:
        return []
    ctx = process._ctx()
    d, tmp = process._data(data)
    try:
        _network_vb_set(ctx, process, q, kappa0, nu0)
        states = _vb_device_loop(ctx, d, q.size, max_steps, rtol, trace)
        pull_params_(process, ctx)
        m = network_posterior_means(process, states[-1])
        process.network.rho, process.network.pv = m["rho"], m["A"]
        return states
    finally:
        if tmp:
            d.free()


def adjacency_info(ctx=None):
    """Diagnostics of the context's last adjacency sweep (nhp_cont_adjacency_info)."""
    ctx = ctx or default_context()
    out = np.zeros(8)
    ctx.lib.nhp_cont_adjacency_info(ctx.h, out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
    keys = ("steps", "batches", "flips", "recomputed_steps", "pairs", "virtual_columns", "sweep_ms", "build_ms")
    d = dict(zip(keys, out.tolist()))
    nv = np.floor(d["virtual_columns"] + 1e-9)
    frac = d["virtual_columns"] - nv  # .CCCBBB: cluster size (CTAs per column; 0 = single-CTA streaming form), bytes per cached pair
    d["virtual_columns"], d["cluster"], d["bytes_per_pair"] = nv, int(round(frac * 1e3 - 0.4)) if frac > 0 else 0, int(round((frac * 1e3 % 1.0) * 1e3)) if frac > 0 else 0
    return d


def mcmc_(process, data, nsteps=1000, log_freq=100, verbose=False, seed=0, device_draws=False, store_every=1, baseline_on_device=False):
    """`mcmc!` (inference.jl:49-70): data is uploaded once and stays on the device.  `device_draws=True` keeps the whole
    sweep on the GPU (resample_on_device_): parameters are pushed once and pulled every `store_every` sweeps (and at the
    end), so neither the K^2 statistics nor the K^2 parameters cross PCIe in between.  With it, `baseline_on_device=True` also
    runs the elliptical-slice update of LogGaussianCoxProcess curves on the device."""
    rng = np.random.default_rng(seed)
    d = process.upload(data)
    t0 = time.time()
    samples = []
    for step in range(nsteps):
        if device_draws:
            keep = (step + 1) % store_every == 0 or step == nsteps - 1
            x = resample_on_device_(process, d, rng, seed=seed, counter=step, push=(step == 0), pull=keep, baseline_on_device=baseline_on_device)
            if keep:
                samples.append(x)
        else:
            samples.append(resample_(process, d, rng, seed=seed, counter=step))
        if verbose and (step + 1) % log_freq == 0:
            print(f" > step: {step + 1}, elapsed: {time.time() - t0:.3f}")
    return MarkovChainMonteCarlo(samples, time.time() - t0)


class MaximumLikelihood:  # inference.jl:1-12
    def __init__(self, maximizer, maximum, steps, elapsed, status):
        self.maximizer, self.maximum, self.steps, self.elapsed, self.status = maximizer, maximum, steps, elapsed, status


def mle_(process, data, regularize=False, guess=None, f_abstol=1e-6, max_iter=200, seed=0, gradient="auto"):
    """`mle!` (continuous.jl:144-198): box-constrained quasi-Newton on [1e-6, 10]; every objective evaluation is one GPU
    log-likelihood on the resident data (SciPy L-BFGS-B stands in for Optim's Fminbox(BFGS())).  `gradient="finite"` is
    the reference's behaviour (finite differences: ~2P sweeps per gradient); `"analytic"` uses the gradient sweep
    (nhp_cont_loglik_grad: two sweeps per objective + gradient).  The default `"auto"` takes the analytic gradient once the
    model has more than 64 parameters (K >= 6): below that 2P tiny log-likelihood launches are cheaper than the scatter
    sweep, whose shared-memory atomics collide when there are only a handful of parent nodes (README example, K = 2:
    0.5 s vs 1.3 s).  With `regularize` the log-prior is differentiated numerically on the host (it costs no sweep)."""
    from scipy.optimize import approx_fprime, minimize
    d = process.upload(data)
    rng = np.random.default_rng(seed)
    x0 = rng.random(process.params().size) if guess is None else np.asarray(guess, dtype=np.float64)
    if gradient == "auto":
        gradient = "analytic" if process.params().size > 64 else "finite"
    analytic = gradient == "analytic" and isinstance(process, ContinuousStandardHawkesProcess)

    def prior(x):
        process.params_(x)
        return process.logprior()

    def objective(x):
        process.params_(x)
        if analytic:
            ll, g = loglikelihood_gradient(process, d)
            gv = gradient_vector(process, g)
            if regularize:
                return -ll - process.logprior(), -gv - approx_fprime(x, prior, 1e-7)
            return -ll, -gv
        ll = loglikelihood(process, d)
        return -ll - process.logprior() if regularize else -ll

    t0 = time.time()
    res = minimize(objective, x0, jac=analytic, method="L-BFGS-B", bounds=[(1e-6, 10.0)] * x0.size, options=dict(ftol=f_abstol * 1e-3, maxiter=max_iter))
    process.params_(res.x)
    return MaximumLikelihood(res.x, -res.fun, res.nit, time.time() - t0, "success" if res.success else "failure")


# ------------------------------------------------------------------------------------------
# rand: on the device (nhp_cont_rand) or on the host (the reference's recursive cluster simulator,
# continuous.jl:16-37, 131-142, 335-348; kept for tiny samples and as an independent check of the device one)
# ------------------------------------------------------------------------------------------
def rand_device(process, duration, seed=0, max_events=None):
    """`rand(process, duration)` simulated on the GPU; returns device-resident data (`.download()` gives the host tuple)."""
    ctx = process._ctx()
    process._push(ctx)
    if max_events is None:  # stationary mean (I - W^T)^-1 lambda0 T with head room; curves: their integrals over [0, duration]
        Weff = process.weights.W if process.adjacency_matrix is None else process.adjacency_matrix * process.weights.W
        rad = float(np.max(np.sum(Weff, axis=1))) if Weff.size else 0.0
        b = process.baseline
        base = float(np.sum(b.integrated_intensity_on(duration))) if isinstance(b, LogGaussianCoxProcess) else float(np.sum(b.lam)) * duration
        mean = base / max(1.0 - min(rad, 0.95), 0.05)
        max_events = int(min(2.1e9, 2.0 * mean + 10.0 * np.sqrt(mean) + 1000))
    h = ctypes.c_void_p()
    ctx.check(ctx.lib.nhp_cont_rand(ctx.h, float(duration), int(seed), int(max_events), ctypes.byref(h)))
    return ContinuousData.from_handle(ctx, h, process.ndims())


def rand(process, duration, rng=None):
    rng = rng or np.random.default_rng()
    K = process.ndims()
    A = process.adjacency_matrix
    W = process.weights.W
    lgcp = isinstance(process.baseline, LogGaussianCoxProcess)
    if lgcp:
        process.baseline._clipped(duration)  # ValueError before any draw when the grid does not cover [0, duration]
    per_node = [[] for _ in range(K)]
    stack = []
    for node in range(K):
        if lgcp:
            ts = process.baseline.sample(node, duration, rng)
        else:
            n = rng.poisson(process.baseline.lam[node] * duration)  # baselines.jl:67-70
            ts = np.sort(rng.uniform(0.0, duration, n))
        per_node[node].extend(ts.tolist())
        stack.extend((t, node) for t in ts)
    while stack:
        t0, p = stack.pop()
        for c in range(K):
            if A is not None and A[p, c] != 1:
                continue
            n = rng.poisson(W[p, c])  # weights.jl:25-27
            if n == 0:
                continue
            ts = t0 + process.impulses.sample(p, c, n, rng)
            ts = ts[ts <= duration]  # truncate (continuous.jl:39-48)
            per_node[c].extend(ts.tolist())
            stack.extend((t, c) for t in ts)
    times = np.concatenate([np.asarray(v, dtype=np.float64) for v in per_node]) if K else np.zeros(0)
    nodes = np.concatenate([np.full(len(v), k + 1, dtype=np.int64) for k, v in enumerate(per_node)]) if K else np.zeros(0, np.int64)
    idx = np.argsort(times, kind="stable")
    return times[idx], nodes[idx], float(duration)
