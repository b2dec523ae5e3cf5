"""Host-side mirror of the reference's discrete-time API over libnhp.

  components  DiscreteHomogeneousProcess (baselines.jl:358-382), DiscreteGaussianImpulseResponse (impulses.jl:272-288)
  processes   DiscreteStandardHawkesProcess (discrete.jl:161-170), DiscreteNetworkHawkesProcess (discrete.jl:395-402)
  functions   basis, convolve, intensity, loglikelihood, resample_parents (reduced over t: counts[c, k]),
              update_ (one VB step, discrete.jl:369-375), resample_ (one Gibbs sweep, discrete.jl:361-367 / 416-424),
              resample_adjacency_matrix_, mcmc_, mcmc_device_ (the chain and its trace on the device), vb_, vb_device_ (the VB loop
              and its trace on the device), svi_schedule and svi_device_ (stochastic VI over windows of bins, on the device),
              network_vb_device_ / network_svi_device_ (VB and SVI of a network process with a variational adjacency matrix, on
              the device) and their host twin network_update_ / network_vb_targets,
              rand (host) and rand_device (nhp_disc_rand: the sample stays on the device)
`data` is an N x T integer matrix (numpy row = node) as in the reference; arrays indexed theta[p, c, b].
"""
import ctypes
import time
import weakref

import numpy as np
from scipy.special import digamma, gammaln

from .continuous import BernoulliNetworkModel, DenseNetworkModel, DenseWeightModel  # noqa: F401
from .core import _f64, _fmat, _ptr, default_context


class DiscreteHomogeneousProcess:
    """baselines.jl:358-382"""

    def __init__(self, lam, dt=1.0, alpha0=1.0, beta0=1.0):
        self.lam = np.array(lam, dtype=np.float64).reshape(-1)
        if np.any(self.lam < 0):
            raise ValueError("DiscreteHomogeneousProcess: intensity parameter λ must be non-negative")
        if not dt > 0:
            raise ValueError("DiscreteHomogeneousProcess: time step dt must be non-negative")
        self.dt, self.alpha0, self.beta0 = float(dt), float(alpha0), float(beta0)
        self.alphav, self.betav = np.ones_like(self.lam), np.ones_like(self.lam)

    def ndims(self):
        return self.lam.size

    def variational_log_expectation(self):
        return digamma(self.alphav) - np.log(self.betav)  # baselines.jl:454-456


class DiscreteGaussianImpulseResponse:
    """impulses.jl:272-288: theta[p, c, b] (rows sum to one over b), nlags, dt."""

    def __init__(self, theta, nlags, dt=1.0, gamma=1.0):
        self.theta = np.array(theta, dtype=np.float64)
        if not np.all(np.sum(self.theta, axis=2) == 1.0) and not np.allclose(np.sum(self.theta, axis=2), 1.0):
            raise ValueError("Invalid discrete basis parameter.")  # impulses.jl:282
        self.nlags, self.dt, self.gamma = int(nlags), float(dt), float(gamma)
        self.gammav = np.ones_like(self.theta)

    def nbasis(self):
        return self.theta.shape[2]

    def basis(self):
        """impulses.jl:321-335 -> phi[l, b] (computed by libnhp's nhp_disc_basis)."""
        from . import _lib
        L, B = self.nlags, self.nbasis()
        phi = np.empty(L * B)
        rc = _lib.load().nhp_disc_basis(L, B, self.dt, _ptr(phi))
        if rc != 0:
            raise ValueError("invalid basis dimensions")
        return phi.reshape(B, L).T.copy()

    def variational_log_expectation(self):
        return digamma(self.gammav) - digamma(np.sum(self.gammav, axis=2, keepdims=True))  # impulses.jl:373-375


class DiscreteData:
    """Device-resident count matrix + its convolution (nhp_disc)."""

    def __init__(self, ctx, data, t_halo=0):
        self.ctx = ctx
        d = np.asarray(data)
        if d.ndim != 2:
            raise ValueError("data must be an N x T matrix")
        self.N, self.T = d.shape
        flat = np.ascontiguousarray(d.T, dtype=np.int64).ravel()  # data[n + N*t]
        h = ctypes.c_void_p()
        ctx.check(ctx.lib.nhp_disc_upload(ctx.h, _ptr(flat), self.N, self.T, int(t_halo), ctypes.byref(h)))
        self.h = h
        self.convolved = False
        self._fin = weakref.finalize(self, ctx.lib.nhp_disc_free, ctx.h, h)

    @classmethod
    def from_handle(cls, ctx, h, N, T):
        """Wrap an unsharded count handle the library created on the device (nhp_disc_rand)."""
        self = cls.__new__(cls)
        self.ctx, self.h, self.N, self.T = ctx, h, int(N), int(T)
        self.convolved = False
        self._fin = weakref.finalize(self, ctx.lib.nhp_disc_free, ctx.h, h)
        return self

    def download(self):
        """The N x T int64 count matrix on the host (every bin, halo included)."""
        flat = np.empty(self.N * self.T, dtype=np.int64)
        self.ctx.check(self.ctx.lib.nhp_disc_download(self.ctx.h, self.h, _ptr(flat)))
        return flat.reshape(self.T, self.N).T.copy()  # data[n + N*t] -> [n, t]

    def events_count(self):
        """Events in the handle's own bins (nhp_disc_events_count)."""
        return int(self.ctx.lib.nhp_disc_events_count(self.h))

    def free(self):
        self._fin()


class DiscreteHawkesProcess:
    adjacency_matrix = None

    def ndims(self):
        return self.baseline.ndims()

    def _ctx(self):
        if getattr(self, "ctx", None) is None:
            self.ctx = default_context()
        return self.ctx

    def _theta_flat(self, th):
        return np.ascontiguousarray(np.asarray(th, dtype=np.float64).transpose(2, 1, 0)).ravel()  # theta[p + N*(c + N*b)]

    def _push(self, ctx):
        N, B = self.ndims(), self.impulses.nbasis()
        if self.weights.W.shape != (N, N) or self.impulses.theta.shape != (N, N, B):
            raise ValueError("parameter shapes do not match the number of nodes")
        A = None if self.adjacency_matrix is None else _fmat(self.adjacency_matrix)
        lam, W, th = _f64(self.baseline.lam), _fmat(self.weights.W), self._theta_flat(self.impulses.theta)
        ctx.check(ctx.lib.nhp_disc_params_set(ctx.h, N, B, _ptr(lam), _ptr(W), _ptr(A), _ptr(th), self.dt))

    def upload(self, data):
        return data if isinstance(data, DiscreteData) else DiscreteData(self._ctx(), data)

    def effective_weights(self):
        """e[p, c] = [A]W[p, c] sum_b theta[p, c, b] sum_l phi_b[l] dt: the expected children on node c of one event on node p."""
        W = self.weights.W if self.adjacency_matrix is None else self.adjacency_matrix * self.weights.W
        return W * np.einsum("pcb,b->pc", self.impulses.theta, self.impulses.basis().sum(axis=0) * self.dt)

    def _ready(self, data):
        d = self.upload(data)
        if not d.convolved:
            convolve(self, d, export=False)
        return d


class DiscreteStandardHawkesProcess(DiscreteHawkesProcess):
    """discrete.jl:161-170"""

    def __init__(self, baseline, impulses, weights, dt=1.0):
        if baseline.dt != dt or impulses.dt != dt:
            raise ValueError("Baseline and impulse response time step must match process time step.")  # intent of discrete.jl:167 (quirk Q13)
        self.baseline, self.impulses, self.weights, self.dt = baseline, impulses, weights, float(dt)

    def params(self):
        eff = (self.weights.W[:, :, None] * self.impulses.theta).transpose(2, 1, 0).ravel()  # vec(W .* theta)
        return np.concatenate([self.baseline.lam, eff])  # discrete.jl:178-182

    def variational_params(self):
        b, w, i = self.baseline, self.weights, self.impulses
        return np.concatenate([b.alphav, b.betav, i.gammav.transpose(2, 1, 0).ravel(), w.kappav.T.ravel(), w.nuv.T.ravel()])  # discrete.jl:204-209


class DiscreteNetworkHawkesProcess(DiscreteHawkesProcess):
    """discrete.jl:395-402"""

    def __init__(self, baseline, impulses, weights, adjacency_matrix, network, dt=1.0):
        self.baseline, self.impulses, self.weights, self.network, self.dt = baseline, impulses, weights, network, float(dt)
        self.adjacency_matrix = np.array(adjacency_matrix, dtype=np.float64)

    def params(self):
        return np.concatenate([self.network.params(), self.baseline.lam, self.weights.W.T.ravel(), self.impulses.theta.transpose(2, 1, 0).ravel(),
                               self.adjacency_matrix.T.ravel()])  # discrete.jl:406-414


# ------------------------------------------------------------------------------------------
def convolve(process, data, export=True):
    """discrete.jl:146-151 -> conv[t, n, b]; the result also stays on the device inside `data` (DiscreteData)."""
    ctx = process._ctx()
    d = process.upload(data)
    phi = process.impulses.basis()
    L, B = phi.shape
    ph = np.ascontiguousarray(phi.T).ravel()
    out = np.empty(d.T * d.N * B) if export else None
    ctx.check(ctx.lib.nhp_disc_convolve(ctx.h, d.h, _ptr(ph), L, B, _ptr(out)))
    d.convolved = True
    return out.reshape(B, d.N, d.T).transpose(2, 1, 0).copy() if export else None


def intensity(process, data):
    """discrete.jl:115-129 -> lam[t, c]."""
    ctx = process._ctx()
    d = process._ready(data)
    process._push(ctx)
    lam = np.empty(d.T * d.N)
    ctx.check(ctx.lib.nhp_disc_intensity(ctx.h, d.h, _ptr(lam)))
    return lam.reshape(d.N, d.T).T.copy()


def loglikelihood(process, data):
    """discrete.jl:86-102."""
    ctx = process._ctx()
    d = process._ready(data)
    process._push(ctx)
    ll = ctypes.c_double()
    ctx.check(ctx.lib.nhp_disc_loglik(ctx.h, d.h, ctypes.byref(ll)))
    return ll.value


def loglikelihood_gradient(process, data):
    """Extension for `mle!` (discrete.jl:211-296; the reference differentiates numerically): the log-likelihood and its analytic
    gradient (nhp_disc_loglik_grad).  Returns `(ll, grads)` with `lambda0 [N]`, `W [p, c]`, `theta [p, c, b]`."""
    ctx = process._ctx()
    d = process._ready(data)
    process._push(ctx)
    N, B = d.N, process.impulses.nbasis()
    ll = ctypes.c_double()
    g0, gW, gT = np.empty(N), np.empty(N * N), np.empty(N * N * B)
    ctx.check(ctx.lib.nhp_disc_loglik_grad(ctx.h, d.h, ctypes.byref(ll), _ptr(g0), _ptr(gW), _ptr(gT)))
    return ll.value, dict(lambda0=g0, W=gW.reshape(N, N).T.copy(), theta=gT.reshape(B, N, N).transpose(2, 1, 0).copy())


def resample_parents(process, data, seed=0, counter=0, u=None):
    """parents.jl:82-117 reduced over t: counts[c, k], k = 0 baseline, k = 1 + p*B + b."""
    ctx = process._ctx()
    d = process._ready(data)
    process._push(ctx)
    N, B = d.N, process.impulses.nbasis()
    NK = 1 + N * B
    counts = np.empty(N * NK)
    uu = None if u is None else _f64(u)
    ctx.check(ctx.lib.nhp_disc_gibbs_counts(ctx.h, d.h, int(seed), int(counter), _ptr(uu), 0 if uu is None else uu.size, _ptr(counts)))
    return counts.reshape(NK, N).T.copy()


def vb_statistics(process, data, e0, E):
    """parents.jl:136-177 fused with baselines.jl:444-452, weights.jl:70-91, impulses.jl:355-371."""
    ctx = process._ctx()
    d = process._ready(data)
    N, B = d.N, process.impulses.nbasis()
    a, k, nu, g = np.empty(N), np.empty(N * N), np.empty(N * N), np.empty(N * N * B)
    Ef = process._theta_flat(E)
    ctx.check(ctx.lib.nhp_disc_vb_stats(ctx.h, d.h, _ptr(_f64(e0)), _ptr(Ef), _ptr(a), _ptr(k), _ptr(nu), _ptr(g)))
    f = lambda v: v.reshape(N, N).T.copy()
    return dict(alpha_sum=a, kappa_sum=f(k), nu_sum=f(nu), gamma_sum=g.reshape(B, N, N).transpose(2, 1, 0).copy())


def update_(process, data):
    """One mean-field VB step, `update!` (discrete.jl:369-375)."""
    b, w, imp = process.baseline, process.weights, process.impulses
    if not hasattr(w, "kappav"):
        w.kappav, w.nuv = np.ones_like(w.W), np.ones_like(w.W)
    e0 = np.exp(b.variational_log_expectation())
    ElogW = digamma(w.kappav) - np.log(w.nuv)  # weights.jl:95-97
    E = np.exp(imp.variational_log_expectation() + ElogW[:, :, None])
    st = vb_statistics(process, data, e0, E)
    d = process.upload(data)
    b.alphav = b.alpha0 + st["alpha_sum"]
    b.betav = 1.0 / b.beta0 + d.T * process.dt * np.ones(d.N)  # baselines.jl:450 (as written in the reference)
    w.kappav = w.kappa + st["kappa_sum"]
    w.nuv = w.nu + st["nu_sum"]
    imp.gammav = imp.gamma + st["gamma_sum"]
    return process.variational_params()


def resample_adjacency_matrix_(process, data, seed=0, counter=0, u=None):
    """discrete.jl:426-460; mutates process.adjacency_matrix."""
    ctx = process._ctx()
    d = process._ready(data)
    process._push(ctx)
    N = d.N
    A = _fmat(process.adjacency_matrix).copy()
    rho = _fmat(process.network.link_probability())
    uu = None if u is None else _fmat(u)
    ctx.check(ctx.lib.nhp_disc_resample_adjacency(ctx.h, d.h, _ptr(rho), int(seed), int(counter), _ptr(uu), _ptr(A)))
    process.adjacency_matrix = A.reshape(N, N).T.copy()
    return process.adjacency_matrix


def resample_(process, data, rng, seed=0, counter=0):
    """One Gibbs sweep, `resample!` (discrete.jl:361-367 / 416-424); conjugate draws on the host (SURVEY.md section 10)."""
    d = process._ready(data)
    N, B = d.N, process.impulses.nbasis()
    C = resample_parents(process, d, seed=seed, counter=counter)  # [c, k]
    b, w, imp = process.baseline, process.weights, process.impulses
    b.lam = rng.gamma(b.alpha0 + C[:, 0], 1.0 / (b.beta0 + d.T * process.dt))  # intended form of baselines.jl:413-419 (quirk Q2)
    Cpb = C[:, 1:].reshape(N, N, B)  # [c, p, b]
    Mnm = Cpb.sum(axis=2).T  # [p, c]
    Mn = vb_row_sums(process, d)
    w.W = rng.gamma(w.kappa + Mnm, (1.0 / (w.nu + Mn))[:, None] * np.ones((N, N)))
    g = imp.gamma + Cpb.transpose(1, 0, 2)  # [p, c, b]
    th = rng.gamma(g, 1.0)
    imp.theta = th / th.sum(axis=2, keepdims=True)  # Dirichlet (impulses.jl:337-353)
    if process.adjacency_matrix is not None:
        resample_adjacency_matrix_(process, d, seed=seed, counter=counter + (1 << 40))
        process.network.resample_(process.adjacency_matrix, rng)
    return process.params()


def resample_on_device_(process, data, rng=None, seed=0, counter=0):
    """One Gibbs sweep, `resample!` (discrete.jl:361-367 / 416-424), with the conjugate draws on the device: the counts of the parent
    sweep stay there (nhp_disc_gibbs_counts with no host copy) and nhp_disc_resample_params draws lambda0, W and the Dirichlet theta
    from them (Philox: seed, counter); the adjacency sweep and the network draw follow as in `resample_`.  `rng` only feeds the
    host-side network draw."""
    d = process._ready(data)
    ctx = process._ctx()
    N, B = d.N, process.impulses.nbasis()
    b, w, imp = process.baseline, process.weights, process.impulses
    Mn = _f64(vb_row_sums(process, d))  # events per node (cached with the data)
    process._push(ctx)
    ctx.check(ctx.lib.nhp_disc_gibbs_counts(ctx.h, d.h, int(seed), int(counter), None, 0, None))
    hy = np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)
    lam, W, th = np.empty(N), np.empty(N * N), np.empty(N * N * B)
    ctx.check(ctx.lib.nhp_disc_resample_params(ctx.h, d.h, int(seed), int(counter), _ptr(Mn), _ptr(hy), hy.size, _ptr(lam), _ptr(W), _ptr(th)))
    b.lam = lam
    w.W = W.reshape(N, N).T.copy()                             # W[p + N c] -> [p, c]
    imp.theta = th.reshape(B, N, N).transpose(2, 1, 0).copy()  # theta[p + N (c + N b)] -> [p, c, b]
    if process.adjacency_matrix is not None:
        resample_adjacency_matrix_(process, d, seed=seed, counter=counter + (1 << 40))
        process.network.resample_(process.adjacency_matrix, rng if rng is not None else np.random.default_rng(seed + counter))
    return process.params()


def vb_row_sums(process, d):
    if not hasattr(d, "_rowsum"):
        N, B = d.N, process.impulses.nbasis()
        st = vb_statistics(process, d, np.ones(N), np.ones((N, N, B)))
        d._rowsum = st["nu_sum"][:, 0].copy()
    return d._rowsum


def mcmc_(process, data, nsteps=1000, seed=0):
    rng = np.random.default_rng(seed)
    d = process._ready(data)
    t0 = time.time()
    samples = [resample_(process, d, rng, seed=seed, counter=s) for s in range(nsteps)]
    from .continuous import MarkovChainMonteCarlo
    return MarkovChainMonteCarlo(samples, time.time() - t0)


def mcmc_device_(process, data, nsteps=1000, seed=0):
    """`mcmc!` (inference.jl:49-70) with the chain AND its sample trace on the device: the parameters (and rho of a Bernoulli network)
    go up once, every sweep is one nhp_disc_gibbs_sweep (Philox keyed by (seed, step), as resample_on_device_; it appends its sample
    to the device-side trace), and the trace comes back in one read at the end.  Returns MarkovChainMonteCarlo with the samples in
    the order of `params(process)` ([rho;] lambda0; vec(W); vec(theta); vec(A) for a network process, discrete.jl:406-414;
    lambda0; vec(W .* theta) for a standard one, discrete.jl:178-182); the process holds the last sample."""
    ctx = process._ctx()
    d = process._ready(data)
    t0 = time.time()
    N, B = d.N, process.impulses.nbasis()
    net = process.adjacency_matrix is not None
    bern = net and isinstance(process.network, BernoulliNetworkModel)
    b, w, imp = process.baseline, process.weights, process.impulses
    process._push(ctx)
    if bern:
        ctx.check(ctx.lib.nhp_disc_network_set(ctx.h, float(process.network.rho)))
    hy = np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)
    ctx.check(ctx.lib.nhp_disc_trace_begin(ctx.h, int(nsteps)))
    try:
        for step in range(nsteps):
            ctx.check(ctx.lib.nhp_disc_gibbs_sweep(ctx.h, d.h, int(seed), int(step), _ptr(hy), hy.size,
                                                   float(process.network.alpha) if bern else 0.0, float(process.network.beta) if bern else 0.0))
        rho, lam, W, th = np.empty(nsteps), np.empty((nsteps, N)), np.empty((nsteps, N * N)), np.empty((nsteps, N * N * B))
        A = np.empty((nsteps, N * N)) if net else None
        ctx.check(ctx.lib.nhp_disc_trace_read(ctx.h, 0, int(nsteps), _ptr(rho), _ptr(lam), _ptr(W), _ptr(A), _ptr(th)))
    finally:
        ctx.check(ctx.lib.nhp_disc_trace_free(ctx.h))
    b.lam = lam[-1].copy()
    w.W = W[-1].reshape(N, N).T.copy()                              # W[p + N c] -> [p, c]
    imp.theta = th[-1].reshape(B, N, N).transpose(2, 1, 0).copy()   # theta[p + N (c + N b)] -> [p, c, b]
    if net:
        process.adjacency_matrix = A[-1].reshape(N, N).T.copy()
    if bern:
        process.network.rho = float(rho[-1])
    samples = []
    for k in range(nsteps):
        if net:    # discrete.jl:406-414: [network; baseline; vec(W); vec(theta); vec(A)]
            parts = ([rho[k:k + 1]] if bern else [process.network.params()]) + [lam[k], W[k], th[k], A[k]]
        else:      # discrete.jl:178-182: [baseline; vec(W .* theta)]
            parts = [lam[k], np.tile(W[k], B) * th[k]]
        samples.append(np.concatenate(parts))
    from .continuous import MarkovChainMonteCarlo
    return MarkovChainMonteCarlo(samples, time.time() - t0)


def vb_(process, data, max_steps=100):
    """`vb!` (inference.jl:153-181; the reference's convergence test is commented out, so it runs max_steps)."""
    d = process._ready(data)
    trace = [update_(process, d) for _ in range(max_steps)]
    return trace


def set_variational_params_(process, q):
    """Inverse of `variational_params` (discrete.jl:204-209): q = [alphav; betav; vec(gammav); vec(kappav); vec(nuv)]."""
    b, w, imp = process.baseline, process.weights, process.impulses
    N, B = process.ndims(), imp.nbasis()
    q = np.asarray(q, dtype=np.float64).reshape(-1)
    if q.size != 2 * N + N * N * (B + 2):
        raise ValueError(f"variational parameter vector of {q.size} entries; N = {N}, B = {B} needs {2 * N + N * N * (B + 2)}")
    o = 2 * N + N * N * B
    b.alphav, b.betav = q[:N].copy(), q[N:2 * N].copy()
    imp.gammav = q[2 * N:o].reshape(B, N, N).transpose(2, 1, 0).copy()  # gammav[p + N (c + N b)] -> [p, c, b]
    w.kappav = q[o:o + N * N].reshape(N, N).T.copy()                     # [p + N c] -> [p, c]
    w.nuv = q[o + N * N:].reshape(N, N).T.copy()


def _vb_device_run(process, d, nsteps, step, network=False):
    """The device VB loop shared by vb_device_, svi_device_ and their network forms: the variational parameters (kappav / nuv
    initialised as update_ does; for `network`, the state of network_variational_params) and the hyper-parameters go up once
    (nhp_disc_vb_set, nhp_disc_vb_network_set), the trace is open for nsteps slots, step(ctx, k) runs step k and returns True to stop
    after it; the trace comes back in one read and the process holds the last state."""
    ctx = process._ctx()
    b, w, imp = process.baseline, process.weights, process.impulses
    N, B = d.N, imp.nbasis()
    if network:
        q = _f64(network_variational_params(process))
        if q.size != _network_q_size(N, B):
            raise ValueError("variational parameter shapes do not match the data's number of nodes")
        hy = _network_hyper(process)
        ctx.check(ctx.lib.nhp_disc_vb_network_set(ctx.h, N, B, process.dt, _ptr(hy), hy.size, _ptr(q)))
    else:
        if not hasattr(w, "kappav"):
            w.kappav, w.nuv = np.ones_like(w.W), np.ones_like(w.W)
        q = _f64(process.variational_params())
        if q.size != 2 * N + N * N * (B + 2):
            raise ValueError("variational parameter shapes do not match the data's number of nodes")
        hy = np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)
        ctx.check(ctx.lib.nhp_disc_vb_set(ctx.h, N, B, process.dt, _ptr(hy), hy.size, _ptr(q)))
    ctx.check(ctx.lib.nhp_disc_vb_trace_begin(ctx.h, int(nsteps)))
    try:
        steps = 0
        for k in range(nsteps):
            stop = step(ctx, k)
            steps += 1
            if stop:
                break
        out = np.empty((steps, q.size))
        ctx.check(ctx.lib.nhp_disc_vb_trace_read(ctx.h, 0, steps, _ptr(out)))
    finally:
        ctx.check(ctx.lib.nhp_disc_vb_trace_free(ctx.h))
    (set_network_variational_params_ if network else set_variational_params_)(process, out[-1])
    return list(out)


def _refuse_network(process, name):
    if isinstance(process, DiscreteNetworkHawkesProcess):
        raise ValueError(f"{name}: the reference's update! of a DiscreteNetworkHawkesProcess is non-functional (quirk Q10); "
                         "VB runs on DiscreteStandardHawkesProcess")


def vb_device_(process, data, max_steps=100, rtol=None):
    """`vb!` (inference.jl:153-181) with the loop and its trace on the device.  The variational parameters (kappav / nuv initialised
    as update_ does) and the hyper-parameters go up once (nhp_disc_vb_set); each step is one nhp_disc_vb_step, the `update!` of
    discrete.jl:369-375 with digamma on the device, which appends the new state to the device-side VB trace; the trace comes back
    in one read.  Without `rtol` it runs max_steps steps, as vb_.  With `rtol` it stops after the first step whose largest relative
    change of any variational parameter, max_i |q_new[i] - q_old[i]| / q_old[i], is <= rtol: a criterion of this package, since the
    reference's own convergence test is commented out (inference.jl:163-176).  Returns the list of variational_params vectors, one
    per step, as vb_; the process holds the last state.  A network process raises ValueError: the reference's update! for it is
    non-functional (quirk Q10)."""
    _refuse_network(process, "vb_device_")
    d = process._ready(data)
    if max_steps < 1:
        return []
    change = ctypes.c_double()

    def step(ctx, k):
        ctx.check(ctx.lib.nhp_disc_vb_step(ctx.h, d.h, None if rtol is None else ctypes.byref(change)))
        return rtol is not None and change.value <= rtol

    return _vb_device_run(process, d, max_steps, step)


def _whole(x, name):
    if isinstance(x, (bool, np.bool_)) or not float(x).is_integer():
        raise ValueError(f"{name} must be an integer, got {x!r}")
    return int(x)


def svi_schedule(T, nsteps, batch_bins, tau0=1.0, kappa=0.75, seed=0):
    """The windows and step sizes of stochastic VI (Hoffman et al. 2013) over T bins: t_begin[k] uniform on [0, T) (an int64 array
    from np.random.default_rng(seed)) and step[k] = (k + 1 + tau0)^(-kappa) for the steps k = 0 .. nsteps - 1, so the first step is
    at most 1 and the steps satisfy sum step = inf, sum step^2 < inf.  Window k covers the batch_bins bins (t_begin[k] + j) mod T; it
    wraps around the end, which keeps every bin's chance of being in it at batch_bins / T.  Checks, with ValueError and before anything
    else: T >= 1, 1 <= batch_bins <= T, 0.5 < kappa <= 1, tau0 >= 0, nsteps >= 0."""
    T, nsteps, batch_bins = _whole(T, "T"), _whole(nsteps, "nsteps"), _whole(batch_bins, "batch_bins")
    if T < 1:
        raise ValueError(f"svi_schedule: T = {T} bins; need at least one")
    if not 1 <= batch_bins <= T:
        raise ValueError(f"svi_schedule: batch_bins = {batch_bins} outside [1, T = {T}]")
    if not 0.5 < kappa <= 1.0:
        raise ValueError(f"svi_schedule: kappa = {kappa} outside (0.5, 1]")
    if not tau0 >= 0.0 or not np.isfinite(tau0):
        raise ValueError(f"svi_schedule: tau0 = {tau0} must be finite and >= 0")
    if nsteps < 0:
        raise ValueError(f"svi_schedule: nsteps = {nsteps} is negative")
    t_begin = np.random.default_rng(seed).integers(0, T, size=nsteps, dtype=np.int64)
    step = (np.arange(1, nsteps + 1, dtype=np.float64) + float(tau0)) ** (-float(kappa))
    return t_begin, step


def svi_device_(process, data, nsteps, batch_bins, tau0=1.0, kappa=0.75, seed=0):
    """Stochastic variational inference (the reference's `svi!`, inference.jl:183-190, is an empty stub) with the loop and its trace
    on the device, shaped like vb_device_: the state goes up once, step k is one nhp_disc_svi_step on the window (t_begin[k],
    batch_bins) with step size step[k] of svi_schedule(T, nsteps, batch_bins, tau0, kappa, seed), and the trace comes back in one read.
    Each step reads only the window's bins and moves q to (1 - step) q + step q*, where q* is the VB update from the window's
    statistics scaled by T / batch_bins.  Returns the list of variational_params vectors, one per step; the process holds the last
    state.  Bad schedule arguments and a network process (quirk Q10) raise ValueError before any device call."""
    T = data.T if isinstance(data, DiscreteData) else np.shape(data)[1]
    t_begin, steps = svi_schedule(T, nsteps, batch_bins, tau0, kappa, seed)
    _refuse_network(process, "svi_device_")
    d = process._ready(data)
    if nsteps < 1:
        return []
    n = int(batch_bins)

    def step(ctx, k):
        ctx.check(ctx.lib.nhp_disc_svi_step(ctx.h, d.h, int(t_begin[k]), n, float(steps[k]), None))
        return False

    return _vb_device_run(process, d, nsteps, step)


# ------------------------------------------------------------------------------------------
# VB and SVI of a network process.  W enters the intensity directly and has a Gamma mixture prior: W | A=1 ~ Gamma(kappa, nu) (the
# slab: the weights model's kappa, nu), W | A=0 ~ Gamma(kappa0, nu0) (the spike, mean kappa0 / nu0), A[p,c] ~ Bernoulli(rho),
# rho ~ Beta(alpha, beta) of the BernoulliNetworkModel.  A true spike W = 0 cannot be used: E[ln W] would be -inf wherever
# q(A=1) < 1.  The factors: q(W | A=1) = Gamma(kappav, nuv), q(W | A=0) = Gamma(kappa0v, nu0v) (weights.kappa0v / nu0v),
# q(A[p,c] = 1) = pv (network.pv), q(rho) = Beta(alphav, betav) (network.alphav / betav).
# ------------------------------------------------------------------------------------------
def _network_q_size(N, B):
    return 2 * N + N * N * (B + 5) + 2


def _spike(w):
    return float(getattr(w, "kappa0", 0.1)), float(getattr(w, "nu0", 10.0))


def _network_hyper(process):
    """[alpha0, beta0, kappa, nu, gamma, kappa0, nu0, alpha_rho, beta_rho], the hyper-parameters of nhp_disc_vb_network_set."""
    b, w, imp, net = process.baseline, process.weights, process.impulses, process.network
    return np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma, *_spike(w), net.alpha, net.beta], dtype=np.float64)


def network_variational_params(process):
    """The network VB state q = [alphav(N); betav(N); vec(gammav)(N*N*B); vec(kappav); vec(nuv); vec(kappa0v); vec(nu0v); vec(pv);
    alpharhov; betarhov] (matrices column-major, [p + N c]): variational_params of the standard process followed by the spike,
    the link probabilities and q(rho).  Missing factors start at kappav = nuv = 1 (as update_), kappa0v = kappa0, nu0v = nu0 (the
    weights' spike hyper-parameters, default 0.1 and 10), pv = rho and q(rho) = Beta(alpha, beta).  adjacency_matrix, W and rho are
    left as they are."""
    b, w, imp, net = process.baseline, process.weights, process.impulses, process.network
    N = process.ndims()
    if not hasattr(w, "kappav"):
        w.kappav, w.nuv = np.ones((N, N)), np.ones((N, N))
    if not hasattr(w, "kappa0v"):
        k0, n0 = _spike(w)
        w.kappa0v, w.nu0v = np.full((N, N), k0), np.full((N, N), n0)
    if not hasattr(net, "pv"):
        net.pv = np.full((N, N), float(net.rho))
    if not hasattr(net, "alphav"):
        net.alphav, net.betav = float(net.alpha), float(net.beta)
    f = lambda M: np.asarray(M, dtype=np.float64).T.ravel()
    return np.concatenate([b.alphav, b.betav, imp.gammav.transpose(2, 1, 0).ravel(), f(w.kappav), f(w.nuv), f(w.kappa0v), f(w.nu0v), f(net.pv),
                           [net.alphav, net.betav]])


def set_network_variational_params_(process, q):
    """Inverse of network_variational_params."""
    b, w, imp, net = process.baseline, process.weights, process.impulses, process.network
    N, B = process.ndims(), imp.nbasis()
    q = np.asarray(q, dtype=np.float64).reshape(-1)
    if q.size != _network_q_size(N, B):
        raise ValueError(f"network variational parameter vector of {q.size} entries; N = {N}, B = {B} needs {_network_q_size(N, B)}")
    NN, o = N * N, 2 * N + N * N * B
    m = lambda k: q[o + k * NN:o + (k + 1) * NN].reshape(N, N).T.copy()  # [p + N c] -> [p, c]
    b.alphav, b.betav = q[:N].copy(), q[N:2 * N].copy()
    imp.gammav = q[2 * N:o].reshape(B, N, N).transpose(2, 1, 0).copy()
    w.kappav, w.nuv, w.kappa0v, w.nu0v, net.pv = m(0), m(1), m(2), m(3), m(4)
    net.alphav, net.betav = float(q[-2]), float(q[-1])


def _network_blocks(q, N, B):
    """Views of the blocks of a network state: alphav, betav, gammav[p, c, b], then kappav, nuv, kappa0v, nu0v, pv as [p, c]."""
    NN, o = N * N, 2 * N + N * N * B
    m = lambda k: q[o + k * NN:o + (k + 1) * NN].reshape(N, N).T
    return q[:N], q[N:2 * N], q[2 * N:o].reshape(B, N, N).transpose(2, 1, 0), m(0), m(1), m(2), m(3), m(4)


def network_expectations(q, N, B):
    """The exp-expectations of a network state in the layouts of vb_statistics: e0[c] = exp(psi(alphav) - ln betav) and
    E[p, c, b] = exp(psi(gammav) - psi(sum_b gammav) + E[ln W]) with the mixture E[ln W] = pv (psi(kappav) - ln nuv) +
    (1 - pv) (psi(kappa0v) - ln nu0v)."""
    q = np.asarray(q, dtype=np.float64)
    av, bv, gv, kv, nv, k0v, n0v, pv = _network_blocks(q, N, B)
    lw = pv * (digamma(kv) - np.log(nv)) + (1.0 - pv) * (digamma(k0v) - np.log(n0v))
    return np.exp(digamma(av) - np.log(bv)), np.exp((digamma(gv) - digamma(gv.sum(axis=2, keepdims=True))) + lw[:, :, None])


def _sigmoid(x):
    with np.errstate(over="ignore", invalid="ignore"):
        return np.where(x >= 0.0, 1.0 / (1.0 + np.exp(-x)), np.exp(x) / (1.0 + np.exp(x)))


def network_vb_targets(q, stats, events, T, dt, hyper, s=1.0):
    """The target q* of one network VB step from the state q and the statistics of a window scaled by s (s = 1 and the whole series
    for VB): `stats` as vb_statistics returns them (alpha_sum[N], kappa_sum[p, c], gamma_sum[p, c, b]) for the expectations of q,
    `events[p]` the events of node p in the window, `hyper` as _network_hyper.  With G = s kappa_sum and E = s events[p]:
    alphav* = alpha0 + s alpha_sum, betav* = 1/beta0 + T dt, gammav* = gamma + s gamma_sum, kappav* = kappa + G, nuv* = nu + E,
    kappa0v* = kappa0 + G, nu0v* = nu0 + E,
      logit pv* = psi(alpharhov) - psi(betarhov) + [lgamma(kappav*) - kappav* ln nuv*] - [lgamma(kappa0v*) - kappa0v* ln nu0v*]
                  + [kappa ln nu - lgamma(kappa)] - [kappa0 ln nu0 - lgamma(kappa0)],
    and, with S = sum pv*, alpharhov* = alpha_rho + S, betarhov* = beta_rho + N^2 - S (N^2 counts links and is not scaled)."""
    q = np.asarray(q, dtype=np.float64)
    h = np.asarray(hyper, dtype=np.float64)
    a = np.asarray(stats["alpha_sum"], dtype=np.float64)
    N = a.size
    NN = N * N
    B = (q.size - 2 * N - 2) // NN - 5
    if q.size != _network_q_size(N, B):
        raise ValueError(f"network variational parameter vector of {q.size} entries does not fit N = {N}")
    G = s * np.asarray(stats["kappa_sum"], dtype=np.float64).T.ravel()
    E = s * np.tile(np.asarray(events, dtype=np.float64), N)  # events[p] at p + N c
    k1, n1, k0, n0 = h[2] + G, h[3] + E, h[5] + G, h[6] + E
    cprior = (h[2] * np.log(h[3]) - gammaln(h[2])) - (h[5] * np.log(h[6]) - gammaln(h[5]))
    logit = (digamma(q[-2]) - digamma(q[-1])) + (gammaln(k1) - k1 * np.log(n1)) - (gammaln(k0) - k0 * np.log(n0)) + cprior
    p = _sigmoid(logit)
    S = float(np.sum(p))
    gs = np.asarray(stats["gamma_sum"], dtype=np.float64).transpose(2, 1, 0).ravel()
    return np.concatenate([h[0] + s * a, np.full(N, 1.0 / h[1] + T * dt), h[4] + s * gs, k1, n1, k0, n0, p, [h[7] + S, (h[8] + NN) - S]])


def network_posterior_means(q, N, B):
    """Posterior means of a network state: A = pv, W = pv kappav / nuv + (1 - pv) kappa0v / nu0v (both [p, c]), theta[p, c, b] =
    gammav / sum_b gammav, lambda0 = alphav / betav and rho = alpharhov / (alpharhov + betarhov)."""
    q = np.asarray(q, dtype=np.float64)
    av, bv, gv, kv, nv, k0v, n0v, pv = _network_blocks(q, N, B)
    return dict(A=pv.copy(), W=pv * kv / nv + (1.0 - pv) * k0v / n0v, theta=gv / gv.sum(axis=2, keepdims=True), lambda0=av / bv,
                rho=float(q[-2] / (q[-2] + q[-1])))


def _network_checks(process, name, kappa0, nu0):
    if not isinstance(process, DiscreteNetworkHawkesProcess):
        raise ValueError(f"{name}: needs a DiscreteNetworkHawkesProcess (vb_device_ / svi_device_ run a standard process)")
    if not isinstance(process.network, BernoulliNetworkModel):
        raise ValueError(f"{name}: network VB needs a BernoulliNetworkModel, got {type(process.network).__name__}")
    for nm, v in (("kappa0", kappa0), ("nu0", nu0)):
        if isinstance(v, (bool, np.bool_)) or not (float(v) > 0.0 and np.isfinite(float(v))):
            raise ValueError(f"{name}: {nm} = {v!r} must be positive and finite")


def network_update_(process, data, kappa0=0.1, nu0=10.0):
    """The host twin of one network VB step (nhp_disc_vb_step on a network state): the expectations of network_expectations, the
    statistics of vb_statistics (device), the events per node of the data and the targets of network_vb_targets with s = 1.  The
    process holds the new state, which is returned."""
    _network_checks(process, "network_update_", kappa0, nu0)
    d = process._ready(data)
    N, B = d.N, process.impulses.nbasis()
    process.weights.kappa0, process.weights.nu0 = float(kappa0), float(nu0)
    q = network_variational_params(process)
    e0, E = network_expectations(q, N, B)
    st = vb_statistics(process, d, e0, E)
    qs = network_vb_targets(q, st, vb_row_sums(process, d), d.T, process.dt, _network_hyper(process), 1.0)
    set_network_variational_params_(process, qs)
    return qs


def network_vb_device_(process, data, max_steps=100, rtol=None, kappa0=0.1, nu0=10.0):
    """Mean-field VB of a discrete network process (BernoulliNetworkModel) with the loop and its trace on the device, shaped like
    vb_device_: network_variational_params(process) and the hyper-parameters go up once (nhp_disc_vb_network_set), each step is one
    nhp_disc_vb_step on the network state (the model and step are those of network_update_), the trace comes back in one read.  With
    `rtol` it stops after the first step whose change (largest relative change of a positive entry, largest absolute change of a
    link probability) is <= rtol.  Returns the list of state vectors, one per step; the process holds the last state.  A standard
    process, another network model or a kappa0 / nu0 that is not positive and finite raise ValueError before any device call."""
    _network_checks(process, "network_vb_device_", kappa0, nu0)
    d = process._ready(data)
    if max_steps < 1:
        return []
    process.weights.kappa0, process.weights.nu0 = float(kappa0), float(nu0)
    change = ctypes.c_double()

    def step(ctx, k):
        ctx.check(ctx.lib.nhp_disc_vb_step(ctx.h, d.h, None if rtol is None else ctypes.byref(change)))
        return rtol is not None and change.value <= rtol

    return _vb_device_run(process, d, max_steps, step, network=True)


def network_svi_device_(process, data, nsteps, batch_bins, tau0=1.0, kappa=0.75, seed=0, kappa0=0.1, nu0=10.0):
    """Stochastic VI of a discrete network process with the loop and its trace on the device, shaped like svi_device_: step k is one
    nhp_disc_svi_step on the network state over the window (t_begin[k], batch_bins) with step size step[k] of svi_schedule(T, nsteps,
    batch_bins, tau0, kappa, seed).  Returns the list of state vectors, one per step; the process holds the last state.  Bad schedule
    arguments and the refusals of network_vb_device_ raise ValueError before any device call."""
    T = data.T if isinstance(data, DiscreteData) else np.shape(data)[1]
    t_begin, steps = svi_schedule(T, nsteps, batch_bins, tau0, kappa, seed)
    _network_checks(process, "network_svi_device_", kappa0, nu0)
    d = process._ready(data)
    if nsteps < 1:
        return []
    process.weights.kappa0, process.weights.nu0 = float(kappa0), float(nu0)
    n = int(batch_bins)

    def step(ctx, k):
        ctx.check(ctx.lib.nhp_disc_svi_step(ctx.h, d.h, int(t_begin[k]), n, float(steps[k]), None))
        return False

    return _vb_device_run(process, d, nsteps, step, network=True)


# ------------------------------------------------------------------------------------------
# rand: on the device (nhp_disc_rand) or on the host (discrete.jl:20-38; sequential over bins, kept for small samples and as an
# independent check of the device one)
# ------------------------------------------------------------------------------------------
def rand_device(process, T, seed=0, max_events=None):
    """`rand(process, T)` simulated on the GPU: an N x T sample with the law `loglikelihood` evaluates, left on the device as
    DiscreteData (`.download()` gives the N x T int64 matrix).  Deterministic in (parameters, T, nlags, seed)."""
    ctx = process._ctx()
    process._push(ctx)
    N, T = process.ndims(), int(T)
    if max_events is None:  # stationary mean (I - e^T)^-1 lambda0 dt T with head room
        e, l0 = process.effective_weights(), process.baseline.lam * process.dt
        rad = float(np.max(np.sum(e, axis=1))) if N else 0.0
        mean = float(np.sum(l0)) * T / max(1.0 - min(rad, 0.95), 0.05)
        if 0 < N <= 2048:  # the exact mean where it is cheap: the row-sum bound misses non-normal e (a chain of strong links)
            m = np.linalg.solve(np.eye(N) - e.T, l0)
            if np.all(np.isfinite(m)) and np.all(m >= 0):  # a non-negative solution: spectral radius of e below 1
                mean = max(mean, float(np.sum(m)) * T)
        max_events = int(min(2.1e9, 2.0 * mean + 10.0 * np.sqrt(mean) + 1000))
    h = ctypes.c_void_p()
    ctx.check(ctx.lib.nhp_disc_rand(ctx.h, T, process.impulses.nlags, int(seed), int(max_events), ctypes.byref(h)))
    return DiscreteData.from_handle(ctx, h, N, T)


def rand(process, T, rng=None):
    """`rand(process, T)` on the host: bin by bin, data[:, t] ~ Poisson(lambda[t, :]) given the earlier bins, with lambda as `intensity`
    computes it (lambda0 dt + sum over lags l = 1..L of data[:, t - l] @ ([A]W theta phi[l] dt)).  Returns the N x T int64 matrix."""
    rng = rng or np.random.default_rng()
    N, T = process.ndims(), int(T)
    W = process.weights.W if process.adjacency_matrix is None else process.adjacency_matrix * process.weights.W
    phi = process.impulses.basis()  # [l, b]
    L = phi.shape[0]
    ir = np.einsum("pcb,lb->lpc", W[:, :, None] * process.impulses.theta, phi) * process.dt  # ir[l - 1, p, c]
    base = process.baseline.lam * process.dt
    data = np.zeros((N, T), dtype=np.int64)
    for t in range(T):
        w = min(L, t)
        lam = base + np.einsum("pl,lpc->c", data[:, t - w:t][:, ::-1], ir[:w]) if w else base
        data[:, t] = rng.poisson(lam)
    return data
