"""NumPy restatement of the continuous event-history formulas with a piecewise-linear baseline (LogGaussianCoxProcess,
baselines.jl:187-336; utils/interpolation.jl:27-36) -- TEST INFRASTRUCTURE ONLY.

The C oracle (oracle/) restates the reference with a homogeneous baseline.  This module states the same formulas with the baseline
read per event, lambda0_c(t_i), so that the device's grid-baseline paths have a reference: the windowed log-likelihood with the
trapezoid compensator, the intensities at the events and at query times, and the adjacency Gibbs sweep (continuous.jl:444-519) whose
total intensity (continuous.jl:391-405) carries the curve.  With `x = None` every function takes the homogeneous `lambda0` instead,
which tests/test_grid_reference_cpu.py pins against the C oracle."""
import numpy as np

INVSQRT2PI = 0.3989422804014327


def interp(x, y, t):
    """LinearInterpolator(x, y)(t) in the form of grid_interp (csrc/cont_baseline.cu): y[G-1] at t = x[G-1] exactly, else the
    interpolation.jl:31 form on the last segment with x[g] <= t.  Times outside [x[0], x[G-1]] raise (the reference's DomainError)."""
    x, y, t = np.asarray(x, np.float64), np.asarray(y, np.float64), np.asarray(t, np.float64)
    if np.any(t < x[0]) or np.any(t > x[-1]):
        raise ValueError("Value is outside interpolation support")
    lo = np.clip(np.searchsorted(x, t, side="right") - 1, 0, x.size - 2)
    x0, x1 = x[lo], x[lo + 1]
    v = (y[lo + 1] * (t - x0) + y[lo] * (x1 - t)) / (x1 - x0)
    return np.where(t >= x[-1], y[-1], v)


def trapezoid(x, y):
    """integrate(LinearInterpolator): the trapezoid sum, term by term in grid order (baselines.jl:336)."""
    s = 0.0
    for g in range(len(x) - 1):
        s += 0.5 * (y[g] + y[g + 1]) * (x[g + 1] - x[g])
    return s


class Model:
    """kind 0: Exponential (p1 = theta), 1: LogitNormal (p1 = mu, p2 = tau).  Matrices are [parent, child]; A = None: Standard
    process.  x, lam: the curves (lam[k, g] at x[g]), or x = None for the homogeneous lambda0."""

    def __init__(self, kind, lambda0, W, p1, p2=None, A=None, dtmax=np.inf, x=None, lam=None):
        self.kind, self.dtmax = int(kind), float(dtmax)
        self.lambda0 = np.asarray(lambda0, np.float64)
        self.K = self.lambda0.size
        self.W, self.p1 = np.asarray(W, np.float64), np.asarray(p1, np.float64)
        self.p2 = None if p2 is None else np.asarray(p2, np.float64)
        self.A = None if A is None else np.asarray(A, np.float64)
        self.x = None if x is None else np.asarray(x, np.float64)
        self.lam = None if lam is None else np.asarray(lam, np.float64)

    # ---- pieces
    def pdf(self, p, c, dt):
        """impulses.jl:106-108 (Exponential(1 ./ theta)) and :174-178 (LogitNormal, no 1/dtmax Jacobian), elementwise."""
        dt = np.asarray(dt, np.float64)
        if self.kind == 0:
            rate = 1.0 / (1.0 / self.p1[p, c])
            return np.where(dt < 0.0, 0.0, rate * np.exp(-rate * np.where(dt < 0.0, 0.0, dt)))
        x = dt / self.dtmax
        ok = (0.0 < x) & (x < 1.0)
        xs = np.where(ok, x, 0.5)
        sigma = self.p2[p, c] ** -0.5
        z = (np.log(xs / (1.0 - xs)) - self.p1[p, c]) / sigma
        return np.where(ok, np.exp(-(z * z) / 2.0) * INVSQRT2PI / sigma / (xs * (1.0 - xs)), 0.0)

    def rates(self, c, t):
        """lambda0_c(t) for nodes c (0-based) at times t."""
        c, t = np.asarray(c), np.asarray(t, np.float64)
        if self.x is None:
            return self.lambda0[c] + 0.0 * t
        out = np.empty(t.shape)
        for k in np.unique(c):
            sel = c == k
            out[sel] = interp(self.x, self.lam[k], t[sel])
        return out

    def integral(self, duration):
        """sum_k integrated_intensity(baseline_k, duration)."""
        if self.x is None:
            return float(np.sum(self.lambda0 * duration))
        return float(sum(trapezoid(self.x, self.lam[k]) for k in range(self.K)))

    def pairs(self, events, idx):
        """(child position in idx, predecessor j) of every event idx[r] and every j in its window: the earlier events with
        t_j > t_i - dtmax (continuous.jl:391-405)."""
        lo = np.searchsorted(events, events[idx] - self.dtmax, side="right")
        lo = np.minimum(lo, idx)
        cnt = idx - lo
        r = np.repeat(np.arange(idx.size), cnt)
        j = np.repeat(lo, cnt) + (np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt))
        return r, j

    def column_impulses(self, events, nodes, c):
        """G[r, p] = W[p, c] sum_{j in win(i_r), node j = p} h_pc(t_i - t_j) for the events i_r on column c (0-based)."""
        idx = np.flatnonzero(nodes - 1 == c)
        r, j = self.pairs(events, idx)
        p = nodes[j] - 1
        G = np.zeros((idx.size, self.K))
        np.add.at(G, (r, p), self.W[p, c] * self.pdf(p, c, events[idx][r] - events[j]))
        return idx, G

    # ---- reference functions
    def event_intensity(self, events, nodes):
        events, nodes = np.asarray(events, np.float64), np.asarray(nodes, np.int64)
        out = self.rates(nodes - 1, events)
        for c in range(self.K):
            idx, G = self.column_impulses(events, nodes, c)
            if idx.size:
                out[idx] += G @ (np.ones(self.K) if self.A is None else self.A[:, c])
        return out

    def loglik(self, events, nodes, duration):
        """The windowed log-likelihood (continuous.jl:210-239 / 360-389): -sum_k integrate(lambda0_k) - sum_i rowsum(c_i) +
        sum_i log lambda_i."""
        events, nodes = np.asarray(events, np.float64), np.asarray(nodes, np.int64)
        Aeff = self.W if self.A is None else self.A * self.W
        comp = float(np.sum(Aeff.sum(axis=1)[nodes - 1]))
        return float(np.sum(np.log(self.event_intensity(events, nodes)))) - self.integral(duration) - comp

    def intensity(self, events, nodes, times):
        """continuous.jl:76-96: strict window t0 - dtmax < t_j < t0, all K children; out[q, c]."""
        events, nodes, times = np.asarray(events, np.float64), np.asarray(nodes, np.int64), np.asarray(times, np.float64)
        Aeff = self.W if self.A is None else self.A * self.W
        out = np.empty((times.size, self.K))
        for q, t0 in enumerate(times):
            sel = (t0 - self.dtmax < events) & (events < t0)
            p = nodes[sel] - 1
            for c in range(self.K):
                out[q, c] = self.rates(np.array([c]), np.array([t0]))[0] + np.sum(Aeff[p, c] * self.pdf(p, c, t0 - events[sel]))
        return out

    def resample_adjacency(self, A, rho, events, nodes, duration, u, col_begin=0, col_stride=1):
        """continuous.jl:444-487 on the columns c % col_stride == col_begin: for p = 1..K in order, ll0 / ll1 with A[p, c] = 0 / 1,
        A[p, c] = (u[p, c] <= exp(ll1 - logsumexp(ll0, ll1))).  The first event never contributes its log term (quirk Q4)."""
        events, nodes = np.asarray(events, np.float64), np.asarray(nodes, np.int64)
        A = np.array(A, np.float64)
        rho, u = np.broadcast_to(np.asarray(rho, np.float64), A.shape), np.asarray(u, np.float64)
        counts = np.bincount(nodes - 1, minlength=self.K).astype(np.float64)
        for c in range(col_begin, self.K, col_stride):
            idx, G = self.column_impulses(events, nodes, c)
            keep = idx != 0
            b = self.rates(np.full(idx.size, c), events[idx])
            I0 = self.lambda0[c] * duration if self.x is None else trapezoid(self.x, self.lam[c])
            for p in range(self.K):
                ll = []
                for a in (0.0, 1.0):
                    A[p, c] = a
                    lam = b + G @ A[:, c]
                    ll.append(-(I0 + float(np.sum(A[:, c] * self.W[:, c] * counts))) + float(np.sum(np.log(lam[keep]))))
                ll0, ll1 = ll[0] + np.log(1.0 - rho[p, c]), ll[1] + np.log(rho[p, c])
                mx = max(ll0, ll1)
                Z = mx + np.log(np.exp(ll0 - mx) + np.exp(ll1 - mx))
                A[p, c] = 1.0 if u[p, c] <= np.exp(ll1 - Z) else 0.0
        return A
