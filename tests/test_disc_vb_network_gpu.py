"""VB and SVI of discrete network processes on the device (nhp_disc_vb_network_set, nhp_disc_vb_step / nhp_disc_svi_step on a network
state, discrete.network_vb_device_ / network_svi_device_).

A step takes the expectations of the old state (the mixture E[ln W] on the device), the statistics of nhp_disc_vb_reduce, and writes
the targets of discrete.network_vb_targets blended with the step size.  The host twin discrete.network_update_ uses the same
statistics kernels and SciPy's digamma / gammaln, so the standard blocks agree to the last bits of the digamma, and pv to the
cancellation of its lgamma brackets (each bracket is of the size of kappav* ln nuv*, up to 1e5 here).

Tolerances are the figures measured on a B200 (1000 W power limit), rounded up; where the statistics kernels take part they are
rounded up generously, because the kernels' floating-point atomics sum in an order that changes from run to run."""
import ctypes

import numpy as np
import pytest

import nhp_b200 as nhp
import oracle_ffi as orc
from nhp_b200 import _lib
from nhp_b200 import discrete as D
from nhp_b200.core import Context, _ptr
from test_disc_vb_network_cpu import bound

pytestmark = pytest.mark.gpu


def make(N, T, B, L, seed, rate=0.1):
    rng = np.random.default_rng(seed)
    lam0 = rng.uniform(0.5, 1.5, N) * rate
    A = (rng.random((N, N)) < 0.3).astype(np.float64)
    W = rng.uniform(0.1, 1.0, (N, N)) * 0.5 / N * A
    theta = rng.dirichlet(np.ones(B), (N, N))
    data = rng.poisson(rate, (N, T)).astype(np.int64)
    proc = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W), A,
                                          nhp.BernoulliNetworkModel(0.3, N))
    return proc, data


def random_q(N, B, seed):
    """A network state with every block spread over orders of magnitude and link probabilities on all of (0, 1)."""
    rng = np.random.default_rng(seed)
    u = lambda lo, hi, n: np.exp(rng.uniform(np.log(lo), np.log(hi), n))
    NN = N * N
    return np.concatenate([u(1.0, 100.0, N), u(0.5, 10.0, N), u(0.05, 5.0, NN * B), u(0.1, 20.0, NN), u(0.5, 50.0, NN), u(0.02, 1.0, NN),
                           u(1.0, 50.0, NN), rng.uniform(0.0, 1.0, NN), u(0.5, 20.0, 2)])


def pv_slice(N, B):
    o = 2 * N + N * N * (B + 4)
    return slice(o, o + N * N)


def net_set(ctx, proc, q, N, B):
    hy = D._network_hyper(proc)
    ctx.check(ctx.lib.nhp_disc_vb_network_set(ctx.h, N, B, proc.dt, _ptr(hy), hy.size, _ptr(np.ascontiguousarray(q))))


def vb_get(ctx, n):
    q = np.empty(n)
    ctx.check(ctx.lib.nhp_disc_vb_get(ctx.h, _ptr(q)))
    return q


def vb_step(ctx, d):
    ch = ctypes.c_double()
    ctx.check(ctx.lib.nhp_disc_vb_step(ctx.h, d.h, ctypes.byref(ch)))
    return ch.value


def svi_step(ctx, d, t_begin, n_bins, step):
    ch = ctypes.c_double()
    ctx.check(ctx.lib.nhp_disc_svi_step(ctx.h, d.h, t_begin, n_bins, step, ctypes.byref(ch)))
    return ch.value


def net_change(new, old, N, B):
    """The step's change: relative over the positive entries, absolute over pv."""
    ps = pv_slice(N, B)
    rel = np.abs(new - old) / old
    rel[ps] = np.abs(new[ps] - old[ps])
    return float(np.max(rel))


def compare(q_dev, q_ref, N, B, rtol, atol_pv):
    ps = pv_slice(N, B)
    keep = np.ones(q_dev.size, bool)
    keep[ps] = False
    keep[-2:] = False
    err = float(np.max(np.abs(q_dev[keep] - q_ref[keep]) / np.abs(q_ref[keep])))
    err_pv = float(np.max(np.abs(q_dev[ps] - q_ref[ps])))
    err_rho = float(np.max(np.abs(q_dev[-2:] - q_ref[-2:]) / q_ref[-2:]))
    print(f"rel {err:.3g}, pv abs {err_pv:.3g}, rho rel {err_rho:.3g}")
    assert err <= rtol and err_pv <= atol_pv and err_rho <= atol_pv, (err, err_pv, err_rho)


@pytest.mark.parametrize("N,T,B,L,warp", [(12, 3000, 3, 5, "1"), (12, 3000, 3, 5, "0"), (200, 20000, 6, 12, "1"), (200, 20000, 6, 12, "0")],
                         ids=["small", "small_block_kernel", "config3_shape", "config3_shape_block_kernel"])
def test_one_step_equals_network_update(N, T, B, L, warp, monkeypatch):
    """From a random network state, one nhp_disc_vb_step == discrete.network_update_: the standard blocks, kappa0v and nu0v at rtol
    5e-14, pv at atol 1e-11, q(rho) at rtol 1e-11; the change equals the host's change of the host state to 1e-11."""
    monkeypatch.setenv("NHP_DISC_WARP", warp)
    proc, data = make(N, T, B, L, 7 + N)
    ctx = proc._ctx()
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    q0 = random_q(N, B, 3)
    D.set_network_variational_params_(proc, q0)
    np.testing.assert_array_equal(D.network_variational_params(proc), q0)
    net_set(ctx, proc, q0, N, B)
    change = vb_step(ctx, d)
    q_dev = vb_get(ctx, q0.size)
    q_host = D.network_update_(proc, d)
    compare(q_dev, q_host, N, B, 5e-14, 1e-11)
    print(f"change {change!r} host {net_change(q_host, q0, N, B)!r}")
    assert change == pytest.approx(net_change(q_host, q0, N, B), rel=1e-11, abs=1e-11)
    d.free()


def expected_step(proc, data, L, B, q0, t_begin, n_bins, step):
    N, T = data.shape
    e0, E = D.network_expectations(q0, N, B)
    idx = (t_begin + np.arange(n_bins)) % T
    masked = np.zeros_like(data)
    masked[:, idx] = data[:, idx]
    st = orc.disc_vb_stats(masked, orc.disc_convolve(data, orc.disc_basis(L, B)), e0, E)
    target = D.network_vb_targets(q0, st, masked.sum(axis=1).astype(np.float64), T, proc.dt, D._network_hyper(proc), T / n_bins)
    return (1.0 - step) * q0 + step * target


T_W = 3000
WINDOWS = {"interior": (700, 900), "wrapped": (2500, 1000), "one_bin": None, "full": (0, T_W)}


@pytest.mark.parametrize("warp", ["1", "0"], ids=["warp_kernel", "block_kernel"])
@pytest.mark.parametrize("step", [1.0, 0.3])
@pytest.mark.parametrize("window", list(WINDOWS))
def test_window_against_the_oracle(window, step, warp, monkeypatch):
    """One SVI step on a network state == network_vb_targets of the oracle's statistics of the window (data zeroed outside it, the
    full data's convolution), blended in NumPy: standard blocks rtol 5e-14, pv atol 1e-11; change as the host's.  The full window at
    step 1 also equals the VB step."""
    monkeypatch.setenv("NHP_DISC_WARP", warp)
    N, B, L = 12, 3, 5
    proc, data = make(N, T_W, B, L, 71)
    t_begin, n_bins = WINDOWS[window] or (int(np.flatnonzero(data[:, 400:].sum(axis=0))[0]) + 400, 1)
    ctx = proc._ctx()
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    q0 = random_q(N, B, 5)
    net_set(ctx, proc, q0, N, B)
    ch = svi_step(ctx, d, t_begin, n_bins, step)
    q_dev = vb_get(ctx, q0.size)
    ref = expected_step(proc, data, L, B, q0, t_begin, n_bins, step)
    compare(q_dev, ref, N, B, 5e-14, 1e-11)
    assert ch == pytest.approx(net_change(ref, q0, N, B), rel=1e-11, abs=1e-11)
    if window == "full" and step == 1.0:
        net_set(ctx, proc, q0, N, B)
        vb_step(ctx, d)
        compare(vb_get(ctx, q0.size), q_dev, N, B, 5e-14, 1e-11)
    d.free()


def test_trace_and_the_kind_of_state():
    """VB and SVI steps on a network state share the open trace; a trace begun for one kind refuses a step on the other
    (NHP_ERR_STATE) and leaves the state alone; after nhp_disc_vb_set replaces the network state, a standard step equals update_."""
    N, T, B, L = 10, 2000, 3, 5
    proc, data = make(N, T, B, L, 31)
    ctx = Context()
    proc.ctx = ctx
    lib = ctx.lib
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    q0 = random_q(N, B, 9)
    net_set(ctx, proc, q0, N, B)
    ctx.check(lib.nhp_disc_vb_trace_begin(ctx.h, 5))
    states = []
    for window in [(100, 300, 0.5), "vb", (1900, 400, 0.8), "vb", (5, 1, 0.2)]:
        if window == "vb":
            vb_step(ctx, d)
        else:
            svi_step(ctx, d, *window)
        states.append(vb_get(ctx, q0.size))
    allq = np.empty((5, q0.size))
    ctx.check(lib.nhp_disc_vb_trace_read(ctx.h, 0, 5, _ptr(allq)))
    np.testing.assert_array_equal(allq, np.array(states))
    # a standard state on the network trace
    std = D.DiscreteStandardHawkesProcess(proc.baseline, proc.impulses, proc.weights)
    std.ctx = ctx
    qs = q0[:2 * N + N * N * (B + 2)].copy()
    D.set_variational_params_(std, qs)
    hy = np.array([std.baseline.alpha0, std.baseline.beta0, std.weights.kappa, std.weights.nu, std.impulses.gamma])
    ctx.check(lib.nhp_disc_vb_set(ctx.h, N, B, 1.0, _ptr(hy), 5, _ptr(qs)))
    assert int(lib.nhp_disc_vb_step(ctx.h, d.h, None)) == _lib.NHP_ERR_STATE
    assert int(lib.nhp_disc_svi_step(ctx.h, d.h, 0, 10, 0.5, None)) == _lib.NHP_ERR_STATE
    np.testing.assert_array_equal(vb_get(ctx, qs.size), qs)
    ctx.check(lib.nhp_disc_vb_trace_free(ctx.h))
    vb_step(ctx, d)
    np.testing.assert_allclose(vb_get(ctx, qs.size), D.update_(std, d), rtol=5e-15)
    # a network state on a standard trace
    ctx.check(lib.nhp_disc_vb_trace_begin(ctx.h, 2))
    net_set(ctx, proc, q0, N, B)
    assert int(lib.nhp_disc_vb_step(ctx.h, d.h, None)) == _lib.NHP_ERR_STATE
    np.testing.assert_array_equal(vb_get(ctx, q0.size), q0)
    ctx.check(lib.nhp_disc_vb_trace_free(ctx.h))
    d.free()


def test_refusals_leave_the_state_unchanged():
    """_network_set refuses n_hyper != 9, a pv outside [0, 1] or NaN, a non-positive entry elsewhere and a non-positive hyper-parameter
    (INVALID); a step refuses sharded data (UNSUPPORTED), N or B not those of the data (INVALID) and unconvolved data (STATE).  The
    kept state is as it was after each."""
    N, T, B, L = 8, 1500, 3, 5
    proc, data = make(N, T, B, L, 41)
    ctx = Context()
    proc.ctx = ctx
    lib = ctx.lib
    q0 = random_q(N, B, 11)
    n = q0.size
    net_set(ctx, proc, q0, N, B)
    hy = D._network_hyper(proc)
    ps = pv_slice(N, B)
    bad = []
    for k, v in ((ps.start, 1.5), (ps.start + 3, -0.1), (ps.stop - 1, np.nan), (2 * N + 1, 0.0), (n - 1, -1.0), (ps.start - 1, np.inf)):
        qb = q0.copy()
        qb[k] = v
        bad.append((qb, hy, 9))
    bad += [(q0, hy[:5], 5), (q0, np.append(hy, 1.0), 10), (q0, np.where(np.arange(9) == 6, 0.0, hy), 9)]
    for qb, hb, nh in bad:
        assert int(lib.nhp_disc_vb_network_set(ctx.h, N, B, 1.0, _ptr(np.ascontiguousarray(hb)), nh, _ptr(qb))) == _lib.NHP_ERR_INVALID
    np.testing.assert_array_equal(vb_get(ctx, n), q0)
    d = proc.upload(data)
    step = lambda h: int(lib.nhp_disc_vb_step(ctx.h, h, None))
    assert step(d.h) == _lib.NHP_ERR_STATE  # not convolved
    D.convolve(proc, d, export=False)
    sh = D.DiscreteData(ctx, data[:, 100:], t_halo=L)
    D.convolve(proc, sh, export=False)
    assert step(sh.h) == _lib.NHP_ERR_UNSUPPORTED
    other, odata = make(N + 1, T, B, L, 42)
    other.ctx = ctx
    od = D.DiscreteData(ctx, odata)
    D.convolve(other, od, export=False)
    assert step(od.h) == _lib.NHP_ERR_INVALID
    wide, _ = make(N, T, B + 1, L, 43)
    wide.ctx = ctx
    wd = D.DiscreteData(ctx, data)
    D.convolve(wide, wd, export=False)
    assert step(wd.h) == _lib.NHP_ERR_INVALID
    np.testing.assert_array_equal(vb_get(ctx, n), q0)
    assert step(d.h) == _lib.NHP_OK
    for h in (sh, od, wd, d):
        h.free()


def test_saturated_links():
    """A state with pv exactly 0 and 1 on some links steps without NaN; pv stays in [0, 1] and the change is finite."""
    N, T, B, L = 10, 3000, 3, 5
    proc, data = make(N, T, B, L, 51)
    ctx = proc._ctx()
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    q0 = random_q(N, B, 13)
    ps = pv_slice(N, B)
    q0[ps.start:ps.start + 30] = 0.0
    q0[ps.start + 30:ps.start + 60] = 1.0
    net_set(ctx, proc, q0, N, B)
    for s in range(3):
        ch = vb_step(ctx, d) if s != 1 else svi_step(ctx, d, 100, 500, 0.5)
        q = vb_get(ctx, q0.size)
        assert np.isfinite(ch) and np.all(np.isfinite(q)), s
        assert np.all((q[ps] >= 0.0) & (q[ps] <= 1.0))
    D.set_network_variational_params_(proc, q0)
    q_host = D.network_update_(proc, d)
    net_set(ctx, proc, q0, N, B)
    vb_step(ctx, d)
    compare(vb_get(ctx, q0.size), q_host, N, B, 5e-14, 1e-11)
    d.free()


def recovery_process(seed=0):
    """N = 10, rho = 0.3, on-link weights of a spectral radius of 0.7, lambda0 in [0.02, 0.05]."""
    N, B, L = 10, 3, 5
    rng = np.random.default_rng(seed)
    lam0 = rng.uniform(0.02, 0.05, N)
    A = (rng.random((N, N)) < 0.3).astype(np.float64)
    W = rng.uniform(0.5, 1.0, (N, N)) * A
    W *= 0.7 / np.max(np.abs(np.linalg.eigvals(W)))
    th = rng.dirichlet(np.full(B, 2.0), (N, N))
    proc = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(th, L), nhp.DenseWeightModel(W), A,
                                          nhp.BernoulliNetworkModel(0.3, N))
    return proc, A


def test_recovery_of_the_adjacency_matrix():
    """A rand_device sample of recovery_process (T = 1e5, seed 3), 100 steps of network_vb_device_.  From pv = 1 (every link on at the
    start), pv > 0.5 matches at least 95 of the 100 entries of the true A.  From the default start pv = rho = 0.3 mean-field VB
    falls into the optimum with every link off: the first E[ln W] is mostly the spike's, so the first responsibilities give the links
    almost no events; it matches only the absent links and ends at a lower bound than the start from pv = 1.  The bound of both device
    traces, evaluated on the host, does not decrease (1e-9 relative)."""
    T, S = 100000, 100
    ref, A = recovery_process()
    d = D.rand_device(ref, T, seed=3)
    data = d.download()
    N, B, L = 10, 3, 5
    conv = orc.disc_convolve(data, orc.disc_basis(L, B))
    out = {}
    for name, pv0 in (("default", None), ("all_links", 1.0)):
        proc, _ = recovery_process()
        proc.ctx = ref.ctx
        if pv0 is not None:
            proc.network.pv = np.full((N, N), pv0)
        q0 = D.network_variational_params(proc)
        tr = D.network_vb_device_(proc, d, max_steps=S)
        assert len(tr) == S
        np.testing.assert_array_equal(D.network_variational_params(proc), tr[-1])
        hy = D._network_hyper(proc)
        Ls = [bound(q, data, conv, N, B, 1.0, hy) for q in [q0] + tr]
        falls = [(Ls[k] - Ls[k + 1]) / abs(Ls[k]) for k in range(S)]
        found = int(np.sum((proc.network.pv > 0.5) == (A > 0.5)))
        out[name] = (found, Ls[-1], max(falls))
        print(name, out[name], int(A.sum()))
        assert max(falls) <= 1e-9, (name, max(falls))
    assert out["all_links"][0] >= 95, out
    assert out["default"][0] >= int(N * N - A.sum()) - 5, out
    assert out["all_links"][1] > out["default"][1], out
    d.free()
