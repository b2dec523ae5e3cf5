"""Discrete mean-field VB on the device (nhp_disc_vb_set / _get / _step, nhp_disc_vb_trace_*, discrete.vb_device_).

One step is `update!` (discrete.jl:369-375): the exp-expectations from the state q = variational_params (digamma on the device), the
statistics of nhp_disc_vb_stats, then q in place.  Given the same statistics the update is the same IEEE arithmetic as discrete.update_,
so device and host differ only where the device digamma / log / exp differ from SciPy / NumPy.

Tolerances are the figures measured on a B200 (1000 W power limit), rounded up.  Where the statistics kernels take part they are
rounded up generously: the kernels' floating-point atomics sum in an order that changes from run to run, and so do the last bits."""
import ctypes
import copy

import mpmath
import numpy as np
import pytest
from scipy.special import digamma

import nhp_b200 as nhp
import oracle_ffi as orc
from nhp_b200 import _lib
from nhp_b200 import discrete as D
from nhp_b200.core import Context, _ptr

pytestmark = pytest.mark.gpu

ROOT_X = 1.4616321449683622  # the positive root of digamma


def psi_dev(ctx, x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    ctx.check(ctx.lib.nhp_test_fastmath(ctx.h, 2, _ptr(x), x.size, _ptr(out)))
    return out


def test_digamma_against_mpmath(ctx):
    """nhp_digamma (which = 2) against mpmath at 50 digits on 3000 points: error <= 1.3e-15 * max(1, |psi|) (measured 1.29e-15, at
    x = 1.4619 next to the root, where the recurrence cancels; SciPy's own error on these points is 2.5e-16)."""
    rng = np.random.default_rng(0)
    x = np.concatenate([10.0 ** rng.uniform(-6, 12, 2000), rng.uniform(1, 3, 500), ROOT_X + rng.uniform(-1e-3, 1e-3, 500)])
    got = psi_dev(ctx, x)
    with mpmath.workdps(50):
        ref = np.array([float(mpmath.digamma(mpmath.mpf(float(v)))) for v in x])
    err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
    assert err.max() <= 1.3e-15, (err.max(), x[err.argmax()])


def test_digamma_against_scipy(ctx):
    """3e5 points (log-spaced 1e-6 ... 1e12, [1, 3], around the root) against scipy.special.digamma: error <= 1.7e-15 * max(1, |psi|)
    (measured 1.67e-15); NaN for x <= 0 and NaN, +inf at +inf."""
    rng = np.random.default_rng(1)
    x = np.concatenate([np.logspace(-6, 12, 200000), rng.uniform(1, 3, 50000), ROOT_X + rng.uniform(-0.05, 0.05, 50000)])
    got, ref = psi_dev(ctx, x), digamma(x)
    err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
    assert err.max() <= 1.7e-15, (err.max(), x[err.argmax()])
    edge = psi_dev(ctx, np.array([0.0, -1.0, -1e300, np.nan, np.inf]))
    assert np.all(np.isnan(edge[:4])) and edge[4] == np.inf


def make(N, T, B, L, seed, rate=0.1):
    rng = np.random.default_rng(seed)
    lam0 = rng.uniform(0.5, 1.5, N) * rate
    W = rng.uniform(0.1, 1.0, (N, N)) * 0.5 / N
    theta = rng.dirichlet(np.ones(B), (N, N))
    data = rng.poisson(rate, (N, T)).astype(np.int64)
    proc = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W))
    return proc, data


def random_q(N, B, seed):
    """A non-trivial state: every block spread over orders of magnitude, small gammav values exercise the digamma recurrence."""
    rng = np.random.default_rng(seed)
    u = lambda lo, hi, n: np.exp(rng.uniform(np.log(lo), np.log(hi), n))
    return np.concatenate([u(1.0, 100.0, N), u(0.5, 10.0, N), u(0.05, 5.0, N * N * B), u(0.1, 20.0, N * N), u(0.5, 50.0, N * N)])


def hyper(proc):
    b, w, imp = proc.baseline, proc.weights, proc.impulses
    return np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)


def vb_set(ctx, proc, q, N, B):
    hy = hyper(proc)
    ctx.check(ctx.lib.nhp_disc_vb_set(ctx.h, N, B, proc.dt, _ptr(hy), 5, _ptr(np.ascontiguousarray(q))))


def vb_get(ctx, n):
    q = np.empty(n)
    ctx.check(ctx.lib.nhp_disc_vb_get(ctx.h, _ptr(q)))
    return q


def vb_step(ctx, d):
    ch = ctypes.c_double()
    ctx.check(ctx.lib.nhp_disc_vb_step(ctx.h, d.h, ctypes.byref(ch)))
    return ch.value


def rel_change(new, old):
    return np.max(np.abs(new - old) / old)


@pytest.mark.parametrize("N,T,B,L,warp", [(12, 3000, 3, 5, "1"), (12, 3000, 3, 5, "0"), (200, 20000, 6, 12, "1"), (200, 20000, 6, 12, "0")],
                         ids=["small", "small_block_kernel", "config3_shape", "config3_shape_block_kernel"])
def test_one_step_equals_update(N, T, B, L, warp, monkeypatch):
    """From a random state, one nhp_disc_vb_step == one discrete.update_ at rtol 5e-15 (measured 1.8e-15 to 2.2e-15), for both
    statistics kernels; its change is the host's max relative change (measured: equal)."""
    monkeypatch.setenv("NHP_DISC_WARP", warp)
    proc, data = make(N, T, B, L, 7 + N)
    ctx = proc._ctx()
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    q0 = random_q(N, B, 3)
    D.set_variational_params_(proc, q0)
    np.testing.assert_array_equal(proc.variational_params(), q0)
    vb_set(ctx, proc, q0, N, B)
    change = vb_step(ctx, d)
    q_dev = vb_get(ctx, q0.size)
    q_host = D.update_(proc, d)
    np.testing.assert_allclose(q_dev, q_host, rtol=5e-15)
    assert change == pytest.approx(rel_change(q_host, q0), rel=1e-14)
    d.free()


def test_one_step_equals_the_stats_reference():
    """The step == the reference statistics (orc.disc_vb_stats) fed with SciPy's e0 / E, plus the update formulas, at rtol 1e-14
    (measured 1.7e-15)."""
    N, T, B, L = 16, 4000, 4, 6
    proc, data = make(N, T, B, L, 17)
    ctx = proc._ctx()
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    q0 = random_q(N, B, 5)
    vb_set(ctx, proc, q0, N, B)
    vb_step(ctx, d)
    q_dev = vb_get(ctx, q0.size)
    NN, o = N * N, 2 * N + N * N * B
    av, bv = q0[:N], q0[N:2 * N]
    gv = q0[2 * N:o].reshape(B, N, N).transpose(2, 1, 0)
    kv, nv = q0[o:o + NN].reshape(N, N).T, q0[o + NN:].reshape(N, N).T
    e0 = np.exp(digamma(av) - np.log(bv))
    E = np.exp((digamma(gv) - digamma(gv.sum(axis=2, keepdims=True))) + (digamma(kv) - np.log(nv))[:, :, None])
    st = orc.disc_vb_stats(data, orc.disc_convolve(data, orc.disc_basis(L, B)), e0, E)
    hy = hyper(proc)
    ref = np.concatenate([hy[0] + st["alpha_sum"], 1.0 / hy[1] + T * proc.dt * np.ones(N), (hy[4] + st["gamma_sum"]).transpose(2, 1, 0).ravel(),
                          (hy[2] + st["kappa_sum"]).T.ravel(), (hy[3] + st["nu_sum"]).T.ravel()])
    np.testing.assert_allclose(q_dev, ref, rtol=1e-14)
    d.free()


def test_chain_equals_host_chain_and_rtol_stops_at_the_same_step():
    """30 device steps == 30 steps of vb_ (every trace entry at rtol 2e-14; measured 8.0e-15 and 1.1e-14 in two runs); each step's
    change == the host's max relative change of consecutive vectors (rtol 2e-14; measured 8.8e-15 and 9.8e-15); with rtol,
    vb_device_ stops at the step a host loop with the same rule stops at."""
    N, T, B, L, S = 20, 5000, 4, 8, 30
    dev, data = make(N, T, B, L, 23, rate=0.15)
    host = copy.deepcopy(dev)
    d = dev.upload(data)
    tr_dev = D.vb_device_(dev, d, max_steps=S)
    tr_host = D.vb_(host, d, max_steps=S)
    assert len(tr_dev) == len(tr_host) == S
    for k in range(S):
        np.testing.assert_allclose(tr_dev[k], tr_host[k], rtol=2e-14, err_msg=f"step {k}")
    np.testing.assert_array_equal(dev.variational_params(), tr_dev[-1])
    # the change of every step, from the default (all-ones) state
    ctx = dev._ctx()
    fresh, _ = make(N, T, B, L, 23, rate=0.15)
    fresh.weights.kappav, fresh.weights.nuv = np.ones((N, N)), np.ones((N, N))
    q0 = fresh.variational_params()
    vb_set(ctx, fresh, q0, N, B)
    ch_dev = np.array([vb_step(ctx, d) for _ in range(S)])
    ch_host = np.array([rel_change(tr_host[k], tr_host[k - 1] if k else q0) for k in range(S)])
    np.testing.assert_allclose(ch_dev, ch_host, rtol=2e-14)
    # rtol: the first step whose change is <= rtol ends the loop; pick a threshold just above one step's change and well below
    # every earlier step's
    j = next(k for k in range(3, S) if ch_host[k] * 1.01 < ch_host[:k].min() and ch_host[k] > 1e-8)
    r = ch_host[j] * 1.001
    early, _ = make(N, T, B, L, 23, rate=0.15)
    tr_r = D.vb_device_(early, d, max_steps=S, rtol=r)
    assert len(tr_r) == j + 1
    np.testing.assert_allclose(tr_r[-1], tr_host[j], rtol=2e-14)
    d.free()


def test_trace_contract():
    """_read equals _get after every step; a full trace stops taking slots while the steps go on; reads outside the stored slots are
    NHP_ERR_INVALID; the trace needs a state."""
    N, T, B, L = 10, 2000, 3, 5
    proc, data = make(N, T, B, L, 31)
    ctx = Context()
    proc.ctx = ctx
    lib = ctx.lib
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    assert int(lib.nhp_disc_vb_trace_begin(ctx.h, 3)) == _lib.NHP_ERR_STATE
    q0 = random_q(N, B, 9)
    n = q0.size
    vb_set(ctx, proc, q0, N, B)
    ctx.check(lib.nhp_disc_vb_trace_begin(ctx.h, 3))
    states = []
    for s in range(5):
        vb_step(ctx, d)
        states.append(vb_get(ctx, n))
        cnt, cap = ctypes.c_int64(), ctypes.c_int64()
        ctx.check(lib.nhp_disc_vb_trace_count(ctx.h, ctypes.byref(cnt), ctypes.byref(cap)))
        assert (cnt.value, cap.value) == (min(s + 1, 3), 3)
        if s < 3:
            slot = np.empty(n)
            ctx.check(lib.nhp_disc_vb_trace_read(ctx.h, s, 1, _ptr(slot)))
            np.testing.assert_array_equal(slot, states[-1])
    assert not np.array_equal(states[3], states[2])  # the steps went on
    allq = np.empty((3, n))
    ctx.check(lib.nhp_disc_vb_trace_read(ctx.h, 0, 3, _ptr(allq)))
    np.testing.assert_array_equal(allq, np.array(states[:3]))
    buf = np.empty(4 * n)
    assert int(lib.nhp_disc_vb_trace_read(ctx.h, 2, 2, _ptr(buf))) == _lib.NHP_ERR_INVALID
    assert int(lib.nhp_disc_vb_trace_read(ctx.h, -1, 1, _ptr(buf))) == _lib.NHP_ERR_INVALID
    assert int(lib.nhp_disc_vb_trace_read(ctx.h, 0, -1, _ptr(buf))) == _lib.NHP_ERR_INVALID
    ctx.check(lib.nhp_disc_vb_trace_free(ctx.h))
    assert int(lib.nhp_disc_vb_trace_read(ctx.h, 0, 1, _ptr(buf))) == _lib.NHP_ERR_INVALID
    d.free()


def test_refusals_leave_the_state_unchanged():
    """Each refusal returns before anything changes: a step with no state or on unconvolved data (STATE), on time-sharded data
    (UNSUPPORTED), with N or B not those of the data (INVALID), with an open trace begun for another B (STATE); _set refuses a
    non-positive or non-finite entry, hyper-parameter or dt (INVALID).  VB steps leave the discrete parameters, the Gibbs trace and
    nhp_disc_vb_stats untouched."""
    N, T, B, L = 8, 1500, 3, 5
    proc, data = make(N, T, B, L, 41)
    ctx = Context()
    proc.ctx = ctx
    lib = ctx.lib
    d = proc.upload(data)
    step = lambda h: int(lib.nhp_disc_vb_step(ctx.h, h, None))
    assert step(d.h) == _lib.NHP_ERR_STATE  # no state
    q0 = random_q(N, B, 11)
    n = q0.size
    vb_set(ctx, proc, q0, N, B)
    assert step(d.h) == _lib.NHP_ERR_STATE  # not convolved
    D.convolve(proc, d, export=False)
    sh = D.DiscreteData(ctx, data[:, 100:], t_halo=L)
    D.convolve(proc, sh, export=False)
    assert step(sh.h) == _lib.NHP_ERR_UNSUPPORTED
    other, odata = make(N + 1, T, B, L, 42)
    other.ctx = ctx
    od = D.DiscreteData(ctx, odata)
    D.convolve(other, od, export=False)
    assert step(od.h) == _lib.NHP_ERR_INVALID  # N
    wide, _ = make(N, T, B + 1, L, 43)
    wide.ctx = ctx
    wd = D.DiscreteData(ctx, data)
    D.convolve(wide, wd, export=False)
    assert step(wd.h) == _lib.NHP_ERR_INVALID  # B
    np.testing.assert_array_equal(vb_get(ctx, n), q0)
    # _set: bad entries leave the kept state alone
    hy = hyper(proc)
    for bad_q, bad_h, dt in ((np.where(np.arange(n) == 5, 0.0, q0), hy, 1.0), (np.where(np.arange(n) == n - 1, np.nan, q0), hy, 1.0),
                             (q0, np.array([1.0, 1.0, -1.0, 1.0, 1.0]), 1.0), (q0, np.array([1.0, np.inf, 1.0, 1.0, 1.0]), 1.0), (q0, hy, 0.0)):
        assert int(lib.nhp_disc_vb_set(ctx.h, N, B, dt, _ptr(bad_h), 5, _ptr(bad_q))) == _lib.NHP_ERR_INVALID
    assert int(lib.nhp_disc_vb_set(ctx.h, N, B, 1.0, _ptr(hy), 4, _ptr(q0))) == _lib.NHP_ERR_INVALID
    np.testing.assert_array_equal(vb_get(ctx, n), q0)
    # an open trace of the (N, B) state, then a state of another B on data of that B
    ctx.check(lib.nhp_disc_vb_trace_begin(ctx.h, 4))
    qw = random_q(N, B + 1, 12)
    vb_set(ctx, wide, qw, N, B + 1)
    assert step(wd.h) == _lib.NHP_ERR_STATE
    np.testing.assert_array_equal(vb_get(ctx, qw.size), qw)
    ctx.check(lib.nhp_disc_vb_trace_free(ctx.h))
    ctx.check(lib.nhp_disc_vb_step(ctx.h, wd.h, None))  # closed: the step runs
    # the discrete parameters, the Gibbs trace and the statistics are the model's, not the VB state's
    proc._push(ctx)
    ctx.check(lib.nhp_disc_trace_begin(ctx.h, 2))
    ctx.check(lib.nhp_disc_trace_push(ctx.h))
    rng = np.random.default_rng(5)
    e0, E = rng.uniform(0.5, 1.5, N), rng.uniform(0.01, 0.2, (N, N, B))
    st0 = D.vb_statistics(proc, d, e0, E)
    P0 = [np.empty(N), np.empty(N * N), np.empty(N * N * B)]
    ctx.check(lib.nhp_disc_params_get(ctx.h, _ptr(P0[0]), _ptr(P0[1]), None, _ptr(P0[2])))
    vb_set(ctx, proc, q0, N, B)
    for _ in range(3):
        vb_step(ctx, d)
    P1 = [np.empty_like(x) for x in P0]
    ctx.check(lib.nhp_disc_params_get(ctx.h, _ptr(P1[0]), _ptr(P1[1]), None, _ptr(P1[2])))
    for a, b in zip(P0, P1):
        np.testing.assert_array_equal(a, b)
    cnt = ctypes.c_int64()
    ctx.check(lib.nhp_disc_trace_count(ctx.h, ctypes.byref(cnt), None))
    assert cnt.value == 1
    lam = np.empty(N)
    ctx.check(lib.nhp_disc_trace_read(ctx.h, 0, 1, None, _ptr(lam), None, None, None))
    np.testing.assert_array_equal(lam, P0[0])
    st1 = D.vb_statistics(proc, d, e0, E)
    for k in st0:
        np.testing.assert_allclose(st1[k], st0[k], rtol=1e-14)
    ctx.check(lib.nhp_disc_trace_free(ctx.h))
    for h in (sh, od, wd, d):
        h.free()


def test_data_without_events():
    """No non-zero bins: the statistics are zero, so the step leaves alphav = alpha0, gammav = gamma, kappav = kappa, nuv = nu and
    betav = 1/beta0 + T dt, equal to update_."""
    N, T, B, L = 6, 500, 3, 4
    proc, _ = make(N, T, B, L, 51)
    data = np.zeros((N, T), dtype=np.int64)
    ctx = proc._ctx()
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    q0 = random_q(N, B, 13)
    D.set_variational_params_(proc, q0)
    vb_set(ctx, proc, q0, N, B)
    vb_step(ctx, d)
    q_dev = vb_get(ctx, q0.size)
    np.testing.assert_array_equal(q_dev, D.update_(proc, d))
    hy = hyper(proc)
    NN, o = N * N, 2 * N + N * N * B
    np.testing.assert_array_equal(q_dev[:N], hy[0])
    np.testing.assert_array_equal(q_dev[2 * N:o], hy[4])
    np.testing.assert_array_equal(q_dev[o:o + NN], hy[2])
    np.testing.assert_array_equal(q_dev[o + NN:], hy[3])
    d.free()


def test_network_process_is_refused():
    """The reference's update! of a network process is non-functional (quirk Q10): vb_device_ raises, as vb_ cannot run one."""
    N, B, L = 4, 2, 3
    rng = np.random.default_rng(61)
    proc = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(np.full(N, 0.1)), D.DiscreteGaussianImpulseResponse(rng.dirichlet(np.ones(B), (N, N)), L),
                                          nhp.DenseWeightModel(np.full((N, N), 0.1)), np.ones((N, N)), nhp.BernoulliNetworkModel(0.5, N))
    with pytest.raises(ValueError):
        D.vb_device_(proc, rng.poisson(0.1, (N, 200)).astype(np.int64))
