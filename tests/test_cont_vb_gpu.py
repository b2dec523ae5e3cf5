"""Continuous mean-field VB on the device (nhp_cont_vb_set / _get / _stats / _step, nhp_cont_vb_trace_*, continuous.vb_device_),
against the NumPy twin of tests/cont_vb_reference.py.

The twin evaluates every event's window on its own (brute force) at the effective parameters of the state; the device runs the
intensity sweep and the gradient's child-major scatter with shared-memory or global floating-point atomics, so its sums come in an
order that changes from run to run.  Tolerances are the figures measured on an NVIDIA B200 (1000 W power limit), rounded up."""
import ctypes

import numpy as np
import pytest

import cont_vb_reference as R
import nhp_b200 as nhp
from nhp_b200 import _lib
from nhp_b200 import continuous as C
from nhp_b200.core import Context, ContinuousData, _fmat, _ptr

pytestmark = pytest.mark.gpu

EXP, LN = R.EXP, R.LN
HYPER = {EXP: [1.5, 0.5, 2.0, 3.0, 2.0, 1.0], LN: [1.5, 0.5, 2.0, 3.0, 0.2, 1.5, 2.0, 0.7]}


def stream(counts, T, seed, ties=0):
    """Times uniform on [0, T), sorted, with exactly counts[k] events on node k (0-based) and `ties` events sharing one time."""
    rng = np.random.default_rng(seed)
    c = rng.permutation(np.repeat(np.arange(len(counts)), counts))
    t = np.sort(rng.uniform(0.0, T, c.size))
    if ties:
        k = c.size // 2
        t[k:k + ties] = t[k]
    return t, c


def random_state(K, kind, seed, wscale=1.0):
    rng = np.random.default_rng(seed)
    mats = [rng.uniform(0.5, 3.0, (K, K)), rng.uniform(3.0, 30.0, (K, K)) * wscale]
    if kind == EXP:
        mats += [rng.uniform(2.0, 10.0, (K, K)), rng.uniform(0.5, 3.0, (K, K))]
    else:
        mats += [rng.normal(0.0, 1.0, (K, K)), rng.uniform(0.5, 5.0, (K, K)), rng.uniform(1.0, 6.0, (K, K)), rng.uniform(0.5, 3.0, (K, K))]
    return R.pack(rng.uniform(2.0, 10.0, K), rng.uniform(1.0, 5.0, K), mats)


def push(ctx, kind, K, dtmax, lam0=None, W=None, p1=None, p2=None, A=None):
    lam0 = np.ones(K) if lam0 is None else lam0
    W = np.full((K, K), 0.05) if W is None else W
    p1 = (np.ones((K, K)) if kind == EXP else np.zeros((K, K))) if p1 is None else p1
    p2 = (None if kind == EXP else np.ones((K, K))) if p2 is None else p2
    ctx.check(ctx.lib.nhp_cont_params_set(ctx.h, kind, K, _ptr(np.ascontiguousarray(lam0, dtype=np.float64)), _ptr(_fmat(W)),
                                          None if A is None else _ptr(_fmat(A)), _ptr(_fmat(p1)), None if p2 is None else _ptr(_fmat(p2)), float(dtmax)))


def vb_set(ctx, kind, q):
    hy = np.asarray(HYPER[kind], dtype=np.float64)
    ctx.check(ctx.lib.nhp_cont_vb_set(ctx.h, _ptr(hy), hy.size, _ptr(np.ascontiguousarray(q, dtype=np.float64))))


def vb_get(ctx, kind, K):
    q = np.empty(2 * K + R.nplanes(kind) * K * K)
    ctx.check(ctx.lib.nhp_cont_vb_get(ctx.h, _ptr(q)))
    return q


def dev_stats(ctx, d, K):
    M0, Mnm, S1, S2 = np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
    ctx.check(ctx.lib.nhp_cont_vb_stats(ctx.h, d.h, _ptr(M0), _ptr(Mnm), _ptr(S1), _ptr(S2)))
    f = lambda v: v.reshape(K, K).T
    return dict(M0=M0, Mnm=f(Mnm), S1=f(S1), S2=f(S2))


def step(ctx, d):
    ch = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_vb_step(ctx.h, d.h, ctypes.byref(ch)))
    return ch.value


def params_get(ctx, kind, K):
    lam, W, p1 = np.empty(K), np.empty(K * K), np.empty(K * K)
    p2 = np.empty(K * K) if kind == LN else None
    ctx.check(ctx.lib.nhp_cont_params_get(ctx.h, _ptr(lam), _ptr(W), None, _ptr(p1), _ptr(p2)))
    f = lambda v: None if v is None else v.reshape(K, K).T.copy()
    return lam, f(W), f(p1), f(p2)


def nerr(a, b):
    """Normwise relative error of an array: max |a - b| / max |b|."""
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


class Owned:
    """The contexts and events handles one test makes."""

    def __init__(self):
        self.ctxs, self.data = [], []

    def context(self):
        self.ctxs.append(Context(0))
        return self.ctxs[-1]

    def upload(self, ctx, *args, **kw):
        self.data.append(ContinuousData(ctx, *args, **kw))
        return self.data[-1]


@pytest.fixture
def own():
    """Frees a test's events handles, then its contexts, when it ends.  Left to the collector, a reference cycle (a caught exception's
    traceback holds the test's frame) could finalize a context before its handles, whose release then runs on a destroyed stream."""
    o = Owned()
    yield o
    for d in o.data:
        d.free()
    for c in o.ctxs:
        c._fin()


def setup(own, kind, K, dtmax, counts, T, seed, ties=0, wscale=1.0):
    ctx = own.context()
    t, c = stream(counts, T, seed, ties)
    d = own.upload(ctx, t, c + 1, T, K)
    q = random_state(K, kind, seed + 100, wscale)
    push(ctx, kind, K, dtmax)
    vb_set(ctx, kind, q)
    return ctx, d, t, c, q


STATS_CASES = [
    # kind, dtmax, K, events per node, duration, tied events
    (EXP, np.inf, 1, [1], 1.0, 0),          # a single event
    (LN, 1.0, 1, [1], 1.0, 0),
    (EXP, np.inf, 1, [700], 100.0, 5),
    (EXP, 2.0, 3, [255, 256, 257], 60.0, 4),  # the 256-event work items of the child-major sweep
    (EXP, np.inf, 3, [255, 256, 257], 60.0, 4),
    (LN, 1.0, 3, [255, 256, 257], 60.0, 4),
    (EXP, 0.5, 17, [120] * 17, 150.0, 3),
    (LN, 1.5, 17, [120] * 17, 150.0, 3),
    (EXP, np.inf, 64, [40] * 64, 100.0, 6),
    (LN, 1.0, 64, [40] * 64, 100.0, 6),
]


@pytest.mark.parametrize("kind,dtmax,K,counts,T,ties", STATS_CASES)
def test_stats_match_twin(own, kind, dtmax, K, counts, T, ties):
    """nhp_cont_vb_stats against the brute-force twin: M0 entrywise, Mnm / S1 / S2 normwise, relative error <= 1e-12 (measured at most
    4.1e-14), and q unchanged by the call."""
    ctx, d, t, c, q = setup(own, kind, K, dtmax, counts, T, 7 * K + kind)
    dev = dev_stats(ctx, d, K)
    ref = R.expected_stats(t, c, K, kind, q, dtmax)
    errs = [nerr(dev[k], ref[k]) for k in ("M0", "Mnm", "S1") + (("S2",) if kind == LN else ())]
    print("stats error", kind, K, dtmax, max(errs))
    assert np.all(np.abs(dev["M0"] - ref["M0"]) <= 1e-12 * ref["M0"])
    for k in ("Mnm", "S1") + (("S2",) if kind == LN else ()):
        assert nerr(dev[k], ref[k]) <= 1e-12, (k, nerr(dev[k], ref[k]))
    if kind == EXP:
        assert not np.any(dev["S2"])
    assert np.array_equal(vb_get(ctx, kind, K), q)


def test_stats_match_twin_global_accumulators(own):
    """K = 5000 Exponential: the columns' accumulators no longer fit in shared memory, so the scatter adds into the K^2 planes with
    global atomics.  Same tolerance as above (measured at most 8.3e-16)."""
    K = 5000
    rng = np.random.default_rng(3)
    counts = np.bincount(rng.integers(0, K, 3000), minlength=K)
    ctx, d, t, c, q = setup(own, EXP, K, np.inf, counts, 30.0, 11, ties=3, wscale=50.0)
    dev = dev_stats(ctx, d, K)
    ref = R.expected_stats(t, c, K, EXP, q, np.inf)
    print("stats error K=5000", nerr(dev["M0"], ref["M0"]), nerr(dev["Mnm"], ref["Mnm"]), nerr(dev["S1"], ref["S1"]))
    assert np.all(np.abs(dev["M0"] - ref["M0"]) <= 1e-12 * ref["M0"])
    assert nerr(dev["Mnm"], ref["Mnm"]) <= 1e-12 and nerr(dev["S1"], ref["S1"]) <= 1e-12


@pytest.mark.parametrize("kind,dtmax", [(EXP, np.inf), (LN, 1.0)])
def test_rao_blackwell(own, kind, dtmax):
    """The expected statistics are the mean of the sampled ones: with the effective parameters pushed (nhp_cont_params_set), R parent
    sweeps give counts whose mean lies within 5 sigma of nhp_cont_vb_stats, sigma^2 = sum u (1 - u) / R (an upper bound of the variance
    of one sweep's count)."""
    K, Rs = 4, 400
    ctx, d, t, c, q = setup(own, kind, K, dtmax, [500] * K, 200.0, 21 + kind)
    dev = dev_stats(ctx, d, K)
    ref = R.expected_stats(t, c, K, kind, q, dtmax)
    lam0, W, p1, p2 = R.effective_params(q, K, kind)
    push(ctx, kind, K, dtmax, lam0, W, p1, p2)
    sM0, sMnm = np.zeros(K), np.zeros((K, K))
    M0, Mnm = np.empty(K), np.empty(K * K)
    for r in range(Rs):
        ctx.check(ctx.lib.nhp_cont_resample_parents(ctx.h, d.h, 5, r, None, None, None))
        ctx.check(ctx.lib.nhp_cont_suffstats(ctx.h, d.h, _ptr(M0), None, _ptr(Mnm), None, None))
        sM0 += M0
        sMnm += Mnm.reshape(K, K).T
    vM0, vMnm = np.zeros(K), np.zeros((K, K))
    for i, (u0, js, u) in enumerate(ref["resp"]):
        vM0[c[i]] += u0 * (1 - u0)
        np.add.at(vMnm, (c[js], c[i]), u * (1 - u))
    for mean, exp_, var in ((sM0 / Rs, dev["M0"], vM0), (sMnm / Rs, dev["Mnm"], vMnm)):
        sig = np.sqrt(var / Rs)
        assert np.all(np.abs(mean - exp_) <= 5 * sig + 1e-9 * np.abs(exp_)), np.max(np.abs(mean - exp_) / np.maximum(sig, 1e-300))


@pytest.mark.parametrize("kind,dtmax", [(EXP, np.inf), (EXP, 3.0), (LN, 1.0)])
def test_steps_match_twin(own, kind, dtmax):
    """One step, then 10 chained steps, against the twin's update from the same state: positive entries relative, mv absolute,
    <= 1e-12 after one step and <= 1e-11 after ten (measured 1.2e-14 and 8.6e-14); `change` as the twin's to 1e-12
    (measured 8.2e-14)."""
    K = 4
    ctx, d, t, c, q = setup(own, kind, K, dtmax, [400, 300, 350, 450], 150.0, 31 + kind, ties=3)
    nq = q.size
    mvsl = slice(2 * K + 2 * K * K, 2 * K + 3 * K * K) if kind == LN else slice(0, 0)
    pos = np.ones(nq, bool)
    pos[mvsl] = False

    def err(a, b):
        return max(float(np.max(np.abs(a[pos] - b[pos]) / b[pos])), float(np.max(np.abs(a[mvsl] - b[mvsl]), initial=0.0)))

    qt = q
    for k in range(10):
        ch = step(ctx, d)
        qt, cht, _ = R.vb_step(t, c, K, kind, qt, HYPER[kind], 150.0, dtmax)
        qd = vb_get(ctx, kind, K)
        assert err(qd, qt) <= (1e-12 if k == 0 else 1e-11), (k, err(qd, qt))
        assert abs(ch - cht) <= 1e-12 * max(cht, 1e-3), (k, ch, cht)


@pytest.mark.parametrize("kind,dtmax", [(EXP, np.inf), (LN, 1.0)])
def test_context_holds_posterior_means(own, kind, dtmax):
    """After a step the parameters are the posterior means of the new state, bit for bit, and the log-likelihood of the context is the
    one of those means pushed from the host."""
    K = 3
    ctx, d, t, c, q = setup(own, kind, K, dtmax, [300, 200, 250], 100.0, 41 + kind)
    step(ctx, d)
    qn = vb_get(ctx, kind, K)
    got = params_get(ctx, kind, K)
    want = R.posterior_means(qn, K, kind)
    for a, b in zip(got, want):
        assert (a is None and b is None) or np.array_equal(a, b)
    ll1, ll2 = ctypes.c_double(), ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll1)))
    push(ctx, kind, K, dtmax, *want)
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll2)))
    assert abs(ll1.value - ll2.value) <= 1e-13 * abs(ll2.value)


def test_trace(own):
    """The trace keeps the state of every step while it has room: count, capacity, and every slot equal to nhp_cont_vb_get after the
    step that pushed it; a step after it is full still runs and pushes nothing."""
    K, kind = 3, LN
    ctx, d, t, c, q = setup(own, kind, K, 1.0, [200, 200, 200], 80.0, 51)
    ctx.check(ctx.lib.nhp_cont_vb_trace_begin(ctx.h, 3))
    seen = []
    cnt, cap = ctypes.c_int64(), ctypes.c_int64()
    for k in range(5):
        step(ctx, d)
        seen.append(vb_get(ctx, kind, K))
        ctx.check(ctx.lib.nhp_cont_vb_trace_count(ctx.h, ctypes.byref(cnt), ctypes.byref(cap)))
        assert (cnt.value, cap.value) == (min(k + 1, 3), 3)
    out = np.empty((3, q.size))
    ctx.check(ctx.lib.nhp_cont_vb_trace_read(ctx.h, 0, 3, _ptr(out)))
    for k in range(3):
        assert np.array_equal(out[k], seen[k])
    assert not np.array_equal(seen[3], seen[2])
    with pytest.raises(nhp.NHPError) as e:
        ctx.check(ctx.lib.nhp_cont_vb_trace_read(ctx.h, 2, 2, _ptr(out)))
    assert e.value.code == _lib.NHP_ERR_INVALID
    ctx.check(ctx.lib.nhp_cont_vb_trace_free(ctx.h))
    ctx.check(ctx.lib.nhp_cont_vb_trace_count(ctx.h, ctypes.byref(cnt), ctypes.byref(cap)))
    assert (cnt.value, cap.value) == (0, 0)


def test_refusals_change_nothing(own):
    """Every refusal leaves the state and the parameters as they were."""
    K, kind = 3, EXP
    ctx, d, t, c, q = setup(own, kind, K, np.inf, [100, 100, 100], 50.0, 61)
    lam0, W, p1 = np.array([0.5, 0.6, 0.7]), np.full((K, K), 0.07), np.full((K, K), 1.3)

    def expect(code, fn, *params):
        with pytest.raises(nhp.NHPError) as e:
            ctx.check(fn())
        assert e.value.code == code, e.value
        assert np.array_equal(vb_get(ctx, kind, K), q)
        got = params_get(ctx, *params[:2])
        for a, b in zip(got, params[2:]):
            assert (a is None and b is None) or np.array_equal(a, b)

    push(ctx, EXP, K, np.inf, lam0, W, p1, A=np.ones((K, K)))  # a network process
    expect(_lib.NHP_ERR_UNSUPPORTED, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, d.h, None), EXP, K, lam0, W, p1, None)
    push(ctx, EXP, K, np.inf, lam0, W, p1)
    x, v = np.array([0.0, 60.0]), np.ones(2 * K)
    ctx.check(ctx.lib.nhp_cont_baseline_grid(ctx.h, 2, _ptr(x), _ptr(v)))  # curves
    expect(_lib.NHP_ERR_UNSUPPORTED, lambda: ctx.lib.nhp_cont_vb_stats(ctx.h, d.h, None, None, None, None), EXP, K, lam0, W, p1, None)
    push(ctx, EXP, K, np.inf, lam0, W, p1)
    shard = own.upload(ctx, t, c + 1, 50.0, K, n_halo=10, index_base=0, flags=1)  # a time shard
    expect(_lib.NHP_ERR_UNSUPPORTED, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, shard.h, None), EXP, K, lam0, W, p1, None)
    other = own.upload(ctx, t, np.minimum(c + 1, 2), 50.0, 2)  # events of another K
    expect(_lib.NHP_ERR_INVALID, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, other.h, None), EXP, K, lam0, W, p1, None)
    ctx.check(ctx.lib.nhp_cont_vb_trace_begin(ctx.h, 2))
    push(ctx, LN, K, 1.0, lam0, W, np.zeros((K, K)), np.ones((K, K)))  # kind changed since _set
    expect(_lib.NHP_ERR_STATE, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, d.h, None), LN, K, lam0, W, np.zeros((K, K)), np.ones((K, K)))
    push(ctx, EXP, K, np.inf, lam0, W, p1)
    ctx.check(ctx.lib.nhp_cont_vb_trace_free(ctx.h))
    hy = np.asarray(HYPER[LN])
    push(ctx, LN, K, 1.0, lam0, W, np.zeros((K, K)), np.ones((K, K)))
    ctx.check(ctx.lib.nhp_cont_vb_trace_begin(ctx.h, 2))  # a trace of the EXP state ...
    ctx.check(ctx.lib.nhp_cont_vb_set(ctx.h, _ptr(hy), hy.size, _ptr(random_state(K, LN, 1))))
    qln = vb_get(ctx, LN, K)
    with pytest.raises(nhp.NHPError) as e:  # ... refuses a step of the LN state
        ctx.check(ctx.lib.nhp_cont_vb_step(ctx.h, d.h, None))
    assert e.value.code == _lib.NHP_ERR_STATE and np.array_equal(vb_get(ctx, LN, K), qln)
    ctx.check(ctx.lib.nhp_cont_vb_trace_free(ctx.h))
    push(ctx, EXP, K, np.inf, lam0, W, p1)
    bad = q.copy()
    bad[2 * K] = -1.0
    for hyp, qq, n in ((HYPER[EXP], bad, 6), (HYPER[EXP][:5] + [0.0], q, 6), (HYPER[EXP], q, 8)):
        h = np.asarray(hyp + [1.0] * (n - len(hyp)), dtype=np.float64)
        with pytest.raises(nhp.NHPError) as e:
            ctx.check(ctx.lib.nhp_cont_vb_set(ctx.h, _ptr(h), n, _ptr(qq)))
        assert e.value.code == _lib.NHP_ERR_INVALID
    # K changed since _set (the LN state above is the kept one)
    push(ctx, LN, 2, 1.0, lam0[:2], W[:2, :2], np.zeros((2, 2)), np.ones((2, 2)))
    with pytest.raises(nhp.NHPError) as e:
        ctx.check(ctx.lib.nhp_cont_vb_step(ctx.h, other.h, None))
    assert e.value.code == _lib.NHP_ERR_STATE and np.array_equal(vb_get(ctx, LN, K), qln)
    fresh = own.context()  # no state
    push(fresh, EXP, K, np.inf)
    df = own.upload(fresh, t, c + 1, 50.0, K)
    with pytest.raises(nhp.NHPError) as e:
        fresh.check(fresh.lib.nhp_cont_vb_step(fresh.h, df.h, None))
    assert e.value.code == _lib.NHP_ERR_STATE


@pytest.mark.parametrize("kind,dtmax", [(EXP, 4.0), (LN, 1.0)])
def test_python_layer(kind, dtmax):
    """continuous.vb_statistics and vb_device_ (with and without the trace) on host data: the statistics and the states of the
    twin, to the tolerances above; the process ends at the posterior means of the last state."""
    K, T = 3, 80.0
    t, c = stream([150, 180, 210], T, 81 + kind)
    p = recovery_process(kind, K, 82)
    if kind == EXP:
        p.impulses.dtmax = dtmax
    p.baseline.alpha0, p.baseline.beta0, p.weights.kappa, p.weights.nu = HYPER[kind][:4]
    if kind == EXP:
        p.impulses.alpha, p.impulses.beta = HYPER[kind][4:]
    else:
        p.impulses.mumu, p.impulses.kappamu, p.impulses.alpha0, p.impulses.beta0 = HYPER[kind][4:]
    data = (t, c + 1, T)
    q0 = C.prior_variational_params(p)
    st = C.vb_statistics(p, data, q0)
    ref = R.expected_stats(t, c, K, kind, q0, dtmax)
    for k in ("M0", "Mnm", "S1") + (("S2",) if kind == LN else ()):
        assert nerr(st[k], ref[k]) <= 1e-12, k
    states = C.vb_device_(p, data, max_steps=4)
    assert len(states) == 4
    q = q0
    for k in range(4):
        q, _, _ = R.vb_step(t, c, K, kind, q, HYPER[kind], T, dtmax)
        assert np.allclose(states[k], q, rtol=1e-11, atol=1e-11)
    last = C.vb_device_(p, data, max_steps=4, trace=False)
    assert len(last) == 1 and np.allclose(last[0], states[-1], rtol=1e-13, atol=1e-13)
    m = C.posterior_means(p, last[0])
    assert np.array_equal(p.baseline.lam, m["lambda0"]) and np.array_equal(p.weights.W, m["W"])
    assert np.array_equal(p.impulses.p1(), m["p1"])


def recovery_process(kind, K, seed):
    rng = np.random.default_rng(seed)
    lam0 = rng.uniform(0.5, 1.0, K)
    W = rng.uniform(0.02, 0.18, (K, K))
    if kind == EXP:
        imp = nhp.ExponentialImpulseResponse(rng.uniform(1.0, 3.0, (K, K)))
    else:
        imp = nhp.LogitNormalImpulseResponse(rng.normal(0.0, 0.5, (K, K)), rng.uniform(1.0, 3.0, (K, K)), 1.0)
    return nhp.ContinuousStandardHawkesProcess(nhp.HomogeneousProcess(lam0), imp, nhp.DenseWeightModel(W))


@pytest.mark.parametrize("kind", [EXP, LN])
def test_recovery_against_device_chain(kind):
    """A rand_device sample of about 2e5 events (K = 5); VB from the prior reaches change <= 1e-8 (measured: after 8753 steps for
    Exponential, 1377 for LogitNormal; the Exponential impulse's theta is a slow direction of mean-field VB), and its posterior means
    of lambda0 and W lie within 3 standard deviations (of the chain) of the means of a 2000-sweep mcmc_device_ chain, the first 500
    dropped (measured: within 0.83 of them for Exponential, 0.58 for LogitNormal)."""
    K = 5
    p = recovery_process(kind, K, 70 + kind)
    rate = np.linalg.solve(np.eye(K) - p.weights.W.T, p.baseline.lam).sum()
    d = nhp.rand_device(p, 2e5 / rate, seed=3)
    assert 1.5e5 < d.n < 2.5e5
    chain = nhp.mcmc_device_(p, d, nsteps=2000, seed=9)
    S = np.array(chain.samples[500:])
    np_imp = K * K * (1 if kind == EXP else 2)
    lam_s, W_s = S[:, :K], S[:, K + np_imp:K + np_imp + K * K]
    states = C.vb_device_(p, d, max_steps=12000, rtol=1e-8, trace=False)
    q = states[-1]
    m = C.posterior_means(p, q)
    assert np.array_equal(p.baseline.lam, m["lambda0"]) and np.array_equal(p.weights.W, m["W"])  # the process holds the means
    # converged: one more step moves nothing by more than 1e-8
    ctx = p._ctx()
    assert step(ctx, d) <= 1e-8
    for vb, s in ((m["lambda0"], lam_s), (m["W"].T.ravel(), W_s)):
        mu, sd = s.mean(axis=0), s.std(axis=0)
        print("recovery", kind, np.max(np.abs(vb - mu) / sd))
        assert np.all(np.abs(vb - mu) <= 3 * sd), np.max(np.abs(vb - mu) / sd)
