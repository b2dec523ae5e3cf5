"""Continuous network VB on the device (nhp_cont_vb_network_set, nhp_cont_vb_stats / _step / _get and the VB trace on a network state,
continuous.network_vb_device_), against the NumPy twin of tests/cont_vb_network_reference.py.

The device runs the intensity sweep and the gradient's child-major scatter with floating-point atomics, so its sums come in an order
that changes from run to run; the tolerances are those of tests/test_cont_vb_gpu.py."""
import ctypes

import numpy as np
import pytest

import cont_vb_network_reference as RN
import cont_vb_reference as R
import nhp_b200 as nhp
from nhp_b200 import _lib
from nhp_b200 import continuous as C
from nhp_b200.core import Context, ContinuousData, _fmat, _ptr

pytestmark = pytest.mark.gpu

EXP, LN = R.EXP, R.LN
HYPER = {EXP: [1.5, 0.5, 2.0, 3.0, 2.0, 1.0, 0.1, 10.0, 1.0, 1.0], LN: [1.5, 0.5, 2.0, 3.0, 0.2, 1.5, 2.0, 0.7, 0.1, 10.0, 1.0, 1.0]}


def stream(counts, T, seed):
    rng = np.random.default_rng(seed)
    c = rng.permutation(np.repeat(np.arange(len(counts)), counts))
    return np.sort(rng.uniform(0.0, T, c.size)), c


def random_state(K, kind, seed, wscale=1.0):
    rng = np.random.default_rng(seed)
    mats = [rng.uniform(0.5, 3.0, (K, K)), rng.uniform(3.0, 30.0, (K, K)) * wscale]
    if kind == EXP:
        mats += [rng.uniform(2.0, 10.0, (K, K)), rng.uniform(0.5, 3.0, (K, K))]
    else:
        mats += [rng.normal(0.0, 1.0, (K, K)), rng.uniform(0.5, 5.0, (K, K)), rng.uniform(1.0, 6.0, (K, K)), rng.uniform(0.5, 3.0, (K, K))]
    qs = R.pack(rng.uniform(2.0, 10.0, K), rng.uniform(1.0, 5.0, K), mats)
    return RN.join(qs, rng.uniform(0.05, 0.5, (K, K)), rng.uniform(2.0, 20.0, (K, K)) * wscale, rng.uniform(0.0, 1.0, (K, K)),
                   rng.uniform(1.0, 4.0), rng.uniform(1.0, 4.0))


def push(ctx, kind, K, dtmax, lam0=None, W=None, p1=None, p2=None, A="ones"):
    lam0 = np.ones(K) if lam0 is None else lam0
    W = np.full((K, K), 0.05) if W is None else W
    p1 = (np.ones((K, K)) if kind == EXP else np.zeros((K, K))) if p1 is None else p1
    p2 = (None if kind == EXP else np.ones((K, K))) if p2 is None else p2
    A = np.ones((K, K)) if isinstance(A, str) else A
    ctx.check(ctx.lib.nhp_cont_params_set(ctx.h, kind, K, _ptr(np.ascontiguousarray(lam0, dtype=np.float64)), _ptr(_fmat(W)),
                                          None if A is None else _ptr(_fmat(A)), _ptr(_fmat(p1)), None if p2 is None else _ptr(_fmat(p2)), float(dtmax)))


def net_set(ctx, kind, q, hyper=None):
    hy = np.asarray(HYPER[kind] if hyper is None else hyper, dtype=np.float64)
    ctx.check(ctx.lib.nhp_cont_vb_network_set(ctx.h, _ptr(hy), hy.size, _ptr(np.ascontiguousarray(q, dtype=np.float64))))


def vb_get(ctx, n):
    q = np.empty(n)
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
    lam, W, A, p1 = np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
    p2 = np.empty(K * K) if kind == LN else None
    ctx.check(ctx.lib.nhp_cont_params_get(ctx.h, _ptr(lam), _ptr(W), _ptr(A), _ptr(p1), _ptr(p2)))
    f = lambda v: None if v is None else v.reshape(K, K).T.copy()
    return lam, f(W), f(A), f(p1), f(p2)


def rho_get(ctx):
    r = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_network_get(ctx.h, ctypes.byref(r)))
    return r.value


def nerr(a, b):
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


def masks(K, kind):
    """(positive entries, mv and pv) of a network state: the entries compared relatively and absolutely."""
    n = 2 * K + R.nplanes(kind) * K * K + 3 * K * K + 2
    ab = np.zeros(n, bool)
    if kind == LN:
        ab[2 * K + 2 * K * K:2 * K + 3 * K * K] = True
    p0 = 2 * K + R.nplanes(kind) * K * K + 2 * K * K
    ab[p0:p0 + K * K] = True
    return ~ab, ab


def state_err(a, b, K, kind):
    pos, ab = masks(K, kind)
    return max(float(np.max(np.abs(a[pos] - b[pos]) / b[pos])), float(np.max(np.abs(a[ab] - b[ab]))))


class Owned:
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
    """Frees a test's events handles, then its contexts, when it ends."""
    o = Owned()
    yield o
    for d in o.data:
        d.free()
    for c in o.ctxs:
        c._fin()


def setup(own, kind, K, dtmax, counts, T, seed, wscale=1.0):
    ctx = own.context()
    t, c = stream(counts, T, seed)
    d = own.upload(ctx, t, c + 1, T, K)
    q = random_state(K, kind, seed + 100, wscale)
    push(ctx, kind, K, dtmax)
    net_set(ctx, kind, q)
    return ctx, d, t, c, q


STATS_CASES = [
    # kind, dtmax, K, events per node, duration
    (EXP, np.inf, 1, [700], 100.0),
    (LN, 1.0, 1, [700], 100.0),
    (EXP, np.inf, 3, [255, 256, 257], 60.0),
    (LN, 1.0, 3, [255, 256, 257], 60.0),
    (EXP, 0.5, 17, [120] * 17, 150.0),
    (LN, 1.5, 17, [120] * 17, 150.0),
    (EXP, np.inf, 64, [40] * 64, 100.0),
    (LN, 1.0, 64, [40] * 64, 100.0),
]


@pytest.mark.parametrize("kind,dtmax,K,counts,T", STATS_CASES)
def test_stats_match_twin(own, kind, dtmax, K, counts, T):
    """nhp_cont_vb_stats of a network state against the twin: M0 entrywise, Mnm / S1 / S2 normwise, relative error <= 1e-12; q is not
    changed by the call."""
    ctx, d, t, c, q = setup(own, kind, K, dtmax, counts, T, 7 * K + kind)
    dev = dev_stats(ctx, d, K)
    ref = RN.expected_stats(t, c, K, kind, q, dtmax)
    assert np.all(np.abs(dev["M0"] - ref["M0"]) <= 1e-12 * ref["M0"])
    for k in ("Mnm", "S1") + (("S2",) if kind == LN else ()):
        assert nerr(dev[k], ref[k]) <= 1e-12, (k, nerr(dev[k], ref[k]))
    assert np.array_equal(vb_get(ctx, q.size), q)


@pytest.mark.parametrize("kind,dtmax", [(EXP, 2.0), (LN, 1.0)])
def test_stats_match_twin_config4_width(own, kind, dtmax):
    """K = 1000 (config 4's width; the columns' accumulators in shared memory) on 2e4 events, to the same tolerance."""
    K = 1000
    rng = np.random.default_rng(5 + kind)
    counts = np.bincount(rng.integers(0, K, 20000), minlength=K)
    ctx, d, t, c, q = setup(own, kind, K, dtmax, counts, 100.0, 13 + kind, wscale=100.0)
    dev = dev_stats(ctx, d, K)
    ref = RN.expected_stats(t, c, K, kind, q, dtmax)
    errs = [nerr(dev[k], ref[k]) for k in ("Mnm", "S1") + (("S2",) if kind == LN else ())]
    print("stats error K=1000", kind, errs)
    assert np.all(np.abs(dev["M0"] - ref["M0"]) <= 1e-12 * ref["M0"])
    assert max(errs) <= 1e-12


@pytest.mark.parametrize("kind,dtmax", [(EXP, np.inf), (EXP, 3.0), (LN, 1.0)])
def test_steps_match_twin(own, kind, dtmax):
    """One step, then 10 chained steps, against the twin, from a state with some link probabilities exactly 0 and 1: positive entries
    relative, mv and pv absolute, <= 1e-12 after one step and <= 1e-11 after ten; `change` as the twin's to 1e-12."""
    K = 4
    ctx = own.context()
    t, c = stream([400, 300, 350, 450], 150.0, 31 + kind)
    d = own.upload(ctx, t, c + 1, 150.0, K)
    q = random_state(K, kind, 131 + kind)
    qs, k0v, n0v, pv, ar, br = RN.split(q, K, kind)
    pv[0, :2], pv[1, 2:] = 0.0, 1.0
    q = RN.join(qs, k0v, n0v, pv, ar, br)
    push(ctx, kind, K, dtmax)
    net_set(ctx, kind, q)
    qt = q
    for k in range(10):
        ch = step(ctx, d)
        qt, cht, _ = RN.vb_step(t, c, K, kind, qt, HYPER[kind], 150.0, dtmax)
        qd = vb_get(ctx, q.size)
        assert state_err(qd, qt, K, kind) <= (1e-12 if k == 0 else 1e-11), (k, state_err(qd, qt, K, kind))
        assert abs(ch - cht) <= 1e-12 * max(cht, 1e-3), (k, ch, cht)


@pytest.mark.parametrize("kind,dtmax", [(EXP, np.inf), (LN, 1.0)])
def test_device_trace_bound_never_decreases(own, kind, dtmax):
    """The twin's bound of every state of a 25-step device trace from the all-links start never decreases."""
    K, T = 3, 60.0
    ctx = own.context()
    t, c = stream([80, 60, 90], T, 41 + kind)
    d = own.upload(ctx, t, c + 1, T, K)
    q = RN.prior_state(K, kind, HYPER[kind])
    push(ctx, kind, K, dtmax)
    net_set(ctx, kind, q)
    ctx.check(ctx.lib.nhp_cont_vb_trace_begin(ctx.h, 25))
    for _ in range(25):
        step(ctx, d)
    out = np.empty((25, q.size))
    ctx.check(ctx.lib.nhp_cont_vb_trace_read(ctx.h, 0, 25, _ptr(out)))
    ctx.check(ctx.lib.nhp_cont_vb_trace_free(ctx.h))
    prev = RN.elbo(t, c, K, kind, q, HYPER[kind], T, dtmax)
    for k in range(25):
        cur = RN.elbo(t, c, K, kind, out[k], HYPER[kind], T, dtmax)
        assert cur >= prev - 1e-12 * abs(prev), (k, prev, cur)
        prev = cur


@pytest.mark.parametrize("kind,dtmax", [(EXP, 3.0), (LN, 1.0)])
def test_spike_equal_to_slab_is_the_standard_step(own, kind, dtmax):
    """kappa0 = kappa, nu0 = nu, kappa0v = kappav, nu0v = nuv: the standard part of a network step equals nhp_cont_vb_step on the matching
    standard state (1e-12), and pv = sigmoid(psi(alpharhov) - psi(betarhov))."""
    from scipy.special import digamma, expit
    K = 3
    t, c = stream([200, 150, 250], 80.0, 51 + kind)
    q = random_state(K, kind, 151 + kind)
    qs, _, _, pv, ar, br = RN.split(q, K, kind)
    _, _, P = R.planes(qs, K, kind)
    q = RN.join(qs, P[0], P[1], pv, ar, br)
    h = list(HYPER[kind])
    ns = RN.nstd(kind)
    h[ns], h[ns + 1] = h[2], h[3]
    cn, cs = own.context(), own.context()
    dn, ds = own.upload(cn, t, c + 1, 80.0, K), own.upload(cs, t, c + 1, 80.0, K)
    push(cn, kind, K, dtmax)
    net_set(cn, kind, q, h)
    push(cs, kind, K, dtmax, A=None)
    hs = np.asarray(h[:ns], dtype=np.float64)
    cs.check(cs.lib.nhp_cont_vb_set(cs.h, _ptr(hs), hs.size, _ptr(qs)))
    step(cn, dn)
    step(cs, ds)
    qn, qsd = vb_get(cn, q.size), vb_get(cs, qs.size)
    np.testing.assert_allclose(RN.split(qn, K, kind)[0], qsd, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(RN.split(qn, K, kind)[3], expit(digamma(ar) - digamma(br)), rtol=1e-12)


@pytest.mark.parametrize("kind,dtmax", [(EXP, np.inf), (LN, 1.0)])
def test_context_holds_the_point_estimate(own, kind, dtmax):
    """After a step the context holds lambda0, the slab mean of W, p1, p2, A = [pv > 1/2] (bit for bit) and rho = alpharhov /
    (alpharhov + betarhov); its log-likelihood is that of those values pushed from the host, and a Gibbs sweep runs from them."""
    K = 3
    ctx, d, t, c, q = setup(own, kind, K, dtmax, [300, 200, 250], 100.0, 61 + kind)
    qs, k0v, n0v, pv, ar, br = RN.split(q, K, kind)
    pv[:] = np.array([[0.9, 0.2, 0.6], [0.1, 0.8, 0.3], [0.7, 0.4, 0.95]])
    net_set(ctx, kind, RN.join(qs, k0v, n0v, pv, ar, br))
    step(ctx, d)
    qn = vb_get(ctx, q.size)
    qsn, _, _, pvn, arn, brn = RN.split(qn, K, kind)
    lam, W, A, p1, p2 = params_get(ctx, kind, K)
    l0w, Ww, p1w, p2w = R.posterior_means(qsn, K, kind)
    assert np.array_equal(lam, l0w) and np.array_equal(W, Ww) and np.array_equal(p1, p1w)
    assert (p2 is None) if kind == EXP else np.array_equal(p2, p2w)
    assert np.array_equal(A, (pvn > 0.5).astype(float))
    assert rho_get(ctx) == arn / (arn + brn)
    ll1, ll2 = ctypes.c_double(), ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll1)))
    push(ctx, kind, K, dtmax, l0w, Ww, p1w, p2w, A=A)
    ctx.check(ctx.lib.nhp_cont_loglik(ctx.h, d.h, 0, ctypes.byref(ll2)))
    assert abs(ll1.value - ll2.value) <= 1e-13 * abs(ll2.value)
    net_set(ctx, kind, q)  # again from the step's point estimate, then one Gibbs sweep of the network process
    step(ctx, d)
    hy = np.asarray(HYPER[kind][:RN.nstd(kind)], dtype=np.float64)
    ctx.check(ctx.lib.nhp_cont_gibbs_sweep(ctx.h, d.h, d.h, 1, 0, 100.0, _ptr(hy), hy.size, 1.0, 1.0))
    lam, W, A, _, _ = params_get(ctx, kind, K)
    assert np.all(np.isfinite(lam)) and np.all(np.isfinite(W)) and set(np.unique(A)) <= {0.0, 1.0}
    assert 0.0 < rho_get(ctx) < 1.0


def test_trace_with_both_kinds_of_state(own):
    """The trace takes the slot size of the state at _begin: a network trace keeps network states, a standard one standard states; a
    step on a trace begun for the other kind of state is refused and changes nothing."""
    K, kind = 3, LN
    ctx, d, t, c, q = setup(own, kind, K, 1.0, [200, 200, 200], 80.0, 71)
    ctx.check(ctx.lib.nhp_cont_vb_trace_begin(ctx.h, 3))
    seen = []
    for _ in range(4):
        step(ctx, d)
        seen.append(vb_get(ctx, q.size))
    cnt, cap = ctypes.c_int64(), ctypes.c_int64()
    ctx.check(ctx.lib.nhp_cont_vb_trace_count(ctx.h, ctypes.byref(cnt), ctypes.byref(cap)))
    assert (cnt.value, cap.value) == (3, 3)
    out = np.empty((3, q.size))
    ctx.check(ctx.lib.nhp_cont_vb_trace_read(ctx.h, 0, 3, _ptr(out)))
    assert all(np.array_equal(out[k], seen[k]) for k in range(3))
    # a standard state on a network trace: refused (the parameters lose their adjacency matrix for the standard state)
    qs = RN.split(q, K, kind)[0]
    hs = np.asarray(HYPER[kind][:8], dtype=np.float64)
    push(ctx, kind, K, 1.0, A=None)
    ctx.check(ctx.lib.nhp_cont_vb_set(ctx.h, _ptr(hs), hs.size, _ptr(qs)))
    with pytest.raises(nhp.NHPError) as e:
        ctx.check(ctx.lib.nhp_cont_vb_step(ctx.h, d.h, None))
    assert e.value.code == _lib.NHP_ERR_STATE and np.array_equal(vb_get(ctx, qs.size), qs)
    ctx.check(ctx.lib.nhp_cont_vb_trace_begin(ctx.h, 2))  # a standard trace now
    step(ctx, d)
    slot = np.empty(qs.size)
    ctx.check(ctx.lib.nhp_cont_vb_trace_read(ctx.h, 0, 1, _ptr(slot)))
    assert np.array_equal(slot, vb_get(ctx, qs.size))
    push(ctx, kind, K, 1.0)  # ... and a network state on it: refused
    net_set(ctx, kind, q)
    with pytest.raises(nhp.NHPError) as e:
        ctx.check(ctx.lib.nhp_cont_vb_step(ctx.h, d.h, None))
    assert e.value.code == _lib.NHP_ERR_STATE and np.array_equal(vb_get(ctx, q.size), q)
    ctx.check(ctx.lib.nhp_cont_vb_trace_free(ctx.h))


def test_refusals_change_nothing(own):
    """Every refusal of a network state leaves the state and the parameters as they were."""
    K, kind = 3, EXP
    ctx, d, t, c, q = setup(own, kind, K, np.inf, [100, 100, 100], 50.0, 81)
    lam0, W, p1, A = np.array([0.5, 0.6, 0.7]), np.full((K, K), 0.07), np.full((K, K), 1.3), np.eye(K)

    def expect(code, fn, pk=EXP, pK=K, pdt=np.inf, pA=A, pp1=p1, pp2=None):
        with pytest.raises(nhp.NHPError) as e:
            ctx.check(fn())
        assert e.value.code == code, e.value
        assert np.array_equal(vb_get(ctx, q.size), q)
        got = params_get(ctx, pk, pK) if pA is not None else None
        if got is not None:
            for a, b in zip(got, (lam0[:pK], W[:pK, :pK], pA, pp1, pp2)):
                assert (a is None and b is None) or np.array_equal(a, b)

    push(ctx, EXP, K, np.inf, lam0, W, p1, A=None)  # no adjacency matrix
    expect(_lib.NHP_ERR_STATE, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, d.h, None), pA=None)
    push(ctx, EXP, K, np.inf, lam0, W, p1, A=A)
    x, v = np.array([0.0, 60.0]), np.ones(2 * K)
    ctx.check(ctx.lib.nhp_cont_baseline_grid(ctx.h, 2, _ptr(x), _ptr(v)))  # curves
    expect(_lib.NHP_ERR_UNSUPPORTED, lambda: ctx.lib.nhp_cont_vb_stats(ctx.h, d.h, None, None, None, None))
    push(ctx, EXP, K, np.inf, lam0, W, p1, A=A)
    shard = own.upload(ctx, t, c + 1, 50.0, K, n_halo=10, index_base=0, flags=1)  # a time shard
    expect(_lib.NHP_ERR_UNSUPPORTED, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, shard.h, None))
    other = own.upload(ctx, t, np.minimum(c + 1, 2), 50.0, 2)  # events of another K
    expect(_lib.NHP_ERR_INVALID, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, other.h, None))
    push(ctx, LN, K, 1.0, lam0, W, np.zeros((K, K)), np.ones((K, K)), A=A)  # kind changed since _set
    expect(_lib.NHP_ERR_STATE, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, d.h, None), LN, K, 1.0, A, np.zeros((K, K)), np.ones((K, K)))
    push(ctx, EXP, 2, np.inf, lam0[:2], W[:2, :2], p1[:2, :2], A=A[:2, :2])  # K changed since _set
    expect(_lib.NHP_ERR_STATE, lambda: ctx.lib.nhp_cont_vb_step(ctx.h, other.h, None), EXP, 2, np.inf, A[:2, :2], p1[:2, :2])
    push(ctx, EXP, K, np.inf, lam0, W, p1, A=A)
    hy = np.asarray(HYPER[EXP], dtype=np.float64)
    pv0 = 2 * K + 6 * K * K
    for bad_i, bad_v in ((pv0, 1.5), (pv0 + 1, -0.1), (pv0, np.nan), (q.size - 1, 0.0), (2 * K + 4 * K * K, -1.0)):
        qq = q.copy()
        qq[bad_i] = bad_v
        expect(_lib.NHP_ERR_INVALID, lambda: ctx.lib.nhp_cont_vb_network_set(ctx.h, _ptr(hy), hy.size, _ptr(qq)))
    for hh, n in ((np.concatenate([hy[:6], [0.0], hy[7:]]), 10), (hy, 6), (np.concatenate([hy[:9], [np.inf]]), 10)):
        expect(_lib.NHP_ERR_INVALID, lambda: ctx.lib.nhp_cont_vb_network_set(ctx.h, _ptr(np.ascontiguousarray(hh)), n, _ptr(q)))
    fresh = own.context()  # no parameters
    with pytest.raises(nhp.NHPError) as e:
        fresh.check(fresh.lib.nhp_cont_vb_network_set(fresh.h, _ptr(hy), hy.size, _ptr(q)))
    assert e.value.code == _lib.NHP_ERR_STATE
    # a standard state still refuses a network process
    hs = np.asarray(HYPER[EXP][:6], dtype=np.float64)
    qs = RN.split(q, K, EXP)[0]
    ctx.check(ctx.lib.nhp_cont_vb_set(ctx.h, _ptr(hs), hs.size, _ptr(qs)))
    with pytest.raises(nhp.NHPError) as e:
        ctx.check(ctx.lib.nhp_cont_vb_step(ctx.h, d.h, None))
    assert e.value.code == _lib.NHP_ERR_UNSUPPORTED and np.array_equal(vb_get(ctx, qs.size), qs)


def test_python_layer(own):
    """network_vb_statistics and network_vb_device_ on host data: the twin's statistics and states; the process ends at the device's
    point estimate with network.rho and network.pv of the last state."""
    K, T, kind, dtmax = 3, 80.0, LN, 1.0
    t, c = stream([150, 180, 210], T, 91)
    rng = np.random.default_rng(92)
    imp = nhp.LogitNormalImpulseResponse(rng.normal(0.0, 0.5, (K, K)), rng.uniform(1.0, 3.0, (K, K)), dtmax, 0.2, 1.5, 2.0, 0.7)
    p = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(rng.uniform(0.5, 1.0, K), 1.5, 0.5), imp,
                                           nhp.DenseWeightModel(rng.uniform(0.02, 0.18, (K, K)), 2.0, 3.0), np.ones((K, K)),
                                           nhp.BernoulliNetworkModel(0.5, K, 1.0, 1.0))
    data = (t, c + 1, T)
    q0 = C.network_prior_variational_params(p)
    st = C.network_vb_statistics(p, data, q0)
    ref = RN.expected_stats(t, c, K, kind, q0, dtmax)
    for k in ("M0", "Mnm", "S1", "S2"):
        assert nerr(st[k], ref[k]) <= 1e-12, k
    states = C.network_vb_device_(p, data, max_steps=4)
    q = q0
    for k in range(4):
        q, _, _ = RN.vb_step(t, c, K, kind, q, HYPER[kind], T, dtmax)
        assert state_err(states[k], q, K, kind) <= 1e-11
    last = C.network_vb_device_(p, data, max_steps=4, trace=False)
    assert len(last) == 1 and state_err(last[0], states[-1], K, kind) <= 1e-13
    m = C.network_posterior_means(p, last[0])
    assert np.array_equal(p.weights.W, m["W_slab"]) and np.array_equal(p.baseline.lam, m["lambda0"])
    assert np.array_equal(p.adjacency_matrix, (m["A"] > 0.5).astype(float))
    assert p.network.rho == m["rho"] and np.array_equal(p.network.pv, m["A"])


def recovery_process(seed):
    """K = 6 LogitNormal network process: 12 of the 36 links on, their weights in [0.1, 0.25]."""
    K = 6
    rng = np.random.default_rng(seed)
    A = np.zeros(K * K)
    A[rng.permutation(K * K)[:12]] = 1.0
    A = A.reshape(K, K)
    W = rng.uniform(0.1, 0.25, (K, K))
    imp = nhp.LogitNormalImpulseResponse(rng.normal(0.0, 0.5, (K, K)), rng.uniform(1.0, 3.0, (K, K)), 1.0)
    return nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(rng.uniform(0.5, 1.0, K)), imp, nhp.DenseWeightModel(W), A,
                                              nhp.BernoulliNetworkModel(1.0 / 3.0, K))


def test_recovery_against_device_chain():
    """A rand_device sample of about 2e5 events (K = 6, 12 links on, their weights in [0.1, 0.25]).  VB from the default start (every
    link on) reaches change <= 1e-8 (measured on an NVIDIA B200, 1000 W power limit: after 1416 steps); [pv > 1/2] is the true adjacency
    matrix (measured: pv of the on links 0.63 to 0.83, of the off links at most 0.041) and the slab means of the on links lie within 3
    standard deviations of the means of a 2000-sweep mcmc_device_ chain, the first 500 dropped (measured: within 0.19 of them).

    The chain's own majority A is not the true one: an off link's weight is drawn from Gamma(kappa, nu + Mn[p]) (about 3e-5 here), at
    which the adjacency sweep's odds are those of rho, and rho's Beta draw counts those links, so the chain sits at rho = 0.93 with every
    off link on in 94 % of the samples, at weights of at most 0.02.  Its majority of effective links (A = 1 and a sampled weight above
    0.01) is the true A, and that is what [pv > 1/2] must equal.

    From pv = rho (the default start of the discrete network VB) the run stops after 264 steps with one link on: 7 on links settle at
    pv ~ 5e-6 and the other 5 between 0.39 and 0.54, since the first E-step's weights come mostly from the spike.  That is asserted too."""
    p = recovery_process(17)
    K = 6
    A_true = p.adjacency_matrix.copy()
    rate = np.linalg.solve(np.eye(K) - (A_true * p.weights.W).T, p.baseline.lam).sum()
    d = nhp.rand_device(p, 2e5 / rate, seed=5)
    assert 1.5e5 < d.n < 2.5e5
    chain = nhp.mcmc_device_(p, d, nsteps=2000, seed=9)
    S = np.array(chain.samples[500:])
    # [rho; lambda0; W; mu; tau; vec(A)]
    rho_s, W_s, A_s = S[:, 0], S[:, 1 + K:1 + K + K * K], S[:, 1 + K + 3 * K * K:]
    f = lambda v: v.reshape(K, K).T
    A_major = f(A_s.mean(axis=0) > 0.5).astype(float)
    A_eff = f((A_s * (W_s > 0.01)).mean(axis=0) > 0.5).astype(float)
    off = A_true == 0.0
    print("chain: rho mean", float(rho_s.mean()), "off links: A = 1 in", float(f(A_s.mean(axis=0))[off].mean()), "of the samples, largest W",
          float(f(W_s.max(axis=0))[off].max()), "majority A == A_true", np.array_equal(A_major, A_true), "effective == A_true", np.array_equal(A_eff, A_true))
    states = C.network_vb_device_(p, d, max_steps=20000, rtol=1e-8)
    m = C.network_posterior_means(p, states[-1])
    A_vb = (m["A"] > 0.5).astype(float)
    on = A_true.T.ravel() == 1.0
    mu, sd = W_s.mean(axis=0), W_s.std(axis=0)
    margin = np.abs(m["W_slab"].T.ravel() - mu)[on] / sd[on]
    print("recovery: steps", len(states), "A_vb == A_true", np.array_equal(A_vb, A_true), "max margin", float(np.max(margin)),
          "pv on", np.sort(m["A"][A_true == 1.0]).tolist(), "pv off max", float(np.max(m["A"][off])), "rho", m["rho"])
    ctx = p._ctx()
    last_change = step(ctx, d)
    # from pv = rho (the discrete path's default start)
    q_rho = C.network_prior_variational_params(p, pv=1.0 / 3.0)
    tr = C.network_vb_device_(p, d, max_steps=20000, rtol=1e-8, q0=q_rho)
    mr = C.network_posterior_means(p, tr[-1])
    print("from pv = rho: steps", len(tr), "links on", int(np.sum(mr["A"] > 0.5)), "equal to A_true", np.array_equal((mr["A"] > 0.5).astype(float), A_true),
          "pv on", np.sort(mr["A"][A_true == 1.0]).tolist(), "pv off max", float(np.max(mr["A"][off])))
    assert np.array_equal(A_vb, A_true) and np.array_equal(A_vb, A_eff)
    assert np.all(margin <= 3.0), margin
    assert last_change <= 1e-8
    assert int(np.sum(mr["A"] > 0.5)) < int(A_true.sum())
