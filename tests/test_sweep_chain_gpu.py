"""Chained device Gibbs sweeps checked stage by stage against the oracle, and the cached pair structure of an events handle
shared by models of another impulse kind or dtmax.

A step of the device chain (what bench.py times) is nhp_cont_loglik_dist followed by nhp_cont_gibbs_sweep on one resident
handle: parent sweep with fused statistics, second pass, conjugate draws, adjacency sweep over the handle's cached pair
structure, commit (masked tables, abits), Beta draw of rho.  Every stage reads what the stage before it left on the device.  The
conjugate and Beta draws are not reproducible on the host; everything else is, given the values read back: the parents and the
adjacency sweep use Philox uniforms (synth.philox_uniform), the statistics and the log-likelihood are deterministic."""
import ctypes

import numpy as np
import pytest

import nhp_b200 as nhp
import oracle_ffi as orc
import synth
from nhp_b200 import continuous
from nhp_b200.core import _ptr
from test_cont_gpu import make_exp, make_ln

pytestmark = pytest.mark.gpu

SEED, STEPS, RHO0 = 4242, 6, 0.15


@pytest.fixture(scope="module", autouse=True)
def oracle_threads():
    """The oracle's adjacency sweep runs its columns in parallel (they are independent: the same result on any thread count)."""
    orc.set_threads(orc.max_threads())
    yield
    orc.set_threads(1)


def read_params(ctx, K, ln):
    """nhp_cont_params_get + nhp_cont_network_get: (dict of [parent, child] matrices, rho)."""
    l0, W, A, p1 = np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
    p2 = np.empty(K * K) if ln else None
    ctx.check(ctx.lib.nhp_cont_params_get(ctx.h, _ptr(l0), _ptr(W), _ptr(A), _ptr(p1), _ptr(p2)))
    rho = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_network_get(ctx.h, ctypes.byref(rho)))
    unf = lambda v: None if v is None else v.reshape(K, K).T.copy()
    return dict(lambda0=l0, W=unf(W), A=unf(A), p1=unf(p1), p2=unf(p2)), rho.value


def oracle(P, A, ln, dtmax):
    return orc.Cont(1 if ln else 0, P["lambda0"], P["W"], P["p1"], P["p2"], A=A, dtmax=dtmax)


def assert_params_equal(P, Q):
    for key in ("lambda0", "W", "A", "p1", "p2"):
        if P[key] is not None or Q[key] is not None:
            np.testing.assert_array_equal(P[key], Q[key], err_msg=key)


def device_loglik(ctx, d):
    ll = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_loglik_dist(ctx.h, d.h, d.h, 0, ctypes.byref(ll)))
    return ll.value


# id: (impulse, environment, bytes per cached pair, cluster size: 1, 0 (streaming form) or "multi" (2..8 CTAs per column))
VARIANTS = {
    "ln_payload": ("ln", {}, 18, 1),
    "ln_lags": ("ln", {"NHP_ADJ_PRE": "0"}, 10, 1),
    "exp_moving_horizon": ("exp", {}, 10, 1),
    "ln_chunk64_cluster": ("ln", {"NHP_ADJ_CHUNK": "64"}, 18, "multi"),
    "ln_chunk7_streaming": ("ln", {"NHP_ADJ_CHUNK": "7"}, 18, 0),
    "ln_chunk64_forced_streaming": ("ln", {"NHP_ADJ_CHUNK": "64", "NHP_ADJ_CLUSTER": "0"}, 18, 0),
}


@pytest.mark.parametrize("mode", ["free", "rewind"])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_chained_gibbs_sweeps_match_oracle_stage_by_stage(monkeypatch, variant, mode):
    """Six chained steps on one handle.  Before step s the device holds P_s, rho_s; then
    - log-likelihood == oracle and == the window sweep; from step 1 on, while the network is sparse, it goes through the structure
      (every step of the rewind chain, at least two of the free one);
    - parents == oracle's given the Philox uniforms of (SEED, event, s); statistics == oracle's of those parents;
    - adjacency matrix after the sweep == oracle's sweep with the freshly drawn lambda0, W, impulse, the old A_s and rho_s, given the
      Philox uniforms of (SEED, p + K c, s + 2^40) (comm.cu: draws, then adjacency, then the Beta draw of rho);
    - the device trace holds every step's sample bit for bit.
    rewind: params_restore + network_set before every step (the benchmark's chain), so every P_s == P_0."""
    kind, env, bytes_per_pair, cluster = VARIANTS[variant]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ln = kind == "ln"
    # Weights small enough for the Poisson data that a free chain stays near its initial density: with larger ones the draws
    # shrink lambda0, links switch on and the network is past the structure log-likelihood's density limit within two steps.
    if ln:  # mean window 40 events at D = 1: buckets of ~550 entries per (column, parent) straddle many 32-entry groups
        K, n, D = 24, 8000, 1.0
        t, nodes, T = synth.poisson_stream(n, K, 40.0, 17)
        proc, _ = make_ln(K, 19, density=RHO0, wmax=0.25 / (K * RHO0), dtmax=D)
    else:  # dtmax = Inf: the sampler's cut-off horizon moves with every theta draw (the oracle scans the whole history: small n)
        K, n, D = 12, 3000, np.inf
        t, nodes, T = synth.poisson_stream(n, K, 20.0, 18)
        proc, _ = make_exp(K, 20, density=RHO0, wmax=0.1 / (K * RHO0), dtmax=D)
    ctx = proc._ctx()
    lib = ctx.lib
    d = proc.upload((t, nodes, T))
    proc._push(ctx)
    ctx.check(lib.nhp_cont_network_set(ctx.h, RHO0))
    hyper = continuous._hyper(proc)
    P0, _ = read_params(ctx, K, ln)
    kk = (np.arange(K)[:, None] + K * np.arange(K)[None, :]).astype(np.uint64)  # u[p, c] is keyed by p + K c
    samples, structure_steps = [], 0
    ctx.check(lib.nhp_cont_trace_begin(ctx.h, STEPS))
    try:
        if mode == "rewind":
            ctx.check(lib.nhp_cont_params_save(ctx.h))
        for s in range(STEPS):
            if mode == "rewind":
                ctx.check(lib.nhp_cont_params_restore(ctx.h))
                ctx.check(lib.nhp_cont_network_set(ctx.h, RHO0))
            P, rho = read_params(ctx, K, ln)
            if mode == "rewind":
                assert_params_equal(P, P0)
                assert rho == RHO0
            om = oracle(P, P["A"], ln, D)
            # ---- log-likelihood of P_s
            ll = device_loglik(ctx, d)
            assert ll == pytest.approx(om.loglik(t, nodes, T, recursive=False), rel=1e-10), s
            if s > 0 and np.count_nonzero(P["A"] * P["W"]) <= 0.25 * K * K:  # nhp_cont_try_adj_loglik's density limit
                structure_steps += 1  # the handle carries the structure: this log-likelihood streamed its active buckets
            monkeypatch.setenv("NHP_ADJ_LOGLIK", "0")
            ll_window = device_loglik(ctx, d)
            monkeypatch.delenv("NHP_ADJ_LOGLIK")
            assert ll == pytest.approx(ll_window, rel=1e-12), s
            # ---- the sweep
            ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, d.h, d.h, SEED, s, float(T), _ptr(hyper), hyper.size, 1.0, 1.0))
            # ---- parents and statistics, from P_s
            par, pn = np.empty(n, np.int64), np.empty(n, np.int64)
            ctx.check(lib.nhp_cont_parents_get(ctx.h, d.h, _ptr(par), _ptr(pn)))
            opar, opn = om.resample_parents(t, nodes, synth.philox_uniform(SEED, np.arange(n, dtype=np.uint64), s))
            assert np.count_nonzero(par != opar) == 0, s
            np.testing.assert_array_equal(pn, opn)
            M0, Mn, Mnm, S1, S2 = np.empty(K), np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
            ctx.check(lib.nhp_cont_suffstats_read(ctx.h, _ptr(M0), _ptr(Mn), _ptr(Mnm), _ptr(S1), _ptr(S2)))
            ost = orc.suffstats(1 if ln else 0, t, nodes, opar, opn, K, D)
            unf = lambda v: v.reshape(K, K).T
            np.testing.assert_array_equal(M0, ost["M0"])
            np.testing.assert_array_equal(Mn, ost["Mn"])
            np.testing.assert_array_equal(unf(Mnm), ost["Mnm"])
            np.testing.assert_allclose(unf(S1), ost["S1"], rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(unf(S2), ost["S2"], rtol=1e-10, atol=1e-12)
            # ---- adjacency sweep: new lambda0, W, impulse; old A and rho
            P1, rho1 = read_params(ctx, K, ln)
            A_ref = oracle(P1, P["A"], ln, D).resample_adjacency(P["A"], np.full((K, K), rho), t, nodes, T, synth.philox_uniform(SEED, kk, s + 2 ** 40))
            np.testing.assert_array_equal(P1["A"], A_ref, err_msg=f"step {s}")
            info = nhp.adjacency_info(ctx)
            assert info["pairs"] > 0 and info["bytes_per_pair"] == bytes_per_pair
            assert (2 <= info["cluster"] <= 8) if cluster == "multi" else info["cluster"] == cluster
            # ---- Beta draw of rho (its distribution: test_adjacency_gpu.py::test_network_draw_moments)
            assert 0.0 < rho1 < 1.0
            samples.append((P1, rho1))
        assert structure_steps >= (STEPS - 1 if mode == "rewind" else 2)
        # ---- the trace holds (rho_{s+1}, P'_s) of every step
        tl0, tW, tA, tp1 = np.empty((STEPS, K)), np.empty((STEPS, K * K)), np.empty((STEPS, K * K)), np.empty((STEPS, K * K))
        trho, tp2 = np.empty(STEPS), (np.empty((STEPS, K * K)) if ln else None)
        ctx.check(lib.nhp_cont_trace_read(ctx.h, 0, STEPS, _ptr(trho), _ptr(tl0), _ptr(tW), _ptr(tA), _ptr(tp1), _ptr(tp2)))
        for s, (P1, rho1) in enumerate(samples):
            assert trho[s] == rho1
            unf = lambda v: v.reshape(K, K).T
            assert_params_equal(P1, dict(lambda0=tl0[s], W=unf(tW[s]), A=unf(tA[s]), p1=unf(tp1[s]), p2=unf(tp2[s]) if ln else None))
    finally:
        ctx.check(lib.nhp_cont_trace_free(ctx.h))
        d.free()


# ------------------------------------------------------------------------------------------------------------------------------
# One handle, two models: the cached structure was built for one impulse kind (and, with the 18-byte LogitNormal payload, one
# dtmax); a model of another kind or dtmax must not read its payload.
def build_ln_structure(data, K, pre):
    """A LogitNormal (D = 1) adjacency sweep on a fresh handle of the default context: the handle keeps its pair structure."""
    proc, _ = make_ln(K, 3, density=0.5, wmax=1.5 / K, dtmax=1.0)
    proc.network = nhp.BernoulliNetworkModel(0.3, K)
    d = proc.upload(data)
    nhp.resample_adjacency_matrix_(proc, d, u=np.random.default_rng(1).random((K, K)))
    assert nhp.adjacency_info()["bytes_per_pair"] == (18 if pre else 10)
    return d


def sweep_both(proc, om, d, data, rho, seed):
    t, nodes, T = data
    K = proc.ndims()
    proc.network = nhp.BernoulliNetworkModel(rho, K)
    A0 = proc.adjacency_matrix.copy()
    u = np.random.default_rng(seed).random((K, K))
    A_gpu = nhp.resample_adjacency_matrix_(proc, d, u=u).copy()
    return A_gpu, om.resample_adjacency(A0, np.full((K, K), rho), t, nodes, T, u)


def sampler_horizon(lam0, W, theta, n):
    """Look-back horizon of the Exponential adjacency sampler with dtmax = Inf (adj_horizon_value, cont_adjacency.cu): the
    cut-off taken over every entry with W != 0."""
    on = W != 0
    return np.log(n * np.max(np.abs(W * theta)[on]) / (1e-14 * lam0.min())) / theta[on].min()


def test_exponential_sweep_after_a_logitnormal_payload_structure():
    """(a) theta in [0.5, 2]: the cut-off lies beyond dtmax = 1, so the Exponential horizon equals the LogitNormal structure's."""
    K, n = 12, 4000
    data = synth.poisson_stream(n, K, 40.0, 31)
    d = build_ln_structure(data, K, pre=True)
    proc, om = make_exp(K, 5, density=0.5, wmax=1.5 / K, dtmax=1.0)
    A_gpu, A_ref = sweep_both(proc, om, d, data, 0.3, 2)
    np.testing.assert_array_equal(A_gpu, A_ref)
    assert nhp.adjacency_info()["bytes_per_pair"] == 10  # rebuilt for the Exponential model
    d.free()


def test_exponential_loglikelihood_after_a_logitnormal_payload_structure():
    """(b) a sparse Exponential network (dtmax = 1) evaluated on a handle that carries a LogitNormal structure."""
    K, n = 12, 4000
    t, nodes, T = data = synth.poisson_stream(n, K, 40.0, 32)
    d = build_ln_structure(data, K, pre=True)
    proc, om = make_exp(K, 6, density=0.15, wmax=2.0 / (K * 0.15), dtmax=1.0)
    assert 0 < np.count_nonzero(proc.adjacency_matrix * proc.weights.W) <= 0.25 * K * K
    ll = nhp.loglikelihood(proc, d, recursive=False)
    assert ll == pytest.approx(om.loglik(t, nodes, T, recursive=False), rel=1e-10)
    d.free()


@pytest.mark.parametrize("pre", [True, False])  # False: the lag payload, which any dtmax may read (slow_pair_ln is 0 outside (0, D))
def test_logitnormal_loglikelihood_after_dtmax_shrinks(monkeypatch, pre):
    """(c) a structure built for D = 1, then a sparse LogitNormal network with dtmax = 0.5 on the same handle: the 18-byte payload
    holds logit(dt / 1) and 1 / (dt (1 - dt)), and pairs with 0.5 < dt < 1 lie outside the new support."""
    if not pre:
        monkeypatch.setenv("NHP_ADJ_PRE", "0")
    K, n = 16, 5000
    t, nodes, T = data = synth.poisson_stream(n, K, 40.0, 33)
    d = build_ln_structure(data, K, pre=pre)
    proc, om = make_ln(K, 7, density=0.15, wmax=2.0 / (K * 0.15), dtmax=0.5)
    assert 0 < np.count_nonzero(proc.adjacency_matrix * proc.weights.W) <= 0.25 * K * K
    ll = nhp.loglikelihood(proc, d, recursive=False)
    assert ll == pytest.approx(om.loglik(t, nodes, T, recursive=False), rel=1e-10)
    d.free()


def test_exponential_moving_horizon_inside_a_logitnormal_structure():
    """(d) dtmax = Inf with theta in [50, 80]: the sampler's cut-off horizon lies in [0.5, 1], so a D = 1 structure covers it
    within the 2x reuse margin of a moving horizon."""
    K, n = 8, 3000
    data = synth.poisson_stream(n, K, 40.0, 34)
    d = build_ln_structure(data, K, pre=True)
    lam0, W, theta, A = synth.exp_params(K, 8, wmax=1.5 / K, density=0.5)
    theta = np.random.default_rng(9).uniform(50.0, 80.0, (K, K))
    assert 0.5 <= sampler_horizon(lam0, W, theta, n) <= 1.0
    proc = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.ExponentialImpulseResponse(theta), nhp.DenseWeightModel(W), A,
                                              nhp.BernoulliNetworkModel(0.3, K))
    om = orc.Cont(0, lam0, W, theta, A=A, dtmax=np.inf)
    A_gpu, A_ref = sweep_both(proc, om, d, data, 0.3, 3)
    np.testing.assert_array_equal(A_gpu, A_ref)
    d.free()


def test_logitnormal_model_on_an_exponential_structure():
    """Control: an Exponential structure (lags) of dtmax = 1, then a LogitNormal model of the same D: sweep and sparse
    log-likelihood on that handle."""
    K, n = 12, 4000
    t, nodes, T = data = synth.poisson_stream(n, K, 40.0, 35)
    ex, om_ex = make_exp(K, 5, density=0.5, wmax=1.5 / K, dtmax=1.0)
    d = ex.upload(data)
    A_gpu, A_ref = sweep_both(ex, om_ex, d, data, 0.3, 4)
    np.testing.assert_array_equal(A_gpu, A_ref)
    proc, om = make_ln(K, 7, density=0.5, wmax=1.5 / K, dtmax=1.0)
    A_gpu, A_ref = sweep_both(proc, om, d, data, 0.3, 5)
    np.testing.assert_array_equal(A_gpu, A_ref)
    sp, om_sp = make_ln(K, 8, density=0.15, wmax=2.0 / (K * 0.15), dtmax=1.0)
    assert 0 < np.count_nonzero(sp.adjacency_matrix * sp.weights.W) <= 0.25 * K * K
    assert nhp.loglikelihood(sp, d, recursive=False) == pytest.approx(om_sp.loglik(t, nodes, T, recursive=False), rel=1e-10)
    d.free()


def test_logitnormal_sweep_after_dtmax_changes():
    """Control: a D = 1 structure, then a LogitNormal sweep with dtmax = 0.5 (another horizon: the structure is rebuilt)."""
    K, n = 12, 4000
    data = synth.poisson_stream(n, K, 40.0, 36)
    d = build_ln_structure(data, K, pre=True)
    proc, om = make_ln(K, 9, density=0.5, wmax=1.5 / K, dtmax=0.5)
    A_gpu, A_ref = sweep_both(proc, om, d, data, 0.3, 6)
    np.testing.assert_array_equal(A_gpu, A_ref)
    d.free()
