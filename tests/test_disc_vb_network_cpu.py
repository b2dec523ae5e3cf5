"""Network VB of discrete processes on the host (discrete.network_vb_targets and the state layout), with the C oracle's statistics.

The model: W | A=1 ~ Gamma(kappa, nu), W | A=0 ~ Gamma(kappa0, nu0), A ~ Bernoulli(rho), rho ~ Beta(alpha_rho, beta_rho); lambda0 and
theta as for the standard process.  One step is coordinate ascent on the collapsed bound (the responsibilities at their optimum):

  L(q) = sum_{t,c} data ln(dt (e0_c + sum_{p,b} conv ET)) - sum ln data! - sum_c E[lambda0_c] T dt - sum_{p,c} E[W] events[p] - KL(q || prior)

so the bound of successive states never decreases; a decrease means an error in the update formulas."""
import numpy as np
import pytest
from scipy.special import betaln, digamma, expit, gammaln, xlogy

import nhp_b200 as nhp
import oracle_ffi as orc
from nhp_b200 import discrete as D


def network_process(N, B, L, seed, rho=0.4):
    """A stable network process with on-link weights large enough to see and a self-link on every node."""
    rng = np.random.default_rng(seed)
    lam0 = rng.uniform(0.1, 0.2, N)
    A = (rng.random((N, N)) < rho).astype(np.float64)
    np.fill_diagonal(A, 1.0)
    W = rng.uniform(0.5, 1.0, (N, N)) * A
    W *= 0.7 / np.max(np.abs(np.linalg.eigvals(W)))
    th = rng.dirichlet(np.full(B, 2.0), (N, N))
    proc = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(th, L), nhp.DenseWeightModel(W), A,
                                          nhp.BernoulliNetworkModel(rho, N))
    return proc, A


def gamma_kl(a, b, a0, b0):
    """KL(Gamma(a, rate b) || Gamma(a0, rate b0))."""
    return (a - a0) * digamma(a) - gammaln(a) + gammaln(a0) + a0 * (np.log(b) - np.log(b0)) + a * (b0 - b) / b


def bound(q, data, conv, N, B, dt, hy):
    """The collapsed bound L(q) of the module docstring; the prior of lambda0 is Gamma(alpha0, rate 1/beta0), the rate the update's
    betav = 1/beta0 + T dt assumes (the reference's form of baselines.jl:450; with beta0 = 1 it is the model's)."""
    T = data.shape[1]
    a0, b0, kap, nu, gam, kap0, nu0, ar0, br0 = hy
    av, bv, gv, kv, nv, k0v, n0v, pv = D._network_blocks(np.asarray(q), N, B)
    e0, E = D.network_expectations(q, N, B)
    rate = dt * (e0[None, :] + np.einsum("tpb,pcb->tc", conv, E))
    ll = float(np.sum(xlogy(data.T, rate)) - np.sum(gammaln(data + 1.0)))
    EW = pv * kv / nv + (1.0 - pv) * k0v / n0v
    ll -= float(np.sum(av / bv) * T * dt + np.sum(EW * data.sum(axis=1)[:, None]))
    kl = np.sum(gamma_kl(av, bv, a0, 1.0 / b0))
    gs = gv.sum(axis=2)
    kl += np.sum(gammaln(gs) - gammaln(gv).sum(axis=2) - gammaln(B * gam) + B * gammaln(gam) + ((gv - gam) * (digamma(gv) - digamma(gs)[:, :, None])).sum(axis=2))
    ar, br = q[-2], q[-1]
    eln1, eln0 = digamma(ar) - digamma(ar + br), digamma(br) - digamma(ar + br)
    kl += np.sum(xlogy(pv, pv) - pv * eln1 + pv * gamma_kl(kv, nv, kap, nu))
    kl += np.sum(xlogy(1.0 - pv, 1.0 - pv) - (1.0 - pv) * eln0 + (1.0 - pv) * gamma_kl(k0v, n0v, kap0, nu0))
    kl += betaln(ar0, br0) - betaln(ar, br) + (ar - ar0) * digamma(ar) + (br - br0) * digamma(br) + (ar0 - ar + br0 - br) * digamma(ar + br)
    return ll - float(kl)


def host_step(q, data, conv, N, B, dt, hy, events):
    e0, E = D.network_expectations(q, N, B)
    st = orc.disc_vb_stats(data, conv, e0, E)
    return D.network_vb_targets(q, st, events, data.shape[1], dt, hy, 1.0)


@pytest.mark.parametrize("pv0", [None, 1.0], ids=["default_start", "all_links_start"])
def test_bound_never_decreases(pv0):
    """N = 5, T = 4000, B = 3, L = 5, beta0 = 1, 40 steps: the bound rises or stays within 1e-9 relative (measured: the largest fall is
    4e-16 relative, rounding), from the default start (pv = rho, kappa0v / nu0v = the spike's hyper-parameters) and from pv = 1."""
    N, T, B, L = 5, 4000, 3, 5
    proc, A = network_process(N, B, L, seed=3)
    data = D.rand(proc, T, np.random.default_rng(11))
    conv = orc.disc_convolve(data, orc.disc_basis(L, B))
    hy = D._network_hyper(proc)
    if pv0 is not None:
        proc.network.pv = np.full((N, N), pv0)
    q = D.network_variational_params(proc)
    events = data.sum(axis=1).astype(np.float64)
    L_prev = bound(q, data, conv, N, B, proc.dt, hy)
    first = L_prev
    for k in range(40):
        q = host_step(q, data, conv, N, B, proc.dt, hy, events)
        Lk = bound(q, data, conv, N, B, proc.dt, hy)
        assert Lk >= L_prev - 1e-9 * abs(L_prev), (k, Lk, L_prev)
        L_prev = Lk
    assert L_prev > first
    found = int(np.sum((D.network_posterior_means(q, N, B)["A"] > 0.5) == (A > 0.5)))
    print(f"bound {first:.6g} -> {L_prev:.6g}; entries of A recovered {found}/{N * N}")


def test_links_are_recovered_from_the_all_links_start():
    """The data of test_bound_never_decreases from pv = 1: after 40 steps pv > 0.5 matches at least 21 of the 25 entries of the true A
    (measured 22, at a bound of -16832).  From the default start pv = rho the same steps end at a lower optimum (bound -17489, every
    pv near 0, 12 of 25): there the first E[ln W] is mostly the spike's, psi(kappa0) - ln nu0, so the first responsibilities give the
    links almost no events and the slab loses every link at once."""
    N, T, B, L = 5, 4000, 3, 5
    proc, A = network_process(N, B, L, seed=3)
    data = D.rand(proc, T, np.random.default_rng(11))
    conv = orc.disc_convolve(data, orc.disc_basis(L, B))
    hy = D._network_hyper(proc)
    proc.network.pv = np.ones((N, N))
    q = D.network_variational_params(proc)
    events = data.sum(axis=1).astype(np.float64)
    for _ in range(40):
        q = host_step(q, data, conv, N, B, proc.dt, hy, events)
    found = int(np.sum((D.network_posterior_means(q, N, B)["A"] > 0.5) == (A > 0.5)))
    assert found >= 21, found


def test_spike_equal_to_slab_is_the_standard_update():
    """kappa0 = kappa, nu0 = nu and kappa0v = kappav, nu0v = nuv: the standard block of q* is the standard update of the same statistics
    (rtol 1e-14; measured 0), kappa0v* = kappav*, nu0v* = nuv*, and pv* = expit(psi(alpharhov) - psi(betarhov)) (the two brackets cancel
    up to rounding of their sizes: rtol 1e-12, measured 2e-15)."""
    N, T, B, L = 4, 3000, 3, 4
    proc, _ = network_process(N, B, L, seed=5)
    proc.weights.kappa, proc.weights.nu = 1.5, 2.0
    proc.weights.kappa0, proc.weights.nu0 = 1.5, 2.0
    data = D.rand(proc, T, np.random.default_rng(2))
    conv = orc.disc_convolve(data, orc.disc_basis(L, B))
    rng = np.random.default_rng(7)
    q = D.network_variational_params(proc)
    NN, o = N * N, 2 * N + N * N * B
    q[:o + 2 * NN] = rng.uniform(0.5, 5.0, o + 2 * NN)
    q[o + 2 * NN:o + 4 * NN] = q[o:o + 2 * NN]
    q[o + 4 * NN:o + 5 * NN] = rng.uniform(0.0, 1.0, NN)
    q[-2:] = [2.5, 7.0]
    hy = D._network_hyper(proc)
    e0, E = D.network_expectations(q, N, B)
    st = orc.disc_vb_stats(data, conv, e0, E)
    events = data.sum(axis=1).astype(np.float64)
    qs = D.network_vb_targets(q, st, events, T, proc.dt, hy, 1.0)
    std = np.concatenate([hy[0] + st["alpha_sum"], 1.0 / hy[1] + T * proc.dt * np.ones(N), (hy[4] + st["gamma_sum"]).transpose(2, 1, 0).ravel(),
                          (hy[2] + st["kappa_sum"]).T.ravel(), (hy[3] + st["nu_sum"]).T.ravel()])
    np.testing.assert_allclose(qs[:o + 2 * NN], std, rtol=1e-14)
    np.testing.assert_array_equal(qs[o + 2 * NN:o + 4 * NN], qs[o:o + 2 * NN])
    p = qs[o + 4 * NN:o + 5 * NN]
    np.testing.assert_allclose(p, expit(digamma(2.5) - digamma(7.0)), rtol=1e-12)
    np.testing.assert_allclose(qs[-2:], [hy[7] + p.sum(), hy[8] + NN - p.sum()], rtol=1e-15)
    # the standard expectations too: with kappa0v = kappav the mixture E[ln W] is psi(kappav) - ln nuv
    av, bv, gv, kv, nv = q[:N], q[N:2 * N], q[2 * N:o].reshape(B, N, N).transpose(2, 1, 0), q[o:o + NN].reshape(N, N).T, q[o + NN:o + 2 * NN].reshape(N, N).T
    E_std = np.exp((digamma(gv) - digamma(gv.sum(axis=2, keepdims=True))) + (digamma(kv) - np.log(nv))[:, :, None])
    np.testing.assert_allclose(E, E_std, rtol=1e-14)
    np.testing.assert_array_equal(e0, np.exp(digamma(av) - np.log(bv)))


def test_window_scale():
    """The targets of a window scale G, E and alpha_sum by s and leave betav and the link count N^2 of q(rho) unscaled."""
    N, B = 3, 2
    rng = np.random.default_rng(1)
    st = dict(alpha_sum=rng.uniform(1, 5, N), kappa_sum=rng.uniform(0, 9, (N, N)), gamma_sum=rng.uniform(0, 3, (N, N, B)))
    hy = np.array([1.0, 1.0, 1.0, 1.0, 1.0, 0.1, 10.0, 1.0, 1.0])
    q = np.concatenate([np.ones(2 * N + N * N * (B + 2)), np.full(2 * N * N, 0.5), np.full(N * N, 0.3), [1.0, 1.0]])
    ev = rng.uniform(10, 20, N)
    a = D.network_vb_targets(q, st, ev, 100, 0.5, hy, 4.0)
    st4 = {k: 4.0 * v for k, v in st.items()}
    b = D.network_vb_targets(q, st4, 4.0 * ev, 100, 0.5, hy, 1.0)
    np.testing.assert_allclose(a, b, rtol=1e-15)
    assert a[N] == 1.0 + 100 * 0.5
    p = a[-2 - N * N:-2]
    assert a[-2] == 1.0 + p.sum() and a[-1] == (1.0 + N * N) - p.sum()


def test_layout_round_trip_and_defaults():
    """Missing factors start as documented, adjacency_matrix / W / rho stay as they are, and state -> process -> state is exact."""
    N, B, L = 4, 3, 4
    proc, A = network_process(N, B, L, seed=9, rho=0.3)
    W0 = proc.weights.W.copy()
    q = D.network_variational_params(proc)
    NN, o = N * N, 2 * N + N * N * B
    assert q.size == 2 * N + N * N * (B + 5) + 2
    np.testing.assert_array_equal(q[o:o + 2 * NN], 1.0)
    np.testing.assert_array_equal(q[o + 2 * NN:o + 3 * NN], 0.1)
    np.testing.assert_array_equal(q[o + 3 * NN:o + 4 * NN], 10.0)
    np.testing.assert_array_equal(q[o + 4 * NN:o + 5 * NN], 0.3)
    np.testing.assert_array_equal(q[-2:], [1.0, 1.0])
    r = np.random.default_rng(4).uniform(0.01, 3.0, q.size)
    r[o + 4 * NN:o + 5 * NN] = np.random.default_rng(5).uniform(0.0, 1.0, NN)
    D.set_network_variational_params_(proc, r)
    np.testing.assert_array_equal(D.network_variational_params(proc), r)
    assert proc.network.pv[1, 2] == r[o + 4 * NN + 1 + N * 2]  # [p + N c]
    np.testing.assert_array_equal(proc.adjacency_matrix, A)
    np.testing.assert_array_equal(proc.weights.W, W0)
    assert proc.network.rho == 0.3
    with pytest.raises(ValueError):
        D.set_network_variational_params_(proc, r[:-1])
    m = D.network_posterior_means(r, N, B)
    k = o + 4 * NN + 1 + N * 2
    pv = r[k]
    assert m["A"][1, 2] == pv
    assert m["W"][1, 2] == pytest.approx(pv * r[k - 4 * NN] / r[k - 3 * NN] + (1 - pv) * r[k - 2 * NN] / r[k - NN], rel=1e-15)
    assert m["rho"] == pytest.approx(r[-2] / (r[-2] + r[-1]), rel=1e-15)
    np.testing.assert_allclose(m["theta"].sum(axis=2), 1.0, rtol=1e-15)


def test_refusals_come_before_any_device_call(monkeypatch):
    """A standard process, a DenseNetworkModel, a kappa0 / nu0 that is not positive and finite, and bad schedule arguments raise
    ValueError without a context: the context factory is not reached."""
    import nhp_b200
    from nhp_b200 import core

    def no_device(*a, **k):
        raise AssertionError("a device context was requested")

    monkeypatch.setattr(core, "default_context", no_device)
    monkeypatch.setattr(D, "default_context", no_device)
    monkeypatch.setattr(nhp_b200, "default_context", no_device, raising=False)
    N, B = 3, 2
    rng = np.random.default_rng(0)
    theta = rng.dirichlet(np.ones(B), (N, N))
    data = rng.poisson(0.1, (N, 100)).astype(np.int64)
    mk = lambda: (D.DiscreteHomogeneousProcess(np.full(N, 0.1)), D.DiscreteGaussianImpulseResponse(theta, 3), nhp_b200.DenseWeightModel(np.full((N, N), 0.1)))
    std = D.DiscreteStandardHawkesProcess(*mk())
    dense = D.DiscreteNetworkHawkesProcess(*mk(), np.ones((N, N)), nhp_b200.DenseNetworkModel(N) if _dense_takes_n() else nhp_b200.DenseNetworkModel())
    net = D.DiscreteNetworkHawkesProcess(*mk(), np.ones((N, N)), nhp_b200.BernoulliNetworkModel(0.5, N))
    runs = (lambda p, **kw: D.network_vb_device_(p, data, 5, **kw), lambda p, **kw: D.network_svi_device_(p, data, 5, 10, **kw),
            lambda p, **kw: D.network_update_(p, data, **kw))
    for run in runs:
        for p, kw in ((std, {}), (dense, {}), (net, dict(kappa0=0.0)), (net, dict(nu0=-1.0)), (net, dict(kappa0=float("nan"))),
                      (net, dict(nu0=float("inf")))):
            with pytest.raises(ValueError):
                run(p, **kw)
    for kw in (dict(batch_bins=0), dict(batch_bins=101), dict(batch_bins=10, kappa=2.0), dict(batch_bins=10, tau0=-1.0)):
        with pytest.raises(ValueError):
            D.network_svi_device_(net, data, 5, **kw)
    assert not hasattr(net.network, "pv")  # nothing was initialised


def _dense_takes_n():
    import inspect
    return len(inspect.signature(nhp.DenseNetworkModel.__init__).parameters) > 1
