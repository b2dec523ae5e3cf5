"""CPU checks of tests/grid_reference.py, the NumPy statement of the continuous formulas with a per-event baseline that the GPU
tests of grid baselines compare against: without curves it must reproduce the C oracle, with curves a plain event-by-event loop
over the reference's definitions."""
import numpy as np
import pytest

import grid_reference as gr
import oracle_ffi as orc
import synth


def _models(kind, K, seed, density, dtmax):
    if kind == 1:
        lam0, W, mu, tau, A = synth.ln_params(K, seed, wmax=1.5 / K, density=density)
        return lam0, W, mu, tau, A, orc.Cont(1, lam0, W, mu, tau, A=A, dtmax=dtmax)
    lam0, W, theta, A = synth.exp_params(K, seed, wmax=1.5 / K, density=density)
    return lam0, W, theta, None, A, orc.Cont(0, lam0, W, theta, A=A, dtmax=dtmax)


def _curves(K, G, T, seed):
    rng = np.random.default_rng(seed)
    x = np.linspace(0.0, T, G)
    return x, np.exp(rng.normal(0.0, 0.5, (K, 1)) + 0.8 * np.sin(rng.uniform(0.5, 3.0, (K, 1)) * x[None, :] / T * 6.0 + rng.uniform(0, 6, (K, 1))))


@pytest.mark.parametrize("kind,dtmax,density", [(1, 1.0, 0.5), (0, 1.0, None), (0, np.inf, 0.6)])
def test_without_curves_the_statement_is_the_oracle(kind, dtmax, density):
    K, n = 5, 700
    t, nodes, T = synth.poisson_stream(n, K, 15.0, 3)
    lam0, W, p1, p2, A, om = _models(kind, K, 4, density, dtmax)
    ref = gr.Model(kind, lam0, W, p1, p2, A=A, dtmax=dtmax)
    np.testing.assert_allclose(ref.event_intensity(t, nodes), om.event_intensity(t, nodes), rtol=1e-12)
    assert ref.loglik(t, nodes, T) == pytest.approx(om.loglik(t, nodes, T, recursive=False), rel=1e-12)
    tq = np.linspace(0.0, T, 23)
    np.testing.assert_allclose(ref.intensity(t, nodes, tq), om.intensity(t, nodes, tq), rtol=1e-12)
    if A is not None:
        rho = np.full((K, K), 0.4)
        for rep in range(3):
            u = np.random.default_rng(10 + rep).random((K, K))
            np.testing.assert_array_equal(ref.resample_adjacency(A, rho, t, nodes, T, u), om.resample_adjacency(A, rho, t, nodes, T, u))


def test_interpolation_is_the_device_form():
    x = np.array([0.0, 0.5, 2.0, 3.0])
    y = np.array([1.0, 3.0, 0.5, 2.0])
    t = np.array([0.0, 0.25, 0.5, 1.9, 2.0, 2.999, 3.0])
    np.testing.assert_allclose(gr.interp(x, y, t), np.interp(t, x, y), rtol=1e-15)
    assert gr.interp(x, y, np.array([3.0]))[0] == 2.0 and gr.interp(x, y, np.array([0.5]))[0] == 3.0
    with pytest.raises(ValueError):
        gr.interp(x, y, np.array([3.0 + 1e-12]))
    assert gr.trapezoid(x, y) == pytest.approx(np.sum(0.5 * (y[1:] + y[:-1]) * np.diff(x)), rel=1e-15)


def _loop_intensity(m, t, nodes, i, c, base):
    """total_intensity (continuous.jl:391-405) of child node c (0-based) for event index i, one predecessor at a time"""
    lam = base
    for j in range(i - 1, -1, -1):
        if not (t[j] > t[i] - m.dtmax):
            break
        p = nodes[j] - 1
        a = 1.0 if m.A is None else m.A[p, c]
        lam += a * m.W[p, c] * float(m.pdf(p, c, t[i] - t[j]))
    return lam


@pytest.mark.parametrize("kind,dtmax", [(1, 1.0), (0, np.inf)])
def test_with_curves_the_statement_is_the_event_loop(kind, dtmax):
    K, n = 4, 300
    t, nodes, T = synth.poisson_stream(n, K, 12.0, 5)
    lam0, W, p1, p2, A, _ = _models(kind, K, 6, 0.6, dtmax)
    x, lam = _curves(K, 9, T, 7)
    ref = gr.Model(kind, lam0, W, p1, p2, A=A, dtmax=dtmax, x=x, lam=lam)
    want = np.array([_loop_intensity(ref, t, nodes, i, nodes[i] - 1, np.interp(t[i], x, lam[nodes[i] - 1])) for i in range(n)])
    np.testing.assert_allclose(ref.event_intensity(t, nodes), want, rtol=1e-12)
    comp = sum(float(np.sum((A * W)[nodes[i] - 1])) for i in range(n))
    trapz = float(np.sum(0.5 * (lam[:, 1:] + lam[:, :-1]) * np.diff(x)[None, :]))
    assert ref.loglik(t, nodes, T) == pytest.approx(float(np.sum(np.log(want))) - trapz - comp, rel=1e-12)
    tq = np.linspace(0.0, T, 11)
    got = ref.intensity(t, nodes, tq)
    for q, t0 in enumerate(tq):
        for c in range(K):
            s = np.interp(t0, x, lam[c])
            for j in range(n):
                if t0 - dtmax < t[j] < t0:
                    p = nodes[j] - 1
                    s += A[p, c] * W[p, c] * float(ref.pdf(p, c, t0 - t[j]))
            assert got[q, c] == pytest.approx(s, rel=1e-12)


def test_adjacency_statement_with_curves_is_the_full_conditional():
    """Each step against ll0 / ll1 summed event by event (continuous.jl:477-483) with the curves as the baseline; constant curves
    equal to lambda0 give the oracle's homogeneous sweep."""
    K, n, rho = 4, 260, 0.45
    t, nodes, T = synth.poisson_stream(n, K, 10.0, 8)
    lam0, W, p1, p2, A0, om = _models(1, K, 9, 0.5, 1.0)
    x, lam = _curves(K, 7, T, 10)
    ref = gr.Model(1, lam0, W, p1, p2, A=A0, dtmax=1.0, x=x, lam=lam)
    u = np.random.default_rng(11).random((K, K))
    got = ref.resample_adjacency(A0, rho, t, nodes, T, u)
    A = A0.copy()
    counts = np.bincount(nodes - 1, minlength=K)
    for c in range(K):
        ev = [i for i in range(1, n) if nodes[i] == c + 1]
        for p in range(K):
            ll = []
            for a in (0.0, 1.0):
                A[p, c] = a
                ref.A = A
                s = sum(np.log(_loop_intensity(ref, t, nodes, i, c, np.interp(t[i], x, lam[c]))) for i in ev)
                ll.append(s - gr.trapezoid(x, lam[c]) - float(np.sum(A[:, c] * W[:, c] * counts)))
            l0, l1 = ll[0] + np.log(1.0 - rho), ll[1] + np.log(rho)
            A[p, c] = 1.0 if u[p, c] <= 1.0 / (1.0 + np.exp(l0 - l1)) else 0.0
    np.testing.assert_array_equal(got, A)
    flat = gr.Model(1, lam0, W, p1, p2, A=A0, dtmax=1.0, x=x, lam=np.repeat(lam0[:, None], x.size, axis=1))
    np.testing.assert_array_equal(flat.resample_adjacency(A0, rho, t, nodes, T, u), om.resample_adjacency(A0, np.full((K, K), rho), t, nodes, T, u))
