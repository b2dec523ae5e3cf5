"""The host simulator with LogGaussianCox curves (nhp.rand: thinning of Poisson(max * duration) candidates for generation 0): by the
time-rescaling theorem its samples are those of the curve model, and not those of the curves' time averages or of the curves reversed
in time (tests/cont_compensator.py)."""
import numpy as np
import pytest

import cont_compensator as cc
import nhp_b200 as nhp
import synth


def skewed_curves(K, T, G, seed, spread=0.5):
    """+-50 % curves on a grid of [0, T], not symmetric in time (a sine of a power of t), so that reversing them changes them."""
    rng = np.random.default_rng(seed)
    x = np.linspace(0.0, T, G)
    s = x / T
    return x, 1.0 + spread * np.sin(2 * np.pi * (1.5 * s[None, :] ** 1.5 + rng.uniform(0.0, 1.0, (K, 1))))


def process(x, lam, kind, W, seed):
    K = lam.shape[0]
    if kind == "ln":
        _, _, mu, tau, _ = synth.ln_params(K, seed)
        imp, model = nhp.LogitNormalImpulseResponse(mu, tau, 1.0), dict(kind="ln", p1=mu, p2=tau, dtmax=1.0)
    else:
        _, _, theta, _ = synth.exp_params(K, seed)
        imp, model = nhp.ExponentialImpulseResponse(theta), dict(kind="exp", p1=theta)
    proc = nhp.ContinuousStandardHawkesProcess(nhp.LogGaussianCoxProcess(x, lam), imp, nhp.DenseWeightModel(W))
    return proc, dict(model, W=W)


@pytest.mark.parametrize("kind,wmax", [("ln", 0.0), ("ln", 0.2), ("exp", 0.2)])
def test_host_sample_rescales_to_a_unit_poisson_process(kind, wmax):
    K, T = 4, 4000.0
    x, lam = skewed_curves(K, T, 17, 1)
    W = synth.ln_params(K, 3, wmax=max(wmax, 1e-3))[1] * (wmax > 0)
    proc, model = process(x, lam, kind, W, 4)
    t, nodes, dur = nhp.rand(proc, T, np.random.default_rng(5))
    assert dur == T and np.all(np.diff(t) >= 0) and t[0] >= 0.0 and t[-1] <= T
    assert np.all(np.bincount(nodes - 1, minlength=K) > 3000)
    ok, p = cc.rescaling_holds(t, nodes, x, lam, **model)
    assert ok, p
    for control in (cc.time_averaged(x, lam, T), cc.reversed_in_time(x, lam)):
        assert not np.allclose(control, lam)
        assert cc.rescaling_pvalues(t, nodes, x, control, **model).min() < 1e-6


def test_grid_must_cover_the_duration():
    K = 2
    for x in (np.linspace(0.5, 100.0, 5), np.linspace(0.0, 90.0, 5)):
        proc, _ = process(x, np.ones((K, 5)), "ln", np.zeros((K, K)), 6)
        with pytest.raises(ValueError, match="does not cover"):
            nhp.rand(proc, 100.0, np.random.default_rng(7))
    # a grid beyond the interval on both sides is fine, and only [0, duration] holds events
    x = np.linspace(-20.0, 120.0, 8)
    proc, _ = process(x, np.ones((K, 8)), "ln", np.zeros((K, K)), 6)
    t, _, _ = nhp.rand(proc, 100.0, np.random.default_rng(7))
    assert t.size > 100 and t.min() >= 0.0 and t.max() <= 100.0
    np.testing.assert_allclose(proc.baseline.integrated_intensity_on(100.0), [100.0, 100.0])


def test_homogeneous_branch_draws_as_before():
    """The homogeneous generation 0 consumes the generator as it always did: Poisson count, then uniforms, node by node."""
    K, T = 3, 50.0
    lam0 = np.array([0.5, 1.0, 2.0])
    proc = nhp.ContinuousStandardHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.ExponentialImpulseResponse(np.ones((K, K))),
                                               nhp.DenseWeightModel(np.zeros((K, K))))
    t, nodes, _ = nhp.rand(proc, T, np.random.default_rng(8))
    rng = np.random.default_rng(8)
    ref = [np.sort(rng.uniform(0.0, T, rng.poisson(lam0[k] * T))) for k in range(K)]
    for k in range(K):
        np.testing.assert_array_equal(t[nodes == k + 1], ref[k])
