"""discrete.svi_schedule: the windows and step sizes of stochastic VI, computed on the host before any device call."""
import numpy as np
import pytest

from nhp_b200 import discrete as D


def test_deterministic_in_the_seed():
    a, sa = D.svi_schedule(1000, 50, 10, seed=3)
    b, sb = D.svi_schedule(1000, 50, 10, seed=3)
    c, _ = D.svi_schedule(1000, 50, 10, seed=4)
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(sa, sb)
    assert not np.array_equal(a, c)
    assert a.dtype == np.int64 and a.shape == sa.shape == (50,)
    np.testing.assert_array_equal(a, np.random.default_rng(3).integers(0, 1000, size=50, dtype=np.int64))


def test_step_size_formula():
    _, s = D.svi_schedule(100, 6, 5, tau0=2.5, kappa=0.6)
    np.testing.assert_array_equal(s, (np.arange(1, 7) + 2.5) ** -0.6)
    _, s = D.svi_schedule(100, 4, 5, tau0=0.0, kappa=1.0)
    np.testing.assert_array_equal(s, 1.0 / np.arange(1, 5))  # tau0 = 0: the first step takes the target whole
    assert np.all((s > 0) & (s <= 1))
    assert np.all(np.diff(D.svi_schedule(100, 30, 5)[1]) < 0)


def test_windows_cover_the_series_uniformly_and_wrap():
    T, n, K = 50, 20, 20000
    t, _ = D.svi_schedule(T, K, n, seed=1)
    assert t.min() >= 0 and t.max() < T
    assert np.any(t + n > T)  # windows that wrap around the end occur
    hits = np.zeros(T)
    for tb in t:
        hits[(tb + np.arange(n)) % T] += 1
    # with wrapping every bin is in a window with probability n / T: 8000 expected hits, binomial sd 69
    assert np.all(np.abs(hits - K * n / T) < 6 * np.sqrt(K * n / T * (1 - n / T)))


def test_empty_schedule():
    t, s = D.svi_schedule(10, 0, 1)
    assert t.size == 0 and s.size == 0


@pytest.mark.parametrize("kw", [dict(T=0, nsteps=1, batch_bins=1), dict(T=10, nsteps=1, batch_bins=0), dict(T=10, nsteps=1, batch_bins=11),
                                dict(T=10, nsteps=1, batch_bins=2, kappa=0.5), dict(T=10, nsteps=1, batch_bins=2, kappa=1.01),
                                dict(T=10, nsteps=1, batch_bins=2, kappa=float("nan")), dict(T=10, nsteps=1, batch_bins=2, tau0=-0.1),
                                dict(T=10, nsteps=1, batch_bins=2, tau0=float("nan")), dict(T=10, nsteps=-1, batch_bins=2),
                                dict(T=10, nsteps=1.5, batch_bins=2), dict(T=10, nsteps=1, batch_bins=2.5)],
                         ids=["T0", "batch0", "batch_gt_T", "kappa_half", "kappa_gt1", "kappa_nan", "tau0_neg", "tau0_nan", "nsteps_neg",
                              "nsteps_frac", "batch_frac"])
def test_refusals(kw):
    with pytest.raises(ValueError):
        D.svi_schedule(**kw)


def test_svi_device_refuses_before_any_device_call(monkeypatch):
    """Bad schedule arguments and a network process raise ValueError without a context: the context factory is not reached."""
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
    std = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(np.full(N, 0.1)), D.DiscreteGaussianImpulseResponse(theta, 3),
                                          nhp_b200.DenseWeightModel(np.full((N, N), 0.1)))
    data = rng.poisson(0.1, (N, 100)).astype(np.int64)
    for kw in (dict(batch_bins=0), dict(batch_bins=101), dict(batch_bins=10, kappa=2.0), dict(batch_bins=10, tau0=-1.0)):
        with pytest.raises(ValueError):
            D.svi_device_(std, data, 5, **kw)
    net = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(np.full(N, 0.1)), D.DiscreteGaussianImpulseResponse(theta, 3),
                                         nhp_b200.DenseWeightModel(np.full((N, N), 0.1)), np.ones((N, N)), nhp_b200.BernoulliNetworkModel(0.5, N))
    with pytest.raises(ValueError, match="Q10"):
        D.svi_device_(net, data, 5, 10)
