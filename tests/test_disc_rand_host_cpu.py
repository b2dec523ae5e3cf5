"""CPU test of the host discrete simulator (discrete.rand, discrete.jl:20-38), the independent check of the device one: its samples
have the conditional law of the likelihood, with lambda from the C oracle's discrete convolution and intensity."""
import numpy as np

import nhp_b200 as nhp
import oracle_ffi as orc
from disc_rand_law import law_holds
from nhp_b200 import discrete as D


def test_host_sample_has_the_conditional_law_of_the_likelihood():
    """N = 4, T = 1e5, network process with mixed theta (measured: KS p 0.47, z -0.41, per-node |z| <= 1.7); the intensity of
    W x 1.1 fails (z -76)."""
    N, B, L = 4, 3, 12
    rng = np.random.default_rng(1)
    lam0 = rng.uniform(0.2, 0.4, N)
    A = (rng.random((N, N)) < 0.6).astype(np.float64)
    np.fill_diagonal(A, 1.0)
    W = rng.uniform(0.5, 1.0, (N, N)) * A
    W *= 0.85 / np.max(np.abs(np.linalg.eigvals(W)))
    th = rng.dirichlet(np.ones(B), (N, N))
    proc = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(th, L), nhp.DenseWeightModel(W), A,
                                          nhp.BernoulliNetworkModel(0.5, N))
    data = D.rand(proc, 100000, np.random.default_rng(5))
    assert data.shape == (N, 100000) and data.dtype == np.int64 and data.sum() > 300000
    conv = orc.disc_convolve(data, orc.disc_basis(L, B))
    ok, st = law_holds(data, orc.Disc(lam0, W, th, A=A).intensity(conv))
    assert ok, st
    bad, st = law_holds(data, orc.Disc(lam0, W * 1.1, th, A=A).intensity(conv))
    assert not bad and st[1] < -20, st


def test_host_sample_is_a_function_of_the_generator():
    proc = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess([0.1, 0.2]), D.DiscreteGaussianImpulseResponse(np.full((2, 2, 2), 0.5), 4),
                                           nhp.DenseWeightModel(np.full((2, 2), 0.2)))
    a, b = D.rand(proc, 500, np.random.default_rng(3)), D.rand(proc, 500, np.random.default_rng(3))
    assert np.array_equal(a, b) and a[:, 0].sum() <= a.sum()
