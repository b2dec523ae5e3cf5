"""Mean-field VB of a discrete network Hawkes process with a variational adjacency matrix, on the device."""
import _path  # noqa: F401
import numpy as np

import nhp_b200 as nhp
from nhp_b200 import discrete as D

rng = np.random.default_rng(0)
N, T, B, L = 6, 40000, 3, 5
A = (rng.random((N, N)) < 0.3).astype(np.float64)
np.fill_diagonal(A, 1.0)
W = rng.uniform(0.5, 1.0, (N, N)) * A
W *= 0.7 / np.max(np.abs(np.linalg.eigvals(W)))
theta = rng.dirichlet(np.full(B, 2.0), (N, N))
process = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(np.full(N, 0.1)), D.DiscreteGaussianImpulseResponse(theta, L),
                                         nhp.DenseWeightModel(W), A, nhp.BernoulliNetworkModel(0.3, N))
d = D.rand_device(process, T, seed=0)
process.network.pv = np.ones((N, N))  # start with every link on: from pv = rho the first steps switch every link off
trace = D.network_vb_device_(process, d, max_steps=100)
m = D.network_posterior_means(trace[-1], N, process.impulses.nbasis())
print("q(A = 1) > 0.5 matches the true A on", int(np.sum((m["A"] > 0.5) == (A > 0.5))), "of", N * N, "entries")
print("E[W] =\n", np.round(m["W"], 3), "\ntruth\n", np.round(W, 3))
print("E[rho] =", round(m["rho"], 3))
