"""Mean-field VB of a discrete Gaussian-basis standard Hawkes process (examples/discrete-gaussian-standard-hawkes-vb.jl)."""
import _path  # noqa: F401
import numpy as np

import nhp_b200 as nhp
from nhp_b200 import discrete as D

rng = np.random.default_rng(0)
N, T, B, L = 2, 20000, 3, 4
theta = rng.dirichlet(np.ones(B), (N, N))
W = np.array([[0.2, 0.1], [0.1, 0.2]])
process = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(np.array([0.1, 0.2])), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W))
d = D.rand_device(process, T, seed=0)  # rand(process, T) (discrete.jl:20-38) on the device; the sample stays there
print("events:", d.events_count(), " loglikelihood:", D.loglikelihood(process, d))
D.vb_(process, d, max_steps=50)
b, w, i = process.baseline, process.weights, process.impulses
print("E[lambda] =", b.alphav / b.betav, " truth", [0.1, 0.2])        # posterior means as the reference example prints them
print("E[W] =\n", w.kappav / w.nuv, "\ntruth\n", W)
