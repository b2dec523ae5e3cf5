"""Mean-field VB of a continuous network Hawkes process with a variational adjacency matrix, on the device, then a Gibbs chain that
starts from the VB point estimate."""
import _path  # noqa: F401
import numpy as np

import nhp_b200 as nhp
from nhp_b200 import continuous as C

rng = np.random.default_rng(0)
K = 6
A = np.zeros(K * K)
A[rng.permutation(K * K)[:12]] = 1.0
A = A.reshape(K, K)
W = rng.uniform(0.1, 0.25, (K, K))
process = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(rng.uniform(0.5, 1.0, K)),
                                             nhp.LogitNormalImpulseResponse(rng.normal(0.0, 0.5, (K, K)), rng.uniform(1.0, 3.0, (K, K)), 1.0),
                                             nhp.DenseWeightModel(W), A, nhp.BernoulliNetworkModel(1.0 / 3.0, K))
d = nhp.rand_device(process, 20000.0, seed=0)
states = C.network_vb_device_(process, d, max_steps=5000, rtol=1e-8, trace=False)  # from every link on
m = C.network_posterior_means(process, states[-1])
print(d.n, "events; q(A = 1) > 0.5 matches the true A on", int(np.sum((m["A"] > 0.5) == (A > 0.5))), "of", K * K, "entries")
print("q(A = 1) =\n", np.round(m["A"], 3))
print("slab means of W on the true links:", np.round(m["W_slab"][A > 0.5], 3), "truth:", np.round(W[A > 0.5], 3))
print("E[rho] =", round(m["rho"], 3), "(the process now holds rho, pv and the point estimate)")
chain = nhp.mcmc_device_(process, d, nsteps=200, seed=1)  # a Gibbs chain from the VB point estimate
# the chain also switches on links whose sampled weight is negligible (their adjacency odds are those of rho)
A_last, W_last = process.adjacency_matrix, process.weights.W
print("chain: links in the last sample", int(A_last.sum()), "of which with a weight above 0.01:", int(np.sum(A_last * W_last > 0.01)))
