"""Small run through every kernel family (for compute-sanitizer memcheck): sizes of a few thousand events."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "networkhawkesprocesses.jl_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import nhp_b200 as nhp  # noqa: E402
from nhp_b200 import discrete as D  # noqa: E402
import synth  # noqa: E402


def cont(kind, K, n, rate, density, env):
    for k, v in env.items():
        os.environ[k] = v
    t, nodes, T = synth.poisson_stream(n, K, rate, 3)
    if kind == "ln":
        lam0, W, mu, tau, A = synth.ln_params(K, 4, density=density, wmax=0.3 / K)
        imp = nhp.LogitNormalImpulseResponse(mu, tau, 1.0)
    else:
        lam0, W, th, A = synth.exp_params(K, 4, density=density, wmax=0.3 / K)
        imp = nhp.ExponentialImpulseResponse(th, dtmax=1.5)
    base, wts = nhp.HomogeneousProcess(lam0), nhp.DenseWeightModel(W)
    proc = nhp.ContinuousStandardHawkesProcess(base, imp, wts) if A is None else nhp.ContinuousNetworkHawkesProcess(base, imp, wts, A, nhp.BernoulliNetworkModel(0.3, K))
    d = proc.upload((t, nodes, T))
    ll = nhp.loglikelihood(proc, d, recursive=False)
    nhp.event_intensity(proc, d)
    nhp.resample_parents(proc, d, seed=1, counter=2, with_loglik=True)
    nhp.sufficient_statistics(proc, d)
    nhp.intensity(proc, d, np.linspace(0, T, 50))
    if A is not None:
        nhp.resample_adjacency_matrix_(proc, d, seed=3)
    for k in env:
        os.environ.pop(k, None)
    return ll


print(cont("ln", 20, 3000, 60.0, None, {}))
print(cont("exp", 20, 3000, 60.0, None, {"NHP_G": "32"}))
print(cont("ln", 40, 3000, 60.0, 0.1, {"NHP_SPARSE": "1"}))
print(cont("exp", 1100, 3000, 60.0, 0.1, {"NHP_SPARSE": "1"}))
print(cont("ln", 12, 3000, 60.0, None, {"NHP_CHILD": "1", "NHP_SPARSE": "0"}))
print(cont("ln", 6, 4000, 3000.0, 0.3, {"NHP_SPARSE": "1"}))  # windows beyond the staging buffer
rng = np.random.default_rng(0)
N, T, B, L = 20, 700, 4, 6
theta = rng.dirichlet(np.ones(B), (N, N))
A = (rng.random((N, N)) < 0.5).astype(float)
proc = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(np.full(N, 0.1)), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(rng.uniform(0, 0.02, (N, N))),
                                      A, nhp.BernoulliNetworkModel(0.4, N))
data = rng.poisson(0.1, (N, T))
dd = proc.upload(data)
D.convolve(proc, dd)
print(D.loglikelihood(proc, dd), D.intensity(proc, dd).shape)
for w in ("1", "0"):
    os.environ["NHP_DISC_WARP"] = w
    D.resample_parents(proc, dd, seed=1)
    D.vb_statistics(proc, dd, np.ones(N), np.full((N, N, B), 0.1))
D.resample_adjacency_matrix_(proc, dd, seed=2)
print("all kernels ran")
