"""The discrete device simulator at config 3: nhp_disc_rand against the host upload of a matrix of the same shape, and one Gibbs sweep
and one VB step on the true sample next to the Poisson surrogate the other discrete tools use.

    python tools/disc_rand_bench.py [--reps 5] [--out FILE]

Model: bench.py's config 3 (N = 200, T = 1e6 bins, B = 6, L = 12, spectral radius 0.5, rho = 0.1; the parameters of
disc_chain_bench.config3).  Every figure is the median over `reps` timed calls after one warm-up call, timed on the host clock around
work that ends in a device synchronisation:

  rand            nhp_disc_rand of the network process: the whole sample, from the parameters to a ready (unconvolved) count handle
  upload          nhp_disc_upload of the N x T Int64 matrix from host memory: today's way to get such data onto the device (1.6 GB
                  over PCIe, then the same handle build)
  gibbs_sweep     one nhp_disc_gibbs_sweep (network process, rho ~ Beta(1, 1)), each from the config-3 parameters
  vb_step         one nhp_disc_vb_step (the standard process of the same W and theta), chained from the all-ones state
the last two on the true sample ("true") and on rng.poisson(0.04, (N, T)) ("poisson").

The card's name and power limit are read in the same process.  One JSON object goes to stdout (and to --out)."""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "networkhawkesprocesses.jl_b200"))
sys.path.insert(0, HERE)
from disc_chain_bench import card, config3  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 1:
        ap.error("--reps must be positive")
    import nhp_b200 as nhp
    from nhp_b200 import discrete as D
    from nhp_b200.core import _ptr
    lam0, W, A, theta, surrogate, L = config3()
    N, B, T = lam0.size, theta.shape[2], surrogate.shape[1]
    net = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W), A,
                                         nhp.BernoulliNetworkModel(0.1, N))
    std = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W))
    ctx = net._ctx()
    lib = ctx.lib
    sync = lambda: ctx.check(lib.nhp_disc_params_get(ctx.h, None, None, None, None))  # synchronises the context's stream

    def timed(fn, setup=None):
        out = []
        for r in range(args.reps + 1):  # r = 0: warm-up
            if setup:
                setup()
            sync()
            t0 = time.perf_counter()
            fn()
            sync()
            if r > 0:
                out.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(out)), out

    res = {"tool": "disc_rand_bench", "card": card(), "workload": "config 3: discrete Gaussian network Hawkes, N=200, T=1e6 bins, B=6, L=12, "
           "spectral radius 0.5, rho=0.1", "reps": args.reps, "ms_median": {}, "ms": {}}

    def record(name, m):
        res["ms_median"][name], res["ms"][name] = m

    net._push(ctx)
    handles = []

    def simulate():
        handles.append(D.rand_device(net, T, seed=len(handles)))

    record("rand", timed(simulate))
    true = handles[-1]
    res["events_true"] = true.events_count()
    res["events_poisson"] = int(surrogate.sum())
    res["same_sample_for_same_seed"] = bool(np.array_equal(D.rand_device(net, T, seed=len(handles) - 1).download(), true.download()))
    del handles[:-1]
    host = true.download()
    uploaded = []
    record("upload", timed(lambda: uploaded.append(D.DiscreteData(ctx, host)), setup=lambda: uploaded.clear()))
    res["upload_equals_sample"] = uploaded[-1].events_count() == true.events_count() == int(host.sum())
    uploaded.clear()
    del host
    pois = D.DiscreteData(ctx, surrogate)
    hy = np.array([net.baseline.alpha0, net.baseline.beta0, net.weights.kappa, net.weights.nu, net.impulses.gamma], dtype=np.float64)
    for name, d in (("true", true), ("poisson", pois)):
        D.convolve(net, d, export=False)

        def reset():
            net._push(ctx)
            ctx.check(lib.nhp_disc_network_set(ctx.h, 0.1))

        record("gibbs_sweep_" + name, timed(lambda: ctx.check(lib.nhp_disc_gibbs_sweep(ctx.h, d.h, 1, 7, _ptr(hy), 5, 1.0, 1.0)), setup=reset))
        std.weights.kappav, std.weights.nuv = np.ones_like(W), np.ones_like(W)
        q = np.ones(2 * N + N * N * (B + 2))
        ctx.check(lib.nhp_disc_vb_set(ctx.h, N, B, std.dt, _ptr(hy), 5, _ptr(q)))
        change = ctypes.c_double()
        record("vb_step_" + name, timed(lambda: ctx.check(lib.nhp_disc_vb_step(ctx.h, d.h, ctypes.byref(change)))))
    res["rand_over_upload"] = res["ms_median"]["rand"] / res["ms_median"]["upload"]
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
