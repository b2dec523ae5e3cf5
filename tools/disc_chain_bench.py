"""The discrete Gibbs chain at config 3: one device sweep (nhp_disc_gibbs_sweep, trace on) against discrete.resample_on_device_.

    python tools/disc_chain_bench.py [--block 20] [--blocks 5] [--out FILE]

Data and model: bench.py's config 3 (N = 200, T = 1e6 bins, B = 6, L = 12, rho = 0.1, the same seeds).  The arms alternate, one
block of `block` chained sweeps each, `blocks` rounds, after one warm-up block each; every block starts from the config-3 parameters.
A block is timed on the host clock around work that ends in a device synchronisation; the figure is the median over the blocks of
(block time / block).  Arms:

  device_sweep        nhp_disc_gibbs_sweep with the discrete trace open: counts, draws, table refresh, in-place adjacency sweep,
                      Beta draw of rho, trace push; only scalars cross PCIe
  resample_on_device  discrete.resample_on_device_: the same sweep with the parameters, A and the N x N link probability crossing
                      PCIe between its calls, and the Beta draw of rho on the host
  gibbs_counts, adjacency_dev
                      the sweep's two large kernels on their own (nhp_disc_gibbs_counts without a host copy,
                      nhp_disc_resample_adjacency_dev), for the share of the sweep that is neither

The card's name and power limit are read in the same process.  One JSON object goes to stdout (and to --out)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "networkhawkesprocesses.jl_b200"))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return out.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def config3():
    """bench.py other_configs_table, cfg3: the same generator calls in the same order."""
    N, Tb, B, L = 200, 1_000_000, 6, 12
    rng = np.random.default_rng(3)
    lam0 = np.full(N, 0.02)
    A = (rng.random((N, N)) < 0.1).astype(np.float64)
    W = rng.uniform(0.0, 0.5, (N, N)) * A
    W *= 0.5 / max(1e-9, np.max(np.abs(np.linalg.eigvals(W))))
    theta = rng.dirichlet(np.ones(B), (N, N))
    data = rng.poisson(0.04, (N, Tb)).astype(np.int64)
    return lam0, W, A, theta, data, L


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--block", type=int, default=20)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.block < 1 or args.blocks < 1:
        ap.error("--block and --blocks must be positive")
    import nhp_b200 as nhp
    from nhp_b200 import discrete as D
    from nhp_b200.core import _ptr
    lam0, W, A, theta, data, L = config3()
    N, B = lam0.size, theta.shape[2]
    proc = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W), A,
                                          nhp.BernoulliNetworkModel(0.1, N))
    ctx = proc._ctx()
    lib = ctx.lib
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    D.vb_row_sums(proc, d)  # resample_on_device_ caches the events per node with the data: not part of a sweep
    b, w, imp = proc.baseline, proc.weights, proc.impulses
    hy = np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)
    counter = [0]

    def reset():
        b.lam, w.W, imp.theta, proc.adjacency_matrix, proc.network.rho = lam0.copy(), W.copy(), theta.copy(), A.copy(), 0.1
        proc._push(ctx)
        ctx.check(lib.nhp_disc_network_set(ctx.h, 0.1))

    def nxt():
        counter[0] += 1
        return counter[0]

    def device_sweep():
        ctx.check(lib.nhp_disc_gibbs_sweep(ctx.h, d.h, 1, nxt(), _ptr(hy), 5, proc.network.alpha, proc.network.beta))

    def host_sweep():
        D.resample_on_device_(proc, d, seed=1, counter=nxt())

    def gibbs_counts():
        ctx.check(lib.nhp_disc_gibbs_counts(ctx.h, d.h, 1, nxt(), None, 0, None))

    def adjacency_dev():
        ctx.check(lib.nhp_disc_resample_adjacency_dev(ctx.h, d.h, -1.0, 1, nxt()))

    arms = {"device_sweep": device_sweep, "resample_on_device": host_sweep, "gibbs_counts": gibbs_counts, "adjacency_dev": adjacency_dev}
    times = {k: [] for k in arms}
    reset()  # the trace's slot layout follows the pushed model
    ctx.check(lib.nhp_disc_trace_begin(ctx.h, (args.blocks + 1) * args.block))
    sync = lambda: ctx.check(lib.nhp_disc_params_get(ctx.h, None, None, None, None))  # synchronises the context's stream
    for rnd in range(args.blocks + 1):  # round 0: warm-up
        for name, fn in arms.items():
            reset()
            sync()
            t0 = time.perf_counter()
            for _ in range(args.block):
                fn()
            sync()
            if rnd > 0:
                times[name].append((time.perf_counter() - t0) * 1e3 / args.block)
    count = ctypes.c_int64()
    ctx.check(lib.nhp_disc_trace_count(ctx.h, ctypes.byref(count), None))
    ctx.check(lib.nhp_disc_trace_free(ctx.h))
    d.free()
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {"tool": "disc_chain_bench", "card": card(), "workload": "config 3: discrete Gaussian network Hawkes, N=200, T=1e6 bins, B=6, L=12, rho=0.1",
           "block": args.block, "blocks": args.blocks, "ms_per_sweep_median": med, "ms_per_sweep_blocks": times, "trace_samples": int(count.value),
           "speedup_device_sweep": med["resample_on_device"] / med["device_sweep"],
           "device_sweep_minus_counts_and_adjacency_ms": med["device_sweep"] - med["gibbs_counts"] - med["adjacency_dev"]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
