"""The network VB step at config 3: one device step on a network state against the standard VB step and a network SVI step.

    python tools/disc_vb_network_bench.py [--block 10] [--blocks 5] [--batch-bins 10000] [--out FILE]

Data and shape: bench.py's config 3 (N = 200, T = 1e6 bins, B = 6, L = 12, A ~ Bernoulli(0.1), the same seeds, through
disc_chain_bench.config3), modelled as a DiscreteNetworkHawkesProcess with a BernoulliNetworkModel.  The arms alternate, one block of
`block` chained steps each, `blocks` rounds, after one warm-up block each; every block starts from the default variational state
(network_variational_params of a fresh process; the all-ones standard state for the standard arm).  A block is timed on the host
clock around work that ends in a device synchronisation; the figure is the median over the blocks of (block time / block).  Arms:

  network_vb_step    nhp_disc_vb_step on the network state (nhp_disc_vb_network_set), reading `change` back every step
  standard_vb_step   nhp_disc_vb_step on the standard state of the same data (nhp_disc_vb_set)
  network_svi_step   nhp_disc_svi_step on the network state over windows of batch_bins bins (the windows and step sizes of
                     svi_schedule, seed 0)

The network step adds O(N^2) work (the per-link expectations, the lgamma targets and the sum of q(A=1)) to the statistics reduction
over the non-zero bins; the difference of the first two arms is its cost.  The card's name and power limit are read in the same
process.  One JSON object goes to stdout (and to --out)."""
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
    ap.add_argument("--block", type=int, default=10)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--batch-bins", type=int, default=10000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.block < 1 or args.blocks < 1:
        ap.error("--block and --blocks must be positive")
    import nhp_b200 as nhp
    from nhp_b200 import discrete as D
    from nhp_b200.core import _ptr
    lam0, W, A, theta, data, L = config3()
    N, B, T = lam0.size, theta.shape[2], data.shape[1]
    if not 1 <= args.batch_bins <= T:
        ap.error(f"--batch-bins must be in [1, {T}]")

    def fresh():
        return D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W),
                                              A, nhp.BernoulliNetworkModel(0.1, N))

    proc = fresh()
    ctx = proc._ctx()
    lib = ctx.lib
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    proc._push(ctx)  # for the synchronising nhp_disc_params_get below; VB does not read the parameters
    q_net = D.network_variational_params(fresh())
    hy_net = D._network_hyper(proc)
    b, w, imp = proc.baseline, proc.weights, proc.impulses
    hy_std = np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)
    q_std = np.ones(2 * N + N * N * (B + 2))
    nsvi = (args.blocks + 1) * args.block
    t_begin, steps = D.svi_schedule(T, nsvi, args.batch_bins, seed=0)
    change = ctypes.c_double()
    k_svi = [0]

    def net_reset():
        ctx.check(lib.nhp_disc_vb_network_set(ctx.h, N, B, proc.dt, _ptr(hy_net), hy_net.size, _ptr(q_net)))

    def std_reset():
        ctx.check(lib.nhp_disc_vb_set(ctx.h, N, B, proc.dt, _ptr(hy_std), hy_std.size, _ptr(q_std)))

    def vb_step():
        ctx.check(lib.nhp_disc_vb_step(ctx.h, d.h, ctypes.byref(change)))

    def svi_step():
        k = k_svi[0] % nsvi
        k_svi[0] += 1
        ctx.check(lib.nhp_disc_svi_step(ctx.h, d.h, int(t_begin[k]), args.batch_bins, float(steps[k]), ctypes.byref(change)))

    arms = {"network_vb_step": (net_reset, vb_step), "standard_vb_step": (std_reset, vb_step), "network_svi_step": (net_reset, svi_step)}
    times = {k: [] for k in arms}
    sync = lambda: ctx.check(lib.nhp_disc_params_get(ctx.h, None, None, None, None))  # synchronises the context's stream
    last_change = {}
    for rnd in range(args.blocks + 1):  # round 0: warm-up
        for name, (reset, fn) in arms.items():
            reset()
            sync()
            t0 = time.perf_counter()
            for _ in range(args.block):
                fn()
            sync()
            last_change[name] = change.value
            if rnd > 0:
                times[name].append((time.perf_counter() - t0) * 1e3 / args.block)
    # the device step against its host twin after one step from the default state
    net_reset()
    vb_step()
    q_dev = np.empty(q_net.size)
    ctx.check(lib.nhp_disc_vb_get(ctx.h, _ptr(q_dev)))
    twin = fresh()
    twin.ctx = ctx
    q_host = D.network_update_(twin, d)
    o = 2 * N + N * N * (B + 4)
    keep = np.ones(q_net.size, bool)
    keep[o:o + N * N] = False
    d.free()
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {"tool": "disc_vb_network_bench", "card": card(), "workload": "config 3 data: discrete Gaussian network Hawkes VB, N=200, T=1e6 bins, B=6, L=12, "
           "A ~ Bernoulli(0.1), from the default variational state", "block": args.block, "blocks": args.blocks, "svi_batch_bins": args.batch_bins,
           "ms_per_step_median": med, "ms_per_step_blocks": times, "network_minus_standard_vb_ms": med["network_vb_step"] - med["standard_vb_step"],
           "state_mb": q_net.size * 8 / 1e6, "last_change": last_change,
           "one_step_max_rel_diff_vs_host_twin": float(np.max(np.abs(q_dev[keep] - q_host[keep]) / np.abs(q_host[keep]))),
           "one_step_max_abs_diff_pv_vs_host_twin": float(np.max(np.abs(q_dev[o:o + N * N] - q_host[o:o + N * N])))}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
