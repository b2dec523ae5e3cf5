"""Stochastic VI steps on windows of bins at config 3: nhp_disc_svi_step at n_bins / T in {1, 0.1, 0.01, 0.001} against nhp_disc_vb_step.

    python tools/disc_svi_bench.py [--block 50] [--blocks 5] [--out FILE]

Data and shape: bench.py's config 3 (N = 200, T = 1e6 bins, B = 6, L = 12, the same seeds, through disc_chain_bench.config3), modelled
as a DiscreteStandardHawkesProcess starting from the all-ones variational parameters.  The arms alternate, one block of `block`
chained steps each, `blocks` rounds, after one warm-up round; every block starts from the all-ones state.  The SVI arms take their
windows and step sizes from discrete.svi_schedule (kappa = 0.75, tau0 = 1, the round as the seed), so windows wrap around the end as
they do in svi_device_.  Steps pass no `change` pointer, as svi_device_ and vb_device_ without rtol do, and the VB trace is closed; a
block is timed on the host clock around work that ends in a device synchronisation, and the figure is the median over the blocks of
(block time / block).  The cost of a window step should be a fixed part (digamma expectations, update, launches) plus the share of
the statistics kernel's time that the window's bins take.

Also: from the same state, the full window (t_begin = 0, n_bins = T, step = 1) against nhp_disc_vb_step (largest relative difference,
which is the run-to-run order of the statistics kernel's atomics).  The card's name and power limit are read in the same process.
One JSON object goes to stdout (and to --out)."""
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

FRACTIONS = (1.0, 0.1, 0.01, 0.001)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--block", type=int, default=50)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.block < 1 or args.blocks < 1:
        ap.error("--block and --blocks must be positive")
    import nhp_b200 as nhp
    from nhp_b200 import discrete as D
    from nhp_b200.core import _ptr
    lam0, W, _, theta, data, L = config3()
    N, T, B = lam0.size, data.shape[1], theta.shape[2]
    proc = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W))
    ctx = proc._ctx()
    lib = ctx.lib
    d = proc.upload(data)
    events_total = int(data.sum())
    del data
    D.convolve(proc, d, export=False)
    proc._push(ctx)  # for the synchronising nhp_disc_params_get below; VB does not read the parameters
    b, w, imp = proc.baseline, proc.weights, proc.impulses
    hy = np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)
    nq = 2 * N + N * N * (B + 2)
    ones = np.ones(nq)

    def reset():
        ctx.check(lib.nhp_disc_vb_set(ctx.h, N, B, proc.dt, _ptr(hy), 5, _ptr(ones)))

    def vb_block(seed):
        for _ in range(args.block):
            ctx.check(lib.nhp_disc_vb_step(ctx.h, d.h, None))

    def svi_block(frac):
        n = max(1, int(round(frac * T)))

        def run(seed):
            t_begin, step = D.svi_schedule(T, args.block, n, seed=seed)
            for k in range(args.block):
                ctx.check(lib.nhp_disc_svi_step(ctx.h, d.h, int(t_begin[k]), n, float(step[k]), None))
        return run

    arms = {"vb_step": vb_block}
    arms.update({f"svi_step_{f:g}": svi_block(f) for f in FRACTIONS})
    times = {k: [] for k in arms}
    sync = lambda: ctx.check(lib.nhp_disc_params_get(ctx.h, None, None, None, None))  # synchronises the context's stream
    for rnd in range(args.blocks + 1):  # round 0: warm-up
        for name, fn in arms.items():
            reset()
            sync()
            t0 = time.perf_counter()
            fn(rnd)
            sync()
            if rnd > 0:
                times[name].append((time.perf_counter() - t0) * 1e3 / args.block)
    # the full window is the VB step
    ch_vb, ch_svi = ctypes.c_double(), ctypes.c_double()
    reset()
    ctx.check(lib.nhp_disc_vb_step(ctx.h, d.h, ctypes.byref(ch_vb)))
    q_vb = np.empty(nq)
    ctx.check(lib.nhp_disc_vb_get(ctx.h, _ptr(q_vb)))
    reset()
    ctx.check(lib.nhp_disc_svi_step(ctx.h, d.h, 0, T, 1.0, ctypes.byref(ch_svi)))
    q_svi = np.empty(nq)
    ctx.check(lib.nhp_disc_vb_get(ctx.h, _ptr(q_svi)))
    d.free()
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {"tool": "disc_svi_bench", "card": card(), "workload": "config 3 data: discrete Gaussian standard Hawkes VB / SVI, N=200, T=1e6 bins, B=6, L=12, "
           f"{events_total} events, from all-ones variational parameters", "block": args.block, "blocks": args.blocks,
           "ms_per_step_median": med, "ms_per_step_blocks": times,
           "svi_over_vb": {k: med[k] / med["vb_step"] for k in med if k != "vb_step"},
           "max_rel_diff_full_window_vs_vb_step": float(np.max(np.abs(q_svi - q_vb) / q_vb)), "change_vb": ch_vb.value, "change_full_window": ch_svi.value}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
