"""The discrete VB step at config 3: one device step (nhp_disc_vb_step, VB trace open) against discrete.update_.

    python tools/disc_vb_bench.py [--block 10] [--blocks 5] [--out FILE]

Data and shape: bench.py's config 3 (N = 200, T = 1e6 bins, B = 6, L = 12, the same seeds, through disc_chain_bench.config3), modelled
as a DiscreteStandardHawkesProcess (VB has no network form) starting from the default all-ones variational parameters.  The arms
alternate, one block of `block` chained steps each, `blocks` rounds, after one warm-up block each; every block starts from the
all-ones state.  A block is timed on the host clock around work that ends in a device synchronisation; the figure is the median over
the blocks of (block time / block).  Arms:

  device_step   nhp_disc_vb_step with the VB trace open, reading `change` back every step: digamma expectations, statistics,
                in-place update, trace push; only the change crosses PCIe
  host_update   discrete.update_: digamma / exp on the host, E up, the statistics down, the update in NumPy
  vb_stats      nhp_disc_vb_stats alone (host e0 / E up, the sums down): the statistics kernel with its PCIe copies

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
    ap.add_argument("--block", type=int, default=10)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.block < 1 or args.blocks < 1:
        ap.error("--block and --blocks must be positive")
    import nhp_b200 as nhp
    from nhp_b200 import discrete as D
    from nhp_b200.core import _ptr
    lam0, W, _, theta, data, L = config3()
    N, B = lam0.size, theta.shape[2]
    proc = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W))
    ctx = proc._ctx()
    lib = ctx.lib
    d = proc.upload(data)
    D.convolve(proc, d, export=False)
    proc._push(ctx)  # for the synchronising nhp_disc_params_get below; VB does not read the parameters
    b, w, imp = proc.baseline, proc.weights, proc.impulses
    hy = np.array([b.alpha0, b.beta0, w.kappa, w.nu, imp.gamma], dtype=np.float64)
    nq = 2 * N + N * N * (B + 2)
    ones = np.ones(nq)
    e0, E = np.ones(N), np.ones(N * N * B)
    st = [np.empty(N), np.empty(N * N), np.empty(N * N), np.empty(N * N * B)]
    change = ctypes.c_double()

    def reset():
        D.set_variational_params_(proc, ones)
        ctx.check(lib.nhp_disc_vb_set(ctx.h, N, B, proc.dt, _ptr(hy), 5, _ptr(ones)))

    def device_step():
        ctx.check(lib.nhp_disc_vb_step(ctx.h, d.h, ctypes.byref(change)))

    def host_update():
        D.update_(proc, d)

    def vb_stats():
        ctx.check(lib.nhp_disc_vb_stats(ctx.h, d.h, _ptr(e0), _ptr(E), *[_ptr(x) for x in st]))

    arms = {"device_step": device_step, "host_update": host_update, "vb_stats": vb_stats}
    times = {k: [] for k in arms}
    reset()
    ctx.check(lib.nhp_disc_vb_trace_begin(ctx.h, (args.blocks + 1) * args.block))
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
    ctx.check(lib.nhp_disc_vb_trace_count(ctx.h, ctypes.byref(count), None))
    # the two paths agree after `block` steps from the same state
    reset()
    for _ in range(args.block):
        device_step()
        host_update()
    q = np.empty(nq)
    ctx.check(lib.nhp_disc_vb_get(ctx.h, _ptr(q)))
    max_rel_diff = float(np.max(np.abs(q - proc.variational_params()) / proc.variational_params()))
    ctx.check(lib.nhp_disc_vb_trace_free(ctx.h))
    d.free()
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {"tool": "disc_vb_bench", "card": card(), "workload": "config 3 data: discrete Gaussian standard Hawkes VB, N=200, T=1e6 bins, B=6, L=12, "
           "from all-ones variational parameters", "block": args.block, "blocks": args.blocks, "ms_per_step_median": med, "ms_per_step_blocks": times,
           "trace_slots": int(count.value), "trace_slot_mb": nq * 8 / 1e6, "speedup_device_step_vs_host_update": med["host_update"] / med["device_step"],
           "device_step_minus_vb_stats_ms": med["device_step"] - med["vb_stats"], "last_change": change.value,
           "max_rel_diff_device_vs_host_after_block": max_rel_diff}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
