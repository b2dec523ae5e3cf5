"""Adjacency sweep and structure log-likelihood with LogGaussianCoxProcess baselines at config 4's shape.

    python tools/adjacency_lgcp_bench.py [--nodes 1000] [--events 1e8] [--reps 3] [--out FILE]

Data: the homogeneous cfg4 model (K = 1000, rho = 0.05, LogitNormal, dtmax = 1) drawn on the device with nhp_cont_rand (data from
the homogeneous model are enough for timing).  On that one events handle the script alternates four baselines, `reps` rounds:

  homogeneous   the cfg4 lambda0
  constant      curves equal to that lambda0 everywhere: the same decisions, so the difference is the cost of reading the rates
  curves_30     curves with the same mean and +-30 % variation (41 grid points per node)
  dips_1pct     the same curves, each dipping to 1 % of the mean at one grid point

and reports per run the adjacency sweep (nhp_last_kernel_ms, batches and recomputed steps of nhp_cont_adjacency_info), the structure
log-likelihood against the window sweep (NHP_ADJ_LOGLIK=0), and the one-off cost of the per-event / by-node baseline rates: the
wall-clock time of the first sweep after a new curve version minus that of the next sweep on the same version.  Every sweep starts
from the cfg4 parameters (nhp_cont_params_restore).  The card's name and power limit are read in the same process.  One JSON
object goes to stdout (and to --out)."""
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

RATE, DTMAX, RHO, BRANCHING, SEED = 64.0, 1.0, 0.05, 0.5, 20261018  # bench.py's config 4


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return out.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=1000)
    ap.add_argument("--events", type=float, default=1e8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import nhp_b200 as nhp
    import synth
    from nhp_b200.core import _f64, _fmat, _ptr
    ctx = nhp.default_context(0)
    lib = ctx.lib
    K = args.nodes
    lam0 = np.full(K, RATE * (1.0 - BRANCHING) / K)
    _, W, mu, tau, A = synth.ln_params(K, 2, wmax=2.0 * BRANCHING / (K * RHO), density=RHO)
    ctx.check(lib.nhp_cont_params_set(ctx.h, 1, K, _ptr(_f64(lam0)), _ptr(_fmat(W)), _ptr(_fmat(A)), _ptr(_fmat(mu)), _ptr(_fmat(tau)), DTMAX))
    T = args.events / RATE
    ev = ctypes.c_void_p()
    ctx.check(lib.nhp_cont_rand(ctx.h, T, SEED, int(args.events * 1.25) + 100000, ctypes.byref(ev)))
    n = int(lib.nhp_events_count(ev))
    ctx.check(lib.nhp_cont_params_save(ctx.h))

    rng = np.random.default_rng(7)
    G = 41
    x = np.linspace(0.0, T, G)
    c30 = lam0[:, None] * (1.0 + 0.3 * np.sin(2 * np.pi * rng.uniform(1.0, 4.0, (K, 1)) * x[None, :] / T + rng.uniform(0, 2 * np.pi, (K, 1))))
    dips = c30.copy()
    dips[np.arange(K), rng.integers(1, G - 1, K)] = 0.01 * lam0
    baselines = {"homogeneous": None, "constant": np.repeat(lam0[:, None], G, axis=1), "curves_30": c30, "dips_1pct": dips}

    def set_baseline(vals):
        if vals is None:
            ctx.check(lib.nhp_cont_baseline_grid(ctx.h, 0, None, None))
        else:
            ctx.check(lib.nhp_cont_baseline_grid(ctx.h, G, _ptr(_f64(x)), _ptr(_f64(vals.ravel()))))

    def sweep(counter):
        ctx.check(lib.nhp_cont_params_restore(ctx.h))
        ctx.check(lib.nhp_cont_network_set(ctx.h, RHO))
        t0 = time.perf_counter()
        ctx.check(lib.nhp_cont_resample_adjacency_dev(ctx.h, ev, RHO, 11, counter, 0, 1, 0))
        wall = (time.perf_counter() - t0) * 1e3
        return wall, ctx.last_kernel_ms, nhp.adjacency_info(ctx)

    def loglik(window):
        if window:
            os.environ["NHP_ADJ_LOGLIK"] = "0"
        try:
            ll = ctypes.c_double()
            ctx.check(lib.nhp_cont_loglik(ctx.h, ev, 0, ctypes.byref(ll)))
            return ll.value, ctx.last_kernel_ms
        finally:
            os.environ.pop("NHP_ADJ_LOGLIK", None)

    # warm-up: the pair structure, the node index, the module loads
    sweep(0)
    ctx.check(lib.nhp_cont_params_restore(ctx.h))
    loglik(False)
    loglik(True)
    runs = []
    counter = 1
    for rep in range(args.reps):
        for name, vals in baselines.items():
            set_baseline(vals)
            w1, ms1, _ = sweep(counter)       # first sweep of this curve version: builds the baseline rates
            w2, ms2, info = sweep(counter)    # same version, same uniforms
            counter += 1
            ctx.check(lib.nhp_cont_params_restore(ctx.h))
            ll_s, ms_s = loglik(False)
            ll_w, ms_w = loglik(True)
            runs.append({"rep": rep, "baseline": name, "sweep_ms": ms2, "sweep_ms_first": ms1, "batches": info["batches"],
                         "recomputed_steps": info["recomputed_steps"], "flips": info["flips"], "steps": info["steps"],
                         "rates_build_ms": w1 - w2, "loglik_structure_ms": ms_s, "loglik_window_ms": ms_w,
                         "loglik_rel_diff": abs(ll_s - ll_w) / abs(ll_w)})
            print(json.dumps(runs[-1]), file=sys.stderr)
    lib.nhp_events_free(ctx.h, ev)
    out = {"what": "adjacency sweep / structure log-likelihood with grid baselines, cfg4 shape", "card": card(), "nodes": K, "events": n,
           "grid_points": G, "runs": runs}
    for name in baselines:
        rs = [r for r in runs if r["baseline"] == name]
        out[name] = {k: [float(np.min([r[k] for r in rs])), float(np.max([r[k] for r in rs]))]
                     for k in ("sweep_ms", "batches", "recomputed_steps", "rates_build_ms", "loglik_structure_ms", "loglik_window_ms")}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
