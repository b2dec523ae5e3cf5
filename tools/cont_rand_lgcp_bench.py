"""Simulation with LogGaussianCoxProcess curves, and the sweeps on data drawn from the curves, at config 4's shape.

    python tools/cont_rand_lgcp_bench.py [--nodes 1000] [--events 1e8] [--reps 3] [--out FILE]

Model: the cfg4 network (K = 1000, rho = 0.05, LogitNormal, dtmax = 1, 1e8 events) with the +-30 % curves of
tools/adjacency_lgcp_bench.py (same rng, 41 grid points over [0, T]) as its baseline, and the GP prior of their logarithms
(m = log lambda0, sigma = 0.3, eta = T / 10).  In `reps` alternating rounds the script measures

  curves        nhp_cont_rand with the curves set (wall-clock ms, events generated), and on that sample, with its true curves and the
                prior set, one adjacency sweep (nhp_last_kernel_ms of the second sweep on the handle, batches and recomputed steps of
                nhp_cont_adjacency_info) and one nhp_cont_gibbs_sweep (wall-clock ms);
  homogeneous   nhp_cont_rand of the homogeneous cfg4 model, and the same sweeps with the same curves on its sample: the situation
                tools/adjacency_lgcp_bench.py and tools/baseline_slice_bench.py measure.

Every sweep starts from the pushed model.  The card's name and power limit are read in the same process.  One JSON object goes to
stdout (and to --out)."""
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
    from nhp_b200.continuous import _hyper
    from nhp_b200.core import _ptr
    ctx = nhp.default_context(0)
    lib = ctx.lib
    K = args.nodes
    lam0 = np.full(K, RATE * (1.0 - BRANCHING) / K)
    _, W, mu, tau, A = synth.ln_params(K, 2, wmax=2.0 * BRANCHING / (K * RHO), density=RHO)
    T = args.events / RATE
    rng = np.random.default_rng(7)
    G = 41
    x = np.linspace(0.0, T, G)
    c30 = lam0[:, None] * (1.0 + 0.3 * np.sin(2 * np.pi * rng.uniform(1.0, 4.0, (K, 1)) * x[None, :] / T + rng.uniform(0, 2 * np.pi, (K, 1))))

    def process(curves):
        base = nhp.LogGaussianCoxProcess(x, c30.copy(), m=float(np.log(lam0[0])), sigma=0.3, eta=T / 10.0) if curves else nhp.HomogeneousProcess(lam0)
        proc = nhp.ContinuousNetworkHawkesProcess(base, nhp.LogitNormalImpulseResponse(mu, tau, DTMAX), nhp.DenseWeightModel(W), A.copy(),
                                                  nhp.BernoulliNetworkModel(RHO, K))
        proc.ctx = ctx
        return proc

    lgcp, hom = process(True), process(False)
    hy = _hyper(lgcp)
    cap = int(args.events * 1.25) + 100000

    def rand(proc, seed):
        proc._push(ctx)
        ev = ctypes.c_void_p()
        t0 = time.perf_counter()
        ctx.check(lib.nhp_cont_rand(ctx.h, T, seed, cap, ctypes.byref(ev)))
        return ev, (time.perf_counter() - t0) * 1e3, int(lib.nhp_events_count(ev))

    def set_model():  # the curve model with its prior, from the start
        lgcp.baseline.lam_grid = c30.copy()
        lgcp._push(ctx)
        lgcp.baseline.push_prior(ctx)
        ctx.check(lib.nhp_cont_network_set(ctx.h, RHO))

    def sweeps(ev, counter):
        set_model()
        ctx.check(lib.nhp_cont_resample_adjacency_dev(ctx.h, ev, RHO, 11, counter, 0, 1, 0))  # builds the baseline rates
        set_model()
        ctx.check(lib.nhp_cont_resample_adjacency_dev(ctx.h, ev, RHO, 11, counter, 0, 1, 0))
        adj_ms, info = ctx.last_kernel_ms, nhp.adjacency_info(ctx)
        set_model()
        t0 = time.perf_counter()
        ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, ev, ev, 12, counter, float(T), _ptr(hy), hy.size, float(lgcp.network.alpha), float(lgcp.network.beta)))
        gibbs_ms = (time.perf_counter() - t0) * 1e3
        return {"adjacency_ms": adj_ms, "batches": info["batches"], "recomputed_steps": info["recomputed_steps"], "gibbs_sweep_ms": gibbs_ms}

    # One sample at a time: the adjacency sampler keeps its pair structure with the events handle only while it fits in its share of
    # the free memory, and with two 1e8-event handles resident the second one's does not (its sweeps take the uncached path, ~1 s).
    # Round 0 warms every path up.
    runs = []
    for rep in range(args.reps + 1):
        for name, proc in (("curves", lgcp), ("homogeneous", hom)):
            ev, ms, n = rand(proc, SEED + rep)
            r = dict(sweeps(ev, rep), rand_ms=ms, events=n, rep=rep, what=name)
            lib.nhp_events_free(ctx.h, ev)
            if rep > 0:
                runs.append(r)
                print(json.dumps(r), file=sys.stderr)
    out = {"what": "nhp_cont_rand with +-30 % curves and the sweeps on data from the curves, cfg4 shape", "card": card(), "nodes": K,
           "grid_points": G, "runs": runs}
    for name in ("curves", "homogeneous"):
        rs = [r for r in runs if r["what"] == name]
        keys = [k for k in rs[0] if k not in ("rep", "what")]
        out[name] = {k: [float(np.min([r[k] for r in rs])), float(np.max([r[k] for r in rs]))] for k in keys}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
