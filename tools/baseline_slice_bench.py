"""The elliptical-slice update of LogGaussianCoxProcess curves at config 4's shape: on the device against the host path.

    python tools/baseline_slice_bench.py [--nodes 1000] [--events 1e8] [--reps 3] [--host-reps 2] [--out FILE]

Data: the homogeneous cfg4 model (K = 1000, rho = 0.05, LogitNormal, dtmax = 1) drawn on the device with nhp_cont_rand, as in
tools/adjacency_lgcp_bench.py.  Baseline: curves with the cfg4 mean and +-30 % variation on 41 grid points per node, with the GP
prior of a LogGaussianCoxProcess (sigma = 1, length scale T / 10, m = log of the mean).  Every measurement starts from the same
curves and the parents of one parent sweep with them.  Reported, with the card's name and power limit read in the same process:

  device     nhp_cont_resample_baseline (Philox): wall ms, split into the list build and the rounds (nhp_cont_slice_info), rounds,
             work items, mean / max attempts per node
  host       the path it replaces: LogGaussianCoxProcess.resample_ (one nhp_cont_baseline_loglik pass over all events per attempt
             round) followed by nhp_cont_baseline_grid
  rebuild    the first per-event rate rebuild after new curves (both paths pay it): a parent sweep on a new curve version minus one
             on the same version
  sweep      nhp_cont_gibbs_sweep with curves and a prior against the homogeneous cfg4 sweep on the same handle (sweep_info)

One JSON object goes to stdout (and to --out)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time
import types

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


def spread(v):
    return [float(np.min(v)), float(np.median(v)), float(np.max(v))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=1000)
    ap.add_argument("--events", type=float, default=1e8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-reps", type=int, default=2)
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
    hyper = _f64([1.0] * 8)

    rng = np.random.default_rng(7)
    G = 41
    x = np.linspace(0.0, T, G)
    c30 = lam0[:, None] * (1.0 + 0.3 * np.sin(2 * np.pi * rng.uniform(1.0, 4.0, (K, 1)) * x[None, :] / T + rng.uniform(0, 2 * np.pi, (K, 1))))
    base = nhp.LogGaussianCoxProcess(x, c30, m=float(np.log(lam0.mean())), sigma=1.0, eta=T / 10.0)
    d = types.SimpleNamespace(h=ev)

    def start(with_prior=True):
        """cfg4 parameters, the curves c30 (a new curve version), their prior, one parent sweep"""
        ctx.check(lib.nhp_cont_params_restore(ctx.h))
        ctx.check(lib.nhp_cont_baseline_grid(ctx.h, G, _ptr(_f64(x)), _ptr(_f64(c30.ravel()))))
        if with_prior:
            base.lam_grid = c30.copy()
            base.push_prior(ctx)
        ctx.check(lib.nhp_cont_resample_parents(ctx.h, ev, 3, 0, None, None, None))

    def parent_sweep_ms():
        t0 = time.perf_counter()
        ctx.check(lib.nhp_cont_resample_parents(ctx.h, ev, 3, 1, None, None, None))
        return (time.perf_counter() - t0) * 1e3

    def gibbs(counter, curves):
        ctx.check(lib.nhp_cont_params_restore(ctx.h))
        if curves:
            ctx.check(lib.nhp_cont_baseline_grid(ctx.h, G, _ptr(_f64(x)), _ptr(_f64(c30.ravel()))))
            base.push_prior(ctx)
        else:
            ctx.check(lib.nhp_cont_baseline_grid(ctx.h, 0, None, None))
        ctx.check(lib.nhp_cont_network_set(ctx.h, RHO))
        t0 = time.perf_counter()
        ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, ev, ev, 11, counter, float(T), _ptr(hyper), hyper.size, 1.0, 1.0))
        wall = (time.perf_counter() - t0) * 1e3
        info = np.zeros(8)
        ctx.check(lib.nhp_cont_sweep_info(ctx.h, info.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
        return wall, info

    # warm-up: node index, pair structure, module loads, the update's buffers
    start()
    ctx.check(lib.nhp_cont_resample_baseline(ctx.h, ev, 5, 0, None, None, None))
    gibbs(0, False)
    gibbs(0, True)

    device, rebuild = [], []
    for rep in range(args.reps):
        start()
        att = np.zeros(K, dtype=np.int64)
        t0 = time.perf_counter()
        ctx.check(lib.nhp_cont_resample_baseline(ctx.h, ev, 5, 1 + rep, None, None, _ptr(att)))
        wall = (time.perf_counter() - t0) * 1e3
        info = np.zeros(4)
        ctx.check(lib.nhp_cont_slice_info(ctx.h, info.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
        first = parent_sweep_ms()   # new curve version: rebuilds the per-event rates
        second = parent_sweep_ms()  # same version
        rebuild.append(first - second)
        device.append({"ms": wall, "build_ms": info[0], "rounds_ms": info[1], "rounds": int(info[2]), "work_items": int(info[3]),
                       "attempts_mean": float(att.mean()), "attempts_max": int(att.max()), "rebuild_ms": first - second})
        print(json.dumps({"device": device[-1]}), file=sys.stderr)

    host = []
    for rep in range(args.host_reps):
        start(with_prior=False)
        base.lam_grid = c30.copy()
        calls = [0]
        orig = lib.nhp_cont_baseline_loglik

        class Counting:  # count the likelihood passes of the host update
            def __getattr__(self, name):
                return getattr(lib, name)

            @staticmethod
            def nhp_cont_baseline_loglik(*a):
                calls[0] += 1
                return orig(*a)
        hctx = types.SimpleNamespace(h=ctx.h, lib=Counting(), check=ctx.check)
        t0 = time.perf_counter()
        base.resample_(hctx, d, np.random.default_rng([5, rep]))
        t1 = time.perf_counter()
        ctx.check(lib.nhp_cont_baseline_grid(ctx.h, G, _ptr(_f64(x)), _ptr(_f64(base.lam_grid.ravel()))))
        t2 = time.perf_counter()
        host.append({"ms": (t2 - t0) * 1e3, "slice_ms": (t1 - t0) * 1e3, "upload_ms": (t2 - t1) * 1e3, "loglik_passes": calls[0]})
        print(json.dumps({"host": host[-1]}), file=sys.stderr)

    sweeps = {"homogeneous": [], "curves_prior": []}
    counter = 1
    for rep in range(args.reps):
        for name in sweeps:
            wall, info = gibbs(counter, name == "curves_prior")
            counter += 1
            sweeps[name].append({"ms": wall, "parents_ms": info[0], "draws_ms": info[1], "adjacency_ms": info[2], "slice_ms": info[3], "slice_rounds": info[4]})
            print(json.dumps({name: sweeps[name][-1]}), file=sys.stderr)
    lib.nhp_events_free(ctx.h, ev)
    out = {"what": "elliptical-slice update of LGCP curves, cfg4 shape", "card": card(), "nodes": K, "events": n, "grid_points": G,
           "device": {k: spread([r[k] for r in device]) for k in device[0]},
           "host": {k: spread([r[k] for r in host]) for k in host[0]},
           "rebuild_ms": spread(rebuild),
           "gibbs_sweep": {name: {k: spread([r[k] for r in rs]) for k in rs[0]} for name, rs in sweeps.items()},
           "runs": {"device": device, "host": host, "sweeps": sweeps}}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
