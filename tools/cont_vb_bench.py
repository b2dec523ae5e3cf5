"""The continuous VB step against the two other device passes over the events: one nhp_cont_vb_step, one nhp_cont_loglik_grad (the
same two sweeps: intensities, then the child-major scatter) and one nhp_cont_gibbs_sweep.

    python tools/cont_vb_bench.py --config {2,5} [--rounds 5] [--events N] [--out FILE]

Shapes (bench.py's Poisson-surrogate streams and parameters, through the same generator calls as tools/bench_configs.py):
  --config 2   LogitNormal standard, K = 50, 1e6 events, rate 100, dtmax 1
  --config 5   Exponential standard, K = 5000, 1.25e8 events (one GPU's share), rate 3.2, dtmax Inf; no VB trace is kept (a state
               is 800 MB)
All three arms use the windowed (non-recursive) semantics.  The VB state is concentrated at the configuration's parameters (every
shape parameter 1e3, rates set so that the posterior means are the parameters), so that its effective parameters, and with them the
Exponential cut-off window, are those the gradient and the Gibbs sweep run with.  Each round times one call of every arm, in turn,
after resetting that arm's state (VB state, or the parameters) outside the timed region; round 0 is the warm-up.  A call is timed on
the host clock around work that ends in a device synchronisation; the figure is the median over the rounds.  `device_ms` is the
library's own CUDA-event time of the call (nhp_last_kernel_ms) for the two arms whose timer spans the whole call: the VB step (the
two table rebuilds included) and the gradient.  The card's name and power limit are read in the same process.  One JSON object goes to stdout (and to --out)."""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(ROOT, "networkhawkesprocesses.jl_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, HERE)
from disc_chain_bench import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, choices=(2, 5), required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--events", type=float, default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.rounds < 1:
        ap.error("--rounds must be positive")
    import nhp_b200 as nhp
    import synth
    from nhp_b200.core import _fmat, _ptr
    cfg = args.config
    K, rate = (50, 100.0) if cfg == 2 else (5000, 3.2)
    n = int(args.events) if args.events else (1_000_000 if cfg == 2 else 125_000_000)
    if cfg == 2:
        lam0, W, p1, p2, _ = synth.ln_params(K, 2)
        kind, dtmax = 1, 1.0
    else:
        lam0, W, p1, _ = synth.exp_params(K, 2)
        p2, kind, dtmax = None, 0, float("inf")
    ctx = nhp.Context(0)
    lib = ctx.lib
    rng = np.random.Generator(np.random.Philox(key=0x4E485030 + 16 * cfg))
    t = np.cumsum(rng.exponential(1.0 / rate, n))
    nodes = rng.integers(1, K + 1, n, dtype=np.int64)
    duration = float(t[-1]) * (1 + 1e-9)
    h = ctypes.c_void_p()
    ctx.check(lib.nhp_events_upload(ctx.h, _ptr(t), _ptr(nodes), n, duration, K, 0, 0, 1, ctypes.byref(h)))
    del t, nodes
    fl = [_fmat(W), _fmat(p1), None if p2 is None else _fmat(p2)]
    lam0 = np.ascontiguousarray(lam0)

    def push():
        ctx.check(lib.nhp_cont_params_set(ctx.h, kind, K, _ptr(lam0), _ptr(fl[0]), None, _ptr(fl[1]), _ptr(fl[2]), dtmax))

    # hyper-parameters: the defaults of the Python components
    hy = np.array([1.0, 1.0, 1.0, 1.0, 1.0, 1.0] if kind == 0 else [1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0])
    s = 1e3
    planes = [np.full(K * K, s), s / fl[0]] + ([np.full(K * K, s), s / fl[1]] if kind == 0 else [fl[1], np.full(K * K, s), np.full(K * K, s), s / fl[2]])
    q0 = np.concatenate([np.full(K, s), s / lam0] + planes)
    del planes
    hz = ctypes.c_double()
    push()
    ctx.check(lib.nhp_cont_horizon(ctx.h, n, 0, ctypes.byref(hz)))
    sync = lambda: ctx.check(lib.nhp_cont_params_get(ctx.h, None, None, None, None, None))  # synchronises the context's stream
    change = ctypes.c_double()

    def reset_vb():
        push()
        ctx.check(lib.nhp_cont_vb_set(ctx.h, _ptr(hy), hy.size, _ptr(q0)))

    arms = {
        "vb_step": (reset_vb, lambda: ctx.check(lib.nhp_cont_vb_step(ctx.h, h, ctypes.byref(change)))),
        "loglik_grad": (push, lambda: ctx.check(lib.nhp_cont_loglik_grad_dev(ctx.h, h, 0))),
        "gibbs_sweep": (push, lambda: ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, h, h, 7, 1, duration, _ptr(hy), hy.size, 0.0, 0.0))),
    }
    wall = {k: [] for k in arms}
    dev = {k: [] for k in arms if k != "gibbs_sweep"}
    for rnd in range(args.rounds + 1):
        for name, (reset, fn) in arms.items():
            reset()
            sync()
            t0 = time.perf_counter()
            fn()
            sync()
            if rnd > 0:
                wall[name].append((time.perf_counter() - t0) * 1e3)
                if name != "gibbs_sweep":  # its timer covers its last stage only
                    dev[name].append(ctx.last_kernel_ms)
    ctx.check(lib.nhp_events_free(ctx.h, h))
    med = {k: float(np.median(v)) for k, v in wall.items()}
    res = {"tool": "cont_vb_bench", "card": card(), "config": cfg,
           "workload": "cfg%d: %s standard, K=%d, %d events, rate %.1f, look-back horizon %.2f at the configuration's parameters"
                       % (cfg, "LogitNormal" if kind else "Exponential", K, n, rate, hz.value),
           "rounds": args.rounds, "ms_median": med, "ms_rounds": wall, "device_ms_median": {k: float(np.median(v)) for k, v in dev.items()},
           "vb_step_over_loglik_grad": med["vb_step"] / med["loglik_grad"], "vb_step_over_gibbs_sweep": med["vb_step"] / med["gibbs_sweep"],
           "vb_state_mb": q0.size * 8 / 1e6, "last_change": change.value}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
