"""The continuous network VB step against the standard VB step on the same events and one Gibbs sweep of the network process, at
config 4's shape.

    python tools/cont_vb_network_bench.py [--nodes 1000] [--events 1e8] [--rounds 3] [--out FILE]

Workload: the cfg4 network (LogitNormal, K = 1000, rho = 0.05, dtmax = 1, bench.py's parameters through the generator calls of
tools/cont_rand_lgcp_bench.py), and a sample of about `events` events drawn from it on the device (nhp_cont_rand).  Arms, one call
each per round, in turn:

  network_vb_step   nhp_cont_vb_step on a network state (nhp_cont_vb_network_set): slab concentrated at W (shape 1e3), pv = A, the
                    spike at its prior (kappa0 = 0.1, nu0 = 10), the other factors concentrated at the parameters as in
                    tools/cont_vb_bench.py
  vb_step           nhp_cont_vb_step on the standard state of the same factors, the parameters pushed without A
  gibbs_sweep       nhp_cont_gibbs_sweep of the network process (adjacency sweep and the draw of rho included)

Every arm's state (VB state, or the parameters and rho) is reset outside the timed region; round 0 is the warm-up.  A call is timed on
the host clock around work that ends in a device synchronisation; the figure is the median over the rounds.  The card's name and power
limit are read in the same process.  One JSON object goes to stdout (and to --out)."""
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
from cont_rand_lgcp_bench import BRANCHING, DTMAX, RATE, RHO, SEED, card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=1000)
    ap.add_argument("--events", type=float, default=1e8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.rounds < 1:
        ap.error("--rounds must be positive")
    import nhp_b200 as nhp
    import synth
    from nhp_b200 import continuous as C
    from nhp_b200.core import _fmat, _ptr
    ctx = nhp.default_context(0)
    lib = ctx.lib
    K = args.nodes
    lam0 = np.full(K, RATE * (1.0 - BRANCHING) / K)
    _, W, mu, tau, A = synth.ln_params(K, 2, wmax=2.0 * BRANCHING / (K * RHO), density=RHO)
    T = args.events / RATE
    proc = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.LogitNormalImpulseResponse(mu, tau, DTMAX), nhp.DenseWeightModel(W),
                                              A.copy(), nhp.BernoulliNetworkModel(RHO, K))
    proc.ctx = ctx
    proc._push(ctx)
    ev = ctypes.c_void_p()
    ctx.check(lib.nhp_cont_rand(ctx.h, T, SEED, int(args.events * 1.25) + 100000, ctypes.byref(ev)))
    n = int(lib.nhp_events_count(ev))
    lam0c, Wf, muf, tauf, Af = np.ascontiguousarray(lam0), _fmat(W), _fmat(mu), _fmat(tau), _fmat(A)

    def push(net):
        ctx.check(lib.nhp_cont_params_set(ctx.h, 1, K, _ptr(lam0c), _ptr(Wf), _ptr(Af) if net else None, _ptr(muf), _ptr(tauf), DTMAX))
        if net:
            ctx.check(lib.nhp_cont_network_set(ctx.h, RHO))

    hy_std = C._hyper(proc)
    hy_net = C.network_hyper(proc)
    s = 1e3
    KK = K * K
    q_std = np.concatenate([np.full(K, s), s / lam0c, np.full(KK, s), s / Wf, muf, np.full(KK, s), np.full(KK, s), s / tauf])
    q_net = np.concatenate([q_std, np.full(KK, 0.1), np.full(KK, 10.0), Af, [proc.network.alpha + RHO * KK, proc.network.beta + (1 - RHO) * KK]])
    sync = lambda: ctx.check(lib.nhp_cont_params_get(ctx.h, None, None, None, None, None))  # synchronises the context's stream
    change = ctypes.c_double()

    def reset_net():
        push(True)
        ctx.check(lib.nhp_cont_vb_network_set(ctx.h, _ptr(hy_net), hy_net.size, _ptr(q_net)))

    def reset_std():
        push(False)
        ctx.check(lib.nhp_cont_vb_set(ctx.h, _ptr(hy_std), hy_std.size, _ptr(q_std)))

    arms = {
        "network_vb_step": (reset_net, lambda: ctx.check(lib.nhp_cont_vb_step(ctx.h, ev, ctypes.byref(change)))),
        "vb_step": (reset_std, lambda: ctx.check(lib.nhp_cont_vb_step(ctx.h, ev, ctypes.byref(change)))),
        "gibbs_sweep": (lambda: push(True), lambda: ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, ev, ev, 7, 1, float(T), _ptr(hy_std), hy_std.size,
                                                                                      proc.network.alpha, proc.network.beta))),
    }
    wall = {k: [] for k in arms}
    for rnd in range(args.rounds + 1):
        for name, (reset, fn) in arms.items():
            reset()
            sync()
            t0 = time.perf_counter()
            fn()
            sync()
            if rnd > 0:
                wall[name].append((time.perf_counter() - t0) * 1e3)
    # the network step's outcome from the concentrated start: links kept on and rho
    reset_net()
    ctx.check(lib.nhp_cont_vb_step(ctx.h, ev, ctypes.byref(change)))
    q = np.empty(q_net.size)
    ctx.check(lib.nhp_cont_vb_get(ctx.h, _ptr(q)))
    pv = q[-2 - KK:-2]
    lib.nhp_events_free(ctx.h, ev)
    med = {k: float(np.median(v)) for k, v in wall.items()}
    res = {"tool": "cont_vb_network_bench", "card": card(),
           "workload": "cfg4: LogitNormal network, K=%d, rho=%.2f, %d events (nhp_cont_rand), dtmax %.1f" % (K, RHO, n, DTMAX),
           "rounds": args.rounds, "ms_median": med, "ms_rounds": wall,
           "network_over_standard_vb_step": med["network_vb_step"] / med["vb_step"], "network_vb_step_over_gibbs_sweep": med["network_vb_step"] / med["gibbs_sweep"],
           "vb_state_mb": q_net.size * 8 / 1e6, "links": int(np.sum(A)), "links_on_after_one_step": int(np.sum(pv > 0.5)),
           "rho_after_one_step": float(q[-2] / (q[-2] + q[-1]))}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
