#!/usr/bin/env python
"""bench.py -- headline benchmark of the event-history hot path (BASELINE.json metric:
"loglik & Gibbs-sweep events/s at 1/2/4/8 B200, % roofline, vs CPU Threads").

Workload (BASELINE.json configs[3], the configuration the north_star target is quoted on; it fits one GPU): continuous
LogitNormal *network* Hawkes process, Bernoulli(rho = 0.05) adjacency, K = 1000 nodes, 1e8 events, total rate 64 events/s,
dtmax = 1 (mean predecessor window 64).

A step = one log-likelihood evaluation + one FULL Gibbs sweep of `resample!` (continuous.jl:350-358): parent resampling
fused with the sufficient statistics, the two-pass variance statistic, the conjugate draws of lambda0 / W / (mu, tau) with the
table rebuild, the adjacency-matrix sweep (continuous.jl:444-519) and the Beta draw of rho -- all on the device, through
nhp_cont_loglik + nhp_cont_gibbs_sweep of the C ABI.

Multi-GPU (torchrun, one process per GPU): STRONG scaling by default -- the 1e8-event stream is cut into contiguous time shards
with a dtmax halo for the log-likelihood / parent sweep (NCCL all-reduce of the statistics inside the library), and the adjacency
sweep partitions the child columns over the ranks on the replicated stream (NCCL all-gather of the columns).  `--scaling weak`
keeps 1e8 events per GPU instead.

Data: `--data hawkes` (default) draws the stream from the model itself with the device branching simulator (nhp_cont_rand), so the
chain runs on data that carry the network (few links flip per sweep once mixed, as in a real `mcmc!` run); `--data surrogate` is
round 1's Poisson surrogate (iid gaps, uniform nodes; SURVEY.md section 8d).  Every step starts from the workload's parameters
(`--chain rewind`, default; `--chain free` lets the chain keep its state).

  python bench.py [--gpus N] [--steps K] [--warmup W]           (torchrun launches N > 1)
  python bench.py --impl reference ...                          (CPU oracle arm, all host threads)
  python bench.py --config {2,3,5} ...                          (the other BASELINE configs as their own line)
  python bench.py --dump-outputs DIR ...                        (also write the last timed step's outputs as DIR/<name>.npy)
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "networkhawkesprocesses.jl_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "loglik+gibbs_sweep_events_per_s"
UNIT = "events/s"
RATE, DTMAX, RHO, BRANCHING = 64.0, 1.0, 0.05, 0.5
# SURVEY.md section 8d: algorithmic work per unit
FLOPS_PER_LN_PAIR, FLOPS_PER_EVENT = 96.0, 40.0   # nominal FP64 flops (libdevice-class accuracy)
BYTES_LOGLIK, BYTES_PARENTS = 12.0, 12.0          # per event: 8 B time + 4 B node (parents stay on the device as fused statistics)
BYTES_EXTRA_WLEN, BYTES_EXTRA_POFF = 2.0, 4.0     # implementation extras, stated separately: cached window length read, parent offset written
BYTES_PER_ADJ_PAIR = 10.0                         # cached adjacency structure: u16 event index + f64 lag per (child event, window predecessor);
                                                  # 18 B with the LogitNormal payload (u16 + logit + Jacobian) -- the form the library reports is used
SEED = 20261018
DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=[2, 3, 4, 5])
    ap.add_argument("--events", type=float, default=None, help="events in total (strong scaling) or per GPU (weak); default 1e8 (config 4)")
    ap.add_argument("--nodes", type=int, default=1000)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--data", default="hawkes", choices=["hawkes", "surrogate"])
    ap.add_argument("--chain", default="rewind", choices=["rewind", "free"],
                    help="rewind: every step is one sweep from the workload's parameters (stationary, reproducible timing); free: the chain keeps its state")
    ap.add_argument("--cpu-sample", type=float, default=1e6, help="events of the CPU-baseline sample (log-likelihood + parent sweep)")
    ap.add_argument("--cpu-adj-sample", type=float, default=1e5, help="events of the CPU-baseline sample of the adjacency sweep")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config table (cfg2 / cfg3 / cfg5 shape) of the default N = 1 run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (its log-likelihood and the sample of its Gibbs sweep) as DIR/<name>.npy in float64, "
                         "to compare two builds output for output (config 4, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or args.config != 4):
        ap.error("--dump-outputs is implemented for the headline workload (--config 4, --impl ours)")
    args.events_given = args.events is not None
    if args.events is None:
        args.events = 1e8
    return args


def emit(line):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = None


def host_threads():
    """All the host cores this process may use (torchrun exports OMP_NUM_THREADS=1: ignore it for the CPU arm)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------
def make_params(K, data_mode, seed=2):
    """cfg4 parameters.  hawkes: lambda0 and W scaled so that the stationary total rate is RATE with branching ratio BRANCHING."""
    import synth
    lam0, W, mu, tau, A = synth.ln_params(K, seed, wmax=2.0 * BRANCHING / (K * RHO), density=RHO)
    if data_mode == "hawkes":
        lam0 = np.full(K, RATE * (1.0 - BRANCHING) / K)
    return lam0, W, mu, tau, A


def surrogate_stream(n, K, seed):
    rng = np.random.default_rng(seed)
    t = np.cumsum(rng.exponential(1.0 / RATE, n))
    nodes = rng.integers(1, K + 1, n, dtype=np.int64)
    return t, nodes, float(t[-1] * (1 + 1e-9))


def host_hawkes_sample(lam0, W, mu, tau, A, T, seed):
    """Generation-by-generation numpy simulator of the same cluster process (continuous.jl:16-37), for the CPU arm's sample."""
    rng = np.random.default_rng(seed)
    K = lam0.size
    Weff = W * A
    rowsum = Weff.sum(axis=1)
    cdf = np.cumsum(Weff, axis=1)
    n0 = rng.poisson(lam0 * T)
    t = rng.uniform(0.0, T, int(n0.sum()))
    c = np.repeat(np.arange(K), n0)
    ts, cs = [t], [c]
    while t.size:
        m = rng.poisson(rowsum[c])
        par_t, par_c = np.repeat(t, m), np.repeat(c, m)
        if par_t.size == 0:
            break
        u = rng.random(par_t.size) * rowsum[par_c]
        child = np.array([np.searchsorted(cdf[p], x, side="right") for p, x in zip(par_c, u)], dtype=np.int64) if par_t.size < 1000 else \
            _rowwise_search(cdf, par_c, u)
        child = np.minimum(child, K - 1)
        z = rng.normal(mu[par_c, child], 1.0 / np.sqrt(tau[par_c, child]))
        tt = par_t + DTMAX / (1.0 + np.exp(-z))
        keep = tt <= T
        t, c = tt[keep], child[keep]
        ts.append(t); cs.append(c)
    t, c = np.concatenate(ts), np.concatenate(cs)
    idx = np.argsort(t, kind="stable")
    return t[idx], (c[idx] + 1).astype(np.int64), float(T)


def _rowwise_search(cdf, rows, x):
    out = np.empty(rows.size, dtype=np.int64)
    order = np.argsort(rows, kind="stable")
    rs = rows[order]
    bounds = np.flatnonzero(np.diff(rs)) + 1
    for seg in np.split(np.arange(rows.size), bounds):
        if seg.size:
            r = rs[seg[0]]
            out[order[seg]] = np.searchsorted(cdf[r], x[order[seg]], side="right")
    return out


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons DURING the timed region (NVML; nvidia-smi as fallback)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.max_mhz = index, [], False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            while not self.stop_flag:
                mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((mhz, [k for k, b in bits.items() if r & b]))
                time.sleep(0.02)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                self.max_mhz = float(f[1])
                self.rows.append((float(f[0]), [n for i, n in enumerate(names) if f[2 + i].lower().startswith("active")]))
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        reasons = sorted({r for _, rs in self.rows for r in rs})
        return {"sm_mhz": float(np.median([m for m, _ in self.rows])), "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(self.rows)}


def hbm_peak():
    f = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(f):
        with open(f) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback (of fallback)"


def workload_config(args, world, n_total, n_shard):
    return {"workload": "cfg4: continuous LogitNormal network Hawkes, Bernoulli(rho=0.05) adjacency, K=%d, %.3g events, rate 64/s, dtmax=1 (mean window 64); "
                        "step = loglikelihood + full Gibbs sweep (parents + fused statistics + conjugate draws + adjacency sweep + rho draw)" % (args.nodes, n_total),
            "K": args.nodes, "global_events": int(n_total), "events_per_gpu": int(n_shard), "mean_window": RATE * DTMAX, "rho": RHO,
            "data_mode": args.data, "chain": args.chain,
            "sharding": ("contiguous time shards + dtmax halo (log-likelihood, parent sweep, statistics); child columns c % N == rank on the replicated stream "
                         "(adjacency sweep)") if world > 1 else "single GPU",
            "l2_policy": "inputs (1.2 GB of events, 116 GB of cached adjacency pairs) are larger than the 126 MB L2; no explicit flush"}


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle (restated reference, C + OpenMP at the reference's Threads.@threads sites)
# ------------------------------------------------------------------------------------------
def cpu_sample_data(args):
    """The CPU arm's bounded sample of the same workload: true Hawkes draws of the cfg4 model (or the surrogate stream)."""
    K = args.nodes
    lam0, W, mu, tau, A = make_params(K, args.data)
    n1, n2 = int(args.cpu_sample), int(args.cpu_adj_sample)
    if args.data == "hawkes":
        t, nodes, T = host_hawkes_sample(lam0, W, mu, tau, A, n1 / RATE, 7)
    else:
        t, nodes, T = surrogate_stream(n1, K, 1000)
    m = min(n2, t.size)
    return (lam0, W, mu, tau, A), (t, nodes, T), (t[:m].copy(), nodes[:m].copy(), float(t[m - 1] * (1 + 1e-9)))


def cpu_step_time(args, reps, sample=None):
    """Seconds per event of the reference algorithm on the host cores, split into (log-likelihood + parent sweep + statistics) on
    the first sample and the adjacency sweep on a smaller one restricted to `cols` columns (the reference's 2 K^2 N algorithm does
    not finish on anything larger); the column subset is scaled by K / cols, which is exact for its cost (columns are independent
    and equally expensive) and stated in the output."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_ffi as orc
    K = args.nodes
    params, d1, d2 = sample or cpu_sample_data(args)
    lam0, W, mu, tau, A = params
    cores = host_threads()
    orc.set_threads(cores)
    om = orc.Cont(1, lam0, W, mu, tau, A=A, dtmax=DTMAX)
    t, nodes, T = d1
    t2, nodes2, T2 = d2
    u = np.random.default_rng(5).random(t.size)
    ua = np.random.default_rng(6).random((K, K))
    cols = min(K, max(cores, 8))
    stride = K // cols
    rho = np.full((K, K), RHO)
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        ll = om.loglik(t, nodes, T)
        par, pn = om.resample_parents(t, nodes, u)
        orc.suffstats(1, t, nodes, par, pn, K, DTMAX)
        t1 = time.perf_counter()
        om.resample_adjacency(A, rho, t2, nodes2, T2, ua, 0, stride)
        t2_ = time.perf_counter()
        ncols = len(range(0, K, stride))
        per_event = (t1 - t0) / t.size + (t2_ - t1) * (K / ncols) / t2.size
        out.append({"per_event_s": per_event, "sweeps_s": t1 - t0, "adjacency_s": t2_ - t1, "adjacency_cols": ncols, "ll": ll})
    desc = ("oracle/liboracle.so on %d threads: loglik + resample_parents + sufficient statistics on %d events, adjacency sweep "
            "(2 K^2 passes) on %d events restricted to %d of %d columns and scaled by %d/%d; seconds per event of the two added"
            % (cores, t.size, t2.size, out[0]["adjacency_cols"], K, K, out[0]["adjacency_cols"]))
    return out, cores, desc, (params, d1, d2)


def run_reference(args, rank, world):
    if rank != 0:
        return
    if args.config != 4:
        return run_reference_other(args)
    rows, cores, desc, _ = cpu_step_time(args, args.warmup + args.steps)
    timed = rows[args.warmup:]
    per_event = float(np.mean([r["per_event_s"] for r in timed]))
    value = 1.0 / per_event
    step_s = float(np.mean([r["sweeps_s"] + r["adjacency_s"] for r in timed]))
    n_total = int(args.events) * (world if args.scaling == "weak" else 1)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * step_s, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, world, n_total, n_total // world),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------
# GPU arm (config 4)
# ------------------------------------------------------------------------------------------
def setup_distributed(local_rank, world):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    return torch, dist, dev


def make_context(torch, dev, local_rank, rank, world, dist):
    """One libnhp context on an explicit stream; for N > 1 the library's own NCCL communicator (nhp_comm_init), the 128-byte id
    travelling through torch.distributed (any host-side channel would do)."""
    import nhp_b200 as nhp
    ctx = nhp.Context(local_rank)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx.check(ctx.lib.nhp_set_stream(ctx.h, ctypes.c_void_p(stream.cuda_stream)))
    if world > 1:
        idbuf = (ctypes.c_ubyte * 128)()
        if rank == 0:
            ctx.check(ctx.lib.nhp_comm_unique_id(idbuf))
        tid = torch.tensor(list(bytes(idbuf)), dtype=torch.uint8, device=dev)
        dist.broadcast(tid, 0)
        raw = bytes(tid.cpu().tolist())
        ctx.check(ctx.lib.nhp_comm_init(ctx.h, ctypes.c_char_p(raw), rank, world))
    return ctx, stream


def run_ours(args, rank, world, local_rank):
    torch, dist, dev = setup_distributed(local_rank, world)
    import nhp_b200 as nhp
    from nhp_b200.core import _fmat, _ptr
    ctx, stream = make_context(torch, dev, local_rank, rank, world, dist)
    lib = ctx.lib
    K = args.nodes
    K2 = K * K
    n_target = int(args.events) * (world if args.scaling == "weak" else 1)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lam0, W, mu, tau, A = make_params(K, args.data)
    pl0, pW, pA, pmu, ptau = (np.ascontiguousarray(lam0), _fmat(W), _fmat(A), _fmat(mu), _fmat(tau))
    hyper = np.ones(8)

    def set_params():
        ctx.check(lib.nhp_cont_params_set(ctx.h, 1, K, _ptr(pl0), _ptr(pW), _ptr(pA), _ptr(pmu), _ptr(ptau), DTMAX))
        ctx.check(lib.nhp_cont_network_set(ctx.h, RHO))

    set_params()
    # ---- the stream: identical on every rank (same seed); full copy on the device for the adjacency sweep, pinned host copy for
    #      the shards and the end-to-end leg
    t_gen0 = time.perf_counter()
    if args.data == "hawkes":
        T = n_target / RATE
        h_full = ctypes.c_void_p()
        ctx.check(lib.nhp_cont_rand(ctx.h, T, SEED, int(n_target * 1.25) + 100000, ctypes.byref(h_full)))
        n_total = int(lib.nhp_events_count(h_full))
        h_t = torch.empty(n_total, dtype=torch.float64, pin_memory=True)
        h_c = torch.empty(n_total, dtype=torch.int64, pin_memory=True)
        ctx.check(lib.nhp_events_download(ctx.h, h_full, ctypes.c_void_p(h_t.data_ptr()), ctypes.c_void_p(h_c.data_ptr()), None))
        duration = T
    else:
        t_np, c_np, duration = surrogate_stream(n_target, K, 1000)
        n_total = n_target
        h_t = torch.empty(n_total, dtype=torch.float64, pin_memory=True)
        h_c = torch.empty(n_total, dtype=torch.int64, pin_memory=True)
        h_t.numpy()[:] = t_np
        h_c.numpy()[:] = c_np
        del t_np, c_np
        h_full = None
    gen_s = time.perf_counter() - t_gen0
    tt = h_t.numpy()
    # ---- this rank's time shard [i0, i1) + halo
    i0, i1 = rank * n_total // world, (rank + 1) * n_total // world
    n = i1 - i0
    lo = int(np.searchsorted(tt, tt[i0] - DTMAX, side="right")) if rank > 0 else 0
    lo = min(lo, i0)
    n_halo = i0 - lo

    def upload(first, count, halo, flags):
        h = ctypes.c_void_p()
        ctx.check(lib.nhp_events_upload(ctx.h, ctypes.c_void_p(h_t.data_ptr() + 8 * (first - halo)), ctypes.c_void_p(h_c.data_ptr() + 8 * (first - halo)),
                                        count + halo, duration, K, halo, first - halo, flags, ctypes.byref(h)))
        return h

    def upload_shard():
        return upload(i0, n, n_halo, 1 if rank == 0 else 0)

    if world == 1:
        if h_full is None:
            h_full = upload(0, n_total, 0, 1)
        ev_shard = h_full
    else:
        if h_full is None:
            h_full = upload(0, n_total, 0, 1)
        ev_shard = upload_shard()
    ev_full = h_full
    if args.chain == "rewind":
        ctx.check(lib.nhp_cont_params_save(ctx.h))

    op_ms = {"loglik": [], "parents": [], "draws": [], "adjacency": [], "step": []}
    adj_rows = []

    def step(counter, record=False):
        if args.chain == "rewind":
            # Every step is one sweep from the workload's parameters (device-to-device copy + table rebuild, ~0.5 ms, inside the timed region).
            # Left alone, the chain does not stay at cfg4's 5 % density: the model resamples W from its prior where A = 0 (weights.jl:59-64,
            # quirk Q14), so uninformative links switch on with probability ~rho, rho follows (networks.jl:72-78), and A fills up sweep by
            # sweep -- a property of the reference's sampler, kept as is, but not a stationary workload to time.
            ctx.check(lib.nhp_cont_params_restore(ctx.h))
            ctx.check(lib.nhp_cont_network_set(ctx.h, RHO))
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ll = ctypes.c_double()
        ctx.check(lib.nhp_cont_loglik_dist(ctx.h, ev_shard, ev_full, 0, ctypes.byref(ll)))  # N > 1: the rank's share (its columns of the structure once it exists, else its time shard)
        llk = ctx.last_kernel_ms
        llv = np.array([ll.value])
        ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(llv), 1))
        ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, ev_shard, ev_full, SEED, counter, float(duration), _ptr(hyper), hyper.size, 1.0, 1.0))
        e1.record(stream)
        if record:
            e1.synchronize()
            info, ainfo = np.zeros(8), np.zeros(8)
            lib.nhp_cont_sweep_info(ctx.h, info.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
            lib.nhp_cont_adjacency_info(ctx.h, ainfo.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
            op_ms["loglik"].append(llk); op_ms["parents"].append(info[0]); op_ms["draws"].append(info[1]); op_ms["adjacency"].append(info[2])
            op_ms["step"].append(e0.elapsed_time(e1))
            adj_rows.append(ainfo.copy())
        return float(llv[0])

    # ---- roofline denominators measured on this device
    peaks = {}
    if rank == 0:
        for which, key in ((0, "fp64_fma_tflops"), (1, "ln_pairs_per_s"), (2, "exp_pairs_per_s"), (3, "dmma_tflops"), (4, "probes_per_s")):
            r = ctypes.c_double()
            ctx.check(lib.nhp_bench_fp64(ctx.h, which, ctypes.byref(r)))
            peaks[key] = r.value

    # ---- parity check of what is being timed against the oracle (N = 1 default run): log-likelihood to 1e-10 and Philox parents
    #      bit-exact on the head of the stream, with the workload's parameters
    parity = None
    cpu_sample = None
    if world == 1 and not args.no_cpu_baseline:
        parity, cpu_sample = parity_check(args, ctx, (lam0, W, mu, tau, A), h_t, h_c)
        set_params()
        if args.chain == "rewind":
            ctx.check(lib.nhp_cont_params_save(ctx.h))

    for w in range(args.warmup):
        step(w)
    sync_all()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ctx.launches
    t_begin = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    t_begin.record(stream)
    ll_last = None
    for k in range(args.steps):
        ll_last = step(args.warmup + k, record=True)
    t_end.record(stream)
    sync_all()
    total_ms = t_begin.elapsed_time(t_end)
    launches = ctx.launches - launches0
    sampler.stop_flag = True
    sampler.join(timeout=3)
    tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = float(tmax.item())
    value = n_total * args.steps / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_step_outputs(ctx, K, ll_last))

    # ---- full-size checks (size-independent properties on the whole timed stream; outside the timed region):
    #      the two independent log-likelihood algorithms agree (window sweep over the time-sorted stream vs the active buckets of the
    #      parent-bucketed pair structure), every event got exactly one parent (sum M0 + sum Mnm = sum Mn = events), A stays 0/1
    full = None
    if world == 1:
        set_params()
        lls = {}
        for name, env in (("structure", None), ("window", "0")):
            if env is None:
                os.environ.pop("NHP_ADJ_LOGLIK", None)
            else:
                os.environ["NHP_ADJ_LOGLIK"] = env
            llv = ctypes.c_double()
            ctx.check(lib.nhp_cont_loglik(ctx.h, ev_full, 0, ctypes.byref(llv)))
            lls[name] = llv.value
            lls[name + "_ms"] = float(lib.nhp_last_kernel_ms(ctx.h))
        os.environ.pop("NHP_ADJ_LOGLIK", None)
        ctx.check(lib.nhp_cont_resample_parents(ctx.h, ev_full, SEED, 777, None, None, None))
        M0, Mn, Mnm = np.empty(K), np.empty(K), np.empty(K2)
        ctx.check(lib.nhp_cont_suffstats_read(ctx.h, _ptr(M0), _ptr(Mn), _ptr(Mnm), None, None))
        Acur = np.empty(K2)
        ctx.check(lib.nhp_cont_params_get(ctx.h, None, None, _ptr(Acur), None, None))
        full = {"events": n_total, "loglik_structure": lls["structure"], "loglik_window": lls["window"],
                "loglik_structure_ms": lls["structure_ms"], "loglik_window_ms": lls["window_ms"],
                "loglik_rel_diff": abs(lls["structure"] - lls["window"]) / abs(lls["window"]),
                "parents_assigned": float(M0.sum() + Mnm.sum()), "events_per_node_sum": float(Mn.sum()),
                "parents_on_inactive_links": float(Mnm[Acur == 0.0].sum()), "adjacency_is_binary": bool(np.all((Acur == 0.0) | (Acur == 1.0)))}
        full["ok"] = bool(full["loglik_rel_diff"] <= 1e-10 and full["parents_assigned"] == n_total and full["events_per_node_sum"] == n_total
                          and full["parents_on_inactive_links"] == 0.0 and full["adjacency_is_binary"])
        if not full["ok"]:
            raise SystemExit("bench.py: full-size property check failed: %r" % full)

    # ---- e2e with the data resident (what `mcmc!` does: upload once, then per sweep only parameters go up and the sample comes back)
    o_l0, o_W, o_A, o_p1, o_p2 = np.empty(K), np.empty(K2), np.empty(K2), np.empty(K2), np.empty(K2)
    sync_all()
    ub = torch.cuda.Event(enable_timing=True); ue = torch.cuda.Event(enable_timing=True)
    ub.record(stream)
    once_steps = max(1, min(args.steps, 3))
    for k in range(once_steps):
        set_params()
        ll = ctypes.c_double()
        ctx.check(lib.nhp_cont_loglik_dist(ctx.h, ev_shard, ev_full, 0, ctypes.byref(ll)))  # N > 1: the rank's share (its columns of the structure once it exists, else its time shard)
        llv = np.array([ll.value])
        ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(llv), 1))
        ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, ev_shard, ev_full, SEED, 2000 + k, float(duration), _ptr(hyper), hyper.size, 1.0, 1.0))
        ctx.check(lib.nhp_cont_params_get(ctx.h, _ptr(o_l0), _ptr(o_W), _ptr(o_A), _ptr(o_p1), _ptr(o_p2)))
    ue.record(stream)
    sync_all()
    once_ms = torch.tensor([ub.elapsed_time(ue)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(once_ms, op=dist.ReduceOp.MAX)
    e2e_once_value = n_total * once_steps / (float(once_ms.item()) * 1e-3)

    # ---- e2e: the public-API call sequence with HOST buffers: parameters + events go up, one step runs (the adjacency structure of the
    #      fresh handle is rebuilt inside it), the sample (parameters + adjacency matrix) comes back; all inside the timed region
    e2e_steps = max(1, min(args.steps, 4))
    if ev_shard is not ev_full:
        lib.nhp_events_free(ctx.h, ev_shard)
    lib.nhp_events_free(ctx.h, ev_full)
    e2e_parts = {"params_set": 0.0, "upload": 0.0, "loglik": 0.0, "gibbs_sweep(incl. adjacency structure build)": 0.0, "readback+free": 0.0}

    def e2e_step(k, timed):
        w0 = time.perf_counter()
        set_params()
        w1 = time.perf_counter()
        if world == 1:
            evf = upload(0, n_total, 0, 1)
            evs = evf
        else:  # every rank uploads its own shard only; the replicated stream of the adjacency sweep is gathered over NVLink
            evs = upload_shard()
            evf = ctypes.c_void_p()
            ctx.check(lib.nhp_comm_allgather_events(ctx.h, evs, ctypes.byref(evf)))
        w2 = time.perf_counter()
        ll = ctypes.c_double()
        ctx.check(lib.nhp_cont_loglik(ctx.h, evs, 0, ctypes.byref(ll)))
        llv = np.array([ll.value])
        ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(llv), 1))
        w3 = time.perf_counter()
        ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, evs, evf, SEED, 1000 + k, float(duration), _ptr(hyper), hyper.size, 1.0, 1.0))
        stream.synchronize()
        w4 = time.perf_counter()
        ctx.check(lib.nhp_cont_params_get(ctx.h, _ptr(o_l0), _ptr(o_W), _ptr(o_A), _ptr(o_p1), _ptr(o_p2)))
        if evs is not evf:
            lib.nhp_events_free(ctx.h, evs)
        lib.nhp_events_free(ctx.h, evf)
        w5 = time.perf_counter()
        if timed:
            for key, dtv in zip(e2e_parts, (w1 - w0, w2 - w1, w3 - w2, w4 - w3, w5 - w4)):
                e2e_parts[key] += 1e3 * dtv / e2e_steps

    e2e_step(-1, False)  # one untimed warm-up step: first-use costs of this call sequence (NCCL broadcast channels, allocator pools)
    sync_all()
    tb = torch.cuda.Event(enable_timing=True); te = torch.cuda.Event(enable_timing=True)
    tb.record(stream)
    for k in range(e2e_steps):
        e2e_step(k, True)
    te.record(stream)
    sync_all()
    e2e_ms = torch.tensor([tb.elapsed_time(te)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = n_total * e2e_steps / (float(e2e_ms.item()) * 1e-3)
    h2d = (n_total if world == 1 else n + n_halo) * 16 + (K + 4 * K2) * 8  # per rank
    d2h = 8 + (K + 4 * K2) * 8

    if rank != 0:
        if world > 1:
            lib.nhp_comm_destroy(ctx.h)
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (per-launch device time measured live with CUDA events on the launching stream)
    med = {k: float(np.median(v)) for k, v in op_ms.items() if v}
    arow = np.median(np.array(adj_rows), axis=0)
    pairs = float(arow[4])               # cached (child event, window predecessor) pairs this rank streams per adjacency sweep
    hbm, hbm_src = hbm_peak()
    density = float(np.count_nonzero(A * W)) / A.size
    probes = n * RATE * DTMAX
    active_pairs = probes * density
    adj_s = med["adjacency"] * 1e-3
    frac5 = float(arow[5]) * 1e3 % 1.0   # adjacency_info[5] = virtual columns + 1e-3 cluster size + 1e-6 bytes per pair
    bpp = float(round(frac5 * 1e3)) if arow[5] > 0 else BYTES_PER_ADJ_PAIR
    if bpp not in (10.0, 18.0):
        bpp = BYTES_PER_ADJ_PAIR
    adj_bytes = pairs * bpp
    dom = "adjacency" if med["adjacency"] >= max(med["loglik"], med["parents"]) else ("parents" if med["parents"] >= med["loglik"] else "loglik")
    # DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this command (same workload: pair counts agree)
    traffic = None
    try:
        cap = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_dominant_kernel.json")))
        if world == 1 and abs(cap["pairs"] - pairs) <= 0.02 * pairs:
            traffic = cap["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        pass
    if dom == "adjacency":
        roofline = {"kernel": "k_adj_sweep<LOGITNORMAL> (adjacency Gibbs sweep, continuous.jl:444-519)", "bound": "hbm", "achieved": adj_bytes / adj_s / 1e9, "peak": hbm,
                    "unit": "GB/s", "frac": adj_bytes / adj_s / 1e9 / hbm, "traffic": traffic, "peak_source": hbm_src, "algorithmic_bytes_per_launch": adj_bytes,
                    "algorithmic_unit": "%.0f B per cached (child event, window predecessor) pair (u16 event index + %s) x %.4g pairs, streamed once per sweep"
                                        % (bpp, "f64 logit + f64 Jacobian of the lag" if bpp == 18.0 else "f64 lag", pairs),
                    "binding_resource": "HBM stream of the cached pairs plus instruction issue: one table-driven exp, one shared-memory intensity look-up and two "
                                        "running products per pair (profiles/r02_ncu_step_kernels.md); fp64_view compares with full LogitNormal pair evaluations",
                    "fp64_view": {"bound": "fp64 impulse evaluations", "achieved": pairs / adj_s, "peak": peaks["ln_pairs_per_s"], "unit": "pairs/s",
                                  "frac": pairs / adj_s / peaks["ln_pairs_per_s"],
                                  "peak_source": "register-resident LogitNormal pair evaluations measured in this run (nhp_bench_fp64 which=1); FP64 FMA peak %.1f TFLOP/s" % peaks["fp64_fma_tflops"]},
                    "kernel_ms": med}
    else:
        secs = med[dom] * 1e-3
        bytes_alg = n * (BYTES_LOGLIK if dom == "loglik" else BYTES_PARENTS)
        roofline = {"kernel": "k_sweep_sparse<LOGITNORMAL, %s>" % dom.upper(), "bound": "hbm", "achieved": bytes_alg / secs / 1e9, "peak": hbm, "unit": "GB/s",
                    "frac": bytes_alg / secs / 1e9 / hbm, "traffic": None, "peak_source": hbm_src, "algorithmic_bytes_per_launch": bytes_alg, "kernel_ms": med}
    # the sparse window sweeps against their own measured ceilings (adjacency-bit probes; active-pair FP64 evaluations)
    sweeps = {}
    for op, extra in (("loglik", BYTES_EXTRA_WLEN), ("parents", BYTES_EXTRA_WLEN + BYTES_EXTRA_POFF)):
        secs = med[op] * 1e-3
        sweeps[op] = {"ms": med[op], "events_per_s": n / secs, "hbm_frac": n * BYTES_LOGLIK / secs / 1e9 / hbm,
                      "algorithmic_bytes_per_event": BYTES_LOGLIK, "implementation_extra_bytes_per_event": extra,
                      "probes_per_s": probes / secs, "probe_ceiling_per_s": peaks["probes_per_s"], "probe_frac": probes / secs / peaks["probes_per_s"],
                      "fp64_tflops": (active_pairs * FLOPS_PER_LN_PAIR + n * FLOPS_PER_EVENT) / secs / 1e12, "fp64_peak_tflops": peaks["fp64_fma_tflops"]}
    if world == 1 and density <= 0.25 and pairs > 0:
        # once the handle carries the pair structure the log-likelihood streams the buckets of the active links (k_adj_loglik) instead of probing
        # every window entry: its probe figures above are window-sweep EQUIVALENTS (events x mean window / time), not probes executed
        secs = med["loglik"] * 1e-3
        sweeps["loglik"]["path"] = "k_adj_loglik: active buckets of the cached pair structure (probes_per_s / probe_frac are window-sweep equivalents)"
        sweeps["loglik"]["structure_bytes"] = pairs * density * bpp
        sweeps["loglik"]["structure_hbm_frac"] = pairs * density * bpp / secs / 1e9 / hbm
    roofline["window_sweeps"] = sweeps
    roofline["adjacency_sweep"] = {"ms": med["adjacency"], "pairs": pairs, "pairs_per_s": pairs / adj_s, "hbm_gbs": adj_bytes / adj_s / 1e9,
                                   "steps": float(arow[0]), "batches": float(arow[1]), "flips": float(arow[2]), "recomputed_steps": float(arow[3]),
                                   "virtual_columns": float(arow[5]), "structure_build_ms": float(arow[7])}
    ms_step = total_ms / args.steps
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(args, world, n_total, n), "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "what": "nhp_cont_params_set + nhp_events_upload (pinned host buffers; N > 1: this rank's time shard, then nhp_comm_allgather_events over "
                            "NVLink for the replicated stream) + nhp_cont_loglik + nhp_cont_gibbs_sweep (builds the adjacency structure of the fresh handle) + "
                            "nhp_cont_params_get (the sample); bytes are per rank",
                    "host_ms_per_step": e2e_parts,
                    "data_resident": {"value": e2e_once_value, "unit": UNIT, "h2d_bytes_per_step": (K + 4 * K2) * 8, "d2h_bytes_per_step": d2h, "steps": once_steps,
                                      "what": "the events stay on the device (as in mcmc!: data is uploaded once); per step nhp_cont_params_set from host "
                                              "arrays + nhp_cont_loglik + nhp_cont_gibbs_sweep + nhp_cont_params_get"}},
            "gpu_launches": int(launches), "roofline": roofline,
            "detail": {"loglik_events_per_s": n_total / (med["loglik"] * 1e-3),
                       "full_gibbs_sweep_ms": ms_step - med["loglik"],
                       "full_gibbs_sweep_events_per_s": n_total / ((ms_step - med["loglik"]) * 1e-3),
                       "phase_ms_rank0": med, "log_likelihood_last_step": ll_last,
                       "data_generation_s": gen_s, "events_total": n_total, "parity_checked": bool(parity and parity.get("ok")), "parity": parity, "full_size_checks": full}}

    if world == 1 and not args.no_cpu_baseline:
        rows, cores, desc, _ = cpu_step_time(args, 1, cpu_sample)
        line["cpu_baseline"] = {"value": 1.0 / rows[0]["per_event_s"], "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
                                "sweeps_s": rows[0]["sweeps_s"], "adjacency_s": rows[0]["adjacency_s"]}
    if world == 1 and not args.no_configs:
        try:
            line["detail"]["configs"] = other_configs_table(ctx, torch, stream, peaks, hbm)
        except Exception as e:  # the table is auxiliary: never lose the headline line to it
            line["detail"]["configs"] = {"error": repr(e)}
    emit(line)
    if world > 1:
        lib.nhp_comm_destroy(ctx.h)
        dist.destroy_process_group()


def last_step_outputs(ctx, K, ll):
    """What a caller of the timed step receives: its log-likelihood and the sample its Gibbs sweep leaves in the context
    (nhp_cont_params_get, nhp_cont_network_get), matrices as X[parent, child]."""
    from nhp_b200.core import _ptr
    l0, W, A, mu, tau = np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
    ctx.check(ctx.lib.nhp_cont_params_get(ctx.h, _ptr(l0), _ptr(W), _ptr(A), _ptr(mu), _ptr(tau)))
    rho = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_network_get(ctx.h, ctypes.byref(rho)))
    unf = lambda v: v.reshape(K, K).T
    return {"loglik": np.array([ll]), "rho": np.array([rho.value]), "lambda0": l0, "W": unf(W), "A": unf(A), "mu": unf(mu), "tau": unf(tau)}


def dump_outputs(out_dir, arrays):
    """out_dir/<name>.npy in float64, DUMP_BYTES at most in all: past that budget an array larger than its even share is written as
    its entries at a fixed, seeded set of flat positions (in ascending order), the same positions in every run of the same shape."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    budget = DUMP_BYTES - 1024 * len(arrays)  # room for the .npy headers
    share = budget // (8 * len(arrays))
    sample = sum(a.nbytes for a in arrays.values()) > budget
    for name, a in arrays.items():
        if sample and a.size > share:
            a = a.ravel()[np.sort(np.random.default_rng(SEED).choice(a.size, share, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def parity_check(args, ctx, params, h_t, h_c):
    """GPU == oracle on the head of the stream that is being timed, with the workload's parameters: log-likelihood to 1e-10,
    parents bit-exact given the same Philox uniforms, counts exact, adjacency columns identical."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_ffi as orc
    import nhp_b200 as nhp
    import synth
    lam0, W, mu, tau, A = params
    K = args.nodes
    sample = cpu_sample_data(args)
    m = int(min(args.cpu_sample, h_t.numel()))
    t, nodes = h_t.numpy()[:m].copy(), h_c.numpy()[:m].copy()
    T = float(t[-1] * (1 + 1e-9))
    orc.set_threads(host_threads())
    om = orc.Cont(1, lam0, W, mu, tau, A=A, dtmax=DTMAX)
    proc = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.LogitNormalImpulseResponse(mu, tau, DTMAX), nhp.DenseWeightModel(W), A,
                                              nhp.BernoulliNetworkModel(RHO, K))
    proc.ctx = ctx
    d = proc.upload((t, nodes, T))
    ll_gpu, ll_ref = nhp.loglikelihood(proc, d), om.loglik(t, nodes, T)
    u = synth.philox_uniform(SEED, np.arange(m, dtype=np.uint64), 3)
    par, pn = nhp.resample_parents(proc, d, seed=SEED, counter=3)
    opar, opn = om.resample_parents(t, nodes, u)
    st = nhp.sufficient_statistics(proc, d)
    ost = orc.suffstats(1, t, nodes, opar, opn, K, DTMAX)
    # adjacency: a 40 000-event head, every 100th column
    ma = min(m, 40000)
    ta, na, Ta = t[:ma], nodes[:ma], float(t[ma - 1] * (1 + 1e-9))
    ua = np.random.default_rng(9).random((K, K))
    A_gpu = nhp.resample_adjacency_matrix_(proc, (ta, na, Ta), u=ua, col_begin=7, col_stride=100).copy()
    A_ref = om.resample_adjacency(A, np.full((K, K), RHO), ta, na, Ta, ua, 7, 100)
    d.free()
    res = {"events": m, "loglik_rel_err": abs(ll_gpu - ll_ref) / abs(ll_ref), "parent_mismatches": int(np.count_nonzero(par != opar)),
           "count_mismatches": int(np.count_nonzero(st["Mnm"] != ost["Mnm"]) + np.count_nonzero(st["M0"] != ost["M0"])),
           "S1_max_rel_err": float(np.max(np.abs(st["S1"] - ost["S1"]) / np.maximum(1.0, np.abs(ost["S1"])))),
           "adjacency_events": ma, "adjacency_columns": len(range(7, K, 100)), "adjacency_mismatches": int(np.count_nonzero(A_gpu != A_ref))}
    res["ok"] = bool(res["loglik_rel_err"] <= 1e-10 and res["parent_mismatches"] == 0 and res["count_mismatches"] == 0 and res["S1_max_rel_err"] <= 1e-10
                     and res["adjacency_mismatches"] == 0)
    if not res["ok"]:
        raise SystemExit("bench.py: GPU result differs from the oracle on the timed workload: %r" % res)
    return res, sample


# ------------------------------------------------------------------------------------------
# the other BASELINE configs: a per-config table in the default run, and their own lines with --config
# ------------------------------------------------------------------------------------------
def _timed(ctx, fn, reps=5):
    ms = []
    for _ in range(reps):
        fn()
        ms.append(ctx.last_kernel_ms)
    return float(np.median(ms[1:])) if len(ms) > 1 else ms[0]


def other_configs_table(ctx, torch, stream, peaks, hbm):
    """cfg2 (dense LogitNormal sweeps, K = 50, 1e6 events), cfg3 (discrete: convolve, FP64 tensor-core contraction, Gibbs, VB,
    adjacency; N = 200, T = 1e6, B = 6) and the cfg5 shape (K = 5000 Exponential, 2e7 events, child-major sweep + analytic gradient),
    each with kernel ms and its own roofline fraction.  Single GPU, device-resident inputs."""
    import nhp_b200 as nhp
    import synth
    from nhp_b200 import discrete as D
    out = {}
    # ---- cfg2
    K, n = 50, 1_000_000
    t, nodes, T = synth.poisson_stream(n, K, 100.0, 1)
    lam0, W, mu, tau, _ = synth.ln_params(K, 2)
    proc = nhp.ContinuousStandardHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.LogitNormalImpulseResponse(mu, tau, 1.0), nhp.DenseWeightModel(W))
    proc.ctx = ctx
    d = proc.upload((t, nodes, T))
    ll_ms = _timed(ctx, lambda: nhp.loglikelihood(proc, d))
    cnt = [0]

    def par():
        cnt[0] += 1
        nhp.resample_parents(proc, d, seed=1, counter=cnt[0], export=False)
    par_ms = _timed(ctx, par)
    pairs = n * 100.0
    out["cfg2"] = {"workload": "continuous LogitNormal standard, K=50, 1e6 events, mean window 100", "loglik_ms": ll_ms, "parents_ms": par_ms,
                   "loglik_pairs_per_s": pairs / (ll_ms * 1e-3), "parents_events_per_s": n / (par_ms * 1e-3),
                   "roofline": {"bound": "fp64 impulse evaluations", "achieved": pairs / (ll_ms * 1e-3), "peak": peaks["ln_pairs_per_s"], "unit": "pairs/s",
                                "frac": pairs / (ll_ms * 1e-3) / peaks["ln_pairs_per_s"]}}
    d.free()
    # ---- cfg5 shape
    K, n = 5000, 20_000_000
    t, nodes, T = synth.poisson_stream(n, K, 3.2, 1)
    lam0, W, theta, _ = synth.exp_params(K, 2)
    proc = nhp.ContinuousStandardHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.ExponentialImpulseResponse(theta), nhp.DenseWeightModel(W))
    proc.ctx = ctx
    d = proc.upload((t, nodes, T))
    ll_ms = _timed(ctx, lambda: nhp.loglikelihood(proc, d, recursive=True), reps=3)
    proc._push(ctx)

    def grad():
        ctx.check(ctx.lib.nhp_cont_loglik_grad_dev(ctx.h, d.h, 1))
        ctx.lib.nhp_cont_loglik_grad_read(ctx.h, d.h, None, None, None, None, None)
    g_ms = _timed(ctx, grad, reps=3)
    hz = ctypes.c_double()
    ctx.check(ctx.lib.nhp_cont_horizon(ctx.h, n, 1, ctypes.byref(hz)))
    pairs = n * 3.2 * hz.value
    out["cfg5_shape"] = {"workload": "continuous Exponential standard, K=5000, 2e7 events (1/50 of cfg5), recursive semantics, cut-off window %.0f pairs/event" % (3.2 * hz.value),
                         "loglik_ms": ll_ms, "loglik_plus_gradient_ms": g_ms, "loglik_events_per_s": n / (ll_ms * 1e-3),
                         "roofline": {"bound": "hbm (window reads of the child-major sweep, 12 B per pair)", "achieved": pairs * 12.0 / (ll_ms * 1e-3) / 1e9, "peak": hbm,
                                      "unit": "GB/s", "frac": pairs * 12.0 / (ll_ms * 1e-3) / 1e9 / hbm,
                                      "fp64_pairs_per_s": pairs / (ll_ms * 1e-3), "fp64_pair_ceiling": peaks["exp_pairs_per_s"]}}
    d.free()
    del t, nodes
    # ---- cfg3
    N, Tb, B, L = 200, 1_000_000, 6, 12
    rng = np.random.default_rng(3)
    lam0 = np.full(N, 0.02)
    A = (rng.random((N, N)) < 0.1).astype(np.float64)
    W = rng.uniform(0.0, 0.5, (N, N)) * A
    W *= 0.5 / max(1e-9, np.max(np.abs(np.linalg.eigvals(W))))
    theta = rng.dirichlet(np.ones(B), (N, N))
    data = rng.poisson(0.04, (N, Tb)).astype(np.int64)
    proc = D.DiscreteNetworkHawkesProcess(D.DiscreteHomogeneousProcess(lam0), D.DiscreteGaussianImpulseResponse(theta, L), nhp.DenseWeightModel(W), A,
                                          nhp.BernoulliNetworkModel(0.1, N))
    proc.ctx = ctx
    d = proc.upload(data)
    conv_ms = _timed(ctx, lambda: D.convolve(proc, d, export=False), reps=3)
    ll_ms = _timed(ctx, lambda: D.loglikelihood(proc, d), reps=4)
    cnt = [0]

    def gib():
        cnt[0] += 1
        D.resample_parents(proc, d, seed=1, counter=cnt[0])
    gibbs_ms = _timed(ctx, gib, reps=3)
    e0, E = np.ones(N), rng.uniform(0.01, 0.2, (N, N, B))
    vb_ms = _timed(ctx, lambda: D.vb_statistics(proc, d, e0, E), reps=3)

    def adj():
        cnt[0] += 1
        D.resample_adjacency_matrix_(proc, d, seed=2, counter=cnt[0])
    adj_ms = _timed(ctx, adj, reps=3)
    flops = 2.0 * Tb * N * N * B
    conv_bytes = 4.0 * N * Tb + 8.0 * Tb * N * B
    out["cfg3"] = {"workload": "discrete Gaussian network Hawkes, N=200, T=1e6 bins, B=6, L=12, ~4 % non-zero bins",
                   "convolve_ms": conv_ms, "loglik_contraction_ms": ll_ms, "gibbs_counts_ms": gibbs_ms, "vb_stats_ms": vb_ms, "adjacency_ms": adj_ms,
                   "bins_per_s_loglik": Tb / (ll_ms * 1e-3),
                   "roofline": {"bound": "fp64 tensor (DMMA m8n8k4)", "achieved": flops / (ll_ms * 1e-3) / 1e12, "peak": peaks["dmma_tflops"], "unit": "TFLOP/s",
                                "frac": flops / (ll_ms * 1e-3) / 1e12 / peaks["dmma_tflops"]},
                   "convolve_roofline": {"bound": "hbm", "achieved": conv_bytes / (conv_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                         "frac": conv_bytes / (conv_ms * 1e-3) / 1e9 / hbm}}
    d.free()
    return out


def run_reference_other(args):
    emit({"impl": "reference", "unavailable": "the CPU reference arm is implemented for the headline workload (--config 4) only"})


def run_ours_other(args, rank, world, local_rank):
    """--config 2 | 3 | 5 as their own JSON line (N >= 1): time-sharded log-likelihood / sweeps with the library's NCCL collectives."""
    import bench_configs
    bench_configs.run(args, rank, world, local_rank, emit, setup_distributed, make_context, ClockSampler, hbm_peak)


def main():
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # NCCL / torch banners must not pollute the single JSON line
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.config == 4:
        run_ours(args, rank, world, local_rank)
    else:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        run_ours_other(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
