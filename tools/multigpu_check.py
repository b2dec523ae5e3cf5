#!/usr/bin/env python3
"""Multi-GPU parity check of the library's own collectives (csrc/comm.cu), run under torchrun on N >= 2 GPUs:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/multigpu_check.py

Every rank builds the same small data set; rank r then works on its time shard / its columns through nhp_comm_* (NCCL inside
libnhp) and the result is compared with the single-GPU computation of the same thing on the same rank:
  * log-likelihood: sum of the shard shares (nhp_comm_allreduce_host) == unsharded, 1e-12
  * parent sweep + statistics: all-reduced counts == unsharded counts exactly (same Philox uniforms: keyed by the global event index)
  * adjacency sweep: column partition + nhp_comm_allgather_adjacency == full sweep, identical matrix
  * nhp_cont_gibbs_sweep: the composite call leaves identical parameters on every rank (checked through an all-reduce of a checksum)
  * LogGaussianCoxProcess curves with a prior: nhp_cont_resample_baseline on the time shards (per-node sums all-reduced) == the update
    of the unsharded stream on a context without communicator, 1e-12 with identical attempt counts; then three composite sweeps
    leave identical curves on every rank
  * discrete time shards with an L-bin halo: log-likelihood and Gibbs counts summed over ranks == unsharded
Prints one JSON line on rank 0; exit code 1 on any mismatch."""
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "networkhawkesprocesses.jl_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import bench
    import nhp_b200 as nhp
    import synth
    from nhp_b200 import discrete as D
    from nhp_b200.core import ContinuousData, _fmat, _ptr
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch, dist, dev = bench.setup_distributed(local, world)
    ctx, stream = bench.make_context(torch, dev, local, rank, world, dist)
    lib = ctx.lib
    res = {"world": world}
    ok = True

    # ---------------- continuous network process
    K, n, rho = 40, 60000, 0.2
    t, nodes, T = synth.poisson_stream(n, K, 80.0, 5)
    lam0, W, mu, tau, A = synth.ln_params(K, 6, wmax=1.0 / (K * rho), density=rho)
    proc = nhp.ContinuousNetworkHawkesProcess(nhp.HomogeneousProcess(lam0), nhp.LogitNormalImpulseResponse(mu, tau, 1.0), nhp.DenseWeightModel(W), A,
                                              nhp.BernoulliNetworkModel(rho, K))
    proc.ctx = ctx
    full = ContinuousData(ctx, t, nodes, T, K)
    i0, i1 = rank * n // world, (rank + 1) * n // world
    lo = int(np.searchsorted(t, t[i0] - 1.0, side="right")) if rank > 0 else 0
    shard = ContinuousData(ctx, t[lo:i1], nodes[lo:i1], T, K, n_halo=i0 - lo, index_base=lo, flags=1 if rank == 0 else 0)
    proc._push(ctx)
    ll_full, ll_sh = ctypes.c_double(), ctypes.c_double()
    ctx.check(lib.nhp_cont_loglik(ctx.h, full.h, 0, ctypes.byref(ll_full)))
    ctx.check(lib.nhp_cont_loglik(ctx.h, shard.h, 0, ctypes.byref(ll_sh)))
    v = np.array([ll_sh.value])
    ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(v), 1))
    res["loglik_rel_err"] = abs(v[0] - ll_full.value) / abs(ll_full.value)
    ok &= res["loglik_rel_err"] < 1e-12

    def stats():
        M0, Mn, Mnm, S1, S2 = np.empty(K), np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
        ctx.check(lib.nhp_cont_suffstats_read(ctx.h, _ptr(M0), _ptr(Mn), _ptr(Mnm), _ptr(S1), _ptr(S2)))
        return M0, Mn, Mnm, S1, S2

    ctx.check(lib.nhp_cont_resample_parents(ctx.h, full.h, 11, 3, None, None, None))
    ctx.check(lib.nhp_cont_suffstats_second_pass(ctx.h, full.h))
    ref = stats()
    ctx.check(lib.nhp_cont_resample_parents(ctx.h, shard.h, 11, 3, None, None, None))
    ctx.check(lib.nhp_comm_allreduce_stats(ctx.h, 0))
    ctx.check(lib.nhp_cont_suffstats_second_pass(ctx.h, shard.h))
    ctx.check(lib.nhp_comm_allreduce_stats(ctx.h, 1))
    got = stats()
    res["count_mismatches"] = int(sum(np.count_nonzero(a != b) for a, b in zip(ref[:3], got[:3])))
    res["S1_max_rel_err"] = float(np.max(np.abs(ref[3] - got[3]) / np.maximum(1.0, np.abs(ref[3]))))
    res["S2_max_rel_err"] = float(np.max(np.abs(ref[4] - got[4]) / np.maximum(1.0, np.abs(ref[4]))))
    ok &= res["count_mismatches"] == 0 and res["S1_max_rel_err"] < 1e-11 and res["S2_max_rel_err"] < 1e-9

    # the replicated stream gathered from the shards over NVLink == the uploaded full stream
    if world > 1:
        gathered = ctypes.c_void_p()
        ctx.check(lib.nhp_comm_allgather_events(ctx.h, shard.h, ctypes.byref(gathered)))
        tg, cg = np.empty(n), np.empty(n, dtype=np.int64)
        Tg = ctypes.c_double()
        ctx.check(lib.nhp_events_download(ctx.h, gathered, _ptr(tg), cg.ctypes.data_as(ctypes.c_void_p), ctypes.byref(Tg)))
        ll_g = ctypes.c_double()
        ctx.check(lib.nhp_cont_loglik(ctx.h, gathered, 0, ctypes.byref(ll_g)))
        res["gathered_stream_mismatches"] = int(np.count_nonzero(tg != t) + np.count_nonzero(cg != nodes)) + int(lib.nhp_events_count(gathered) != n)
        res["gathered_loglik_rel_err"] = abs(ll_g.value - ll_full.value) / abs(ll_full.value)
        ok &= res["gathered_stream_mismatches"] == 0 and res["gathered_loglik_rel_err"] < 1e-14
        lib.nhp_events_free(ctx.h, gathered)

    # adjacency: full sweep on this GPU vs column partition + all-gather
    def get_A():
        out = np.empty(K * K)
        ctx.check(lib.nhp_cont_params_get(ctx.h, None, None, _ptr(out), None, None))
        return out

    proc._push(ctx)
    ctx.check(lib.nhp_cont_resample_adjacency_dev(ctx.h, full.h, rho, 21, 4, 0, 1, 1))
    A_full = get_A()
    proc._push(ctx)
    ctx.check(lib.nhp_cont_resample_adjacency_dev(ctx.h, full.h, rho, 21, 4, rank, world, 0))
    ctx.check(lib.nhp_comm_allgather_adjacency(ctx.h))
    A_part = get_A()
    res["adjacency_mismatches"] = int(np.count_nonzero(A_full != A_part))
    res["adjacency_links"] = int(A_full.sum())
    ok &= res["adjacency_mismatches"] == 0

    # distributed log-likelihood: the share through this rank's columns of the structure (built by the partitioned sweep above)
    proc._push(ctx)
    ctx.check(lib.nhp_cont_loglik(ctx.h, full.h, 0, ctypes.byref(ll_full)))
    share = ctypes.c_double()
    ctx.check(lib.nhp_cont_loglik_dist(ctx.h, shard.h, full.h, 0, ctypes.byref(share)))
    v = np.array([share.value])
    ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(v), 1))
    res["loglik_dist_rel_err"] = abs(v[0] - ll_full.value) / abs(ll_full.value)
    ok &= res["loglik_dist_rel_err"] < 1e-12

    # composite sweep: identical parameters on every rank
    proc._push(ctx)
    ctx.check(lib.nhp_cont_network_set(ctx.h, rho))
    hyper = np.ones(8)
    for sweep in range(3):
        ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, shard.h, full.h, 31, sweep, float(T), _ptr(hyper), hyper.size, 1.0, 1.0))
    l0, Wd, Ad, p1, p2 = np.empty(K), np.empty(K * K), np.empty(K * K), np.empty(K * K), np.empty(K * K)
    ctx.check(lib.nhp_cont_params_get(ctx.h, _ptr(l0), _ptr(Wd), _ptr(Ad), _ptr(p1), _ptr(p2)))
    chk = np.array([l0.sum(), Wd.sum(), Ad.sum(), p1.sum(), p2.sum()])
    tot = chk.copy()
    ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(tot), tot.size))
    res["composite_param_spread"] = float(np.max(np.abs(tot / world - chk) / np.maximum(1.0, np.abs(chk))))
    res["composite_links"] = int(Ad.sum())
    ok &= res["composite_param_spread"] < 1e-12 and np.all(np.isfinite(chk))

    # ---------------- LGCP network with a prior: the slice update of the curves on the time shards
    G = 41
    rg = np.random.default_rng(8)
    xg = np.linspace(0.0, T, G)
    cv = lam0[:, None] * (1.0 + 0.3 * np.sin(2 * np.pi * rg.uniform(1.0, 4.0, (K, 1)) * xg[None, :] / T + rg.uniform(0, 2 * np.pi, (K, 1))))
    zs, us = rg.standard_normal(K * G), rg.random(K * 101)

    def lgcp_update(c, ev):
        lg = nhp.ContinuousNetworkHawkesProcess(nhp.LogGaussianCoxProcess(xg, cv, m=float(np.log(lam0.mean())), eta=T / 10.0),
                                                nhp.LogitNormalImpulseResponse(mu, tau, 1.0), nhp.DenseWeightModel(W), A, nhp.BernoulliNetworkModel(rho, K))
        lg.ctx = c
        lg._push(c)
        c.check(c.lib.nhp_cont_resample_parents(c.h, ev.h, 41, 2, None, None, None))
        lg.baseline.resample_device_(c, ev, z=zs, u=us)
        return lg, lg.baseline.lam_grid.copy(), lg.baseline.last_attempts.copy()

    single = nhp.Context(local)
    full1 = ContinuousData(single, t, nodes, T, K)
    _, cur_ref, att_ref = lgcp_update(single, full1)
    full1.free()
    lg, cur, att = lgcp_update(ctx, shard)
    res["lgcp_curves_max_rel_err"] = float(np.max(np.abs(cur - cur_ref) / cur_ref))
    res["lgcp_attempt_mismatches"] = int(np.count_nonzero(att != att_ref))
    res["lgcp_attempts_max"] = int(att.max())
    ok &= res["lgcp_curves_max_rel_err"] < 1e-12 and res["lgcp_attempt_mismatches"] == 0
    ctx.check(lib.nhp_cont_network_set(ctx.h, rho))
    for sweep in range(3):
        ctx.check(lib.nhp_cont_gibbs_sweep(ctx.h, shard.h, full.h, 32, sweep, float(T), _ptr(hyper), hyper.size, 1.0, 1.0))
    cur = lg.baseline.pull_(ctx).ravel()
    tot = cur.copy()
    ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(tot), tot.size))
    res["lgcp_composite_curve_spread"] = float(np.max(np.abs(tot / world - cur) / cur))
    ok &= res["lgcp_composite_curve_spread"] < 1e-12

    # ---------------- intensity(process, data, times): the query times are sharded, the stream is replicated, no exchange but the gather
    proc._push(ctx)
    nq = 2001
    tq = np.linspace(0.0, T, nq)
    lam_full = nhp.intensity(proc, full, tq)                      # [nq, K]
    q0, q1 = rank * nq // world, (rank + 1) * nq // world
    lam_mine = nhp.intensity(proc, full, tq[q0:q1])
    gathered_q = np.zeros((nq, K))
    gathered_q[q0:q1] = lam_mine
    flat = np.ascontiguousarray(gathered_q.ravel())
    ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(flat), flat.size))  # disjoint slices: the sum is the gather
    res["query_shard_max_abs_err"] = float(np.max(np.abs(flat.reshape(nq, K) - lam_full)))
    ok &= res["query_shard_max_abs_err"] == 0.0

    # ---------------- discrete process: time shards with an L-bin halo
    N, Tb, B, L = 12, 6000, 4, 8
    rng = np.random.default_rng(4)
    l0d, Wdd, thd = rng.uniform(0.05, 0.15, N), rng.uniform(0.0, 0.6 / N, (N, N)), rng.dirichlet(np.ones(B), (N, N))
    data = rng.poisson(0.1, (N, Tb)).astype(np.int64)
    pd_ = D.DiscreteStandardHawkesProcess(D.DiscreteHomogeneousProcess(l0d), D.DiscreteGaussianImpulseResponse(thd, L), nhp.DenseWeightModel(Wdd))
    pd_.ctx = ctx
    dfull = D.DiscreteData(ctx, data)
    ll_ref = D.loglikelihood(pd_, dfull)
    t0, t1 = rank * Tb // world, (rank + 1) * Tb // world
    halo = min(L, t0)
    dsh = D.DiscreteData(ctx, data[:, t0 - halo:t1], t_halo=halo)
    v = np.array([D.loglikelihood(pd_, dsh)])
    ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(v), 1))
    res["disc_loglik_rel_err"] = abs(v[0] - ll_ref) / abs(ll_ref)
    st_ref = D.vb_statistics(pd_, dfull, np.ones(N), np.full((N, N, B), 0.1))
    st_sh = D.vb_statistics(pd_, dsh, np.ones(N), np.full((N, N, B), 0.1))
    g = np.ascontiguousarray(st_sh["gamma_sum"])
    ctx.check(lib.nhp_comm_allreduce_host(ctx.h, _ptr(g), g.size))
    res["disc_vb_max_rel_err"] = float(np.max(np.abs(g - st_ref["gamma_sum"]) / np.maximum(1e-12, np.abs(st_ref["gamma_sum"]))))
    ok &= res["disc_loglik_rel_err"] < 1e-12 and res["disc_vb_max_rel_err"] < 1e-10

    flag = torch.tensor([0 if ok else 1], device=dev)
    if world > 1:
        dist.all_reduce(flag)
    res["ok"] = bool(flag.item() == 0)
    if rank == 0:
        print(json.dumps(res), flush=True)
    if world > 1:
        lib.nhp_comm_destroy(ctx.h)
        dist.destroy_process_group()
    sys.exit(0 if res["ok"] else 1)


if __name__ == "__main__":
    main()
