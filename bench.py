#!/usr/bin/env python
"""bench.py -- PodGang placements/sec on the 50k-node / 10k-gang synthetic snapshot (BASELINE.json).

A "step" is one scheduling cycle: every pending PodGang of the snapshot goes through fit -> (score) -> admit -> commit
and comes out admitted or rejected, with the result of the SEQUENTIAL priority-ordered pass (oracle/grove_oracle_seq.c).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C4] [--impl reference]

`value`       whole-job admitted gangs / second, node table already resident in HBM (per step: device->device reset of
              the node table, then the cycle).
`e2e`         the same metric through the C ABI with HOST buffers every step: grove_load_nodes + grove_submit_gangs +
              grove_run_cycle + grove_get_placements + grove_get_gang_status.
`roofline`    the HBM-bound kernel of the path (K2, the score matrix) timed alone with CUDA events, against the measured copy
              bandwidth in MEASURED_PEAKS.json -- K2 is built on request and is NOT on the cycle's critical path (the admission
              never reads it); the whole-cycle fractions and K3's own figures of merit are next to it.
`cpu_baseline`/--impl reference   the CPU oracle (a C restatement: the reference tree holds no scheduler and there is no Go
              toolchain) on this box's host cores.  The gang loop of the sequential pass cannot be parallelised; OpenMP
              threads split each gang's fit/score rows over the nodes.
--gpus N      N > 1: replicas (DESIGN.md section 7): one cluster is one sequential dependency chain of ~1.6 MB of state, so
              every rank schedules ITS OWN cluster snapshot (same shape, rank-specific seed), no data-path collective;
              value = gangs admitted by all ranks / max-over-ranks time, scaling "weak".
--config C4X  the part of the path that DOES shard: the score pass (K1 + K2) on a cluster 4x C4, node-range shards, one rank per
              GPU, ONE all-reduce of per-shard feasibility / capacity counts (NCCL); strong scaling, pairs scored per second.
--config C5   steady-state churn (BASELINE.json config 5); C1..C3 the smaller configurations.
--dump-outputs DIR   C1..C4 on the GPU: after the timed steps, what the last one computed (placements, gang status, scope
              domains, committed node table; rank 0's cluster) goes to DIR as one float64 .npy per field.  The inputs are
              seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from grove_b200 import synth, tables as T  # noqa: E402


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_workload(name: str, replica: int = 0):
    """replica r > 0: an independent cluster of the same shape (rank-specific seed)"""
    cfg = synth.CONFIGS[name]() if replica == 0 or name == "C1" else synth.CONFIGS[name](seed=synth.SEED_BASE + int(name[1]) + 1000 * replica)
    g, c, s = cfg["tables"]
    return cfg["nodes"], cfg["n_levels"], g, c, s


def host_cores() -> int:
    """threads this process may actually run on: its affinity mask, capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except (OSError, ValueError):
        pass
    return n


def workload_desc(name, n_nodes, n_gangs, n_cliques, n_gpus):
    """identical for both arms (the driver compares the dicts): what is scheduled, nothing about how it went"""
    return {"workload": f"{name}: {n_nodes} nodes / {n_gangs} PodGangs / {n_cliques} PodCliques, "
                        + {"C4": "4-level tree zone/block/rack/host, hierarchical PCSG gangs (base + scaled)",
                           "C3": "3-level tree, prefill+decode cliques", "C2": "flat", "C1": "simple1.yaml"}[name],
            "nodes": int(n_nodes), "gangs": int(n_gangs), "cliques": int(n_cliques),
            "pairs_per_full_pass": int(n_nodes) * int(n_cliques),
            "semantics": "sequential pass in (priority desc, submission index asc) order",
            "parallelism": "1 cluster on 1 GPU" if n_gpus == 1 else f"replicas only: {n_gpus} independent clusters, one per GPU",
            "l2": "inputs change every step (node table reset, claims rebuilt); the 126 MB L2 holds the working set by design"}


DUMP_BYTES = 60 << 20


def dump_outputs(out_dir, tables):
    """every field of the result tables as DIR/<table>.<field>.npy in float64 (exact: the fields are integers below 2**53);
    a table whose fields would exceed its share of DUMP_BYTES is cut to a fixed, seeded sample of its rows, whose indices
    go to DIR/<table>.rows.npy"""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(tables)
    for name, a in tables.items():
        row_bytes = 8 * (1 + sum(int(np.prod(a.dtype[f].shape)) for f in a.dtype.names))
        if len(a) * row_bytes > share:
            rows = np.sort(np.random.default_rng(0).choice(len(a), share // row_bytes, replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, f"{name}.rows.npy"), rows.astype(np.float64))
        for f in a.dtype.names:
            np.save(os.path.join(out_dir, f"{name}.{f}.npy"), a[f].astype(np.float64))


def prefix_sample(g, c, s, keep):
    """the first `keep` PodGangs of the table (grown until every base-gang reference stays inside): a self-contained
    sub-workload for the bounded CPU legs"""
    keep = min(keep, len(g))
    while keep < len(g):
        bg = g["base_gang"][:keep]
        if not ((bg != T.NONE_U32) & (bg >= keep)).any():
            break
        keep += 1
    gs = g[:keep].copy()
    nc = int(gs["clique_off"][-1] + gs["n_cliques"][-1]); ns = int(gs["scope_off"][-1] + gs["n_scopes"][-1])
    return gs, c[:nc], s[:ns]


def time_oracle(nodes, L, g, c, s, threads, budget_s):
    """one timed oracle run sized to ~budget_s: the full workload when it fits, else a prefix sample (the sequential pass
    costs the same per gang wherever it stands in the order); -> (gangs/s, description, result of the run, full?)"""
    from oracle import oracle_py as O
    probe_g, probe_c, probe_s = prefix_sample(g, c, s, min(len(g), 200))
    t0 = time.perf_counter(); O.run_cycle(nodes, L, probe_g, probe_c, probe_s, threads=threads); per_gang = (time.perf_counter() - t0) / len(probe_g)
    keep = len(g) if per_gang * len(g) <= budget_s else max(200, int(budget_s / per_gang))
    full = keep >= len(g)
    sg, sc, ss = (g, c, s) if full else prefix_sample(g, c, s, keep)
    t0 = time.perf_counter(); r = O.run_cycle(nodes, L, sg, sc, ss, threads=threads); dt = time.perf_counter() - t0
    what = ("the full workload" if full else f"the first {len(sg)} of {len(g)} PodGangs (rank-order prefix, all base gangs inside)") + \
           f" against all {len(nodes)} nodes, {dt:.2f} s"
    return r["stats"]["gangs_admitted"] / dt, what, r, full


def run_reference(args):
    """--impl reference: the CPU oracle with all the host threads it can use.  The reference tree holds no scheduler (the
    path lives in KAI-Scheduler, not vendored) and is Go with no toolchain here, so this arm times the C restatement.  A step
    is one cycle over the full workload when K steps fit a few minutes, else a bounded sample of it."""
    from oracle import oracle_py as O
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nodes, L, g, c, s = make_workload(args.config)
    cores = host_cores()
    O.build()
    desc = workload_desc(args.config, len(nodes), len(g), len(c), args.gpus)
    total_steps = max(1, args.steps + args.warmup)
    budget = 150.0 / total_steps
    _, what, _, full = time_oracle(nodes, L, g, c, s, cores, budget)
    sg, sc, ss = (g, c, s) if full else prefix_sample(g, c, s, int(what.split()[2]))
    for _ in range(args.warmup):
        O.run_cycle(nodes, L, sg, sc, ss, threads=cores)
    t0 = time.perf_counter()
    adm = 0
    for _ in range(args.steps):
        r = O.run_cycle(nodes, L, sg, sc, ss, threads=cores)
        adm = r["stats"]["gangs_admitted"]
    dt = (time.perf_counter() - t0) / args.steps
    val = adm / dt
    line = {
        "impl": "reference", "metric": "podgang_placements_per_sec", "value": val, "unit": "gangs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak" if args.gpus > 1 else "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": desc,
        "cpu_baseline": {"value": val, "unit": "gangs/s", "cores": cores, "kind": "port",
                         "sample": "per step: " + what.rsplit(",", 1)[0] + "; sequential gang loop, OpenMP over the nodes of each "
                                   "gang's fit/score rows; C restatement (no scheduler in the reference tree, Go toolchain absent)"},
        "e2e": {"value": val, "unit": "gangs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def ncu_traffic():
    """DRAM bytes (read + write) of one k_score launch over the whole C4 submission, from the committed `ncu --set full`
    capture (profiles/r2_ncu_k_score_raw.csv); None when the capture is absent."""
    import csv
    for name in ("r2_ncu_k_score_raw.csv", "r1_ncu_k_score_raw.csv"):
        try:
            rows = list(csv.reader(open(os.path.join(ROOT, "profiles", name))))
            h, units, vals = rows[0], rows[1], rows[2]
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            tot = sum(float(vals[h.index(k)].replace(",", "")) * scale[units[h.index(k)]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
            return tot, name
        except (OSError, ValueError, KeyError, IndexError):
            continue
    return None, None


def run_gpu(args):
    import torch
    from grove_b200 import build
    from grove_b200.engine import PlacementEngine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path (use --impl reference for the CPU oracle)")
    # one rank per GPU shares the box's cores: the engine's host thread team (table validation, derived tables) is sized to this
    # rank's share, and one core per rank stays free for the thread that follows the relaxation
    os.environ.setdefault("GROVE_HOST_THREADS", str(max(1, min(8, host_cores() // max(world, 1) - 1))))
    build.build()
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist_.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_
    # replicas only (DESIGN.md section 7): rank r schedules its own cluster, no data-path collective
    nodes, L, g, c, s = make_workload(args.config, replica=rank)
    eng = PlacementEngine(L, device=local)
    eng.load_nodes(nodes)
    eng.submit_gangs(g, c, s)
    d_nodes = torch.from_numpy(nodes.view(np.uint8).reshape(-1)).cuda()  # pristine snapshot, resident in HBM
    h2d = nodes.nbytes + g.nbytes + c.nbytes + s.nbytes

    def step_dev():
        eng.load_nodes_device(d_nodes.data_ptr(), len(nodes))
        return eng.run_cycle()

    def step_e2e():
        eng.load_nodes(nodes); eng.submit_gangs(g, c, s)
        st = eng.run_cycle()
        return st, eng.placements(copy=False), eng.gang_status(copy=False)

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # sampled from the warm-up on: a cycle is milliseconds, nvidia-smi samples every 20 ms
    for _ in range(args.warmup):
        step_dev()
    sync()
    t0 = time.perf_counter()
    acc = {k: 0.0 for k in ("ms_fit", "ms_admit", "ms_commit", "ms_total")}
    launches = evals = 0
    for _ in range(args.steps):
        st = step_dev()
        for k in acc:
            acc[k] += st[k]
        launches += st["kernel_launches"] + 1  # + k_gather of the node-table reset
        evals += st["evaluations"]
    sync()
    dt = time.perf_counter() - t0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"placements": eng.placements(), "gang_status": eng.gang_status(),
                                         "scope_domains": eng.scope_domains(), "nodes": eng.nodes()})
    # e2e through the C ABI with host buffers
    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    sync()
    t1 = time.perf_counter()
    for _ in range(args.steps):
        st_e, pl, gs = step_e2e()
    sync()
    dt_e = time.perf_counter() - t1
    clocks = sampler.stop() if rank == 0 else None  # covers warm-up, the timed steps and the e2e steps
    adm_all, rej_all = st["gangs_admitted"], st["gangs_rejected"]
    if dist is not None:
        tt = torch.tensor([dt, dt_e], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt, dt_e = tt.tolist()
        cnt = torch.tensor([adm_all, rej_all], device="cuda", dtype=torch.int64)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        adm_all, rej_all = cnt.tolist()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    ms_step = dt / args.steps * 1e3
    ms_e2e = dt_e / args.steps * 1e3
    peak, peak_src = peaks()
    # K2 (score matrix): per (clique,node) pair it reads 1 fit bit and writes 1 score byte.  Built on request; timed alone
    # here with CUDA events on the engine's stream, K steps after W warm-ups.
    pairs = len(c) * len(nodes)
    k2_bytes = pairs * (1.0 + 1.0 / 8.0)
    for _ in range(args.warmup):
        eng.build_score_matrix()
    k2_ms = float(np.mean([eng.build_score_matrix() for _ in range(args.steps)]))
    achieved = k2_bytes / (k2_ms * 1e-3) / 1e9 if k2_ms > 0 else 0.0
    traffic, traffic_src = ncu_traffic() if args.config == "C4" else (None, None)
    d2h = pl.nbytes + gs.nbytes
    ms_cycle = acc["ms_total"] / args.steps
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import oracle_py as O
        O.build()
        cores = host_cores()
        v1, what1, _, _ = time_oracle(nodes, L, g, c, s, 1, 10.0)
        vn, whatn, r, full = time_oracle(nodes, L, g, c, s, cores, 20.0)
        same = None
        if full:   # the multi-thread leg ran the whole workload: compare every output with the GPU's
            same = bool(np.array_equal(r["placements"], pl) and np.array_equal(r["status"], gs))
        cpu = {"value": vn, "unit": "gangs/s", "cores": cores, "kind": "port", "sample": whatn + "; sequential gang loop, OpenMP "
               "over the nodes of each gang's fit/score rows; C restatement timed on this box (reference tree has no scheduler; Go toolchain absent)",
               "single_thread": {"value": v1, "cores": 1, "sample": what1},
               "outputs_identical_to_gpu": same}
    line = {
        "metric": "podgang_placements_per_sec", "value": adm_all / (ms_step * 1e-3), "unit": "gangs/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak" if world > 1 else "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_desc(args.config, len(nodes), len(g), len(c), world),
        "result": {"admitted": int(adm_all), "rejected": int(rej_all), "pods_bound_rank0": st["pods_bound"],
                   "gangs_decided_per_sec": (adm_all + rej_all) / (ms_step * 1e-3), "relaxation_rounds_rank0": st["rounds"],
                   "gang_evaluations_per_cycle_rank0": evals / args.steps},
        "clocks": clocks,
        "e2e": {"value": adm_all / (ms_e2e * 1e-3), "unit": "gangs/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": int(d2h) * world},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "k_score (K2 topology-distance score matrix), timed alone", "bound": "hbm", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_note": None if traffic is None else f"DRAM read+write of one k_score launch over the whole submission, profiles/{traffic_src}",
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": k2_bytes, "ms_per_launch": k2_ms,
                     "on_critical_path": False,
                     "note": "the admission (K3) derives its visiting order from the anchor's domain ranges and never reads the score matrix: K2 is "
                             "built on request (grove_build_score_matrix) and is not part of `value`; it is write-dominated (1 B written per 1/8 B read), "
                             "so ~0.6 of the copy peak is its DRAM ceiling",
                     "whole_cycle": {"ms_device": ms_cycle,
                                     "frac_k2_bytes_model": (k2_bytes / (ms_cycle * 1e-3) / 1e9) / peak,
                                     "frac_survey_model_2.375B_per_pair": (2.375 * pairs / (ms_cycle * 1e-3) / 1e9) / peak,
                                     "note": "what the cycle would reach IF it moved the 3-kernel formulation's bytes; it does not: fit rows are per signature, "
                                             "K3 reads only the domains it visits -- the cycle is a latency chain of relaxation rounds, not an HBM stream"},
                     "k3": {"gang_evaluations_per_sec": evals / args.steps / (ms_cycle * 1e-3), "ms_admit_per_cycle": acc["ms_admit"] / args.steps,
                            "rounds_per_cycle": st["rounds"]}},
        "kernel_ms_per_step": {k: v / args.steps for k, v in acc.items()},
        "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def run_sharded(args):
    """--config C4X: the multi-GPU SCORE PASS on a cluster 4x C4 (200 000 nodes / 40 000 PodGangs / 110 000 PodCliques; a 22 GB score
    matrix): K1 + K2 over node-range shards, one rank per GPU, and the ONE all-reduce of per-shard feasibility / capacity counts
    (grove_b200/sharded.py; BASELINE.json north_star's sharding).  The admission (K3) does not shard and is not part of this line.
    A step = grove_run_score_pass + grove_shard_summary_device + all_reduce(SUM) on every rank; value = (clique, node) pairs scored
    per second by the whole job (strong scaling: the matrix is fixed, the ranks split its columns)."""
    import torch
    from grove_b200 import build
    from grove_b200.engine import PlacementEngine
    from grove_b200.sharded import engine_summary, infeasible_from_sum, sharded_score_pass
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path")
    os.environ.setdefault("GROVE_HOST_THREADS", str(max(1, min(8, host_cores() // max(world, 1) - 1))))
    build.build()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist_.init_process_group("nccl", device_id=dev)
        dist = dist_
    cfg = synth.config_c4(n=200000, g=40000)
    nodes, L = cfg["nodes"], cfg["n_levels"]
    g, c, s = cfg["tables"]
    eng = PlacementEngine(L, device=local, rank=rank, world=world)
    eng.load_nodes(nodes); eng.submit_gangs(g, c, s)
    summ = engine_summary(eng, dev)

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier(); torch.cuda.synchronize()

    def step():
        ms = eng.run_score_pass()
        total, t_coll = sharded_score_pass(dist, world, summ, rank)
        return ms, total, t_coll

    def step_e2e():
        eng.load_nodes(nodes); eng.submit_gangs(g, c, s)
        return step()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step()
    sync()
    t0 = time.perf_counter()
    ms_k, t_c = 0.0, 0.0
    for _ in range(args.steps):
        ms, total, tc = step()
        ms_k += ms; t_c += tc
    sync()
    dt = time.perf_counter() - t0
    step_e2e(); sync()
    t1 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    sync()
    dt_e = time.perf_counter() - t1
    clocks = sampler.stop() if rank == 0 else None
    lo, hi = eng.shard_range()
    tt = torch.tensor([dt, dt_e, ms_k / args.steps, t_c / args.steps], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt, dt_e, ms_kernel, s_coll = tt.tolist()
    if rank == 0:
        pairs = len(c) * len(nodes)
        peak, peak_src = peaks()
        bad = infeasible_from_sum(total, g, c)
        ms_step, ms_e2e = dt / args.steps * 1e3, dt_e / args.steps * 1e3
        shard_bytes = 1.125 * len(c) * (hi - lo)
        ach = shard_bytes / (ms_kernel * 1e-3) / 1e9
        line = {
            "metric": "score_pass_pairs_per_sec", "value": pairs / (ms_step * 1e-3), "unit": "clique-node pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"C4X: score pass (K1 + K2 + per-shard feasibility, no admission) on {len(nodes)} nodes / {len(g)} PodGangs / "
                                   f"{len(c)} PodCliques, 4-level tree; node-range shards cut at zone boundaries, one all-reduce(SUM) of int32[G + Q]",
                       "nodes": len(nodes), "gangs": len(g), "cliques": len(c), "pairs_per_full_pass": pairs,
                       "parallelism": f"{world} node-range shard(s), one per GPU", "l2": "each step writes a score-matrix shard far larger than the 126 MB L2"},
            "result": {"gangs_infeasible_from_snapshot": int(bad.sum()), "all_reduce_bytes": int(4 * (len(g) + len(c))),
                       "collective_s_per_step_max_over_ranks": s_coll, "shard_nodes_rank0": int(hi - lo), "score_matrix_bytes_total": int(pairs)},
            "clocks": clocks,
            "e2e": {"value": pairs / (ms_e2e * 1e-3), "unit": "clique-node pairs/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": int(nodes.nbytes + g.nbytes + c.nbytes + s.nbytes) * world, "d2h_bytes_per_step": int(4 * (len(g) + len(c))) * world},
            "gpu_launches": int(args.steps * 7 * world),
            "roofline": {"kernel": "k_fit + k_score over this rank's node range (grove_run_score_pass), slowest rank", "bound": "hbm", "achieved": ach,
                         "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": shard_bytes, "ms_per_launch": ms_kernel,
                         "note": "1 B written + 1/8 B read per (clique, node) pair of the shard; the pass is write-dominated (~0.6 of the copy peak is its DRAM ceiling)"},
            "cpu_baseline": None,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def run_churn(args):
    """--config C5 (BASELINE.json config 5, steady-state churn): the C4 cluster, 100 PodGang arrivals per 100 ms tick
    (1 000 /s) joining the gangs still pending, ~1 % of the running gangs finishing per tick (their resources come back
    through grove_update_nodes).  A step is one tick: update_nodes + submit_gangs + run_cycle + results to host buffers,
    all through the C ABI with host arrays (e2e); `value` counts the cycle alone (tables already resident)."""
    import torch
    from grove_b200 import build
    from grove_b200.engine import PlacementEngine
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        raise SystemExit("bench.py --config C5 is a single-GPU line (the churn host loop is sequential)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path")
    build.build()
    ch = synth.ChurnC5(n=50000, arrivals=100, release_pct=1)
    sampler = ClockSampler(0)
    sampler.start()
    t_tick, t_cycle, adm, launches, pend, h2d, d2h = [], [], 0, 0, [], 0, 0
    cpu_t, cpu_adm, same, kept = 0.0, 0, True, []
    idx = recs = None
    with PlacementEngine(ch.n_levels) as e:
        e.load_nodes(ch.nodes)
        for tick in range(args.warmup + args.steps):
            specs, tabs = ch.begin_tick()
            g, c, s = tabs
            before = ch.nodes
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if idx is not None and len(idx):
                e.update_nodes(idx, recs)
            e.submit_gangs(g, c, s)
            st = e.run_cycle()
            pl, gs = e.placements(), e.gang_status()
            dt = time.perf_counter() - t0
            if tick >= args.warmup:
                t_tick.append(dt * 1e3); t_cycle.append(st["ms_total"]); adm += st["gangs_admitted"]
                launches += st["kernel_launches"]; pend.append(len(g))
                h2d += g.nbytes + c.nbytes + s.nbytes + (0 if idx is None else idx.nbytes + recs.nbytes); d2h += pl.nbytes + gs.nbytes
            if not args.no_cpu_baseline and args.warmup <= tick < args.warmup + 5:   # bounded CPU sample: five ticks, replayed below
                kept.append((before.copy(), g, c, s, pl.copy(), gs.copy()))
            idx, recs = ch.end_tick(specs, tabs, gs, pl, e.nodes())
    # the CPU leg runs AFTER the timed ticks: the oracle's OpenMP team (all cores) and the engine's (8 threads) share one
    # libgomp, and alternating team sizes makes it re-create its threads -- tens of milliseconds that belong to neither
    for before, g, c, s, pl, gs in kept:
        from oracle import oracle_py as O
        tc = time.perf_counter()
        r = O.run_cycle(before, ch.n_levels, g, c, s, threads=host_cores())
        cpu_t += time.perf_counter() - tc; cpu_adm += r["stats"]["gangs_admitted"]
        same &= bool(np.array_equal(r["placements"], pl) and np.array_equal(r["status"], gs))
    clocks = sampler.stop()
    ms_tick, ms_cyc = float(np.mean(t_tick)), float(np.mean(t_cycle))
    line = {
        "metric": "podgang_placements_per_sec", "value": adm / (sum(t_cycle) * 1e-3), "unit": "gangs/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_cyc, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "C5: steady-state churn on the C4 cluster (50000 nodes, 4-level tree): 100 PodGang arrivals per 100 ms tick "
                               "+ carried-over pending gangs, ~1 % of running gangs finish per tick (grove_update_nodes)",
                   "nodes": 50000, "arrivals_per_tick": 100, "tick_budget_ms": 100.0, "pending_per_tick_mean": float(np.mean(pend)),
                   "pending_per_tick_last": int(pend[-1]), "admitted": int(adm), "tick_ms_mean": ms_tick, "tick_ms_max": float(np.max(t_tick)),
                   "tick_budget_used": ms_tick / 100.0, "arrivals_per_sec_sustained_at_this_latency": 100.0 / (ms_tick * 1e-3),
                   "l2": "inputs change every tick (arrivals, releases)"},
        "clocks": clocks,
        "e2e": {"value": adm / (sum(t_tick) * 1e-3), "unit": "gangs/s", "ms_per_step": ms_tick,
                "h2d_bytes_per_step": int(h2d / args.steps), "d2h_bytes_per_step": int(d2h / args.steps)},
        "gpu_launches": int(launches),
        "roofline": None,
        "cpu_baseline": None if args.no_cpu_baseline else {
            "value": cpu_adm / cpu_t if cpu_t else 0.0, "unit": "gangs/s", "cores": host_cores(), "kind": "port",
            "sample": "the first five timed ticks (same inputs, C restatement on this box's host cores)", "placements_identical_to_gpu": same},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="C4", choices=sorted(synth.CONFIGS) + ["C5", "C4X"])
    ap.add_argument("--impl", default="grove_b200", choices=["grove_b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config in ("C5", "C4X")):
        ap.error("--dump-outputs covers the single-cycle lines on the GPU (C1-C4, --impl grove_b200)")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        if args.config == "C4X":
            raise SystemExit("bench.py: C4X is the multi-GPU score-pass line of this repo; --impl reference covers C1-C4")
        if args.config == "C5":
            raise SystemExit("bench.py: the C5 line times the CPU oracle itself (cpu_baseline, five ticks); --impl reference covers C1-C4")
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        if args.config == "C5":
            run_churn(args)
        elif args.config == "C4X":
            run_sharded(args)
        else:
            run_gpu(args)


if __name__ == "__main__":
    main()
