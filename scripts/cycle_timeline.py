#!/usr/bin/env python
"""cycle_timeline.py -- the device timeline of scheduling cycles: where the GPU works and where it waits.

  python scripts/cycle_timeline.py [--config C4] [--warmup 5] [--cycles 3] [--out DIR]

Runs the `bench.py` device-resident step (node-table reset + grove_run_cycle) `--warmup` times, then `--cycles` more under
torch.profiler with CUDA activities, and writes the chrome trace to DIR/cycle_timeline.pt.trace.json.  For every profiled
cycle (k_reset .. the last kernel before the next cycle) it prints:
  - launches by kernel name,
  - span: first kernel start to last kernel end,
  - busy: the union of the kernel intervals over all streams,
  - idle = span - busy, in total and per relaxation round,
  - the median duration of each kernel,
  - idle by the pair of kernels on either side of each gap.
The summary also goes to DIR/cycle_timeline.json.  Run it in a process of its own: tracing slows the host, so the cycle
times it shows are not the bench values.  Set GROVE_PLACE_LIB to time another build of the engine.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ENGINE_KERNELS = ("k_reset", "k_eval", "k_apply", "k_detect")   # must all be in the trace, or the capture missed the engine


def short_name(name: str) -> str:
    """'void grove::k_eval<true, 1, false>(grove::Topo, ...)' -> 'k_eval<true, 1, false>'"""
    n = name[5:] if name.startswith("void ") else name
    depth, cut = 0, len(n)
    for i, ch in enumerate(n):   # the parameter list starts at the first '(' outside template brackets
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            cut = i
            break
    return re.sub(r"\b[A-Za-z_]\w*::", "", n[:cut]).strip()


def union_length(iv):
    busy, end = 0.0, -np.inf
    for a, b in sorted(iv):
        if b <= end:
            continue
        busy += b - max(a, end)
        end = b
    return busy


def analyse(kernels, rounds):
    """kernels: [(start_us, end_us, short name)] of one cycle, sorted by start"""
    span = max(k[1] for k in kernels) - kernels[0][0]
    busy = union_length([(k[0], k[1]) for k in kernels])
    idle = span - busy
    by_name = collections.defaultdict(list)
    for a, b, n in kernels:
        by_name[n].append(b - a)
    # gaps between consecutive kernels of the cycle (over all streams: a gap is a time no kernel runs), named by its neighbours
    gaps = collections.defaultdict(lambda: [0, 0.0])
    end, last = kernels[0][1], kernels[0][2]
    for a, b, n in kernels[1:]:
        if a > end:
            g = gaps[f"{last} -> {n}"]
            g[0] += 1
            g[1] += a - end
        if b >= end:
            end, last = b, n
    return {
        "span_us": span, "busy_us": busy, "idle_us": idle, "idle_frac": idle / span if span else 0.0,
        "relaxation_rounds": rounds, "idle_us_per_round": idle / rounds if rounds else None,
        "launches": {n: len(v) for n, v in sorted(by_name.items())},
        "n_launches": len(kernels),
        "median_us": {n: float(np.median(v)) for n, v in sorted(by_name.items())},
        "total_us": {n: float(np.sum(v)) for n, v in sorted(by_name.items())},
        "idle_by_gap": {k: {"gaps": c, "us": round(t, 2)} for k, (c, t) in sorted(gaps.items(), key=lambda kv: -kv[1][1])},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C4")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--cycles", type=int, default=3)
    ap.add_argument("--out", default="cycle_timeline")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    from grove_b200 import synth
    from grove_b200.engine import PlacementEngine

    if not torch.cuda.is_available():
        raise SystemExit("cycle_timeline.py: no CUDA device")
    os.makedirs(args.out, exist_ok=True)
    cfg = synth.CONFIGS[args.config]()
    nodes, L = cfg["nodes"], cfg["n_levels"]
    g, c, s = cfg["tables"]
    eng = PlacementEngine(L, device=0)
    eng.load_nodes(nodes)
    eng.submit_gangs(g, c, s)
    d_nodes = torch.from_numpy(nodes.view(np.uint8).reshape(-1)).cuda()

    def step():
        eng.load_nodes_device(d_nodes.data_ptr(), len(nodes))
        return eng.run_cycle()

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    stats = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.cycles):
            stats.append(step())
        torch.cuda.synchronize()
    trace = os.path.join(args.out, "cycle_timeline.pt.trace.json")
    prof.export_chrome_trace(trace)

    with open(trace) as f:
        ev = json.load(f)["traceEvents"]
    kernels = sorted((float(e["ts"]), float(e["ts"]) + float(e["dur"]), short_name(e["name"]))
                     for e in ev if e.get("cat") == "kernel")
    other = collections.Counter(e.get("cat") for e in ev if e.get("cat") in ("gpu_memcpy", "gpu_memset"))
    names = {k[2].split("<")[0] for k in kernels}
    missing = [k for k in ENGINE_KERNELS if k not in names]
    if missing:
        raise SystemExit(f"cycle_timeline.py: the trace holds none of {missing}; kernels seen: {sorted(names)}")
    starts = [i for i, k in enumerate(kernels) if k[2] == "k_reset"]
    if len(starts) != args.cycles:
        raise SystemExit(f"cycle_timeline.py: {len(starts)} k_reset launches in the trace for {args.cycles} cycles")
    cycles = []
    for j, i0 in enumerate(starts):
        i1 = starts[j + 1] if j + 1 < len(starts) else len(kernels)
        ks = [k for k in kernels[i0:i1] if not k[2].startswith("k_gather")]   # k_gather is the next step's node-table reset
        cycles.append(analyse(ks, int(stats[j]["rounds"])))

    import torch.cuda as tc
    summary = {"config": args.config, "device": tc.get_device_name(0), "engine": os.environ.get("GROVE_PLACE_LIB", "in-tree"),
               "memcpy_memset_ops": dict(other), "cycles": cycles,
               "median": {k: float(np.median([cy[k] for cy in cycles])) for k in ("span_us", "busy_us", "idle_us", "idle_frac", "idle_us_per_round")}}
    with open(os.path.join(args.out, "cycle_timeline.json"), "w") as f:
        json.dump(summary, f, indent=1)

    cy = cycles[len(cycles) // 2]
    print(f"{args.config} on {summary['device']}, engine {summary['engine']}; {len(cycles)} profiled cycles, the middle one:")
    print(f"  launches {cy['n_launches']}, relaxation rounds {cy['relaxation_rounds']}")
    for n, k in cy["launches"].items():
        print(f"    {n:34s} {k:4d} launches, median {cy['median_us'][n]:8.2f} us, total {cy['total_us'][n]:8.1f} us")
    print(f"  span {cy['span_us']:.1f} us, busy {cy['busy_us']:.1f} us, idle {cy['idle_us']:.1f} us "
          f"({100 * cy['idle_frac']:.1f} % of the span, {cy['idle_us_per_round']:.2f} us per round)")
    print("  idle by gap (previous kernel -> next kernel):")
    for k, v in list(cy["idle_by_gap"].items())[:12]:
        print(f"    {k:60s} {v['gaps']:4d} gaps {v['us']:8.1f} us")
    m = summary["median"]
    print(f"  median over cycles: span {m['span_us']:.1f} us, idle {m['idle_us']:.1f} us ({100 * m['idle_frac']:.1f} %), "
          f"{m['idle_us_per_round']:.2f} us per round")
    print(json.dumps({"timeline": {"config": args.config, "engine": summary["engine"], **m}}))


if __name__ == "__main__":
    main()
