#!/usr/bin/env python3
"""Measures the batched derivative-free time allocation (tg_time_alloc_dfo_batch, csrc/tg_dfo.cuh) on one GPU: B = $TG_DFO_B (16384)
random-flier problems of 11 waypoints (S = 10) with the node's vertex recipe (ends fixed up to acceleration, interior positions) and
the node's 12 magnitude constraints, per method 0, 1, 3, 4 and the default parameters (max_iterations 10, f_rel 0.05).
Per method: device ms per call (CUDA events around the call, copies included; median of three after a warm-up), problems/s, the
per-kernel table of one extra profiled call, and for contrast the wall time of one B = 1 call per problem over the first 256 problems
(what a caller looping over problems gets).  The card's name and power limit are read first.
Usage (GPU box): python tools/bench_derivative_free.py OUT.json"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import mrs_uav_trajectory_generation_b200 as tg  # noqa: E402
from mrs_uav_trajectory_generation_b200 import workloads as W  # noqa: E402
import oracle_lib as O  # noqa: E402

CONSTRAINTS = [(d, k, v) for d, lim in enumerate(((4.0, 2.0, 20.0), (4.0, 2.0, 20.0), (2.0, 1.0, 20.0), (1.0, 2.0, 10.0)))
               for k, v in zip((1, 2, 3), lim)]


def problems(B, V=11):
    off = np.arange(B + 1, dtype=np.int32) * V
    mask = np.ones((B, V), np.uint8)
    mask[:, 0] = mask[:, -1] = 0b111
    vals = np.zeros((B, V, 5, 4))
    times = np.zeros((B, V - 1))
    for p in range(B):
        wp = W.random_flier_path(p, V)
        vals[p, :, 0] = wp
        times[p] = O.estimate_times(wp)[0]
    return off, mask.reshape(-1), vals.reshape(B * V, 5, 4), times.reshape(-1)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    B = int(os.environ.get("TG_DFO_B", "16384"))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    lines = [{"card": q.stdout.strip()}]
    print(json.dumps(lines[0]), flush=True)
    ctx = tg.Context(tg.Library(), 0)
    off, mask, vals, times = problems(B)
    n_free = sum(5 - bin(int(m)).count("1") for m in mask[:11])
    for method in (0, 1, 3, 4):
        P = ctx.L.default_dfo_params(time_alloc_method=method)
        ms = []
        for rep in range(4):
            out = ctx.time_alloc_dfo_batch(off, mask, vals, times, P, CONSTRAINTS)
            ms.append(ctx.last_device_ms())
        dev = float(np.median(ms[1:]))
        codes = {int(c): int((out["code"] == c).sum()) for c in np.unique(out["code"])}
        line = {"method": method, "problems": B, "segments_per_problem": 10, "variables_per_problem": 10 if method < 3 else 10 + 4 * n_free,
                "device_ms": dev, "problems_per_s_device": B / (1e-3 * dev) if dev > 0 else None, "mean_iterations": float(out["n_iterations"].mean()),
                "codes": codes, "note": "device_ms = CUDA events around the call (copies in and out included); median of 3 after a warm-up"}
        ctx.set_profiling(True)
        ctx.time_alloc_dfo_batch(off, mask, vals, times, P, CONSTRAINTS)
        prof = ctx.profile()
        ctx.set_profiling(False)
        line["kernel_ms"] = {k: [round(v[0], 3), int(v[1])] for k, v in prof.items()}  # kernel: [ms, launches]
        nb = min(256, B)
        same = True
        t0 = time.perf_counter()
        for p in range(nb):
            one = ctx.time_alloc_dfo_batch(off[:2], mask[p * 11:(p + 1) * 11], vals[p * 11:(p + 1) * 11], times[p * 10:(p + 1) * 10], P, CONSTRAINTS)
            same = same and np.array_equal(one["times"], out["times"][p * 10:(p + 1) * 10]) and one["total"][0] == out["total"][p]
        wall = time.perf_counter() - t0
        line["single_problem_loop_problems_per_s_wall"] = nb / wall
        line["single_problem_loop_equals_batch_first_%d" % nb] = bool(same)
        lines.append(line)
        print(json.dumps(line), flush=True)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
