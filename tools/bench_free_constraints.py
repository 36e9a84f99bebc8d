#!/usr/bin/env python3
"""Measures the free-constraint entry points on one GPU: tg_solve_linear_free_batch_nd (solveLinear + getFreeConstraints + getSegments +
computeCost) and tg_set_free_constraints_batch_nd (setFreeConstraints + getSegments + computeCost) for B = $TG_FREE_B (65536)
random-flier problems of 11 vertices with the node's vertex recipe (ends fixed up to acceleration, interior positions), r = 2, D = 4,
at N = 10 and N = 12.  For comparison the same problems through tg_solve_linear_batch_nd and, at N = 10, the tuned
tg_solve_linear_batch.  Per call: device ms (CUDA events around the call, copies in and out included; median of three after a
warm-up), wall ms, problems/s, and the kernel table of one extra profiled call.  The card's name and power limit are read first.
Usage (GPU box): python tools/bench_free_constraints.py OUT.json"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mrs_uav_trajectory_generation_b200 as tg  # noqa: E402
from mrs_uav_trajectory_generation_b200 import workloads as W  # noqa: E402


def problems(B, n_coef, V=11, r=2):
    wp_off, wp = W.random_flier_paths_fast(B, V)
    mask = np.ones((B, V), np.uint8)
    mask[:, 0] = mask[:, -1] = (1 << (r + 1)) - 1
    vals = np.zeros((B * V, n_coef // 2, 4))
    vals[:, 0] = wp
    w = wp.reshape(B, V, 4)
    times = (np.linalg.norm(w[:, 1:, :3] - w[:, :-1, :3], axis=2) / 1.5 + 0.2).ravel()
    return wp_off, mask.ravel(), vals, times


def timed(ctx, fn):
    dev, wall = [], []
    for _ in range(4):
        t0 = time.perf_counter()
        out = fn()
        wall.append(1e3 * (time.perf_counter() - t0))
        dev.append(ctx.last_device_ms())
    ctx.set_profiling(True)
    fn()
    prof = ctx.profile()
    ctx.set_profiling(False)
    return out, float(np.median(dev[1:])), float(np.median(wall[1:])), {k: [round(v[0], 3), int(v[1])] for k, v in prof.items()}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    B, r = int(os.environ.get("TG_FREE_B", "65536")), 2
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    lines = [{"card": q.stdout.strip()}]
    print(json.dumps(lines[0]), flush=True)
    ctx = tg.Context(tg.Library(), 0)
    for n_coef in (10, 12):
        off, mask, vals, times = problems(B, n_coef, 11, r)
        calls = {"tg_solve_linear_free_batch_nd": lambda: ctx.solve_linear_free_batch_nd(n_coef, 4, off, mask, vals, times, r),
                 "tg_solve_linear_batch_nd": lambda: ctx.solve_linear_batch_nd(n_coef, 4, off, mask, vals, times, r)}
        if n_coef == 10:
            calls["tg_solve_linear_batch"] = lambda: ctx.solve_linear_batch(off, mask, vals, times, r)
        results = {}
        for name, fn in calls.items():
            results[name] = timed(ctx, fn)
        coef, cost, free = results["tg_solve_linear_free_batch_nd"][0]
        results["tg_set_free_constraints_batch_nd"] = timed(ctx, lambda: ctx.set_free_constraints_batch_nd(n_coef, 4, off, mask, vals, times, free, r))
        c_set, k_set = results["tg_set_free_constraints_batch_nd"][0]
        same = {"set(get) == solve": bool(np.array_equal(c_set, coef) and np.array_equal(k_set, cost)),
                "free call == solve_linear_batch_nd": bool(np.array_equal(results["tg_solve_linear_batch_nd"][0][0], coef))}
        if n_coef == 10:
            same["free call == tuned solve"] = bool(np.array_equal(results["tg_solve_linear_batch"][0][0], coef))
        for name, (_, dev, wall, prof) in results.items():
            line = {"N": n_coef, "D": 4, "r": r, "call": name, "problems": B, "segments_per_problem": 10,
                    "free_per_problem": int(free[0].size), "device_ms": dev, "wall_ms": wall,
                    "problems_per_s_device": B / (1e-3 * dev) if dev > 0 else None, "kernel_ms": prof, "same_bits": same,
                    "note": "device_ms = CUDA events around the call (copies in and out included); median of 3 after a warm-up"}
            lines.append(line)
            print(json.dumps({k: v for k, v in line.items() if k != "kernel_ms"}), flush=True)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
