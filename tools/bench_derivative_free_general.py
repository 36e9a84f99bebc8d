#!/usr/bin/env python3
"""Measures the derivative-free time allocation for PolynomialOptimization<N> (tg_time_alloc_dfo_batch_nd, csrc/tg_dfo_generic.cuh)
on one GPU: B = $TG_DFO_B (16384) random-flier problems of 11 vertices (S = 10) with the node's vertex recipe (ends fixed up to
acceleration, interior positions) and the node's 12 magnitude constraints, default parameters (max_iterations 10, f_rel 0.05),
methods 0, 1, 3, 4, for N = 6, 8, 10, 12 on 4 dimensions and N = 10 on 3 dimensions.  At N = 10 on 4 dimensions the tuned
tg_time_alloc_dfo_batch runs on the same problems, and whether both give the same bits is recorded.
Per call: device ms (CUDA events around the call, copies included; median of two after a warm-up), problems/s and the mean
iteration count.  The card's name and power limit are read first.
Usage (GPU box): python tools/bench_derivative_free_general.py OUT.json"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import mrs_uav_trajectory_generation_b200 as tg  # noqa: E402
from mrs_uav_trajectory_generation_b200 import workloads as W  # noqa: E402
import oracle_lib as O  # noqa: E402

CONSTRAINTS = [(d, k, v) for d, lim in enumerate(((4.0, 2.0, 20.0), (4.0, 2.0, 20.0), (2.0, 1.0, 20.0), (1.0, 2.0, 10.0)))
               for k, v in zip((1, 2, 3), lim)]
SHAPES = [(6, 4), (8, 4), (10, 4), (12, 4), (10, 3)]


def problems(B, n_coef, dims, V=11):
    H = n_coef // 2
    off = np.arange(B + 1, dtype=np.int32) * V
    mask = np.ones((B, V), np.uint8)
    mask[:, 0] = mask[:, -1] = 0b111
    vals = np.zeros((B, V, H, dims))
    times = np.zeros((B, V - 1))
    for p in range(B):
        wp = W.random_flier_path(p, V)
        vals[p, :, 0] = wp[:, :dims]
        times[p] = O.estimate_times(wp)[0]
    return off, mask.reshape(-1), vals.reshape(B * V, H, dims), times.reshape(-1)


def timed(ctx, fn, reps=3):
    ms, out = [], None
    for _ in range(reps):
        out = fn()
        ms.append(ctx.last_device_ms())
    return float(np.median(ms[1:])), out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    B = int(os.environ.get("TG_DFO_B", "16384"))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    lines = [{"card": q.stdout.strip(), "problems": B, "segments_per_problem": 10, "constraints": len(CONSTRAINTS),
              "note": "device_ms = CUDA events around the call (copies in and out included); median of 2 after a warm-up"}]
    print(json.dumps(lines[0]), flush=True)
    ctx = tg.Context(tg.Library(), 0)
    for n_coef, dims in SHAPES:
        off, mask, vals, times = problems(B, n_coef, dims)
        n_free = sum(n_coef // 2 - bin(int(m)).count("1") for m in mask[:11])
        for method in (0, 1, 3, 4):
            P = ctx.L.default_dfo_params(time_alloc_method=method)
            dev, out = timed(ctx, lambda: ctx.time_alloc_dfo_batch_nd(n_coef, dims, off, mask, vals, times, P, CONSTRAINTS))
            line = {"N": n_coef, "D": dims, "method": method, "call": "tg_time_alloc_dfo_batch_nd",
                    "variables_per_problem": 10 if method < 3 else 10 + dims * n_free, "device_ms": dev,
                    "problems_per_s_device": B / (1e-3 * dev) if dev > 0 else None, "mean_iterations": float(out["n_iterations"].mean()),
                    "codes": {int(c): int((out["code"] == c).sum()) for c in np.unique(out["code"])}}
            if (n_coef, dims) == (10, 4):
                dev_t, tuned = timed(ctx, lambda: ctx.time_alloc_dfo_batch(off, mask, vals, times, P, CONSTRAINTS))
                line["tuned_device_ms"] = dev_t
                line["tuned_problems_per_s_device"] = B / (1e-3 * dev_t) if dev_t > 0 else None
                line["nd_over_tuned"] = dev / dev_t if dev_t > 0 else None
                line["same_bits_as_tuned"] = bool(all(np.array_equal(out[k], tuned[k]) for k in ("times", "coef", "code", "n_iterations", "total", "parts")))
            lines.append(line)
            print(json.dumps(line), flush=True)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
