#!/usr/bin/env python3
"""Measures the general-shape path (csrc/tg_generic.cuh) on one GPU beside the CPU oracle compiled for the same N, on B problems of 11
vertices (10 segments):
  * linear optimisation (tg_solve_linear_batch_nd), B = $TG_GS_B (65536), five shapes;
  * Mellinger time allocation (tg_time_alloc_batch_nd), B = $TG_GS_TA_B (16384), D = 4, N in {6, 8, 10, 12}.
Prints the card (name, power limit, max SM clock) first, then one JSON object per measurement; the N = 10, D = 4 lines also time the
tuned kernels on the same problems and say whether both paths give the same bits.
Usage (GPU box): python tools/bench_general_shape.py > profiles/rNN_general_shape.json"""
import ctypes as C
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
import oracle_lib as O  # noqa: E402


def problems(n_coef, dims, B, V=11, seed=0):
    rng = np.random.default_rng(seed + n_coef)
    H = n_coef // 2
    mask = np.ones((B, V), np.uint8)
    mask[:, 0] = mask[:, -1] = (1 << min(H, 3)) - 1
    vals = np.zeros((B, V, H, dims))
    vals[:, :, 0, :] = np.cumsum(rng.normal(size=(B, V, dims)) * 2.0, axis=1)
    times = rng.uniform(0.5, 3.0, (B, V - 1))
    off = np.arange(B + 1, dtype=np.int32) * V
    return off, mask.reshape(-1), vals.reshape(B * V, H, dims), times.reshape(-1)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"card": q.stdout.strip()}


def time_alloc_lines(ctx, B):
    """PolynomialOptimizationNonLinear<N>(4)::optimize() with the Mellinger method for B problems per call."""
    for n_coef in (6, 8, 10, 12):
        r = 2
        off, mask, vals, times = problems(n_coef, 4, B, seed=7)
        P = ctx.L.default_params(derivative_to_optimize=r)
        ms = []
        for rep in range(4):
            out = ctx.time_alloc_batch_nd(n_coef, 4, off, mask, vals, times, P)
            ms.append(ctx.last_device_ms())
        dev = float(np.median(ms[1:]))
        line = {"time_alloc": {"N": n_coef, "D": 4, "derivative_to_optimize": r}, "problems": B, "segments_per_problem": 10,
                "device_ms": dev, "problems_per_s_device": B / (1e-3 * dev) if dev > 0 else None,
                "mean_evaluations": float(out["n_evals"].mean()), "mean_scale_passes": float(out["n_scale_passes"].mean()),
                "note": "device_ms = CUDA events around the call (copies in and out included); no Bernstein pruning, dense evaluation launches"}
        ctx.set_profiling(True)
        ctx.time_alloc_batch_nd(n_coef, 4, off, mask, vals, times, P)
        prof = ctx.profile()
        ctx.set_profiling(False)
        line["kernel_ms"] = {k: [round(v[0], 3), int(v[1])] for k, v in prof.items()}  # kernel: [ms, launches]
        if n_coef == 10:
            tm = []
            for rep in range(4):
                tuned = ctx.time_alloc_batch(off, mask, vals, times, P)
                tm.append(ctx.last_device_ms())
            line["tuned_kernels_device_ms"] = float(np.median(tm[1:]))
            line["general_equals_tuned_bit_for_bit"] = bool(all(np.array_equal(out[k], tuned[k]) for k in out))
        orc = O.OracleN(n_coef)
        v4 = vals  # D = 4 already
        Po = O.Params()
        C.memmove(C.byref(Po), C.byref(P), C.sizeof(O.Params))
        nb, same, t0 = 64, True, time.perf_counter()
        for p in range(nb):
            t = np.array(times[p * 10:(p + 1) * 10])
            c = np.zeros((10, 4, n_coef))
            code, ev, ps, cost = C.c_int(), C.c_int(), C.c_int(), C.c_double()
            m = np.ascontiguousarray(mask[p * 11:(p + 1) * 11])
            vv = np.ascontiguousarray(v4[p * 11:(p + 1) * 11])
            orc.lib.orc_time_alloc(11, m.ctypes.data_as(C.POINTER(C.c_uint8)), vv.ctypes.data_as(C.POINTER(C.c_double)),
                                   t.ctypes.data_as(C.POINTER(C.c_double)), r, C.byref(Po), c.ctypes.data_as(C.POINTER(C.c_double)), C.byref(code),
                                   C.byref(ev), C.byref(ps), C.byref(cost))
            same = same and np.array_equal(t, out["times"][p * 10:(p + 1) * 10]) and np.array_equal(c, out["coef"][p * 10:(p + 1) * 10])
        line["cpu_oracle_problems_per_s_one_thread"] = nb / (time.perf_counter() - t0)
        line["bit_exact_vs_oracle_first_64"] = bool(same)
        print(json.dumps(line), flush=True)


def main():
    B = int(os.environ.get("TG_GS_B", "65536"))
    ctx = tg.Context(tg.Library(), 0)
    print(json.dumps(card()), flush=True)
    for n_coef, dims, r in ((6, 3, 2), (8, 4, 3), (10, 4, 2), (12, 4, 4), (12, 1, 5)):
        off, mask, vals, times = problems(n_coef, dims, B)
        ms, wall = [], []
        for rep in range(6):
            t0 = time.perf_counter()
            coef, cost = ctx.solve_linear_batch_nd(n_coef, dims, off, mask, vals, times, r)
            wall.append(time.perf_counter() - t0)
            ms.append(ctx.last_device_ms())
        line = {"shape": {"N": n_coef, "D": dims, "derivative_to_optimize": r}, "problems": B, "segments_per_problem": 10,
                "device_ms": float(np.median(ms[1:])), "problems_per_s_device": B / (1e-3 * float(np.median(ms[1:]))),
                "problems_per_s_host_buffers": B / float(np.median(wall[1:])),
                "note": "device_ms = CUDA events around the call: host-to-device copies, three kernel launches, copy back"}
        # kernel-only times (CUDA events around every launch of one extra call)
        ctx.set_profiling(True)
        ctx.solve_linear_batch_nd(n_coef, dims, off, mask, vals, times, r)
        prof = ctx.profile()
        ctx.set_profiling(False)
        line["kernel_ms"] = {k: round(v[0], 3) for k, v in prof.items() if "gen::" in k}
        kern = sum(line["kernel_ms"].values()) * 1e-3
        line["kernel_problems_per_s"] = B / kern if kern > 0 else None
        if n_coef == 10 and dims == 4:
            tm = []
            for rep in range(6):
                c_t, cost_t = ctx.solve_linear_batch(off, mask, vals, times, r)
                tm.append(ctx.last_device_ms())
            line["tuned_kernels_device_ms"] = float(np.median(tm[1:]))
            line["general_equals_tuned_bit_for_bit"] = bool(np.array_equal(c_t, coef) and np.array_equal(cost_t, cost))
        # CPU oracle for the same N on a sample, one thread
        orc = O.OracleN(n_coef)
        nb = 256
        v4 = np.zeros((nb * 11, n_coef // 2, 4))
        v4[:, :, :dims] = vals[: nb * 11]
        t0 = time.perf_counter()
        same = True
        for p in range(nb):
            c_o, cost_o = orc.solve_linear(mask[p * 11:(p + 1) * 11], v4[p * 11:(p + 1) * 11], times[p * 10:(p + 1) * 10], r)
            same = same and np.array_equal(c_o[:, :dims], coef[p * 10:(p + 1) * 10]) and cost_o == cost[p]
        cpu = time.perf_counter() - t0
        line["cpu_oracle_problems_per_s_one_thread"] = nb / cpu
        line["bit_exact_vs_oracle_first_256"] = bool(same)
        print(json.dumps(line), flush=True)
    time_alloc_lines(ctx, int(os.environ.get("TG_GS_TA_B", "16384")))


if __name__ == "__main__":
    main()
