#!/usr/bin/env python3
"""Measures windowed sampling on one GPU: tg_sample_range_batch_nd and tg_evaluate_range_batch_nd for B = $TG_RANGE_B (65536)
random-flier trajectories of 11 waypoints (10 segments; ends fixed up to acceleration, r = 2, D = 4), at N = 10 and N = 12, each with a
2 s window at a random start inside the trajectory and dt = 0.01 -- "the next 2 s of every trajectory".  Per call: device ms (CUDA
events around the call, copies in and out included; median of three after a warm-up) of the counting call (outputs NULL) and of the
outputs call, samples/s, and the kernel table of one extra profiled call; "not_in_kernels" = 1 - kernel time / device time of the
outputs call, i.e. the share taken by the copies and the gaps between launches.  For contrast, Trajectory::evaluateRange as the C++
header did it before this entry point (a host walk, then one tg_evaluate_batch call per segment the window touches; restated here in
Python) on 1000 of the trajectories, one trajectory at a time, next to tg_evaluate_range_batch_nd with B = 1 per trajectory and
one batched call.  The card's name and power limit are read first.
Usage (GPU box): python tools/bench_sample_range.py OUT.json"""
import ctypes as C
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

dp, ip, llp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_longlong)


def _p(a, t=dp):
    return None if a is None else a.ctypes.data_as(t)


def trajectories(ctx, B, n_coef, V=11, r=2):
    wp_off, wp = W.random_flier_paths_fast(B, V)
    mask = np.ones((B, V), np.uint8)
    mask[:, 0] = mask[:, -1] = (1 << (r + 1)) - 1
    vals = np.zeros((B * V, n_coef // 2, 4))
    vals[:, 0] = wp
    w = wp.reshape(B, V, 4)
    times = (np.linalg.norm(w[:, 1:, :3] - w[:, :-1, :3], axis=2) / 1.5 + 0.2).ravel()
    coef, _ = ctx.solve_linear_batch_nd(n_coef, 4, wp_off, mask.ravel(), vals, times, r)
    seg_off = (np.asarray(wp_off) - np.arange(B + 1)).astype(np.int32)
    return seg_off, coef, times


def timed(ctx, fn):
    dev, wall = [], []
    for _ in range(4):
        t0 = time.perf_counter()
        fn()
        wall.append(1e3 * (time.perf_counter() - t0))
        dev.append(ctx.last_device_ms())
    ctx.set_profiling(True)
    fn()
    prof = ctx.profile()
    ctx.set_profiling(False)
    return float(np.median(dev[1:])), float(np.median(wall[1:])), {k: [round(v[0], 3), int(v[1])] for k, v in prof.items()}


def old_evaluate_range(ctx, coef, T, t_start, t_end, dt, deriv):
    """the C++ header's former evaluateRange: host walk, one tg_evaluate_batch call per run of samples in one segment"""
    ts, seg_of, acc, i = [], [], 0.0, 0
    for i in range(len(T)):
        acc += T[i]
        if acc > t_start:
            break
    acc -= T[i]
    tin = t_start - acc
    while acc < t_end:
        if tin > T[i]:
            tin -= T[i]
            i += 1
            if i >= len(T):
                break
            continue
        ts.append(tin)
        seg_of.append(i)
        tin += dt
        acc += dt
    out, k0 = [], 0
    while k0 < len(ts):
        k1 = k0
        while k1 < len(ts) and seg_of[k1] == seg_of[k0]:
            k1 += 1
        s = seg_of[k0]
        out.append(ctx.evaluate(coef[s:s + 1], T[s:s + 1], np.array(ts[k0:k1]), deriv)[0])
        k0 = k1
    return np.concatenate(out) if out else np.zeros((0, 4))


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    B, dt, H = int(os.environ.get("TG_RANGE_B", "65536")), 0.01, 2.0
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    lines = [{"card": q.stdout.strip()}]
    print(json.dumps(lines[0]), flush=True)
    ctx = tg.Context(tg.Library(), 0)
    lib = ctx.L.lib
    rng = np.random.default_rng(1)
    for n_coef in (10, 12):
        seg_off, coef, times = trajectories(ctx, B, n_coef)
        ends = np.add.reduceat(times, seg_off[:-1])
        starts = rng.uniform(0.0, 1.0, B) * np.maximum(ends - H, 0.0)
        win = np.ascontiguousarray(np.column_stack([starts, starts + H]))
        counts = np.zeros(B, np.int32)

        def sample(samples=None, t_ns=None):
            rc = lib.tg_sample_range_batch_nd(ctx.h, n_coef, 4, B, _p(seg_off, ip), _p(coef), _p(times), _p(win), C.c_double(dt), _p(counts, ip),
                                              _p(samples), None, _p(t_ns, llp))
            assert rc == 0, tg.TgError(lib.tg_last_error(ctx.h))

        sample()
        rows = int(counts.sum())
        samples, t_ns = np.empty((rows, 4)), np.empty(rows, np.int64)
        vals, st = np.empty((rows, 4)), np.empty(rows)

        def evaluate(out=None, s=None):
            rc = lib.tg_evaluate_range_batch_nd(ctx.h, n_coef, 4, B, _p(seg_off, ip), _p(coef), _p(times), _p(win), C.c_double(dt), 1,
                                                _p(counts, ip), _p(out), _p(s))
            assert rc == 0

        res = {"tg_sample_range_batch_nd counts": timed(ctx, sample), "tg_sample_range_batch_nd samples+t_ns": timed(ctx, lambda: sample(samples, t_ns)),
               "tg_evaluate_range_batch_nd counts": timed(ctx, evaluate), "tg_evaluate_range_batch_nd values+times": timed(ctx, lambda: evaluate(vals, st))}
        for name, (dev, wall, prof) in res.items():
            kern = sum(v[0] for v in prof.values())
            line = {"N": n_coef, "D": 4, "call": name, "trajectories": B, "window_s": H, "dt": dt, "samples": rows, "device_ms": dev, "wall_ms": wall,
                    "samples_per_s_device": rows / (1e-3 * dev) if dev > 0 else None, "kernel_ms_sum": kern,
                    "not_in_kernels": (1.0 - kern / dev) if dev > 0 else None, "kernel_ms": prof,
                    "note": "device_ms = CUDA events around the call (copies in and out included); median of 3 after a warm-up"}
            lines.append(line)
            print(json.dumps({k: v for k, v in line.items() if k != "kernel_ms"}), flush=True)
        if n_coef == 10:  # one trajectory at a time: the former per-segment path against the new entry point
            n = 1000
            so = [np.array([0, seg_off[p + 1] - seg_off[p]], np.int32) for p in range(n)]
            cs = [np.ascontiguousarray(coef[seg_off[p]:seg_off[p + 1]]) for p in range(n)]
            ts = [np.ascontiguousarray(times[seg_off[p]:seg_off[p + 1]]) for p in range(n)]
            for rep in range(2):  # the first pass warms up
                t0 = time.perf_counter()
                old = [old_evaluate_range(ctx, cs[p], ts[p], win[p, 0], win[p, 1], dt, 1) for p in range(n)]
                t_old = time.perf_counter() - t0
                t0 = time.perf_counter()
                new = [ctx.evaluate_range_batch_nd(10, 4, so[p], cs[p], ts[p], win[p:p + 1], dt, 1)[1] for p in range(n)]
                t_new = time.perf_counter() - t0
            t0 = time.perf_counter()
            _, batched, _ = ctx.evaluate_range_batch_nd(10, 4, seg_off[:n + 1], coef[:seg_off[n]], times[:seg_off[n]], win[:n], dt, 1)
            t_batch = time.perf_counter() - t0
            same = all(np.array_equal(a, b) for a, b in zip(old, new)) and np.array_equal(np.concatenate(new), batched)
            line = {"N": 10, "D": 4, "call": "evaluateRange, 1000 trajectories, velocity", "former_per_segment_calls_wall_s": t_old,
                    "tg_evaluate_range_batch_nd_B1_per_trajectory_wall_s": t_new, "tg_evaluate_range_batch_nd_one_call_wall_s": t_batch,
                    "same_bits": bool(same), "note": "host wall clock over the Python loop (each call ends in a device synchronise)"}
            lines.append(line)
            print(json.dumps(line), flush=True)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
