#!/usr/bin/env python3
"""Measures the segment-time estimates on one GPU: tg_estimate_segment_times_batch (both outputs) for 65 536 and 1 048 576 random-flier
paths of 11 waypoints (10 segments each), with the node's synthetic limits.  Per size: device ms (tg_last_device_ms = CUDA events
around the call: the copies of vtx_off and the positions in, the kernel, the two outputs back; median of 5 after a warm-up), wall ms
of the call from pageable numpy buffers, the kernel alone (a profiled call of its own), and the host-to-device copy of the positions
alone (the same pageable buffer copied by torch, CUDA events) -- the part the call cannot avoid.  For contrast the oracle
(oracle/ restatement, deterministic math mode, tests/cpp/oracle_estimate_times.cpp) on one host core and on every host core, with the
core count, and whether every output bit equals the device's.  The card's name and power limit are read first, in the same run.
Usage (GPU box, after __graft_entry__.build()): python tools/bench_segment_times.py OUT.json"""
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
from mrs_uav_trajectory_generation_b200 import workloads as W  # noqa: E402
import oracle_lib as O  # noqa: E402
from test_segment_times import oracle_times  # noqa: E402

dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)


def _p(a, t=dp):
    return None if a is None else a.ctypes.data_as(t)


def main():
    import torch

    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    lines = [{"card": q.stdout.strip(), "host_cores": os.cpu_count()}]
    print(json.dumps(lines[0]), flush=True)
    ctx = tg.Context(tg.Library(), 0)
    lib = ctx.L.lib
    L9 = np.array(O.DEFAULT_LIMITS, dtype=np.float64)
    L8 = np.ascontiguousarray(L9[:8])
    for B in (65536, 1 << 20):
        wp_off, wp = W.random_flier_paths_fast(B, 11)
        totS = B * 10
        e, b = np.empty(totS), np.empty(totS)

        def call():
            rc = lib.tg_estimate_segment_times_batch(ctx.h, B, _p(wp_off, ip), _p(wp), _p(L8), _p(e), _p(b))
            assert rc == 0, lib.tg_last_error(ctx.h)

        dev, wall = [], []
        for _ in range(6):
            t0 = time.perf_counter()
            call()
            wall.append(1e3 * (time.perf_counter() - t0))
            dev.append(ctx.last_device_ms())
        ctx.set_profiling(True)
        call()
        prof = {k: [round(v[0], 4), int(v[1])] for k, v in ctx.profile().items()}
        ctx.set_profiling(False)
        kern = sum(v[0] for v in prof.values())
        # the positions' host-to-device copy alone, from the same pageable buffer
        src = torch.from_numpy(wp)
        dst = torch.empty(wp.shape, dtype=torch.float64, device="cuda")
        h2d = []
        for _ in range(6):
            s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            dst.copy_(src)
            t.record()
            t.synchronize()
            h2d.append(s.elapsed_time(t))
        O.set_math_mode(O.MATH_DET)
        oracle = {}
        for n in (1, os.cpu_count()):
            t0 = time.perf_counter()
            oe, ob = oracle_times(wp_off, wp, L9, nthreads=n)
            oracle[n] = 1e3 * (time.perf_counter() - t0)
        line = {"call": "tg_estimate_segment_times_batch (Euclidean + Baca)", "paths": B, "waypoints": 11, "segments": totS,
                "device_ms": float(np.median(dev[1:])), "wall_ms": float(np.median(wall[1:])), "kernel_ms": kern,
                "positions_h2d_ms": float(np.median(h2d[1:])), "positions_bytes": int(wp.nbytes),
                "segments_per_s_device": totS / (1e-3 * float(np.median(dev[1:]))), "oracle_1_core_ms": oracle[1],
                f"oracle_{os.cpu_count()}_cores_ms": oracle[os.cpu_count()], "same_bits_as_oracle": bool(np.array_equal(e, oe) and np.array_equal(b, ob)),
                "kernels": prof,
                "note": "device_ms = CUDA events around the call (copies in and out included), wall_ms = host clock around it (pageable "
                        "buffers), median of 5 after a warm-up; kernel_ms from one profiled call; positions_h2d_ms = torch copy of the same "
                        "pageable positions array, median of 5; oracle = host restatement, deterministic math mode"}
        lines.append(line)
        print(json.dumps({k: v for k, v in line.items() if k != "note"}), flush=True)
    if out_path:
        with open(out_path, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
