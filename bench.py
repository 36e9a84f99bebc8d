#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 trajectory path (contract: see the build prompt / DESIGN.md "Measurement").

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference ...                     (the reference arm: CPU restatement on the host cores)
  python bench.py ... --dump-outputs DIR                   (also writes the last timed step's outputs to DIR/*.npy)

Workload = BASELINE.json configs[2] ("65536 random paths, full nonlinear time allocation and feasibility subdivision"),
the configuration the metric "optimized+sampled trajectories/sec (10-seg, N=10, fp64) at 1/2/4/8 B200" is quoted on.
One step = one pass of the whole hot path (optimize(): findTrajectory + validation + subdivision rounds) over one batch
of synthetic random-flier paths per GPU (weak scaling: every rank owns its own batch, no data-path collective).
"""
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "optimized+sampled trajectories/sec (10-seg, N=10, fp64)"
UNIT = "trajectories/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(n_paths, first_index, nthreads=0, keep=False):
    """The oracle (CPU restatement of the reference, `kind: port`) on a bounded sample of the same workload."""
    import oracle_lib as O
    from mrs_uav_trajectory_generation_b200 import workloads as W

    O.build_oracle(ref=False)
    O.set_math_mode(O.MATH_DET)
    wp_off, wp = W.random_flier_paths_fast(n_paths, first_index=first_index)
    t0 = time.perf_counter()
    r = O.optimize_batch(wp_off, wp, cap_wp=700, cap_samples=4000, nthreads=nthreads, want_outputs=True)
    dt = time.perf_counter() - t0
    ok = sum(1 for x in r["res"] if x.success)
    if keep:
        return n_paths / dt, r["threads"], dt, ok, (wp_off, wp, r)
    return n_paths / dt, r["threads"], dt, ok


def parity_on_sample(ctx, P, sample):
    """Outside the timed region: the GPU's outputs for the cpu_baseline sample (the first paths of the bench batch) against the
    oracle outputs that leg has just computed -- verdicts and counts exactly, coefficients / samples bit for bit."""
    import parity_checks as PC

    wp_off, wp, ref = sample
    res, _ = ctx.optimize_batch(wp_off, wp, None, None, P)
    out = ctx.fetch_outputs()
    n = len(wp_off) - 1
    ints = ("status", "success", "nlopt_code", "n_evals", "rounds", "safe", "n_waypoints", "n_samples", "n_scale_passes")
    verdicts, exact, worst_c, worst_s = 0, 0, 0.0, 0.0
    for p in range(n):
        r, g = ref["res"][p], res[p]
        same = all(getattr(r, k) == g[k] for k in ints)
        verdicts += int(same)
        if not same or not g["success"]:
            exact += int(same)
            continue
        s0, s1 = out["seg_off"][p], out["seg_off"][p + 1]
        m0, m1 = out["smp_off"][p], out["smp_off"][p + 1]
        S, M = s1 - s0, m1 - m0
        rc, rt, rs = ref["coeffs"][p, :S], ref["times"][p, :S], ref["samples"][p, :M]
        worst_c = max(worst_c, PC.coef_rel_err(out["coef"][s0:s1], rc, rt))
        worst_s = max(worst_s, float(np.abs(out["samples"][m0:m1, :3] - rs[:, :3]).max()))
        exact += int(np.array_equal(out["coef"][s0:s1], rc) and np.array_equal(out["times"][s0:s1], rt) and np.array_equal(out["samples"][m0:m1], rs))
    return {"paths": n, "verdicts_and_counts_equal": verdicts, "bit_exact": exact, "worst_coef_rel": worst_c, "worst_sample_pos_m": worst_s,
            "against": "oracle (CPU restatement, pinned bit for bit to the reference's own eth_trajectory_generation sources compiled with stand-in "
                       "Eigen/NLopt: tests/test_ref_eth.py); a build of the reference with real glibc/Eigen/NLopt differs by the numeric floor "
                       "(~1e-6 relative on coefficients, DESIGN.md)"}


def single_path_latency(ctx, P, n=101):
    """BASELINE metric's 'p50 latency': one 11-waypoint path at a time through the host-buffer API (waypoints in, samples and the
    result record out), n different paths; median / p90 of the wall time per call."""
    from mrs_uav_trajectory_generation_b200 import workloads as W

    ts = []
    for i in range(n + 5):
        wp = W.random_flier_path(90000 + i, 11)
        off = np.array([0, len(wp)], np.int32)
        t0 = time.perf_counter()
        res, _ = ctx.optimize_batch(off, wp, None, None, P)
        ctx.fetch_outputs(want=("smp_off", "samples"))
        dt = time.perf_counter() - t0
        if i >= 5:
            ts.append(1e3 * dt)
    ts = np.sort(np.array(ts))
    return {"p50_ms": float(np.median(ts)), "p90_ms": float(ts[int(0.9 * len(ts))]), "n": n,
            "what": "single 11-waypoint random-flier path per call, host waypoints in -> samples + result record on the host (configs[0]-style single problem)"}


DUMP_PATHS = 4096            # paths whose full outputs are written
DUMP_LIMIT = 64 << 20        # bytes, all files together


def dump_outputs(out_dir, ctx, res):
    """Writes what a caller of the timed call receives for the last timed step, as float64 .npy files that two builds can be
    compared with file by file.  For a fixed seeded sample of paths (path_index.npy, ascending): their final waypoints, segment
    times, coefficients and samples, concatenated in path order (path p contributes n_waypoints[p] waypoints, n_waypoints[p] - 1
    segments and n_samples[p] samples).  The result records (result_<field>.npy, one value per path) cover every path while they
    take at most half of DUMP_LIMIT (batches up to 262144 paths), the sampled paths only beyond that.  The sample is halved until
    all files fit DUMP_LIMIT; one path always fits."""
    out = ctx.fetch_outputs()
    B = len(res)
    all_records = B * len(res.dtype.names) * 8 <= DUMP_LIMIT // 2

    def gather(idx):
        s0, s1 = out["seg_off"][idx], out["seg_off"][idx + 1]
        m0, m1 = out["smp_off"][idx], out["smp_off"][idx + 1]
        cat = lambda a, lo, hi: np.concatenate([a[l:h] for l, h in zip(lo, hi)]).astype(np.float64)
        rec = res if all_records else res[idx]
        arrays = {"result_" + k: rec[k].astype(np.float64) for k in res.dtype.names}
        arrays.update({"path_index": idx.astype(np.float64), "wp": cat(out["wp"], s0 + idx, s1 + idx + 1), "times": cat(out["times"], s0, s1),
                       "coef": cat(out["coef"], s0, s1), "samples": cat(out["samples"], m0, m1)})
        return arrays

    idx = np.sort(np.random.default_rng(20261020).permutation(B)[:DUMP_PATHS])
    arrays = gather(idx)
    while len(idx) > 1 and sum(a.nbytes for a in arrays.values()) > DUMP_LIMIT:
        idx = idx[::2]
        arrays = gather(idx)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_reference(args, rank, world):
    if rank != 0:
        return
    n = args.ref_paths
    vals = []
    cores = os.cpu_count()
    for _ in range(args.warmup):
        cpu_baseline(max(64, n // 8), 0)
    t_tot = 0.0
    for k in range(args.steps):
        v, cores, dt, ok = cpu_baseline(n, 1 + k)
        vals.append(v)
        t_tot += dt
    value = n * args.steps / t_tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "configs[2]: random-flier paths (11 waypoints), full optimize(): time allocation + scaling + deviation subdivision + dt=0.2 sampling",
                   "paths_per_step": n, "note": "reference arm = oracle (Eigen-free CPU restatement; the reference itself needs Eigen/NLopt/ROS, absent here), all host threads"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": f"{n} paths per step x {args.steps} steps, {cores} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=RESULT_OUT or sys.stdout, flush=True)


RESULT_OUT = None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="paths per GPU per step")
    ap.add_argument("--ref-paths", type=int, default=2048, help="paths per step of the CPU reference arm")
    ap.add_argument("--cpu-sample", type=int, default=4096, help="paths of the cpu_baseline leg")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--same-batch", action="store_true", help="diagnostic: every rank gets rank 0's batch (separates batch-to-batch work variance from the box)")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE line, the JSON result: anything libraries print on fd 1 meanwhile (NCCL's version banner
    # under NCCL_DEBUG=VERSION, for one) is sent to stderr
    sys.stdout.flush()
    result_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        global RESULT_OUT
        RESULT_OUT = result_out
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import mrs_uav_trajectory_generation_b200 as tg
    from mrs_uav_trajectory_generation_b200 import workloads as W

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = tg.Context(tg.Library(os.environ.get("TG_LIB") or None), local_rank)
    P = ctx.L.default_params()
    B = args.batch
    wp_off, wp = W.random_flier_paths_fast(B, first_index=0 if args.same_batch else rank)
    d_wp = torch.from_numpy(wp).cuda()
    h_wp = torch.from_numpy(wp).pin_memory()
    wp_pinned = h_wp.numpy()

    def step_resident():
        res, totals = ctx.optimize_batch(wp_off, d_wp.data_ptr(), None, None, P, inputs_on_device=True)
        return res, totals, ctx.last_device_ms()

    for _ in range(args.warmup):
        res, totals, _ = step_resident()
    c0 = ctx.counters()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    dev_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res, totals, ms = step_resident()
        dev_ms += ms
    torch.cuda.synchronize()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    clocks = sampler.stop()
    barrier()
    c1 = ctx.counters()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, res)
    tmax = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dev_ms_max, wall_ms_max = float(tmax[0]), float(tmax[1])
    # per-rank breakdown (what the scaling residual is made of): device ms, wall ms and median SM clock of every rank
    mine = torch.tensor([dev_ms / args.steps, wall_ms / args.steps, clocks.get("sm_mhz") or 0.0, float(res["rounds"].max()), float(res["n_waypoints"].sum() - B)],
                        dtype=torch.float64, device="cuda")
    if world > 1:
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
    else:
        allr = [mine]
    # every rank draws its own batch (first_index = rank): subdivision rounds and final segments say how much work it happened to get
    per_rank = [{"rank": i, "dev_ms": round(float(t[0]), 3), "wall_ms": round(float(t[1]), 3), "sm_mhz": float(t[2]), "max_rounds": int(t[3]), "final_segments": int(t[4])}
                for i, t in enumerate(allr)]
    value = world * B * args.steps / (dev_ms_max * 1e-3)

    # ---- e2e: host (pinned) inputs, H2D inside the call, samples + per-problem results read back every step
    out_bufs = None
    totM = int(totals[1])
    pin_samples = torch.empty((int(totM * 1.05) + 1024, 4), dtype=torch.float64).pin_memory()
    h2d = wp.nbytes + wp_off.nbytes
    d2h = 0
    barrier()
    t0 = time.perf_counter()
    pin_np = pin_samples.numpy()
    for _ in range(args.steps):
        # host buffers in, samples + per-path results out: the call a user makes (tg_optimize_batch_streamed copies the samples of the
        # paths that have finished while the later subdivision rounds still run; path p owns rows begin[p] : begin[p] + n_samples[p])
        res_e, totals_e, begin_e = ctx.optimize_batch_streamed(wp_off, wp_pinned, pin_np, None, None, P, inputs_on_device=False)
        d2h = int(totals_e[1]) * 32 + begin_e.nbytes + res_e.nbytes
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    # outside the timed region: the streamed rows are, path by path, the rows tg_fetch_outputs returns
    chk = ctx.fetch_outputs(want=("smp_off", "samples"))
    streamed_ok = True
    for p in range(0, B, max(1, B // 4096)):
        n, m0 = int(res_e["n_samples"][p]), int(chk["smp_off"][p])
        streamed_ok = streamed_ok and bool(np.array_equal(pin_np[begin_e[p]:begin_e[p] + n], chk["samples"][m0:m0 + n]))
    if not streamed_ok:
        raise RuntimeError("streamed samples differ from tg_fetch_outputs")
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(te[0])

    # ---- per-kernel profile of one extra step (not timed) -> roofline of the dominant kernel
    roofline = None
    prof_table = None
    if rank == 0 and not args.no_profile:
        fp64_fma = ctx.fp64_peak_tflops(0)
        fp64_nofma = ctx.fp64_peak_tflops(1)
        ctx.set_profiling(True)
        ca = ctx.counters()
        step_resident()
        cb = ctx.counters()
        prof = ctx.profile()
        ctx.set_profiling(False)
        tot_ms = sum(v[0] for v in prof.values())
        prof_table = {k: {"ms": round(v[0], 3), "launches": v[1], "share": round(v[0] / tot_ms, 4)} for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
        hbm_peak, how = load_peaks()
        traffic_db = {}
        try:  # DRAM bytes per launch from the committed ncu --set full captures (never measured under the bench itself)
            with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
                traffic_db = json.load(f)
        except Exception:
            pass

        def kernel_flops(name, items):
            if name.startswith("refill:ExtremaRawFn") or name.startswith("jt:"):
                return float(items)  # counted in the kernel: stage-machine blocks executed x their operation counts
            if "CoefCost" in name:
                return None
            if "Solve" in name:
                return None  # split below between the solve launches by their instance counts
            if "SetupMellinger" in name or "SetupBase" in name:
                return None
            return None

        solve_names = [k for k in prof if "Solve" in k and "CoefCost" not in k and "CostSum" not in k]
        solve_items = sum(prof[k][2] for k in solve_names) or 1
        setup_names = [k for k in prof if "Setup" in k]
        coef_names = [k for k in prof if "CoefCost" in k]
        coef_items = sum(prof[k][2] for k in coef_names) or 1
        # record setup runs in two stages: heads (Q, Dinv, X: 3(N-r)^2 + 525 = 717 flop per item) and rows of H (4 N^2 = 400 flop per item)
        def setup_weight(k):
            return 400.0 if "SetupMellingerFn<1>" in k else (717.0 if "SetupMellingerFn<0>" in k else 4717.0)

        setup_items = sum(prof[k][2] * setup_weight(k) for k in setup_names) or 1
        rooflines = {}
        for name, (ms, launches, items) in prof.items():
            fl = kernel_flops(name, items)
            if fl is None and name in solve_names:
                fl = (cb["flops_solve"] - ca["flops_solve"]) * items / solve_items
            if fl is None and name in coef_names:
                fl = (cb["flops_coef"] - ca["flops_coef"]) * items / coef_items
            if fl is None and name in setup_names:
                fl = (cb["flops_setup"] - ca["flops_setup"]) * items * setup_weight(name) / setup_items
            if not fl or ms <= 0:
                continue
            achieved = fl / (ms * 1e-3) / 1e12
            tr = traffic_db.get(name)
            rooflines[name] = {"bound": "fp64", "kernel": name, "achieved": achieved, "peak": fp64_nofma, "unit": "TFLOP/s",
                               "frac": achieved / fp64_nofma if fp64_nofma else None,
                               "traffic": tr["bytes_per_launch"] if tr else None, "traffic_note": ("ncu dram__bytes_read.sum + dram__bytes_write.sum, " + tr["launch"]) if tr else None,
                               "avg_launch_ms": ms / launches, "launches": launches, "share_of_step": ms / tot_ms, "algorithmic_flops_per_launch": fl / launches}
        if rooflines:
            top_name = max(rooflines, key=lambda k: rooflines[k]["share_of_step"])
            roofline = dict(rooflines[top_name])
            roofline["peak_note"] = (f"FP64 pipe measured live: DMUL+DADD (-fmad=false mix) {fp64_nofma:.2f} TFLOP/s, DFMA {fp64_fma:.2f} TFLOP/s; "
                                     f"HBM {hbm_peak} GB/s ({how}) is not the bound for this path (SURVEY.md 8d)")
            roofline["flops_note"] = ("Jenkins-Traub kernels: operations counted in the kernel per executed stage-machine block; solve / setup / coefficient kernels: "
                                      "SURVEY.md 8(d) formulas x the instances launched")
            roofline["others"] = {k: {"frac": round(v["frac"], 4), "achieved": round(v["achieved"], 3), "share_of_step": round(v["share_of_step"], 4)}
                                  for k, v in sorted(rooflines.items(), key=lambda kv: -kv[1]["share_of_step"]) if k != top_name}

    # ---- CPU baseline on a bounded sample (rank 0, N = 1 only)
    cpu = None
    parity = None
    latency = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, cores, dt, ok, sample = cpu_baseline(args.cpu_sample, 0, keep=True)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"first {args.cpu_sample} paths of the same workload, oracle (Eigen-free C++ restatement, -O3, no FMA), {cores} host threads, {dt:.1f} s"}
        parity = parity_on_sample(ctx, P, sample)
    if rank == 0:
        latency = single_path_latency(ctx, P)

    if rank == 0:
        launches = (c1["launches"] - c0["launches"])
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {
                "workload": "configs[2]: 65536 random-flier paths (11 waypoints = 10 segments) per GPU, full optimize(): Mellinger time allocation by NLopt-LD_LBFGS-style PLIS (maxeval 10, every evaluation with its gradient), "
                            "Jenkins-Traub time scaling, deviation check 0.05 m with <=6 midpoint-subdivision rounds, dt=0.2 s sampling",
                "paths_per_gpu_per_step": B, "parallelism": f"problem-index sharding x{world}, no data-path collective",
                "l2": "per-step working set (segment records ~3.4 GB per evaluation) >> 126 MB L2, no explicit flush needed",
                "timing": "CUDA events on the library's stream around each batch call (tg_last_device_ms), max over ranks",
                "wall_ms_per_step": wall_ms_max / args.steps,
                "batches": "every rank gets rank 0's batch (--same-batch diagnostic)" if args.same_batch else "rank r draws its own batch (generator stream r)",
            },
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": int(d2h) * world,
                    "call": "tg_optimize_batch_streamed: pinned host waypoints in; per-path results and all samples out into pinned host memory, "
                            "the samples of finished paths copied while later subdivision rounds run; wall clock over the timed steps",
                    "streamed_equals_fetched": bool(streamed_ok)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "per_rank": per_rank,
            "stats": {"success_rate": float(res["success"].mean()), "safe_rate": float(res["safe"].mean()), "mean_rounds": float(res["rounds"].mean()),
                      "mean_final_segments": float(res["n_waypoints"].mean() - 1), "mean_samples": float(res["n_samples"].mean()),
                      "solves_per_step": int((c1["solves"] - c0["solves"]) / args.steps), "root_finds_reference_equivalent_per_step": int((c1["root_finds"] - c0["root_finds"]) / args.steps),
                      "root_finds_executed_per_step": int((c1["root_finds_executed"] - c0["root_finds_executed"]) / args.steps)},
        }
        if roofline:
            line["roofline"] = roofline
        if prof_table:
            line["kernel_profile"] = prof_table
        if cpu:
            line["cpu_baseline"] = cpu
        if parity:
            line["parity"] = parity
        if latency:
            line["p50_latency_ms"] = latency["p50_ms"]
            line["latency"] = latency
        print(json.dumps(line), file=result_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
