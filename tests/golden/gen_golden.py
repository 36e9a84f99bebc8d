#!/usr/bin/env python3
"""Generates the committed golden fixtures of tests/golden/ (run where a checkout of the reference is present:
$TG_REFERENCE_DIR, else BASELINE.json's reference_path).

  rpoly_reference.npz   zeros returned by the REFERENCE's own Jenkins-Traub file
                        (src/eth_trajectory_generation/rpoly/rpoly_ak1.cpp of that checkout, compiled unmodified by
                        oracle/Makefile into oracle/_ref/libref_rpoly.so) for 600 polynomials of the kinds the path meets:
                        extremum polynomials of real trajectory segments (degrees 15/13/11/7/6/5), random polynomials
                        with exact zeros at the origin, vanishing leading coefficients, clustered zeros.
  ref_eth.npz           outputs of the REFERENCE's own eth_trajectory_generation classes (every translation unit of the
                        library compiled unmodified by oracle/Makefile into oracle/_ref/libref_eth.so against the stand-ins of
                        oracle/ref_shim/) for eight random-flier problems: linear solve (coefficients, cost), Euclidean / Baca
                        segment times, per-segment maxima, scaleSegmentTimesToMeetConstraints, sampleWholeTrajectory,
                        PolynomialOptimizationNonLinear::optimize (Mellinger + LD_LBFGS stand-in).  The oracle must
                        reproduce them bit for bit in glibc math mode (tests/test_golden.py); the GPU is compared with them
                        within the published numeric floor (tests/test_gpu_parity.py).
  pipeline_oracle.npz   outputs of the oracle's full pipeline (findTrajectory + validation + subdivision) for the two
                        config-1 fixtures (SURVEY.md 8d F1a, F1b) and eight random-flier paths: final waypoints, segment
                        times, coefficients, samples, verdicts and counts.  A regression pin of the node-level restatement
                        (src/mrs_trajectory_generation.cpp needs ROS and cannot be compiled here).
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_lib as O  # noqa: E402
from mrs_uav_trajectory_generation_b200 import workloads as W  # noqa: E402


def extremum_polys(coef):
    """Increasing-power coefficient vectors handed to findRootsJenkinsTraub for one segment (eth/segment.cpp:122-145)."""
    out = []
    fact = lambda k, j: float(np.prod(np.arange(j - k + 1, j + 1))) if j >= k else 0.0
    for k in (1, 2, 3):
        nd, ndd = 10 - k, 9 - k
        acc = np.zeros(nd + ndd - 1)
        for dim in (0, 1):
            c = coef[dim]
            d = np.array([c[j + k] * fact(k, j + k) for j in range(nd)])
            dd = np.array([c[j + k + 1] * fact(k + 1, j + k + 1) for j in range(ndd)])
            acc += np.convolve(d, dd)
        out.append(acc)
        for dim in (2, 3):
            c = coef[dim]
            v = np.zeros(10)
            for j in range(10 - k - 1):
                v[j] = c[j + k + 1] * fact(k + 1, j + k + 1)
            out.append(v)
    return out


def ref_eth_fixtures():
    """Class-level input / output pairs computed by the reference's own code (oracle/_ref/libref_eth.so)."""
    ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_eth.so"))
    dp, u8p = C.POINTER(C.c_double), C.POINTER(C.c_uint8)
    P = lambda a, t=dp: a.ctypes.data_as(t)
    L = np.array(O.DEFAULT_LIMITS, dtype=np.float64)
    store = {"n": np.array(8), "limits": L}
    for q in range(8):
        V = 11 if q < 6 else 4 + q
        r = 2 if q % 3 != 2 else 4
        wp = np.ascontiguousarray(W.random_flier_path(700 + q, V))
        m = np.ones(V, np.uint8)
        m[0] = m[-1] = (1 << (r + 1)) - 1
        v = np.zeros((V, 5, 4))
        v[:, 0, :] = wp
        S = V - 1
        e, b = np.zeros(S), np.zeros(S)
        ref.ref_estimate_times(V, P(wp), P(L), P(e), P(b))
        coef = np.zeros((S, 4, 10))
        cost = C.c_double()
        assert ref.ref_solve_linear(V, P(m, u8p), P(v), P(e), r, P(coef), C.byref(cost), None, None) == 0
        mx = np.zeros((S, 9))
        ref.ref_segment_maxima(S, P(coef), P(e), P(mx))
        sc, st = coef.copy(), e.copy()
        within = C.c_int()
        ref.ref_scale_times(S, P(sc), P(st), P(L), C.byref(within))
        smp = np.zeros((4096, 19))
        tns = np.zeros(4096, np.int64)
        n = ref.ref_sample(S, P(sc), P(st), C.c_double(0.2), 4096, P(smp), tns.ctypes.data_as(C.POINTER(C.c_int64)))
        assert n > 0
        at, ac = e.copy(), np.zeros((S, 4, 10))
        code, ne, fc = C.c_int(), C.c_int(), C.c_double()
        ref.ref_time_alloc(V, P(m, u8p), P(v), P(at), r, 10, C.c_double(0.05), C.c_double(0.1), P(L), P(ac), C.byref(code), C.byref(ne), C.byref(fc))
        store.update({f"wp_{q}": wp, f"mask_{q}": m, f"vals_{q}": v, f"r_{q}": np.array(r), f"euclid_{q}": e, f"baca_{q}": b, f"coef_{q}": coef,
                      f"cost_{q}": np.array(cost.value), f"maxima_{q}": mx, f"scaled_coef_{q}": sc, f"scaled_times_{q}": st,
                      f"within_{q}": np.array(within.value), f"samples_{q}": smp[:n].copy(), f"tns_{q}": tns[:n].copy(), f"alloc_times_{q}": at,
                      f"alloc_coef_{q}": ac, f"alloc_meta_{q}": np.array([code.value, ne.value]), f"alloc_cost_{q}": np.array(fc.value)})
    np.savez_compressed(os.path.join(HERE, "ref_eth.npz"), **store)
    print("ref_eth.npz: 8 problems")


def main():
    O.build_oracle(ref=True)
    assert O.ref_lib() is not None, "needs a checkout of ctu-mrs/mrs_uav_trajectory_generation (TG_REFERENCE_DIR or BASELINE.json reference_path)"
    O.set_math_mode(O.MATH_DET)
    rng = np.random.default_rng(20261017)
    polys = []
    # extremum polynomials of real segments
    for p in range(12):
        r = O.optimize_path(W.random_flier_path(p, 11), params=O.default_params(check_deviation=0))
        for s in range(0, len(r["times"]), 3):
            polys += extremum_polys(r["coeffs"][s])
    # synthetic stress cases
    for i in range(240):
        n = int(rng.integers(3, 17))
        c = rng.standard_normal(n) * np.exp(rng.uniform(-4, 4, n))
        if i % 5 == 0:
            c[: int(rng.integers(1, 3))] = 0.0          # zeros at the origin
        if i % 7 == 0:
            c[-int(rng.integers(1, 3)):] = 0.0          # vanishing leading coefficients (trimmed by the wrapper)
        if i % 11 == 0:
            roots = np.concatenate([np.full(3, rng.uniform(-2, 2)), rng.uniform(-3, 3, max(n - 4, 1))])
            c = np.poly(roots)[::-1]                    # a triple zero
        polys.append(c)
    polys = polys[:600]
    L = max(len(c) for c in polys)
    P = np.zeros((len(polys), L))
    n_c = np.zeros(len(polys), np.int32)
    RE = np.zeros((len(polys), L))
    IM = np.zeros((len(polys), L))
    n_r = np.zeros(len(polys), np.int32)
    ok = np.zeros(len(polys), np.uint8)
    for i, c in enumerate(polys):
        re, im, success = O.find_roots(c, use_ref=True)
        P[i, : len(c)] = c
        n_c[i] = len(c)
        RE[i, : len(re)] = re
        IM[i, : len(im)] = im
        n_r[i] = len(re)
        ok[i] = success
    np.savez_compressed(os.path.join(HERE, "rpoly_reference.npz"), coeffs=P, n_coeffs=n_c, re=RE, im=IM, n_roots=n_r, ok=ok)
    print("rpoly_reference.npz:", len(polys), "polynomials,", int(n_r.sum()), "zeros")

    ref_eth_fixtures()

    paths = [W.F1A_WAYPOINTS, W.F1B_WAYPOINTS] + [W.random_flier_path(100 + p, 11) for p in range(8)]
    inits = [W.init14(W.F1A_INIT_HEADING), W.init14(W.F1B_INIT_HEADING)] + [None] * 8
    store = {}
    for p, (wp, init) in enumerate(zip(paths, inits)):
        r = O.optimize_path(wp, init=init)
        res = r["res"]
        store[f"wp_in_{p}"] = np.asarray(wp, dtype=np.float64)
        store[f"init_{p}"] = np.zeros(0) if init is None else init
        store[f"wp_{p}"] = r["wp"]
        store[f"times_{p}"] = r["times"]
        store[f"coef_{p}"] = r["coeffs"]
        store[f"samples_{p}"] = r["samples"]
        store[f"meta_{p}"] = np.array([res.success, res.rounds, res.safe, res.n_waypoints, res.n_samples, res.nlopt_code, res.n_evals, res.n_scale_passes],
                                      dtype=np.int64)
    store["n"] = np.array(len(paths))
    np.savez_compressed(os.path.join(HERE, "pipeline_oracle.npz"), **store)
    print("pipeline_oracle.npz:", len(paths), "paths")


if __name__ == "__main__":
    main()
