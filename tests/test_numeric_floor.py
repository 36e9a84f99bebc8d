"""The numeric floor of this path: how far two CORRECT implementations of the reference's algorithm may land from each other.

north_star asks for coefficients within 1e-9 relative of the reference's CPU path.  That holds bit for bit between the CUDA
kernels and the oracle because both follow one written-down operation order and one deterministic libm
(include/tg_detmath.h).  Against a build of the reference with a real libm and real Eigen it cannot hold, for a reason that
has nothing to do with this implementation: the reduced system Rpp has cond ~ 1e8 .. 1e13, so a single-ulp difference
anywhere upstream (glibc's pow is not correctly rounded on ~0.2 % of its calls; Eigen's products and SparseQR sum in an
order that cannot be known here) moves the solution by cond * 2^-53.  These tests MEASURE that floor and pin the verdicts,
counts and sample tolerances that do survive it:

  1. oracle in detmath mode vs oracle in glibc mode, full pipeline: verdicts, subdivision rounds, evaluation / scaling-pass /
     waypoint / sample counts identical on every path; sample positions within 1e-6 m; coefficient deviation recorded;
  2. band LU (this project's solver) vs a Householder QR of the same matrix (the reference's own code compiled against the
     stand-in Eigen with REF_SHIM_QR_HOUSEHOLDER, oracle/_ref/libref_eth_qr.so): coefficient deviation recorded;
  3. both against an mpmath (50 digit) solve of the same fp64 matrix: forward error of the free derivatives relative to
     cond(Rpp) * eps -- the band LU without pivoting is as accurate as the QR on these matrices.
The recorded numbers are quoted in DESIGN.md ("numeric floor").
"""
import ctypes as C
import os

import mpmath as mp
import numpy as np
import pytest

import oracle_lib as O
import parity_checks as PC
from mrs_uav_trajectory_generation_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _meta(r):
    return (r.success, r.rounds, r.safe, r.n_waypoints, r.n_samples, r.nlopt_code, r.n_evals, r.n_scale_passes, r.status)


def test_detmath_vs_glibc_pipeline(oracle, record_property):
    B = 256
    off, wp = W.random_flier_paths_fast(B)[:2]
    outs = {}
    try:
        for mode in (O.MATH_DET, O.MATH_LIBM):
            O.set_math_mode(mode)
            outs[mode] = O.optimize_batch(off, wp, cap_wp=96, cap_samples=2048)
    finally:
        O.set_math_mode(O.MATH_DET)
    a, b = outs[O.MATH_DET], outs[O.MATH_LIBM]
    exact, worst_c, worst_s, worst_t = 0, 0.0, 0.0, 0.0
    for p in range(B):
        ra, rb = a["res"][p], b["res"][p]
        assert _meta(ra) == _meta(rb), p  # feasibility verdicts, subdivision and sample counts survive the libm change
        S, M = ra.n_waypoints - 1, ra.n_samples
        ca, cb = a["coeffs"][p, :S], b["coeffs"][p, :S]
        sa, sb = a["samples"][p, :M], b["samples"][p, :M]
        ta, tb = a["times"][p, :S], b["times"][p, :S]
        assert np.array_equal(a["wp"][p, : S + 1], b["wp"][p, : S + 1])
        exact += int(np.array_equal(ca, cb) and np.array_equal(sa, sb) and np.array_equal(ta, tb))
        worst_c = max(worst_c, PC.coef_rel_err(ca, cb, tb))
        worst_s = max(worst_s, float(np.abs(sa[:, :3] - sb[:, :3]).max()))
        worst_t = max(worst_t, float(np.abs(ta / tb - 1.0).max()))
    print(f"detmath vs glibc, {B} paths: verdicts/counts identical on all; bit-identical outputs on {exact}; worst coefficient deviation "
          f"{worst_c:.2e} relative, worst sample position deviation {worst_s:.2e} m, worst segment-time deviation {worst_t:.2e} relative")
    record_property("floor_det_vs_libm", (exact, worst_c, worst_s, worst_t))
    assert worst_s <= 1e-6      # north_star: sampled positions within 1e-6 m
    assert worst_c <= 1e-4      # the floor itself (measured ~1e-6); a regression here means a real difference, not rounding


def _problem(i, V=11):
    wp = W.random_flier_path(900 + i, V)
    m = np.ones(V, np.uint8)
    m[0] = m[-1] = 7
    v = np.zeros((V, 5, 4))
    v[:, 0, :] = wp
    t = O.estimate_times(wp)[0]
    return m, v, t


def _mp_solve(m, v, t):
    """Exact (50 digit) solution of the reduced system as formed in fp64: d_p = Rpp^-1 (-(Rpf d_f)); returns d_p [4][n_free], cond."""
    mp.mp.dps = 50
    V = len(m)
    R = O.dense_R(m, v, t, 2)
    fixed = [(vv, k) for vv in range(V) for k in range(5) if (m[vv] >> k) & 1]
    nf = len(fixed)
    n = R.shape[0] - nf
    Rpp, Rpf = R[nf:, nf:], R[nf:, :nf]
    A = mp.matrix(Rpp.tolist())
    out = np.zeros((4, n))
    for d in range(4):
        df = np.array([v[vv, k, d] for vv, k in fixed])
        rhs = mp.matrix([-sum(mp.mpf(float(Rpf[i, j])) * mp.mpf(float(df[j])) for j in range(nf)) for i in range(n)])
        x = mp.lu_solve(A, rhs)
        out[d] = [float(x[i]) for i in range(n)]
    return out, float(np.linalg.cond(Rpp))


def test_band_lu_vs_qr_vs_exact(oracle, record_property):
    qr = None
    if O.REFERENCE:
        O.build_oracle(ref=True)
        qr = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_eth_qr.so"))
    O.set_math_mode(O.MATH_LIBM)
    try:
        worst_lu, worst_qr, worst_lu_qr, worst_cond = 0.0, 0.0, 0.0, 0.0
        for i in range(8):
            m, v, t = _problem(i)
            # stretch two cases towards the ill-conditioned end (short next to long segments)
            if i >= 6:
                t = t * np.where(np.arange(len(t)) % 2 == 0, 0.15, 4.0)
            c, cost, d, dims = O.solve_linear(m, v, t, 2)
            exact, cond = _mp_solve(m, v, t)
            scale = np.abs(exact).max(axis=1, keepdims=True)
            e_lu = float((np.abs(d - exact) / scale).max())
            worst_lu = max(worst_lu, e_lu / (cond * 2.0 ** -53))
            worst_cond = max(worst_cond, cond)
            if qr is not None:
                V = len(m)
                c2 = np.zeros((V - 1, 4, 10))
                cost2 = C.c_double()
                d2 = np.zeros(4 * 5 * V)
                dims2 = np.zeros(2, np.int32)
                dp = C.POINTER(C.c_double)
                qr.ref_solve_linear(V, m.ctypes.data_as(C.POINTER(C.c_uint8)), np.ascontiguousarray(v).ctypes.data_as(dp), np.ascontiguousarray(t).ctypes.data_as(dp), 2,
                                    c2.ctypes.data_as(dp), C.byref(cost2), d2.ctypes.data_as(dp), dims2.ctypes.data_as(C.POINTER(C.c_int)))
                dq = d2[: 4 * dims2[1]].reshape(4, dims2[1])
                worst_qr = max(worst_qr, float((np.abs(dq - exact) / scale).max()) / (cond * 2.0 ** -53))
                worst_lu_qr = max(worst_lu_qr, PC.coef_rel_err(c, c2, t))
        print(f"reduced systems: cond(Rpp) up to {worst_cond:.1e}; forward error / (cond * eps): band LU {worst_lu:.3f}, Householder QR {worst_qr:.3f}; "
              f"coefficients LU vs QR differ by up to {worst_lu_qr:.2e} relative")
        record_property("floor_lu_qr", (worst_cond, worst_lu, worst_qr, worst_lu_qr))
        # unpivoted LU on the full band is backward stable here: its forward error stays a small fraction of cond * eps
        assert worst_lu <= 1.0
        if qr is not None:
            assert worst_qr <= 1.0
    finally:
        O.set_math_mode(O.MATH_DET)
