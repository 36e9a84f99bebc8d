"""Oracle pinned to the REFERENCE's own source.

oracle/Makefile compiles the reference's eth_trajectory_generation library UNMODIFIED from a checkout of the reference
($TG_REFERENCE_DIR, else the reference_path BASELINE.json records) (polynomial.cpp,
segment.cpp, trajectory.cpp, trajectory_sampling.cpp, vertex.cpp, motion_defines.cpp, timing.cpp, rpoly/rpoly_ak1.cpp and the
header templates PolynomialOptimization<10> / PolynomialOptimizationNonLinear<10>) against the stand-ins of oracle/ref_shim/
(Eigen, NLopt, mrs_lib, ROS messages, boost are absent from this image) into oracle/_ref/libref_eth.so.  These tests run the
same inputs through that library and through the restatement (oracle/liboracle.so, glibc math mode = the pure restatement)
and require the results to be BIT-IDENTICAL: every branch, loop bound, operand order and libm call of the restatement is
thereby checked against the reference's own code for SURVEY rows a3-a13, a14-a21, a23-a25.  What this does NOT pin: the
rounding of real Eigen's products / SparseQR and of a real NLopt build -- the stand-ins implement this project's numeric
contract for those (oracle/ref_shim/Eigen/shim_impl.h, oracle/plis.cpp).

The reference's sources are not part of this repository: these tests run where that checkout is present and skip elsewhere.
Without it only part of what they check is compared with stored reference outputs (tests/golden/ref_eth.npz, eight problems,
tests/test_golden.py): segment-time estimates, linear-solve coefficients and cost (r = 2, 4), per-segment maxima, time
scaling, sampling and the Mellinger time allocation.  The mapping / inverse / cost matrices, the dense R, the free derivatives,
r = 3, computeMaximumOfMagnitude, Trajectory::evaluate and the soft-constraint objectives have no stored counterpart.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
import parity_checks as PC
from mrs_uav_trajectory_generation_b200 import workloads as W

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
dp = C.POINTER(C.c_double)
u8p = C.POINTER(C.c_uint8)
ip = C.POINTER(C.c_int)


def _p(a, t=dp):
    return a.ctypes.data_as(t)


@pytest.fixture(scope="module")
def ref():
    if not O.REFERENCE:
        pytest.skip("needs a checkout of the original ctu-mrs/mrs_uav_trajectory_generation (TG_REFERENCE_DIR or BASELINE.json reference_path)")
    O.build_oracle(ref=True)
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_eth.so"))
    O.set_math_mode(O.MATH_LIBM)
    yield lib
    O.set_math_mode(O.MATH_DET)


def ref_solve_linear(lib, mask, vals, times, r):
    V = len(mask)
    S = V - 1
    coef = np.zeros((S, 4, 10))
    cost = C.c_double()
    dims = np.zeros(2, np.int32)
    dpv = np.zeros(4 * 5 * V)
    rc = lib.ref_solve_linear(V, _p(np.ascontiguousarray(mask, np.uint8), u8p), _p(np.ascontiguousarray(vals, np.float64)),
                              _p(np.ascontiguousarray(times, np.float64)), int(r), _p(coef), C.byref(cost), _p(dpv), _p(dims, ip))
    assert rc == 0
    return coef, cost.value, dpv[: 4 * dims[1]].reshape(4, dims[1]).copy(), dims


@pytest.mark.parametrize("r", [2, 3, 4])
def test_segment_matrices(ref, r):
    """setupMappingMatrix, invertMappingMatrix, computeQuadraticCostJacobian (lin_impl.h:112-121, 147-177, 605-618)."""
    for T in [0.01, 0.11, 0.37, 1.0, 2.5, 7.3, 41.0]:
        A, Ai, Q = O.segment_matrices(T, r)
        A2, Ai2, Q2 = np.zeros((10, 10)), np.zeros((10, 10)), np.zeros((10, 10))
        ref.ref_segment_matrices(C.c_double(T), r, _p(A2), _p(Ai2), _p(Q2))
        assert np.array_equal(A, A2) and np.array_equal(Ai, Ai2) and np.array_equal(Q, Q2), T


@pytest.mark.parametrize("r", [2, 3, 4])
def test_linear_solve(ref, r):
    """setupFromVertices, setupConstraintReorderingMatrix, constructR, solveLinear, updateSegmentsFromCompactConstraints,
    computeCost (lin_impl.h:61-106, 183-257, 310-373, 263-282, 127-141) on the vertex recipes the node and the tests build."""
    rng = np.random.default_rng(100 + r)
    for p in range(30):
        V = int(rng.integers(2, 16))
        m, v, t = PC.random_linear_problem(rng, V, kind=p % 6)
        c, co, d, dims = O.solve_linear(m, v, t, r)
        c2, co2, d2, dims2 = ref_solve_linear(ref, m, v, t, r)
        assert list(dims) == list(dims2)
        assert np.array_equal(d, d2), (p, np.abs(d - d2).max())
        assert np.array_equal(c, c2), (p, PC.coef_rel_err(c, c2, t))
        assert co == co2, (p, co, co2)


def test_dense_R(ref):
    """constructR (lin_impl.h:310-334): R = C^T blockdiag(H) C, every entry."""
    rng = np.random.default_rng(7)
    for p in range(6):
        V = int(rng.integers(3, 9))
        m, v, t = PC.random_linear_problem(rng, V, kind=p % 5)
        R = O.dense_R(m, v, t, 2)
        n = R.shape[0]
        R2 = np.zeros((n, n))
        assert ref.ref_dense_R(V, _p(np.ascontiguousarray(m, np.uint8), u8p), _p(np.ascontiguousarray(v)), _p(np.ascontiguousarray(t)), 2, _p(R2)) == 0
        assert np.array_equal(R, R2), np.abs(R - R2).max()


def test_segment_time_estimates(ref):
    """estimateSegmentTimes (Euclidean) and estimateSegmentTimesBaca (eth/vertex.cpp:491-565, 301-485), incl. vertical
    segments, zero-length segments, heading-dominated segments and relaxed heading limits (FLT_MAX)."""
    rng = np.random.default_rng(3)
    cases = [W.random_flier_path(i, 11) for i in range(20)]
    cases.append(np.array([[0, 0, 0, 0], [0, 0, 5, 0], [0, 0, 5, 3.0], [0, 0, 5, 3.0], [4, 0, 1, -3.0]], float))
    cases.append(np.cumsum(rng.uniform(-3, 3, (9, 4)), axis=0))
    for lim in (O.DEFAULT_LIMITS, (4.0, 2.0, 2.0, 1.0, 20.0, 20.0, 3.4028234663852886e38, 3.4028234663852886e38, 3.4028234663852886e38)):
        for wp in cases:
            e, b = O.estimate_times(wp, lim)
            V = len(wp)
            e2, b2 = np.zeros(V - 1), np.zeros(V - 1)
            L = np.array(lim, dtype=np.float64)
            ref.ref_estimate_times(V, _p(np.ascontiguousarray(wp, np.float64)), _p(L), _p(e2), _p(b2))
            assert np.array_equal(e, e2) and np.array_equal(b, b2)


def _solved(i, V=11, r=2):
    wp = W.random_flier_path(i, V)
    m = np.ones(V, np.uint8)
    m[0] = m[-1] = (1 << (r + 1)) - 1
    v = np.zeros((V, 5, 4))
    v[:, 0, :] = wp
    t = O.estimate_times(wp)[0]
    c = O.solve_linear(m, v, t, r)[0]
    return m, v, t, c


def test_extrema_and_scaling(ref):
    """computeMaxDerivatives{Horizontal,Vertical,Heading} per segment -> computeMinMaxMagnitude ->
    Segment::computeMinMaxMagnitudeCandidates -> Polynomial::computeMinMaxCandidates -> findRootsJenkinsTraub
    (eth/trajectory.cpp:211-280, 422-565; eth/segment.cpp:113-212; eth/polynomial.cpp:36-85) and
    scaleSegmentTimesToMeetConstraints (eth/trajectory.cpp:598-692)."""
    L = np.array(O.DEFAULT_LIMITS, dtype=np.float64)
    for i in range(12):
        m, v, t, c = _solved(200 + i)
        S = len(t)
        mx = O.segment_maxima(c, t)
        mx2 = np.zeros((S, 9))
        ref.ref_segment_maxima(S, _p(np.ascontiguousarray(c)), _p(np.ascontiguousarray(t)), _p(mx2))
        assert np.array_equal(mx, mx2), np.abs(mx - mx2).max()
        c1, t1, passes, within = O.scale_times(c, t)
        c2, t2 = np.ascontiguousarray(c).copy(), np.ascontiguousarray(t).copy()
        w2 = C.c_int()
        ref.ref_scale_times(S, _p(c2), _p(t2), _p(L), C.byref(w2))
        assert np.array_equal(t1, t2) and np.array_equal(c1, c2) and bool(within) == bool(w2.value)


def test_max_of_magnitude(ref):
    """computeMaximumOfMagnitude (lin_impl.h:477-508), derivatives 1..4."""
    for i in range(6):
        m, v, t, c = _solved(300 + i)
        for k in (1, 2, 3, 4):
            tm, val, idx = O.max_magnitude(c, t, k)
            a, b, ci = C.c_double(), C.c_double(), C.c_int()
            assert ref.ref_solve_max_magnitude(len(m), _p(m, u8p), _p(np.ascontiguousarray(v)), _p(np.ascontiguousarray(t)), 2, k, C.byref(a), C.byref(b),
                                               C.byref(ci)) == 0
            assert (tm, val, idx) == (a.value, b.value, ci.value)


def test_sampling_and_evaluate(ref):
    """sampleWholeTrajectory -> sampleTrajectoryInRange -> evaluateRange (eth/trajectory_sampling.cpp:49-124,
    eth/trajectory.cpp:93-151) incl. the quaternion round trip of the heading, time_from_start_ns, and Trajectory::evaluate
    (eth/trajectory.cpp:55-87)."""
    for i in range(8):
        m, v, t, c = _solved(400 + i, V=4 + i)
        S = len(t)
        for dt in (0.2, 0.01 * (i + 1), 0.37):
            smp, tns = O.sample(c, t, dt)
            out = np.zeros((len(smp) + 8, 19))
            tn2 = np.zeros(len(smp) + 8, np.int64)
            n = ref.ref_sample(S, _p(np.ascontiguousarray(c)), _p(np.ascontiguousarray(t)), C.c_double(dt), len(out), _p(out), tn2.ctypes.data_as(C.POINTER(C.c_int64)))
            assert n == len(smp)                                    # sample count: exact
            assert np.array_equal(tns, tn2[:n])                     # time_from_start_ns: exact
            assert np.array_equal(smp, out[:n]), np.abs(smp - out[:n]).max()
        tot = float(np.sum(t))
        for tq in (0.0, 0.3 * tot, float(t[0]), tot, tot + 1.0):
            for k in range(5):
                val, ok = O.trajectory_evaluate(c, t, tq, k)
                v2 = np.zeros(4)
                ok2 = ref.ref_trajectory_evaluate(S, _p(np.ascontiguousarray(c)), _p(np.ascontiguousarray(t)), C.c_double(tq), k, _p(v2))
                assert bool(ok) == bool(ok2)
                if ok:
                    assert np.array_equal(val, v2)


@pytest.mark.parametrize("r", [2, 4])
def test_time_allocation(ref, r):
    """PolynomialOptimizationNonLinear<10>::setupFromVertices / addMaximumMagnitudeConstraint / optimize ->
    optimizeTimeMellingerOuterLoop, objectiveFunctionTimeMellingerOuterLoop, getCostAndGradientMellinger,
    scaleSegmentTimesWithViolation (nl_impl.h:51-118, 159-234, 256-427, 616-649) driving the reference's own code through the
    nlopt stand-in (LD_LBFGS = oracle/plis.cpp): result code, evaluation count, final cost, times and coefficients."""
    L = np.array(O.DEFAULT_LIMITS, dtype=np.float64)
    for i in range(10):
        V = 3 + i
        wp = W.random_flier_path(500 + i, V)
        m = np.ones(V, np.uint8)
        m[0] = m[-1] = (1 << (r + 1)) - 1
        v = np.zeros((V, 5, 4))
        v[:, 0, :] = wp
        t = O.estimate_times(wp)[0]
        a = O.time_alloc(m, v, t, r, O.default_params(derivative_to_optimize=r))
        t2 = np.ascontiguousarray(t).copy()
        c2 = np.zeros((V - 1, 4, 10))
        code, ne, fc = C.c_int(), C.c_int(), C.c_double()
        ref.ref_time_alloc(V, _p(m, u8p), _p(np.ascontiguousarray(v)), _p(t2), r, 10, C.c_double(0.05), C.c_double(0.1), _p(L), _p(c2), C.byref(code), C.byref(ne),
                           C.byref(fc))
        assert (a["nlopt_code"], a["n_evals"]) == (code.value, ne.value), i
        assert a["final_cost"] == fc.value
        assert np.array_equal(a["times"], t2) and np.array_equal(a["coef"], c2), i


@pytest.mark.parametrize("method", [0, 1, 3, 4])
def test_soft_constraint_objectives(ref, method):
    """objectiveFunctionTime / objectiveFunctionTimeAndConstraints with evaluateMaximumMagnitudeAsSoftConstraint
    (nl_impl.h:567-614, 651-762), evaluated by the reference's own code at candidate vectors."""
    rng = np.random.default_rng(40 + method)
    m, v, t, c = _solved(600 + method, V=6)
    V, S = len(m), len(t)
    d = O.solve_linear(m, v, t, 2)[2]
    nfree = d.shape[1]
    K = 5
    if method >= 3:
        nvar = S + 4 * nfree
        x = np.zeros((K, nvar))
        for k in range(K):
            x[k, :S] = t * np.exp(rng.uniform(-0.2, 0.2, S))
            x[k, S:] = d.reshape(-1) * (1.0 + rng.uniform(-0.05, 0.05, 4 * nfree))
    else:
        nvar = S
        x = t[None, :] * np.exp(rng.uniform(-0.3, 0.3, (K, S)))
    cd = np.array([1, 2], np.int32)
    cv = np.array([4.0, 2.0])
    tot, parts = O.objective(m, v, 2, method, x, con_deriv=cd, con_value=cv, nthreads=1)
    tot2, parts2 = np.zeros(K), np.zeros((K, 3))
    ref.ref_objective(V, _p(m, u8p), _p(np.ascontiguousarray(v)), 2, method, K, _p(np.ascontiguousarray(x)), nvar, C.c_double(500.0), 1, C.c_double(100.0), 2,
                      _p(cd, ip), _p(cv), _p(tot2), _p(parts2))
    assert np.array_equal(parts, parts2), np.abs(parts - parts2).max()
    assert np.array_equal(tot, tot2)
