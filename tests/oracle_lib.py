"""ctypes access to oracle/liboracle.so and oracle/_ref/libref_rpoly.so (TEST INFRASTRUCTURE ONLY).

The oracle is the CPU restatement of the reference; the product package never imports this module.
"""
import ctypes as C
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
N, D, HALF = 10, 4, 5

MATH_LIBM, MATH_DET = 0, 1


class Params(C.Structure):
    """Mirrors tg_params (include/tg_b200.h) and orc_params (oracle/capi.cpp)."""

    _fields_ = [
        ("derivative_to_optimize", C.c_int),
        ("max_evals", C.c_int),
        ("f_rel", C.c_double),
        ("x_rel", C.c_double),
        ("limits", C.c_double * 9),
        ("dt", C.c_double),
        ("check_deviation", C.c_int),
        ("max_deviation", C.c_double),
        ("max_deviation_iters", C.c_int),
        ("first_segment_checked", C.c_int),
        ("max_len_factor", C.c_double),
        ("min_len_factor", C.c_double),
        ("run_time_alloc", C.c_int),
        ("override_heading_atan2", C.c_int),
    ]


# SURVEY.md 8(d): builder-chosen dynamics limits for all synthetic runs
DEFAULT_LIMITS = (4.0, 2.0, 2.0, 1.0, 20.0, 20.0, 1.0, 2.0, 10.0)


def default_params(**kw):
    p = Params()
    p.derivative_to_optimize = 2
    p.max_evals = 10
    p.f_rel = 0.05
    p.x_rel = 0.1
    for i, v in enumerate(DEFAULT_LIMITS):
        p.limits[i] = v
    p.dt = 0.2
    p.check_deviation = 1
    p.max_deviation = 0.05
    p.max_deviation_iters = 6
    p.first_segment_checked = 1
    p.max_len_factor = 3.0
    p.min_len_factor = 0.33
    p.run_time_alloc = 1
    for k, v in kw.items():
        if k == "limits":
            for i, x in enumerate(v):
                p.limits[i] = x
        else:
            setattr(p, k, v)
    return p


class Result(C.Structure):
    _fields_ = [
        ("status", C.c_int),
        ("success", C.c_int),
        ("nlopt_code", C.c_int),
        ("n_evals", C.c_int),
        ("rounds", C.c_int),
        ("safe", C.c_int),
        ("n_waypoints", C.c_int),
        ("n_samples", C.c_int),
        ("n_scale_passes", C.c_int),
        ("overflow", C.c_int),
        ("max_dev", C.c_double),
        ("final_cost", C.c_double),
        ("baca_total", C.c_double),
        ("total_solves", C.c_longlong),
        ("total_root_calls", C.c_longlong),
        ("total_evals", C.c_longlong),
    ]


def reference_dir():
    """The checkout of the original ctu-mrs/mrs_uav_trajectory_generation that oracle/Makefile compiles into oracle/_ref/:
    $TG_REFERENCE_DIR, else the reference_path BASELINE.json records (the same rule as oracle/Makefile); None where it is
    absent.  The repository does not contain it: without it the live comparisons with the reference's own code skip, and only
    the reference outputs stored under tests/golden/ are compared with."""
    d = os.environ.get("TG_REFERENCE_DIR")
    if not d:
        with open(os.path.join(ROOT, "BASELINE.json")) as f:
            d = json.load(f).get("reference_path")
    return os.path.abspath(d) if d and os.path.isdir(d) else None


REFERENCE = reference_dir()


def build_oracle(ref=True):
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "liboracle.so"])
    if ref and REFERENCE:
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "ref", "REFERENCE=" + REFERENCE])


_lib = None
_ref = None
dp = C.POINTER(C.c_double)
u8p = C.POINTER(C.c_uint8)
ip = C.POINTER(C.c_int)


def _ptr(a, t=dp):
    return a.ctypes.data_as(t) if a is not None else None


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(ORACLE_DIR, "liboracle.so")
        if not os.path.exists(path):
            build_oracle(ref=False)
        _lib = C.CDLL(path)
        _lib.orc_math.restype = C.c_double
        _lib.orc_math.argtypes = [C.c_int, C.c_double, C.c_double]
        _lib.orc_dist_from_segment.restype = C.c_double
    return _lib


def ref_lib():
    """The reference's own rpoly_ak1.cpp, compiled by oracle/Makefile (None when unavailable)."""
    global _ref
    if _ref is None:
        path = os.path.join(ORACLE_DIR, "_ref", "libref_rpoly.so")
        if not os.path.exists(path):
            if not REFERENCE:
                return None
            build_oracle(ref=True)
        _ref = C.CDLL(path)
    return _ref


def set_math_mode(mode):
    lib().orc_set_math_mode(int(mode))


def set_scale_tolerance(tol):
    lib().orc_set_scale_tolerance.argtypes = [C.c_double]
    lib().orc_set_scale_tolerance(float(tol))


def math_fn(fn, x, y=0.0):
    return lib().orc_math(fn, float(x), float(y))


def segment_matrices(T, r):
    A = np.zeros((N, N))
    Ai = np.zeros((N, N))
    Q = np.zeros((N, N))
    lib().orc_segment_matrices(C.c_double(T), int(r), _ptr(A), _ptr(Ai), _ptr(Q))
    return A, Ai, Q


def solve_linear(mask, vals, times, r):
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    times = np.ascontiguousarray(times, dtype=np.float64)
    V = mask.shape[0]
    S = V - 1
    coeffs = np.zeros((S, D, N))
    cost = C.c_double()
    dims = (C.c_int * 2)()
    dpv = np.zeros(D * HALF * V)
    rc = lib().orc_solve_linear(V, _ptr(mask, u8p), _ptr(vals), _ptr(times), int(r), _ptr(coeffs), C.byref(cost), _ptr(dpv), dims)
    assert rc == 0
    nfree = dims[1]
    return coeffs, cost.value, dpv[: D * nfree].reshape(D, nfree), (dims[0], dims[1])


def time_alloc(mask, vals, times, r=2, params=None):
    """PolynomialOptimizationNonLinear::optimize() from vertices (Mellinger loop + time scaling + final solve)."""
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    t = np.array(times, dtype=np.float64, copy=True)
    V = len(mask)
    coeffs = np.empty((V - 1, D, N))
    code, ev, passes = C.c_int(0), C.c_int(0), C.c_int(0)
    cost = C.c_double(0)
    P = params or default_params()
    rc = lib().orc_time_alloc(V, _ptr(mask, u8p), _ptr(vals), _ptr(t), int(r), C.byref(P), _ptr(coeffs), C.byref(code),
                              C.byref(ev), C.byref(passes), C.byref(cost))
    assert rc == 0
    return {"times": t, "coef": coeffs, "nlopt_code": code.value, "n_evals": ev.value, "n_scale_passes": passes.value, "final_cost": cost.value}


def dense_R(mask, vals, times, r):
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    times = np.ascontiguousarray(times, dtype=np.float64)
    V = mask.shape[0]
    n = HALF * V
    R = np.zeros((n, n))
    assert lib().orc_dense_R(V, _ptr(mask, u8p), _ptr(vals), _ptr(times), int(r), _ptr(R)) == 0
    return R


def find_roots(coeffs_increasing, use_ref=False):
    c = np.ascontiguousarray(coeffs_increasing, dtype=np.float64)
    re = np.zeros(64)
    im = np.zeros(64)
    ok = C.c_int()
    if use_ref:
        n = ref_lib().ref_find_roots_jt(_ptr(c), len(c), _ptr(re), _ptr(im), C.byref(ok))
    else:
        n = lib().orc_find_roots(_ptr(c), len(c), _ptr(re), _ptr(im), C.byref(ok))
    return re[:n].copy(), im[:n].copy(), bool(ok.value)


def segment_maxima(coeffs, times):
    coeffs = np.ascontiguousarray(coeffs, dtype=np.float64)
    times = np.ascontiguousarray(times, dtype=np.float64)
    S = len(times)
    out = np.zeros((S, 9))
    lib().orc_segment_maxima(S, _ptr(coeffs), _ptr(times), _ptr(out))
    return out


def max_magnitude(coeffs, times, derivative):
    """computeMaximumOfMagnitude (lin_impl.h:477-508) of one trajectory -> (time, value, segment_idx)."""
    coeffs = np.ascontiguousarray(coeffs, dtype=np.float64)
    times = np.ascontiguousarray(times, dtype=np.float64)
    t, v, i = C.c_double(), C.c_double(), C.c_int()
    lib().orc_max_magnitude(len(times), _ptr(coeffs), _ptr(times), int(derivative), C.byref(t), C.byref(v), C.byref(i))
    return t.value, v.value, i.value


def scale_times(coeffs, times, limits=DEFAULT_LIMITS):
    coeffs = np.array(coeffs, dtype=np.float64, order="C")
    times = np.array(times, dtype=np.float64)
    lim = np.array(limits, dtype=np.float64)
    w = C.c_int()
    passes = lib().orc_scale_times(len(times), _ptr(coeffs), _ptr(times), _ptr(lim), C.byref(w))
    return coeffs, times, passes, bool(w.value)


def estimate_times(pos4, limits=DEFAULT_LIMITS):
    pos4 = np.ascontiguousarray(pos4, dtype=np.float64)
    V = pos4.shape[0]
    lim = np.array(limits, dtype=np.float64)
    e = np.zeros(V - 1)
    b = np.zeros(V - 1)
    lib().orc_estimate_times(V, _ptr(pos4), _ptr(lim), _ptr(e), _ptr(b))
    return e, b


def sample(coeffs, times, dt, cap=100000):
    coeffs = np.ascontiguousarray(coeffs, dtype=np.float64)
    times = np.ascontiguousarray(times, dtype=np.float64)
    out = np.zeros((cap, 19))
    tns = np.zeros(cap, dtype=np.int64)
    n = lib().orc_sample(len(times), _ptr(coeffs), _ptr(times), C.c_double(dt), cap, _ptr(out), tns.ctypes.data_as(C.POINTER(C.c_int64)))
    assert n >= 0
    return out[:n].copy(), tns[:n].copy()


def trajectory_evaluate(coeffs, times, t, deriv):
    coeffs = np.ascontiguousarray(coeffs, dtype=np.float64)
    times = np.ascontiguousarray(times, dtype=np.float64)
    out = np.zeros(4)
    ok = lib().orc_trajectory_evaluate(len(times), _ptr(coeffs), _ptr(times), C.c_double(t), int(deriv), _ptr(out))
    return out, bool(ok)


def preprocess_path(wp, stop_at=None, min_dist=0.05, straightener=False, max_dev=0.05, max_hdg_dev=0.1):
    wp = np.ascontiguousarray(wp, dtype=np.float64)
    V = len(wp)
    stop = np.zeros(V, np.uint8) if stop_at is None else np.ascontiguousarray(stop_at, dtype=np.uint8)
    owp = np.zeros((V, 4))
    ostop = np.zeros(V, np.uint8)
    n = lib().orc_preprocess_path(V, _ptr(wp), _ptr(stop, u8p), C.c_double(min_dist), int(bool(straightener)), C.c_double(max_dev), C.c_double(max_hdg_dev),
                                  _ptr(owp), _ptr(ostop, u8p))
    return owp[:n].copy(), ostop[:n].copy()


def fallback_sample(wp, stop_at=None, limits=DEFAULT_LIMITS, dt=0.2, stopping_time=2.0, cap=200000):
    wp = np.ascontiguousarray(wp, dtype=np.float64)
    V = len(wp)
    stop = np.zeros(V, np.uint8) if stop_at is None else np.ascontiguousarray(stop_at, dtype=np.uint8)
    lim = np.array(limits, dtype=np.float64)
    out = np.zeros((cap, 4))
    n = lib().orc_fallback_sample(V, _ptr(wp), _ptr(stop, u8p), _ptr(lim), C.c_double(dt), C.c_double(stopping_time), cap, _ptr(out))
    assert n >= 0
    return out[:n].copy()


def waypoint_idxs(samples, wp):
    samples = np.ascontiguousarray(samples, dtype=np.float64)
    wp = np.ascontiguousarray(wp, dtype=np.float64)
    idx = np.zeros(len(wp) + 1, dtype=np.int32)
    n = lib().orc_waypoint_idxs(len(samples), _ptr(samples), len(wp), _ptr(wp), idx.ctypes.data_as(C.POINTER(C.c_int)))
    return idx[:n].copy()


def dist_from_segment(p, a, b):
    p, a, b = (np.ascontiguousarray(x, dtype=np.float64) for x in (p, a, b))
    return lib().orc_dist_from_segment(_ptr(p), _ptr(a), _ptr(b))


def init14(heading, vel=(0, 0, 0, 0), acc=(0, 0, 0, 0), jerk=(0, 0, 0, 0)):
    return np.array([1.0, heading, *vel, *acc, *jerk], dtype=np.float64)


def optimize_path(wp, stop_at=None, init=None, params=None, cap_wp=None, cap_samples=20000):
    wp = np.ascontiguousarray(wp, dtype=np.float64)
    V = wp.shape[0]
    stop = np.zeros(V, dtype=np.uint8) if stop_at is None else np.ascontiguousarray(stop_at, dtype=np.uint8)
    params = params or default_params()
    cap_wp = cap_wp or (V - 1) * 64 + 1
    res = Result()
    wp_out = np.zeros((cap_wp, 4))
    times = np.zeros(cap_wp - 1)
    coeffs = np.zeros((cap_wp - 1, D, N))
    smp = np.zeros((cap_samples, 4))
    lib().orc_optimize_path(V, _ptr(wp), _ptr(stop, u8p), _ptr(init) if init is not None else None, C.byref(params), C.byref(res),
                            cap_wp, _ptr(wp_out), _ptr(times), _ptr(coeffs), cap_samples, _ptr(smp))
    assert not res.overflow
    Vf = res.n_waypoints
    return dict(res=res, wp=wp_out[:Vf].copy(), times=times[: Vf - 1].copy(), coeffs=coeffs[: Vf - 1].copy(),
                samples=smp[: res.n_samples].copy())


def optimize_batch(wp_off, wp, stop_at=None, init=None, params=None, cap_wp=64, cap_samples=1024, nthreads=0, want_outputs=True):
    wp_off = np.ascontiguousarray(wp_off, dtype=np.int32)
    wp = np.ascontiguousarray(wp, dtype=np.float64)
    B = len(wp_off) - 1
    params = params or default_params()
    res = (Result * B)()
    if want_outputs:
        wp_out = np.zeros((B, cap_wp, 4))
        times = np.zeros((B, cap_wp - 1))
        coeffs = np.zeros((B, cap_wp - 1, D, N))
        smp = np.zeros((B, cap_samples, 4))
    else:
        wp_out = times = coeffs = smp = None
    stop = None if stop_at is None else np.ascontiguousarray(stop_at, dtype=np.uint8)
    used = lib().orc_optimize_batch(B, _ptr(wp_off, ip), _ptr(wp), _ptr(stop, u8p) if stop is not None else None,
                                    _ptr(init) if init is not None else None, C.byref(params), res, cap_wp, _ptr(wp_out),
                                    _ptr(times), _ptr(coeffs), cap_samples, _ptr(smp), int(nthreads))
    return dict(res=res, wp=wp_out, times=times, coeffs=coeffs, samples=smp, threads=used)


def objective(mask, vals, r, method, x, time_penalty=500.0, use_soft=True, soft_weight=100.0, con_deriv=(), con_value=(), nthreads=0):
    """objectiveFunctionTime / objectiveFunctionTimeAndConstraints (nl_impl.h:567-722) at K candidate vectors -> total[K], parts[K][3]."""
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    x = np.ascontiguousarray(x, dtype=np.float64)
    K, nvar = x.shape
    cd = np.ascontiguousarray(con_deriv, dtype=np.int32)
    cv = np.ascontiguousarray(con_value, dtype=np.float64)
    total, parts = np.zeros(K), np.zeros((K, 3))
    lib().orc_objective(len(mask), _ptr(mask, C.POINTER(C.c_uint8)), _ptr(vals), int(r), int(method), K, _ptr(x), nvar, C.c_double(time_penalty),
                        int(bool(use_soft)), C.c_double(soft_weight), len(cd), _ptr(cd, C.POINTER(C.c_int)), _ptr(cv), _ptr(total), _ptr(parts),
                        int(nthreads))
    return total, parts


def sweep_costs(mask, vals, r, cand_times, nthreads=0):
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    cand = np.ascontiguousarray(cand_times, dtype=np.float64)
    K = cand.shape[0]
    costs = np.zeros(K)
    lib().orc_sweep_costs(mask.shape[0], _ptr(mask, u8p), _ptr(vals), int(r), K, _ptr(cand), _ptr(costs), int(nthreads))
    return costs


class OracleN:
    """The restatement compiled for another even coefficient count (oracle/Makefile: liboracle_n{6,8,12}.so = the same sources
    with -DORC_N); n = 10 is liboracle.so itself.  Each library has its own math-mode switch."""

    def __init__(self, n, mode=MATH_DET):
        self.N, self.HALF = int(n), int(n) // 2
        name = "liboracle.so" if self.N == 10 else f"liboracle_n{self.N}.so"
        path = os.path.join(ORACLE_DIR, name)
        if not os.path.exists(path):
            subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, name])
        self.lib = C.CDLL(path)
        self.lib.orc_set_math_mode(int(mode))

    def solve_linear(self, mask, vals, times, r):
        """vals [V][N/2][4] -> coef [S][4][N], cost"""
        mask = np.ascontiguousarray(mask, dtype=np.uint8)
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        V = mask.shape[0]
        coeffs = np.zeros((V - 1, D, self.N))
        cost = C.c_double()
        dims = (C.c_int * 2)()
        dpv = np.zeros(D * self.HALF * V)
        rc = self.lib.orc_solve_linear(V, _ptr(mask, u8p), _ptr(vals), _ptr(times), int(r), _ptr(coeffs), C.byref(cost), _ptr(dpv), dims)
        assert rc == 0
        return coeffs, cost.value

    def trajectory_evaluate(self, coeffs, times, t, deriv):
        coeffs = np.ascontiguousarray(coeffs, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        out = np.zeros(4)
        ok = self.lib.orc_trajectory_evaluate(len(times), _ptr(coeffs), _ptr(times), C.c_double(float(t)), int(deriv), _ptr(out))
        return out, bool(ok)

    def sample(self, coeffs, times, dt, cap=100000):
        coeffs = np.ascontiguousarray(coeffs, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        out = np.zeros((cap, 19))
        n = self.lib.orc_sample(len(times), _ptr(coeffs), _ptr(times), C.c_double(float(dt)), cap, _ptr(out), None)
        assert n >= 0
        return out[:n].copy()
