"""ctypes binding of the C ABI in include/tg_b200.h (libtg_b200.so).

This is the thin FFI layer; the reference-shaped host API lives in api.py.  There is no CPU fallback: if the CUDA
library is missing or no GPU is usable, loading / context creation raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(_HERE, "libtg_b200.so")

N, D, HALF = 10, 4, 5


class Params(C.Structure):
    """tg_params (include/tg_b200.h)."""

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


class DfoParams(C.Structure):
    """tg_dfo_params (include/tg_b200.h): the NonlinearOptimizationParameters fields the derivative-free methods read."""

    _fields_ = [
        ("time_alloc_method", C.c_int),
        ("derivative_to_optimize", C.c_int),
        ("max_iterations", C.c_int),
        ("f_rel", C.c_double),
        ("x_rel", C.c_double),
        ("initial_stepsize_rel", C.c_double),
        ("time_penalty", C.c_double),
        ("use_soft_constraints", C.c_int),
        ("soft_constraint_weight", C.c_double),
    ]


class Result(C.Structure):
    """tg_result (include/tg_b200.h)."""

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


RESULT_DTYPE = np.dtype(
    [
        ("status", "i4"), ("success", "i4"), ("nlopt_code", "i4"), ("n_evals", "i4"), ("rounds", "i4"), ("safe", "i4"),
        ("n_waypoints", "i4"), ("n_samples", "i4"), ("n_scale_passes", "i4"), ("overflow", "i4"),
        ("max_dev", "f8"), ("final_cost", "f8"), ("baca_total", "f8"),
        ("total_solves", "i8"), ("total_root_calls", "i8"), ("total_evals", "i8"),
    ],
    align=True,
)
assert RESULT_DTYPE.itemsize == C.sizeof(Result)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_u8p = C.POINTER(C.c_uint8)
_llp = C.POINTER(C.c_longlong)


class TgError(RuntimeError):
    pass


def _p(a, t=_dp):
    if a is None:
        return None
    if isinstance(a, int):  # raw (device) address
        return C.cast(C.c_void_p(a), t)
    return a.ctypes.data_as(t)


class Library:
    """A loaded libtg_b200.so (or, in tests only, the host emulation library with the same ABI)."""

    def __init__(self, path=None):
        path = path or DEFAULT_LIB
        if not os.path.exists(path):
            raise TgError(
                f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback."
            )
        self.path = path
        L = self.lib = C.CDLL(path)
        L.tg_version.restype = C.c_char_p
        L.tg_last_error.restype = C.c_char_p
        L.tg_last_error.argtypes = [C.c_void_p]
        L.tg_last_device_ms.restype = C.c_double
        L.tg_last_device_ms.argtypes = [C.c_void_p]
        L.tg_detmath_eval.restype = C.c_double
        L.tg_detmath_eval.argtypes = [C.c_int, C.c_double, C.c_double]
        L.tg_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.tg_ctx_destroy.argtypes = [C.c_void_p]
        L.tg_get_counters.argtypes = [C.c_void_p, _llp]
        L.tg_get_flop_counters.argtypes = [C.c_void_p, _dp]
        L.tg_optimize_batch.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _u8p, _dp, C.POINTER(Params), C.c_int, C.c_void_p, _llp]
        L.tg_optimize_batch_streamed.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _u8p, _dp, C.POINTER(Params), C.c_int, C.c_void_p, _llp, _dp,
                                                  C.c_longlong, _llp]
        L.tg_fetch_outputs.argtypes = [C.c_void_p, _ip, _dp, _dp, _dp, _ip, _dp]
        L.tg_solve_linear_batch.argtypes = [C.c_void_p, C.c_int, _ip, _u8p, _dp, _dp, C.c_int, _dp, _dp]
        L.tg_time_alloc_batch.argtypes = [C.c_void_p, C.c_int, _ip, _u8p, _dp, _dp, C.POINTER(Params), _dp, _ip, _ip, _ip, _dp]
        L.tg_preprocess_paths.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _u8p, C.c_double, C.c_int, C.c_double, C.c_double, _ip, _dp, _u8p]
        L.tg_fallback_sample_batch.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _u8p, _dp, C.c_double, C.c_double, _ip, _dp]
        L.tg_waypoint_idxs_batch.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _ip, _dp, _ip, _ip]
        L.tg_sample_batch.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _dp, C.c_double, _ip, _dp, _dp]
        L.tg_evaluate_batch.argtypes = [C.c_void_p, C.c_int, _dp, _dp, C.c_int, _dp, C.c_int, _dp, _u8p]
        L.tg_extrema_batch.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp]
        L.tg_solve_linear_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _u8p, _dp, _dp, C.c_int, _dp, _dp]
        L.tg_solve_linear_free_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _u8p, _dp, _dp, C.c_int, _dp, _dp, _dp]
        L.tg_set_free_constraints_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _u8p, _dp, _dp, C.c_int, _dp, _dp, _dp]
        L.tg_evaluate_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, C.c_int, _dp, C.c_int, _dp, _u8p]
        L.tg_sample_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, C.c_double, _ip, _dp, _dp]
        L.tg_sample_range_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, _dp, C.c_double, _ip, _dp, _dp, _llp]
        L.tg_evaluate_range_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, _dp, C.c_double, C.c_int, _ip, _dp, _dp]
        L.tg_extrema_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp]
        L.tg_max_magnitude_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, C.c_int, _dp, _dp, _ip]
        L.tg_scale_times_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _dp, _dp, _dp, _ip, _u8p]
        L.tg_time_alloc_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _u8p, _dp, _dp, C.POINTER(Params), _dp, _ip, _ip, _ip, _dp]
        L.tg_objective_batch.argtypes = [C.c_void_p, C.c_int, _u8p, _dp, C.c_int, C.c_int, C.c_longlong, _dp, C.c_int, C.c_double, C.c_int, C.c_double,
                                         C.c_int, _ip, _dp, _dp, _dp, _dp]
        L.tg_default_dfo_params.argtypes = [C.POINTER(DfoParams)]
        L.tg_time_alloc_dfo_batch.argtypes = [C.c_void_p, C.c_int, _ip, _u8p, _dp, _dp, C.POINTER(DfoParams), C.c_int, _ip, _ip, _dp, _dp, _dp, _ip,
                                              _ip, _dp, _dp]
        L.tg_objective_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _u8p, _dp, C.c_int, C.c_int, C.c_longlong, _dp, C.c_int, C.c_double,
                                            C.c_int, C.c_double, C.c_int, _ip, _dp, _dp, _dp, _dp]
        L.tg_time_alloc_dfo_batch_nd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _ip, _u8p, _dp, _dp, C.POINTER(DfoParams), C.c_int, _ip, _ip,
                                                 _dp, _dp, _dp, _ip, _ip, _dp, _dp]
        L.tg_max_magnitude_batch.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _dp, C.c_int, _dp, _dp, _ip]
        L.tg_scale_times_batch.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _dp, _dp, _ip, _u8p]
        L.tg_estimate_segment_times_batch.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _dp, _dp, _dp]
        L.tg_sweep_costs.argtypes = [C.c_void_p, C.c_int, _u8p, _dp, C.c_int, C.c_longlong, _dp, C.c_int, _dp, _llp, _dp]
        L.tg_default_params.argtypes = [C.POINTER(Params)]
        L.tg_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.tg_get_profile.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int, _dp, _llp, _llp]
        L.tg_measure_fp64_peak.restype = C.c_double
        L.tg_measure_fp64_peak.argtypes = [C.c_void_p, C.c_int]

    def version(self):
        return self.lib.tg_version().decode()

    def default_params(self, **kw):
        p = Params()
        self.lib.tg_default_params(C.byref(p))
        for k, v in kw.items():
            if k == "limits":
                for i, x in enumerate(v):
                    p.limits[i] = x
            else:
                setattr(p, k, v)
        return p

    def default_dfo_params(self, **kw):
        p = DfoParams()
        self.lib.tg_default_dfo_params(C.byref(p))
        for k, v in kw.items():
            setattr(p, k, v)
        return p

    @staticmethod
    def copy_params(p):
        q = Params()
        C.memmove(C.byref(q), C.byref(p), C.sizeof(Params))
        return q

    def detmath(self, fn, x, y=0.0):
        return self.lib.tg_detmath_eval(int(fn), float(x), float(y))


class Context:
    """tg_ctx: one CUDA device + stream.  Not thread-safe; use one per GPU / thread."""

    def __init__(self, library=None, device=0):
        self.L = library or Library()
        h = C.c_void_p()
        rc = self.L.lib.tg_ctx_create(int(device), C.byref(h))
        if rc != 0 or not h:
            raise TgError(f"tg_ctx_create(device={device}) failed with code {rc}: no usable CUDA device (no CPU fallback)")
        self.h = h
        self._B = 0

    def close(self):
        if self.h:
            self.L.lib.tg_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise TgError(f"tg call failed ({rc}): {self.L.lib.tg_last_error(self.h).decode()}")

    def counters(self):
        c = (C.c_longlong * 16)()
        self.L.lib.tg_get_counters(self.h, c)
        f = (C.c_double * 4)()
        self.L.lib.tg_get_flop_counters(self.h, f)
        return dict(launches=c[0], solves=c[1], evals=c[2], root_finds=c[3], segment_setups=c[4], samples=c[5],
                    mellinger_solves=c[6], mellinger_launches=c[7], root_finds_executed=c[8], flops_solve=f[0], flops_setup=f[1], flops_sample=f[2],
                    flops_coef=f[3])

    def set_profiling(self, on):
        self.L.lib.tg_set_profiling(self.h, 1 if on else 0)

    def profile(self):
        """Per-kernel device time since profiling was switched on: {kernel: (ms, launches, items)}."""
        import subprocess

        cap = 64
        names = C.create_string_buffer(1 << 16)
        ms = (C.c_double * cap)()
        ln = (C.c_longlong * cap)()
        it = (C.c_longlong * cap)()
        n = self.L.lib.tg_get_profile(self.h, cap, names, len(names), ms, ln, it)
        out = {}
        mangled = names.value.decode().split("\n")[:max(n, 0)]
        for i, m in enumerate(mangled):
            prefix, _, core = m.rpartition(":")  # "thread:<typeid>" / "refill:ExtremaRawFn<1>" / "<typeid>"
            try:
                nm = subprocess.run(["c++filt", "-t", core], capture_output=True, text=True).stdout.strip() or core
            except Exception:
                nm = core
            out[(prefix + ":" if prefix else "") + nm.replace("tg::", "")] = (ms[i], ln[i], it[i])
        return out

    def test_find_roots(self, coeffs, ncoef):
        """Test hook: the device Jenkins-Traub on polynomials coeffs[n][16] (increasing powers, ncoef[n] used) -> re, im [n][16], nroots[n]."""
        c = np.ascontiguousarray(coeffs, dtype=np.float64)
        nc = np.ascontiguousarray(ncoef, dtype=np.int32)
        n = len(nc)
        assert c.shape == (n, 16)
        re, im, nr = np.zeros((n, 16)), np.zeros((n, 16)), np.zeros(n, dtype=np.int32)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
        self._check(self.L.lib.tg_test_find_roots_batch(self.h, n, c.ctypes.data_as(dp), nc.ctypes.data_as(ip), re.ctypes.data_as(dp), im.ctypes.data_as(dp),
                                                        nr.ctypes.data_as(ip)))
        return re, im, nr

    def test_set_scale_tolerance(self, tol):
        self.L.lib.tg_test_set_scale_tolerance.argtypes = [C.c_void_p, C.c_double]
        self._check(self.L.lib.tg_test_set_scale_tolerance(self.h, float(tol)))

    def fp64_peak_tflops(self, mode=1):
        return self.L.lib.tg_measure_fp64_peak(self.h, int(mode))

    def last_device_ms(self):
        return self.L.lib.tg_last_device_ms(self.h)

    # ---- the hot path ------------------------------------------------------------------------------------------
    def optimize_batch(self, wp_off, wp, stop_at=None, init14=None, params=None, inputs_on_device=False):
        """wp_off: int32[B+1]; wp: float64[totV,4] (or a device address when inputs_on_device); returns (results, totals)."""
        wp_off = np.ascontiguousarray(wp_off, dtype=np.int32)
        B = len(wp_off) - 1
        if not inputs_on_device:
            wp = np.ascontiguousarray(wp, dtype=np.float64)
            stop_at = None if stop_at is None else np.ascontiguousarray(stop_at, dtype=np.uint8)
            init14 = None if init14 is None else np.ascontiguousarray(init14, dtype=np.float64)
        params = params or self.L.default_params()
        res = np.zeros(B, dtype=RESULT_DTYPE)
        totals = (C.c_longlong * 2)()
        self._check(self.L.lib.tg_optimize_batch(self.h, B, _p(wp_off, _ip), _p(wp), _p(stop_at, _u8p), _p(init14), C.byref(params),
                                                 1 if inputs_on_device else 0, res.ctypes.data_as(C.c_void_p), totals))
        self._B = B
        self._totals = (totals[0], totals[1])
        return res, self._totals

    def optimize_batch_streamed(self, wp_off, wp, samples_out, stop_at=None, init14=None, params=None, inputs_on_device=False):
        """tg_optimize_batch_streamed: optimize_batch with the samples copied into `samples_out` (float64 [cap, 4]; page-locked for a
        real overlap) while later rounds still run.  Returns (results, totals, smp_begin): path p owns rows
        smp_begin[p] : smp_begin[p] + results['n_samples'][p] (completion order, not path order)."""
        wp_off = np.ascontiguousarray(wp_off, dtype=np.int32)
        B = len(wp_off) - 1
        if not inputs_on_device:
            wp = np.ascontiguousarray(wp, dtype=np.float64)
            stop_at = None if stop_at is None else np.ascontiguousarray(stop_at, dtype=np.uint8)
            init14 = None if init14 is None else np.ascontiguousarray(init14, dtype=np.float64)
        if samples_out.dtype != np.float64 or not samples_out.flags["C_CONTIGUOUS"] or samples_out.ndim != 2 or samples_out.shape[1] != 4:
            raise ValueError("samples_out: C-contiguous float64 [cap, 4]")
        params = params or self.L.default_params()
        res = np.zeros(B, dtype=RESULT_DTYPE)
        totals = (C.c_longlong * 2)()
        begin = np.zeros(B, dtype=np.int64)
        self._check(self.L.lib.tg_optimize_batch_streamed(self.h, B, _p(wp_off, _ip), _p(wp), _p(stop_at, _u8p), _p(init14), C.byref(params),
                                                          1 if inputs_on_device else 0, res.ctypes.data_as(C.c_void_p), totals,
                                                          _p(samples_out), int(samples_out.shape[0]), _p(begin, _llp)))
        self._B = B
        self._totals = (totals[0], totals[1])
        return res, self._totals, begin

    def fetch_outputs(self, want=("seg_off", "wp", "times", "coef", "smp_off", "samples"), out=None):
        """Copies the last batch's outputs to host arrays (optionally into caller-provided pinned buffers `out`)."""
        B = self._B
        totS, totM = self._totals
        o = dict(out or {})

        def buf(name, shape, dtype):
            if name not in want:
                return None
            if name not in o:
                o[name] = np.empty(shape, dtype=dtype)
            return o[name]

        seg_off = buf("seg_off", B + 1, np.int32)
        wp = buf("wp", (totS + B, 4), np.float64)
        times = buf("times", totS, np.float64)
        coef = buf("coef", (totS, D, N), np.float64)
        smp_off = buf("smp_off", B + 1, np.int32)
        samples = buf("samples", (totM, 4), np.float64)
        self._check(self.L.lib.tg_fetch_outputs(self.h, _p(seg_off, _ip), _p(wp), _p(times), _p(coef), _p(smp_off, _ip), _p(samples)))
        return o

    # ---- class-level pieces --------------------------------------------------------------------------------------
    def solve_linear_batch(self, vtx_off, vmask, vval, times, r=2):
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        B = len(vtx_off) - 1
        totS = int(vtx_off[-1]) - B
        coef = np.empty((totS, D, N))
        cost = np.empty(B)
        self._check(self.L.lib.tg_solve_linear_batch(self.h, B, _p(vtx_off, _ip), _p(vmask, _u8p), _p(vval), _p(times), int(r), _p(coef), _p(cost)))
        return coef, cost

    def time_alloc_batch(self, vtx_off, vmask, vval, times, params=None):
        """PolynomialOptimizationNonLinear::optimize() for B problems given as vertices.  Returns a dict with the allocated
        times, the coefficients of the final solve, nlopt_code / n_evals / n_scale_passes / final_cost per problem."""
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        times = np.array(times, dtype=np.float64, copy=True)
        B = len(vtx_off) - 1
        totS = int(vtx_off[-1]) - B
        P = params or self.L.default_params()
        coef = np.empty((totS, D, N))
        code = np.zeros(B, dtype=np.int32)
        evals = np.zeros(B, dtype=np.int32)
        passes = np.zeros(B, dtype=np.int32)
        cost = np.zeros(B)
        self._check(self.L.lib.tg_time_alloc_batch(self.h, B, _p(vtx_off, _ip), _p(vmask, _u8p), _p(vval), _p(times), C.byref(P), _p(coef),
                                                   _p(code, _ip), _p(evals, _ip), _p(passes, _ip), _p(cost)))
        return {"times": times, "coef": coef, "nlopt_code": code, "n_evals": evals, "n_scale_passes": passes, "final_cost": cost}

    def time_alloc_dfo_batch(self, vtx_off, vmask, vval, times, params=None, constraints=()):
        """PolynomialOptimizationNonLinear::optimize() with a derivative-free method (0, 1, 3, 4) for B problems given as vertices.
        constraints: (dimension, derivative, value) shared by every problem.  Returns a dict with the allocated times, the
        coefficients at the final point, vval (methods 3, 4: the free slots at their final values), code / n_iterations / total per
        problem and parts [B][3] = cost_trajectory, cost_time, cost_soft_constraints."""
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        times = np.array(times, dtype=np.float64, copy=True)
        B = len(vtx_off) - 1
        totS = int(vtx_off[-1]) - B
        P = params or self.L.default_dfo_params()
        cdim = np.ascontiguousarray([c[0] for c in constraints], dtype=np.int32)
        cder = np.ascontiguousarray([c[1] for c in constraints], dtype=np.int32)
        cval = np.ascontiguousarray([c[2] for c in constraints], dtype=np.float64)
        coef = np.empty((totS, D, N))
        vval_out = vval.copy() if P.time_alloc_method >= 3 else None
        code = np.zeros(B, dtype=np.int32)
        iters = np.zeros(B, dtype=np.int32)
        total = np.zeros(B)
        parts = np.zeros((B, 3))
        self._check(self.L.lib.tg_time_alloc_dfo_batch(self.h, B, _p(vtx_off, _ip), _p(vmask, _u8p), _p(vval), _p(times), C.byref(P), len(cdim),
                                                       _p(cdim, _ip), _p(cder, _ip), _p(cval), _p(coef), _p(vval_out), _p(code, _ip),
                                                       _p(iters, _ip), _p(total), _p(parts)))
        return {"times": times, "coef": coef, "vval": vval_out, "code": code, "n_iterations": iters, "total": total, "parts": parts}

    def estimate_segment_times_batch(self, vtx_off, pos4, limits8, euclidean=True, baca=True):
        """estimateSegmentTimes (Euclidean) and estimateSegmentTimesBaca (eth/vertex.cpp:491-565, 301-485) for B vertex lists
        (tg_estimate_segment_times_batch): vtx_off int32[B+1], pos4 float64[totV, 4] = x y z heading, limits8 = v_h, v_v, a_h, a_v,
        j_h, j_v, heading speed, heading acceleration.  Returns (euclid [totS] or None, baca [totS] or None); segment s of problem p
        at vtx_off[p] - p + s."""
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        pos4 = np.ascontiguousarray(pos4, dtype=np.float64)
        lim = np.ascontiguousarray(limits8, dtype=np.float64)
        B = len(vtx_off) - 1
        if lim.shape != (8,) or pos4.ndim != 2 or pos4.shape[1] != 4 or B < 1 or pos4.shape[0] != int(vtx_off[-1]):
            raise ValueError("vtx_off [B+1] with B >= 1, pos4 [vtx_off[-1], 4] and eight limits are needed")
        totS = max(int(vtx_off[-1]) - B, 0)
        e = np.empty(totS) if euclidean else None
        b = np.empty(totS) if baca else None
        self._check(self.L.lib.tg_estimate_segment_times_batch(self.h, B, _p(vtx_off, _ip), _p(pos4), _p(lim), _p(e), _p(b)))
        return e, b

    # ---- the steps either side of the path (SURVEY.md 8f) ---------------------------------------------------------------
    def preprocess_paths(self, wp_off, wp, stop_at=None, min_waypoint_distance=0.05, straightener=False, max_deviation=0.05, max_hdg_deviation=0.1):
        """preprocessPath (node.cpp:431-500).  Returns (wp_off_out, wp_out, stop_out) as a compact ragged batch."""
        wp_off = np.ascontiguousarray(wp_off, dtype=np.int32)
        wp = np.ascontiguousarray(wp, dtype=np.float64)
        stop = None if stop_at is None else np.ascontiguousarray(stop_at, dtype=np.uint8)
        B = len(wp_off) - 1
        cnt = np.zeros(B, dtype=np.int32)
        owp = np.zeros_like(wp)
        ostop = np.zeros(len(wp), dtype=np.uint8)
        self._check(self.L.lib.tg_preprocess_paths(self.h, B, _p(wp_off, _ip), _p(wp), _p(stop, _u8p), float(min_waypoint_distance), int(bool(straightener)),
                                                   float(max_deviation), float(max_hdg_deviation), _p(cnt, _ip), _p(owp), _p(ostop, _u8p)))
        keep = np.concatenate([np.arange(wp_off[p], wp_off[p] + cnt[p]) for p in range(B)]) if B else np.zeros(0, int)
        off = np.zeros(B + 1, dtype=np.int32)
        off[1:] = np.cumsum(cnt)
        return off, owp[keep], ostop[keep]

    def fallback_sample_batch(self, wp_off, wp, stop_at=None, limits=None, dt=0.2, stopping_time=2.0):
        """findTrajectoryFallback (node.cpp:1215-1395).  Returns (smp_off, samples [M, 4])."""
        wp_off = np.ascontiguousarray(wp_off, dtype=np.int32)
        wp = np.ascontiguousarray(wp, dtype=np.float64)
        stop = None if stop_at is None else np.ascontiguousarray(stop_at, dtype=np.uint8)
        lim = np.array(list(self.L.default_params().limits) if limits is None else limits, dtype=np.float64)
        B = len(wp_off) - 1
        cnt = np.zeros(B, dtype=np.int32)
        self._check(self.L.lib.tg_fallback_sample_batch(self.h, B, _p(wp_off, _ip), _p(wp), _p(stop, _u8p), _p(lim), float(dt), float(stopping_time),
                                                        _p(cnt, _ip), None))
        smp = np.zeros((int(cnt.sum()), 4))
        if len(smp):
            self._check(self.L.lib.tg_fallback_sample_batch(self.h, B, _p(wp_off, _ip), _p(wp), _p(stop, _u8p), _p(lim), float(dt), float(stopping_time),
                                                            _p(cnt, _ip), _p(smp)))
        off = np.zeros(B + 1, dtype=np.int32)
        off[1:] = np.cumsum(cnt)
        return off, smp

    def waypoint_idxs_batch(self, smp_off, samples, wp_off, wp):
        """getWaypointInTrajectoryIdxs (node.cpp:1461-1499).  Returns a list of index arrays, one per path."""
        smp_off = np.ascontiguousarray(smp_off, dtype=np.int32)
        samples = np.ascontiguousarray(samples, dtype=np.float64)
        wp_off = np.ascontiguousarray(wp_off, dtype=np.int32)
        wp = np.ascontiguousarray(wp, dtype=np.float64)
        B = len(wp_off) - 1
        cnt = np.zeros(B, dtype=np.int32)
        idx = np.zeros(max(len(wp), 1), dtype=np.int32)
        self._check(self.L.lib.tg_waypoint_idxs_batch(self.h, B, _p(smp_off, _ip), _p(samples), _p(wp_off, _ip), _p(wp), _p(cnt, _ip), _p(idx, _ip)))
        return [idx[wp_off[p]: wp_off[p] + cnt[p]].copy() for p in range(B)]

    def sample_batch(self, seg_off, coef, times, dt, full=False):
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int32)
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        B = len(seg_off) - 1
        counts = np.zeros(B, dtype=np.int32)
        self._check(self.L.lib.tg_sample_batch(self.h, B, _p(seg_off, _ip), _p(coef), _p(times), float(dt), _p(counts, _ip), None, None))
        tot = int(counts.sum())
        samples = np.empty((tot, 4))
        fullv = np.empty((tot, 19)) if full else None
        self._check(self.L.lib.tg_sample_batch(self.h, B, _p(seg_off, _ip), _p(coef), _p(times), float(dt), _p(counts, _ip), _p(samples), _p(fullv)))
        return counts, samples, fullv

    def evaluate(self, coef, times, t, derivative=0):
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        t = np.ascontiguousarray(np.atleast_1d(t), dtype=np.float64)
        out = np.empty((len(t), 4))
        ok = np.zeros(len(t), dtype=np.uint8)
        self._check(self.L.lib.tg_evaluate_batch(self.h, len(times), _p(coef), _p(times), len(t), _p(t), int(derivative), _p(out), _p(ok, _u8p)))
        return out, ok.astype(bool)

    # ---- general shape: N in {6, 8, 10, 12} coefficients, D in 1..4 dimensions (tg_*_nd, csrc/tg_generic.cuh) ----
    def solve_linear_batch_nd(self, n_coef, dim, vtx_off, vmask, vval, times, r=2):
        """PolynomialOptimization<n_coef>(dim): vval [totV][n_coef/2][dim] -> coef [totS][dim][n_coef], cost [B]."""
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        B = len(vtx_off) - 1
        totS = int(vtx_off[-1]) - B
        assert vval.size == int(vtx_off[-1]) * (n_coef // 2) * dim and times.size == totS
        coef = np.empty((totS, dim, n_coef))
        cost = np.empty(B)
        self._check(self.L.lib.tg_solve_linear_batch_nd(self.h, int(n_coef), int(dim), B, _p(vtx_off, _ip), _p(vmask, _u8p), _p(vval), _p(times),
                                                        int(r), _p(coef), _p(cost)))
        return coef, cost

    @staticmethod
    def free_counts(n_coef, vtx_off, vmask):
        """n_free of every problem: the clear mask bits below n_coef/2 over its vertices."""
        bits = (np.asarray(vmask, dtype=np.uint8)[:, None] >> np.arange(n_coef // 2, dtype=np.uint8)) & 1
        cs = np.concatenate([[0], np.cumsum(n_coef // 2 - bits.sum(axis=1, dtype=np.int64))])
        off = np.asarray(vtx_off, dtype=np.int64)
        return cs[off[1:]] - cs[off[:-1]]

    def solve_linear_free_batch_nd(self, n_coef, dim, vtx_off, vmask, vval, times, r=2):
        """solveLinear + getFreeConstraints + getSegments + computeCost: (coef [totS][dim][n_coef], cost [B], free), free = one
        [dim][n_free] array per problem (the d_p of lin_impl.h:340-373, dimension-major)."""
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        B = len(vtx_off) - 1
        totS = int(vtx_off[-1]) - B
        assert vval.size == int(vtx_off[-1]) * (n_coef // 2) * dim and times.size == totS
        nf = self.free_counts(n_coef, vtx_off, vmask)
        coef = np.empty((totS, dim, n_coef))
        cost = np.empty(B)
        free = np.empty(max(int(nf.sum()) * dim, 1))
        self._check(self.L.lib.tg_solve_linear_free_batch_nd(self.h, int(n_coef), int(dim), B, _p(vtx_off, _ip), _p(vmask, _u8p), _p(vval), _p(times),
                                                             int(r), _p(coef), _p(cost), _p(free)))
        off = np.concatenate([[0], np.cumsum(nf * dim)])
        return coef, cost, [free[off[p]:off[p + 1]].reshape(dim, nf[p]) for p in range(B)]

    def set_free_constraints_batch_nd(self, n_coef, dim, vtx_off, vmask, vval, times, free, r=2):
        """setFreeConstraints + getSegments + computeCost: free = one [dim][n_free] array per problem -> (coef, cost)."""
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        B = len(vtx_off) - 1
        totS = int(vtx_off[-1]) - B
        assert vval.size == int(vtx_off[-1]) * (n_coef // 2) * dim and times.size == totS and len(free) == B
        nf = self.free_counts(n_coef, vtx_off, vmask)
        for p in range(B):
            if np.shape(free[p]) != (dim, nf[p]):
                raise ValueError(f"problem {p}: the free constraints are [{dim}][{nf[p]}], got {np.shape(free[p])}")
        flat = np.ascontiguousarray(np.concatenate([np.asarray(f, dtype=np.float64).reshape(-1) for f in free] + [np.zeros(1)]))
        coef = np.empty((totS, dim, n_coef))
        cost = np.empty(B)
        self._check(self.L.lib.tg_set_free_constraints_batch_nd(self.h, int(n_coef), int(dim), B, _p(vtx_off, _ip), _p(vmask, _u8p), _p(vval),
                                                                _p(times), int(r), _p(flat), _p(coef), _p(cost)))
        return coef, cost

    def evaluate_nd(self, n_coef, dim, coef, times, t, derivative=0):
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        t = np.ascontiguousarray(np.atleast_1d(t), dtype=np.float64)
        assert coef.size == len(times) * dim * n_coef
        out = np.empty((len(t), dim))
        ok = np.zeros(len(t), dtype=np.uint8)
        self._check(self.L.lib.tg_evaluate_batch_nd(self.h, int(n_coef), int(dim), len(times), _p(coef), _p(times), len(t), _p(t), int(derivative),
                                                    _p(out), _p(ok, _u8p)))
        return out, ok.astype(bool)

    def sample_batch_nd(self, n_coef, dim, seg_off, coef, times, dt, full=False):
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int32)
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        B = len(seg_off) - 1
        assert coef.size == int(seg_off[-1]) * dim * n_coef
        counts = np.zeros(B, dtype=np.int32)
        lib = self.L.lib
        self._check(lib.tg_sample_batch_nd(self.h, int(n_coef), int(dim), B, _p(seg_off, _ip), _p(coef), _p(times), float(dt), _p(counts, _ip), None, None))
        tot = int(counts.sum())
        samples = np.empty((tot, 4))
        fullv = np.empty((tot, 19)) if full else None
        self._check(lib.tg_sample_batch_nd(self.h, int(n_coef), int(dim), B, _p(seg_off, _ip), _p(coef), _p(times), float(dt), _p(counts, _ip),
                                           _p(samples), _p(fullv)))
        return counts, samples, fullv

    def _range_inputs(self, n_coef, dim, seg_off, coef, times, t_range):
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int32)
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        t_range = np.ascontiguousarray(t_range, dtype=np.float64).reshape(-1, 2)
        B = len(seg_off) - 1
        assert coef.size == int(seg_off[-1]) * dim * n_coef and t_range.shape[0] == B
        return seg_off, coef, times, t_range, B

    def sample_range_batch_nd(self, n_coef, dim, seg_off, coef, times, t_range, dt, full=False):
        """sampleTrajectoryInRange's walk over window p = t_range[p] = (t_start, t_end) of every trajectory (tg_sample_range_batch_nd):
        counts [B], samples [sum][4] (x y z heading), full [sum][19] or None, t_ns [sum] (time_from_start_ns), rows in trajectory order."""
        seg_off, coef, times, t_range, B = self._range_inputs(n_coef, dim, seg_off, coef, times, t_range)
        counts = np.zeros(B, dtype=np.int32)
        lib = self.L.lib
        args = (self.h, int(n_coef), int(dim), B, _p(seg_off, _ip), _p(coef), _p(times), _p(t_range), float(dt), _p(counts, _ip))
        self._check(lib.tg_sample_range_batch_nd(*args, None, None, None))
        tot = int(counts.sum())
        samples, t_ns = np.empty((tot, 4)), np.empty(tot, dtype=np.int64)
        fullv = np.empty((tot, 19)) if full else None
        self._check(lib.tg_sample_range_batch_nd(*args, _p(samples), _p(fullv), _p(t_ns, _llp)))
        return counts, samples, fullv, t_ns

    def evaluate_range_batch_nd(self, n_coef, dim, seg_off, coef, times, t_range, dt, derivative=0):
        """Trajectory::evaluateRange over window p = t_range[p] of every trajectory (tg_evaluate_range_batch_nd): counts [B],
        values [sum][dim] of the derivative, sampling_times [sum], rows in trajectory order."""
        seg_off, coef, times, t_range, B = self._range_inputs(n_coef, dim, seg_off, coef, times, t_range)
        counts = np.zeros(B, dtype=np.int32)
        lib = self.L.lib
        args = (self.h, int(n_coef), int(dim), B, _p(seg_off, _ip), _p(coef), _p(times), _p(t_range), float(dt), int(derivative), _p(counts, _ip))
        self._check(lib.tg_evaluate_range_batch_nd(*args, None, None))
        tot = int(counts.sum())
        out, st = np.empty((tot, dim)), np.empty(tot)
        self._check(lib.tg_evaluate_range_batch_nd(*args, _p(out), _p(st)))
        return counts, out, st

    def extrema_nd(self, n_coef, dim, coef, times):
        """Nine maxima per segment of N-coefficient, D-dimensional segments: coef [totS][dim][n_coef] -> maxima [totS][9]."""
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        assert coef.size == len(times) * dim * n_coef
        m = np.empty((len(times), 9))
        self._check(self.L.lib.tg_extrema_batch_nd(self.h, int(n_coef), int(dim), len(times), _p(coef), _p(times), _p(m)))
        return m

    def max_magnitude_nd(self, n_coef, dim, seg_off, coef, times, derivative):
        """computeMaximumOfMagnitude(derivative) of PolynomialOptimization<n_coef>(dim) per trajectory -> time[B], value[B], segment_idx[B]."""
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int32)
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        B = len(seg_off) - 1
        assert coef.size == int(seg_off[-1]) * dim * n_coef and times.size == int(seg_off[-1])
        v, t, i = np.empty(B), np.empty(B), np.empty(B, dtype=np.int32)
        self._check(self.L.lib.tg_max_magnitude_batch_nd(self.h, int(n_coef), int(dim), B, _p(seg_off, _ip), _p(coef), _p(times), int(derivative),
                                                         _p(v), _p(t), _p(i, _ip)))
        return t, v, i

    def scale_times_nd(self, n_coef, dim, seg_off, coef, times, limits):
        """scaleSegmentTimesToMeetConstraints on copies of coef [totS][dim][n_coef] / times -> coef, times, passes[B], within[B]."""
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int32)
        coef = np.array(coef, dtype=np.float64, order="C")
        times = np.array(times, dtype=np.float64)
        lim = np.ascontiguousarray(limits, dtype=np.float64)
        B = len(seg_off) - 1
        assert coef.size == int(seg_off[-1]) * dim * n_coef and times.size == int(seg_off[-1]) and lim.size == 9
        passes = np.zeros(B, dtype=np.int32)
        within = np.zeros(B, dtype=np.uint8)
        self._check(self.L.lib.tg_scale_times_batch_nd(self.h, int(n_coef), int(dim), B, _p(seg_off, _ip), _p(coef), _p(times), _p(lim), _p(passes, _ip),
                                                       _p(within, _u8p)))
        return coef, times, passes, within.astype(bool)

    def time_alloc_batch_nd(self, n_coef, dim, vtx_off, vmask, vval, times, params=None):
        """PolynomialOptimizationNonLinear<n_coef>(dim)::optimize() (Mellinger) for B problems given as vertices: vval [totV][n_coef/2][dim].
        Returns the dict of time_alloc_batch with coef [totS][dim][n_coef]."""
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        times = np.array(times, dtype=np.float64, copy=True)
        B = len(vtx_off) - 1
        totS = int(vtx_off[-1]) - B
        assert vval.size == int(vtx_off[-1]) * (n_coef // 2) * dim and times.size == totS
        P = params or self.L.default_params()
        coef = np.empty((totS, dim, n_coef))
        code = np.zeros(B, dtype=np.int32)
        evals = np.zeros(B, dtype=np.int32)
        passes = np.zeros(B, dtype=np.int32)
        cost = np.zeros(B)
        self._check(self.L.lib.tg_time_alloc_batch_nd(self.h, int(n_coef), int(dim), B, _p(vtx_off, _ip), _p(vmask, _u8p), _p(vval), _p(times), C.byref(P),
                                                      _p(coef), _p(code, _ip), _p(evals, _ip), _p(passes, _ip), _p(cost)))
        return {"times": times, "coef": coef, "nlopt_code": code, "n_evals": evals, "n_scale_passes": passes, "final_cost": cost}

    def objective_nd(self, n_coef, dim, mask, vals, r, method, x, time_penalty=500.0, use_soft=True, soft_weight=100.0, con_deriv=(),
                     con_value=(), want_coef=False):
        """objective() for PolynomialOptimizationNonLinear<n_coef>(dim): vals [V][n_coef/2][dim]; x [K][nvar], nvar = S or S + dim * n_free
        (the free derivatives dimension-major) -> total[K], parts[K][3] (and coef [K][S][dim][n_coef] with want_coef)."""
        mask = np.ascontiguousarray(mask, dtype=np.uint8)
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        x = np.ascontiguousarray(x, dtype=np.float64)
        K, nvar = x.shape
        cd = np.ascontiguousarray(con_deriv, dtype=np.int32)
        cv = np.ascontiguousarray(con_value, dtype=np.float64)
        total, parts = np.empty(K), np.empty((K, 3))
        coef = np.empty((K, len(mask) - 1, dim, n_coef)) if want_coef else None
        self._check(self.L.lib.tg_objective_batch_nd(self.h, int(n_coef), int(dim), len(mask), _p(mask, _u8p), _p(vals), int(r), int(method), K, _p(x),
                                                     nvar, float(time_penalty), int(bool(use_soft)), float(soft_weight), len(cd), _p(cd, _ip), _p(cv),
                                                     _p(total), _p(parts), _p(coef) if want_coef else None))
        return (total, parts, coef) if want_coef else (total, parts)

    def time_alloc_dfo_batch_nd(self, n_coef, dim, vtx_off, vmask, vval, times, params=None, constraints=()):
        """time_alloc_dfo_batch for PolynomialOptimizationNonLinear<n_coef>(dim): vval [totV][n_coef/2][dim], derivative_to_optimize
        0 .. n_coef/2-1.  Returns the dict of time_alloc_dfo_batch with coef [totS][dim][n_coef] and vval [totV][n_coef/2][dim]."""
        vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        times = np.array(times, dtype=np.float64, copy=True)
        B = len(vtx_off) - 1
        totS = int(vtx_off[-1]) - B
        assert vval.size == int(vtx_off[-1]) * (n_coef // 2) * dim and times.size == totS
        P = params or self.L.default_dfo_params()
        cdim = np.ascontiguousarray([c[0] for c in constraints], dtype=np.int32)
        cder = np.ascontiguousarray([c[1] for c in constraints], dtype=np.int32)
        cval = np.ascontiguousarray([c[2] for c in constraints], dtype=np.float64)
        coef = np.empty((totS, dim, n_coef))
        vval_out = vval.copy() if P.time_alloc_method >= 3 else None
        code = np.zeros(B, dtype=np.int32)
        iters = np.zeros(B, dtype=np.int32)
        total = np.zeros(B)
        parts = np.zeros((B, 3))
        self._check(self.L.lib.tg_time_alloc_dfo_batch_nd(self.h, int(n_coef), int(dim), B, _p(vtx_off, _ip), _p(vmask, _u8p), _p(vval), _p(times),
                                                          C.byref(P), len(cdim), _p(cdim, _ip), _p(cder, _ip), _p(cval), _p(coef), _p(vval_out),
                                                          _p(code, _ip), _p(iters, _ip), _p(total), _p(parts)))
        return {"times": times, "coef": coef, "vval": vval_out, "code": code, "n_iterations": iters, "total": total, "parts": parts}

    def extrema(self, coef, times):
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        m = np.empty((len(times), 9))
        self._check(self.L.lib.tg_extrema_batch(self.h, len(times), _p(coef), _p(times), _p(m)))
        return m

    def objective(self, mask, vals, r, method, x, time_penalty=500.0, use_soft=True, soft_weight=100.0, con_deriv=(), con_value=(),
                  want_coef=False):
        """objectiveFunctionTime / objectiveFunctionTimeAndConstraints (nl_impl.h:567-722) at K candidates -> total[K], parts[K][3]."""
        mask = np.ascontiguousarray(mask, dtype=np.uint8)
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        x = np.ascontiguousarray(x, dtype=np.float64)
        K, nvar = x.shape
        cd = np.ascontiguousarray(con_deriv, dtype=np.int32)
        cv = np.ascontiguousarray(con_value, dtype=np.float64)
        total, parts = np.empty(K), np.empty((K, 3))
        coef = np.empty((K, len(mask) - 1, 4, 10)) if want_coef else None
        self._check(self.L.lib.tg_objective_batch(self.h, len(mask), _p(mask, _u8p), _p(vals), int(r), int(method), K, _p(x), nvar, float(time_penalty),
                                                  int(bool(use_soft)), float(soft_weight), len(cd), _p(cd, _ip), _p(cv), _p(total), _p(parts),
                                                  _p(coef) if want_coef else None))
        return (total, parts, coef) if want_coef else (total, parts)

    def max_magnitude(self, seg_off, coef, times, derivative):
        """computeMaximumOfMagnitude(derivative) per trajectory (lin_impl.h:477-508) -> time[B], value[B], segment_idx[B]."""
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int32)
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        times = np.ascontiguousarray(times, dtype=np.float64)
        B = len(seg_off) - 1
        v, t, i = np.empty(B), np.empty(B), np.empty(B, dtype=np.int32)
        self._check(self.L.lib.tg_max_magnitude_batch(self.h, B, _p(seg_off, _ip), _p(coef), _p(times), int(derivative), _p(v), _p(t), _p(i, _ip)))
        return t, v, i

    def scale_times(self, seg_off, coef, times, limits):
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int32)
        coef = np.array(coef, dtype=np.float64, order="C")
        times = np.array(times, dtype=np.float64)
        lim = np.ascontiguousarray(limits, dtype=np.float64)
        B = len(seg_off) - 1
        passes = np.zeros(B, dtype=np.int32)
        within = np.zeros(B, dtype=np.uint8)
        self._check(self.L.lib.tg_scale_times_batch(self.h, B, _p(seg_off, _ip), _p(coef), _p(times), _p(lim), _p(passes, _ip), _p(within, _u8p)))
        return coef, times, passes, within.astype(bool)

    @staticmethod
    def sweep_best(contexts, vmask, vval, cand, r=2):
        """tg_sweep_best: candidates sharded over several contexts (one per device) of this process -> (best_cost, best_index, best_times)."""
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        cand = np.ascontiguousarray(cand, dtype=np.float64)
        K, S = cand.shape
        lib = contexts[0].L.lib
        hs = (C.c_void_p * len(contexts))(*[c.h for c in contexts])
        bi, bc = C.c_longlong(), C.c_double()
        bt = np.empty(S)
        lib.tg_sweep_best.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, _u8p, _dp, C.c_int, C.c_longlong, _dp, C.POINTER(C.c_longlong), C.POINTER(C.c_double), _dp]
        lib.tg_sweep_best.restype = C.c_int
        contexts[0]._check(lib.tg_sweep_best(hs, len(contexts), len(vmask), _p(vmask, _u8p), _p(vval), int(r), int(K), _p(cand), C.byref(bi), C.byref(bc), _p(bt)))
        return bc.value, bi.value, bt

    def sweep_costs(self, vmask, vval, cand, r=2, want_costs=True, cand_on_device=False, K=None):
        vmask = np.ascontiguousarray(vmask, dtype=np.uint8)
        vval = np.ascontiguousarray(vval, dtype=np.float64)
        V = len(vmask)
        if not cand_on_device:
            cand = np.ascontiguousarray(cand, dtype=np.float64)
            K = cand.shape[0]
        costs = np.empty(K) if want_costs else None
        bi = C.c_longlong()
        bc = C.c_double()
        self._check(self.L.lib.tg_sweep_costs(self.h, V, _p(vmask, _u8p), _p(vval), int(r), int(K), _p(cand), 1 if cand_on_device else 0,
                                              _p(costs), C.byref(bi), C.byref(bc)))
        return costs, bi.value, bc.value
