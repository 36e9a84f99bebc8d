"""tg_time_alloc_dfo_batch: the derivative-free time allocation (methods 0, 1, 3, 4; nl_impl.h:120-157, 429-536) for many problems in
one device call.  Every problem must come out exactly as the single-problem search it replaces: ReferenceSearch below is that search,
the host loop over tg_objective_batch (ctx.objective) and tg_solve_linear_batch, kept here as the pin.  Checked on the host emulation
(all three solve dispatches, a small matrix) and on the B200 (the full matrix and one call with 16 384 problems)."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
import mrs_uav_trajectory_generation_b200.api as A
from mrs_uav_trajectory_generation_b200 import workloads as W
from mrs_uav_trajectory_generation_b200._capi import D, HALF, N

TG_ERR_INVALID = -3


class ReferenceSearch:
    """The single-problem search, one tg_objective_batch call per iteration (the former DerivativeFreeTimeAllocation.optimize)."""

    kTimeLowerBound = 0.01  # kOptimizationTimeLowerBound (nl.h:143)

    def __init__(self, mask, vals, times, derivative_to_optimize, parameters, constraints, ctx):
        self.ctx = ctx
        self.P = parameters
        self.r = derivative_to_optimize
        self.mask, self.vals = mask, vals
        self.times0 = np.asarray(times, dtype=np.float64)
        self.S = len(self.times0)
        self.constraints = list(constraints)  # (dimension, derivative, value) in the order they were added
        self.with_free = parameters.time_alloc_method in (3, 4)

    def _objective(self, x, want_coef=False):
        cd = [c[1] for c in self.constraints]
        cv = [c[2] for c in self.constraints]
        return self.ctx.objective(self.mask, self.vals, self.r, self.P.time_alloc_method, x, self.P.time_penalty, self.P.use_soft_constraints,
                                  self.P.soft_constraint_weight, cd, cv, want_coef=want_coef)

    def _bounds(self, x0, free_slots):
        n = len(x0)
        lo, hi = np.full(n, -np.finfo(np.float64).max), np.full(n, np.finfo(np.float64).max)
        lo[: self.S] = self.kTimeLowerBound
        if self.with_free:
            # setFreeEndpointDerivativeHardConstraints (nl_impl.h:764-805), INCLUDING its index arithmetic: free_deriv_counter
            # advances only for derivatives <= derivative_to_optimize while the variables hold every free slot (0..4), so for
            # derivative_to_optimize < 4 the bounds land where the reference puts them, not on the slots one would expect
            n_free = len(free_slots)
            for dim, deriv, value in self.constraints:
                counter = 0
                for v in range(len(self.mask)):
                    for k in range(self.r + 1):
                        if not (self.mask[v] >> k) & 1:
                            if k == deriv:
                                at = self.S + dim * n_free + counter
                                if at < n:
                                    lo[at] = -abs(value)
                                    hi[at] = abs(value)
                            counter += 1
        # "Check if initial solution isn't already out of bounds" (nl_impl.h:497-503)
        lo = np.minimum(lo, x0)
        hi = np.maximum(hi, x0)
        return lo, hi

    def optimize(self):
        x = self.times0.copy()
        free_slots = []
        if self.with_free:
            # initial solution: solveLinear + getFreeConstraints (nl_impl.h:436-462), dimension-major
            # (read off the solved segments: derivative k at a vertex = k! c_k of the segment that starts there, or the
            # last segment's polynomial at its end)
            vtx_off = np.array([0, len(self.mask)], dtype=np.int32)
            coef, _ = self.ctx.solve_linear_batch(vtx_off, self.mask, self.vals, self.times0, self.r)
            fact = [1.0, 1.0, 2.0, 6.0, 24.0]
            for v in range(len(self.mask)):
                for k in range(5):
                    if not (self.mask[v] >> k) & 1:
                        free_slots.append((v, k))
            dp = np.zeros((D, len(free_slots)))
            for j, (v, k) in enumerate(free_slots):
                for d in range(D):
                    if v < self.S:
                        dp[d, j] = fact[k] * coef[v, d, k]
                    else:
                        c, T, acc = coef[self.S - 1, d], self.times0[-1], 0.0
                        for i in range(N - 1, k - 1, -1):
                            acc = acc * T + np.prod(np.arange(i - k + 1, i + 1, dtype=np.float64)) * c[i]
                        dp[d, j] = acc
            x = np.concatenate([x, dp.reshape(-1)])
        n = len(x)
        lo, hi = self._bounds(x, free_slots)
        step = np.where(np.abs(x) <= np.finfo(np.float64).eps, 1e-13, self.P.initial_stepsize_rel * np.abs(x))  # nl_impl.h:488-495
        f = float(self._objective(x[None, :])[0][0])
        self.n_iterations, code = 0, 5
        while self.n_iterations < self.P.max_iterations:
            self.n_iterations += 1
            cand = np.repeat(x[None, :], 2 * n, axis=0)
            idx = np.arange(n)
            cand[idx, idx] = np.minimum(x + step, hi)
            cand[n + idx, idx] = np.maximum(x - step, lo)
            tot, _ = self._objective(cand)
            k = int(np.argmin(tot))  # first minimum
            if tot[k] < f:
                f_old, f = f, float(tot[k])
                x = cand[k].copy()
                if abs(f_old - f) <= self.P.f_rel * abs(f):  # NLopt ftol_rel
                    code = 3
                    break
            else:
                step *= 0.5
                if np.all(step <= self.P.x_rel * np.abs(x)):  # NLopt xtol_rel
                    code = 4
                    break
        self.x, self.cost = x, f
        tot, parts, coef = self._objective(x[None, :], want_coef=True)
        self.cost_parts = parts[0]
        self.coef, self.times = coef[0], x[: self.S].copy()
        return code


# ---- problems -----------------------------------------------------------------------------------------------------------------
NODE_CONSTRAINTS = [(d, k, v) for d, lim in enumerate(((4.0, 2.0, 20.0), (4.0, 2.0, 20.0), (2.0, 1.0, 20.0), (1.0, 2.0, 10.0)))
                    for k, v in zip((1, 2, 3), lim)]  # the node's 12 (x, y, z, heading x velocity, acceleration, jerk)
# small limits: the free-derivative bounds bind, and land on the slots the counter quirk picks for r < 4
TIGHT_CONSTRAINTS = [(0, 1, 0.3), (1, 2, 0.2), (2, 3, 0.5), (3, 1, 0.1), (1, 1, 0.25), (0, 4, 0.4)]


def make_problems(seed, B, S_max, r):
    """Ragged random-flier problems: S = 1 .. S_max, ends fixed up to r, interior positions; some with a stop_at vertex (v, a, j
    fixed at zero), random masks and values, an initial state, no free slot at all, or initial times below 0.01."""
    rng = np.random.default_rng(seed)
    probs = []
    for p in range(B):
        S = 1 + p % S_max
        V = S + 1
        wp = W.random_flier_path(500 + seed * 1000 + p, V)
        mask = np.ones(V, np.uint8)
        vals = np.zeros((V, HALF, D))
        vals[:, 0] = wp
        mask[0] = mask[-1] = (1 << (r + 1)) - 1
        kind = p % 6
        if kind == 1 and V > 2:
            mask[V // 2] = 0b1111
        if kind == 2:
            for v in range(1, V - 1):
                mask[v] = 1 | int(rng.integers(0, 16)) << 1
                vals[v, 1:] = rng.uniform(-0.5, 0.5, (HALF - 1, D))
        if kind == 3:
            mask[:] = 31
            vals[:, 1:] = rng.uniform(-0.2, 0.2, (V, HALF - 1, D))
        if kind == 4:
            mask[0] = 0b1111
            vals[0, 1:4] = rng.uniform(-1.0, 1.0, (3, D))
        times = O.estimate_times(wp)[0].copy()
        if kind == 5:
            times[0] = 0.004
        probs.append((mask, vals, times))
    return probs


def pack(probs):
    vtx_off = np.cumsum([0] + [len(m) for m, _, _ in probs]).astype(np.int32)
    return vtx_off, np.concatenate([m for m, _, _ in probs]), np.concatenate([v for _, v, _ in probs]), np.concatenate([t for _, _, t in probs])


def nl_params(method, iters, soft, f_rel=1e-6):
    P = A.NonlinearOptimizationParameters()
    P.time_alloc_method, P.max_iterations, P.use_soft_constraints, P.f_rel = method, iters, soft, f_rel
    return P


def dfo_params(ctx, P, r):
    return ctx.L.default_dfo_params(time_alloc_method=P.time_alloc_method, derivative_to_optimize=r, max_iterations=P.max_iterations, f_rel=P.f_rel,
                                    x_rel=P.x_rel, initial_stepsize_rel=P.initial_stepsize_rel, time_penalty=P.time_penalty,
                                    use_soft_constraints=int(P.use_soft_constraints), soft_constraint_weight=P.soft_constraint_weight)


def free_values(mask, vval):
    """the free slots of vval [V][5][4], dimension-major as the search's variables hold them"""
    f = [vval[v, k] for v in range(len(mask)) for k in range(HALF) if not (mask[v] >> k) & 1]
    return np.array(f).reshape(-1, D).T.reshape(-1)


def problem_out(out, probs, p):
    vtx_off = np.cumsum([0] + [len(m) for m, _, _ in probs])
    v0, v1 = vtx_off[p], vtx_off[p + 1]
    s0, s1 = v0 - p, v1 - p - 1
    o = {"code": int(out["code"][p]), "n_iterations": int(out["n_iterations"][p]), "times": out["times"][s0:s1], "coef": out["coef"][s0:s1],
         "total": out["total"][p], "parts": out["parts"][p]}
    o["x"] = o["times"] if out["vval"] is None else np.concatenate([o["times"], free_values(probs[p][0], out["vval"][v0:v1])])
    return o


def same(a, b):
    return (a["code"] == b["code"] and a["n_iterations"] == b["n_iterations"] and np.array_equal(a["times"], b["times"])
            and np.array_equal(a["coef"], b["coef"]) and np.array_equal(a["x"], b["x"]) and a["total"] == b["total"]
            and np.array_equal(a["parts"], b["parts"]))


def check_against_reference(ctx, method, r, iters, soft, constraints, seed, B=24, S_max=12, oracle=None):
    probs = make_problems(seed, B, S_max, r)
    P = nl_params(method, iters, soft)
    out = ctx.time_alloc_dfo_batch(*pack(probs), dfo_params(ctx, P, r), constraints)
    cd, cv = [c[1] for c in constraints], [c[2] for c in constraints]
    for p, (mask, vals, times) in enumerate(probs):
        ref = ReferenceSearch(mask, vals, times, r, P, constraints, ctx)
        code = ref.optimize()
        want = {"code": code, "n_iterations": ref.n_iterations, "times": ref.times, "coef": ref.coef, "total": ref.cost, "parts": ref.cost_parts,
                "x": ref.x}
        got = problem_out(out, probs, p)
        assert same(got, want), (method, r, iters, soft, len(constraints), p, got["code"], code, got["n_iterations"], ref.n_iterations)
        if oracle is not None:  # the three terms are the oracle's objective at the returned x
            _, rp = oracle.objective(mask, vals, r, method, got["x"][None, :], P.time_penalty, soft, P.soft_constraint_weight, cd, cv)
            assert np.array_equal(got["parts"], rp[0]), (method, p)
    return out, probs


# the emulator matrix: every method, r and constraint count, the iteration limits spread over the cases (the reference search
# evaluates every candidate in full on the host, which is where the time goes)
EMU_CASES = [
    (0, 2, 25, True, NODE_CONSTRAINTS, 6), (0, 3, 1, False, [], 12), (0, 4, 10, True, TIGHT_CONSTRAINTS, 8),
    (1, 2, 10, True, TIGHT_CONSTRAINTS, 12), (1, 4, 0, True, NODE_CONSTRAINTS, 6), (1, 3, 25, False, NODE_CONSTRAINTS, 6),
    (3, 2, 10, True, TIGHT_CONSTRAINTS, 6), (3, 3, 1, True, NODE_CONSTRAINTS, 5), (3, 4, 0, False, [], 4),
    (4, 2, 10, True, NODE_CONSTRAINTS, 4), (4, 3, 10, True, TIGHT_CONSTRAINTS, 5), (4, 4, 1, False, TIGHT_CONSTRAINTS, 6),
]


@pytest.mark.parametrize("case", range(len(EMU_CASES)))
def test_equals_reference_search_on_host_emulation(emu_ctx, oracle, case):
    method, r, iters, soft, cons, S_max = EMU_CASES[case]
    check_against_reference(emu_ctx, method, r, iters, soft, cons, seed=case, S_max=S_max, oracle=oracle if case % 3 == 0 else None)


@pytest.mark.gpu
@pytest.mark.parametrize("method", [0, 1, 3, 4])
def test_equals_reference_search_on_gpu(gpu_ctx, oracle, method):
    for r in (2, 3, 4):
        for iters, soft, cons in ((0, True, NODE_CONSTRAINTS), (1, False, TIGHT_CONSTRAINTS), (10, True, TIGHT_CONSTRAINTS), (25, True, []),
                                  (25, False, TIGHT_CONSTRAINTS), (10, True, NODE_CONSTRAINTS)):
            check_against_reference(gpu_ctx, method, r, iters, soft, cons, seed=100 * method + 10 * r + iters, oracle=oracle)


def check_independence(ctx, lib, method):
    """each problem's outputs equal its own B = 1 call, and a context whose small TG_SEG_BUDGET cuts the batch into several groups
    gives the same bits"""
    from mrs_uav_trajectory_generation_b200 import Context

    r, cons = 2, TIGHT_CONSTRAINTS
    probs = make_problems(7 + method, 9, 5, r)
    P = nl_params(method, 10, True)
    prm = dfo_params(ctx, P, r)
    out = ctx.time_alloc_dfo_batch(*pack(probs), prm, cons)
    for p in range(len(probs)):
        one = ctx.time_alloc_dfo_batch(*pack(probs[p:p + 1]), prm, cons)
        assert same(problem_out(out, probs, p), problem_out(one, probs[p:p + 1], 0)), (method, p)
    old = os.environ.get("TG_SEG_BUDGET")
    os.environ["TG_SEG_BUDGET"] = "100"
    try:
        small = Context(lib, 0)
    finally:
        if old is None:
            os.environ.pop("TG_SEG_BUDGET")
        else:
            os.environ["TG_SEG_BUDGET"] = old
    out2 = small.time_alloc_dfo_batch(*pack(probs), dfo_params(small, P, r), cons)
    for p in range(len(probs)):
        assert same(problem_out(out, probs, p), problem_out(out2, probs, p)), (method, p)


@pytest.mark.parametrize("method", [0, 4])
def test_independence_on_host_emulation(emu_ctx, emu_lib, method):
    check_independence(emu_ctx, emu_lib, method)


@pytest.mark.gpu
@pytest.mark.parametrize("method", [0, 1, 3, 4])
def test_independence_on_gpu(gpu_ctx, method):
    from mrs_uav_trajectory_generation_b200 import Library

    check_independence(gpu_ctx, Library(), method)


def check_refusals(ctx):
    probs = make_problems(3, 3, 4, 2)
    vtx_off, masks, vals, times = pack(probs)
    B, totS, totV = 3, len(times), len(masks)

    def call(B=B, vtx_off=vtx_off, params=None, cons=((0, 1, 2.0),)):
        prm = params or ctx.L.default_dfo_params(time_alloc_method=3)
        cd = np.array([c[0] for c in cons], np.int32)
        ck = np.array([c[1] for c in cons], np.int32)
        cv = np.array([c[2] for c in cons], np.float64)
        outs = [times.copy(), np.full((totS, D, N), 7.0), np.full((totV, HALF, D), 7.0), np.full(B + 1, 7, np.int32), np.full(B + 1, 7, np.int32),
                np.full(B + 1, 7.0), np.full((B + 1, 3), 7.0)]
        ip, dp = C.POINTER(C.c_int), C.POINTER(C.c_double)
        rc = ctx.L.lib.tg_time_alloc_dfo_batch(ctx.h, B, vtx_off.ctypes.data_as(ip), masks.ctypes.data_as(C.POINTER(C.c_uint8)), vals.ctypes.data_as(dp),
                                               outs[0].ctypes.data_as(dp), C.byref(prm), len(cons), cd.ctypes.data_as(ip), ck.ctypes.data_as(ip),
                                               cv.ctypes.data_as(dp), outs[1].ctypes.data_as(dp), outs[2].ctypes.data_as(dp), outs[3].ctypes.data_as(ip),
                                               outs[4].ctypes.data_as(ip), outs[5].ctypes.data_as(dp), outs[6].ctypes.data_as(dp))
        untouched = (np.array_equal(outs[0], times) and np.all(outs[1] == 7.0) and np.all(outs[2] == 7.0) and np.all(outs[3] == 7)
                     and np.all(outs[4] == 7) and np.all(outs[5] == 7.0) and np.all(outs[6] == 7.0))
        return rc, untouched

    assert call()[0] == 0
    bad = [dict(B=0), dict(vtx_off=np.array([0, 1, vtx_off[2], vtx_off[3]], np.int32))]
    bad += [dict(params=ctx.L.default_dfo_params(time_alloc_method=m)) for m in (2, 5, -1)]
    bad += [dict(params=ctx.L.default_dfo_params(derivative_to_optimize=k)) for k in (1, 5)]
    bad += [dict(cons=[(0, 1, 1.0)] * 17), dict(cons=[(0, 0, 1.0)]), dict(cons=[(0, 5, 1.0)]), dict(cons=[(4, 1, 1.0)]), dict(cons=[(-1, 1, 1.0)]),
            dict(cons=[(0, 1, 1.0), (1, 2, 0.0)])]
    for kw in bad:
        rc, untouched = call(**kw)
        assert rc == TG_ERR_INVALID and untouched, kw


def test_refusals_on_host_emulation(emu_ctx):
    check_refusals(emu_ctx)


@pytest.mark.gpu
def test_refusals_on_gpu(gpu_ctx):
    check_refusals(gpu_ctx)


def check_classes(ctx):
    """DerivativeFreeTimeAllocation (through PolynomialOptimizationNonLinear.optimize) and TrajectoryGenerator.time_alloc_derivative_free
    give the batched call's results"""
    probs = make_problems(11, 4, 4, 2)
    for method in (1, 3):
        P = nl_params(method, 10, True, f_rel=0.05)
        verts_all = []
        for mask, vals, times in probs:
            verts = []
            for v in range(len(mask)):
                vx = A.Vertex(4)
                for k in range(HALF):
                    if (mask[v] >> k) & 1:
                        vx.addConstraint(k, vals[v, k])
                verts.append(vx)
            verts_all.append(verts)
        trajs, codes = A.TrajectoryGenerator(ctx=ctx).time_alloc_derivative_free(verts_all, [t for _, _, t in probs], P, NODE_CONSTRAINTS)
        for p, (mask, vals, times) in enumerate(probs):
            opt = A.PolynomialOptimizationNonLinear(4, P, ctx=ctx)
            assert opt.setupFromVertices(verts_all[p], times, 2)
            for c in NODE_CONSTRAINTS:
                opt.addMaximumMagnitudeConstraint(*c)
            assert opt.optimize() == codes[p]
            ref = ReferenceSearch(mask, vals, times, 2, P, NODE_CONSTRAINTS, ctx)
            assert ref.optimize() == codes[p]
            assert np.array_equal(opt._dfo.x, ref.x) and opt._dfo.cost == ref.cost and opt._dfo.n_iterations == ref.n_iterations
            assert np.array_equal(trajs[p].times, ref.times) and np.array_equal(trajs[p].coef, ref.coef)
            assert np.array_equal(opt.getTrajectory().coef, ref.coef)


def test_classes_on_host_emulation(emu_ctx):
    check_classes(emu_ctx)


@pytest.mark.gpu
def test_classes_on_gpu(gpu_ctx):
    check_classes(gpu_ctx)


def _run_cpp(libdir, libname, tmp_path):
    from test_cpp_shim import _run_shim

    res = _run_shim(libdir, libname, tmp_path, "test_shim_dfo_batch.cpp")
    assert res["batch_equals_single"][0][0] == 1.0
    assert res["mixed_refused"][0][0] == 1.0
    assert res["mellinger_refused"][0][0] == 1.0


def test_cpp_optimize_batch_on_host_emulation(emu_lib, tmp_path):
    _run_cpp(os.path.join(os.path.dirname(__file__), "host_emu"), "tg_emu", tmp_path)


@pytest.mark.gpu
def test_cpp_optimize_batch_on_gpu(gpu_ctx, tmp_path):
    _run_cpp(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "mrs_uav_trajectory_generation_b200"), "tg_b200", tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("method", [0, 3])
def test_gpu_at_scale(gpu_ctx, method):
    """one call with 16 384 random-flier problems (S = 10, the node's vertex recipe and 12 constraints): every output finite, and 64
    sampled problems equal the reference search"""
    B, r = 16384, 2
    probs = []
    for p in range(B):
        wp = W.random_flier_path(p, 11)
        mask = np.ones(11, np.uint8)
        mask[0] = mask[-1] = 0b111
        vals = np.zeros((11, HALF, D))
        vals[:, 0] = wp
        probs.append((mask, vals, O.estimate_times(wp)[0].copy()))
    P = nl_params(method, 10, True, f_rel=0.05)
    out = gpu_ctx.time_alloc_dfo_batch(*pack(probs), dfo_params(gpu_ctx, P, r), NODE_CONSTRAINTS)
    for k in ("times", "coef", "total", "parts"):
        assert np.all(np.isfinite(out[k])), k
    if out["vval"] is not None:
        assert np.all(np.isfinite(out["vval"]))
    for p in np.random.default_rng(5).choice(B, 64, replace=False):
        mask, vals, times = probs[p]
        ref = ReferenceSearch(mask, vals, times, r, P, NODE_CONSTRAINTS, gpu_ctx)
        code = ref.optimize()
        want = {"code": code, "n_iterations": ref.n_iterations, "times": ref.times, "coef": ref.coef, "total": ref.cost, "parts": ref.cost_parts,
                "x": ref.x}
        assert same(problem_out(out, probs, p), want), p
