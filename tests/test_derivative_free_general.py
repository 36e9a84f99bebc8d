"""tg_objective_batch_nd and tg_time_alloc_dfo_batch_nd: the derivative-free time allocation (methods 0, 1, 3, 4; nl_impl.h:120-157,
429-536) for PolynomialOptimization<N>, N in {6, 8, 10, 12}, on 1..4 dimensions.

Pinned bit for bit on both sides: the objective equals the oracle's orc_objective compiled for that N (vals and x zero-padded to four
dimensions), and the search equals ReferenceSearchN, the single-problem search of test_derivative_free_batch.py generalised to N and D
and evaluated through that oracle.  At N = 10 on 4 dimensions both calls equal the tuned tg_objective_batch / tg_time_alloc_dfo_batch.
On the host emulation a small matrix, on the B200 the full one and one 16 384-problem call per shape (12, 4) and (6, 3).
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
import mrs_uav_trajectory_generation_b200.api as A
from mrs_uav_trajectory_generation_b200 import workloads as W
from mrs_uav_trajectory_generation_b200._capi import _dp, _ip, _p, _u8p
from test_derivative_free_batch import NODE_CONSTRAINTS, TIGHT_CONSTRAINTS, dfo_params, nl_params
from test_free_constraints import FreeOracle, make_problems, pack

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TG_ERR_INVALID = -3
SHAPES_GPU = [(n, d) for n in (6, 8, 10, 12) for d in (1, 2, 3, 4)]
SHAPES_EMU = [(6, 1), (8, 3), (10, 4), (12, 2)]
CONSTRAINT_SETS = [[], TIGHT_CONSTRAINTS, NODE_CONSTRAINTS]  # 0, 6 and 12 constraints


@pytest.fixture(scope="module")
def free_oracle(oracle, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("oracle_set_free_dfo"))
    cache = {}

    def get(n_coef):
        if n_coef not in cache:
            cache[n_coef] = FreeOracle(n_coef, d)
        return cache[n_coef]

    return get


def orc_objective(orc, mask, vals4, r, method, x4, time_penalty, use_soft, soft_weight, con_deriv, con_value):
    """orc_objective of the oracle compiled for orc.N: x4 [K][S or S + 4 n_free] -> total[K], parts[K][3]"""
    mask = np.ascontiguousarray(mask, dtype=np.uint8)
    vals4 = np.ascontiguousarray(vals4, dtype=np.float64)
    x4 = np.ascontiguousarray(x4, dtype=np.float64)
    K, nvar = x4.shape
    cd = np.ascontiguousarray(con_deriv, dtype=np.int32)
    cv = np.ascontiguousarray(con_value, dtype=np.float64)
    total, parts = np.zeros(K), np.zeros((K, 3))
    orc.orc.lib.orc_objective(len(mask), _p(mask, _u8p), _p(vals4), int(r), int(method), int(K), _p(x4), int(nvar), C.c_double(time_penalty),
                              int(bool(use_soft)), C.c_double(soft_weight), len(cd), _p(cd, _ip), _p(cv), _p(total), _p(parts), 0)
    return total, parts


def free_slots(mask, H):
    return [(v, k) for v in range(len(mask)) for k in range(H) if not (mask[v] >> k) & 1]


def pad_x(x, S, nf, dims):
    """[K][S + dims * nf] -> [K][S + 4 * nf], the missing dimensions zero"""
    x = np.atleast_2d(x)
    out = np.zeros((x.shape[0], S + 4 * nf))
    out[:, : S + dims * nf] = x
    return out


def poly_eval(c, t, k, N):
    """Polynomial::evaluate(t, k) with N coefficients (eth/polynomial.h:115-150): Horner over the base coefficients"""
    def b(k, j):
        out = 1.0
        for q in range(j - k + 1, j + 1):
            out *= float(q)
        return out

    acc = b(k, N - 1) * c[N - 1]
    for j in range(N - 2, k - 1, -1):
        acc = acc * t
        acc = acc + b(k, j) * c[j]
    return acc


class ReferenceSearchN:
    """ReferenceSearch (test_derivative_free_batch.py) for N coefficients and D dimensions: the variables are the S times, then for
    methods 3/4 the free derivatives of the D dimensions, dimension-major; every objective value is the oracle's."""

    kTimeLowerBound = 0.01

    def __init__(self, fo, dims, mask, vals4, times, r, parameters, constraints):
        self.fo, self.N, self.H, self.dims = fo, fo.N, fo.N // 2, dims
        self.P, self.r = parameters, r
        self.mask, self.vals4 = mask, vals4
        self.times0 = np.asarray(times, dtype=np.float64)
        self.S = len(self.times0)
        self.constraints = list(constraints)
        self.with_free = parameters.time_alloc_method in (3, 4)
        self.nf = len(free_slots(mask, self.H))

    def objective(self, x):
        x4 = pad_x(x, self.S, self.nf, self.dims) if self.with_free else np.atleast_2d(x)
        return orc_objective(self.fo, self.mask, self.vals4, self.r, self.P.time_alloc_method, x4, self.P.time_penalty, self.P.use_soft_constraints,
                             self.P.soft_constraint_weight, [c[1] for c in self.constraints], [c[2] for c in self.constraints])

    def optimize(self):
        x = self.times0.copy()
        if self.with_free:  # solveLinear + getFreeConstraints at the initial times, read off the segments (nl_impl.h:436-462)
            coef, _ = self.fo.orc.solve_linear(self.mask, self.vals4, self.times0, self.r)
            dp = np.zeros((self.dims, self.nf))
            for j, (v, k) in enumerate(free_slots(self.mask, self.H)):
                seg, t = (v, 0.0) if v < self.S else (self.S - 1, self.times0[-1])
                for d in range(self.dims):
                    dp[d, j] = poly_eval(coef[seg, d], t, k, self.N)
            x = np.concatenate([x, dp.reshape(-1)])
        n = len(x)
        lo, hi = np.full(n, -np.finfo(np.float64).max), np.full(n, np.finfo(np.float64).max)
        lo[: self.S] = self.kTimeLowerBound
        if self.with_free:  # setFreeEndpointDerivativeHardConstraints with its counter quirk (nl_impl.h:764-805)
            for dim, deriv, value in self.constraints:
                counter = 0
                for v in range(len(self.mask)):
                    for k in range(self.r + 1):
                        if not (self.mask[v] >> k) & 1:
                            if k == deriv:
                                at = self.S + dim * self.nf + counter
                                if at < n:
                                    lo[at], hi[at] = -abs(value), abs(value)
                            counter += 1
        lo, hi = np.minimum(lo, x), np.maximum(hi, x)
        step = np.where(np.abs(x) <= np.finfo(np.float64).eps, 1e-13, self.P.initial_stepsize_rel * np.abs(x))
        f = float(self.objective(x)[0][0])
        self.n_iterations, code = 0, 5
        while self.n_iterations < self.P.max_iterations:
            self.n_iterations += 1
            cand = np.repeat(x[None, :], 2 * n, axis=0)
            idx = np.arange(n)
            cand[idx, idx] = np.minimum(x + step, hi)
            cand[n + idx, idx] = np.maximum(x - step, lo)
            tot, _ = self.objective(cand)
            k = int(np.argmin(tot))
            if tot[k] < f:
                f_old, f = f, float(tot[k])
                x = cand[k].copy()
                if abs(f_old - f) <= self.P.f_rel * abs(f):
                    code = 3
                    break
            else:
                step *= 0.5
                if np.all(step <= self.P.x_rel * np.abs(x)):
                    code = 4
                    break
        self.x, self.cost, self.times = x, f, x[: self.S].copy()
        self.parts = self.objective(x)[1][0]
        if self.with_free:  # updateSegmentTimes + setFreeConstraints
            coef, _ = self.fo.set(self.mask, self.vals4, self.times, self.r, pad_x(x, self.S, self.nf, self.dims)[0, self.S:].reshape(4, self.nf))
        else:  # updateSegmentTimes + solveLinear
            coef, _ = self.fo.orc.solve_linear(self.mask, self.vals4, self.times, self.r)
        self.coef = coef[:, : self.dims]
        return code


def problem_out(out, probs, p, n_coef, dims):
    vtx_off = np.cumsum([0] + [len(m) for m, _, _ in probs])
    v0, v1 = vtx_off[p], vtx_off[p + 1]
    s0, s1 = v0 - p, v1 - p - 1
    o = {"code": int(out["code"][p]), "n_iterations": int(out["n_iterations"][p]), "times": out["times"][s0:s1], "coef": out["coef"][s0:s1],
         "total": out["total"][p], "parts": out["parts"][p]}
    o["x"] = o["times"]
    if out["vval"] is not None:
        vv = out["vval"][v0:v1]
        free = [vv[v, k] for v, k in free_slots(probs[p][0], n_coef // 2)]
        o["x"] = np.concatenate([o["times"], np.array(free).reshape(-1, dims).T.reshape(-1)])
    return o


def same(a, b):
    return (a["code"] == b["code"] and a["n_iterations"] == b["n_iterations"] and np.array_equal(a["times"], b["times"])
            and np.array_equal(a["coef"], b["coef"]) and np.array_equal(a["x"], b["x"]) and a["total"] == b["total"]
            and np.array_equal(a["parts"], b["parts"]))


def reference_out(ref):
    code = ref.optimize()
    return {"code": code, "n_iterations": ref.n_iterations, "times": ref.times, "coef": ref.coef, "total": ref.cost, "parts": ref.parts, "x": ref.x}


# ---- 1. the objective ---------------------------------------------------------------------------------------------------------
def objective_candidates(rng, times, free, dims, method, K=9):
    """K candidate vectors around the problem's times (and free derivatives), the first with a time below 0.01"""
    S = len(times)
    T = times[None, :] * rng.uniform(0.5, 1.5, (K, S))
    T[0, 0] = 0.004
    if method < 3:
        return T
    F = free[None, :] * (1.0 + 0.2 * rng.standard_normal((K, free.size))) + 0.05 * rng.standard_normal((K, free.size))
    return np.concatenate([T, F], axis=1)


def check_objective(ctx, fo, n_coef, dims, seed=0):
    orc = fo(n_coef)
    rng = np.random.default_rng(seed)
    case = 0
    for r in range(n_coef // 2):
        probs = make_problems(n_coef, dims, r, 3000 + 100 * n_coef + 10 * dims + r, B=6, S_max=6)
        for method in (0, 1, 3, 4):
            for mask, vals4, times in probs[case % 3::3]:
                cons = CONSTRAINT_SETS[case % 3]
                soft = case % 2 == 0
                case += 1
                nf = len(free_slots(mask, n_coef // 2))
                _, _, dp, _ = orc.solve(mask, vals4, times, r)
                x = objective_candidates(rng, times, dp[:dims].reshape(-1), dims, method)
                cd, cv = [c[1] for c in cons], [c[2] for c in cons]
                tot, parts, coef = ctx.objective_nd(n_coef, dims, mask, vals4[:, :, :dims], r, method, x, 500.0, soft, 100.0, cd, cv, want_coef=True)
                x4 = pad_x(x, len(times), nf, dims) if method >= 3 else x
                rt, rp = orc_objective(orc, mask, vals4, r, method, x4, 500.0, soft, 100.0, cd, cv)
                assert np.array_equal(tot, rt) and np.array_equal(parts, rp), (n_coef, dims, r, method, len(cons), soft)
                # the coefficients are the oracle's segments at each candidate
                for k in (0, len(x) - 1):
                    if method >= 3:
                        want, _ = orc.set(mask, vals4, x[k, : len(times)], r, x4[k, len(times):].reshape(4, nf))
                    else:
                        want, _ = orc.orc.solve_linear(mask, vals4, x[k], r)
                    assert np.array_equal(coef[k], want[:, :dims]), (n_coef, dims, r, method, k)
                if (n_coef, dims) == (10, 4) and r >= 2:  # the tuned call
                    t2, p2, c2 = ctx.objective(mask, vals4, r, method, x, 500.0, soft, 100.0, cd, cv, want_coef=True)
                    assert np.array_equal(tot, t2) and np.array_equal(parts, p2) and np.array_equal(coef, c2), (r, method)


@pytest.mark.parametrize("n_coef,dims", SHAPES_EMU)
def test_objective_equals_oracle_emulator(emu_ctx, free_oracle, n_coef, dims):
    check_objective(emu_ctx, free_oracle, n_coef, dims)


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", SHAPES_GPU)
def test_objective_equals_oracle_gpu(gpu_ctx, free_oracle, n_coef, dims):
    check_objective(gpu_ctx, free_oracle, n_coef, dims, seed=1)


# ---- 2. the search against ReferenceSearchN -----------------------------------------------------------------------------------
def check_search(ctx, fo, n_coef, dims, method, r, iters, soft, cons, seed, B=12, S_max=12):
    orc = fo(n_coef)
    probs = make_problems(n_coef, dims, r, seed, B=B, S_max=S_max)
    P = nl_params(method, iters, soft)
    out = ctx.time_alloc_dfo_batch_nd(n_coef, dims, *pack(probs, dims), dfo_params(ctx, P, r), cons)
    for p, (mask, vals4, times) in enumerate(probs):
        want = reference_out(ReferenceSearchN(orc, dims, mask, vals4, times, r, P, cons))
        got = problem_out(out, probs, p, n_coef, dims)
        assert same(got, want), (n_coef, dims, method, r, iters, soft, len(cons), p, got["code"], want["code"], got["n_iterations"],
                                 want["n_iterations"])
    return out, probs


def emu_search_cases(n_coef, dims):
    """per shape: every method, r spread over 0 .. N/2-1, iteration limits 0, 1, 10, 25, constraint sets and soft on / off"""
    H = n_coef // 2
    iters = (0, 1, 10, 25)
    return [(m, (3 * i + n_coef) % H, iters[i % 4], i % 3 != 1, CONSTRAINT_SETS[(i + dims) % 3]) for i, m in enumerate((0, 1, 3, 4))]


@pytest.mark.parametrize("n_coef,dims", SHAPES_EMU)
def test_search_equals_reference_emulator(emu_ctx, free_oracle, n_coef, dims):
    for i, (method, r, iters, soft, cons) in enumerate(emu_search_cases(n_coef, dims)):
        check_search(emu_ctx, free_oracle, n_coef, dims, method, r, iters, soft, cons, seed=7000 + 100 * n_coef + 10 * dims + i, B=8, S_max=5)


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", SHAPES_GPU)
@pytest.mark.parametrize("method", [0, 1, 3, 4])
def test_search_equals_reference_gpu(gpu_ctx, free_oracle, n_coef, dims, method):
    """every r, each with one of the four (iterations, soft, constraints) cases in turn (the reference search runs on the host)"""
    cases = ((0, True, NODE_CONSTRAINTS), (1, False, TIGHT_CONSTRAINTS), (10, True, TIGHT_CONSTRAINTS), (25, True, []))
    for r in range(n_coef // 2):
        i = (r + method + dims) % 4
        iters, soft, cons = cases[i]
        check_search(gpu_ctx, free_oracle, n_coef, dims, method, r, iters, soft, cons, seed=9000 + 1000 * method + 100 * n_coef + 10 * r + dims,
                     B=12, S_max=12 if method < 3 else 6)


# ---- 3. the tuned path ----------------------------------------------------------------------------------------------------------
def check_tuned(ctx, methods, rs):
    for method in methods:
        for r in rs:
            probs = make_problems(10, 4, r, 500 + 10 * method + r, B=10, S_max=8)
            P = nl_params(method, 10, True)
            args = pack(probs, 4)
            a = ctx.time_alloc_dfo_batch_nd(10, 4, *args, dfo_params(ctx, P, r), TIGHT_CONSTRAINTS)
            b = ctx.time_alloc_dfo_batch(*args, dfo_params(ctx, P, r), TIGHT_CONSTRAINTS)
            for k in ("times", "coef", "code", "n_iterations", "total", "parts"):
                assert np.array_equal(a[k], b[k]), (method, r, k)
            assert (a["vval"] is None) == (b["vval"] is None) and (a["vval"] is None or np.array_equal(a["vval"], b["vval"]))


def test_tuned_path_emulator(emu_ctx):
    check_tuned(emu_ctx, (0, 3), (2, 4))


@pytest.mark.gpu
def test_tuned_path_gpu(gpu_ctx):
    check_tuned(gpu_ctx, (0, 1, 3, 4), (2, 3, 4))


# ---- 4. independence ----------------------------------------------------------------------------------------------------------
def check_independence(ctx, lib, n_coef, dims, method):
    from mrs_uav_trajectory_generation_b200 import Context

    r = 1
    probs = make_problems(n_coef, dims, r, 40 + method, B=9, S_max=5)
    P = nl_params(method, 10, True)
    out = ctx.time_alloc_dfo_batch_nd(n_coef, dims, *pack(probs, dims), dfo_params(ctx, P, r), TIGHT_CONSTRAINTS)
    for p in range(len(probs)):
        one = ctx.time_alloc_dfo_batch_nd(n_coef, dims, *pack(probs[p:p + 1], dims), dfo_params(ctx, P, r), TIGHT_CONSTRAINTS)
        assert same(problem_out(out, probs, p, n_coef, dims), problem_out(one, probs[p:p + 1], 0, n_coef, dims)), (method, p)
    old = os.environ.get("TG_SEG_BUDGET")
    os.environ["TG_SEG_BUDGET"] = "100"
    try:
        small = Context(lib, 0)
    finally:
        if old is None:
            os.environ.pop("TG_SEG_BUDGET")
        else:
            os.environ["TG_SEG_BUDGET"] = old
    out2 = small.time_alloc_dfo_batch_nd(n_coef, dims, *pack(probs, dims), dfo_params(small, P, r), TIGHT_CONSTRAINTS)
    for p in range(len(probs)):
        assert same(problem_out(out, probs, p, n_coef, dims), problem_out(out2, probs, p, n_coef, dims)), (method, p)


@pytest.mark.parametrize("n_coef,dims,method", [(8, 3, 0), (12, 2, 4)])
def test_independence_emulator(emu_ctx, emu_lib, n_coef, dims, method):
    check_independence(emu_ctx, emu_lib, n_coef, dims, method)


@pytest.mark.gpu
@pytest.mark.parametrize("method", [0, 1, 3, 4])
def test_independence_gpu(gpu_ctx, method):
    from mrs_uav_trajectory_generation_b200 import Library

    check_independence(gpu_ctx, Library(), 6 + 2 * method % 8, 1 + method % 4, method)


# ---- 5. refusals --------------------------------------------------------------------------------------------------------------
def check_refusals(ctx):
    n_coef, dims = 8, 3
    H = n_coef // 2
    probs = make_problems(n_coef, dims, 1, 3, B=3, S_max=4)
    vtx_off, masks, vals, times = pack(probs, dims)
    B, totS, totV = 3, len(times), len(masks)
    lib = ctx.L.lib

    def dfo(N=n_coef, D=dims, B=B, vtx_off=vtx_off, params=None, cons=((0, 1, 2.0),)):
        prm = params or ctx.L.default_dfo_params(time_alloc_method=3, derivative_to_optimize=1)
        cd = np.array([c[0] for c in cons], np.int32)
        ck = np.array([c[1] for c in cons], np.int32)
        cv = np.array([c[2] for c in cons], np.float64)
        outs = [times.copy(), np.full((totS, 4, 12), 7.0), np.full((totV, 6, 4), 7.0), np.full(B + 1, 7, np.int32), np.full(B + 1, 7, np.int32),
                np.full(B + 1, 7.0), np.full((B + 1, 3), 7.0)]
        rc = lib.tg_time_alloc_dfo_batch_nd(ctx.h, N, D, B, _p(vtx_off, _ip), _p(masks, _u8p), _p(vals), _p(outs[0]), C.byref(prm), len(cons),
                                            _p(cd, _ip), _p(ck, _ip), _p(cv), _p(outs[1]), _p(outs[2]), _p(outs[3], _ip), _p(outs[4], _ip),
                                            _p(outs[5]), _p(outs[6]))
        untouched = np.array_equal(outs[0], times) and all(np.all(o == 7) for o in outs[1:])
        return rc, untouched

    assert dfo()[0] == 0
    bad = [dict(N=7), dict(N=14), dict(D=0), dict(D=5), dict(B=0), dict(vtx_off=np.array([0, 1, vtx_off[2], vtx_off[3]], np.int32))]
    bad += [dict(params=ctx.L.default_dfo_params(time_alloc_method=m)) for m in (2, 5, -1)]
    bad += [dict(params=ctx.L.default_dfo_params(derivative_to_optimize=k)) for k in (-1, H)]
    bad += [dict(cons=[(0, 1, 1.0)] * 17), dict(cons=[(0, 0, 1.0)]), dict(cons=[(0, 5, 1.0)]), dict(cons=[(4, 1, 1.0)]), dict(cons=[(-1, 1, 1.0)]),
            dict(cons=[(0, 1, 1.0), (1, 2, 0.0)])]
    for kw in bad:
        rc, untouched = dfo(**kw)
        assert rc == TG_ERR_INVALID and untouched, kw

    mask, vals4, t0 = probs[1]
    V, S = len(mask), len(t0)
    nf = len(free_slots(mask, H))
    v3 = np.ascontiguousarray(vals4[:, :, :dims])

    def obj(N=n_coef, D=dims, V=V, r=1, method=3, K=2, nvar=S + dims * nf, cons=((1, 2.0),)):
        x = np.tile(np.concatenate([t0, np.zeros(max(nvar - S, 0))])[:max(nvar, 1)], (max(K, 1), 1))
        cd = np.array([c[0] for c in cons], np.int32)
        cv = np.array([c[1] for c in cons], np.float64)
        outs = [np.full(max(K, 1), 7.0), np.full((max(K, 1), 3), 7.0), np.full((max(K, 1), S, 4, 12), 7.0)]
        rc = lib.tg_objective_batch_nd(ctx.h, N, D, V, _p(mask, _u8p), _p(v3), r, method, K, _p(x), nvar, 500.0, 1, 100.0, len(cons), _p(cd, _ip),
                                       _p(cv), _p(outs[0]), _p(outs[1]), _p(outs[2]))
        return rc, all(np.all(o == 7.0) for o in outs)

    assert obj()[0] == 0
    bad = [dict(N=9), dict(D=0), dict(D=5), dict(V=1), dict(r=-1), dict(r=H), dict(method=2), dict(method=5), dict(K=0), dict(nvar=S + dims * nf + 1),
           dict(nvar=S + 4 * nf), dict(method=0, nvar=S + dims * nf), dict(cons=[(1, 1.0)] * 17), dict(cons=[(0, 1.0)]), dict(cons=[(5, 1.0)]),
           dict(cons=[(1, 0.0)])]
    for kw in bad:
        rc, untouched = obj(**kw)
        assert rc == TG_ERR_INVALID and untouched, kw

    # NaN inputs are not refused and propagate
    P = nl_params(0, 3, True)
    tn = times.copy()
    tn[0] = np.nan
    out = ctx.time_alloc_dfo_batch_nd(n_coef, dims, vtx_off, masks, vals, tn, dfo_params(ctx, P, 1), TIGHT_CONSTRAINTS)
    assert np.isnan(out["total"][0])
    x = np.tile(t0, (2, 1))
    x[1, 0] = np.nan
    tot, _ = ctx.objective_nd(n_coef, dims, mask, v3, 1, 0, x)
    assert np.isfinite(tot[0]) and np.isnan(tot[1])


def test_refusals_emulator(emu_ctx):
    check_refusals(emu_ctx)


@pytest.mark.gpu
def test_refusals_gpu(gpu_ctx):
    check_refusals(gpu_ctx)


# ---- 6. the Python classes and the C++ batch function ---------------------------------------------------------------------------
def vertices_of(mask, vals4, H, dims):
    verts = []
    for v in range(len(mask)):
        vx = A.Vertex(dims)
        for k in range(H):
            if (mask[v] >> k) & 1:
                vx.addConstraint(k, vals4[v, k, :dims])
        verts.append(vx)
    return verts


def check_classes(ctx, n_coef, dims):
    H, r = n_coef // 2, 1
    probs = make_problems(n_coef, dims, r, 77, B=4, S_max=4)
    for method in (1, 3):
        P = nl_params(method, 10, True, f_rel=0.05)
        verts = [vertices_of(m, v, H, dims) for m, v, _ in probs]
        trajs, codes = A.TrajectoryGenerator(ctx=ctx).time_alloc_derivative_free(verts, [t for _, _, t in probs], P, NODE_CONSTRAINTS, r,
                                                                                 n_coefficients=n_coef, dimension=dims)
        out = ctx.time_alloc_dfo_batch_nd(n_coef, dims, *pack(probs, dims), dfo_params(ctx, P, r), NODE_CONSTRAINTS)
        assert np.array_equal(codes, out["code"])
        for p, (mask, vals4, times) in enumerate(probs):
            got = problem_out(out, probs, p, n_coef, dims)
            assert np.array_equal(trajs[p].times, got["times"]) and np.array_equal(trajs[p].coef, got["coef"])
            dfo = A.DerivativeFreeTimeAllocation(verts[p], times, r, P, NODE_CONSTRAINTS, ctx=ctx, n_coefficients=n_coef, dimension=dims)
            assert dfo.optimize() == got["code"]
            assert np.array_equal(dfo.x, got["x"]) and dfo.cost == got["total"] and np.array_equal(dfo.coef, got["coef"])


def check_class_defaults(ctx):
    """the defaults give the N = 10, D = 4 call"""
    probs = make_problems(10, 4, 2, 78, B=3, S_max=4)
    P = nl_params(3, 10, True, f_rel=0.05)
    verts = [vertices_of(m, v, 5, 4) for m, v, _ in probs]
    trajs, codes = A.TrajectoryGenerator(ctx=ctx).time_alloc_derivative_free(verts, [t for _, _, t in probs], P, NODE_CONSTRAINTS)
    out = ctx.time_alloc_dfo_batch(*pack(probs, 4), dfo_params(ctx, P, 2), NODE_CONSTRAINTS)
    assert np.array_equal(codes, out["code"]) and np.array_equal(np.concatenate([t.coef for t in trajs]), out["coef"])
    dfo = A.DerivativeFreeTimeAllocation(verts[0], probs[0][2], 2, P, NODE_CONSTRAINTS, ctx=ctx)
    assert dfo.optimize() == out["code"][0] and dfo.cost == out["total"][0]


@pytest.mark.parametrize("n_coef,dims", [(6, 3), (12, 4)])
def test_classes_emulator(emu_ctx, n_coef, dims):
    check_classes(emu_ctx, n_coef, dims)


def test_class_defaults_emulator(emu_ctx):
    check_class_defaults(emu_ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", [(6, 3), (8, 1), (12, 4)])
def test_classes_gpu(gpu_ctx, n_coef, dims):
    check_classes(gpu_ctx, n_coef, dims)


@pytest.mark.gpu
def test_class_defaults_gpu(gpu_ctx):
    check_class_defaults(gpu_ctx)


# ---- 7. one call at scale -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", [(12, 4), (6, 3)])
@pytest.mark.parametrize("method", [0, 3])
def test_gpu_at_scale(gpu_ctx, free_oracle, n_coef, dims, method):
    """one call with 16 384 random-flier problems of 11 vertices (ends fixed up to acceleration) and the node's 12 constraints: every
    output finite, and 16 sampled problems equal ReferenceSearchN"""
    B, r, H = 16384, 2, n_coef // 2
    probs = []
    for p in range(B):
        wp = W.random_flier_path(p, 11)
        mask = np.ones(11, np.uint8)
        mask[0] = mask[-1] = 0b111
        vals = np.zeros((11, H, 4))
        vals[:, 0] = wp
        vals[:, :, dims:] = 0.0
        probs.append((mask, vals, O.estimate_times(wp)[0].copy()))
    P = nl_params(method, 10, True, f_rel=0.05)
    out = gpu_ctx.time_alloc_dfo_batch_nd(n_coef, dims, *pack(probs, dims), dfo_params(gpu_ctx, P, r), NODE_CONSTRAINTS)
    for k in ("times", "coef", "total", "parts"):
        assert np.all(np.isfinite(out[k])), k
    orc = free_oracle(n_coef)
    for p in np.random.default_rng(5).choice(B, 16, replace=False):
        mask, vals4, times = probs[p]
        want = reference_out(ReferenceSearchN(orc, dims, mask, vals4, times, r, P, NODE_CONSTRAINTS))
        assert same(problem_out(out, probs, p, n_coef, dims), want), p


# ---- the C++ functions (built as they are and against an Eigen) -------------------------------------------------------------
def run_cpp(libdir, libname, tmp_path):
    from test_cpp_shim import _eigen_flags, _run_shim

    for extra, tag in (((), "plain"), (_eigen_flags(), "eigen")):
        d = tmp_path / tag
        d.mkdir()
        res = _run_shim(libdir, libname, d, "test_shim_dfo_general.cpp", extra)
        keys = [f"N{n}_D{dd}_m{m}" for n, dd in ((6, 3), (8, 1), (10, 4), (12, 2)) for m in (0, 1, 3, 4)]
        keys += [f"N{n}_D{dd}_refused" for n, dd in ((6, 3), (8, 1), (10, 4), (12, 2))]
        for k in keys:
            assert res[k][0][0] == 1.0, (tag, k)


def test_cpp_batch_emulator(emu_lib, tmp_path):
    run_cpp(os.path.join(ROOT, "tests", "host_emu"), "tg_emu", tmp_path)


@pytest.mark.gpu
def test_cpp_batch_gpu(gpu_ctx, tmp_path):
    run_cpp(os.path.join(ROOT, "mrs_uav_trajectory_generation_b200"), "tg_b200", tmp_path)
