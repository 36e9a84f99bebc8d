"""Free and fixed constraints of PolynomialOptimization<N> (lin_impl.h:183-257, 513-522): tg_solve_linear_free_batch_nd (solveLinear +
getFreeConstraints + getSegments + computeCost) and tg_set_free_constraints_batch_nd (setFreeConstraints + getSegments + computeCost) for
N in {6, 8, 10, 12}, D in 1..4 and every derivative_to_optimize, and the classes above them.

Checked bit for bit against the oracle compiled for that N: its solve returns d_p (orc_solve_linear), and tests/cpp/oracle_set_free.cpp
runs its setFreeConstraints path (d_p assigned, segments_from_compact, cost).  On the host emulation of the device code a small matrix,
on the B200 the full one and one call with 65 536 problems.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import mrs_uav_trajectory_generation_b200.api as A
from mrs_uav_trajectory_generation_b200 import workloads as W
from mrs_uav_trajectory_generation_b200._capi import _dp, _ip, _p, _u8p

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TG_ERR_INVALID = -3
SHAPES_GPU = [(n, d) for n in (6, 8, 10, 12) for d in (1, 2, 3, 4)]
SHAPES_EMU = [(6, 1), (8, 3), (10, 4), (12, 2)]


class FreeOracle:
    """The oracle for one N: the solve with its free derivatives, and setFreeConstraints."""

    def __init__(self, n_coef, build_dir):
        self.N, self.H = n_coef, n_coef // 2
        self.orc = O.OracleN(n_coef)  # builds and loads the library the helper links, and sets its math mode
        so = os.path.join(build_dir, f"liboracle_set_free_n{n_coef}.so")
        lib = "oracle" if n_coef == 10 else f"oracle_n{n_coef}"
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", f"-DORC_N={n_coef}", "-o", so,
                               os.path.join(ROOT, "tests", "cpp", "oracle_set_free.cpp"), "-L" + O.ORACLE_DIR, "-l" + lib, "-Wl,-rpath," + O.ORACLE_DIR])
        self.lib = C.CDLL(so)

    def solve(self, mask, vals, times, r):
        """-> coef [S][4][N], cost, d_p [4][n_free], (n_fixed, n_free)"""
        V = len(mask)
        coef = np.zeros((V - 1, 4, self.N))
        cost = C.c_double()
        dims = (C.c_int * 2)()
        dp = np.zeros(4 * self.H * V)
        assert self.orc.lib.orc_solve_linear(V, _p(np.ascontiguousarray(mask), _u8p), _p(np.ascontiguousarray(vals)), _p(np.ascontiguousarray(times)),
                                             int(r), _p(coef), C.byref(cost), _p(dp), dims) == 0
        return coef, cost.value, dp[: 4 * dims[1]].reshape(4, dims[1]), (dims[0], dims[1])

    def set(self, mask, vals, times, r, dp4):
        V = len(mask)
        coef = np.zeros((V - 1, 4, self.N))
        cost = C.c_double()
        dp4 = np.ascontiguousarray(dp4, dtype=np.float64)
        assert self.lib.orc_set_free_constraints(V, _p(np.ascontiguousarray(mask), _u8p), _p(np.ascontiguousarray(vals)),
                                                 _p(np.ascontiguousarray(times)), int(r), _p(dp4), _p(coef), C.byref(cost)) == dp4.shape[1]
        return coef, cost.value


@pytest.fixture(scope="module")
def free_oracle(oracle, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("oracle_set_free"))
    cache = {}

    def get(n_coef):
        if n_coef not in cache:
            cache[n_coef] = FreeOracle(n_coef, d)
        return cache[n_coef]

    return get


def make_problems(n_coef, dims, r, seed, B=24, S_max=12):
    """Ragged random-flier problems: S = 1 .. S_max, ends fixed up to r, interior positions; some with a stop vertex (v, a, j fixed at
    zero), random interior masks and values, every vertex fully fixed (n_free = 0), or an initial time below 0.01.  vals [V][N/2][4],
    dimensions from `dims` on zero."""
    H = n_coef // 2
    full = (1 << H) - 1
    rng = np.random.default_rng(seed)
    probs = []
    for p in range(B):
        S = 1 + p % S_max
        V = S + 1
        wp = W.random_flier_path(700 + seed * 1000 + p, V)
        mask = np.ones(V, np.uint8)
        vals = np.zeros((V, H, 4))
        vals[:, 0] = wp
        mask[0] = mask[-1] = (1 << (r + 1)) - 1
        kind = p % 6
        if kind == 1 and V > 2:
            mask[V // 2] = 0b1111 & full
        if kind == 2:
            for v in range(1, V - 1):
                mask[v] = 1 | int(rng.integers(0, 1 << (H - 1))) << 1
                vals[v, 1:] = rng.uniform(-0.5, 0.5, (H - 1, 4))
        if kind == 3:
            mask[:] = full
            vals[:, 1:] = rng.uniform(-0.2, 0.2, (V, H - 1, 4))
        if kind == 4:
            mask[0] = 0b1111 & full
            vals[0, 1:4] = rng.uniform(-1.0, 1.0, (min(3, H - 1), 4))
        for v in range(V):  # values of free slots are not read; keep them zero so that the layouts compare plainly
            for k in range(H):
                if not (mask[v] >> k) & 1:
                    vals[v, k] = 0.0
        vals[:, :, dims:] = 0.0
        times = O.estimate_times(wp)[0].copy()
        if kind == 5:
            times[0] = 0.004
        probs.append((mask, vals, times))
    return probs


def pack(probs, dims):
    vtx_off = np.cumsum([0] + [len(m) for m, _, _ in probs]).astype(np.int32)
    vals = np.concatenate([v for _, v, _ in probs])
    return vtx_off, np.concatenate([m for m, _, _ in probs]), np.ascontiguousarray(vals[:, :, :dims]), np.concatenate([t for _, _, t in probs])


def seg_offsets(probs):
    return np.cumsum([0] + [len(t) for _, _, t in probs])


def perturbed(rng, free):
    """free vectors near the solution, scaled to the problem's values"""
    out = []
    for f in free:
        scale = np.abs(f).mean() if f.size else 0.0
        out.append(f * (1.0 + 0.25 * rng.standard_normal(f.shape)) + 0.1 * (scale + 1.0) * rng.standard_normal(f.shape))
    return out


def check_get_set(ctx, fo, n_coef, dims, seed=0):
    orc = fo(n_coef)
    for r in range(n_coef // 2):
        probs = make_problems(n_coef, dims, r, 1000 * n_coef + 10 * dims + r + seed)
        args = pack(probs, dims)
        so = seg_offsets(probs)
        coef, cost, free = ctx.solve_linear_free_batch_nd(n_coef, dims, *args, r)
        # 1. get: the solve's bits, the oracle's d_p
        c_nd, k_nd = ctx.solve_linear_batch_nd(n_coef, dims, *args, r)
        assert np.array_equal(coef, c_nd) and np.array_equal(cost, k_nd), (n_coef, dims, r)
        if (n_coef, dims) == (10, 4) and r >= 2:
            c_t, k_t = ctx.solve_linear_batch(*args, r)
            assert np.array_equal(coef, c_t) and np.array_equal(cost, k_t), r
        for p, (mask, vals, times) in enumerate(probs):
            c_o, cost_o, dp_o, (n_fixed, n_free) = orc.solve(mask, vals, times, r)
            assert free[p].shape == (dims, n_free) and n_fixed + n_free == len(mask) * (n_coef // 2)
            assert np.array_equal(free[p], dp_o[:dims]), (n_coef, dims, r, p)
            assert np.array_equal(coef[so[p]:so[p + 1]], c_o[:, :dims]) and cost[p] == cost_o, (n_coef, dims, r, p)
        # 3. round trip: set(get) gives solveLinear's coefficients and cost
        c_rt, k_rt = ctx.set_free_constraints_batch_nd(n_coef, dims, *args, free, r)
        assert np.array_equal(c_rt, coef) and np.array_equal(k_rt, cost), (n_coef, dims, r)
        # 2. set: random free vectors against the oracle's setFreeConstraints
        x = perturbed(np.random.default_rng(seed + r), free)
        c_s, k_s = ctx.set_free_constraints_batch_nd(n_coef, dims, *args, x, r)
        for p, (mask, vals, times) in enumerate(probs):
            dp4 = np.zeros((4, x[p].shape[1]))
            dp4[:dims] = x[p]
            c_o, cost_o = orc.set(mask, vals, times, r, dp4)
            assert np.array_equal(c_s[so[p]:so[p + 1]], c_o[:, :dims]) and k_s[p] == cost_o, (n_coef, dims, r, p)
            if (n_coef, dims) == (10, 4) and r >= 2:  # objectiveFunctionTimeAndConstraints' trajectory term at x = [times ; free]
                _, parts, c_obj = ctx.objective(mask, vals, r, 3, np.concatenate([times, x[p].ravel()])[None], 0.0, False, want_coef=True)
                assert np.array_equal(c_obj[0], c_s[so[p]:so[p + 1]]) and parts[0, 0] == k_s[p], (r, p)


def check_independence(ctx, n_coef, dims):
    r = min(2, n_coef // 2 - 1)
    probs = make_problems(n_coef, dims, r, 55)
    args = pack(probs, dims)
    so = seg_offsets(probs)
    coef, cost, free = ctx.solve_linear_free_batch_nd(n_coef, dims, *args, r)
    x = perturbed(np.random.default_rng(1), free)
    c_s, k_s = ctx.set_free_constraints_batch_nd(n_coef, dims, *args, x, r)
    for p in (0, 5, 11, 23):
        one = pack([probs[p]], dims)
        c1, k1, f1 = ctx.solve_linear_free_batch_nd(n_coef, dims, *one, r)
        assert np.array_equal(c1, coef[so[p]:so[p + 1]]) and k1[0] == cost[p] and np.array_equal(f1[0], free[p]), p
        c2, k2 = ctx.set_free_constraints_batch_nd(n_coef, dims, *one, [x[p]], r)
        assert np.array_equal(c2, c_s[so[p]:so[p + 1]]) and k2[0] == k_s[p], p


def check_refusals(ctx):
    """TG_ERR_INVALID with every output untouched"""
    lib = ctx.L.lib
    probs = make_problems(8, 3, 2, 9, B=3)
    vtx_off, mask, vals, times = pack(probs, 3)
    nv = int(vtx_off[-1])
    big = np.zeros(nv * 6 * 4)
    big[: vals.size] = vals.ravel()
    bad_off = vtx_off.copy()
    bad_off[1] = 1  # problem 0 with one vertex
    cases = [dict(N=7), dict(N=14), dict(N=4), dict(D=0), dict(D=5), dict(r=-1), dict(r=4), dict(B=0), dict(off=bad_off)]
    for case in cases:
        N, D, r, B, off = case.get("N", 8), case.get("D", 3), case.get("r", 2), case.get("B", 3), case.get("off", vtx_off)
        coef = np.full(int(times.size) * 4 * 12, 7.25)
        cost = np.full(3, 7.25)
        free = np.full(nv * 6 * 4, 7.25)
        rc = lib.tg_solve_linear_free_batch_nd(ctx.h, N, D, B, _p(off, _ip), _p(mask, _u8p), _p(big), _p(times), r, _p(coef), _p(cost), _p(free))
        assert rc == TG_ERR_INVALID, case
        assert (coef == 7.25).all() and (cost == 7.25).all() and (free == 7.25).all(), case
        inp = np.zeros(nv * 6 * 4)
        rc = lib.tg_set_free_constraints_batch_nd(ctx.h, N, D, B, _p(off, _ip), _p(mask, _u8p), _p(big), _p(times), r, _p(inp), _p(coef), _p(cost))
        assert rc == TG_ERR_INVALID, case
        assert (coef == 7.25).all() and (cost == 7.25).all(), case
    # NULL outputs are allowed; non-finite free values propagate
    assert lib.tg_solve_linear_free_batch_nd(ctx.h, 8, 3, 3, _p(vtx_off, _ip), _p(mask, _u8p), _p(vals), _p(times), 2, None, None, None) == 0
    _, _, free = ctx.solve_linear_free_batch_nd(8, 3, vtx_off, mask, vals, times, 2)
    free[0][1, 0] = np.nan
    c, k = ctx.set_free_constraints_batch_nd(8, 3, vtx_off, mask, vals, times, free, 2)
    assert np.isnan(k[0]) and np.isfinite(k[1:]).all()


def _vertices(n_coef, dims, seed):
    """A vertex list for the classes (A.Vertex), the matching masks / values and times."""
    H, r = n_coef // 2, min(2, n_coef // 2 - 1)
    probs = make_problems(n_coef, dims, r, seed, B=6)
    lists, times = [], []
    for mask, vals, t in probs[1:4]:
        vl = []
        for v in range(len(mask)):
            x = A.Vertex(dims)
            for k in range(H):
                if (mask[v] >> k) & 1:
                    x.addConstraint(k, vals[v, k, :dims])
            vl.append(x)
        lists.append(vl)
        times.append(t)
    return lists, times, probs[1:4], r


def check_python_class(ctx, fo):
    for n_coef in (6, 8, 10, 12):
        for dims in (3, 4):
            lists, times, probs, r = _vertices(n_coef, dims, 3 * n_coef + dims)
            orc = fo(n_coef)
            # one problem
            opt = A.PolynomialOptimization(dims, ctx=ctx, n_coefficients=n_coef)
            assert opt.setupFromVertices(lists[0], times[0], r)
            mask, vals, t = probs[0]
            _, _, dp_o, (n_fixed, n_free) = orc.solve(mask, vals, t, r)
            assert (opt.getNumberFreeConstraints(), opt.getNumberFixedConstraints(), opt.getNumberAllConstraints()) == (n_free, n_fixed, len(t) * n_coef)
            before = opt.getFreeConstraints()
            assert len(before) == dims and all(np.array_equal(v, np.zeros(n_free)) for v in before)
            fixed = opt.getFixedConstraints()
            want_fixed = [vals[:, :, d][((mask[:, None] >> np.arange(n_coef // 2)) & 1).astype(bool)] for d in range(dims)]
            assert all(np.array_equal(a, b) for a, b in zip(fixed, want_fixed)) and len(fixed) == dims
            assert opt.solveLinear()
            free = opt.getFreeConstraints()
            assert len(free) == dims and np.array_equal(np.array(free).reshape(dims, n_free), dp_o[:dims])
            assert not opt.setFreeConstraints(free[:-1]) and np.array_equal(np.array(opt.getFreeConstraints()).reshape(dims, n_free), dp_o[:dims])
            if n_free:
                free[-1][0] += 0.75
            assert opt.setFreeConstraints(free)
            dp4 = np.zeros((4, n_free))
            dp4[:dims] = np.array(free).reshape(dims, n_free)
            c_o, cost_o = orc.set(mask, vals, t, r, dp4)
            coef, tt = opt.getSegments()
            assert np.array_equal(coef, c_o[:, :dims]) and opt.computeCost() == cost_o and np.array_equal(tt, t)
            assert np.array_equal(np.array(opt.getFreeConstraints()).reshape(dims, n_free), dp4[:dims])
            opt.updateSegmentTimes(t * 1.1)
            assert all(np.array_equal(v, np.zeros(n_free)) for v in opt.getFreeConstraints())
            # a batch: a list in, a list out
            optb = A.PolynomialOptimization(dims, ctx=ctx, n_coefficients=n_coef)
            assert optb.setupFromVertices(lists, times, r) and optb.solveLinear()
            fb = optb.getFreeConstraints()
            assert len(fb) == 3 and optb.getNumberFreeConstraints()[0] == n_free
            x = [[v * 1.5 for v in f] for f in fb]
            assert optb.setFreeConstraints(x)
            costs = optb.computeCost()
            for p, (mask, vals, t) in enumerate(probs):
                nf = orc.solve(mask, vals, t, r)[3][1]
                dp4 = np.zeros((4, nf))
                dp4[:dims] = np.array(x[p]).reshape(dims, nf)
                c_o, cost_o = orc.set(mask, vals, t, r, dp4)
                assert np.array_equal(optb.getSegments(p)[0], c_o[:, :dims]) and costs[p] == cost_o, (n_coef, dims, p)


def _shim_vertices(n_coef, dims):
    """the problem tests/cpp/test_shim_free_constraints.cpp builds"""
    H, r, V = n_coef // 2, min(2, n_coef // 2 - 1), 6
    mask = np.ones(V, np.uint8)
    vals = np.zeros((V, H, 4))
    for i in range(V):
        wp = np.array([1.1 * i, 0.7 if i % 2 == 0 else -0.5, 2.0 + 0.3 * i, 0.2 * i])
        vals[i, 0, :dims] = wp[:dims]
    mask[0] = mask[-1] = (1 << (r + 1)) - 1
    mask[2] |= 0b10
    vals[2, 1, :dims] = 0.4
    times = np.array([0.9 + 0.25 * (i % 3) for i in range(V - 1)])
    return mask, vals, times, r


def _run_shim(libdir, libname, tmp_path, extra=(), tag="plain"):
    exe = str(tmp_path / f"test_shim_free_constraints_{tag}")
    out = exe + ".txt"
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-pthread", *extra, "-o", exe, os.path.join(ROOT, "tests", "cpp", "test_shim_free_constraints.cpp"),
                           "-L" + libdir, "-l" + libname, "-Wl,-rpath," + libdir])
    subprocess.check_call([exe, out])
    res = {}
    for line in open(out):
        f = line.split()
        res[f[0]] = np.array([float.fromhex(x) for x in f[2:]])
    return res


def check_shim(ctx, fo, res):
    for n_coef in (6, 8, 10, 12):
        for dims in (3, 4):
            key = f"n{n_coef}d{dims}"
            mask, vals, times, r = _shim_vertices(n_coef, dims)
            _, _, _, (n_fixed, n_free) = fo(n_coef).solve(mask, vals, times, r)
            assert np.array_equal(res[key + "_counts"], [n_free, n_fixed, len(times) * n_coef]), key
            assert np.array_equal(res[key + "_free_before"], np.zeros(dims * n_free))
            bits = ((mask[:, None] >> np.arange(n_coef // 2)) & 1).astype(bool)
            assert np.array_equal(res[key + "_fixed"], np.concatenate([vals[:, :, d][bits] for d in range(dims)])), key
            off = np.array([0, len(mask)], np.int32)
            coef, cost, free = ctx.solve_linear_free_batch_nd(n_coef, dims, off, mask, np.ascontiguousarray(vals[:, :, :dims]), times, r)
            assert np.array_equal(res[key + "_free"], free[0].ravel()) and np.array_equal(res[key + "_free_again"], free[0].ravel()), key
            assert res[key + "_cost_solve"][0] == cost[0] and res[key + "_cost_after_bad"][0] == cost[0], key
            x = free[0].copy()
            x[dims - 1, 0] += 0.75
            assert np.array_equal(res[key + "_free_set"], x.ravel()), key
            c_s, k_s = ctx.set_free_constraints_batch_nd(n_coef, dims, off, mask, np.ascontiguousarray(vals[:, :, :dims]), times, [x], r)
            assert np.array_equal(res[key + "_coef"], c_s.ravel()) and res[key + "_cost"][0] == k_s[0], key
            t, v, i = ctx.max_magnitude_nd(n_coef, dims, np.array([0, len(times)], np.int32), c_s, times, 2)
            assert np.array_equal(res[key + "_maxacc"], [t[0], v[0], i[0]]), key
            assert np.array_equal(res[key + "_free_after_times"], np.zeros(dims * n_free)), key


def _eigen_flags():
    return ["-I" + os.path.join(ROOT, "oracle", "ref_shim")]


# ---- host emulation (small matrix) ------------------------------------------------------------------------------------------------
def _by_size(ctx):
    if ctx.solve_kernels != "by-size":
        pytest.skip("the general-shape path has one dispatch")


@pytest.mark.parametrize("n_coef,dims", SHAPES_EMU)
def test_get_set_round_trip_emulator(emu_ctx, free_oracle, n_coef, dims):
    _by_size(emu_ctx)
    check_get_set(emu_ctx, free_oracle, n_coef, dims)


def test_independence_and_refusals_emulator(emu_ctx):
    _by_size(emu_ctx)
    check_independence(emu_ctx, 12, 3)
    check_refusals(emu_ctx)


def test_python_class_emulator(emu_ctx, free_oracle):
    _by_size(emu_ctx)
    check_python_class(emu_ctx, free_oracle)


def test_cpp_shim_emulator(emu_ctx, emu_lib, free_oracle, tmp_path):
    _by_size(emu_ctx)
    libdir = os.path.join(ROOT, "tests", "host_emu")
    check_shim(emu_ctx, free_oracle, _run_shim(libdir, "tg_emu", tmp_path))
    check_shim(emu_ctx, free_oracle, _run_shim(libdir, "tg_emu", tmp_path, _eigen_flags(), "eigen"))


# ---- B200 (full matrix) -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", SHAPES_GPU)
def test_get_set_round_trip_gpu(gpu_ctx, free_oracle, n_coef, dims):
    check_get_set(gpu_ctx, free_oracle, n_coef, dims)
    check_get_set(gpu_ctx, free_oracle, n_coef, dims, seed=1)


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", [(6, 4), (10, 4), (12, 3)])
def test_independence_gpu(gpu_ctx, n_coef, dims):
    check_independence(gpu_ctx, n_coef, dims)


@pytest.mark.gpu
def test_refusals_gpu(gpu_ctx):
    check_refusals(gpu_ctx)


@pytest.mark.gpu
def test_python_class_gpu(gpu_ctx, free_oracle):
    check_python_class(gpu_ctx, free_oracle)


@pytest.mark.gpu
def test_cpp_shim_gpu(gpu_ctx, free_oracle, tmp_path):
    libdir = os.path.join(ROOT, "mrs_uav_trajectory_generation_b200")
    check_shim(gpu_ctx, free_oracle, _run_shim(libdir, "tg_b200", tmp_path))
    check_shim(gpu_ctx, free_oracle, _run_shim(libdir, "tg_b200", tmp_path, _eigen_flags(), "eigen"))


def node_problems(B, n_coef, V=11, r=2):
    """B random-flier paths of V waypoints with the node's vertex recipe (ends fixed up to r, interior positions) and times from the
    waypoint distances; vals [B*V][N/2][4]."""
    wp_off, wp = W.random_flier_paths_fast(B, V)
    mask = np.ones((B, V), np.uint8)
    mask[:, 0] = mask[:, -1] = (1 << (r + 1)) - 1
    vals = np.zeros((B * V, n_coef // 2, 4))
    vals[:, 0] = wp
    w = wp.reshape(B, V, 4)
    times = (np.linalg.norm(w[:, 1:, :3] - w[:, :-1, :3], axis=2) / 1.5 + 0.2).ravel()
    return wp_off, mask.ravel(), vals, times


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef", [10, 12])
def test_scale_gpu(gpu_ctx, free_oracle, n_coef):
    """65 536 problems through each entry point; a seeded sample of 256 compared with the oracle"""
    B, V, r = 65536, 11, 2
    off, mask, vals, times = node_problems(B, n_coef, V, r)
    coef, cost, free = gpu_ctx.solve_linear_free_batch_nd(n_coef, 4, off, mask, vals, times, r)
    x = perturbed(np.random.default_rng(3), free)
    c_s, k_s = gpu_ctx.set_free_constraints_batch_nd(n_coef, 4, off, mask, vals, times, x, r)
    assert np.isfinite(coef).all() and np.isfinite(c_s).all() and np.isfinite(cost).all() and np.isfinite(k_s).all()
    orc = free_oracle(n_coef)
    S = V - 1
    for p in np.random.default_rng(11).choice(B, 256, replace=False):
        m, v, t = mask[p * V:(p + 1) * V], vals[p * V:(p + 1) * V], times[p * S:(p + 1) * S]
        c_o, cost_o, dp_o, _ = orc.solve(m, v, t, r)
        assert np.array_equal(free[p], dp_o) and np.array_equal(coef[p * S:(p + 1) * S], c_o) and cost[p] == cost_o, p
        c_o, cost_o = orc.set(m, v, t, r, x[p])
        assert np.array_equal(c_s[p * S:(p + 1) * S], c_o) and k_s[p] == cost_o, p
