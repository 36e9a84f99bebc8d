"""General shape, nonlinear half: per-segment maxima, computeMaximumOfMagnitude, time scaling and the Mellinger time allocation of
PolynomialOptimizationNonLinear<N>(D) for N in {6, 8, 10, 12}, D in 1..4 (tg_extrema_batch_nd, tg_max_magnitude_batch_nd,
tg_scale_times_batch_nd, tg_time_alloc_batch_nd; csrc/tg_generic.cuh).  Checked bit for bit:
  * against the restatement compiled for that N (oracle/liboracle_n{6,8,12}.so), on the zero-padded coefficients -- on the host
    emulation of the device code (CPU) and on the GPU;
  * N = 10, D = 4: every general-shape entry point against its tuned sibling;
  * the restatement for N = 6, 8, 12 against the reference's own templates (oracle/_ref/libref_eth_n{N}.so), where a checkout of
    the reference is present.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
from test_general_shape import SHAPES, random_batch, random_vertices

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
dp, u8p, ip = C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(C.c_int)


def _p(a, t=dp):
    return a.ctypes.data_as(t)


# ---- the oracle compiled for N: [S][4][N] coefficients, [V][N/2][4] vertex values ------------------------------------------------
def orc_maxima(orc, c4, times):
    c4, times = np.ascontiguousarray(c4), np.ascontiguousarray(times)
    out = np.zeros((len(times), 9))
    orc.lib.orc_segment_maxima(len(times), _p(c4), _p(times), _p(out))
    return out


def orc_max_magnitude(orc, c4, times, derivative):
    c4, times = np.ascontiguousarray(c4), np.ascontiguousarray(times)
    t, v, i = C.c_double(), C.c_double(), C.c_int()
    orc.lib.orc_max_magnitude(len(times), _p(c4), _p(times), int(derivative), C.byref(t), C.byref(v), C.byref(i))
    return t.value, v.value, i.value


def orc_scale(orc, c4, times, limits):
    c4, times = np.array(c4, order="C"), np.array(times, dtype=np.float64)
    lim = np.ascontiguousarray(limits, dtype=np.float64)
    w = C.c_int()
    passes = orc.lib.orc_scale_times(len(times), _p(c4), _p(times), _p(lim), C.byref(w))
    return c4, times, passes, bool(w.value)


def orc_set_tolerance(orc, tol):
    orc.lib.orc_set_scale_tolerance.argtypes = [C.c_double]
    orc.lib.orc_set_scale_tolerance(float(tol))


def orc_time_alloc(orc, mask, vals4, times, r, params):
    mask, vals4 = np.ascontiguousarray(mask, dtype=np.uint8), np.ascontiguousarray(vals4)
    t = np.array(times, dtype=np.float64)
    coef = np.zeros((len(t), 4, orc.N))
    code, ev, passes, cost = C.c_int(), C.c_int(), C.c_int(), C.c_double()
    assert orc.lib.orc_time_alloc(len(mask), _p(mask, u8p), _p(vals4), _p(t), int(r), C.byref(params), _p(coef), C.byref(code), C.byref(ev),
                                  C.byref(passes), C.byref(cost)) == 0
    return dict(times=t, coef=coef, nlopt_code=code.value, n_evals=ev.value, n_scale_passes=passes.value, final_cost=cost.value)


def pad4(coef):
    c4 = np.zeros((coef.shape[0], 4, coef.shape[2]))
    c4[:, :coef.shape[1]] = coef
    return c4


def oracle_params(ctx, **kw):
    """The library's tg_params as the oracle's orc_params (the same layout)."""
    p = ctx.L.default_params(**kw)
    q = O.Params()
    C.memmove(C.byref(q), C.byref(p), C.sizeof(O.Params))
    return q


def solved_batch(ctx, n_coef, dims, seed, B=12, r=None):
    """A ragged batch of solved trajectories with a short (0.01 s) and a long (20 s) segment in it -> seg_off, coef, times."""
    rng = np.random.default_rng(seed)
    off, masks, vals, times = random_batch(rng, n_coef, B, dims)
    t = np.concatenate(times)
    t[rng.integers(0, len(t), 2)] = (0.01, 20.0)
    r = min(2, n_coef // 2 - 1) if r is None else r
    coef, _ = ctx.solve_linear_batch_nd(n_coef, dims, off, np.concatenate(masks), np.concatenate(vals)[:, :, :dims], t, r)
    return off - np.arange(len(off), dtype=np.int32), coef, t


def general_only(ctx):
    if getattr(ctx, "solve_kernels", "by-size") != "by-size":
        pytest.skip("the general-shape path has one dispatch")


# ---- checks --------------------------------------------------------------------------------------------------------------------------
def check_maxima(ctx, n_coef, dims):
    orc = O.OracleN(n_coef)
    seg_off, coef, t = solved_batch(ctx, n_coef, dims, 10 * n_coef + dims)
    m = ctx.extrema_nd(n_coef, dims, coef, t)
    assert np.array_equal(m, orc_maxima(orc, pad4(coef), t)), (n_coef, dims)
    for p in range(len(seg_off) - 1):
        s0, s1 = seg_off[p], seg_off[p + 1]
        for k in (1, 2, 3, 4):
            got = ctx.max_magnitude_nd(n_coef, dims, seg_off[p:p + 2] - s0, coef[s0:s1], t[s0:s1], k)
            assert tuple(x[0] for x in got) == orc_max_magnitude(orc, pad4(coef[s0:s1]), t[s0:s1], k), (n_coef, dims, p, k)
    for k in (1, 2, 3, 4):  # the whole ragged batch in one call
        tt, vv, ii = ctx.max_magnitude_nd(n_coef, dims, seg_off, coef, t, k)
        for p in range(len(seg_off) - 1):
            s0, s1 = seg_off[p], seg_off[p + 1]
            assert (tt[p], vv[p], ii[p]) == orc_max_magnitude(orc, pad4(coef[s0:s1]), t[s0:s1], k)


def check_scaling(ctx, n_coef, dims):
    orc = O.OracleN(n_coef)
    rng = np.random.default_rng(7 * n_coef + dims)
    passes_seen = set()
    try:
        for tol in (1e-3, -0.2, -0.6):
            orc_set_tolerance(orc, tol)
            ctx.test_set_scale_tolerance(tol)
            seg_off, coef, t = solved_batch(ctx, n_coef, dims, int(rng.integers(1 << 30)))
            lim = np.array(O.DEFAULT_LIMITS) * np.exp(rng.uniform(-1.5, 0.5, 9))
            c2, t2, passes, within = ctx.scale_times_nd(n_coef, dims, seg_off, coef, t, lim)
            for p in range(len(seg_off) - 1):
                s0, s1 = seg_off[p], seg_off[p + 1]
                rc, rt, rp, rw = orc_scale(orc, pad4(coef[s0:s1]), t[s0:s1], lim)
                assert np.array_equal(c2[s0:s1], rc[:, :dims]) and np.array_equal(t2[s0:s1], rt), (n_coef, dims, tol, p)
                assert passes[p] == rp and bool(within[p]) == rw, (n_coef, dims, tol, p, passes[p], rp)
                passes_seen.add(int(rp))
    finally:
        orc_set_tolerance(orc, 1e-3)
        ctx.test_set_scale_tolerance(1e-3)
    assert max(passes_seen) > 1


def alloc_problems(rng, n_coef, dims, B=24):
    """B problems of S = 1 .. 12 segments (the first one S = 1); problem 1 starts below the 0.01 s bound (nlopt code -1)."""
    off, masks, vals, times = [0], [], [], []
    for p in range(B):
        V = 2 if p == 0 else int(rng.integers(2, 14))
        m, v = random_vertices(rng, n_coef, V, dims)
        t = rng.uniform(0.3, 5.0, V - 1)
        if p == 1:
            t[0] = 0.005
        masks.append(m)
        vals.append(v)
        times.append(t)
        off.append(off[-1] + V)
    return np.array(off, np.int32), masks, vals, times


def check_time_alloc(ctx, n_coef, dims, seed=0, rs=None):
    orc = O.OracleN(n_coef)
    rng = np.random.default_rng(100 * n_coef + dims + 1000 * seed)
    tight = (1.0, 0.5, 0.5, 0.3, 2.0, 2.0, 0.3, 0.3, 1.0)
    for r in (range(n_coef // 2) if rs is None else rs):
        for kw in ({}, {"max_evals": 1}, {"limits": tight}):
            off, masks, vals, times = alloc_problems(rng, n_coef, dims)
            vv = np.concatenate(vals)[:, :, :dims]
            got = ctx.time_alloc_batch_nd(n_coef, dims, off, np.concatenate(masks), vv, np.concatenate(times),
                                          ctx.L.default_params(derivative_to_optimize=r, **kw))
            P = oracle_params(ctx, derivative_to_optimize=r, **kw)
            s0 = 0
            for p in range(len(masks)):
                ref = orc_time_alloc(orc, masks[p], vals[p], times[p], r, P)
                S = len(times[p])
                where = (n_coef, dims, r, kw, p)
                assert got["nlopt_code"][p] == ref["nlopt_code"] and got["n_evals"][p] == ref["n_evals"], where
                assert got["n_scale_passes"][p] == ref["n_scale_passes"] and got["final_cost"][p] == ref["final_cost"], where
                assert np.array_equal(got["times"][s0:s0 + S], ref["times"]), where
                assert np.array_equal(got["coef"][s0:s0 + S], ref["coef"][:, :dims]), where
                s0 += S
            assert got["nlopt_code"][1] == -1 and got["n_evals"][1] == 0
            if "limits" in kw:
                assert got["n_scale_passes"].max() >= 1


def check_tuned_equals_general(ctx):
    """N = 10, D = 4: each _nd entry point gives the bits of its tuned sibling."""
    rng = np.random.default_rng(1234)
    seg_off, coef, t = solved_batch(ctx, 10, 4, 55, B=24)
    assert np.array_equal(ctx.extrema_nd(10, 4, coef, t), ctx.extrema(coef, t))
    for k in (1, 2, 3, 4):
        a, b = ctx.max_magnitude_nd(10, 4, seg_off, coef, t, k), ctx.max_magnitude(seg_off, coef, t, k)
        assert all(np.array_equal(x, y) for x, y in zip(a, b)), k
    try:
        for tol in (1e-3, -0.4):
            ctx.test_set_scale_tolerance(tol)
            lim = np.array(O.DEFAULT_LIMITS) * np.exp(rng.uniform(-1.5, 0.5, 9))
            a, b = ctx.scale_times_nd(10, 4, seg_off, coef, t, lim), ctx.scale_times(seg_off, coef, t, lim)
            assert all(np.array_equal(x, y) for x, y in zip(a, b)), tol
    finally:
        ctx.test_set_scale_tolerance(1e-3)
    for r in (2, 3, 4):
        for kw in ({}, {"limits": (1.0, 0.5, 0.5, 0.3, 2.0, 2.0, 0.3, 0.3, 1.0)}):
            off, masks, vals, times = alloc_problems(rng, 10, 4)
            args = (off, np.concatenate(masks), np.concatenate(vals), np.concatenate(times), ctx.L.default_params(derivative_to_optimize=r, **kw))
            a, b = ctx.time_alloc_batch_nd(10, 4, *args), ctx.time_alloc_batch(*args)
            for key in a:
                assert np.array_equal(a[key], b[key]), (r, kw, key)


def check_refusals(ctx):
    rng = np.random.default_rng(3)
    seg_off, coef, t = solved_batch(ctx, 8, 4, 1, B=3)
    L9 = np.array(O.DEFAULT_LIMITS)
    m, v = random_vertices(rng, 8, 4)
    off = np.array([0, 4], np.int32)
    for n_coef, dims in ((4, 4), (7, 4), (14, 4), (8, 0), (8, 5)):
        n, d = max(n_coef, 1), max(dims, 1)
        c = np.zeros((len(t), d, n))
        with pytest.raises(Exception):
            ctx.extrema_nd(n_coef, dims, c, t)
        with pytest.raises(Exception):
            ctx.max_magnitude_nd(n_coef, dims, seg_off, c, t, 1)
        with pytest.raises(Exception):
            ctx.scale_times_nd(n_coef, dims, seg_off, c, t, L9)
        with pytest.raises(Exception):
            ctx.time_alloc_batch_nd(n_coef, dims, off, m, np.zeros((4, max(n // 2, 1), d)), np.ones(3))
    for k in (0, 5):
        with pytest.raises(Exception):
            ctx.max_magnitude_nd(8, 4, seg_off, coef, t, k)
    for r in (-1, 4):
        with pytest.raises(Exception):
            ctx.time_alloc_batch_nd(8, 4, off, m, v, np.ones(3), ctx.L.default_params(derivative_to_optimize=r))
    with pytest.raises(Exception):
        ctx.time_alloc_batch_nd(8, 4, off, m, v, np.ones(3), ctx.L.default_params(max_evals=0))
    empty = np.array([0], np.int32)  # B = 0
    with pytest.raises(Exception):
        ctx.max_magnitude_nd(8, 4, empty, coef[:0], t[:0], 1)
    with pytest.raises(Exception):
        ctx.scale_times_nd(8, 4, empty, coef[:0], t[:0], L9)
    with pytest.raises(Exception):
        ctx.time_alloc_batch_nd(8, 4, np.array([0], np.int32), m[:0], v[:0], np.ones(0))
    with pytest.raises(Exception):
        ctx.extrema_nd(8, 4, coef[:0], t[:0])
    no_seg = np.array([0, 2, 2, 3], np.int32)  # the second trajectory has no segment
    with pytest.raises(Exception):
        ctx.max_magnitude_nd(8, 4, no_seg, coef[:3], t[:3], 1)
    with pytest.raises(Exception):
        ctx.scale_times_nd(8, 4, no_seg, coef[:3], t[:3], L9)
    with pytest.raises(Exception):
        ctx.time_alloc_batch_nd(8, 4, np.array([0, 4, 5], np.int32), np.concatenate([m, m[:1]]), np.concatenate([v, v[:1]]), np.ones(3))


def check_api(ctx):
    import mrs_uav_trajectory_generation_b200.api as A

    # a (3, 8) trajectory: maxima and time scaling on its own shape
    n_coef, dims, r = 8, 3, 3
    pts = [np.array([1.3 * i, (-1.0) ** i * 0.7, 2.0 + 0.2 * i]) for i in range(6)]
    verts = []
    for i, p in enumerate(pts):
        v = A.Vertex(dims)
        if i in (0, len(pts) - 1):
            v.makeStartOrEnd(p, r)
        else:
            v.addConstraint(A.derivative_order.POSITION, p)
        verts.append(v)
    times = np.array([0.9, 1.1, 0.7, 1.4, 1.0])
    opt = A.PolynomialOptimization(dims, ctx=ctx, n_coefficients=n_coef)
    assert opt.setupFromVertices(verts, times, r) and opt.solveLinear()
    traj = opt.getTrajectory()
    orc = O.OracleN(n_coef)
    c4 = pad4(traj.coef)
    assert np.array_equal(traj.computeMaxDerivatives(), orc_maxima(orc, c4, times))
    lim = (1.0, 0.5, 0.5, 0.3, 2.0, 2.0, 0.3, 0.3, 1.0)
    rc, rt, _, rw = orc_scale(orc, c4, times, lim)
    assert traj.scaleSegmentTimesToMeetConstraints(lim) == rw
    assert np.array_equal(traj.coef, rc[:, :dims]) and np.array_equal(traj.times, rt)
    # PolynomialOptimizationNonLinear<12>(4) from vertices, Mellinger
    n_coef, dims, r = 12, 4, 3
    rng = np.random.default_rng(8)
    pts = [rng.normal(size=4) * 3.0 for _ in range(7)]
    verts = []
    for i, p in enumerate(pts):
        v = A.Vertex(dims)
        if i in (0, len(pts) - 1):
            v.makeStartOrEnd(p, r)
        else:
            v.addConstraint(A.derivative_order.POSITION, p)
        verts.append(v)
    times = np.full(6, 1.5)
    P = A.NonlinearOptimizationParameters()
    nl = A.PolynomialOptimizationNonLinear(dims, P, ctx=ctx, n_coefficients=n_coef)
    assert nl.setupFromVertices(verts, times, r)
    for dim, der, val in ((0, 1, 2.0), (1, 1, 2.0), (2, 1, 1.0), (0, 2, 1.5), (2, 2, 1.0)):
        assert nl.addMaximumMagnitudeConstraint(dim, der, val)
    code = nl.optimize()
    t = nl.getTrajectory()
    _, masks, vals = A.pack_vertices([verts], n_coef // 2, dims)
    Pp = oracle_params(ctx, derivative_to_optimize=r, max_evals=P.max_iterations, f_rel=P.f_rel, x_rel=P.x_rel, check_deviation=0,
                       limits=[nl._limits[i] if nl._limits[i] is not None else 3.4028234663852886e38 for i in range(9)])
    ref = orc_time_alloc(O.OracleN(n_coef), masks, vals, times, r, Pp)
    assert code == ref["nlopt_code"] and np.array_equal(t.times, ref["times"]) and np.array_equal(t.coef, ref["coef"])
    assert not A.PolynomialOptimizationNonLinear(dims, P, ctx=ctx, n_coefficients=8).setupFromVertices(verts, times, 4)  # above N/2 - 1
    P0 = A.NonlinearOptimizationParameters()
    P0.time_alloc_method = 0
    assert not A.PolynomialOptimizationNonLinear(dims, P0, ctx=ctx, n_coefficients=n_coef).setupFromVertices(verts, times, r)


# ---- host emulation (CPU) ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_coef,dims", SHAPES)
def test_maxima_general_shape_emulator(emu_ctx, oracle, n_coef, dims):
    general_only(emu_ctx)
    check_maxima(emu_ctx, n_coef, dims)


@pytest.mark.parametrize("n_coef,dims", SHAPES)
def test_scaling_general_shape_emulator(emu_ctx, oracle, n_coef, dims):
    general_only(emu_ctx)
    check_scaling(emu_ctx, n_coef, dims)


@pytest.mark.parametrize("n_coef,dims", SHAPES)
def test_time_alloc_general_shape_emulator(emu_ctx, oracle, n_coef, dims):
    general_only(emu_ctx)
    check_time_alloc(emu_ctx, n_coef, dims)


def test_nonlinear_tuned_equals_general_emulator(emu_ctx, oracle):
    general_only(emu_ctx)
    check_tuned_equals_general(emu_ctx)


def test_nonlinear_general_shape_refusals_emulator(emu_ctx):
    general_only(emu_ctx)
    check_refusals(emu_ctx)


def test_nonlinear_api_general_shape_emulator(emu_ctx, oracle):
    general_only(emu_ctx)
    check_api(emu_ctx)


# ---- the B200 ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", SHAPES)
def test_maxima_general_shape_gpu(gpu_ctx, oracle, n_coef, dims):
    check_maxima(gpu_ctx, n_coef, dims)


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", SHAPES)
def test_scaling_general_shape_gpu(gpu_ctx, oracle, n_coef, dims):
    check_scaling(gpu_ctx, n_coef, dims)


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", SHAPES)
def test_time_alloc_general_shape_gpu(gpu_ctx, oracle, n_coef, dims):
    check_time_alloc(gpu_ctx, n_coef, dims)


@pytest.mark.gpu
def test_nonlinear_tuned_equals_general_gpu(gpu_ctx, oracle):
    check_tuned_equals_general(gpu_ctx)


@pytest.mark.gpu
def test_nonlinear_general_shape_refusals_gpu(gpu_ctx):
    check_refusals(gpu_ctx)


@pytest.mark.gpu
def test_nonlinear_api_general_shape_gpu(gpu_ctx, oracle):
    check_api(gpu_ctx)


@pytest.mark.gpu
def test_time_alloc_general_shape_large_batch_gpu(gpu_ctx, oracle):
    """4096 problems of N = 12 in one call: all finite, 64 of them equal to the oracle."""
    rng = np.random.default_rng(4096)
    off, masks, vals, times = random_batch(rng, 12, 4096, 4)
    P = gpu_ctx.L.default_params(derivative_to_optimize=3)
    got = gpu_ctx.time_alloc_batch_nd(12, 4, off, np.concatenate(masks), np.concatenate(vals), np.concatenate(times), P)
    assert np.isfinite(got["coef"]).all() and np.isfinite(got["times"]).all() and np.isfinite(got["final_cost"]).all()
    orc = O.OracleN(12)
    Po = oracle_params(gpu_ctx, derivative_to_optimize=3)
    seg_off = off - np.arange(len(off), dtype=np.int32)
    for p in rng.integers(0, 4096, 64):
        ref = orc_time_alloc(orc, masks[p], vals[p], times[p], 3, Po)
        s0, s1 = seg_off[p], seg_off[p + 1]
        assert got["nlopt_code"][p] == ref["nlopt_code"] and got["n_evals"][p] == ref["n_evals"] and got["final_cost"][p] == ref["final_cost"]
        assert np.array_equal(got["times"][s0:s1], ref["times"]) and np.array_equal(got["coef"][s0:s1], ref["coef"])


# ---- the restatement for N = 6, 8, 12 against the reference's own templates --------------------------------------------------------
@pytest.mark.parametrize("n_coef", [6, 8, 12])
def test_nonlinear_restatement_equals_reference_templates(n_coef):
    """Segment maxima, computeMaximumOfMagnitude, time scaling and the Mellinger time allocation of the reference instantiated for N
    (libref_eth_n{N}.so) against the oracle for that N in LIBM mode."""
    if not O.REFERENCE:
        pytest.skip("needs a checkout of the original ctu-mrs/mrs_uav_trajectory_generation (TG_REFERENCE_DIR or BASELINE.json reference_path)")
    O.build_oracle(ref=True)
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", f"libref_eth_n{n_coef}.so"))
    orc = O.OracleN(n_coef, mode=O.MATH_LIBM)
    try:
        rng = np.random.default_rng(31 + n_coef)
        r = 2
        for _ in range(6):
            V = int(rng.integers(2, 10))
            mask, vals = random_vertices(rng, n_coef, V)
            times = rng.uniform(0.3, 5.0, V - 1)
            c4, _ = orc.solve_linear(mask, vals, times, r)
            S = V - 1
            m_ref = np.zeros((S, 9))
            lib.ref_segment_maxima(S, _p(np.ascontiguousarray(c4)), _p(times), _p(m_ref))
            assert np.array_equal(m_ref, orc_maxima(orc, c4, times))
            for k in (1, 2, 3, 4):
                t, v, i = C.c_double(), C.c_double(), C.c_int()
                lib.ref_solve_max_magnitude(V, _p(mask, u8p), _p(np.ascontiguousarray(vals)), _p(times), r, k, C.byref(t), C.byref(v), C.byref(i))
                assert (t.value, v.value, i.value) == orc_max_magnitude(orc, c4, times, k)
            lim = np.array(O.DEFAULT_LIMITS) * 0.5
            cr, tr = np.array(c4), np.array(times)
            w = C.c_int()
            lib.ref_scale_times(S, _p(cr), _p(tr), _p(lim), C.byref(w))  # the reference does not expose its pass count
            rc, rt, _, rw = orc_scale(orc, c4, times, lim)
            assert np.array_equal(cr, rc) and np.array_equal(tr, rt) and bool(w.value) == rw
            P = O.default_params(derivative_to_optimize=r)
            ref = orc_time_alloc(orc, mask, vals, times, r, P)
            tt, cc = np.array(times), np.zeros((S, 4, n_coef))
            code, ev, cost = C.c_int(), C.c_int(), C.c_double()
            assert lib.ref_time_alloc(V, _p(mask, u8p), _p(np.ascontiguousarray(vals)), _p(tt), r, P.max_evals, C.c_double(P.f_rel), C.c_double(P.x_rel),
                                      _p(np.array(list(P.limits))), _p(cc), C.byref(code), C.byref(ev), C.byref(cost)) == 0
            assert np.array_equal(tt, ref["times"]) and np.array_equal(cc, ref["coef"]) and code.value == ref["nlopt_code"]
            assert ev.value == ref["n_evals"] and cost.value == ref["final_cost"]
    finally:
        orc.lib.orc_set_math_mode(O.MATH_DET)


# ---- the C++ header (include/eth_trajectory_generation_b200.hpp): tests/cpp/test_shim_nonlinear_general.cpp -------------------------
def check_cpp(res):
    def vertices(n_coef, dims, r):
        H = n_coef // 2
        mask = np.ones(7, np.uint8)
        mask[0] = mask[-1] = (1 << (r + 1)) - 1
        vals = np.zeros((7, H, 4))
        for i in range(7):
            vals[i, 0, :dims] = np.array([1.9 * i, 0.8 if i % 2 == 0 else -0.5, 2.0 + 0.4 * i, 0.2 * i])[:dims]
        return mask, vals

    times = np.array([0.9 + 0.2 * (i % 3) for i in range(6)])
    big = 3.40282346638528859812e+38
    for key, n_coef, dims, r in (("n8d3", 8, 3, 3), ("n12d4", 12, 4, 4), ("n6d2", 6, 2, 2)):
        orc = O.OracleN(n_coef)
        mask, vals = vertices(n_coef, dims, r)
        P = O.default_params(derivative_to_optimize=r, limits=(2.5, 1.0 if dims >= 3 else big, 1.5, big, big, big, big, big, big))
        ref = orc_time_alloc(orc, mask, vals, times, r, P)
        got = res[key + "_times_code"][0]
        assert np.array_equal(got[:-1], ref["times"]) and int(got[-1]) == ref["nlopt_code"], key
        assert np.array_equal(res[key + "_coef"][0].reshape(-1, dims, n_coef), ref["coef"][:, :dims]), key
        assert res[key + "_dfo_refused"][0][0] == 1.0, key
    orc = O.OracleN(12)
    mask, vals = vertices(12, 4, 3)
    coef, _ = orc.solve_linear(mask, vals, times, 3)
    for k in (1, 2, 3, 4):
        assert np.array_equal(res["n12d4_maxmag"][k - 1], np.array(orc_max_magnitude(orc, coef, times, k), dtype=np.float64)), k


def test_cpp_shim_nonlinear_general_shapes_on_host_emulation(oracle, emu_lib, tmp_path):
    from test_cpp_shim import _run_shim

    check_cpp(_run_shim(os.path.join(ROOT, "tests", "host_emu"), "tg_emu", tmp_path, "test_shim_nonlinear_general.cpp"))


@pytest.mark.gpu
def test_cpp_shim_nonlinear_general_shapes_on_gpu(oracle, gpu_ctx, tmp_path):
    from test_cpp_shim import _run_shim

    check_cpp(_run_shim(os.path.join(ROOT, "mrs_uav_trajectory_generation_b200"), "tg_b200", tmp_path, "test_shim_nonlinear_general.cpp"))
