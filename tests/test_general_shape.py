"""General shape (SURVEY 8f rank 4): PolynomialOptimization<N>(D) for N in {6, 8, 10, 12}, D in 1..4, r in 0 .. N/2-1.

The reference's classes are templates over the number of coefficients N (lin.h:46-55, Polynomial::kMaxN = 12 in
eth/polynomial.h:45-48) and take the dimension at run time.  The product serves those shapes through tg_solve_linear_batch_nd /
tg_evaluate_batch_nd / tg_sample_batch_nd (csrc/tg_generic.cuh).  Checked here, bit for bit:
  * against the restatement compiled for that N (oracle/liboracle_n{6,8,12}.so = the same sources with -DORC_N) -- on the host
    emulation of the device code (CPU) and on the GPU;
  * N = 10, D = 4: the general-shape kernels against the tuned kernels of the benchmarked path;
  * the restatement for N = 6, 8, 12 against the REFERENCE's own templates instantiated for that N
    (oracle/_ref/libref_eth_n{6,8,12}.so, built from a checkout of the reference against the stand-in headers), and against
    the vectors that build left in tests/golden/ref_eth_general.npz (the same inputs) for machines without that checkout.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden", "ref_eth_general.npz")
SHAPES = [(6, 3), (8, 1), (8, 4), (10, 3), (10, 4), (12, 2), (12, 4)]


def random_vertices(rng, n_coef, V, dims=4):
    """Vertex lists of the kind the node and the reference's tests build: end points fixed up to a random derivative, interior
    vertices with a fixed position and now and then a fixed higher derivative (eth/vertex.cpp:134-163)."""
    H = n_coef // 2
    mask = np.zeros(V, np.uint8)
    vals = np.zeros((V, H, 4))
    for v in range(V):
        if v in (0, V - 1):
            up_to = H if rng.random() < 0.6 else int(rng.integers(1, H + 1))
            mask[v] = (1 << up_to) - 1
        else:
            mask[v] = 1
            if rng.random() < 0.25:
                mask[v] |= 1 << int(rng.integers(1, H))
        for k in range(H):
            if (mask[v] >> k) & 1:
                vals[v, k, :dims] = rng.normal(size=dims) * (4.0 if k == 0 else 0.6)
    return mask, vals


def random_batch(rng, n_coef, B, dims):
    off, masks, vals, times = [0], [], [], []
    for _ in range(B):
        V = int(rng.integers(2, 14))
        m, v = random_vertices(rng, n_coef, V, dims)
        masks.append(m)
        vals.append(v)
        times.append(rng.uniform(0.3, 5.0, V - 1))
        off.append(off[-1] + V)
    return np.array(off, np.int32), masks, vals, times


def check_linear(ctx, n_coef, dims, seed=0):
    H = n_coef // 2
    orc = O.OracleN(n_coef)
    rng = np.random.default_rng(1000 * n_coef + 10 * dims + seed)
    for r in range(0, H):
        off, masks, vals, times = random_batch(rng, n_coef, 24, dims)
        vv = np.concatenate(vals)[:, :, :dims]
        coef, cost = ctx.solve_linear_batch_nd(n_coef, dims, off, np.concatenate(masks), vv, np.concatenate(times), r)
        s0 = 0
        for p in range(len(masks)):
            c_o, cost_o = orc.solve_linear(masks[p], vals[p], times[p], r)
            S = len(times[p])
            assert np.array_equal(coef[s0:s0 + S], c_o[:, :dims, :]), (n_coef, dims, r, p)
            assert cost[p] == cost_o, (n_coef, dims, r, p, cost[p], cost_o)
            assert np.all(c_o[:, dims:, :] == 0.0)
            s0 += S


def check_tuned_equals_general(ctx):
    """N = 10, D = 4, r = 2..4: both device paths give the same bits."""
    rng = np.random.default_rng(77)
    for r in (2, 3, 4):
        off, masks, vals, times = random_batch(rng, 10, 32, 4)
        args = (off, np.concatenate(masks), np.concatenate(vals), np.concatenate(times), r)
        c_t, cost_t = ctx.solve_linear_batch(*args)
        c_g, cost_g = ctx.solve_linear_batch_nd(10, 4, *args)
        assert np.array_equal(c_t, c_g) and np.array_equal(cost_t, cost_g), r


def check_evaluate_and_sample(ctx, n_coef, dims):
    orc = O.OracleN(n_coef)
    rng = np.random.default_rng(5 * n_coef + dims)
    off, masks, vals, times = random_batch(rng, n_coef, 6, dims)
    r = min(2, n_coef // 2 - 1)
    vv = np.concatenate(vals)[:, :, :dims]
    coef, _ = ctx.solve_linear_batch_nd(n_coef, dims, off, np.concatenate(masks), vv, np.concatenate(times), r)
    seg_off = off - np.arange(len(off), dtype=np.int32)
    c4 = np.zeros((coef.shape[0], 4, n_coef))
    c4[:, :dims, :] = coef
    for p in range(len(masks)):
        cs, ts = coef[seg_off[p]:seg_off[p + 1]], times[p]
        tq = np.concatenate([[0.0, ts.sum(), ts.sum() + 1.0, ts[0]], rng.uniform(0.0, ts.sum(), 12)])
        for deriv in (0, 1, 2, 4, n_coef - 1, n_coef, n_coef + 3):
            out, ok = ctx.evaluate_nd(n_coef, dims, cs, ts, tq, deriv)
            for k, t in enumerate(tq):
                o, okk = orc.trajectory_evaluate(c4[seg_off[p]:seg_off[p + 1]], ts, t, deriv)
                assert ok[k] == okk and np.array_equal(out[k], o[:dims]), (n_coef, dims, p, deriv, t)
    if dims < 3:
        with pytest.raises(Exception):
            ctx.sample_batch_nd(n_coef, dims, seg_off, coef, np.concatenate(times), 0.2)
        return
    for dt in (0.2, 0.037):
        counts, samples, full = ctx.sample_batch_nd(n_coef, dims, seg_off, coef, np.concatenate(times), dt, full=True)
        m0 = 0
        for p in range(len(masks)):
            ref = orc.sample(c4[seg_off[p]:seg_off[p + 1]], times[p], dt)
            assert counts[p] == len(ref), (n_coef, dims, p, counts[p], len(ref))
            assert np.array_equal(full[m0:m0 + counts[p]], ref)
            assert np.array_equal(samples[m0:m0 + counts[p], :3], ref[:, :3]) and np.array_equal(samples[m0:m0 + counts[p], 3], ref[:, 18])
            m0 += counts[p]


def check_refusals(ctx):
    rng = np.random.default_rng(3)
    m, v = random_vertices(rng, 8, 4)
    t = np.ones(3)
    off = np.array([0, 4], np.int32)
    for n_coef, dims, r in ((7, 4, 2), (14, 4, 2), (4, 4, 1), (8, 5, 2), (8, 0, 2), (8, 4, 4), (8, 4, -1)):
        with pytest.raises(Exception):
            vv = np.zeros((4, max(n_coef // 2, 1), max(dims, 1)))
            ctx.solve_linear_batch_nd(n_coef, dims, off, m, vv, t, r)


def check_api(ctx):
    """The reference-shaped host classes on another shape: Vertex(3), PolynomialOptimization<8>(3), Trajectory, sampleWholeTrajectory."""
    import mrs_uav_trajectory_generation_b200.api as A

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
    assert not A.PolynomialOptimization(dims, ctx=ctx, n_coefficients=n_coef).setupFromVertices(verts, times, 4)  # above N/2 - 1
    traj = opt.getTrajectory()
    assert traj.shape() == (dims, n_coef)
    orc = O.OracleN(n_coef)
    mask = np.ones(len(pts), np.uint8)
    mask[0] = mask[-1] = (1 << (r + 1)) - 1
    vals = np.zeros((len(pts), n_coef // 2, 4))
    for i, p in enumerate(pts):
        vals[i, 0, :dims] = p
    c_o, cost_o = orc.solve_linear(mask, vals, times, r)
    assert np.array_equal(traj.coef, c_o[:, :dims]) and opt.computeCost() == cost_o
    assert np.array_equal(traj.evaluate(2.2, 1), orc.trajectory_evaluate(c_o, times, 2.2, 1)[0][:dims])
    full = A.sample_whole_trajectory(traj, 0.25, full=True)
    assert np.array_equal(full, orc.sample(c_o, times, 0.25))
    # the segment YAML format carries the shape (eth/io.cpp:27-59): write, read back, same trajectory
    back = A.Trajectory.fromYaml(traj.toYaml(), ctx=ctx)
    assert back is not None and back.shape() == (dims, n_coef) and np.array_equal(back.coef, traj.coef)
    assert np.array_equal(back.evaluate(1.1, 2), orc.trajectory_evaluate(c_o, np.floor(times * 1e9) * 1e-9, 1.1, 2)[0][:dims])
    opt4 = A.PolynomialOptimization(4, ctx=ctx, n_coefficients=8)
    assert opt4.setupFromVertices(verts, times, 2)
    with pytest.raises(ValueError):
        opt4.solveLinear()  # three-dimensional vertices in a four-dimensional optimisation


def test_api_general_shape_emulator(emu_ctx, oracle):
    check_api(emu_ctx)


@pytest.mark.gpu
def test_api_general_shape_gpu(gpu_ctx, oracle):
    check_api(gpu_ctx)


@pytest.mark.parametrize("n_coef,dims", SHAPES)
def test_linear_general_shape_emulator(emu_ctx, oracle, n_coef, dims):
    check_linear(emu_ctx, n_coef, dims)


def test_tuned_equals_general_emulator(emu_ctx):
    check_tuned_equals_general(emu_ctx)


@pytest.mark.parametrize("n_coef,dims", [(6, 3), (8, 4), (12, 4), (12, 2)])
def test_evaluate_and_sample_general_shape_emulator(emu_ctx, oracle, n_coef, dims):
    if emu_ctx.solve_kernels != "by-size":
        pytest.skip("the general-shape path has one dispatch")
    check_evaluate_and_sample(emu_ctx, n_coef, dims)


def test_general_shape_refusals_emulator(emu_ctx):
    check_refusals(emu_ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", SHAPES)
def test_linear_general_shape_gpu(gpu_ctx, oracle, n_coef, dims):
    check_linear(gpu_ctx, n_coef, dims)
    check_linear(gpu_ctx, n_coef, dims, seed=1)


@pytest.mark.gpu
def test_tuned_equals_general_gpu(gpu_ctx):
    check_tuned_equals_general(gpu_ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("n_coef,dims", [(6, 3), (8, 4), (12, 4), (12, 2)])
def test_evaluate_and_sample_general_shape_gpu(gpu_ctx, oracle, n_coef, dims):
    check_evaluate_and_sample(gpu_ctx, n_coef, dims)


@pytest.mark.gpu
def test_general_shape_refusals_gpu(gpu_ctx):
    check_refusals(gpu_ctx)


@pytest.mark.gpu
def test_general_shape_large_batch_gpu(gpu_ctx, oracle):
    """4096 problems of N = 12 in one call (one warp each): spot-checked against the oracle, all finite."""
    rng = np.random.default_rng(99)
    off, masks, vals, times = random_batch(rng, 12, 4096, 4)
    coef, cost = gpu_ctx.solve_linear_batch_nd(12, 4, off, np.concatenate(masks), np.concatenate(vals), np.concatenate(times), 3)
    assert np.isfinite(coef).all() and np.isfinite(cost).all() and (cost >= 0).all()
    orc = O.OracleN(12)
    seg_off = off - np.arange(len(off), dtype=np.int32)
    for p in rng.integers(0, 4096, 64):
        c_o, cost_o = orc.solve_linear(masks[p], vals[p], times[p], 3)
        assert np.array_equal(coef[seg_off[p]:seg_off[p + 1]], c_o) and cost[p] == cost_o


# ---- the restatement for N = 6, 8, 12 against the reference's own templates ------------------------------------------------------
dp = C.POINTER(C.c_double)
u8p = C.POINTER(C.c_uint8)
ip = C.POINTER(C.c_int)


def _p(a, t=dp):
    return a.ctypes.data_as(t)


def reference_cases(n_coef):
    """Deterministic inputs shared by the live comparison and the golden file."""
    rng = np.random.default_rng(4242 + n_coef)
    cases = []
    for r in range(0, n_coef // 2):
        for _ in range(6):
            V = int(rng.integers(2, 10))
            m, v = random_vertices(rng, n_coef, V)
            cases.append((r, m, v, rng.uniform(0.3, 5.0, V - 1)))
    return cases


def ref_outputs(lib, n_coef, case):
    r, mask, vals, times = case
    V, H = len(mask), n_coef // 2
    coef = np.zeros((V - 1, 4, n_coef))
    cost = C.c_double()
    dims = np.zeros(2, np.int32)
    dpv = np.zeros(4 * H * V)
    rc = lib.ref_solve_linear(V, _p(np.ascontiguousarray(mask), u8p), _p(np.ascontiguousarray(vals)), _p(np.ascontiguousarray(times)), int(r),
                              _p(coef), C.byref(cost), _p(dpv), _p(dims, ip))
    assert rc == 0
    return coef, cost.value


@pytest.mark.parametrize("n_coef", [6, 8, 12])
def test_restatement_equals_reference_templates(n_coef):
    """PolynomialOptimization<N>::setupFromVertices / solveLinear / computeCost of the reference, instantiated for N, vs oracle/."""
    if not O.REFERENCE:
        pytest.skip("needs a checkout of the original ctu-mrs/mrs_uav_trajectory_generation (TG_REFERENCE_DIR or BASELINE.json reference_path)")
    O.build_oracle(ref=True)
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", f"libref_eth_n{n_coef}.so"))
    orc = O.OracleN(n_coef, mode=O.MATH_LIBM)
    try:
        for case in reference_cases(n_coef):
            c_r, cost_r = ref_outputs(lib, n_coef, case)
            c_o, cost_o = orc.solve_linear(case[1], case[2], case[3], case[0])
            assert np.array_equal(c_r, c_o) and cost_r == cost_o, (n_coef, case[0])
    finally:
        orc.lib.orc_set_math_mode(O.MATH_DET)


@pytest.mark.parametrize("n_coef", [6, 8, 12])
def test_restatement_equals_reference_golden(n_coef):
    """The same comparison against the committed outputs of the reference build (tests/golden/gen_golden_general.py)."""
    g = np.load(GOLDEN)
    orc = O.OracleN(n_coef, mode=O.MATH_LIBM)
    try:
        for i, case in enumerate(reference_cases(n_coef)):
            c_o, cost_o = orc.solve_linear(case[1], case[2], case[3], case[0])
            assert np.array_equal(g[f"n{n_coef}_coef_{i}"], c_o) and g[f"n{n_coef}_cost_{i}"] == cost_o, (n_coef, i)
    finally:
        orc.lib.orc_set_math_mode(O.MATH_DET)
