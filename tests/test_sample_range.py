"""Sampling and evaluation over a time window: tg_sample_range_batch_nd / tg_evaluate_range_batch_nd (csrc/tg_generic.cuh RangeWalkFn,
gen::SampleEvalFn, gen::EvaluateRangeFn) and the Python functions over them.

Checked bit for bit against the restatement's windowed walk (tests/cpp/oracle_sample_range.cpp over the oracle built for each N; over
[0, end] it equals the oracle's own sampleWholeTrajectory),
on the host emulation of the device code and, with -m gpu, on the GPU:
  * every N in {6, 8, 10, 12}; sampling on D in {3, 4}, evaluateRange on D = 1..4 and derivatives 0 .. N+1; ragged batches
    (S = 1 .. 12) of trajectories from tg_solve_linear_batch_nd;
  * windows starting at 0, on a segment boundary, mid-segment, at the end, past the end, below 0; ending past the end, at +inf,
    before the start; dt longer than the trajectory; NaN ends; and a 10^6-sample window;
  * [0, end] against tg_sample_batch_nd and, at N = 10, D = 4, tg_sample_batch; a window alone against the same window inside
    a batch of 4096;
  * the capacity bound, TG_ERR_CAPACITY, and every refusal (TG_ERR_INVALID, outputs untouched);
  * the reference's own sampleTrajectoryInRange / evaluateRange (tests/cpp/ref_sample_range.cpp over oracle/_ref) where a checkout
    of the reference is present.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as O
from test_general_shape import random_batch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
TG_ERR_INVALID, TG_ERR_CAPACITY = -3, -5
dp, ip, llp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_longlong)


def _p(a, t=dp):
    return None if a is None else a.ctypes.data_as(t)


def trajectories(ctx, n_coef, dims, B, seed):
    """B solved trajectories of S = 1 .. 12 segments: seg_off, coef [totS][dims][N], times."""
    rng = np.random.default_rng(seed)
    vtx_off, masks, vals, times = random_batch(rng, n_coef, B, dims)
    vv = np.concatenate(vals)[:, :, :dims]
    t = np.concatenate(times)
    coef, _ = ctx.solve_linear_batch_nd(n_coef, dims, vtx_off, np.concatenate(masks), vv, t, 2)
    seg_off = (vtx_off - np.arange(B + 1)).astype(np.int32)
    return seg_off, coef, t


def end_of(times):
    tot = 0.0
    for x in times:
        tot += float(x)
    return tot


def windows_for(times, rng):
    """(t_start, t_end, dt) edge cases of one trajectory."""
    tot = end_of(times)
    b1 = float(times[0])  # the boundary between segments 0 and 1 as the walk accumulates it
    mid = 0.5 * b1
    w = [(0.0, tot, 0.05), (b1, tot, 0.07), (mid, tot, 0.03), (mid, 0.6 * tot, 0.11), (tot, tot, 0.05), (tot, tot + 5.0, 0.05),
         (tot + 1.0, tot + 2.0, 0.05), (-0.3, 0.5 * tot, 0.05), (mid, tot + 3.0, 0.05), (mid, np.inf, 0.04), (0.0, np.inf, 0.2),
         (0.7 * tot, 0.2 * tot, 0.01), (mid, mid, 0.1), (0.0, tot, 2.0 * tot + 1.0), (mid, tot, 3.0 * tot),
         (np.nan, tot, 0.1), (0.0, np.nan, 0.1), (-np.inf, 0.5 * tot, 0.1)]
    for _ in range(4):
        a = float(rng.uniform(-0.2, 1.1) * tot)
        w.append((a, a + float(rng.uniform(-0.1, 1.0) * tot), float(rng.uniform(0.005, 0.3))))
    return w


def pad4(coef, dims, n_coef):
    c4 = np.zeros((coef.shape[0], 4, n_coef))
    c4[:, :dims] = coef
    return c4


_RANGE_ORACLES = {}


def range_oracle(n_coef):
    """tests/cpp/oracle_sample_range.cpp built against the oracle library for N = n_coef (which OracleN builds, loads and sets to the
    deterministic math mode): orc_sample_range / orc_evaluate_range"""
    if n_coef not in _RANGE_ORACLES:
        O.OracleN(n_coef)
        d = tempfile.mkdtemp(prefix="oracle_sample_range")
        so = os.path.join(d, f"liboracle_sample_range_n{n_coef}.so")
        lib = "oracle" if n_coef == 10 else f"oracle_n{n_coef}"
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", f"-DORC_N={n_coef}", "-o", so,
                               os.path.join(HERE, "cpp", "oracle_sample_range.cpp"), "-L" + O.ORACLE_DIR, "-l" + lib, "-Wl,-rpath," + O.ORACLE_DIR])
        _RANGE_ORACLES[n_coef] = C.CDLL(so)
    return _RANGE_ORACLES[n_coef]


def oracle_sample(orc, coef4, times, t0, t1, dt):
    cap = 4096
    while True:
        out, tns = np.zeros((cap, 19)), np.zeros(cap, np.int64)
        n = orc.orc_sample_range(len(times), _p(coef4), _p(times), C.c_double(t0), C.c_double(t1), C.c_double(dt), cap, _p(out),
                                     tns.ctypes.data_as(C.POINTER(C.c_int64)))
        if n >= 0:
            return out[:n], tns[:n]
        cap = -n


def oracle_evaluate(orc, coef4, times, t0, t1, dt, deriv):
    cap = 4096
    while True:
        out, st = np.zeros((cap, 4)), np.zeros(cap)
        n = orc.orc_evaluate_range(len(times), _p(coef4), _p(times), C.c_double(t0), C.c_double(t1), C.c_double(dt), int(deriv), cap,
                                       _p(out), _p(st))
        if n >= 0:
            return out[:n], st[:n]
        cap = -n


def same(a, b):
    """bit for bit, NaN matching NaN (a window starting at -inf evaluates segment 0 at -inf)"""
    return np.array_equal(a, b, equal_nan=True)


def split(counts, *arrays):
    off = np.concatenate([[0], np.cumsum(counts)])
    return [[a[off[i]:off[i + 1]] for i in range(len(counts))] for a in arrays]


def check_sample_parity(ctx, n_coef, dims, seed):
    orc = range_oracle(n_coef)
    rng = np.random.default_rng(seed)
    seg_off, coef, times = trajectories(ctx, n_coef, dims, 12, seed)
    for dt_group in range(2):  # one call per dt: the device takes one dt per call
        wins, sel = [], []
        for p in range(12):
            T = times[seg_off[p]:seg_off[p + 1]]
            for (a, b, dt) in windows_for(T, rng):
                wins.append((p, a, b, dt))
        dts = sorted({w[3] for w in wins})
        for dt in dts[dt_group::2]:
            sel = [w for w in wins if w[3] == dt]
            idx = [w[0] for w in sel]
            so = np.concatenate([[0], np.cumsum([seg_off[p + 1] - seg_off[p] for p in idx])]).astype(np.int32)
            cf = np.concatenate([coef[seg_off[p]:seg_off[p + 1]] for p in idx])
            tm = np.concatenate([times[seg_off[p]:seg_off[p + 1]] for p in idx])
            rng_ = np.array([(w[1], w[2]) for w in sel])
            counts, samples, full, t_ns = ctx.sample_range_batch_nd(n_coef, dims, so, cf, tm, rng_, dt, full=True)
            fs, ss, ts = split(counts, full, samples, t_ns)
            for k, (p, a, b, _) in enumerate(sel):
                T = times[seg_off[p]:seg_off[p + 1]]
                want, want_ns = oracle_sample(orc, pad4(coef[seg_off[p]:seg_off[p + 1]], dims, n_coef), T, a, b, dt)
                assert counts[k] == len(want), (n_coef, dims, a, b, dt)
                assert same(fs[k], want), (n_coef, dims, a, b, dt)
                assert same(ss[k][:, :3], want[:, :3]) and same(ss[k][:, 3], want[:, 18])
                assert same(ts[k], want_ns)


def check_evaluate_parity(ctx, n_coef, dims, seed):
    orc = range_oracle(n_coef)
    rng = np.random.default_rng(seed + 1)
    seg_off, coef, times = trajectories(ctx, n_coef, dims, 10, seed)
    for deriv in range(n_coef + 2):
        dt = float(rng.uniform(0.02, 0.2))
        B = len(seg_off) - 1
        wins = []
        for p in range(B):
            T = times[seg_off[p]:seg_off[p + 1]]
            ws = windows_for(T, rng)
            a, b, _ = ws[int(rng.integers(len(ws)))]
            wins.append((a, b))
        counts, vals, st = ctx.evaluate_range_batch_nd(n_coef, dims, seg_off, coef, times, np.array(wins), dt, deriv)
        vs, sts = split(counts, vals, st)
        for p in range(B):
            T = times[seg_off[p]:seg_off[p + 1]]
            want, want_t = oracle_evaluate(orc, pad4(coef[seg_off[p]:seg_off[p + 1]], dims, n_coef), T, wins[p][0], wins[p][1], dt, deriv)
            assert counts[p] == len(want), (n_coef, dims, deriv, wins[p])
            assert same(vs[p], want[:, :dims]) and same(sts[p], want_t), (n_coef, dims, deriv, wins[p])
            if deriv >= n_coef:
                assert not vs[p].any()


@pytest.mark.parametrize("n_coef", [6, 8, 10, 12])
def test_range_oracle_whole_window_is_the_oracle_sampler(oracle, n_coef):
    """The windowed restatement over [0, end] gives the oracle's own sampleWholeTrajectory rows (orc_sample), t_ns included at N = 10."""
    rng = np.random.default_rng(n_coef)
    for S in (1, 3, 12):
        coef = rng.normal(size=(S, 4, n_coef))
        times = rng.uniform(0.2, 2.0, S)
        for dt in (0.05, 0.2, 0.37):
            got, got_ns = oracle_sample(range_oracle(n_coef), coef, times, 0.0, end_of(times), dt)
            assert same(got, O.OracleN(n_coef).sample(coef, times, dt)), (n_coef, S, dt)
            if n_coef == 10:
                want, want_ns = O.sample(coef, times, dt)
                assert same(got, want) and same(got_ns, want_ns)


@pytest.mark.parametrize("n_coef", [6, 8, 10, 12])
@pytest.mark.parametrize("dims", [3, 4])
def test_sample_range_parity_emu(emu_ctx, n_coef, dims):
    check_sample_parity(emu_ctx, n_coef, dims, 10 * n_coef + dims)


@pytest.mark.parametrize("n_coef", [6, 8, 10, 12])
@pytest.mark.parametrize("dims", [1, 2, 3, 4])
def test_evaluate_range_parity_emu(emu_ctx, n_coef, dims):
    check_evaluate_parity(emu_ctx, n_coef, dims, 20 * n_coef + dims)


def check_whole_and_batch(ctx, n_coef, dims):
    seg_off, coef, times = trajectories(ctx, n_coef, dims, 12, 7 * n_coef + dims)
    B = len(seg_off) - 1
    whole = np.array([(0.0, end_of(times[seg_off[p]:seg_off[p + 1]])) for p in range(B)])
    counts, samples, full, t_ns = ctx.sample_range_batch_nd(n_coef, dims, seg_off, coef, times, whole, 0.2, full=True)
    c2, s2, f2 = ctx.sample_batch_nd(n_coef, dims, seg_off, coef, times, 0.2, full=True)
    assert same(counts, c2) and same(samples, s2) and same(full, f2)
    want_ns = np.concatenate([(0.0 + 0.2 * np.arange(c, dtype=np.float64)) * 1e9 for c in counts]).astype(np.int64)
    assert same(t_ns, want_ns)
    if (n_coef, dims) == (10, 4):
        c3, s3, f3 = ctx.sample_batch(seg_off, coef, times, 0.2, full=True)
        assert same(counts, c3) and same(samples, s3) and same(full, f3)
    # one window alone == the same window inside a batch of 4096
    rng = np.random.default_rng(3)
    pick = rng.integers(0, B, 4096)
    so = np.concatenate([[0], np.cumsum([seg_off[p + 1] - seg_off[p] for p in pick])]).astype(np.int32)
    cf = np.concatenate([coef[seg_off[p]:seg_off[p + 1]] for p in pick])
    tm = np.concatenate([times[seg_off[p]:seg_off[p + 1]] for p in pick])
    w = np.array([(rng.uniform(-0.5, 1.0) * whole[p, 1], rng.uniform(0.0, 1.2) * whole[p, 1]) for p in pick])
    cb, sb, fb, tb = ctx.sample_range_batch_nd(n_coef, dims, so, cf, tm, w, 0.05, full=True)
    fbs, tbs = split(cb, fb, tb)
    for k in list(range(0, 4096, 97)) + [4095]:
        p = pick[k]
        c1, _, f1, t1 = ctx.sample_range_batch_nd(n_coef, dims, np.array([0, seg_off[p + 1] - seg_off[p]], np.int32), coef[seg_off[p]:seg_off[p + 1]],
                                                  times[seg_off[p]:seg_off[p + 1]], w[k:k + 1], 0.05, full=True)
        assert c1[0] == cb[k] and same(f1, fbs[k]) and same(t1, tbs[k])


@pytest.mark.parametrize("shape", [(6, 3), (8, 4), (10, 4), (12, 3)])
def test_whole_window_and_batch_independence_emu(emu_ctx, shape):
    check_whole_and_batch(emu_ctx, *shape)


def check_million(ctx, orc10):
    """a 10^6-sample window: dt = 1e-5 over 10 s"""
    seg_off, coef, times = trajectories(ctx, 10, 4, 1, 5)
    times = times * (10.0 / end_of(times))
    counts, samples, full, t_ns = ctx.sample_range_batch_nd(10, 4, seg_off, coef, times, [(0.0, 10.0)], 1e-5, full=True)
    want, want_ns = oracle_sample(orc10, coef, times, 0.0, 10.0, 1e-5)
    assert counts[0] == len(want) and counts[0] >= 10 ** 6 - 2
    assert same(full, want) and same(t_ns, want_ns)


def test_million_samples_emu(emu_ctx):
    if emu_ctx.solve_kernels != "by-size":
        pytest.skip("the walk does not depend on the solve dispatch")
    check_million(emu_ctx, range_oracle(10))


def raw_sample(ctx, N, D, seg_off, coef, times, t_range, dt, counts, samples=None, full=None, t_ns=None):
    return ctx.L.lib.tg_sample_range_batch_nd(ctx.h, N, D, len(seg_off) - 1, _p(seg_off, ip), _p(coef), _p(times), _p(t_range), C.c_double(dt),
                                              _p(counts, ip), _p(samples), _p(full), _p(t_ns, llp))


def raw_evaluate(ctx, N, D, seg_off, coef, times, t_range, dt, deriv, counts, out=None, st=None):
    return ctx.L.lib.tg_evaluate_range_batch_nd(ctx.h, N, D, len(seg_off) - 1, _p(seg_off, ip), _p(coef), _p(times), _p(t_range), C.c_double(dt),
                                                int(deriv), _p(counts, ip), _p(out), _p(st))


def check_refusals(ctx):
    seg_off = np.array([0, 2], np.int32)
    times = np.array([1.0, 1.5])
    t_range = np.array([0.2, 2.0])
    for N, D, sample_ok in ((10, 4, True), (8, 3, True), (6, 2, False), (12, 1, False)):
        coef = np.ones((2, D, N)) * 0.1
        cnt, s4, f19, tns = np.full(1, -7, np.int32), np.full((64, 4), 7.0), np.full((64, 19), 7.0), np.full(64, 7, np.int64)
        out, st = np.full((64, D), 7.0), np.full(64, 7.0)

        def untouched():
            return (cnt == -7).all() and (s4 == 7.0).all() and (f19 == 7.0).all() and (tns == 7).all() and (out == 7.0).all() and (st == 7.0).all()

        rc = raw_sample(ctx, N, D, seg_off, coef, times, t_range, 0.1, cnt, s4, f19, tns)
        assert (rc == 0) == sample_ok and (rc == 0 or (rc == TG_ERR_INVALID and untouched())), (N, D, rc)
        cnt[:] = -7
        s4[:], f19[:], tns[:] = 7.0, 7.0, 7
        assert raw_evaluate(ctx, N, D, seg_off, coef, times, t_range, 0.1, 1, cnt, out, st) == 0
        cnt[:] = -7
        out[:], st[:] = 7.0, 7.0
        bad = [dict(N=7), dict(N=14), dict(D=0), dict(D=5), dict(dt=0.0), dict(dt=-0.1), dict(dt=np.nan), dict(seg_off=np.array([0, 2, 1], np.int32)),
               dict(seg_off=np.array([1, 2], np.int32)), dict(t_range=None), dict(times=None), dict(coef=None)]
        for kw in bad:
            a = dict(N=N, D=D, seg_off=seg_off, coef=coef, times=times, t_range=t_range, dt=0.1)
            a.update(kw)
            if "seg_off" in kw and kw["seg_off"][0] == 0:
                a["t_range"] = np.array([0.2, 2.0, 0.2, 2.0])
            rc = raw_sample(ctx, a["N"], a["D"], a["seg_off"], a["coef"], a["times"], a["t_range"], a["dt"], cnt, s4, f19, tns)
            assert rc == TG_ERR_INVALID and untouched(), kw
            rc = raw_evaluate(ctx, a["N"], a["D"], a["seg_off"], a["coef"], a["times"], a["t_range"], a["dt"], 0, cnt, out, st)
            assert rc == TG_ERR_INVALID and untouched(), kw
        assert raw_evaluate(ctx, N, D, seg_off, coef, times, t_range, 0.1, -1, cnt, out, st) == TG_ERR_INVALID and untouched()
        assert raw_sample(ctx, N, D, seg_off, coef, times, t_range, 0.1, None, s4, f19, tns) == TG_ERR_INVALID and untouched()
        assert ctx.L.lib.tg_sample_range_batch_nd(ctx.h, N, D, 0, _p(seg_off, ip), _p(coef), _p(times), _p(t_range), C.c_double(0.1), _p(cnt, ip),
                                                  None, None, None) == TG_ERR_INVALID and untouched()


def test_refusals_emu(emu_ctx):
    check_refusals(emu_ctx)


def check_capacity(ctx):
    """A window no int bounds fails with TG_ERR_CAPACITY and writes nothing; the bound itself holds on every window above."""
    seg_off = np.array([0, 2], np.int32)
    coef, times = np.ones((2, 4, 10)) * 0.1, np.array([1.0, 1.5])
    cnt = np.full(1, -7, np.int32)
    for win, dt in (((-np.inf, np.inf), 0.1), ((0.0, 2.5), 1e-12), ((-1e300, 1.0), 1e-300)):
        rc = raw_sample(ctx, 10, 4, seg_off, coef, times, np.array(win), dt, cnt)
        assert rc == TG_ERR_CAPACITY and cnt[0] == -7, (win, dt, rc)
        assert raw_evaluate(ctx, 10, 4, seg_off, coef, times, np.array(win), dt, 0, cnt) == TG_ERR_CAPACITY and cnt[0] == -7
    # the walk's own sample count stays within the bound min(t_end - segment start, end - t_start) / dt + 4 on windows that are
    # exactly at it: a window [0, end] at dt = end / k samples k or k + 1 times
    for k in (1, 3, 10, 1000):
        win = np.array([0.0, 2.5])
        assert raw_sample(ctx, 10, 4, seg_off, coef, times, win, 2.5 / k, cnt) == 0 and k <= cnt[0] <= k + 1


def test_capacity_emu(emu_ctx):
    check_capacity(emu_ctx)


def check_python_api(ctx):
    import mrs_uav_trajectory_generation_b200 as tg
    import mrs_uav_trajectory_generation_b200.api as A

    seg_off, coef, times = trajectories(ctx, 8, 3, 3, 11)
    trajs = [A.Trajectory(coef[seg_off[p]:seg_off[p + 1]], times[seg_off[p]:seg_off[p + 1]], ctx) for p in range(3)]
    orc = range_oracle(8)
    t = trajs[1]
    tot = t.getMaxTime()
    s = tg.sample_trajectory_in_range(t, 0.25 * tot, 0.75 * tot, 0.05, full=True)
    want, _ = oracle_sample(orc, pad4(t.coef, 3, 8), t.times, 0.25 * tot, 0.75 * tot, 0.05)
    assert same(s, want)
    assert same(tg.sample_trajectory_start_duration(t, 0.25 * tot, 0.5 * tot, 0.05, full=True),
                          tg.sample_trajectory_in_range(t, 0.25 * tot, 0.25 * tot + 0.5 * tot, 0.05, full=True))
    assert tg.sample_trajectory_in_range(t, -0.1, tot, 0.05) is None and tg.sample_trajectory_in_range(t, 0.0, tot + 0.1, 0.05) is None
    assert same(tg.sample_trajectory_in_range(t, 0.0, tot, 0.2), tg.sample_whole_trajectory(t, 0.2))
    wins = [(0.1, 1e9), (0.5 * trajs[1].getMaxTime(), np.inf), (0.0, 0.3)]
    counts, rows, t_ns = tg.sample_trajectories_in_range(trajs, wins, 0.07, full=True)
    parts = split(counts, rows)[0]
    for p in range(3):
        want, want_ns = oracle_sample(orc, pad4(trajs[p].coef, 3, 8), trajs[p].times, wins[p][0], wins[p][1], 0.07)
        assert same(parts[p], want)
    v, st = t.evaluateRange(0.3 * tot, tot, 0.09, 2)
    wv, wt = oracle_evaluate(orc, pad4(t.coef, 3, 8), t.times, 0.3 * tot, tot, 0.09, 2)
    assert same(v, wv[:, :3]) and same(st, wt)


def test_python_api_emu(emu_ctx):
    check_python_api(emu_ctx)


# ---- the reference's own sampleTrajectoryInRange / evaluateRange --------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref():
    if not O.REFERENCE:
        pytest.skip("needs a checkout of the original ctu-mrs/mrs_uav_trajectory_generation (TG_REFERENCE_DIR or BASELINE.json reference_path)")
    O.build_oracle(ref=True)
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    so = os.path.join(tempfile.mkdtemp(prefix="ref_sample_range"), "libref_sample_range.so")
    subprocess.check_call(["g++", "-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-w", "-shared", "-I", os.path.join(ROOT, "oracle", "ref_shim"),
                           "-I", os.path.join(O.REFERENCE, "include"), "-o", so, os.path.join(HERE, "cpp", "ref_sample_range.cpp"), "-L" + ref_dir,
                           "-lref_eth", "-Wl,-rpath," + ref_dir])
    lib = C.CDLL(so)
    O.set_math_mode(O.MATH_LIBM)
    yield lib
    O.set_math_mode(O.MATH_DET)


def test_reference_pin(ref, emu_lib):
    """ref_sample_range / ref_evaluate_range (the reference's code) == the restatement on the windows of §4.3, edges included;
    sampleTrajectoryInRange refuses windows outside [getMinTime(), getMaxTime()]."""
    from mrs_uav_trajectory_generation_b200 import Context

    ctx = Context(emu_lib, 0)
    seg_off, coef, times = trajectories(ctx, 10, 4, 6, 99)
    rng = np.random.default_rng(4)
    for p in range(6):
        c4, T = coef[seg_off[p]:seg_off[p + 1]], times[seg_off[p]:seg_off[p + 1]]
        tot = end_of(T)
        for (a, b, dt) in windows_for(T, rng):
            if np.isnan(a) or np.isnan(b) or np.isinf(a):
                continue
            out, tns, ok = np.zeros((20000, 19)), np.zeros(20000, np.int64), C.c_int()
            n = ref.ref_sample_range(len(T), _p(c4), _p(T), C.c_double(a), C.c_double(b), C.c_double(dt), 20000, _p(out),
                                     tns.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(ok))
            inside = a >= 0.0 and b <= tot
            assert bool(ok.value) == inside, (a, b)
            if inside:
                want, want_ns = oracle_sample(range_oracle(10), c4, T, a, b, dt)
                assert n == len(want) and same(out[:n], want) and same(tns[:n], want_ns), (a, b, dt)
            for deriv in (0, 3, 11):
                v, st = np.zeros((20000, 4)), np.zeros(20000)
                n = ref.ref_evaluate_range(len(T), _p(c4), _p(T), C.c_double(a), C.c_double(b), C.c_double(dt), deriv, 20000, _p(v), _p(st))
                wv, wt = oracle_evaluate(range_oracle(10), c4, T, a, b, dt, deriv)
                assert n == len(wv) and same(v[:n], wv) and same(st[:n], wt), (a, b, dt, deriv)


# ---- on the GPU ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_coef", [6, 8, 10, 12])
def test_sample_range_parity_gpu(gpu_ctx, n_coef):
    for dims in (3, 4):
        check_sample_parity(gpu_ctx, n_coef, dims, 10 * n_coef + dims)
        check_evaluate_parity(gpu_ctx, n_coef, dims, 20 * n_coef + dims)
    for dims in (1, 2):
        check_evaluate_parity(gpu_ctx, n_coef, dims, 20 * n_coef + dims)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(6, 3), (8, 4), (10, 4), (12, 3)])
def test_whole_window_and_batch_independence_gpu(gpu_ctx, shape):
    check_whole_and_batch(gpu_ctx, *shape)


@pytest.mark.gpu
def test_million_refusals_capacity_api_gpu(gpu_ctx):
    check_million(gpu_ctx, range_oracle(10))
    check_refusals(gpu_ctx)
    check_capacity(gpu_ctx)
    check_python_api(gpu_ctx)


# ---- the C++ header -------------------------------------------------------------------------------------------------------------------------
def _check_cpp(res):
    """tests/cpp/test_shim_sample_range.cpp against the oracle: states = t_ns, p3 v3 a3 j3 s3, yaw rate, yaw acceleration."""
    def states(full, t_ns, dims):
        yaw = full[:, [7, 11]] if dims == 4 else np.zeros((len(full), 2))
        return np.column_stack([t_ns.astype(np.float64), full[:, 0:3], full[:, 4:7], full[:, 8:11], full[:, 12:15], full[:, 15:18], yaw])

    shapes = [(10, 4), (10, 4), (8, 3)]
    tr = []
    for i, (n_coef, dims) in enumerate(shapes):
        times = res["times%d" % i][0]
        coef = res["coef%d" % i][0].reshape(len(times), dims, n_coef)
        orc = range_oracle(n_coef)
        c4, end, mid = pad4(coef, dims, n_coef), end_of(times), 0.5 * times[0]
        tr.append((orc, c4, times, end))
        for key, (a, b, dt) in (("in_range", (mid, 0.7 * end, 0.05)), ("start_duration", (mid, mid + 0.3 * end, 0.07)),
                                ("whole_range", (0.0, end, 0.2)), ("whole", (0.0, end, 0.2))):
            full, t_ns = oracle_sample(orc, c4, times, a, b, dt)
            assert same(res["%s%d" % (key, i)][0].reshape(-1, 18), states(full, t_ns, dims)), (key, i)
        assert list(res["ok%d" % i][0]) == [1, 1, 1, 1, 0, 0], i
        v, st = oracle_evaluate(orc, c4, times, mid, end + 1.0, 0.09, 2)
        assert same(res["range%d" % i][0].reshape(-1, dims), v[:, :dims]) and same(res["range_t%d" % i][0], st), i
    assert res["batch_ok"][0][0] == 1.0 and res["mixed_ok"][0][0] == 0.0
    for i, (a, b) in enumerate([(0.3, 1e9), (0.5 * tr[1][3], 2.0 * tr[1][3])]):
        orc, c4, times, _ = tr[i]
        full, t_ns = oracle_sample(orc, c4, times, a, b, 0.04)
        assert len(full) > 0 and same(res["batch%d" % i][0].reshape(-1, 18), states(full, t_ns, 4)), i


def _cpp(libdir, libname, tmp_path, eigen):
    import test_cpp_shim as S

    extra = ["-DTG_TEST_EIGEN_POINT"] + S._eigen_flags() if eigen else ["-DTG_B200_NO_EIGEN"]
    return S._run_shim(libdir, libname, tmp_path, "test_shim_sample_range.cpp", extra)


@pytest.mark.parametrize("eigen", [False, True])
def test_cpp_sample_range_on_host_emulation(oracle, emu_lib, tmp_path, eigen):
    _check_cpp(_cpp(os.path.join(ROOT, "tests", "host_emu"), "tg_emu", tmp_path, eigen))


@pytest.mark.gpu
@pytest.mark.parametrize("eigen", [False, True])
def test_cpp_sample_range_on_gpu(oracle, gpu_ctx, tmp_path, eigen):
    _check_cpp(_cpp(os.path.join(ROOT, "mrs_uav_trajectory_generation_b200"), "tg_b200", tmp_path, eigen))
