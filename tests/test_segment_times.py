"""Initial segment times on the device: tg_estimate_segment_times_batch (csrc/tg_kernels.cuh EstimateTimesFn over the pipeline's own
segment_time_euclidean / segment_time_baca), the Python functions over it and the C++ estimateSegmentTimes / estimateSegmentTimesBaca /
estimateSegmentTimesBatch of the drop-in header.

Checked bit for bit on the host emulation of the device code and, with -m gpu, on the GPU:
  * against the oracle (deterministic math mode) on 4096 random-flier paths, a ragged batch of V = 1 ... 40 vertices (V = 1 and 2 in the
    middle), the edge cases of test_ref_eth.py::test_segment_time_estimates (vertical and zero-length segments, heading-dominated
    segments, FLT_MAX heading limits), headings across +-pi and non-finite inputs; on the GPU also 2^20 paths, every one compared;
  * against tg_optimize_batch (run_time_alloc = 0, no deviation check): its segment times and tg_result.baca_total;
  * against the reference's own outputs (tests/golden/ref_eth.npz) and, where a checkout of the reference is present, its code live;
  * every refusal (TG_ERR_INVALID, outputs untouched), in C, Python and C++;
  * the C++ call sites of findTrajectory (tests/cpp/test_shim_segment_times.cpp).
"""
import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as O
import mrs_uav_trajectory_generation_b200.api as A
from mrs_uav_trajectory_generation_b200 import TgError
from mrs_uav_trajectory_generation_b200 import workloads as W
from test_cpp_shim import _eigen_flags, _run_shim

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
TG_ERR_INVALID = -3
dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
FLT_MAX = 3.4028234663852886e38
LIMITS = np.array(O.DEFAULT_LIMITS, dtype=np.float64)                                    # 9 entries: the oracle reads the ninth
RELAXED = np.array((4.0, 2.0, 2.0, 1.0, 20.0, 20.0, FLT_MAX, FLT_MAX, FLT_MAX))           # relax_heading: FLT_MAX heading limits


def _p(a, t=dp):
    return None if a is None else a.ctypes.data_as(t)


_BATCH_ORACLE = []


def batch_oracle():
    """tests/cpp/oracle_estimate_times.cpp linked against the oracle library: orc_estimate_times over a ragged batch on host threads"""
    if not _BATCH_ORACLE:
        O.build_oracle(ref=False)
        O.set_math_mode(O.MATH_DET)
        so = os.path.join(tempfile.mkdtemp(prefix="oracle_estimate_times"), "liboracle_estimate_times.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-shared", "-o", so,
                               os.path.join(HERE, "cpp", "oracle_estimate_times.cpp"), "-L" + O.ORACLE_DIR, "-loracle", "-Wl,-rpath," + O.ORACLE_DIR])
        _BATCH_ORACLE.append(C.CDLL(so))
    return _BATCH_ORACLE[0]


def oracle_times(vtx_off, pos4, lim9, nthreads=os.cpu_count()):
    vtx_off = np.ascontiguousarray(vtx_off, dtype=np.int32)
    pos4 = np.ascontiguousarray(pos4, dtype=np.float64)
    lim9 = np.ascontiguousarray(lim9, dtype=np.float64)
    B = len(vtx_off) - 1
    e, b = np.empty(int(vtx_off[-1]) - B), np.empty(int(vtx_off[-1]) - B)
    batch_oracle().orc_estimate_times_batch(B, _p(vtx_off, ip), _p(pos4), _p(lim9), _p(e), _p(b), int(nthreads or 1))
    return e, b


def ragged(lists):
    vtx_off = np.concatenate([[0], np.cumsum([len(l) for l in lists])]).astype(np.int32)
    return vtx_off, np.concatenate(lists).reshape(-1, 4)


def same(a, b):
    return np.array_equal(a, b, equal_nan=True)


def check_lists(ctx, lists, lim9):
    """one device call over the lists == the oracle list by list, both outputs; either output alone gives the same bits"""
    vtx_off, pos4 = ragged(lists)
    e, b = ctx.estimate_segment_times_batch(vtx_off, pos4, lim9[:8])
    so = vtx_off - np.arange(len(vtx_off))
    for p, wp in enumerate(lists):
        oe, ob = O.estimate_times(wp, lim9)
        assert same(e[so[p]:so[p + 1]], oe) and same(b[so[p]:so[p + 1]], ob), p
    assert same(ctx.estimate_segment_times_batch(vtx_off, pos4, lim9[:8], baca=False)[0], e)
    assert same(ctx.estimate_segment_times_batch(vtx_off, pos4, lim9[:8], euclidean=False)[1], b)


def edge_lists():
    """the cases of test_ref_eth.py::test_segment_time_estimates, headings across +-pi, and non-finite positions"""
    rng = np.random.default_rng(3)
    out = [np.array([[0, 0, 0, 0], [0, 0, 5, 0], [0, 0, 5, 3.0], [0, 0, 5, 3.0], [4, 0, 1, -3.0]], float),  # vertical, zero length, heading
           np.cumsum(rng.uniform(-3, 3, (9, 4)), axis=0)]
    pi = math.pi
    h = [3.1, -3.1, pi, -pi, 3.0, -2.9, 0.0, pi - 1e-15, -pi + 1e-15, 2.5, -2.5, 6.0, -6.0, pi]
    out.append(np.column_stack([np.arange(len(h)) * 0.7, np.zeros(len(h)), np.full(len(h), 5.0), h]))
    out.append(np.column_stack([np.zeros(6), np.zeros(6), np.full(6, 5.0), [3.0, -3.0, 3.0, -3.0, 0.1, 0.1]]))  # heading only
    nf = W.random_flier_path(9, 6)
    nf[2, 0], nf[4, 3] = np.nan, np.inf
    out.append(nf)
    return out


def check_parity(ctx):
    wp_off, wp = W.random_flier_paths(4096, 11)
    e, b = ctx.estimate_segment_times_batch(wp_off, wp, LIMITS[:8])
    oe, ob = oracle_times(wp_off, wp, LIMITS)
    assert np.array_equal(e, oe) and np.array_equal(b, ob)
    Vs = list(range(3, 41))
    Vs[18:18] = [1, 2]
    rng = np.random.default_rng(11)
    lists = [W.random_flier_path(100 + i, V) if i % 2 else np.cumsum(rng.uniform(-2, 2, (V, 4)), axis=0) for i, V in enumerate(Vs)]
    for lim in (LIMITS, RELAXED):
        check_lists(ctx, lists, lim)
        check_lists(ctx, edge_lists(), lim)
    inf_lim = LIMITS.copy()
    inf_lim[[1, 6]] = np.inf
    check_lists(ctx, edge_lists()[:3], inf_lim)


def test_parity_emu(oracle, emu_ctx):
    if emu_ctx.solve_kernels != "by-size":
        pytest.skip("the estimates do not depend on the solve dispatch")
    check_parity(emu_ctx)


@pytest.mark.gpu
def test_parity_gpu(oracle, gpu_ctx):
    if gpu_ctx.solve_kernels != "by-size":
        pytest.skip("the estimates do not depend on the solve dispatch")
    check_parity(gpu_ctx)


@pytest.mark.gpu
def test_million_paths_gpu(oracle, gpu_ctx):
    """2^20 paths of 11 waypoints in one call, every path compared with the oracle (in chunks); single paths alone == inside the batch"""
    if gpu_ctx.solve_kernels != "by-size":
        pytest.skip("the estimates do not depend on the solve dispatch")
    B, V = 1 << 20, 11
    wp_off, wp = W.random_flier_paths_fast(B, V)
    e, b = gpu_ctx.estimate_segment_times_batch(wp_off, wp, LIMITS[:8])
    chunk = 1 << 16
    for p0 in range(0, B, chunk):
        off = wp_off[p0:p0 + chunk + 1] - wp_off[p0]
        oe, ob = oracle_times(off, wp[wp_off[p0]:wp_off[p0 + chunk]], LIMITS)
        s0 = p0 * (V - 1)
        assert np.array_equal(e[s0:s0 + len(oe)], oe) and np.array_equal(b[s0:s0 + len(ob)], ob), p0
    for p in (0, 1, 777, B // 2, B - 1):
        se, sb = gpu_ctx.estimate_segment_times_batch([0, V], wp[p * V:(p + 1) * V], LIMITS[:8])
        assert np.array_equal(se, e[p * (V - 1):(p + 1) * (V - 1)]) and np.array_equal(sb, b[p * (V - 1):(p + 1) * (V - 1)]), p


def recipe_positions(wp):
    """the vertex positions of the node's recipe without an initial state (build_vertices, node.cpp:931-977): each heading unwrapped from
    the one before, h_0 = wp_0, h_i = h_{i-1} + rad_diff(wp_i, h_{i-1})"""
    pos = np.array(wp, dtype=np.float64, copy=True)
    last = float(wp[0, 3])
    for i in range(len(wp)):
        d = float(wp[i, 3]) - last
        if d < -math.pi:
            d = d + 2.0 * math.pi
        elif d >= math.pi:
            d = d - 2.0 * math.pi
        last = last + d
        pos[i, 3] = last
    return pos


def check_pipeline(ctx, B):
    """tg_optimize_batch without time allocation starts from the same estimates: its times and tg_result.baca_total"""
    wp_off, wp = W.random_flier_paths(B, 11, first_index=5000)
    wp = wp.copy()
    wp[::7, 3] += 2.0 * math.pi * np.where(np.arange(0, len(wp), 7) % 2, 1.0, -1.0)  # raw headings outside [-pi, pi)
    P = ctx.L.default_params(run_time_alloc=0, check_deviation=0)
    res, _ = ctx.optimize_batch(wp_off, wp, params=P)
    out = ctx.fetch_outputs(want=("seg_off", "times"))
    pos = np.concatenate([recipe_positions(wp[wp_off[p]:wp_off[p + 1]]) for p in range(B)])
    e, b = ctx.estimate_segment_times_batch(wp_off, pos, LIMITS[:8])
    so = wp_off - np.arange(B + 1)
    accepted = 0
    for p in range(B):
        tot = 0.0
        for x in b[so[p]:so[p + 1]]:
            tot = tot + float(x)
        assert res["baca_total"][p] == tot, p
        if res["status"][p] == 0:
            accepted += 1
            assert np.array_equal(out["times"][out["seg_off"][p]:out["seg_off"][p + 1]], e[so[p]:so[p + 1]]), p
    assert accepted > B // 2


def test_pipeline_agreement_emu(oracle, emu_ctx):
    check_pipeline(emu_ctx, 512)


@pytest.mark.gpu
def test_pipeline_agreement_gpu(oracle, gpu_ctx):
    check_pipeline(gpu_ctx, 4096)


def check_golden(ctx):
    """the reference's own estimateSegmentTimes / estimateSegmentTimesBaca outputs stored in ref_eth.npz"""
    z = np.load(os.path.join(HERE, "golden", "ref_eth.npz"))
    for q in range(int(z["n"])):
        wp = z[f"wp_{q}"]
        e, b = ctx.estimate_segment_times_batch([0, len(wp)], wp, z["limits"][:8])
        assert np.array_equal(e, z[f"euclid_{q}"]) and np.array_equal(b, z[f"baca_{q}"]), q


def test_reference_outputs_emu(oracle, emu_ctx):
    check_golden(emu_ctx)


@pytest.mark.gpu
def test_reference_outputs_gpu(oracle, gpu_ctx):
    check_golden(gpu_ctx)


def test_reference_live(oracle, emu_lib):
    """where a checkout of the reference is present: its own functions (oracle/_ref ref_estimate_times) on the parity inputs"""
    if not O.REFERENCE:
        pytest.skip("needs a checkout of the original ctu-mrs/mrs_uav_trajectory_generation (TG_REFERENCE_DIR or BASELINE.json reference_path)")
    from mrs_uav_trajectory_generation_b200 import Context

    O.build_oracle(ref=True)
    ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_eth.so"))
    emu_ctx = Context(emu_lib, 0)
    lists = [W.random_flier_path(i, 11) for i in range(64)] + edge_lists()[:4]
    for lim in (LIMITS, RELAXED):
        for wp in lists:
            wp = np.ascontiguousarray(wp, dtype=np.float64)
            e2, b2 = np.zeros(len(wp) - 1), np.zeros(len(wp) - 1)
            ref.ref_estimate_times(len(wp), _p(wp), _p(lim), _p(e2), _p(b2))
            e, b = emu_ctx.estimate_segment_times_batch([0, len(wp)], wp, lim[:8])
            assert np.array_equal(e, e2) and np.array_equal(b, b2)


def check_refusals(ctx):
    lib = ctx.L.lib
    wp = np.ascontiguousarray(W.random_flier_path(5, 6))
    pos = np.ascontiguousarray(np.concatenate([wp, wp]))
    lim = np.ascontiguousarray(LIMITS[:8])

    def call(B, off, pos4, limits, want_e=True, want_b=True):
        e, b = np.full(16, -7.25), np.full(16, -7.25)
        rc = lib.tg_estimate_segment_times_batch(ctx.h, B, _p(off, ip), _p(pos4), _p(limits), _p(e) if want_e else None, _p(b) if want_b else None)
        return rc, bool(np.all(e == -7.25) and np.all(b == -7.25))

    good = np.array([0, 6, 12], np.int32)
    for args in ((0, good, pos, lim), (-1, good, pos, lim), (2, None, pos, lim), (2, good, None, lim), (2, good, pos, None),
                 (2, good, pos, lim, False, False), (2, np.array([1, 6, 12], np.int32), pos, lim), (2, np.array([0, 0, 12], np.int32), pos, lim),
                 (2, np.array([0, 6, 6], np.int32), pos, lim), (3, np.array([0, 6, 6, 12], np.int32), pos, lim),
                 (2, np.array([0, 8, 6], np.int32), pos, lim)):
        rc, untouched = call(*args)
        assert rc == TG_ERR_INVALID and untouched, args[:2]
    rc, untouched = call(2, np.array([0, 1, 2], np.int32), pos, lim)  # lists of one vertex: valid, no segment, nothing written
    assert rc == 0 and untouched
    assert call(2, good, pos, lim)[0] == 0
    with pytest.raises(TgError):
        ctx.estimate_segment_times_batch([0, 6, 6], wp, lim)
    with pytest.raises(TgError):
        ctx.estimate_segment_times_batch([0, 6], wp, lim, euclidean=False, baca=False)
    with pytest.raises(ValueError):
        ctx.estimate_segment_times_batch([0, 6], wp, LIMITS)  # nine limits
    with pytest.raises(TgError):
        A.estimate_segment_times([], lim, ctx=ctx)
    v3 = A.Vertex(3)
    v3.addConstraint(0, [0.0, 1.0, 2.0])
    with pytest.raises(ValueError):
        A.estimate_segment_times([v3, v3], lim, ctx=ctx)
    v4 = A.Vertex(4)
    v4.addConstraint(1, [0.0, 1.0, 2.0, 0.0])
    with pytest.raises(ValueError):
        A.estimate_segment_times_baca([v4, v4], lim, ctx=ctx)


def test_refusals_emu(emu_ctx):
    check_refusals(emu_ctx)


@pytest.mark.gpu
def test_refusals_gpu(gpu_ctx):
    check_refusals(gpu_ctx)


def check_python_api(ctx):
    lists = [W.random_flier_path(30 + i, V) for i, V in enumerate((11, 1, 2, 5))]
    vertex_lists = []
    for wp in lists:
        vl = []
        for i, w in enumerate(wp):
            v = A.Vertex(4)
            if i in (0, len(wp) - 1):
                v.makeStartOrEnd(w, 2)
            else:
                v.addConstraint(A.derivative_order.POSITION, w)
            vl.append(v)
        vertex_lists.append(vl)
    es, bs = A.estimate_segment_times_batch(vertex_lists, LIMITS[:8], ctx=ctx)
    for wp, vl, e, b in zip(lists, vertex_lists, es, bs):
        oe, ob = O.estimate_times(wp)
        assert np.array_equal(e, oe) and np.array_equal(b, ob)
        assert np.array_equal(A.estimate_segment_times(vl, LIMITS[:8], ctx=ctx), oe)
        assert np.array_equal(A.estimate_segment_times_euclidean(vl, LIMITS[:8], ctx=ctx), oe)
        assert np.array_equal(A.estimate_segment_times_baca(vl, LIMITS[:8], ctx=ctx), ob)


def test_python_api_emu(emu_ctx):
    check_python_api(emu_ctx)


@pytest.mark.gpu
def test_python_api_gpu(gpu_ctx):
    check_python_api(gpu_ctx)


def test_symbol_declared_and_exported(emu_lib):
    import test_abi

    assert "tg_estimate_segment_times_batch" in test_abi._declared_symbols()
    assert hasattr(emu_lib.lib, "tg_estimate_segment_times_batch")


# ---- C++ (tests/cpp/test_shim_segment_times.cpp) ------------------------------------------------------------------------------
CPP_WP = np.array([[0.0, 0.0, 3.0, 3.0], [2.0, 0.5, 4.0, -3.0], [4.0, -0.5, 5.0, 2.9], [4.0, -0.5, 7.5, -3.1], [6.0, 0.5, 5.0, 0.5],
                   [8.0, -0.5, 5.0, 3.1], [10.0, 0.5, 5.0, -2.0]])


def _check_cpp(res):
    pos = recipe_positions(CPP_WP)
    e, b = O.estimate_times(pos)
    assert np.array_equal(res["times"][0], e) and np.array_equal(res["baca"][0], b) and np.array_equal(res["euclidean"][0], e)
    tot = 0.0
    for x in b:
        tot += float(x)
    assert res["baca_sum"][0][0] == tot
    V, r = len(pos), 2
    mask = np.ones(V, np.uint8)
    mask[0] = mask[-1] = (1 << (r + 1)) - 1
    vals = np.zeros((V, O.HALF, O.D))
    vals[:, 0] = pos
    a = O.time_alloc(mask, vals, e, r)
    assert (int(res["nl_meta"][0][0]), int(res["nl_meta"][0][1])) == (a["nlopt_code"], a["n_evals"])
    assert np.array_equal(res["nl_times"][0], a["times"]) and np.array_equal(res["nl_coef"][0].reshape(-1, 4, 10), a["coef"])
    assert list(res["batch_ok"][0]) == [1.0, 1.0]
    for i, n in enumerate((V, 1, 2)):
        oe, ob = O.estimate_times(pos[:n])
        assert np.array_equal(res["batch_e"][i], oe) and np.array_equal(res["batch_b"][i], ob) and np.array_equal(res["batch_b_only"][i], ob)
    assert list(res["refused"][0]) == [1.0] * 5


def test_cpp_segment_times_on_host_emulation(oracle, emu_lib, tmp_path):
    _check_cpp(_run_shim(os.path.join(ROOT, "tests", "host_emu"), "tg_emu", tmp_path, "test_shim_segment_times.cpp", _eigen_flags()))


@pytest.mark.gpu
def test_cpp_segment_times_on_gpu(oracle, gpu_ctx, tmp_path):
    _check_cpp(_run_shim(os.path.join(ROOT, "mrs_uav_trajectory_generation_b200"), "tg_b200", tmp_path, "test_shim_segment_times.cpp", _eigen_flags()))
