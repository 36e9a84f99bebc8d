"""The C++ host side (include/eth_trajectory_generation_b200.hpp, the reference's class names over the C ABI): a C++
program written like MrsTrajectoryGeneration::findTrajectory (tests/cpp/test_shim.cpp) is compiled, linked against the
C-ABI library and its results compared bit for bit with the oracle.  CPU runs link the host emulation of the device
code; the GPU run links libtg_b200.so."""
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from mrs_uav_trajectory_generation_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run_shim(libdir, libname, tmp_path, source="test_shim.cpp", extra=()):
    exe = str(tmp_path / source.replace(".cpp", ""))
    out = str(tmp_path / source.replace(".cpp", ".txt"))
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-pthread", *extra, "-o", exe, os.path.join(ROOT, "tests", "cpp", source),
                           "-L" + libdir, "-l" + libname, "-Wl,-rpath," + libdir])
    subprocess.check_call([exe, out])
    res = {}
    for line in open(out):
        f = line.split()
        res.setdefault(f[0], []).append(np.array([float.fromhex(x) for x in f[2:]]))
    return res


def _check(res):
    wps = W.F1B_WAYPOINTS
    V, r = len(wps), 2
    mask = np.ones(V, np.uint8)
    mask[0] = mask[-1] = 0b111
    vals = np.zeros((V, O.HALF, O.D))
    vals[:, 0] = wps
    times = np.array([1.0 + 0.25 * (i % 3) for i in range(V - 1)])
    # PolynomialOptimization<10>
    coef, cost, _, _ = O.solve_linear(mask, vals, times, r)
    assert np.array_equal(res["lin_times"][0], times)
    assert np.array_equal(res["lin_coef"][0].reshape(V - 1, 4, 10), coef)
    assert res["lin_cost"][0][0] == cost
    tq = [0.0, 2.6, float(np.add.accumulate(times)[-1]) * 0.75]
    for k, t in enumerate(tq):
        assert np.array_equal(res["lin_eval_p"][k], O.trajectory_evaluate(coef, times, t, 0)[0])
        assert np.array_equal(res["lin_eval_v"][k], O.trajectory_evaluate(coef, times, t, 1)[0])
    assert res["lin_bad_setup"][0][0] == 0.0  # wrong number of segment times: setupFromVertices returns false
    # PolynomialOptimizationNonLinear<10> + sampleWholeTrajectory
    ref = O.time_alloc(mask, vals, times, r)
    code, evals, passes, fcost = res["nl_meta"][0]
    assert (int(code), int(evals), int(passes)) == (ref["nlopt_code"], ref["n_evals"], ref["n_scale_passes"]) and fcost == ref["final_cost"]
    assert np.array_equal(res["nl_times"][0], ref["times"])
    assert np.array_equal(res["nl_coef"][0].reshape(V - 1, 4, 10), ref["coef"])
    full, t_ns = O.sample(ref["coef"], ref["times"], 0.2)  # [M][19] = p4 v4 a4 j3 s3 yaw
    got = res["nl_samples"][0].reshape(-1, 7)
    assert got.shape[0] == full.shape[0]
    assert np.array_equal(got[:, :3], full[:, :3]) and np.array_equal(got[:, 3], full[:, 18])
    assert np.array_equal(got[:, 4], full[:, 4]) and np.array_equal(got[:, 5], full[:, 10])
    assert np.array_equal(got[:, 6].astype(np.int64), t_ns)
    mx = O.segment_maxima(ref["coef"], ref["times"])
    assert np.array_equal(res["nl_max_h"][0], mx[:, 0:3].max(axis=0))
    for k in (1, 2, 3):
        t, v, i = O.max_magnitude(ref["coef"], ref["times"], k)
        assert np.array_equal(res["nl_maxmag"][k - 1], [t, v, float(i)])
    # evaluateObjectives: objectiveFunctionTime (kSquaredTime) with two soft constraints at three candidate time vectors
    xs = np.stack([times, times * 1.25, times * 0.8])
    rt, rp = O.objective(mask, vals, r, 0, xs, 500.0, True, 100.0, [1, 2], [4.0, 2.0])
    assert np.array_equal(res["obj_total"][0], rt) and np.array_equal(res["obj_parts"][0].reshape(3, 3), rp)
    # TrajectoryGeneratorBatch: optimize() over two paths
    for p, path in enumerate([W.F1B_WAYPOINTS, W.F1A_WAYPOINTS]):
        o = O.optimize_path(path)
        meta = res["batch_meta"][p]
        assert (int(meta[0]), int(meta[1]), int(meta[2]), int(meta[3]), int(meta[4]), int(meta[5])) == \
            (o["res"].success, o["res"].rounds, o["res"].n_waypoints, o["res"].n_samples, o["res"].nlopt_code, o["res"].safe)
        assert np.array_equal(res["batch_times"][p], o["times"])
        assert np.array_equal(res["batch_coef"][p].reshape(-1, 4, 10), o["coeffs"])
        assert np.array_equal(res["batch_samples"][p].reshape(-1, 4), o["samples"])


def _check_requests(res):
    """optimizeRequests: the resolved limits follow node.cpp:972-1040 / 1847-1881 and each request's samples equal the oracle's at them."""
    p1 = np.array([[10, 20, 3.5, 1.2], [-5, -5, 5, 1], [-5, 5, 5, 2], [5, -5, 5, 3], [5, 5, 5, 4]], float)
    FM = float(np.finfo(np.float32).max)
    base = [4.0, 2.0, 3.0, 1.5, 30.0, 20.0, 1.0, 2.0, 10.0]
    over = [6.0, 3.0, 3.5, 2.5, 35.0, 35.0, 1.0, 2.0, 10.0]
    want = [(base[:6] + [FM] * 3, 0.4, 1, 0, 6, 0), (over, 0.05, 1, 1, 5, 1), (base, 0.05, 1, 0, 5, 0)]
    for q in range(3):
        m = res["req_meta"][q]
        L, dev, prepend, overridden, V, stop = want[q]
        assert list(m[:9]) == L and m[9] == dev and (m[10], m[11], m[12], m[13]) == (prepend, overridden, V, stop)
        wp = p1 + np.array([q, 0, 0, 0.0])
        if q == 0:
            wp = np.vstack([wp, wp[:1]])
        vel = (7.0 if q == 2 else 0.4, -0.3, 0.1, 0.0)
        ref = O.optimize_batch(np.array([0, len(wp)], np.int32), wp, stop_at=np.full(len(wp), stop, np.uint8), init=np.asarray([W.init14(1.2, vel=vel)]),
                               params=O.default_params(limits=L, max_deviation=dev), cap_wp=400, cap_samples=4000)
        r = ref["res"][0]
        assert (int(m[14]), int(m[15]), int(m[16]), int(m[17])) == (r.success, r.rounds, r.n_waypoints, r.n_samples)
        assert np.array_equal(res["req_samples"][q].reshape(-1, 4), ref["samples"][0, : r.n_samples])


def _check_side_steps(res):
    raw = W.F1B_WAYPOINTS.copy()
    raw = np.insert(raw, 3, raw[2] + np.array([0.01, 0, 0, 0]), axis=0)
    stop = np.zeros(len(raw), np.uint8)
    stop[6] = 1
    pw, ps = O.preprocess_path(raw, stop)
    got = res["pre"][0].reshape(-1, 5)
    assert np.array_equal(got[:, :4], pw) and np.array_equal(got[:, 4].astype(np.uint8), ps) and len(pw) == len(raw) - 1
    lim = np.array(O.DEFAULT_LIMITS) * np.array([0.75, 0.75, 0.75, 0.75, 1, 1, 1, 1, 1])
    fb = O.fallback_sample(pw, ps, lim, 0.2, 2.0)
    assert np.array_equal(res["fallback"][0].reshape(-1, 4), fb)
    assert np.array_equal(res["idxs"][0].astype(np.int32), O.waypoint_idxs(fb, pw))


def _eigen_flags():
    # the Eigen stand-in (test infrastructure: the tests do not need Eigen) and, where a checkout of the reference is present
    # (oracle_lib.reference_dir()), its own eth_mav_msgs/eigen_mav_msgs.h for the EigenTrajectoryPoint type
    flags = ["-I" + os.path.join(ROOT, "oracle", "ref_shim")]
    if O.REFERENCE and os.path.isdir(os.path.join(O.REFERENCE, "include")):
        flags.append("-I" + os.path.join(O.REFERENCE, "include"))
    return flags


def _check_eigen(res, ctx):
    """tests/cpp/test_shim_eigen.cpp: reference-typed call sites (Eigen::Vector4d in, Eigen::VectorXd / EigenTrajectoryPoint out),
    evaluateRange, optimize() of the derivative-free methods, two contexts side by side."""
    import mrs_uav_trajectory_generation_b200.api as A

    n_wp, r = 7, 2
    wp = np.array([[1.5 * i, 0.4 if i % 2 == 0 else -0.6, 4.0 + 0.1 * i, 0.2 * i] for i in range(n_wp)])
    mask = np.ones(n_wp, np.uint8)
    mask[0], mask[-1] = 0b1111, 0b111
    vals = np.zeros((n_wp, O.HALF, O.D))
    vals[:, 0] = wp
    vals[0, 1], vals[0, 2] = (0.3, -0.1, 0.05, 0.02), (0.0, 0.1, 0.0, 0.0)
    times = np.array([0.9 + 0.2 * (i % 3) for i in range(n_wp - 1)])
    assert np.array_equal(res["vtx0_vel"][0], vals[0, 1])
    ref = O.time_alloc(mask, vals, times, r)
    code, evals, cost = res["nl_meta"][0]
    assert (int(code), int(evals)) == (ref["nlopt_code"], ref["n_evals"]) and cost == ref["final_cost"]
    assert np.array_equal(res["nl_times"][0], ref["times"]) and np.array_equal(res["nl_coef"][0].reshape(-1, 4, 10), ref["coef"])
    tq = 0.37 * float(np.add.accumulate(ref["times"])[-1])  # getMaxTime(): accumulated in segment order
    tot = 0.0
    for t in ref["times"]:
        tot += t
    tq = 0.37 * tot
    assert np.array_equal(res["eval_p"][0], O.trajectory_evaluate(ref["coef"], ref["times"], tq, 0)[0])
    assert np.array_equal(res["eval_s"][0], O.trajectory_evaluate(ref["coef"], ref["times"], tq, 4)[0])
    full, t_ns = O.sample(ref["coef"], ref["times"], 0.2)
    got = res["samples"][0].reshape(-1, 8)
    assert got.shape[0] == full.shape[0]
    assert np.array_equal(got[:, :3], full[:, :3]) and np.array_equal(got[:, 5], full[:, 7]) and np.array_equal(got[:, 6], full[:, 16])
    assert np.array_equal(got[:, 7].astype(np.int64), t_ns)
    # the quaternion is built on the host by the (stand-in) Eigen from the raw heading: w = cos(yaw / 2), z = sin(yaw / 2)
    assert np.allclose(got[:, 3], np.cos(0.5 * full[:, 3]), rtol=0, atol=2e-16) and np.allclose(got[:, 4], np.sin(0.5 * full[:, 3]), rtol=0, atol=2e-16)
    # evaluateRange(t_start inside segment 1, dt 0.3, jerk): the reference's walk (eth/trajectory.cpp:93-151) restated here
    T = ref["times"]
    t_start, t_end, dt = T[0] + 0.05, tot, 0.3
    acc, i = 0.0, 0
    for i in range(len(T)):
        acc += T[i]
        if acc > t_start:
            break
    acc -= T[i]
    in_seg = t_start - acc
    want, want_t = [], []
    while acc < t_end:
        if in_seg > T[i]:
            in_seg = in_seg - T[i]
            i += 1
            if i >= len(T):
                break
            continue
        want.append(O.trajectory_evaluate(ref["coef"][i:i + 1], T[i:i + 1], in_seg, 3)[0])
        want_t.append(acc)
        in_seg += dt
        acc += dt
    assert np.array_equal(res["range_t"][0], np.array(want_t)) and np.array_equal(res["range_jerk"][0].reshape(-1, 4), np.array(want))
    # optimize() of the derivative-free methods == the Python mirror of the same search over the same batched objective
    verts = []
    for v in range(n_wp):
        vx = A.Vertex(4)
        for k in range(5):
            if (mask[v] >> k) & 1:
                vx.addConstraint(k, vals[v, k].copy())
        verts.append(vx)
    for key, method, iters, cons in (("df", 0, 6, [(0, 1, 4.0), (0, 2, 2.0)]), ("df4", 4, 3, [(0, 1, 4.0), (2, 2, 1.0)])):
        P = A.NonlinearOptimizationParameters()
        P.time_alloc_method, P.max_iterations = method, iters
        opt = A.PolynomialOptimizationNonLinear(4, P, ctx=ctx)
        assert opt.setupFromVertices(verts, times, r)
        for c in cons:
            opt.addMaximumMagnitudeConstraint(*c)
        pcode = opt.optimize()
        m = res[key + "_meta"][0]
        assert (int(m[0]), int(m[1])) == (pcode, opt._dfo.n_iterations), (key, m, pcode, opt._dfo.n_iterations)
        assert np.array_equal(res[key + "_times"][0], opt._dfo.times) and np.array_equal(res[key + "_coef"][0].reshape(-1, 4, 10), opt._dfo.coef)
        assert np.array_equal(m[2:5], opt._dfo.cost_parts)
    assert res["r1_refused"][0][0] == 1.0 and res["multi_ctx_same"][0][0] == 1.0
    c1, cost1 = O.OracleN(10).solve_linear(mask, vals, times, 1)  # derivative_to_optimize = 1 through the general-shape kernels
    assert np.array_equal(res["r1_coef_cost"][0][:-1].reshape(-1, 4, 10), c1) and res["r1_coef_cost"][0][-1] == cost1


def _check_general(res):
    """tests/cpp/test_shim_general.cpp: PolynomialOptimization<8>(3), <12>(4), <6>(1), <10>(3) against the oracle compiled for that N."""
    def wp(i, dims):
        return np.array([1.7 * i, 0.6 if i % 2 == 0 else -0.4, 3.0 + 0.25 * i, 0.15 * i])[:dims]

    for key, n_coef, dims, r in (("n8d3", 8, 3, 3), ("n12d4", 12, 4, 4), ("n6d1", 6, 1, 2), ("n10d3", 10, 3, 2)):
        H, V = n_coef // 2, 6
        orc = O.OracleN(n_coef)
        mask = np.ones(V, np.uint8)
        mask[0] = mask[-1] = (1 << (r + 1)) - 1
        mask[2] |= 2
        vals = np.zeros((V, H, 4))
        for i in range(V):
            vals[i, 0, :dims] = wp(i, dims)
        vals[2, 1, :dims] = 0.3
        times = np.array([0.8 + 0.3 * (i % 3) for i in range(V - 1)])
        coef, cost = orc.solve_linear(mask, vals, times, r)
        assert np.array_equal(res[key + "_coef"][0].reshape(V - 1, dims, n_coef), coef[:, :dims]), key
        assert res[key + "_cost"][0][0] == cost, key
        tot = 0.0
        for t in times:
            tot += t
        k = 0
        for tq in (0.0, 1.3, tot * 0.8):
            for deriv in (0, 1, 2):
                assert np.array_equal(res[key + "_eval"][k], orc.trajectory_evaluate(coef, times, tq, deriv)[0][:dims]), (key, tq, deriv)
                k += 1
        # evaluateRange(0.4, max, 0.35, velocity): the reference's walk (eth/trajectory.cpp:93-151)
        acc, i = 0.0, 0
        for i in range(len(times)):
            acc += times[i]
            if acc > 0.4:
                break
        acc -= times[i]
        tin, want = 0.4 - acc, []
        while acc < tot:
            if tin > times[i]:
                tin = tin - times[i]
                i += 1
                if i >= len(times):
                    break
                continue
            want.append(orc.trajectory_evaluate(coef[i:i + 1], times[i:i + 1], tin, 1)[0][:dims])
            tin += 0.35
            acc += 0.35
        assert np.array_equal(res[key + "_range"][0].reshape(-1, dims), np.array(want)), key
        if dims >= 3:
            full = orc.sample(coef, times, 0.2)
            got = res[key + "_samples"][0].reshape(-1, 3, 3)
            assert got.shape[0] == full.shape[0]
            assert np.array_equal(got[:, :, 0], full[:, 0:3]) and np.array_equal(got[:, :, 1], full[:, 4:7]) and np.array_equal(got[:, :, 2], full[:, 15:18])
        else:
            assert res[key + "_samples"][0].size == 0
    # N = 10 on three dimensions: maxima / magnitude / time scaling equal the four-dimensional run with a zero heading
    V = 5
    mask = np.ones(V, np.uint8)
    mask[0] = mask[-1] = 0b111
    vals = np.zeros((V, 5, 4))
    for i in range(V):
        vals[i, 0, :3] = wp(i, 3)
    times = np.full(V - 1, 0.7)
    coef, _, _, _ = O.solve_linear(mask, vals, times, 2)
    mx = O.segment_maxima(coef, times)
    assert np.array_equal(res["n10d3_max"][0], np.concatenate([mx[:, 0:3].max(axis=0), mx[:, 3:6].max(axis=0)]))
    t, v, i = O.max_magnitude(coef, times, 1)
    assert np.array_equal(res["n10d3_maxmag"][0], [t, v, float(i)])
    c2, t2, passes, within = O.scale_times(coef, times)
    assert np.array_equal(res["n10d3_scaled_times"][0][:-1], t2) and res["n10d3_scaled_times"][0][-1] == float(within)
    assert np.array_equal(res["n10d3_scaled_coef"][0].reshape(-1, 3, 10), c2[:, :3])
    assert res["d5_refused"][0][0] == 1.0 and res["n8_scale_refused"][0][0] == 0.0
    # PolynomialOptimizationNonLinear<10>(3), Mellinger: the four-dimensional run with a zero heading, limits as set in the C++ test
    big = 3.40282346638528859812e+38
    P = O.default_params(limits=(4.0, 2.0, 2.0, 1.0, big, big, big, big, big))
    ref = O.time_alloc(mask, vals, times, 2, P)
    assert np.array_equal(res["nl3_times_code"][0][:-1], ref["times"]) and int(res["nl3_times_code"][0][-1]) == ref["nlopt_code"]
    assert np.array_equal(res["nl3_coef"][0].reshape(-1, 3, 10), ref["coef"][:, :3]) and np.all(ref["coef"][:, 3] == 0.0)
    assert res["nl3_dfo_refused"][0][0] == 1.0


def test_cpp_shim_general_shapes_on_host_emulation(oracle, emu_lib, tmp_path):
    _check_general(_run_shim(os.path.join(ROOT, "tests", "host_emu"), "tg_emu", tmp_path, "test_shim_general.cpp"))


@pytest.mark.gpu
def test_cpp_shim_general_shapes_on_gpu(oracle, gpu_ctx, tmp_path):
    _check_general(_run_shim(os.path.join(ROOT, "mrs_uav_trajectory_generation_b200"), "tg_b200", tmp_path, "test_shim_general.cpp"))


def test_cpp_shim_eigen_types_on_host_emulation(oracle, emu_lib, emu_ctx, tmp_path):
    res = _run_shim(os.path.join(ROOT, "tests", "host_emu"), "tg_emu", tmp_path, "test_shim_eigen.cpp", _eigen_flags())
    _check_eigen(res, emu_ctx)


@pytest.mark.gpu
def test_cpp_shim_eigen_types_on_gpu(oracle, gpu_ctx, tmp_path):
    res = _run_shim(os.path.join(ROOT, "mrs_uav_trajectory_generation_b200"), "tg_b200", tmp_path, "test_shim_eigen.cpp", _eigen_flags())
    _check_eigen(res, gpu_ctx)


def test_cpp_shim_on_host_emulation(oracle, emu_lib, tmp_path):
    res = _run_shim(os.path.join(ROOT, "tests", "host_emu"), "tg_emu", tmp_path)
    _check(res)
    _check_side_steps(res)
    _check_requests(res)


@pytest.mark.gpu
def test_cpp_shim_on_gpu(oracle, gpu_ctx, tmp_path):
    res = _run_shim(os.path.join(ROOT, "mrs_uav_trajectory_generation_b200"), "tg_b200", tmp_path)
    _check(res)
    _check_side_steps(res)
    _check_requests(res)
