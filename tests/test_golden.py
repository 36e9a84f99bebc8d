"""Pins of the oracle (not gpu) and of the product against the committed golden fixtures (tests/golden/, made by
tests/golden/gen_golden.py in the build container):
  * rpoly_reference.npz -- zeros computed by the REFERENCE's own rpoly_ak1.cpp (compiled unmodified): the oracle's
    Jenkins-Traub restatement must reproduce them bit for bit with the reference's libm, and with the deterministic
    math layer that the GPU kernels share (include/tg_detmath.h) as well;
  * pipeline_oracle.npz -- the oracle's full-pipeline outputs: a regression pin for the restatement and the golden
    input/output pairs of the GPU tests (the reference cannot be run on the GPU box either)."""
import os

import numpy as np
import pytest

import oracle_lib as O
import parity_checks as PC

HERE = os.path.dirname(os.path.abspath(__file__))
G = os.path.join(HERE, "golden")


def _rpoly_cases():
    z = np.load(os.path.join(G, "rpoly_reference.npz"))
    for i in range(len(z["n_coeffs"])):
        yield z["coeffs"][i, : z["n_coeffs"][i]], z["re"][i, : z["n_roots"][i]], z["im"][i, : z["n_roots"][i]], bool(z["ok"][i])


def test_oracle_rpoly_matches_reference_vectors(oracle):
    """Bit-exact in both math modes: the detmath log/exp agree with glibc on every argument the 600 cases produce, or
    perturb nothing that reaches a zero."""
    try:
        for mode in (O.MATH_LIBM, O.MATH_DET):
            O.set_math_mode(mode)
            bad = 0
            for c, re, im, ok in _rpoly_cases():
                r2, i2, ok2 = O.find_roots(c)
                if not (ok2 == ok and np.array_equal(r2, re) and np.array_equal(i2, im)):
                    bad += 1
            assert bad == 0, (mode, bad)
    finally:
        O.set_math_mode(O.MATH_DET)


def test_oracle_rpoly_matches_live_reference_build(oracle):
    """Where a checkout of the reference is present, the comparison also runs live against oracle/_ref on 300 more polynomials."""
    if O.ref_lib() is None:
        pytest.skip("needs a checkout of the original project (TG_REFERENCE_DIR or BASELINE.json reference_path); "
                    "the 600 stored cases of rpoly_reference.npz are compared instead")
    rng = np.random.default_rng(5)
    O.set_math_mode(O.MATH_LIBM)
    try:
        for _ in range(300):
            n = int(rng.integers(2, 17))
            c = rng.standard_normal(n) * np.exp(rng.uniform(-3, 3, n))
            a, b = O.find_roots(c), O.find_roots(c, use_ref=True)
            assert a[2] == b[2] and np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    finally:
        O.set_math_mode(O.MATH_DET)


def _ref_eth_cases():
    z = np.load(os.path.join(G, "ref_eth.npz"))
    for q in range(int(z["n"])):
        yield q, {k[: -len(f"_{q}")]: z[k] for k in z.files if k.endswith(f"_{q}")}, z["limits"]


def test_oracle_matches_reference_class_vectors(oracle):
    """ref_eth.npz holds outputs of the REFERENCE's own classes (compiled unmodified, oracle/_ref/libref_eth.so); the
    restatement reproduces every one bit for bit in glibc math mode: segment-time estimates, linear solve + cost, per-segment
    maxima, time scaling, sampling (count, time_from_start_ns, all 19 fields), Mellinger time allocation."""
    O.set_math_mode(O.MATH_LIBM)
    try:
        for q, g, L in _ref_eth_cases():
            r = int(g["r"])
            e, b = O.estimate_times(g["wp"], L)
            assert np.array_equal(e, g["euclid"]) and np.array_equal(b, g["baca"]), q
            c, cost, _, _ = O.solve_linear(g["mask"], g["vals"], e, r)
            assert np.array_equal(c, g["coef"]) and cost == float(g["cost"]), q
            assert np.array_equal(O.segment_maxima(c, e), g["maxima"]), q
            sc, st, _, within = O.scale_times(c, e, L)
            assert np.array_equal(sc, g["scaled_coef"]) and np.array_equal(st, g["scaled_times"]) and int(within) == int(g["within"]), q
            smp, tns = O.sample(sc, st, 0.2)
            assert np.array_equal(tns, g["tns"]) and np.array_equal(smp, g["samples"]), q
            a = O.time_alloc(g["mask"], g["vals"], e, r, O.default_params(derivative_to_optimize=r))
            assert [a["nlopt_code"], a["n_evals"]] == list(g["alloc_meta"]) and a["final_cost"] == float(g["alloc_cost"]), q
            assert np.array_equal(a["times"], g["alloc_times"]) and np.array_equal(a["coef"], g["alloc_coef"]), q
    finally:
        O.set_math_mode(O.MATH_DET)


def _pipeline_cases():
    z = np.load(os.path.join(G, "pipeline_oracle.npz"))
    for p in range(int(z["n"])):
        init = z[f"init_{p}"]
        yield p, z[f"wp_in_{p}"], (init if init.size else None), {k: z[f"{k}_{p}"] for k in ("wp", "times", "coef", "samples", "meta")}


def test_oracle_pipeline_regression(oracle):
    for p, wp, init, g in _pipeline_cases():
        r = O.optimize_path(wp, init=init)
        res = r["res"]
        meta = np.array([res.success, res.rounds, res.safe, res.n_waypoints, res.n_samples, res.nlopt_code, res.n_evals, res.n_scale_passes])
        assert np.array_equal(meta, g["meta"]), p
        for k, kk in (("wp", "wp"), ("times", "times"), ("coeffs", "coef"), ("samples", "samples")):
            assert np.array_equal(r[k], g[kk]), (p, k)


def _product_vs_golden(ctx):
    cases = list(_pipeline_cases())
    for with_init in (True, False):
        sel = [c for c in cases if (c[2] is not None) == with_init]
        wp_off = np.cumsum([0] + [len(c[1]) for c in sel]).astype(np.int32)
        wp = np.concatenate([c[1] for c in sel])
        init = np.stack([c[2] for c in sel]) if with_init else None
        res, _ = ctx.optimize_batch(wp_off, wp, None, init, ctx.L.default_params())
        out = ctx.fetch_outputs()
        for q, (p, _, _, g) in enumerate(sel):
            s0, s1 = out["seg_off"][q], out["seg_off"][q + 1]
            m0, m1 = out["smp_off"][q], out["smp_off"][q + 1]
            meta = np.array([res["success"][q], res["rounds"][q], res["safe"][q], res["n_waypoints"][q], res["n_samples"][q], res["nlopt_code"][q],
                             res["n_evals"][q], res["n_scale_passes"][q]])
            assert np.array_equal(meta, g["meta"]), p  # verdicts, subdivision and sample counts: exact
            assert np.array_equal(out["wp"][s0 + q: s1 + q + 1], g["wp"]), p
            # north_star tolerances: coefficients 1e-9 relative, samples 1e-6 m (the kernels are in fact bit-exact)
            assert PC.coef_rel_err(out["coef"][s0:s1], g["coef"], g["times"]) <= 1e-9
            assert np.abs(out["samples"][m0:m1] - g["samples"]).max() <= 1e-6
            assert np.array_equal(out["times"][s0:s1], g["times"]) and np.array_equal(out["coef"][s0:s1], g["coef"])
            assert np.array_equal(out["samples"][m0:m1], g["samples"])


def test_emulated_kernels_match_golden_pipeline(emu_ctx):
    _product_vs_golden(emu_ctx)


@pytest.mark.gpu
def test_gpu_matches_golden_pipeline(gpu_ctx):
    _product_vs_golden(gpu_ctx)
