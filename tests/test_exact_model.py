"""The general-shape kernels against an exact model of the problem (tests/exact_model.py), not against the restatement.

Every other kernel test here asks whether the device code gives the bits of oracle/.  A mistake both share (a falling-factorial
factor, a power of 1/s, the cost convention, a candidate filter) passes those.  These tests compare tg_*_nd -- on the host
emulation of the device code and on the GPU -- with an mpmath model written from the mathematics, at N in {6, 8, 10, 12}, D in
1..4 and every r in 0 .. N/2-1, on ragged batches (S = 1 .. 12) with normal (0.3 .. 5 s) and extreme (0.01 s next to 20 s)
segment times and positions of 1 km and of 6 cm.

Every tolerance is gamma * U * (a condition or magnitude quantity the model computes), gamma a small constant named below; the
worst observed ratio |error| / (U * quantity) per (N, r, check) is printed and recorded with record_property.
"""
import math

import numpy as np
import pytest

import exact_model as EM
from exact_model import U
from test_general_shape import random_vertices

# ---- the constants of the tolerances (multiples of U * the model's quantity) ------------------------------------------------------
G_GRAD = 4.0    # exact reduced gradient H x + g at the kernel's free derivatives vs E |x| + E_pf |d_f| (exact_model.reduced_gradient)
G_SOLVE = 4.0   # free derivatives of the solve vs their componentwise condition xb (exact_model.solve)
G_COEF = 16.0   # coefficients of the solve vs cb = |A^-1| xb + Ahat |d|
G_ENDS = 16.0   # end-point derivatives of the fp64 coefficients vs |A| Ahat |d|
G_SET = 16.0    # set path coefficients vs Ahat |d|
G_COST = 4.0    # a cost vs sum |c_a Q_ab c_b|
NORTH_STAR = 1e-9
CASES = [(N, r) for N in (6, 8, 10, 12) for r in range(N // 2)]
LIM_OF_Q = (0, 2, 4, 1, 3, 5, 6, 7, 8)  # limit index of maxima quantity q (violation_scaling, eth/trajectory.cpp:625-657)
LIMITS = np.array((4.0, 2.0, 2.0, 1.0, 20.0, 20.0, 1.0, 2.0, 10.0))

# (N, r, problem) of the normal band where the scaled coefficient error passes 1e-9 although cond_skeel * U < 1e-12 (worst
# 1.1e-8, at (10, 3, 2)).  The reference forms H = A^-T Q A^-1 and c = A^-1 d with an explicit fp64 A^-1 (lin_impl.h:147-177,
# 271-280, 320); the rounding of that inverse reaches the free derivatives through H and the coefficients directly, and the
# condition of the exact H does not see it.  The error stays within the componentwise bound cb of that formation, which is
# asserted for these problems as for every other.  The set is exact: each test asserts that its (N, r) meets these and no others.
NORTH_STAR_EXCEPTIONS = frozenset({(8, 1, 1), (8, 1, 3), (10, 3, 1), (10, 3, 2)})

# Maxima whose maximising critical point the model classifies as a multiple or near-multiple root (exact_model.NEAR_MULTIPLE):
# the reference drops every root with |im| > DBL_EPSILON (eth/polynomial.cpp:36-63, restated at oracle/trajectory.cpp:79), and
# fp64 root finding returns such a pair as complex, so the kernel may report less than the true maximum there: the lower bound is
# not asserted for them.  Entries are ("extrema", N, segment, quantity) or ("max_magnitude", N, problem, derivative); the inputs
# below meet none, and each test asserts that the cases it meets are exactly the listed ones of its N.
NEAR_MULTIPLE_CASES = frozenset()


def general_only(ctx):
    if getattr(ctx, "solve_kernels", "by-size") != "by-size":
        pytest.skip("the general-shape path has one dispatch")


# ---- inputs ---------------------------------------------------------------------------------------------------------------------
def dims_for(N, r, band):
    return 1 + (N // 2 + r + 2 * band) % 4


def make_problems(N, r, band):
    """Ragged batch of one (N, r, band): band 0 normal times, band 1 with a 0.01 s and a 20 s segment in every problem that has
    two or more segments.  Problem 0 fully fixed, problem 1 interior vertices with position only; positions offset by 1 km
    (problems 1, 4) or scaled to 6 cm (problems 2, 5)."""
    H = N // 2
    rng = np.random.default_rng(7919 * N + 31 * r + band)
    D = dims_for(N, r, band)
    Vs = (5, 13, 2, 7, 4) if band == 0 else (4, 6, 2)
    probs = []
    for p, V in enumerate(Vs):
        m, v = random_vertices(rng, N, V, D)
        if p == 0:
            m[:] = (1 << H) - 1
            v[:, :, :D] = rng.normal(size=(V, H, D)) * np.where(np.arange(H) == 0, 4.0, 0.6)[None, :, None]
        if p == 1:
            m[1:-1] = 1
            v[1:-1, 1:, :] = 0.0
        if p % 3 == 1:
            v[:, 0, :D] += 1000.0
        elif p % 3 == 2:
            v[:, :, :D] *= 0.015
        t = rng.uniform(0.3, 5.0, V - 1)
        if band == 1:
            if V == 2:
                t[0] = 20.0
            else:
                i, j = rng.choice(V - 1, 2, replace=False)
                t[i], t[j] = 0.01, 20.0
        probs.append((m, v, t))
    return D, probs


def batch(probs, D):
    off = np.concatenate([[0], np.cumsum([len(m) for m, _, _ in probs])]).astype(np.int32)
    mask = np.concatenate([m for m, _, _ in probs])
    vals = np.ascontiguousarray(np.concatenate([v for _, v, _ in probs])[:, :, :D])
    times = np.concatenate([t for _, _, t in probs])
    return off, mask, vals, times


@pytest.fixture(scope="module")
def model():
    """The model's results per (N, r, band), computed once for the emulator and the GPU runs."""
    cache = {}

    def get(N, r, band):
        if (N, r, band) not in cache:
            D, probs = make_problems(N, r, band)
            cache[(N, r, band)] = (D, probs, [EM.solve(N, r, m, v, t, D) for m, v, t in probs])
        return cache[(N, r, band)]

    return get


class Worst:
    """Worst ratio per check, printed and recorded."""

    def __init__(self):
        self.w = {}

    def add(self, name, err, scale):
        q = float(err) / scale if scale > 0 else (0.0 if err == 0 else math.inf)
        self.w[name] = max(self.w.get(name, 0.0), q)
        return q

    def report(self, where, record_property):
        line = ", ".join(f"{k} {v:.3g}" for k, v in sorted(self.w.items()))
        print(f"{where}: {line}")
        record_property(where, dict(self.w))


# ---- 1 + 2: the linear solve and the set path -----------------------------------------------------------------------------------
def check_linear(ctx, model, N, r, band, record_property):
    general_only(ctx)
    H = N // 2
    D, probs, exact = model(N, r, band)
    off, mask, vals, times = batch(probs, D)
    coef, cost, free = ctx.solve_linear_free_batch_nd(N, D, off, mask, vals, times, r)
    coef2, cost2 = ctx.solve_linear_batch_nd(N, D, off, mask, vals, times, r)
    assert np.array_equal(coef, coef2) and np.array_equal(cost, cost2)
    W = Worst()
    s0 = 0
    free_exact = []
    north_star_seen = set()
    for p, ((m, v, t), ex) in enumerate(zip(probs, exact)):
        S = len(t)
        fr, _ = EM._slots(N, m)
        where = (N, r, band, p)
        # the kernel's free derivatives make the exact reduced gradient vanish up to the rounding of forming H and g: a solve of any
        # other objective (a wrong entry of Q, A^-1 or H, a wrong right-hand side) leaves their difference here
        for d in range(D):
            if ex["n_free"]:
                res, scale = EM.reduced_gradient(ex, free[p][d], d)
                for i in range(ex["n_free"]):
                    q = W.add("gradient", abs(res[i]), U * scale[i])
                    assert q <= G_GRAD, (where, d, i, q)
        # free derivatives against the optimum, componentwise
        for d in range(D):
            for i in range(ex["n_free"]):
                W.add("free/skeel", abs(EM.X(free[p][d, i]) - ex["x"][d][i]), U * ex["xs"][d, i])
                q = W.add("free/xb", abs(EM.X(free[p][d, i]) - ex["x"][d][i]), U * ex["xb"][d, i])
                assert q <= G_SOLVE, (where, d, i, q)
        free_exact.append(np.array([[float(ex["x"][d][i]) for i in range(ex["n_free"])] for d in range(D)]).reshape(D, ex["n_free"]))
        for s in range(S):
            g = EM.segment(N, r, float(t[s]))
            keys = [(s + w, k) for w in (0, 1) for k in range(H)]
            for d in range(D):
                c = coef[s0 + s, d]
                # (a) the coefficients reproduce the end-point derivatives: fixed values, and the returned free values (so both
                # sides of an interior vertex meet); independent of the conditioning
                dk = np.array([free[p][d, fr[kk]] if kk in fr else v[kk[0], kk[1], d] for kk in keys])
                bound = g["absA"] @ g["Ahat"] @ np.abs(dk)
                for a, kk in enumerate(keys):
                    val, _ = EM.deriv_value(c, 0.0 if a < H else t[s], kk[1])
                    q = W.add("ends", abs(val - EM.X(dk[a])), U * bound[a])
                    assert q <= G_ENDS, (where, s, d, kk, q)
                # (b) the coefficients against the optimum, componentwise and scaled
                ce = ex["coef"][s][d]
                for j in range(N):
                    q = W.add("coef/cb", abs(EM.X(c[j]) - ce[j]), U * ex["cb"][s, d, j])
                    assert q <= G_COEF, (where, s, d, j, q)
                Tj = float(t[s]) ** np.arange(N)
                sc = max(abs(float(ce[j])) * Tj[j] for j in range(N))
                err = max(abs(float(EM.X(c[j]) - ce[j])) * Tj[j] for j in range(N))
                rel = err / sc if sc > 0 else err
                W.add("scaled", rel, 1.0)
                W.add("scaled/cond", rel, U * ex["cond_skeel"])
                if band == 0 and ex["cond_skeel"] * U < 1e-12 and rel > NORTH_STAR:
                    north_star_seen.add((N, r, p))
        # the cost: against the model at the kernel's own coefficients, and against the exact optimum
        own, mag = EM.cost_of(N, r, coef[s0:s0 + S], t)
        q = W.add("cost/own", abs(EM.X(cost[p]) - own), U * mag)
        assert q <= G_COST, (where, q)
        lin = sum(float(np.abs(coef[s0 + s, d]) @ EM.segment(N, r, float(t[s]))["absQ"] @ ex["cb"][s, d]) for s in range(S) for d in range(D))
        quad = sum(float(ex["cb"][s, d] @ EM.segment(N, r, float(t[s]))["absQ"] @ ex["cb"][s, d]) for s in range(S) for d in range(D))
        bound = U * (mag + 2.0 * G_COEF * lin) + (G_COEF * U) ** 2 * quad
        q = W.add("cost/opt", abs(EM.X(cost[p]) - ex["cost"]), bound)
        assert q <= G_COST, (where, q)
        s0 += S
    # 2. the set path, fed the exact free derivatives rounded to fp64
    coef_s, cost_s = ctx.set_free_constraints_batch_nd(N, D, off, mask, vals, times, free_exact, r)
    s0 = 0
    for p, (m, v, t) in enumerate(probs):
        S = len(t)
        ce, cb = EM.coefficients_from_free(N, r, m, v, t, free_exact[p], D)
        for s in range(S):
            for d in range(D):
                for j in range(N):
                    q = W.add("set/coef", abs(EM.X(coef_s[s0 + s, d, j]) - ce[s][d][j]), U * cb[s, d, j])
                    assert q <= G_SET, (N, r, band, p, s, d, j, q)
        own, mag = EM.cost_of(N, r, coef_s[s0:s0 + S], t)
        q = W.add("set/cost", abs(EM.X(cost_s[p]) - own), U * mag)
        assert q <= G_COST, (N, r, band, p, q)
        s0 += S
    assert north_star_seen == ({e for e in NORTH_STAR_EXCEPTIONS if e[:2] == (N, r)} if band == 0 else set()), north_star_seen
    W.w["north-star exceptions"] = float(len(north_star_seen))
    W.w["cond_skeel_max"] = max(ex["cond_skeel"] for ex in exact)
    W.report(f"exact linear N={N} r={r} {'extreme' if band else 'normal'} D={D}", record_property)


@pytest.mark.parametrize("band", [0, 1], ids=["normal", "extreme"])
@pytest.mark.parametrize("N,r", CASES)
def test_linear_exact_emulator(emu_ctx, model, N, r, band, record_property):
    check_linear(emu_ctx, model, N, r, band, record_property)


@pytest.mark.gpu
@pytest.mark.parametrize("band", [0, 1], ids=["normal", "extreme"])
@pytest.mark.parametrize("N,r", CASES)
def test_linear_exact_gpu(gpu_ctx, model, N, r, band, record_property):
    check_linear(gpu_ctx, model, N, r, band, record_property)


# ---- 3. evaluation and sampling -------------------------------------------------------------------------------------------------
def locate(times, t):
    """The segment and local time Trajectory::evaluate uses for global time t (eth/trajectory.cpp:55-87), or None past the end."""
    acc, i = 0.0, 0
    S = len(times)
    for i in range(S):
        acc = acc + float(times[i])
        if acc > t:
            break
    if t > acc:
        return None
    if i >= S:
        i = S - 1
    return i, t - (acc - float(times[i]))


def sample_times(times, dt):
    """(segment, local time) of every sample of sampleWholeTrajectory's dt walk (eth/trajectory.cpp:93-151)."""
    T = [float(x) for x in times]
    S, t_end = len(T), 0.0
    for x in T:
        t_end = t_end + x
    acc, i = 0.0, 0
    for i in range(S):
        acc = acc + T[i]
        if acc > 0.0:
            break
    if 0.0 > acc or i >= S:
        return []
    acc = acc - T[i]
    tin, out = 0.0 - acc, []
    while acc < t_end:
        if tin > T[i]:
            tin = tin - T[i]
            i += 1
            if i >= S:
                break
            continue
        out.append((i, tin))
        tin = tin + dt
        acc = acc + dt
    return out


def horner_bound(N, terms):
    return 2.0 * (N + 1) * U * terms  # one multiply and one add per Horner step


def check_evaluate_sample(ctx, model, N, record_property):
    general_only(ctx)
    W = Worst()
    for band in (0, 1):
        r = N // 2 - 1
        D, probs, _ = model(N, r, band)
        off, mask, vals, times = batch(probs, D)
        coef, _ = ctx.solve_linear_batch_nd(N, D, off, mask, vals, times, r)
        seg_off = off - np.arange(len(off), dtype=np.int32)
        rng = np.random.default_rng(N + 10 * band)
        for p, (_, _, t) in enumerate(probs):
            cs = coef[seg_off[p]:seg_off[p + 1]]
            bnd = np.concatenate([[0.0], np.cumsum(t)])
            tq = np.concatenate([bnd, [bnd[-1] + 1.0, bnd[-1] * (1 + 1e-9)], rng.uniform(0.0, bnd[-1], 6)])
            for k in range(N + 4):
                out, ok = ctx.evaluate_nd(N, D, cs, t, tq, k)
                for qi, tt in enumerate(tq):
                    loc = locate(t, float(tt))
                    assert bool(ok[qi]) == (loc is not None), (N, band, p, k, tt)
                    if loc is None:
                        assert np.all(out[qi] == 0.0)
                        continue
                    i, tin = loc
                    for d in range(D):
                        if k >= N:
                            assert out[qi, d] == 0.0
                            continue
                        val, terms = EM.deriv_value(cs[i, d], tin, k)
                        q = W.add(f"evaluate k={k}", abs(EM.X(out[qi, d]) - val), horner_bound(N, terms))
                        assert q <= 1.0, (N, band, p, k, tt, d, q)
        if D < 3:
            continue
        for dt in (0.2, 0.037):
            counts, samples, full = ctx.sample_batch_nd(N, D, seg_off, coef, times, dt, full=True)
            m0 = 0
            for p, (_, _, t) in enumerate(probs):
                st = sample_times(t, dt)
                assert counts[p] == len(st), (N, band, p, dt)
                cs = coef[seg_off[p]:seg_off[p + 1]]
                fields = [(f, d, 0) for f, d in zip(range(4), range(4))] + [(4 + d, d, 1) for d in range(4)] + \
                    [(8 + d, d, 2) for d in range(4)] + [(12 + d, d, 3) for d in range(3)] + [(15 + d, d, 4) for d in range(3)]
                for m_i, (i, tin) in enumerate(st):
                    row = full[m0 + m_i]
                    assert np.array_equal(samples[m0 + m_i, :3], row[:3])
                    for f, d, k in fields:
                        if d >= D:
                            assert row[f] == 0.0
                            continue
                        val, terms = EM.deriv_value(cs[i, d], tin, k)
                        q = W.add(f"sample k={k}", abs(EM.X(row[f]) - val), horner_bound(N, terms))
                        assert q <= 1.0, (N, band, p, dt, m_i, f, q)
                m0 += counts[p]
    W.report(f"exact evaluate/sample N={N}", record_property)


@pytest.mark.parametrize("N", [6, 8, 10, 12])
def test_evaluate_sample_exact_emulator(emu_ctx, model, N, record_property):
    check_evaluate_sample(emu_ctx, model, N, record_property)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [6, 8, 10, 12])
def test_evaluate_sample_exact_gpu(gpu_ctx, model, N, record_property):
    check_evaluate_sample(gpu_ctx, model, N, record_property)


# ---- 4. maxima ------------------------------------------------------------------------------------------------------------------
def maxima_input(ctx, N):
    """Short trajectories for the maxima: one with a 0.01 s and a 20 s segment (1 km offset), one in the normal band (6 cm),
    solved on the device at r = N/2 - 1; coefficients padded to 4 dimensions."""
    rng = np.random.default_rng(4000 + N)
    D = 4 if N in (6, 12) else 3
    probs = []
    for p, (V, tt) in enumerate(((4, (0.01, 1.7, 20.0)), (3, tuple(rng.uniform(0.3, 5.0, 2))))):
        m, v = random_vertices(rng, N, V, D)
        if p == 0:
            v[:, 0, :D] += 1000.0
        else:
            v[:, :, :D] *= 0.015
        probs.append((m, v, np.array(tt)))
    off, mask, vals, times = batch(probs, D)
    coef, _ = ctx.solve_linear_batch_nd(N, D, off, mask, vals, times, N // 2 - 1)
    return D, off - np.arange(len(off), dtype=np.int32), coef, times


def pad4(c):
    out = np.zeros((c.shape[0], 4, c.shape[2]))
    out[:, :c.shape[1]] = c
    return out


def check_max_value(W, name, got, ex, where, near_multiple):
    """Upper bound and lower bound of one maximum; a near-multiple maximising root is added to near_multiple instead of checked
    from below."""
    q = W.add(f"{name} above", max(0.0, float(EM.X(got) - ex["value"])), ex["err"])
    assert q <= 1.0, (where, "above the true maximum", got, float(ex["value"]))
    rel = float((ex["value"] - EM.X(got)) / ex["value"]) if ex["value"] > 0 else 0.0
    W.add(f"{name} below(rel)", max(rel, 0.0), 1.0)
    if ex["near_multiple"]:
        near_multiple.add(where)
        return
    assert float(EM.X(got) - ex["value"]) >= -(NORTH_STAR * float(ex["value"]) + ex["err"]), (where, "below the true maximum", got,
                                                                                               float(ex["value"]), float(ex["t"]))


def check_maxima(ctx, N, record_property):
    general_only(ctx)
    W = Worst()
    D, seg_off, coef, times = maxima_input(ctx, N)
    c4 = pad4(coef)
    m = ctx.extrema_nd(N, D, coef, times)
    near_multiple = set()
    for s in range(len(times)):
        exs = EM.nine_maxima(c4[s], times[s])
        for q, ex in enumerate(exs):
            where = ("extrema", N, s, q)
            # the end points are candidates: the value is at least theirs
            dims, k = EM.QUANTITIES[q]
            ends = max(math.sqrt(sum(float(EM.deriv_value(c4[s, d], tt, k)[0]) ** 2 for d in dims)) for tt in (0.0, float(times[s])))
            assert m[s, q] >= ends - ex["err"], (where, "below an end point")
            check_max_value(W, f"extrema q={q}", m[s, q], ex, where, near_multiple)
    for k in (1, 2, 3, 4):
        tt, vv, ii = ctx.max_magnitude_nd(N, D, seg_off, coef, times, k)
        for p in range(len(seg_off) - 1):
            s0, s1 = seg_off[p], seg_off[p + 1]
            exs = [EM.maximum(list(c4[s]), times[s], k) for s in range(s0, s1)]
            where = ("max_magnitude", N, p, k)
            i = int(ii[p])
            assert 0 <= i < s1 - s0 and 0.0 <= tt[p] <= times[s0 + i], (where, i, tt[p])
            here = math.sqrt(sum(float(EM.deriv_value(c4[s0 + i, d], tt[p], k)[0]) ** 2 for d in range(4)))
            q = W.add(f"max_magnitude k={k} value at (t, i)", abs(here - vv[p]), exs[i]["err"])
            assert q <= 1.0, (where, here, vv[p])
            best = max(range(len(exs)), key=lambda j: exs[j]["value"])
            check_max_value(W, f"max_magnitude k={k}", vv[p], dict(exs[best], err=max(e["err"] for e in exs)), where, near_multiple)
    assert near_multiple == {c for c in NEAR_MULTIPLE_CASES if c[1] == N}, near_multiple
    W.w["near-multiple maxima"] = float(len(near_multiple))
    W.report(f"exact maxima N={N}", record_property)


@pytest.mark.parametrize("N", [6, 8, 10, 12])
def test_maxima_exact_emulator(emu_ctx, N, record_property):
    check_maxima(emu_ctx, N, record_property)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [6, 8, 10, 12])
def test_maxima_exact_gpu(gpu_ctx, N, record_property):
    check_maxima(gpu_ctx, N, record_property)


# ---- 5. time scaling ------------------------------------------------------------------------------------------------------------
def check_scaling(ctx, N, record_property):
    general_only(ctx)
    W = Worst()
    D, seg_off, coef, times = maxima_input(ctx, N)
    rng = np.random.default_rng(50 + N)
    scaled = 0
    try:
        for tol in (1e-3, -0.2):
            ctx.test_set_scale_tolerance(tol)
            lim = LIMITS * np.exp(rng.uniform(-2.5, -0.5, 9))
            c2, t2, passes, within = ctx.scale_times_nd(N, D, seg_off, coef, times, lim)
            for p in range(len(seg_off) - 1):
                for s in range(seg_off[p], seg_off[p + 1]):
                    where = (N, tol, p, s)
                    assert t2[s] >= times[s], where
                    # the reparametrisation p_new(S t) = p_old(t), S = T_new / T_old: c_new_j S^j = c_old_j up to the rounding of
                    # the passes' factors (j + 1 products per pass on the coefficient, one on the time)
                    Sx = EM.X(t2[s]) / EM.X(times[s])
                    scaled += int(t2[s] != times[s])
                    for d in range(D):
                        for j in range(N):
                            err = abs(EM.X(c2[s, d, j]) * Sx ** j - EM.X(coef[s, d, j]))
                            q = W.add("reparametrisation", err, U * (2 * j + 3) * max(int(passes[p]), 1) * abs(coef[s, d, j]))
                            assert q <= 1.0, (where, d, j, q)
                if within[p] and tol > 0:
                    # the model's maxima of the scaled trajectory meet the limits within the tolerance (eth/trajectory.cpp:660-689)
                    for s in range(seg_off[p], seg_off[p + 1]):
                        for q, ex in enumerate(EM.nine_maxima(pad4(c2[s:s + 1])[0], t2[s])):
                            lq = lim[LIM_OF_Q[q]]
                            over = float(ex["value"]) - lq * (1.0 + tol)
                            qq = W.add("within: above the limit", max(over, 0.0), ex["err"] + 4 * U * lq)
                            assert qq <= 1.0, (N, p, s, q, float(ex["value"]), lq)
    finally:
        ctx.test_set_scale_tolerance(1e-3)
    assert scaled > 0
    W.report(f"exact scaling N={N}", record_property)


@pytest.mark.parametrize("N", [6, 8, 10, 12])
def test_scaling_exact_emulator(emu_ctx, N, record_property):
    check_scaling(emu_ctx, N, record_property)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [6, 8, 10, 12])
def test_scaling_exact_gpu(gpu_ctx, N, record_property):
    check_scaling(gpu_ctx, N, record_property)
