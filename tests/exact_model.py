"""An exact model of the general-shape operations, written from the mathematics (mpmath, DPS digits).

It imports neither oracle/ nor the library: it is the yardstick both are measured against (tests/test_exact_model.py).  Every
fp64 input is taken exactly (mp.mpf of a double is exact), so the model answers "what is the true value for these fp64 inputs",
and the error bounds it returns are the componentwise first-order bounds of the fp64 computation, in units of the unit roundoff U.

Conventions (the reference's, cited where they are fixed):
  * a segment polynomial is p(t) = sum_j c_j t^j on [0, T], N coefficients, N even; vertex derivatives 0 .. N/2-1 at both ends;
  * the cost of a problem is 0.5 sum_segments sum_dims c^T Q c (lin_impl.h:127-141) with the reference's
    Q[i][j] = B[r][i] B[r][j] T^e * 2 / e, e = i + j - 2r + 1 (lin_impl.h:605-618): that is 2 * integral(p^(r) p^(r)), so the
    cost is sum_segments sum_dims integral_0^T (p^(r)(t))^2 dt, which is what `cost_of` computes by exact integration;
  * free derivatives are ordered vertex-major, derivative ascending (the d_p of lin_impl.h:340-373);
  * time scaling by s is the reparametrisation p_new(s t) = p_old(t), so c_new_j s^j = c_old_j (polynomial.cpp:218-224).
"""
import functools
import math

import mpmath as mp
import numpy as np

DPS = 60
U = 2.0 ** -53  # unit roundoff of fp64
# a maximising critical point closer than this (relative to T) to another root of d/dt |p^(k)|^2 is a near-multiple root: fp64
# root finding cannot separate the pair (the discriminant of their quadratic factor is below rounding), see `maximum`
NEAR_MULTIPLE = 64.0 * math.sqrt(U)


def fall(j, k):
    """Falling factorial j (j-1) ... (j-k+1) = d^k/dt^k t^j / t^(j-k); 0 for k > j."""
    if k > j:
        return 0
    p = 1
    for q in range(k):
        p *= j - q
    return p


def X(x):
    return mp.mpf(float(x))


def _absf(M):
    """|M| of an mp matrix as a float numpy array (bounds need a few digits only)."""
    return np.array([[abs(float(M[i, j])) for j in range(M.cols)] for i in range(M.rows)])


# ---- one segment --------------------------------------------------------------------------------------------------------------
def endpoint_matrix(N, T):
    """A(T): rows 0 .. N/2-1 = derivative k at t = 0, rows N/2 + k = derivative k at t = T (eth/polynomial.h:208-226)."""
    H = N // 2
    A = mp.zeros(N, N)
    for k in range(H):
        A[k, k] = fall(k, k)
        for j in range(k, N):
            A[H + k, j] = fall(j, k) * T ** (j - k)
    return A


def cost_matrix(N, r, T):
    """Q with c^T Q c = integral_0^T (p^(r)(t))^2 dt, by exact integration of the monomials."""
    Q = mp.zeros(N, N)
    for a in range(r, N):
        for b in range(r, N):
            e = a + b - 2 * r + 1
            Q[a, b] = fall(a, r) * fall(b, r) * T ** e / e
    return Q


@functools.lru_cache(maxsize=None)
def segment(N, r, T):
    """Exact A, A^-1, Q of a segment of fp64 length T, and the float bound matrices |A|, |Q| and Ahat = |A^-1||A||A^-1| (the
    componentwise first-order error of an A^-1 computed in fp64 from a correctly rounded A, in units of U)."""
    with mp.workdps(DPS):
        Tm = X(T)
        A = endpoint_matrix(N, Tm)
        Ai = A ** -1
        Q = cost_matrix(N, r, Tm)
        K = Ai.T * Q * Ai
    absA, absAi = _absf(A), _absf(Ai)
    return dict(A=A, Ai=Ai, Q=Q, K=K, absA=absA, absAi=absAi, absQ=_absf(Q), Ahat=absAi @ absA @ absAi)


def deriv_value(c, t, k):
    """(p^(k)(t) exactly, sum_j |c_j fall(j, k) t^(j-k)| as a float) for fp64 (or mp) coefficients c."""
    with mp.workdps(DPS):
        tm = t if isinstance(t, mp.mpf) else X(t)
        v, s = mp.mpf(0), mp.mpf(0)
        for j in range(k, len(c)):
            term = (c[j] if isinstance(c[j], mp.mpf) else X(c[j])) * fall(j, k) * tm ** (j - k)
            v += term
            s += abs(term)
        return v, float(s)


def cost_of(N, r, coef, times):
    """Exact sum_segments sum_dims c^T Q c of given coefficients [S][D][N], and sum |c_a Q_ab c_b| as a float."""
    with mp.workdps(DPS):
        tot, mag = mp.mpf(0), 0.0
        for s in range(len(times)):
            g = segment(N, r, float(times[s]))
            for d in range(coef.shape[1]):
                c = mp.matrix([X(x) for x in coef[s, d]])
                tot += (c.T * g["Q"] * c)[0]
                ac = np.abs(coef[s, d])
                mag += float(ac @ g["absQ"] @ ac)
        return tot, mag


# ---- the linear problem of PolynomialOptimization<N>(D) -----------------------------------------------------------------------
def _slots(N, mask):
    H = N // 2
    free, fixed = {}, []
    for v in range(len(mask)):
        for k in range(H):
            if (int(mask[v]) >> k) & 1:
                fixed.append((v, k))
            else:
                free[(v, k)] = len(free)
    return free, fixed


def solve(N, r, mask, vals, times, D):
    """setupFromVertices + solveLinear, exactly.  mask [V], vals [V][N/2][>= D], times [S].  Returns a dict:
      x       [D][n_free] mp   the optimal free derivatives
      coef    [S][D][N] mp     the optimal coefficients;  cost mp: the optimal cost
      cond_skeel               || |H^-1| |H| ||_inf of the reduced Hessian H (invariant under row scaling)
      xb      [D][n_free]      componentwise condition of each free derivative: |H^-1| (E_pp |x| + E_pf |d_f|), where
                               E = sum |A^-1|^T |Q| |A^-1| is the size of the terms the fp64 formation of H and of the right-hand
                               side sums; |x_fp64 - x| <= gamma U xb for a solve that is backward stable against that formation
      xs      [D][n_free]      the Skeel componentwise condition |H^-1| (|H| |x| + |H_pf| |d_f|): what a backward-stable solve of the
                               EXACT H would achieve; reported, not a bound here (H is formed in fp64 from an explicit A^-1)
      cb      [S][D][N]        the same for the coefficients: |A^-1| xb + Ahat |d|, d the segment's end-point derivatives (the
                               free derivatives' error through A^-1, and the error of the computed A^-1 applied to d)
      H, g, E, Eg              the exact reduced Hessian and right-hand sides (mp) and their rounding scales (reduced_gradient)
      d       [S][D][N] mp     the end-point derivatives of every segment (fixed values and x)
    """
    H = N // 2
    V, S = len(mask), len(times)
    free, fixed = _slots(N, mask)
    n = len(free)
    segs = [segment(N, r, float(times[s])) for s in range(S)]
    keys = [[(s + w, k) for w in (0, 1) for k in range(H)] for s in range(S)]
    with mp.workdps(DPS):
        fixval = [{fk: X(vals[fk[0], fk[1], d]) for fk in fixed} for d in range(D)]
        Hm = mp.zeros(n, n)
        g = [mp.zeros(n, 1) for _ in range(D)]
        Hh = np.zeros((n, n))
        gh = np.zeros((D, n))
        for s in range(S):
            K, aAi, aQ = segs[s]["K"], segs[s]["absAi"], segs[s]["absQ"]
            Kh = aAi.T @ aQ @ aAi
            for a, ka in enumerate(keys[s]):
                if ka not in free:
                    continue
                ia = free[ka]
                for b, kb in enumerate(keys[s]):
                    if kb in free:
                        Hm[ia, free[kb]] += K[a, b]
                        Hh[ia, free[kb]] += Kh[a, b]
                    else:
                        for d in range(D):
                            g[d][ia] += K[a, b] * fixval[d][kb]
                            gh[d, ia] += Kh[a, b] * abs(float(vals[kb[0], kb[1], d]))
        if n:
            Hi = mp.inverse(Hm)
            x = [Hi * (-g[d]) for d in range(D)]
            aHi, aH = _absf(Hi), _absf(Hm)
            cond_skeel = float(np.abs(aHi @ aH).sum(axis=1).max())
        else:
            x, cond_skeel = [None] * D, 1.0
        xb, xs = np.zeros((D, n)), np.zeros((D, n))
        if n:
            aHpf = np.zeros((D, n))  # |H_pf| |d_f|
            for s in range(S):
                K = segs[s]["K"]
                for a, ka in enumerate(keys[s]):
                    if ka in free:
                        for b, kb in enumerate(keys[s]):
                            if kb not in free:
                                for d in range(D):
                                    aHpf[d, free[ka]] += abs(float(K[a, b])) * abs(float(vals[kb[0], kb[1], d]))
            for d in range(D):
                ax = np.array([abs(float(x[d][i])) for i in range(n)])
                xb[d] = aHi @ (Hh @ ax + gh[d])
                xs[d] = aHi @ (aH @ ax + aHpf[d])

        def val(d, key):
            return x[d][free[key]] if key in free else fixval[d][key]

        coef = [[None] * D for _ in range(S)]
        dv = [[None] * D for _ in range(S)]
        cb = np.zeros((S, D, N))
        cost = mp.mpf(0)
        for s in range(S):
            for d in range(D):
                dd = mp.matrix([val(d, kk) for kk in keys[s]])
                c = segs[s]["Ai"] * dd
                coef[s][d] = [c[j] for j in range(N)]
                dv[s][d] = [dd[j] for j in range(N)]
                ad = np.array([abs(float(dd[j])) for j in range(N)])
                bx = np.array([xb[d, free[kk]] if kk in free else 0.0 for kk in keys[s]])
                cb[s, d] = segs[s]["absAi"] @ bx + segs[s]["Ahat"] @ ad
                cost += (c.T * segs[s]["Q"] * c)[0]
        return dict(x=[[x[d][i] for i in range(n)] for d in range(D)], coef=coef, d=dv, cost=cost, cond_skeel=cond_skeel, xb=xb, xs=xs,
                    cb=cb, n_free=n, H=Hm, g=g, E=Hh, Eg=gh)


def reduced_gradient(ex, free_vals, d):
    """Half the exact gradient of the cost over the free derivatives, H x + g, at given fp64 free derivatives x (one dimension d of
    a `solve` result), and its rounding scale E |x| + E_pf |d_f|: the size of the terms the fp64 formation of H and g sums
    (E = sum |A^-1|^T |Q| |A^-1|).  A solve of the right objective leaves a residual of a few U times that scale; a solve of a
    different objective leaves the difference of the two gradients."""
    n = ex["n_free"]
    with mp.workdps(DPS):
        xv = mp.matrix([X(free_vals[i]) for i in range(n)])
        res = ex["H"] * xv + ex["g"][d]
        scale = ex["E"] @ np.abs(np.asarray(free_vals, dtype=float)) + ex["Eg"][d]
        return [res[i] for i in range(n)], scale


def coefficients_from_free(N, r, mask, vals, times, free_vals, D):
    """setFreeConstraints + getSegments, exactly: c = A^-1 d per segment from the fixed values and the given free derivatives
    free_vals [D][n_free] (fp64).  Returns coef [S][D][N] mp and the bound Ahat |d| [S][D][N] (units of U)."""
    H = N // 2
    free, _ = _slots(N, mask)
    S = len(times)
    coef, cb = [[None] * D for _ in range(S)], np.zeros((S, D, N))
    with mp.workdps(DPS):
        for s in range(S):
            g = segment(N, r, float(times[s]))
            keys = [(s + w, k) for w in (0, 1) for k in range(H)]
            for d in range(D):
                dd = [X(free_vals[d][free[kk]]) if kk in free else X(vals[kk[0], kk[1], d]) for kk in keys]
                c = g["Ai"] * mp.matrix(dd)
                coef[s][d] = [c[j] for j in range(N)]
                cb[s, d] = g["Ahat"] @ np.array([abs(float(v)) for v in dd])
    return coef, cb


# ---- maxima -------------------------------------------------------------------------------------------------------------------
def maximum(polys, T, k):
    """True max over t in [0, T] of |(p_1^(k)(t), ..., p_m^(k)(t))| for fp64 coefficient rows polys [m][N].

    Candidates: t = 0, t = T and the real roots in [0, T] of d/dt |p^(k)|^2 / 2 = sum_d p_d^(k) p_d^(k+1), found by mp.polyroots
    at high precision in u = t / T (degree <= 2 (N - k) - 3).  Returns dict(value, t, interior, sep, mult, near_multiple, err):
    sep = distance (in t) from the maximising root to the nearest other root, mult = roots within 1e-30 T of it, near_multiple =
    sep < NEAR_MULTIPLE * T, err = an upper bound on the fp64 rounding of the magnitude anywhere on [0, T] (Horner on N
    coefficients, the squares, the sum and the root)."""
    N = len(polys[0])
    with mp.workdps(DPS):
        Tm = X(T)
        q = []  # coefficients in u of p_d^(k)(T u)
        for c in polys:
            q.append([X(c[j]) * fall(j, k) * Tm ** (j - k) for j in range(k, N)])
        L = N - k
        G = [mp.mpf(0)] * max(2 * L - 2, 1)  # sum_d q_d(u) q_d'(u)
        for qd in q:
            for a in range(L):
                for b in range(1, L):
                    G[a + b - 1] += qd[a] * b * qd[b]
        while len(G) > 1 and G[-1] == 0:
            G.pop()

        def mag(u):
            s = mp.mpf(0)
            for qd in q:
                v = mp.mpf(0)
                for j in range(L - 1, -1, -1):
                    v = v * u + qd[j]
                s += v * v
            return mp.sqrt(s)

        best = dict(value=mag(mp.mpf(0)), u=mp.mpf(0), interior=False, sep=math.inf, mult=1)
        vT = mag(mp.mpf(1))
        if vT > best["value"]:
            best.update(value=vT, u=mp.mpf(1))
        roots = []
        if len(G) > 1:
            roots = mp.polyroots(G[::-1], maxsteps=400, extraprec=4 * DPS)
        tiny = mp.mpf(10) ** (-DPS // 2)
        for z in roots:
            if abs(mp.im(z)) > tiny:
                continue
            u = mp.re(z)
            if u < 0 or u > 1:
                continue
            v = mag(u)
            if v > best["value"]:
                others = [abs(w - z) for w in roots if w is not z]
                sep = float(min(others)) if others else math.inf
                mult = 1 + sum(1 for o in others if o < mp.mpf(10) ** -30)
                best.update(value=v, u=u, interior=True, sep=sep, mult=mult)
        err_terms = [float(sum(abs(x) for x in qd)) for qd in q]
    err = (N + 3) * U * math.sqrt(sum(e * e for e in err_terms)) * 2.0
    sep = best["sep"] * T
    return dict(value=best["value"], t=best["u"] * Tm, interior=best["interior"], sep=sep, mult=best["mult"],
                near_multiple=best["interior"] and (best["mult"] > 1 or best["sep"] < NEAR_MULTIPLE), err=err)


# the nine quantities of a segment's maxima (eth/trajectory.cpp:616-622): (dimensions, derivative)
QUANTITIES = [((0, 1), 1), ((0, 1), 2), ((0, 1), 3), ((2,), 1), ((2,), 2), ((2,), 3), ((3,), 1), ((3,), 2), ((3,), 3)]


def nine_maxima(c4, T):
    """The nine maxima of one segment, coefficients [4][N] (dimensions past D are zero rows)."""
    return [maximum([c4[d] for d in dims], T, k) for dims, k in QUANTITIES]
