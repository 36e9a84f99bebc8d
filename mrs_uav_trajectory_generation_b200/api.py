"""Host-side mirror of the reference's interface for the hot path (names, argument meaning and error behaviour follow
the C++ classes of include/eth_trajectory_generation/*.h), implemented on the C ABI of libtg_b200.so.

The reference API is one-object-per-problem; every class here also accepts batches because the GPU path is batched
(SURVEY.md H7).  The C++ shim with the same class names is include/eth_trajectory_generation_b200.hpp.
"""
import math

import numpy as np

from ._capi import Context, Library, N, D, HALF


class derivative_order:  # eth/motion_defines.h
    POSITION, VELOCITY, ACCELERATION, JERK, SNAP = 0, 1, 2, 3, 4
    INVALID = -1


_default_ctx = None


def default_context():
    """Lazily created process-wide context on device 0 (fails loudly without a GPU)."""
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(Library(), 0)
    return _default_ctx


class Vertex:
    """eth_trajectory_generation::Vertex (eth/vertex.h:42-116): derivative -> D-vector constraints."""

    def __init__(self, dimension=D):
        if not 1 <= dimension <= D:
            raise ValueError("the B200 path carries 1 to 4 dimensions (the node uses 4: x, y, z, heading, node.cpp:902)")
        self.D = dimension
        self.constraints = {}

    def addConstraint(self, derivative, value):  # eth/vertex.cpp:134-137
        v = np.asarray(value, dtype=np.float64).reshape(-1)
        if v.shape[0] != self.D:
            raise ValueError("constraint dimension mismatch")
        self.constraints[int(derivative)] = v.copy()

    def makeStartOrEnd(self, value, up_to_derivative):  # eth/vertex.cpp:158-163
        self.addConstraint(derivative_order.POSITION, value)
        for i in range(1, up_to_derivative + 1):
            self.constraints[i] = np.zeros(self.D)

    def removeConstraint(self, derivative):
        return self.constraints.pop(int(derivative), None) is not None

    def hasConstraint(self, derivative):
        return int(derivative) in self.constraints

    def getConstraint(self, derivative):
        return self.constraints.get(int(derivative))

    def mask_and_values(self, half=HALF):
        """Constraints with derivative > N/2 - 1 are dropped, as setupFromVertices does (lin_impl.h:84-102).  Values [half][D]."""
        m = 0
        vals = np.zeros((half, self.D))
        for k, v in self.constraints.items():
            if 0 <= k < half:
                m |= 1 << k
                vals[k] = v
        return m, vals


def pack_vertices(vertex_lists, half=HALF, dimension=D):
    vtx_off = [0]
    masks, vals = [], []
    for vl in vertex_lists:
        for v in vl:
            if v.D != dimension:
                raise ValueError("vertex dimension %d does not match the optimisation's %d" % (v.D, dimension))
            m, x = v.mask_and_values(half)
            masks.append(m)
            vals.append(x)
        vtx_off.append(len(masks))
    return np.array(vtx_off, dtype=np.int32), np.array(masks, dtype=np.uint8), np.array(vals, dtype=np.float64)


class Trajectory:
    """eth_trajectory_generation::Trajectory (eth/trajectory.h): segments = (coefficients [S,4,10], times [S])."""

    def __init__(self, coef=None, times=None, ctx=None):
        self.coef = None if coef is None else np.ascontiguousarray(coef, dtype=np.float64)
        self.times = None if times is None else np.ascontiguousarray(times, dtype=np.float64)
        self._ctx = ctx

    def _c(self):
        return self._ctx or default_context()

    def K(self):
        return 0 if self.times is None else len(self.times)

    def getMinTime(self):
        return 0.0

    def getMaxTime(self):  # eth/trajectory.h:76-83: accumulated in segment order
        t = 0.0
        for x in self.times:
            t += float(x)
        return t

    def toYaml(self):  # trajectoryToYaml / segmentsToFile (eth/io.cpp:66-70, 125-168)
        from . import segment_io

        return segment_io.segments_to_yaml(self.coef, self.times)

    @classmethod
    def fromYaml(cls, text, ctx=None):  # trajectoryFromYaml / segmentsFromFile (eth/io.cpp:114-122, 169-218); None when malformed
        from . import segment_io

        r = segment_io.segments_from_yaml(text)
        if r is None or not (1 <= r[0].shape[1] <= D and r[0].shape[2] in (6, 8, 10, 12)):
            return None  # shapes the device entry points take: N in {6, 8, 10, 12}, 1..4 dimensions
        return cls(r[0], r[1], ctx)

    def getSegmentTimes(self):
        return self.times.copy()

    def shape(self):
        """(D, N) of the segments (Trajectory::D(), N(), eth/trajectory.h:58-60)."""
        return (D, N) if self.coef is None else tuple(self.coef.shape[1:])

    def _tuned(self):
        return self.shape() == (D, N)

    def evaluate(self, t, derivative=derivative_order.POSITION):
        """Trajectory::evaluate (eth/trajectory.cpp:55-87); t may be an array.  Past-the-end queries return zeros."""
        if self._tuned():
            out, ok = self._c().evaluate(self.coef, self.times, t, derivative)
        else:
            d, n = self.shape()
            out, ok = self._c().evaluate_nd(n, d, self.coef, self.times, t, derivative)
        return out[0] if np.isscalar(t) else out

    def computeMaxDerivatives(self):
        """Per-segment maxima [S, 9] = hor v,a,j ; ver v,a,j ; heading v,a,j (eth/trajectory.cpp:422-565)."""
        if self._tuned():
            return self._c().extrema(self.coef, self.times)
        d, n = self.shape()
        return self._c().extrema_nd(n, d, self.coef, self.times)

    def scaleSegmentTimesToMeetConstraints(self, limits9):
        """eth/trajectory.cpp:598-692, in place; returns within_range."""
        seg_off = np.array([0, len(self.times)], dtype=np.int32)
        if self._tuned():
            self.coef, self.times, _, within = self._c().scale_times(seg_off, self.coef, self.times, limits9)
        else:
            d, n = self.shape()
            self.coef, self.times, _, within = self._c().scale_times_nd(n, d, seg_off, self.coef, self.times, limits9)
        return bool(within[0])


def sample_whole_trajectory(trajectory, dt, full=False, ctx=None):
    """eth_trajectory_generation::sampleWholeTrajectory (eth/trajectory_sampling.cpp:119-124).
    Returns samples [M, 4] (x, y, z, heading) or, with full=True, [M, 19] = p4 v4 a4 j3 s3 yaw."""
    c = ctx or trajectory._c()
    seg_off = np.array([0, trajectory.K()], dtype=np.int32)
    if trajectory._tuned():
        counts, samples, fullv = c.sample_batch(seg_off, trajectory.coef, trajectory.times, dt, full=full)
    else:  # any N in {6, 8, 10, 12}; D >= 3 as the reference demands (eth/trajectory_sampling.cpp:58-61)
        d, n = trajectory.shape()
        counts, samples, fullv = c.sample_batch_nd(n, d, seg_off, trajectory.coef, trajectory.times, dt, full=full)
    return fullv if full else samples


class PolynomialOptimization:
    """eth_trajectory_generation::PolynomialOptimization<N> (lin.h:60-233) for one problem or a batch.  N = 10 on 4 dimensions with
    derivative_to_optimize 2..4 (the node's shape) runs on the tuned kernels; N in {6, 8, 10, 12}, 1..4 dimensions and
    derivative_to_optimize 0 .. N/2-1 on the general-shape kernels (tg_solve_linear_batch_nd)."""

    N = N

    def __init__(self, dimension=D, ctx=None, n_coefficients=N):
        if not 1 <= dimension <= D:
            raise ValueError("1 to 4 dimensions")
        if n_coefficients not in (6, 8, 10, 12):
            raise ValueError("N = 6, 8, 10 or 12 coefficients (lin.h:46-55; Polynomial::kMaxN = 12)")
        self.N = n_coefficients
        self.dimension = dimension
        self._ctx = ctx
        self._lists = None
        self.derivative_to_optimize = derivative_order.INVALID
        self.coef = self.cost = None
        self._free = None  # per problem [dimension][n_free] once known; "solve" = the solve's, not fetched yet

    def _c(self):
        return self._ctx or default_context()

    def _packed(self):
        return pack_vertices(self._lists, self.N // 2, self.dimension)

    def _out(self, per_problem):
        return per_problem[0] if self._single else per_problem

    def setupFromVertices(self, vertices, times, derivative_to_optimize):  # lin_impl.h:61-106
        if not (0 <= derivative_to_optimize <= self.N // 2 - 1):  # kHighestDerivativeToOptimize (lin.h:55, lin_impl.h:63-66)
            print("You tried to optimize a derivative that is not possible")  # CHECK prints and continues (eth/misc.h)
            return False
        single = len(vertices) > 0 and isinstance(vertices[0], Vertex)
        self._lists = [vertices] if single else list(vertices)
        self._times = [np.asarray(times, dtype=np.float64)] if single else [np.asarray(t, dtype=np.float64) for t in times]
        for vl, t in zip(self._lists, self._times):
            if len(vl) != len(t) + 1:
                print("Size of times must be one less than positions.")
                return False
        self.derivative_to_optimize = derivative_to_optimize
        self._single = single
        self._free = None
        return True

    def updateSegmentTimes(self, times):  # lin_impl.h:288-304
        self._times = [np.asarray(times, dtype=np.float64)] if self._single else [np.asarray(t, dtype=np.float64) for t in times]
        self._free = None

    def solveLinear(self):  # lin_impl.h:340-373
        vtx_off, masks, vals = self._packed()
        self._free = "solve"
        self._seg_off = vtx_off - np.arange(len(vtx_off), dtype=np.int32)
        if self.N == N and self.dimension == D and self.derivative_to_optimize >= 2:
            self.coef, self.cost = self._c().solve_linear_batch(vtx_off, masks, vals, np.concatenate(self._times), self.derivative_to_optimize)
        else:
            self.coef, self.cost = self._c().solve_linear_batch_nd(self.N, self.dimension, vtx_off, masks, vals, np.concatenate(self._times),
                                                                   self.derivative_to_optimize)
        return True

    def computeCost(self):  # lin_impl.h:127-141
        return float(self.cost[0]) if self._single else self.cost.copy()

    def getSegmentTimes(self):
        return self._times[0].copy() if self._single else [t.copy() for t in self._times]

    def getTrajectory(self, index=0):  # lin.h:153-160
        s0, s1 = self._seg_off[index], self._seg_off[index + 1]
        return Trajectory(self.coef[s0:s1], self._times[index], self._ctx)

    def getSegments(self, index=0):  # lin.h:177
        t = self.getTrajectory(index)
        return t.coef, t.times

    # ---- free and fixed constraints (lin_impl.h:183-257, 513-522): lists of `dimension` vectors, each vertex-major with the derivative
    # ascending; for a batch, one such list per problem
    def _counts(self):
        vtx_off, masks, _ = self._packed()
        nf = Context.free_counts(self.N, vtx_off, masks)
        nv = np.diff(vtx_off)
        return nf, nv * (self.N // 2) - nf, (nv - 1) * self.N

    def getNumberFreeConstraints(self):
        return self._out([int(x) for x in self._counts()[0]])

    def getNumberFixedConstraints(self):
        return self._out([int(x) for x in self._counts()[1]])

    def getNumberAllConstraints(self):  # N/2 start and N/2 end rows per segment
        return self._out([int(x) for x in self._counts()[2]])

    def getFixedConstraints(self):
        vtx_off, masks, vals = self._packed()
        bits = ((masks[:, None] >> np.arange(self.N // 2)) & 1).astype(bool)  # [V][N/2], vertex-major then derivative
        return self._out([[vals[vtx_off[p]:vtx_off[p + 1]][bits[vtx_off[p]:vtx_off[p + 1]], d].copy() for d in range(self.dimension)]
                          for p in range(len(vtx_off) - 1)])

    def getFreeConstraints(self):
        """After solveLinear: the free derivatives d_p of the solve (fetched on the first request).  After setFreeConstraints: what was
        set.  Otherwise (no solve yet, or updateSegmentTimes since): a message and zero vectors."""
        if isinstance(self._free, str):
            vtx_off, masks, vals = self._packed()
            _, _, free = self._c().solve_linear_free_batch_nd(self.N, self.dimension, vtx_off, masks, vals, np.concatenate(self._times),
                                                              self.derivative_to_optimize)
            self._free = free
        if self._free is None:
            print("getFreeConstraints: no linear solution (call solveLinear or setFreeConstraints first)")
            return self._out([[np.zeros(n) for _ in range(self.dimension)] for n in self._counts()[0]])
        return self._out([[row.copy() for row in f] for f in self._free])

    def setFreeConstraints(self, free_constraints):
        """lin_impl.h:519-522: the segments and the cost become A^-1 [fixed ; free] at the current times.  The wrong number of vectors
        or of entries is refused with a message (returns False) and changes nothing."""
        per_problem = [free_constraints] if self._single else list(free_constraints)
        nf = self._counts()[0]
        try:
            free = [np.array([np.asarray(v, dtype=np.float64).reshape(-1) for v in f], dtype=np.float64) for f in per_problem]
        except ValueError:
            free = None
        if free is None or len(free) != len(nf) or any(f.shape != (self.dimension, n) for f, n in zip(free, nf)):
            print("setFreeConstraints: needs %d vectors of n_free entries per problem (n_free = %s)" % (self.dimension, list(nf)))
            return False
        vtx_off, masks, vals = self._packed()
        self.coef, self.cost = self._c().set_free_constraints_batch_nd(self.N, self.dimension, vtx_off, masks, vals, np.concatenate(self._times),
                                                                       free, self.derivative_to_optimize)
        self._seg_off = vtx_off - np.arange(len(vtx_off), dtype=np.int32)
        self._free = free
        return True


class NonlinearOptimizationParameters:
    """nl.h:35-110."""

    kSquaredTime, kRichterTime, kMellingerOuterLoop, kSquaredTimeAndConstraints, kRichterTimeAndConstraints = 0, 1, 2, 3, 4

    def __init__(self):
        self.f_rel = 0.05
        self.x_rel = 0.1
        self.max_iterations = 10
        self.time_alloc_method = 2  # kMellingerOuterLoop (the node's choice, node.cpp:881)
        self.initial_stepsize_rel = 0.1  # nl.h:58
        self.time_penalty = 500.0  # nl.h:73
        self.use_soft_constraints = True  # nl.h:88
        self.soft_constraint_weight = 100.0  # nl.h:91


class DerivativeFreeTimeAllocation:
    """PolynomialOptimizationNonLinear<10>::optimizeTime / optimizeTimeAndFreeConstraints (nl_impl.h:120-157, 429-536) for the
    time-allocation methods 0, 1, 3, 4 (SURVEY.md 8f rank 3).

    The reference hands objectiveFunctionTime / objectiveFunctionTimeAndConstraints to NLopt's LN_BOBYQA (nl_impl.h:68-79); NLopt is
    not vendored, so -- as for LD_LBFGS on the Mellinger path (DESIGN.md, "parity unpinned") -- the objective, bounds, initial steps
    and stopping rules are the reference's and the search itself is ours: a bound-constrained coordinate pattern search whose 2n trial
    points per iteration are evaluated together on the GPU (tg_time_alloc_dfo_batch, here with one problem; TrajectoryGenerator.
    time_alloc_derivative_free runs many).  max_iterations counts those batched iterations, not single evaluations.  Result codes
    as NLopt: 3 ftol_rel, 4 xtol_rel, 5 maxeval.  n_coefficients / dimension: the shape of PolynomialOptimization<N> (N in
    {6, 8, 10, 12}, 1..4 dimensions, derivative_to_optimize 0 .. N/2-1); N = 10 on 4 dimensions runs tg_time_alloc_dfo_batch, every
    other shape tg_time_alloc_dfo_batch_nd.
    """

    kTimeLowerBound = 0.01  # kOptimizationTimeLowerBound (nl.h:143)

    def __init__(self, vertices, times, derivative_to_optimize, parameters, constraints, ctx=None, n_coefficients=N, dimension=D):
        self.ctx = ctx or default_context()
        self.P = parameters
        self.r = derivative_to_optimize
        self.N, self.dimension = n_coefficients, dimension
        self.vertices = list(vertices)
        _, self.mask, self.vals = pack_vertices([vertices], n_coefficients // 2, dimension)
        self.times0 = np.asarray(times, dtype=np.float64)
        self.S = len(self.times0)
        self.constraints = list(constraints)  # (dimension, derivative, value) in the order they were added
        self.with_free = parameters.time_alloc_method in (3, 4)

    def optimize(self):
        vtx_off = np.array([0, len(self.mask)], dtype=np.int32)
        out = _dfo_batch(self.ctx, self.N, self.dimension, vtx_off, self.mask, self.vals, self.times0, _dfo_params(self.ctx, self.P, self.r),
                         self.constraints)
        self.times, self.coef = out["times"], out["coef"]
        self.x = self.times.copy()
        if self.with_free:  # x = the times, then the free derivatives dimension-major (getFreeConstraints, vertex-major slots)
            free = [out["vval"][v, k] for v in range(len(self.mask)) for k in range(self.N // 2) if not (self.mask[v] >> k) & 1]
            self.x = np.concatenate([self.x, np.array(free).reshape(-1, self.dimension).T.reshape(-1)])
        self.cost = float(out["total"][0])
        self.cost_parts = out["parts"][0]
        self.n_iterations = int(out["n_iterations"][0])
        return int(out["code"][0])


def _dfo_batch(ctx, n_coef, dim, vtx_off, masks, vals, times, params, constraints):
    if (n_coef, dim) == (N, D) and params.derivative_to_optimize >= 2:  # the tuned kernels: the same bits
        return ctx.time_alloc_dfo_batch(vtx_off, masks, vals, times, params, constraints)
    return ctx.time_alloc_dfo_batch_nd(n_coef, dim, vtx_off, masks, vals, times, params, constraints)


def _dfo_params(ctx, P, r):
    return ctx.L.default_dfo_params(time_alloc_method=int(P.time_alloc_method), derivative_to_optimize=int(r), max_iterations=int(P.max_iterations),
                                    f_rel=float(P.f_rel), x_rel=float(P.x_rel), initial_stepsize_rel=float(P.initial_stepsize_rel),
                                    time_penalty=float(P.time_penalty), use_soft_constraints=int(bool(P.use_soft_constraints)),
                                    soft_constraint_weight=float(P.soft_constraint_weight))


class PolynomialOptimizationNonLinear:
    """eth_trajectory_generation::PolynomialOptimizationNonLinear<N> (nl.h:147-197).  From waypoints: the node's recipe (N = 10, 4
    dimensions).  From vertices with the Mellinger outer loop: N in {6, 8, 10, 12} on 1..4 dimensions, derivative_to_optimize 2 ..
    N/2-1 -- N = 10 on 4 dimensions on the tuned kernels, every other shape on the general-shape kernels (tg_time_alloc_batch_nd).
    The derivative-free methods take N = 10 on 4 dimensions."""

    def __init__(self, dimension=D, parameters=None, ctx=None, n_coefficients=N):
        if not 1 <= dimension <= D:
            raise ValueError("1 to 4 dimensions")
        if n_coefficients not in (6, 8, 10, 12):
            raise ValueError("N = 6, 8, 10 or 12 coefficients (lin.h:46-55; Polynomial::kMaxN = 12)")
        self.N, self.dimension = n_coefficients, dimension
        self.params = parameters or NonlinearOptimizationParameters()
        self._gen = TrajectoryGenerator(ctx=ctx)
        self._vertices = None
        self._limits = [None] * 9
        self._constraints = []  # (dimension, derivative, value) in the order they were added (inequality_constraints_, nl.h:223)

    def setupFromWaypoints(self, waypoints, initial_state=None, derivative_to_optimize=2):
        """The node builds the vertices from waypoints (node.cpp:923-977); the batched kernel does the same on device."""
        self._wp = np.asarray(waypoints, dtype=np.float64)
        self._init = initial_state
        self._r = derivative_to_optimize
        self._vertices = None
        return True

    def addMaximumMagnitudeConstraint(self, dimension, derivative, maximum_value):  # nl_impl.h:538-565, mapping 355-381
        if derivative not in (1, 2, 3, 4) or dimension not in (0, 1, 2, 3):
            return False
        if derivative <= 3:  # snap limits only enter the soft-constraint objectives
            group = 0 if dimension <= 1 else (1 if dimension == 2 else 2)
            idx = {(0, 1): 0, (1, 1): 1, (0, 2): 2, (1, 2): 3, (0, 3): 4, (1, 3): 5, (2, 1): 6, (2, 2): 7, (2, 3): 8}[(group, derivative)]
            self._limits[idx] = float(maximum_value)
        self._constraints.append((int(dimension), int(derivative), float(maximum_value)))
        return True

    def setupFromVertices(self, vertices, times, derivative_to_optimize):  # nl_impl.h:51-82
        """Vertices (Vertex(dimension)) + initial segment times."""
        self._vertices, self._times0, self._r = list(vertices), np.asarray(times, dtype=np.float64), derivative_to_optimize
        if not 2 <= derivative_to_optimize <= self.N // 2 - 1:
            print("[PolynomialOptimizationNonLinear]: derivative_to_optimize = %d is not supported by the B200 path (2 .. %d)"
                  % (derivative_to_optimize, self.N // 2 - 1))
            return False
        if self.params.time_alloc_method != NonlinearOptimizationParameters.kMellingerOuterLoop and (self.N, self.dimension) != (N, D):
            print("[PolynomialOptimizationNonLinear]: the derivative-free methods take N = 10 on 4 dimensions")
            return False
        return len(self._vertices) == len(self._times0) + 1

    def _params(self):
        return self._gen.params(derivative_to_optimize=self._r, max_evals=self.params.max_iterations, f_rel=self.params.f_rel,
                                x_rel=self.params.x_rel, check_deviation=0,
                                limits=[l if l is not None else 3.4028234663852886e38 for l in self._limits])

    def optimize(self):  # nl_impl.h:89-118 -> returns the nlopt-style code
        if self.params.time_alloc_method != NonlinearOptimizationParameters.kMellingerOuterLoop:
            self._dfo = DerivativeFreeTimeAllocation(self._vertices, self._times0, self._r, self.params, self._constraints, ctx=self._gen.ctx)
            code = self._dfo.optimize()
            self._trajectory = Trajectory(self._dfo.coef, self._dfo.times, self._gen.ctx)
            return code
        if self._vertices is None:  # from waypoints: the node's recipe
            self.result = self._gen.optimize([self._wp], initial_states=None if self._init is None else [self._init], params=self._params())
            self._trajectory = self.result.trajectory(0)
            return int(self.result.results["nlopt_code"][0])
        ctx = self._gen.ctx
        vtx_off, masks, vals = pack_vertices([self._vertices], self.N // 2, self.dimension)
        if (self.N, self.dimension) == (N, D):
            out = ctx.time_alloc_batch(vtx_off, masks, vals, self._times0, self._params())
        else:
            out = ctx.time_alloc_batch_nd(self.N, self.dimension, vtx_off, masks, vals, self._times0, self._params())
        self.info = out
        self._trajectory = Trajectory(out["coef"], out["times"], ctx)
        return int(out["nlopt_code"][0])

    def getTrajectory(self):
        return self._trajectory


class BatchResult:
    def __init__(self, results, out, ctx=None):
        self.results = results
        self.out = out
        self.ctx = ctx  # the generator's context: later evaluate / sample calls on a trajectory stay on its device

    def trajectory(self, p):
        s0, s1 = self.out["seg_off"][p], self.out["seg_off"][p + 1]
        return Trajectory(self.out["coef"][s0:s1], self.out["times"][s0:s1], self.ctx)

    def samples(self, p):
        m0, m1 = self.out["smp_off"][p], self.out["smp_off"][p + 1]
        return self.out["samples"][m0:m1]

    def waypoints(self, p):
        s0, s1 = self.out["seg_off"][p], self.out["seg_off"][p + 1]
        return self.out["wp"][s0 + p: s1 + p + 1]


class DynamicsConstraints:
    """The DynamicsConstraints fields findTrajectory / findTrajectoryFallback read (node.cpp:972-994, 1256-1280)."""

    FIELDS = ("horizontal_speed", "vertical_ascending_speed", "vertical_descending_speed", "horizontal_acceleration",
              "vertical_ascending_acceleration", "vertical_descending_acceleration", "horizontal_jerk", "vertical_ascending_jerk",
              "vertical_descending_jerk", "heading_speed", "heading_acceleration", "heading_jerk")

    def __init__(self, **kw):
        for f in self.FIELDS:
            setattr(self, f, float(kw.pop(f)))
        if kw:
            raise TypeError(f"unknown constraint fields {sorted(kw)}")


class PathRequest:
    """The mrs_msgs::Path fields the path callbacks act on (node.cpp:1847-1902, 2061-2118, 2294-2351).  use_heading and fly_now only
    travel into the outgoing TrajectoryReference (node.cpp:1573-1575); max_execution_time bounds the node's retry loop."""

    def __init__(self, points, use_heading=True, fly_now=False, stop_at_waypoints=False, loop=False, override_constraints=False,
                 override_max_velocity_horizontal=0.0, override_max_acceleration_horizontal=0.0, override_max_jerk_horizontal=0.0,
                 override_max_velocity_vertical=0.0, override_max_acceleration_vertical=0.0, override_max_jerk_vertical=0.0,
                 relax_heading=False, max_deviation_from_path=0.0, dont_prepend_current_state=False, max_execution_time=0.0):
        self.points = np.asarray(points, dtype=np.float64).reshape(-1, 4)
        self.use_heading, self.fly_now, self.stop_at_waypoints, self.loop = use_heading, fly_now, stop_at_waypoints, loop
        self.override_constraints = override_constraints
        self.override_max_velocity_horizontal = override_max_velocity_horizontal
        self.override_max_acceleration_horizontal = override_max_acceleration_horizontal
        self.override_max_jerk_horizontal = override_max_jerk_horizontal
        self.override_max_velocity_vertical = override_max_velocity_vertical
        self.override_max_acceleration_vertical = override_max_acceleration_vertical
        self.override_max_jerk_vertical = override_max_jerk_vertical
        self.relax_heading = relax_heading
        self.max_deviation_from_path = max_deviation_from_path
        self.dont_prepend_current_state = dont_prepend_current_state
        self.max_execution_time = max_execution_time


FLT_MAX = float(np.finfo(np.float32).max)


def resolve_request(req, constraints, base_params, initial_state=None):
    """What a path callback turns one message into before optimize() runs.  Returns (waypoints [V,4], stop_at [V], limits[9],
    max_deviation, prepend_state, overridden).  initial_state: a 14-vector (workloads.init14) or None."""
    wp = req.points.copy()
    if req.loop and len(wp):
        wp = np.vstack([wp, wp[:1]])  # node.cpp:1904-1906
    stop = np.full(len(wp), 1 if req.stop_at_waypoints else 0, np.uint8)
    prepend = initial_state is not None and not req.dont_prepend_current_state  # node.cpp:508-510
    c = constraints
    L = [c.horizontal_speed, min(c.vertical_ascending_speed, c.vertical_descending_speed), c.horizontal_acceleration,
         min(c.vertical_ascending_acceleration, c.vertical_descending_acceleration), c.horizontal_jerk,
         min(c.vertical_ascending_jerk, c.vertical_descending_jerk), c.heading_speed, c.heading_acceleration, c.heading_jerk]
    overridden = False
    if req.override_constraints:
        o_jv = req.override_max_jerk_horizontal  # the callbacks copy the HORIZONTAL jerk into the vertical slot (node.cpp:1856, 2070, 2303)
        can_change = True
        if prepend:  # node.cpp:1002-1009
            s = np.asarray(initial_state, dtype=np.float64)
            v, a, j = s[2:6], s[6:10], s[10:14]
            can_change = (math.hypot(v[0], v[1]) < req.override_max_velocity_horizontal and math.hypot(a[0], a[1]) < req.override_max_acceleration_horizontal
                          and math.hypot(j[0], j[1]) < req.override_max_jerk_horizontal and abs(v[2]) < req.override_max_velocity_vertical
                          and abs(a[2]) < req.override_max_acceleration_vertical and abs(j[2]) < o_jv)
        if can_change:
            L[0], L[2], L[4] = req.override_max_velocity_horizontal, req.override_max_acceleration_horizontal, req.override_max_jerk_horizontal
            L[1], L[3], L[5] = req.override_max_velocity_vertical, req.override_max_acceleration_vertical, o_jv
            overridden = True
    if req.relax_heading:
        L[6] = L[7] = L[8] = FLT_MAX  # node.cpp:1030-1034
    max_dev = req.max_deviation_from_path if req.max_deviation_from_path > 0 else base_params.max_deviation  # node.cpp:1875-1879
    return wp, stop, L, max_dev, prepend, overridden


class TrajectoryGenerator:
    """The numeric core of MrsTrajectoryGeneration::optimize() / findTrajectory() (node.cpp:620-851, 857-1209) for batches."""

    def __init__(self, ctx=None, device=0):
        self.ctx = ctx or (default_context() if device == 0 else Context(Library(), device))

    def params(self, **kw):
        return self.ctx.L.default_params(**kw)

    def optimize(self, paths, stop_at=None, initial_states=None, params=None):
        """paths: list of [V_p, 4] arrays.  initial_states: optional list of 14-vectors (workloads.init14)."""
        wp_off = np.zeros(len(paths) + 1, dtype=np.int32)
        wp_off[1:] = np.cumsum([len(p) for p in paths])
        wp = np.concatenate([np.asarray(p, dtype=np.float64).reshape(-1, 4) for p in paths])
        stop = None if stop_at is None else np.concatenate([np.asarray(s, dtype=np.uint8) for s in stop_at])
        init = None if initial_states is None else np.stack([np.asarray(i, dtype=np.float64) for i in initial_states])
        res, _ = self.ctx.optimize_batch(wp_off, wp, stop, init, params)
        return BatchResult(res, self.ctx.fetch_outputs(), self.ctx)

    def optimize_requests(self, requests, constraints, initial_states=None, params=None):
        """Many path messages at once: requests whose resolved limits / deviation bound / state use agree share one batch call.
        Returns a list of (BatchResult, index inside it), one per request, plus the resolved tuples."""
        base = params or self.params()
        resolved = [resolve_request(r, constraints, base, None if initial_states is None else initial_states[i]) for i, r in enumerate(requests)]
        groups = {}
        for i, (wp, stop, L, max_dev, prepend, _) in enumerate(resolved):
            groups.setdefault((tuple(L), max_dev, prepend), []).append(i)
        placed = [None] * len(requests)
        for (L, max_dev, prepend), members in groups.items():
            p = self.ctx.L.copy_params(base)
            for k in range(9):
                p.limits[k] = L[k]
            p.max_deviation = max_dev
            br = self.optimize([resolved[i][0] for i in members], [resolved[i][1] for i in members],
                               [initial_states[i] for i in members] if prepend else None, p)
            for k, i in enumerate(members):
                placed[i] = (br, k)
        return placed, resolved

    def time_alloc_derivative_free(self, vertex_lists, times_list, parameters, constraints=(), derivative_to_optimize=2, n_coefficients=N,
                                   dimension=D):
        """PolynomialOptimizationNonLinear<N>::optimize() with a derivative-free method (parameters.time_alloc_method 0, 1, 3 or 4) for
        many problems in one call.  vertex_lists: one list of Vertex(dimension) per problem; times_list: their initial segment times;
        constraints: (dimension, derivative, value) added to every problem; n_coefficients in {6, 8, 10, 12}, dimension 1..4.  Returns
        ([Trajectory], codes[B])."""
        vtx_off, masks, vals = pack_vertices(vertex_lists, n_coefficients // 2, dimension)
        times = np.concatenate([np.asarray(t, dtype=np.float64) for t in times_list])
        out = _dfo_batch(self.ctx, n_coefficients, dimension, vtx_off, masks, vals, times, _dfo_params(self.ctx, parameters, derivative_to_optimize),
                         list(constraints))
        seg_off = vtx_off - np.arange(len(vtx_off), dtype=np.int32)
        trajs = [Trajectory(out["coef"][seg_off[p]:seg_off[p + 1]], out["times"][seg_off[p]:seg_off[p + 1]], self.ctx) for p in range(len(vertex_lists))]
        return trajs, out["code"]

    def findTrajectory(self, waypoints, initial_state=None, params=None):
        """One findTrajectory pass without the deviation loop (node.cpp:857-1209)."""
        p = params or self.params()
        p.check_deviation = 0
        r = self.optimize([waypoints], initial_states=None if initial_state is None else [initial_state], params=p)
        return r.samples(0) if r.results["success"][0] else None
