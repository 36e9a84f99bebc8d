/*
 * tg_b200.h -- C ABI of libtg_b200.so, the B200-native (sm_100a) batched polynomial trajectory optimiser.
 *
 * Drop-in boundary for the hot path of ctu-mrs/mrs_uav_trajectory_generation (SURVEY.md section 8b).  The
 * reference has no FFI around this path: it is in-process C++ (static library + header templates, namespace
 * eth_trajectory_generation) called from exactly one place, MrsTrajectoryGeneration::findTrajectory /
 * optimize().  Each entry point below names the reference interface it replaces (file:line under the reference
 * root).  INTEGRATION.md shows the C++ shim (include/eth_trajectory_generation_b200.hpp) with the reference's
 * class names that forwards to these functions, and the ctypes binding used by the tests.
 *
 * Conventions
 *   - plain pointers and sizes only; caller owns every host buffer; the library owns device workspaces in tg_ctx;
 *     no pointer is retained after a call returns.
 *   - every function returns TG_OK (0) or a negative TG_ERR_* code; tg_last_error() gives the text.  Nothing throws
 *     or aborts across the ABI (the reference's CHECK macros print and continue, eth/misc.h:6-38); per-problem
 *     outcomes are reported in tg_result.
 *   - a tg_ctx is bound to one CUDA device and one stream; calls on one ctx are serialised by the caller, several
 *     ctxs (one per GPU / host thread) may run concurrently.  There is NO CPU fallback: creating a ctx fails
 *     loudly without a CUDA device.
 *   - arithmetic: IEEE binary64 everywhere (the reference is fp64 Eigen), compiled without FMA contraction.
 *
 * Ragged batch layout: problem p owns waypoints wp_off[p] .. wp_off[p+1]-1 (V_p = count, S_p = V_p - 1 segments).
 *   waypoint: 4 doubles x, y, z, heading.   coefficients: per segment [4 dims][10], increasing powers
 *   (eth/polynomial.h:35-37).   samples: 4 doubles x, y, z, heading as getTrajectoryReference emits them
 *   (src/mrs_trajectory_generation.cpp:1578-1602).
 */
#ifndef TG_B200_H_
#define TG_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TG_OK 0
#define TG_ERR_NO_DEVICE (-1)
#define TG_ERR_CUDA (-2)
#define TG_ERR_INVALID (-3)
#define TG_ERR_NO_RESULT (-4)
#define TG_ERR_CAPACITY (-5)

typedef struct tg_ctx tg_ctx;

/* Parameters of one batch call.  Defaults (tg_default_params) are the reference's production constants
 * (SURVEY.md section 5): config/private/trajectory_generation.yaml:4-11, config/public/trajectory_generation.yaml:11-36,
 * src/mrs_trajectory_generation.cpp:884-896. */
typedef struct tg_params {
  int derivative_to_optimize;   /* 2 acceleration (default), 3 jerk, 4 snap  (node.cpp:904-919) */
  int max_evals;                /* NLopt maxeval = max_iterations (10) */
  double f_rel, x_rel;          /* 0.05, 0.1 (node.cpp:884-885) */
  double limits[9];             /* v_h, v_v, a_h, a_v, j_h, j_v, v_heading, a_heading, j_heading (node.cpp:981-1038) */
  double dt;                    /* sampling_dt 0.2 s */
  int check_deviation;          /* check_trajectory_deviation/enabled */
  double max_deviation;         /* 0.05 m */
  int max_deviation_iters;      /* 6 */
  int first_segment_checked;    /* max_deviation_first_segment_ (node.cpp:874-878) */
  double max_len_factor, min_len_factor; /* 3.0, 0.33 (node.cpp:1178-1199) */
  int run_time_alloc;           /* 1: full findTrajectory; 0: linear solve at the Euclidean times + sampling */
  int override_heading_atan2;   /* getTrajectoryReference: heading of a sample = direction to the next one (node.cpp:1586-1599); default 0 */
} tg_params;

/* Per-problem outcome of tg_optimize_batch. */
typedef struct tg_result {
  int status;          /* 0 ok, 1 optimiser code rejected (node.cpp:1138-1149), 2 too long, 3 too short (node.cpp:1178-1199), 4 sampling failed, 5 fewer than two waypoints ("the path is empty", node.cpp:676-681),
                          6 a non-finite waypoint or initial-state value (the callbacks' checkNaN, node.cpp:1896-1900; host inputs only) */
  int success;         /* optimize() produced a trajectory */
  int nlopt_code;      /* NLopt-style result code of the last findTrajectory (1,3,4,5 success codes, -1 generic failure) */
  int n_evals;         /* objective evaluations of the last findTrajectory (OptimizationInfo::n_iterations) */
  int rounds;          /* subdivision rounds executed (re-solves) */
  int safe;            /* last validation verdict (validateTrajectorySpatial) */
  int n_waypoints;     /* final vertex count */
  int n_samples;       /* final sample count */
  int n_scale_passes;  /* passes of scaleSegmentTimesToMeetConstraints in the last findTrajectory */
  int overflow;        /* reserved (always 0: outputs are sized by the library) */
  double max_dev;      /* last measured path deviation [m] */
  double final_cost;   /* OptimizationInfo::cost_trajectory: objective at the last point the optimiser evaluated (nl_impl.h:646) */
  double baca_total;   /* sum of estimateSegmentTimesBaca (node.cpp:1048-1056) */
  long long total_solves, total_root_calls, total_evals; /* reference-equivalent work over all rounds */
} tg_result;

/* Library / context ------------------------------------------------------------------------------------------------ */
const char* tg_version(void);
void tg_default_params(tg_params* p);
/* Creates a context on CUDA device `device` (its own stream).  Fails with TG_ERR_NO_DEVICE when no GPU is usable. */
int tg_ctx_create(int device, tg_ctx** out);
void tg_ctx_destroy(tg_ctx* ctx);
const char* tg_last_error(const tg_ctx* ctx);
/* counters[16] (9 used): kernel launches, linear solves, objective evaluations, root finds the REFERENCE would run for the
 * same work, segment setups, samples, solves inside the time-allocation loop, launches of that solve kernel, Jenkins-Traub
 * runs actually launched (after the exact pruning of tg_bound.cuh); cumulative since the context was created. */
int tg_get_counters(const tg_ctx* ctx, long long* counters);
/* flops[4]: ALGORITHMIC flops (SURVEY.md 8(d) formula, DESIGN.md) of the launched work: solve kernels (assembly, banded
 * factorisation, back substitution), segment-setup kernels, sampling, coefficient + cost kernel -- the numerators of the
 * roofline report. */
int tg_get_flop_counters(const tg_ctx* ctx, double* flops);
/* Milliseconds of device time (CUDA events on the context's stream) spent inside the last batch call. */
double tg_last_device_ms(const tg_ctx* ctx);

/* The hot path --------------------------------------------------------------------------------------------------------
 * tg_optimize_batch = for every problem: MrsTrajectoryGeneration::optimize()'s numeric core
 *   (src/mrs_trajectory_generation.cpp:620-851): findTrajectory (857-1209: vertex recipe 923-977, estimateSegmentTimes
 *   + Baca 1045-1056, PolynomialOptimizationNonLinear<10>::setupFromVertices / addMaximumMagnitudeConstraint x12 /
 *   optimize 1063-1083, acceptance 1138-1149, sampleWholeTrajectory 1169, length check 1178-1199), then
 *   validateTrajectorySpatial (1401-1455) and midpoint subdivision + re-solve (729-785) up to max_deviation_iters.
 * init14 (optional, [B][14]): {present, heading, vel[4], acc[4], jerk[4]} = the TrackerCommand fields read at
 *   node.cpp:925-957; NULL means "no initial state" for every problem (dont_prepend_current_state).
 * inputs_on_device != 0: wp, stop_at, init14 are device pointers on the context's device (wp_off stays on the host).
 * results: [B] host.  totals[2]: total segments and total samples of the final trajectories (sizes for tg_fetch_outputs). */
int tg_optimize_batch(tg_ctx* ctx, int B, const int* wp_off, const double* wp, const uint8_t* stop_at, const double* init14,
                      const tg_params* params, int inputs_on_device, tg_result* results, long long* totals);
/* tg_optimize_batch with the samples of every path (what getTrajectoryReference hands to the tracker, node.cpp:1560-1606) copied to
 *   host memory WHILE the later validation / subdivision rounds of optimize() (node.cpp:729-785) still run: a path's samples are final
 *   as soon as its own validation passes, and most paths finish in the first rounds.  samples_out: samples_cap rows of 4 doubles
 *   (x y z heading) in host memory -- page-locked memory for a real overlap --; paths are stored in COMPLETION order:
 *   smp_begin[p] = first row of path p, results[p].n_samples rows.  TG_ERR_CAPACITY when samples_cap < totals[1] (the batch
 *   result is complete and can be read with tg_fetch_outputs).  Everything else as tg_optimize_batch. */
int tg_optimize_batch_streamed(tg_ctx* ctx, int B, const int* wp_off, const double* wp, const uint8_t* stop_at, const double* init14,
                               const tg_params* params, int inputs_on_device, tg_result* results, long long* totals, double* samples_out,
                               long long samples_cap, long long* smp_begin);
/* Copies the outputs of the last tg_optimize_batch to host buffers (any pointer may be NULL):
 *   seg_off[B+1] (segment offsets; vertex offset of problem p = seg_off[p] + p), wp[(totS+B)*4] final waypoint lists,
 *   times[totS], coef[totS*40], smp_off[B+1], samples[totM*4].
 * Replaces PolynomialOptimization::getSegments (lin.h:177), getTrajectory (nl.h:181) and getTrajectoryReference
 * (node.cpp:1560-1606) for the whole batch. */
int tg_fetch_outputs(tg_ctx* ctx, int* seg_off, double* wp, double* times, double* coef, int* smp_off, double* samples);

/* Pieces of the path with the reference's class-level meaning --------------------------------------------------------
 * tg_solve_linear_batch = PolynomialOptimization<10>::setupFromVertices + solveLinear + getSegments + computeCost
 *   (lin_impl.h:61-106, 340-373, 263-282, 127-141) for B independent problems.
 *   vtx_off[B+1] vertex offsets; vmask[totV] bit k set = derivative k fixed (Vertex::addConstraint, eth/vertex.cpp:134-137);
 *   vval[totV][5][4] fixed values; times[totS]; r = derivative_to_optimize.  Outputs: coef[totS*40], cost[B]. */
int tg_solve_linear_batch(tg_ctx* ctx, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, const double* times, int r,
                          double* coef, double* cost);
/* tg_time_alloc_batch = PolynomialOptimizationNonLinear<10>::setupFromVertices + addMaximumMagnitudeConstraint x12 +
 *   optimize() + getTrajectory (nl.h:147-197; nl_impl.h:51-82, 538-565, 89-118 -> optimizeTimeMellingerOuterLoop 159-234 with
 *   the objective / forward-difference gradient of 256-333 -> scaleSegmentTimesWithViolation 335-427) for B problems given
 *   as vertices.  times[totS]: initial segment times in, allocated + stretched times out.  params: derivative_to_optimize,
 *   max_evals, f_rel, x_rel and limits are read.  Outputs (any may be NULL): coef[totS*40] of the final solve,
 *   nlopt_code[B] (NLopt-style result code), n_evals[B] (OptimizationInfo::n_iterations), n_scale_passes[B], final_cost[B]. */
int tg_time_alloc_batch(tg_ctx* ctx, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times,
                        const tg_params* params, double* coef, int* nlopt_code, int* n_evals, int* n_scale_passes, double* final_cost);
/* tg_sample_batch = sampleWholeTrajectory (eth/trajectory_sampling.cpp:119-124, 49-104) for B trajectories given as
 *   seg_off[B+1], coef, times.  Two-call convention: with samples == NULL only counts[B] is filled.
 *   samples: [sum counts][4] (x y z heading); full (optional): [sum counts][19] = p4 v4 a4 j3 s3 yaw. */
int tg_sample_batch(tg_ctx* ctx, int B, const int* seg_off, const double* coef, const double* times, double dt, int* counts,
                    double* samples, double* full);
/* tg_evaluate_batch = Trajectory::evaluate(t, derivative) (eth/trajectory.cpp:55-87) at n query times of ONE trajectory.
 *   out: [n][4]; ok[n] = 0 where t is past the end (the reference logs and returns zeros). */
int tg_evaluate_batch(tg_ctx* ctx, int S, const double* coef, const double* times, int n, const double* t, int derivative, double* out,
                      uint8_t* ok);
/* tg_extrema_batch = Trajectory::computeMaxDerivatives{Horizontal,Vertical,Heading}(.., seg) (eth/trajectory.cpp:422-565)
 *   for totS segments: maxima[totS][9] = hor v,a,j ; ver v,a,j ; heading v,a,j. */
int tg_extrema_batch(tg_ctx* ctx, int totS, const double* coef, const double* times, double* maxima);
/* tg_max_magnitude_batch = PolynomialOptimization<N>::computeMaximumOfMagnitude(derivative, nullptr) (lin_impl.h:477-508,
 *   used by evaluateMaximumMagnitudeConstraint, nl_impl.h:724-738) for B trajectories given as seg_off[B+1], coef, times:
 *   the Extremum {time (inside its segment), value, segment_idx} of the magnitude of the derivative over ALL four
 *   dimensions (the constraint's `dimension` is ignored by the reference, lin_impl.h:407-409).  derivative in 1..4. */
int tg_max_magnitude_batch(tg_ctx* ctx, int B, const int* seg_off, const double* coef, const double* times, int derivative, double* value,
                           double* time, int* segment_idx);
/* tg_scale_times_batch = Trajectory::scaleSegmentTimesToMeetConstraints (eth/trajectory.cpp:598-692), in place on
 *   coef/times; passes[B], within[B]. */
int tg_scale_times_batch(tg_ctx* ctx, int B, const int* seg_off, double* coef, double* times, const double* limits9, int* passes,
                         uint8_t* within);
/* General shape: the reference's classes are templates over the number of coefficients N (lin.h:46-55: even; Polynomial::kMaxN = 12,
 *   eth/polynomial.h:45-48) and take the dimension D at run time (Vertex(D), PolynomialOptimization<N>(D), Trajectory::D()).
 *   The three entry points below are tg_solve_linear_batch / tg_evaluate_batch / tg_sample_batch for N in {6, 8, 10, 12},
 *   D in 1..4 and derivative_to_optimize r in 0 .. N/2-1 (lin_impl.h:61-70 accepts exactly that range):
 *   vmask bit k (k < N/2) = derivative k fixed; vval[totV][N/2][D]; coef[totS][D][N]; out[n][D].
 *   tg_sample_batch_nd needs D >= 3 as sampleTrajectoryInRange does (eth/trajectory_sampling.cpp:58-61); with D = 3 the heading
 *   entries of samples / full are zero (the reference leaves the orientation at identity).
 *   The tuned kernels serve N = 10, D = 4, r in 2..4 (the node's only shape, node.cpp:902, 1063) through the entry points above;
 *   these go through the general-shape kernels of csrc/tg_generic.cuh for every shape, N = 10 included. */
int tg_solve_linear_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, const double* times,
                             int r, double* coef, double* cost);
int tg_evaluate_batch_nd(tg_ctx* ctx, int N, int D, int S, const double* coef, const double* times, int n, const double* t, int derivative,
                         double* out, uint8_t* ok);
int tg_sample_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* seg_off, const double* coef, const double* times, double dt, int* counts,
                       double* samples, double* full);
/* Free and fixed constraints of PolynomialOptimization<N> (lin_impl.h:183-257, 513-522) on the same shapes, inputs as in
 *   tg_solve_linear_batch_nd.  The free derivatives d_p of a problem are dimension-major: D vectors of n_free entries, and within a
 *   dimension vertex-major with the derivative ascending; n_free = the clear mask bits below N/2 over the problem's vertices,
 *   n_fixed = (S+1)*N/2 - n_free.  free[] holds the problems' D*n_free blocks one after the other, in problem order.
 * tg_solve_linear_free_batch_nd = setupFromVertices + solveLinear + getFreeConstraints + getSegments + computeCost
 *   (lin_impl.h:340-373, 513-516, 263-282, 127-141): coef[totS][D][N] and cost[B] carry tg_solve_linear_batch_nd's bits, free the
 *   d_p the solve found.  Any output may be NULL.
 * tg_set_free_constraints_batch_nd = setFreeConstraints + getSegments + computeCost (lin_impl.h:519-522 -> 263-282, 127-141): the
 *   coefficients A^-1 [fixed ; free] of every (segment, dimension) from the given free[] and the cost 1/2 sum c^T Q c in (segment,
 *   dimension) order, with no solve; K candidate free vectors of one problem are K problems.  Non-finite free values are not
 *   refused and propagate.  coef and cost may be NULL.  Setting the free derivatives a solve returned reproduces its coef and cost
 *   bit for bit.
 *   Both refuse with TG_ERR_INVALID, writing no output, N outside {6, 8, 10, 12}, D outside 1..4, r outside 0 .. N/2-1, B < 1
 *   and a problem with fewer than two vertices. */
int tg_solve_linear_free_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval,
                                  const double* times, int r, double* coef, double* cost, double* free);
int tg_set_free_constraints_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval,
                                     const double* times, int r, const double* free, double* coef, double* cost);
/* The nonlinear half on the same shapes, with the contracts of the N = 10 entry points above (coef[totS][D][N] everywhere):
 *   tg_extrema_batch_nd        = tg_extrema_batch: Trajectory::computeMaxDerivatives{Horizontal,Vertical,Heading}
 *                                (eth/trajectory.cpp:422-565) -> maxima[totS][9]; a missing dimension has zero maxima.
 *   tg_max_magnitude_batch_nd  = tg_max_magnitude_batch: PolynomialOptimization<N>::computeMaximumOfMagnitude (lin_impl.h:477-508)
 *                                over the D dimensions; derivative in 1..4.
 *   tg_scale_times_batch_nd    = tg_scale_times_batch: Trajectory::scaleSegmentTimesToMeetConstraints (eth/trajectory.cpp:598-692)
 *                                in place on coef / times.
 *   tg_time_alloc_batch_nd     = tg_time_alloc_batch: PolynomialOptimizationNonLinear<N>::setupFromVertices + optimize() with the
 *                                Mellinger outer loop (nl_impl.h:159-234, 256-333) + scaleSegmentTimesWithViolation (335-427) +
 *                                getTrajectory; vval[totV][N/2][D]; derivative_to_optimize in 0 .. N/2-1.
 *   Every (segment, quantity) maximum is found by exact root finding (no Bernstein pruning: that is built for N = 10), and a
 *   Mellinger evaluation is S+1 dense solves per running problem; both give the tuned kernels' bits at N = 10, D = 4. */
int tg_extrema_batch_nd(tg_ctx* ctx, int N, int D, int totS, const double* coef, const double* times, double* maxima);
int tg_max_magnitude_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* seg_off, const double* coef, const double* times, int derivative,
                              double* value, double* time, int* segment_idx);
int tg_scale_times_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* seg_off, double* coef, double* times, const double* limits9,
                            int* passes, uint8_t* within);
int tg_time_alloc_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times,
                           const tg_params* params, double* coef, int* nlopt_code, int* n_evals, int* n_scale_passes, double* final_cost);
/* tg_sweep_costs (BASELINE config 5) = updateSegmentTimes + solveLinear + computeCost for K candidate time vectors
 *   of ONE problem (lin_impl.h:288-304, 340-373, 127-141).  cand[K][S] host (or device when cand_on_device).
 *   costs (optional) [K] host; best_index / best_cost = argmin (first minimum). */
int tg_sweep_costs(tg_ctx* ctx, int V, const uint8_t* vmask, const double* vval, int r, long long K, const double* cand,
                   int cand_on_device, double* costs, long long* best_index, double* best_cost);

/* tg_sweep_best (SURVEY.md 8b, BASELINE config 5 on several GPUs of one box): the K candidates are cut into n_ctx contiguous shards,
 *   shard g runs tg_sweep_costs on ctxs[g] (one context per device, one host thread per context), and the first minimum of the whole
 *   list is returned: best_index (global), best_cost, best_times[S] (optional).  No device-to-device exchange: each shard returns
 *   16 bytes.  Across processes (one rank per GPU) the same reduction is one all_gather of (cost, index, S times) per rank:
 *   mrs_uav_trajectory_generation_b200/sharding.py sweep_best_distributed (NCCL). */
int tg_sweep_best(tg_ctx* const* ctxs, int n_ctx, int V, const uint8_t* vmask, const double* vval, int r, long long K, const double* cand,
                  long long* best_index, double* best_cost, double* best_times);

/* tg_objective_batch (SURVEY.md 8f rank 3) = the objective functions of the time-allocation methods other than Mellinger's,
 *   PolynomialOptimizationNonLinear<N>::objectiveFunctionTime (nl_impl.h:567-614; methods 0 kSquaredTime, 1 kRichterTime) and
 *   objectiveFunctionTimeAndConstraints (nl_impl.h:651-722; methods 3, 4), with evaluateMaximumMagnitudeAsSoftConstraint
 *   (nl_impl.h:740-762) over computeMaximumOfMagnitude, at K candidate vectors of ONE problem -- the batch a derivative-free
 *   optimiser (the reference drives NLopt LN_BOBYQA, nl_impl.h:68-79) evaluates per iteration.  x[K][nvar]: S segment times,
 *   then for methods 3/4 the free derivatives, dimension-major (4 x n_free) as getFreeConstraints returns them.
 *   total[K] = cost_trajectory + cost_time + cost_soft_constraints; parts (optional) [K][3] = the three terms;
 *   coef (optional) [K][S][4][10] = the segments of every candidate (getSegments after the objective call). */
int tg_objective_batch(tg_ctx* ctx, int V, const uint8_t* vmask, const double* vval, int r, int time_alloc_method, long long K, const double* x,
                       int nvar, double time_penalty, int use_soft_constraints, double soft_constraint_weight, int n_constraints,
                       const int* con_derivative, const double* con_value, double* total, double* parts, double* coef);

/* tg_time_alloc_dfo_batch = PolynomialOptimizationNonLinear<10>::optimize() with the derivative-free time-allocation methods
 *   (optimizeTime / optimizeTimeAndFreeConstraints, nl_impl.h:120-157, 429-536) for B problems in one call.  The reference hands
 *   the objective to NLopt's LN_BOBYQA; here the objective (tg_objective_batch's, bit for bit), the bounds
 *   (kOptimizationTimeLowerBound; setFreeEndpointDerivativeHardConstraints, nl_impl.h:764-805, including its counter that only
 *   advances for derivatives <= derivative_to_optimize), the initial steps (nl_impl.h:488-495) and the stopping rules are the
 *   reference's, and the search is a bound-constrained coordinate pattern search (2n candidates per iteration; first strict
 *   minimum accepted when it improves, every step halved otherwise; codes 3 ftol_rel, 4 xtol_rel, 5 max_iterations).  Methods 3, 4
 *   start the free derivatives at the linear solution of the initial times (nl_impl.h:436-462).
 *   Inputs as tg_time_alloc_batch: vtx_off[B+1], vmask[totV], vval[totV][5][4]; times[totS] initial times in, allocated out.
 *   The constraints (addMaximumMagnitudeConstraint, nl_impl.h:538-565) are shared by every problem: at most 16, dimension 0..3,
 *   derivative 1..4, value != 0.  Outputs (any may be NULL): coef[totS][4][10] at the final point; vval_out[totV][5][4] (methods 3, 4)
 *   the fixed values with every free slot at its final variable; code[B]; n_iterations[B]; total[B] the best objective;
 *   parts[B][3] = {cost_trajectory, cost_time, cost_soft_constraints} at the final point.  TG_ERR_INVALID, with no output written,
 *   for B < 1, a problem with fewer than two vertices, a method other than 0, 1, 3, 4, derivative_to_optimize outside 2..4 or an
 *   invalid constraint.  max_iterations <= 0 runs no iteration (code 5). */
typedef struct tg_dfo_params {
  int time_alloc_method;          /* 0, 1, 3 or 4 */
  int derivative_to_optimize;     /* 2 .. 4 */
  int max_iterations;             /* batched search iterations (10) */
  double f_rel, x_rel, initial_stepsize_rel;  /* 0.05, 0.1, 0.1 */
  double time_penalty;            /* 500 */
  int use_soft_constraints;       /* 1 */
  double soft_constraint_weight;  /* 100 */
} tg_dfo_params;
void tg_default_dfo_params(tg_dfo_params* p);
int tg_time_alloc_dfo_batch(tg_ctx* ctx, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times,
                            const tg_dfo_params* params, int n_constraints, const int* con_dimension, const int* con_derivative,
                            const double* con_value, double* coef, double* vval_out, int* code, int* n_iterations, double* total, double* parts);

/* The derivative-free time allocation for PolynomialOptimization<N>, N in {6, 8, 10, 12}, D in 1..4 dimensions:
 * tg_objective_batch_nd      = tg_objective_batch over N coefficients and D dimensions: vval[V][N/2][D]; x[K][nvar], nvar = S
 *                              (methods 0, 1) or S + D * n_free (methods 3, 4; the free derivatives dimension-major, D x n_free,
 *                              the layout of tg_solve_linear_free_batch_nd); coef (optional) [K][S][D][N].
 * tg_time_alloc_dfo_batch_nd = tg_time_alloc_dfo_batch over N coefficients and D dimensions: the same search, bounds, steps and
 *                              codes, with variables for the D dimensions only (n = S or S + D * n_free); vval, vval_out
 *                              [totV][N/2][D], coef[totS][D][N]; the other outputs as tg_time_alloc_dfo_batch.  A constraint is
 *                              shared by every problem as there (dimension 0..3: a bound that lands outside the variables is
 *                              dropped); its magnitude is taken over the D dimensions.
 *   derivative_to_optimize (r) is 0 .. N/2-1 in both.  Both refuse with TG_ERR_INVALID, writing no output, N outside {6, 8, 10, 12},
 *   D outside 1..4, r outside 0 .. N/2-1, a method other than 0, 1, 3, 4, K or B < 1, a problem with fewer than two vertices, more
 *   than 16 constraints or one with a dimension outside 0..3, a derivative outside 1..4 or a zero value, and a wrong nvar.
 *   Non-finite inputs are not refused and propagate. */
int tg_objective_batch_nd(tg_ctx* ctx, int N, int D, int V, const uint8_t* vmask, const double* vval, int r, int time_alloc_method, long long K,
                          const double* x, int nvar, double time_penalty, int use_soft_constraints, double soft_constraint_weight,
                          int n_constraints, const int* con_derivative, const double* con_value, double* total, double* parts, double* coef);
int tg_time_alloc_dfo_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times,
                               const tg_dfo_params* params, int n_constraints, const int* con_dimension, const int* con_derivative,
                               const double* con_value, double* coef, double* vval_out, int* code, int* n_iterations, double* total,
                               double* parts);

/* The steps either side of the path (SURVEY.md 8f ranks 1-2), batched, one path per thread --------------------------------
 * tg_preprocess_paths = MrsTrajectoryGeneration::preprocessPath (src/mrs_trajectory_generation.cpp:431-500): optional path
 *   straightener (config/public/trajectory_generation.yaml:20-23) then the min_waypoint_distance filter (:27).
 *   Outputs: out_count[B]; out_wp / out_stop_at have the INPUT layout (problem p writes out_count[p] waypoints from wp_off[p]).
 * tg_fallback_sample_batch = findTrajectoryFallback (node.cpp:1215-1395): constant-velocity samples along the polyline with
 *   estimateSegmentTimesBaca times; limits9 already carry fallback_sampling/speed_factor and accel_factor (yaml:47-54);
 *   stopping_time = fallback_sampling/stopping_time.  Two-call convention: samples == NULL fills counts[B] only.
 *   samples: [sum counts][4] = x y z heading as getTrajectoryReference emits them.
 * tg_waypoint_idxs_batch = getWaypointInTrajectoryIdxs (node.cpp:1461-1499): for every path the sample indices at which the
 *   trajectory passes its waypoints (chord within 0.1 m).  idxs has the waypoint layout (problem p writes counts[p] entries
 *   from wp_off[p]). */
int tg_preprocess_paths(tg_ctx* ctx, int B, const int* wp_off, const double* wp, const uint8_t* stop_at, double min_waypoint_distance,
                        int straightener_enabled, double straightener_max_deviation, double straightener_max_hdg_deviation, int* out_count,
                        double* out_wp, uint8_t* out_stop_at);
int tg_fallback_sample_batch(tg_ctx* ctx, int B, const int* wp_off, const double* wp, const uint8_t* stop_at, const double* limits9, double dt,
                             double stopping_time, int* counts, double* samples);
int tg_waypoint_idxs_batch(tg_ctx* ctx, int B, const int* smp_off, const double* samples, const int* wp_off, const double* wp, int* counts, int* idxs);

/* Measurement hooks (bench.py) ------------------------------------------------------------------------------------------
 * tg_set_profiling: when on, every kernel launch is bracketed by CUDA events on the context's stream and accumulated
 *   per kernel (serialises the host; never enabled inside a timed region).  tg_get_profile returns the table.
 * tg_measure_fp64_peak: TFLOP/s of the FP64 pipe; mode 0 = DFMA chains, mode 1 = DMUL+DADD (the -fmad=false mix the
 *   product kernels issue).  This is the roofline denominator for this path. */
int tg_set_profiling(tg_ctx* ctx, int on);
int tg_get_profile(tg_ctx* ctx, int cap, char* names, int names_cap, double* ms, long long* launches, long long* items);
double tg_measure_fp64_peak(tg_ctx* ctx, int mode);

/* Test hook: the tolerance of scaleSegmentTimesToMeetConstraints' global check (1e-3, eth/trajectory.cpp:604).  With the
 * reference's value a second pass practically never happens; tests lower it to drive the multi-pass path. */
int tg_test_set_scale_tolerance(tg_ctx* ctx, double tolerance);

/* Test hook: the device Jenkins-Traub root finder = findRootsJenkinsTraub (eth/rpoly/rpoly_ak1.cpp:76-120) on n arbitrary
 * polynomials.  coeffs[n][16]: increasing powers, ncoef[n] <= 16 of them used; re / im [n][16]: the zeros in the order the
 * reference stores them (zeros at the origin first, then as found); nroots[n]: how many (fewer than the degree = no
 * convergence after 20 shifts, as in the reference).  The production path only ever reads maxima at these zeros. */
int tg_test_find_roots_batch(tg_ctx* ctx, int n, const double* coeffs, const int* ncoef, double* re, double* im, int* nroots);

/* Host-side evaluation of the deterministic math layer (include/tg_detmath.h), for tests:
 *   fn 0 log, 1 exp, 2 sin, 3 cos, 4 atan2(x, y), 5 cbrt, 6 pow(x, (int)y). */
double tg_detmath_eval(int fn, double x, double y);

#ifdef __cplusplus
}
#endif

#endif /* TG_B200_H_ */
