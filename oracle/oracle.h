/*
 * oracle/oracle.h -- CPU restatement of the reference hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * This directory restates, in plain Eigen-free C++17, the algorithm that
 * ctu-mrs/mrs_uav_trajectory_generation runs for one path (SURVEY.md section 8a).
 * It is the checker the CUDA library is compared against; nothing in the
 * product package (mrs_uav_trajectory_generation_b200/) includes, links or calls it.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load liboracle.so.
 *
 * PARITY STATUS: pinned to the reference's own SOURCES, bit for bit, for everything the reference's repository contains; unpinned
 * only where the reference calls third-party BINARIES that are not in its tree.
 *   - oracle/Makefile target _ref/libref_eth.so compiles, unmodified and from where they lie in a checkout of the reference
 *     ($TG_REFERENCE_DIR, else BASELINE.json's reference_path, /root/reference),
 *     src/eth_trajectory_generation/{motion_defines,polynomial,segment,trajectory,trajectory_sampling,vertex,timing,
 *     rpoly/rpoly_ak1}.cpp and the templates impl/polynomial_optimization_{linear,nonlinear}_impl.h, against stand-in headers for
 *     Eigen (oracle/ref_shim/Eigen: eager dense/sparse subset with the summation orders written down), NLopt (ref_shim/nlopt.hpp),
 *     mrs_lib's cyclic angle helpers, geometry_msgs and boost::clamp.  tests/test_ref_eth.py compares this restatement (math mode
 *     LIBM) with that build bit for bit: Q / A / A^-1 / R, solveLinear, coefficients and cost, both time estimates, per-segment
 *     maxima through Jenkins-Traub, computeMaximumOfMagnitude, scaleSegmentTimesToMeetConstraints, sampleWholeTrajectory,
 *     Trajectory::evaluate, the Mellinger time allocation end to end (optimize -> scaleSegmentTimesWithViolation) and the objective
 *     functions of methods 0/1/3/4.  tests/golden/ref_eth.npz holds outputs of that build (generator: tests/golden/gen_golden.py)
 *     for eight problems, so that the time estimates, coefficients and cost, maxima, time scaling, sampling and time allocation
 *     stay pinned on machines without the checkout.
 *   - What the stand-ins stand in for is NOT in the reference tree and cannot be pinned: (i) Eigen::SparseQR<COLAMD> on Rpp
 *     (lin_impl.h:362-369) -- the stand-in's solve is LU without pivoting on the full band (the contract the GPU follows); a
 *     Householder-QR variant of the stand-in (_ref/libref_eth_qr.so) and a 50-digit mpmath solve bound the difference
 *     (tests/test_numeric_floor.py: 5.9e-7 relative on coefficients at cond(Rpp) up to 4.9e15); (ii) NLopt 2.x LD_LBFGS
 *     (nl_impl.h:178-191) -- oracle/plis.cpp restates Luksan's PLIS as NLopt ships it (plis.c / pssubs.c / mssubs.c) from the
 *     published algorithm, call for call; NLopt's binary is absent, so its iterate sequence is restated, not compared;
 *     (iii) glibc's libm -- math mode DET replaces it by include/tg_detmath.h (correctly rounded; glibc is not, so the two modes
 *     differ by the floor measured in tests/test_numeric_floor.py: counts and verdicts identical, coefficients 1.4e-6 relative,
 *     sample positions 1.1e-7 m).
 *   - The node-level steps (mrs_trajectory_generation.cpp: vertex recipe, validation, subdivision, acceptance, sampling into the
 *     tracker's format) need ROS to compile; they are restated in node.cpp with file:line citations and checked through the
 *     reference tests' geometric predicate (0.5 m / 0.2 rad pass-through, test/include/get_path_test.h:10-11,45-68) and the
 *     identities of eth/test_utils.h.
 *
 * Math modes: kMathLibm calls glibc (the pure restatement: pow, exp, log, atan2, sin, cos, cbrt
 * exactly where the reference calls them); kMathDet swaps those calls for include/tg_detmath.h so
 * that results are bit-comparable with the GPU (see that header for why).
 */
#ifndef ORACLE_ORACLE_H_
#define ORACLE_ORACLE_H_

#include <cmath>
#include <cstdint>
#include <array>
#include <vector>

namespace orc {

#ifndef ORC_N
#define ORC_N 10  // the node's only instantiation (node.cpp:1063); liboracle_n{6,8,12}.so are built with -DORC_N for the general-N tests
#endif
constexpr int kN = ORC_N;     // coefficients per polynomial (lin.h:46-55: even, <= Polynomial::kMaxN = 12)
constexpr int kHalf = kN / 2;  // derivative slots per vertex (lin_impl.h:206)
constexpr int kD = 4;          // x, y, z, heading (node.cpp:902)

enum MathMode { kMathLibm = 0, kMathDet = 1 };
void set_math_mode(int mode);
int math_mode();
double m_pow_int(double t, int e);  // pow(t, e), e >= 1
double m_log(double x);
double m_exp(double x);
double m_sin(double x);
double m_cos(double x);
double m_atan2(double y, double x);
double m_cbrt(double x);
double m_hypot(double x, double y);
// the < 1.5 ulp kernels (not the correctly rounded versions) where a last-bit difference cannot reach a result the path reads:
// Jenkins-Traub's starting radius (rpoly_ak1.cpp:227-246) and the heading's quaternion round trip (eth_mav_msgs/common.h:130-140)
double m_log_k(double x);
double m_exp_k(double x);
double m_sin_k(double x);
double m_cos_k(double x);
double m_atan2_k(double y, double x);

// base_coefficients_(k, i) = i!/(i-k)!  (eth/polynomial.cpp:155-170)
double base_coeff(int k, int i);

// ---- vertices / constraints (eth/vertex.h:42-116) ------------------------------------------------
struct Vertex {
  uint8_t mask = 0;             // bit k set <=> derivative k is fixed
  double val[kHalf][kD] = {};   // fixed value per derivative and dimension
  void add(int deriv, const double* v) {
    if (deriv < 0 || deriv >= kHalf) return;  // lin_impl.h:84-102 drops orders > 4
    mask |= (uint8_t)(1u << deriv);
    for (int d = 0; d < kD; ++d) val[deriv][d] = v[d];
  }
  bool has(int deriv) const { return (mask >> deriv) & 1u; }
  // eth/vertex.cpp:158-163
  void make_start_or_end(const double* pos, int up_to) {
    add(0, pos);
    const double z[kD] = {0, 0, 0, 0};
    for (int i = 1; i <= up_to; ++i) add(i, z);
  }
};

struct Segment {
  double T = 0;
  double c[kD][kN] = {};  // increasing powers
};

// ---- linear QP (lin_impl.h) ------------------------------------------------------------------------
struct LinearSolver {
  int S = 0, r = 2;
  std::vector<Vertex> vtx;
  std::vector<double> times;
  // per segment
  std::vector<double> Ainv;  // S x 10 x 10
  std::vector<double> Q;     // S x 10 x 10
  // ordering (lin_impl.h:183-257)
  int n_fixed = 0, n_free = 0;
  std::vector<int> col_of;  // (V x 5): >=0 -> fixed column, <0 -> -(free index)-1
  std::vector<double> d_f;  // kD x n_fixed
  std::vector<double> d_p;  // kD x n_free
  std::vector<Segment> seg;

  bool setup(const std::vector<Vertex>& vertices, const std::vector<double>& t, int deriv_to_opt);
  void update_times(const std::vector<double>& t);  // lin_impl.h:288-304
  bool solve();                                     // lin_impl.h:340-373
  void segments_from_compact();                     // lin_impl.h:263-282
  double cost() const;                              // lin_impl.h:127-141
  // dense R (n_fixed+n_free)^2 for tests (lin_impl.h:310-334)
  void dense_R(std::vector<double>* R) const;
  void segment_H(int i, double* H) const;
};

void setup_mapping_A(double T, double* A);                       // lin_impl.h:112-121
void invert_mapping(const double* A, double* Ainv);              // lin_impl.h:147-177
void cost_jacobian_Q(int r, double T, double* Q);                // lin_impl.h:605-618

// ---- polynomial helpers (eth/polynomial.h, polynomial.cpp) ---------------------------------------------
double poly_eval(const double* c, double t, int deriv);          // polynomial.h:150-163
void poly_deriv_coeffs(const double* c, int deriv, double* out); // polynomial.h:108-119
int find_roots_jt(const double* coeffs_increasing, int n, double* re, double* im, bool* ok);  // rpoly_ak1.cpp:76-120

// extremum of |p^(deriv)| over dims on one segment (eth/segment.cpp:113-212, trajectory.cpp:211-243)
double segment_max_magnitude(const Segment& s, int deriv, const int* dims, int ndims, long* root_calls);
void max_of_magnitude(const std::vector<Segment>& seg, int deriv, double* time, double* value, int* segment_idx);  // lin_impl.h:477-508

// ---- trajectory level ---------------------------------------------------------------------------------
struct Limits {  // order matches scaleSegmentTimesToMeetConstraints' argument meaning
  double v_h, v_v, a_h, a_v, j_h, j_v, v_hdg, a_hdg, j_hdg;
};
extern double g_scale_tolerance;  // 1e-3 (eth/trajectory.cpp:604); a test hook may change it
// eth/trajectory.cpp:598-692 ; returns number of passes executed, *within = final within_range
int scale_times_to_meet_constraints(std::vector<Segment>& seg, const Limits& L, bool* within, long* root_calls);

struct Sample {  // the fields of EigenTrajectoryPoint the node consumes plus the derivatives it carries
  double p[4], v[4], a[4], j[3], s[3];
  double yaw_out;  // yawFromQuaternion(quaternionFromYaw(p[3])) (eth_mav_msgs/common.h:130-140)
  int64_t t_ns;
};
// eth/trajectory_sampling.cpp:49-104,119-124 + eth/trajectory.cpp:93-151
bool sample_whole(const std::vector<Segment>& seg, double dt, std::vector<Sample>* out);
// eth/trajectory.cpp:55-87
bool trajectory_evaluate(const std::vector<Segment>& seg, double t, int deriv, double* out4);

// eth/vertex.cpp:491-565 and 301-485
std::vector<double> estimate_times_euclidean(const std::vector<Vertex>& v, const Limits& L);
std::vector<double> estimate_times_baca(const std::vector<Vertex>& v, const Limits& L);

// mrs_lib cyclic helpers (restated from memory, SURVEY.md 8c(3))
double rad_wrap(double a);           // radians: [0, 2pi)
double rad_diff(double a, double b); // signed shortest a-b in [-pi, pi)
double rad_dist(double a, double b);
double rad_interp(double a, double b, double c);
double srad_unwrap(double what, double from);

// ---- nonlinear time allocation (nl_impl.h) -------------------------------------------------------------
struct NlParams {
  int max_evals = 10;      // config/private/trajectory_generation.yaml:10
  double f_rel = 0.05;     // node.cpp:884
  double x_rel = 0.1;      // node.cpp:885
  double f_abs = -1, x_abs = -1;
  int time_alloc = 2;      // Mellinger outer loop (config/private/...yaml:7)
};
struct NlInfo {
  int code = -1;      // nlopt-style result code
  int n_evals = 0;    // objective evaluations (OptimizationInfo::n_iterations)
  int n_solves = 0;   // linear solves performed
  int n_scale_passes = 0;
  long n_root_calls = 0;
  double final_cost = 0;
};
// nl_impl.h:256-333 ; leaves the solver at `times`
double mellinger_cost_and_grad(LinearSolver& ls, std::vector<double>* grad, int* n_solves);
// NLopt LD_LBFGS = Luksan's PLIS, restated from the published algorithm (oracle/plis.cpp; NLopt is not vendored).
typedef double (*PlisObjective)(int n, const double* x, double* grad, void* data);
struct PlisStop {
  int maxeval = 0;          // 0 = no limit; tested between iterations only
  double xtol_rel = 0, ftol_rel = 0;
  double xtol_abs = -1;     // nlopt_stop_dx's absolute tolerance (one value for all variables)
  double minf_max = -HUGE_VAL;  // stopval
  int nevals = 0;
};
int luksan_plis(int n, PlisObjective f, void* data, const double* lb, const double* ub, double* x, double* minf, PlisStop* stop);
// nl_impl.h:159-234 with nlopt::LD_LBFGS -> luksan_plis
int optimize_time_mellinger(LinearSolver& ls, const NlParams& p, const Limits& L, NlInfo* info);

// ---- node level (src/mrs_trajectory_generation.cpp) --------------------------------------------------------
struct Waypoint {
  double c[4];
  bool stop_at;
};
struct InitialState {  // the TrackerCommand fields findTrajectory reads (node.cpp:925-957)
  bool present = false;
  double heading = 0;
  double vel[4] = {0, 0, 0, 0}, acc[4] = {0, 0, 0, 0}, jerk[4] = {0, 0, 0, 0};
};
struct NodeParams {
  int derivative_to_optimize = 2;  // ACCELERATION
  NlParams nl;
  Limits lim;
  double dt = 0.2;
  bool check_deviation = true;
  double max_deviation = 0.05;
  int max_deviation_iters = 6;
  bool first_segment_checked = true;  // max_deviation_first_segment_ (node.cpp:874-878)
  double max_len_factor = 3.0, min_len_factor = 0.33;
  bool run_time_alloc = true;  // false => config-2 style: linear solve at the Euclidean times + sampling
  bool override_heading_atan2 = false;  // getTrajectoryReference: heading = direction to the next sample (node.cpp:1586-1599)
};
enum FindStatus { kFindOk = 0, kFindNloptRejected = 1, kFindTooLong = 2, kFindTooShort = 3, kFindSampleFail = 4, kFindEmptyPath = 5, kFindNotFinite = 6 };
struct FindResult {
  int status = kFindOk;
  NlInfo nl;
  std::vector<double> times;
  std::vector<Segment> seg;
  std::vector<Sample> samples;
  double baca_total = 0;
};
// node.cpp:857-1209
FindResult find_trajectory(const std::vector<Waypoint>& wp, const InitialState& init, const NodeParams& P);
// getTrajectoryReference (node.cpp:1560-1606): x, y, z, heading of every sample; heading = getYaw(), or with
// override_heading_atan2 the direction towards the next sample (the previous heading when that step is shorter than 0.05 m)
std::vector<std::array<double, 4>> trajectory_reference(const std::vector<Sample>& traj, bool override_heading_atan2);
// node.cpp:1401-1455
struct Validation {
  bool safe = true;
  double max_dev = 0;
  std::vector<uint8_t> seg_ok;
};
Validation validate_spatial(const std::vector<Sample>& traj, const std::vector<Waypoint>& wp, const NodeParams& P);
double dist_from_segment(const double* p, const double* a, const double* b);  // node.cpp:1533-1554
Waypoint interpolate_point(const Waypoint& a, const Waypoint& b, double coeff);  // node.cpp:1612-1625

// ---- the steps either side of the path (SURVEY.md 8f ranks 1-2) ---------------------------------------------------
// preprocessPath (node.cpp:431-500): optional straightener, then the min-distance filter.  Keeps the reference's
// `fabs(radians::diff(a, b) > limit)` expression as written (fabs of a bool, SURVEY.md section 9).
std::vector<Waypoint> preprocess_path(const std::vector<Waypoint>& in, double min_waypoint_distance, bool straightener_enabled,
                                      double straightener_max_deviation, double straightener_max_hdg_deviation);
// findTrajectoryFallback (node.cpp:1215-1395): constant-velocity samples along the polyline, Baca segment times.
// `L` already carries the fallback speed / acceleration factors; out: x, y, z, heading (after the quaternion round trip).
void fallback_sample(const std::vector<Waypoint>& wp, const Limits& L, double dt, double stopping_time, std::vector<std::array<double, 4>>* out);
// getWaypointInTrajectoryIdxs (node.cpp:1461-1499): index of the first sample whose chord passes within 0.1 m of each waypoint
std::vector<int> waypoint_trajectory_idxs(const std::vector<std::array<double, 4>>& samples, const std::vector<Waypoint>& wp);
// node.cpp:620-851 restricted to the numeric part: findTrajectory + validation + subdivision rounds
struct OptimizeResult {
  bool success = false;
  int rounds = 0;  // subdivision rounds executed (re-solves)
  bool safe = false;
  double max_dev = 0;
  std::vector<Waypoint> wp;  // final waypoint list
  FindResult find;
  long total_solves = 0, total_root_calls = 0, total_evals = 0;
};
OptimizeResult optimize_path(const std::vector<Waypoint>& wp_in, const InitialState& init, const NodeParams& P);

}  // namespace orc

#endif  // ORACLE_ORACLE_H_
