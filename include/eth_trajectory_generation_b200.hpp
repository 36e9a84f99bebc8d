// eth_trajectory_generation_b200.hpp -- header-only C++ host side of the B200 path, with the reference's class names.
//
// Drop-in for the classes MrsTrajectoryGeneration::findTrajectory uses (src/mrs_trajectory_generation.cpp:857-1209):
//   eth_trajectory_generation::Vertex                          eth/vertex.h:42-116
//   eth_trajectory_generation::Segment / Trajectory            eth/segment.h, eth/trajectory.h:51-190
//   eth_trajectory_generation::PolynomialOptimization<N>       lin.h:60-233
//   eth_trajectory_generation::NonlinearOptimizationParameters nl.h:35-110
//   eth_trajectory_generation::PolynomialOptimizationNonLinear<N>  nl.h:147-197
//   eth_trajectory_generation::sampleWholeTrajectory           eth/trajectory_sampling.h:44
//   eth_trajectory_generation::sampleTrajectoryInRange / sampleTrajectoryStartDuration  eth/trajectory_sampling.cpp:49-104, eth/trajectory_sampling.h
//   eth_trajectory_generation::estimateSegmentTimes / estimateSegmentTimesBaca   eth/vertex.cpp:491-565, 301-485
// Same method names, argument meaning and error behaviour (bool returns, print-and-continue -- eth/misc.h:6-38 -- and the
// NLopt-style int of optimize()).  Every method marshals into the C ABI of include/tg_b200.h, i.e. into the sm_100a
// kernels of libtg_b200.so; one object = a batch of one.  There is no CPU arithmetic here and no fallback: constructing
// the first object fails (std::runtime_error) when no CUDA device is usable.
//
// Types: the reference passes and returns Eigen::VectorXd.  When <Eigen/Core> can be found (or TG_B200_USE_EIGEN is defined)
// this header includes it and `Vector` IS Eigen::VectorXd, so call sites written against the reference compile unchanged
// (vertex.makeStartOrEnd(Eigen::Vector4d(x, y, z, heading), r), Eigen::VectorXd p = trajectory.evaluate(t), ...); every
// setter is a template over the vector type, so Eigen::Vector4d, Eigen::VectorXd, std::vector<double> and std::array all
// work.  Without Eigen (define TG_B200_NO_EIGEN to force it) `Vector` is std::vector<double>.  sampleWholeTrajectory fills any
// point type with the fields of eth_mav_msgs::EigenTrajectoryPoint (eth_mav_msgs/eigen_mav_msgs.h:188-240) -- the reference's
// own struct when that header is included, or the plain TrajectoryPoint below.
//
// Additions that the one-problem-per-object reference API cannot express: TrajectoryGeneratorBatch (the numeric core of
// optimize()/findTrajectory for many paths in one call, SURVEY.md H7), sampleTrajectoriesInRange (many windows in one call) and
// estimateSegmentTimesBatch (many vertex lists in one call).
#ifndef ETH_TRAJECTORY_GENERATION_B200_HPP_
#define ETH_TRAJECTORY_GENERATION_B200_HPP_

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <limits>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "tg_b200.h"

#if !defined(TG_B200_NO_EIGEN) && (defined(TG_B200_USE_EIGEN) || (defined(__has_include) && __has_include(<Eigen/Core>)))
#include <Eigen/Core>
#define TG_B200_HAVE_EIGEN 1
#endif
#include <thread>
#include <type_traits>
#include <utility>

namespace eth_trajectory_generation {

namespace derivative_order {  // eth/motion_defines.h:33-44
static constexpr int POSITION = 0;
static constexpr int VELOCITY = 1;
static constexpr int ACCELERATION = 2;
static constexpr int JERK = 3;
static constexpr int SNAP = 4;
static constexpr int INVALID = -1;
}  // namespace derivative_order

#if defined(TG_B200_HAVE_EIGEN)
typedef Eigen::VectorXd Vector;
#else
typedef std::vector<double> Vector;
#endif

namespace b200 {
// a Vector of n copies of `value`, and a copy of any indexable vector type (Eigen fixed / dynamic, std::vector, std::array)
inline Vector make_vector(size_t n, double value) {
#if defined(TG_B200_HAVE_EIGEN)
  return Vector::Constant((long)n, value);
#else
  return Vector(n, value);
#endif
}
template <class V>
inline Vector to_vector(const V& v) {
  Vector out = make_vector((size_t)v.size(), 0.0);
  for (size_t i = 0; i < (size_t)v.size(); ++i) out[i] = v[i];
  return out;
}
constexpr int kN = 10;    // coefficients per segment and dimension (node.cpp:1063)
constexpr int kD = 4;     // x, y, z, heading (node.cpp:902)
constexpr int kHalf = 5;  // derivative slots per vertex (lin_impl.h:206)

// One tg_ctx per device for the process, created on first use.
class Context {
 public:
  // slot > 0: a further, independent context on the same device (a tg_ctx serves one host thread at a time)
  static Context& instance(int device = 0, int slot = 0) {
    static std::map<std::pair<int, int>, std::unique_ptr<Context>> all;
    std::unique_ptr<Context>& c = all[std::make_pair(device, slot)];
    if (!c) c.reset(new Context(device));
    return *c;
  }
  tg_ctx* get() const { return ctx_; }
  void check(int rc, const char* what) const {
    if (rc != TG_OK) throw std::runtime_error(std::string(what) + ": " + tg_last_error(ctx_));
  }
  ~Context() {
    if (ctx_) tg_ctx_destroy(ctx_);
  }

 private:
  explicit Context(int device) {
    const int rc = tg_ctx_create(device, &ctx_);
    if (rc != TG_OK || !ctx_) throw std::runtime_error("tg_ctx_create failed: libtg_b200 needs a CUDA device (no CPU fallback)");
  }
  tg_ctx* ctx_ = nullptr;
};
}  // namespace b200

// ---- Vertex (eth/vertex.h:42-116, eth/vertex.cpp:134-177) ----------------------------------------------------------
class Vertex {
 public:
  typedef std::vector<Vertex> Vector;
  typedef eth_trajectory_generation::Vector ConstraintValue;
  typedef std::map<int, ConstraintValue> Constraints;

  explicit Vertex(size_t dimension) : D_(dimension) {}
  size_t D() const { return D_; }

  void addConstraint(int derivative_order, double value) { constraints_[derivative_order] = b200::make_vector(D_, value); }
  // any vector type: Eigen::VectorXd / Vector4d as in the reference's call sites, std::vector<double>, std::array
  template <class V, class = typename std::enable_if<!std::is_arithmetic<V>::value>::type>
  void addConstraint(int type, const V& constraint) {
    if ((size_t)constraint.size() != D_) {
      std::printf("[Vertex]: dimension of the constraint does not match the vertex\n");  // CHECK prints and continues
      return;
    }
    constraints_[type] = b200::to_vector(constraint);
  }
  // start or end vertex: position fixed, derivatives 1 .. up_to_derivative fixed at zero (eth/vertex.cpp:158-163)
  template <class V, class = typename std::enable_if<!std::is_arithmetic<V>::value>::type>
  void makeStartOrEnd(const V& constraint, int up_to_derivative) {
    addConstraint(derivative_order::POSITION, constraint);
    for (int i = 1; i <= up_to_derivative; ++i) constraints_[i] = b200::make_vector(D_, 0.0);
  }
  void makeStartOrEnd(double value, int up_to_derivative) { makeStartOrEnd(b200::make_vector(D_, value), up_to_derivative); }
  bool hasConstraint(int derivative_order) const { return constraints_.find(derivative_order) != constraints_.end(); }
  bool getConstraint(int derivative_order, ConstraintValue* constraint) const {
    const auto it = constraints_.find(derivative_order);
    if (it == constraints_.end()) return false;
    if (constraint) *constraint = it->second;
    return true;
  }
  bool removeConstraint(int type) { return constraints_.erase(type) > 0; }
  size_t getNumberOfConstraints() const { return constraints_.size(); }
  const Constraints& constraints() const { return constraints_; }

 private:
  size_t D_;
  Constraints constraints_;
};

// ---- Segment / Trajectory (eth/segment.h, eth/trajectory.h) -------------------------------------------------------------
struct Extremum {  // eth/extremum.h:31-55: ordered by value
  Extremum() : time(0.0), value(0.0), segment_idx(0) {}
  Extremum(double _time, double _value, int _segment_idx) : time(_time), value(_value), segment_idx(_segment_idx) {}
  bool operator<(const Extremum& rhs) const { return value < rhs.value; }
  bool operator>(const Extremum& rhs) const { return value > rhs.value; }
  double time;      // time inside the segment
  double value;
  int segment_idx;
};

class Segment {
 public:
  typedef std::vector<Segment> Vector;
  Segment() : time_(0.0), N_(b200::kN), D_(b200::kD), coef_(b200::kD * b200::kN, 0.0) {}
  Segment(int N, int D) : time_(0.0), N_(N), D_(D), coef_((size_t)N * D, 0.0) {}  // eth/segment.h:48
  int N() const { return N_; }
  int D() const { return D_; }
  double getTime() const { return time_; }
  void setTime(double t) { time_ = t; }
  // coefficients of dimension `dim`, increasing powers (eth/polynomial.h:35-37)
  const double* coefficients(int dim) const { return coef_.data() + dim * N_; }
  double* coefficients(int dim) { return coef_.data() + dim * N_; }
  const double* data() const { return coef_.data(); }  // [D][N]

 private:
  double time_;
  int N_, D_;
  std::vector<double> coef_;
};

class Trajectory {
 public:
  Trajectory() {}
  // shape of the segments (eth/trajectory.h:58-60; 10 coefficients x 4 dimensions while empty, the node's shape)
  int D() const { return segments_.empty() ? b200::kD : segments_.front().D(); }
  int N() const { return segments_.empty() ? b200::kN : segments_.front().N(); }
  int K() const { return (int)segments_.size(); }
  bool empty() const { return segments_.empty(); }
  void clear() { segments_.clear(); }
  void setSegments(const Segment::Vector& segments) {  // eth/trajectory.h:97-104: every segment must have the same shape
    for (const Segment& sg : segments)
      if (sg.N() != segments.front().N() || sg.D() != segments.front().D()) {
        std::printf("[Trajectory]: segments of different shapes, not set\n");
        return;
      }
    segments_ = segments;
  }
  // the tuned kernels take 10 coefficients x 4 dimensions; other shapes go through the general-shape entry points (tg_*_nd)
  bool tunedShape() const { return N() == b200::kN && D() == b200::kD; }
  void getSegments(Segment::Vector* segments) const {
    if (segments) *segments = segments_;
  }
  const Segment::Vector& segments() const { return segments_; }
  double getMinTime() const { return 0.0; }
  double getMaxTime() const {  // accumulated in segment order (eth/trajectory.h:76-83)
    double t = 0.0;
    for (const Segment& s : segments_) t += s.getTime();
    return t;
  }
  std::vector<double> getSegmentTimes() const {
    std::vector<double> t;
    for (const Segment& s : segments_) t.push_back(s.getTime());
    return t;
  }
  // Trajectory::evaluate(t, derivative) (eth/trajectory.cpp:55-87); past the end: prints, returns zeros.
  Vector evaluate(double t, int derivative = derivative_order::POSITION) const {
    Vector out = b200::make_vector((size_t)D(), 0.0);
    if (segments_.empty()) return out;
    std::vector<double> coef, times;
    pack(&coef, &times);
    uint8_t ok = 0;
    double v4[b200::kD] = {0, 0, 0, 0};
    b200::Context& c = b200::Context::instance();
    if (tunedShape()) c.check(tg_evaluate_batch(c.get(), K(), coef.data(), times.data(), 1, &t, derivative, v4, &ok), "tg_evaluate_batch");
    else c.check(tg_evaluate_batch_nd(c.get(), N(), D(), K(), coef.data(), times.data(), 1, &t, derivative, v4, &ok), "tg_evaluate_batch_nd");
    if (!ok) std::printf("[Trajectory]: time out of range, returning zeros\n");
    for (int d = 0; d < D(); ++d) out[d] = v4[d];
    return out;
  }
  // evaluateRange (eth/trajectory.cpp:93-151): the dt walk of the sampler, derivative `derivative` only
  void evaluateRange(double t_start, double t_end, double dt, int derivative, std::vector<Vector>* result,
                     std::vector<double>* sampling_times = nullptr) const;
  // maxima of |v|, |a|, |j| over the whole trajectory for the three dimension groups (eth/trajectory.cpp:422-565)
  void computeMaxDerivativesHorizontal(double* v_max, double* a_max, double* j_max) const { max_of_group(0, v_max, a_max, j_max); }
  void computeMaxDerivativesVertical(double* v_max, double* a_max, double* j_max) const { max_of_group(1, v_max, a_max, j_max); }
  void computeMaxDerivativesHeading(double* v_max, double* a_max, double* j_max) const { max_of_group(2, v_max, a_max, j_max); }
  // eth/trajectory.cpp:598-692, argument order of the reference
  bool scaleSegmentTimesToMeetConstraints(double v_max_horizontal, double v_max_vertical, double a_max_horizontal, double a_max_vertical,
                                          double j_max_horizontal, double j_max_vertical, double v_max_heading, double a_max_heading,
                                          double j_max_heading) {
    if (segments_.empty()) return true;
    if (!requireTenCoefficients("scaleSegmentTimesToMeetConstraints")) return false;
    std::vector<double> coef, times;
    pack4(&coef, &times);
    const double L[9] = {v_max_horizontal, v_max_vertical, a_max_horizontal, a_max_vertical, j_max_horizontal,
                         j_max_vertical,   v_max_heading,  a_max_heading,    j_max_heading};
    const int seg_off[2] = {0, K()};
    int passes = 0;
    uint8_t within = 0;
    b200::Context& c = b200::Context::instance();
    c.check(tg_scale_times_batch(c.get(), 1, seg_off, coef.data(), times.data(), L, &passes, &within), "tg_scale_times_batch");
    unpack4(coef, times);
    return within != 0;
  }

  // marshalling helpers (also used by the optimisers)
  // coef: [K][D][N] in the trajectory's own shape
  void pack(std::vector<double>* coef, std::vector<double>* times) const {
    const size_t dn = (size_t)D() * N();
    coef->resize((size_t)K() * dn);
    times->resize(K());
    for (int i = 0; i < K(); ++i) {
      (*times)[i] = segments_[i].getTime();
      for (size_t e = 0; e < dn; ++e) (*coef)[(size_t)i * dn + e] = segments_[i].data()[e];
    }
  }
  void unpack(const std::vector<double>& coef, const std::vector<double>& times, int n_coef = b200::kN, int dims = b200::kD) {
    segments_.assign(times.size(), Segment(n_coef, dims));
    for (size_t i = 0; i < times.size(); ++i) {
      segments_[i].setTime(times[i]);
      for (int d = 0; d < dims; ++d)
        for (int k = 0; k < n_coef; ++k) segments_[i].coefficients(d)[k] = coef[(i * dims + d) * n_coef + k];
    }
  }
  // Trajectory's maxima and time scaling take 10 coefficients (the tuned kernels).  Fewer than 4 dimensions are carried as zero
  // dimensions: a zero polynomial adds exact zeros to every sum of squares, so the other dimensions' results do not change.
  bool requireTenCoefficients(const char* what) const {
    if (N() == b200::kN) return true;
    std::printf("[Trajectory]: %s is not available for N = %d on the B200 path (N = 10 only)\n", what, N());
    return false;
  }
  void pack4(std::vector<double>* coef, std::vector<double>* times) const {  // [K][4][10], D() <= 4
    coef->assign((size_t)K() * b200::kD * b200::kN, 0.0);
    times->resize(K());
    for (int i = 0; i < K(); ++i) {
      (*times)[i] = segments_[i].getTime();
      for (int d = 0; d < D(); ++d)
        for (int k = 0; k < b200::kN; ++k) (*coef)[((size_t)i * b200::kD + d) * b200::kN + k] = segments_[i].coefficients(d)[k];
    }
  }
  void unpack4(const std::vector<double>& coef, const std::vector<double>& times) {  // keeps the trajectory's D
    const int dims = D();
    segments_.assign(times.size(), Segment(b200::kN, dims));
    for (size_t i = 0; i < times.size(); ++i) {
      segments_[i].setTime(times[i]);
      for (int d = 0; d < dims; ++d)
        for (int k = 0; k < b200::kN; ++k) segments_[i].coefficients(d)[k] = coef[(i * b200::kD + d) * b200::kN + k];
    }
  }

 private:
  void max_of_group(int group, double* v_max, double* a_max, double* j_max) const {
    double m[3] = {-1.7976931348623157e308, -1.7976931348623157e308, -1.7976931348623157e308};
    if (!segments_.empty() && requireTenCoefficients("computeMaxDerivatives")) {
      std::vector<double> coef, times, maxima((size_t)K() * 9);
      pack4(&coef, &times);
      b200::Context& c = b200::Context::instance();
      c.check(tg_extrema_batch(c.get(), K(), coef.data(), times.data(), maxima.data()), "tg_extrema_batch");
      for (int i = 0; i < K(); ++i)
        for (int q = 0; q < 3; ++q)
          if (m[q] < maxima[(size_t)i * 9 + group * 3 + q]) m[q] = maxima[(size_t)i * 9 + group * 3 + q];
    }
    if (v_max) *v_max = m[0];
    if (a_max) *a_max = m[1];
    if (j_max) *j_max = m[2];
  }
  Segment::Vector segments_;
};

// ---- sampling (eth/trajectory_sampling.h:44, eth_mav_msgs/eigen_mav_msgs.h:188-240) -------------------------------------
// The fields of EigenTrajectoryPoint the sampler fills (eth/trajectory_sampling.cpp:73-88).
struct TrajectoryPoint {
  typedef std::vector<TrajectoryPoint> Vector;
  int64_t time_from_start_ns;
  double position_W[3], velocity_W[3], acceleration_W[3], jerk_W[3], snap_W[3];
  double yaw;                 // getYaw(): yawFromQuaternion(quaternionFromYaw(heading)) (eth_mav_msgs/common.h:130-140)
  double yaw_rate, yaw_acc;   // v[3], a[3]
  double heading_raw;         // p[3] before the quaternion round trip
};

namespace b200 {
// does the point type carry EigenTrajectoryPoint's setFromYaw() (eth_mav_msgs/eigen_mav_msgs.h:226-238)?
template <class P, class = void>
struct has_set_from_yaw : std::false_type {};
template <class P>
struct has_set_from_yaw<P, decltype(std::declval<P&>().setFromYaw(0.0), void())> : std::true_type {};
template <class P>
inline typename std::enable_if<has_set_from_yaw<P>::value>::type fill_heading(P& s, const double* f) {
  s.setFromYaw(f[3]);       // the quaternion is built on the host by the reference's own inline code, as in the reference
  s.setFromYawRate(f[7]);
  s.setFromYawAcc(f[11]);
}
template <class P>
inline typename std::enable_if<!has_set_from_yaw<P>::value>::type fill_heading(P& s, const double* f) {
  s.heading_raw = f[3];
  s.yaw_rate = f[7];
  s.yaw_acc = f[11];
  s.yaw = f[18];
}
}  // namespace b200

namespace b200 {
// The windowed walk of tg_sample_range_batch_nd for trajectories of one shape, window p = [t_range[2p], t_range[2p+1]]: one counting
// call and one call for the rows (p4 v4 a4 j3 s3 yaw, time_from_start_ns), compacted in trajectory order.
inline void sample_ranges(const std::vector<const Trajectory*>& trajs, const double* t_range, double dt, std::vector<int>* counts,
                          std::vector<double>* full, std::vector<long long>* t_ns) {
  const int B = (int)trajs.size(), n_coef = trajs.front()->N(), dims = trajs.front()->D();
  std::vector<int> seg_off(1, 0);
  std::vector<double> coef, times;
  for (const Trajectory* t : trajs) {
    std::vector<double> c, T;
    t->pack(&c, &T);
    coef.insert(coef.end(), c.begin(), c.end());
    times.insert(times.end(), T.begin(), T.end());
    seg_off.push_back(seg_off.back() + t->K());
  }
  counts->assign(B, 0);
  Context& c = Context::instance();
  c.check(tg_sample_range_batch_nd(c.get(), n_coef, dims, B, seg_off.data(), coef.data(), times.data(), t_range, dt, counts->data(), nullptr,
                                   nullptr, nullptr),
          "tg_sample_range_batch_nd");
  size_t rows = 0;
  for (int n : *counts) rows += (size_t)n;
  full->resize(rows * 19);
  t_ns->resize(rows);
  if (rows)
    c.check(tg_sample_range_batch_nd(c.get(), n_coef, dims, B, seg_off.data(), coef.data(), times.data(), t_range, dt, counts->data(), nullptr,
                                     full->data(), t_ns->data()),
            "tg_sample_range_batch_nd");
}
// rows -> the fields of EigenTrajectoryPoint the sampler fills (eth/trajectory_sampling.cpp:73-103)
template <class PointVector>
inline void fill_points(int dims, const double* full, const long long* t_ns, int count, PointVector* states) {
  states->resize(count);
  for (int i = 0; i < count; ++i) {
    auto& s = (*states)[i];
    const double* f = full + (size_t)i * 19;  // p4 v4 a4 j3 s3 yaw
    s.time_from_start_ns = (int64_t)t_ns[i];  // (min_time + dt * i) * 1e9, eth/trajectory_sampling.cpp:98
    for (int k = 0; k < 3; ++k) {
      s.position_W[k] = f[k];
      s.velocity_W[k] = f[4 + k];
      s.acceleration_W[k] = f[8 + k];
      s.jerk_W[k] = f[12 + k];
      s.snap_W[k] = f[15 + k];
    }
    if (dims == 4) fill_heading(s, f);  // eth/trajectory_sampling.cpp:99-103: only a 4-dimensional trajectory sets the yaw
  }
}
inline bool sampling_refused(const char* who, const Trajectory& trajectory, double sampling_interval) {
  if (trajectory.empty() || !(sampling_interval > 0.0)) {
    std::printf("[%s]: empty trajectory or non-positive sampling interval\n", who);
    return true;
  }
  if (trajectory.D() < 3) {
    std::printf("[%s]: Dimension has to be at least 3, but is %d\n", who, trajectory.D());  // eth/trajectory_sampling.cpp:58-61
    return true;
  }
  return false;
}
}  // namespace b200

// sampleTrajectoryInRange (eth/trajectory_sampling.cpp:49-104).  PointVector: std::vector of TrajectoryPoint, or of the reference's
// eth_mav_msgs::EigenTrajectoryPoint (any allocator).  As upstream, a window outside [getMinTime(), getMaxTime()] is refused (false,
// no states); inside it the samples are evaluateRange's walk (DESIGN.md §4.3), which may return no state.  One device call.
template <class PointVector>
inline bool sampleTrajectoryInRange(const Trajectory& trajectory, double min_time, double max_time, double sampling_interval, PointVector* states) {
  if (!states) return false;
  states->clear();
  if (b200::sampling_refused("sampleTrajectoryInRange", trajectory, sampling_interval)) return false;
  if (!(min_time >= trajectory.getMinTime() && max_time <= trajectory.getMaxTime())) {
    std::printf("[sampleTrajectoryInRange]: Sample time should be within [%g %g] but is [%g %g]\n", trajectory.getMinTime(), trajectory.getMaxTime(),
                min_time, max_time);
    return false;
  }
  const double t_range[2] = {min_time, max_time};
  std::vector<int> counts;
  std::vector<double> full;
  std::vector<long long> t_ns;
  b200::sample_ranges({&trajectory}, t_range, sampling_interval, &counts, &full, &t_ns);
  b200::fill_points(trajectory.D(), full.data(), t_ns.data(), counts[0], states);
  return true;
}
// sampleTrajectoryStartDuration: sampleTrajectoryInRange over [start_time, start_time + duration]
template <class PointVector>
inline bool sampleTrajectoryStartDuration(const Trajectory& trajectory, double start_time, double duration, double sampling_interval,
                                          PointVector* states) {
  return sampleTrajectoryInRange(trajectory, start_time, start_time + duration, sampling_interval, states);
}
// sampleWholeTrajectory (eth/trajectory_sampling.cpp:119-124): sampleTrajectoryInRange over [getMinTime(), getMaxTime()], false when
// that gives no sample (a trajectory of zero duration) -- same call as in the reference (node.cpp:1166).
template <class PointVector>
inline bool sampleWholeTrajectory(const Trajectory& trajectory, double sampling_interval, PointVector* states) {
  if (!states) return false;
  return sampleTrajectoryInRange(trajectory, trajectory.getMinTime(), trajectory.getMaxTime(), sampling_interval, states) && !states->empty();
}
// Not a reference name: sampleTrajectoryInRange's walk for many trajectories of one shape in one device call, window i = windows[i] =
// {min_time, max_time}, states_per_trajectory[i] filled as sampleTrajectoryInRange fills its states.  It applies no range check: a
// window running past a trajectory's end stops at that end, as "the next H seconds" of a trajectory near its end should.  false, with
// nothing filled, for an empty list, mismatched sizes or shapes, or what sampleTrajectoryInRange refuses for any trajectory.
template <class PointVector>
inline bool sampleTrajectoriesInRange(const std::vector<Trajectory>& trajectories, const std::vector<std::pair<double, double>>& windows,
                                      double sampling_interval, std::vector<PointVector>* states_per_trajectory) {
  if (!states_per_trajectory) return false;
  states_per_trajectory->clear();
  if (trajectories.empty() || windows.size() != trajectories.size()) {
    std::printf("[sampleTrajectoriesInRange]: one window per trajectory is needed\n");
    return false;
  }
  std::vector<const Trajectory*> trajs;
  std::vector<double> t_range;
  for (size_t i = 0; i < trajectories.size(); ++i) {
    const Trajectory& t = trajectories[i];
    if (b200::sampling_refused("sampleTrajectoriesInRange", t, sampling_interval)) return false;
    if (t.N() != trajectories.front().N() || t.D() != trajectories.front().D()) {
      std::printf("[sampleTrajectoriesInRange]: every trajectory must have the same shape\n");
      return false;
    }
    trajs.push_back(&t);
    t_range.push_back(windows[i].first);
    t_range.push_back(windows[i].second);
  }
  std::vector<int> counts;
  std::vector<double> full;
  std::vector<long long> t_ns;
  b200::sample_ranges(trajs, t_range.data(), sampling_interval, &counts, &full, &t_ns);
  states_per_trajectory->resize(trajs.size());
  size_t row = 0;
  for (size_t i = 0; i < trajs.size(); ++i) {
    b200::fill_points(trajs[i]->D(), full.data() + row * 19, t_ns.data() + row, counts[i], &(*states_per_trajectory)[i]);
    row += (size_t)counts[i];
  }
  return true;
}

inline void Trajectory::evaluateRange(double t_start, double t_end, double dt, int derivative, std::vector<Vector>* result,
                                      std::vector<double>* sampling_times) const {
  // eth/trajectory.cpp:93-151 in one device call (tg_evaluate_range_batch_nd): the walk from the start of the segment holding t_start
  // while the accumulated time is below t_end, derivative `derivative` of every dimension; a start past the end prints and returns
  // nothing
  if (!result) return;
  result->clear();
  if (sampling_times) sampling_times->clear();
  if (segments_.empty() || !(dt > 0.0)) return;
  if (t_start > getMaxTime()) std::printf("[Trajectory]: start time out of range of the trajectory!\n");
  std::vector<double> coef, times;
  pack(&coef, &times);
  const int seg_off[2] = {0, K()};
  const double t_range[2] = {t_start, t_end};
  const int dims = D();
  int count = 0;
  b200::Context& c = b200::Context::instance();
  c.check(tg_evaluate_range_batch_nd(c.get(), N(), dims, 1, seg_off, coef.data(), times.data(), t_range, dt, derivative, &count, nullptr, nullptr),
          "tg_evaluate_range_batch_nd");
  if (count == 0) return;
  std::vector<double> out((size_t)count * dims), st(count);
  c.check(tg_evaluate_range_batch_nd(c.get(), N(), dims, 1, seg_off, coef.data(), times.data(), t_range, dt, derivative, &count, out.data(), st.data()),
          "tg_evaluate_range_batch_nd");
  for (int k = 0; k < count; ++k) {
    Vector v = b200::make_vector((size_t)dims, 0.0);
    for (int d = 0; d < dims; ++d) v[d] = out[(size_t)k * dims + d];
    result->push_back(v);
  }
  if (sampling_times) sampling_times->assign(st.begin(), st.end());
}

// ---- vertex marshalling ------------------------------------------------------------------------------------------------
namespace b200 {
// masks / fixed values ([V][half][dims]) of a vertex list; constraints above derivative half-1 are dropped with a warning
// (lin_impl.h:84-102)
inline bool pack_vertices(const Vertex::Vector& vertices, std::vector<uint8_t>* mask, std::vector<double>* vals, int half = kHalf, int dims = kD) {
  mask->assign(vertices.size(), 0);
  vals->assign(vertices.size() * (size_t)half * dims, 0.0);
  for (size_t v = 0; v < vertices.size(); ++v) {
    if (vertices[v].D() != (size_t)dims) {
      std::printf("[PolynomialOptimization]: vertex %zu has %zu dimensions, the optimisation %d\n", v, vertices[v].D(), dims);
      return false;
    }
    for (const auto& kv : vertices[v].constraints()) {
      if (kv.first < 0 || kv.first >= half) {
        std::printf("[PolynomialOptimization]: constraint of derivative %d ignored (highest possible: %d)\n", kv.first, half - 1);
        continue;
      }
      (*mask)[v] |= (uint8_t)(1u << kv.first);
      for (int d = 0; d < dims; ++d) (*vals)[(v * half + kv.first) * dims + d] = kv.second[d];
    }
  }
  return true;
}

// tg_estimate_segment_times_batch over vertex lists: the POSITION constraint of every vertex (x y z heading) goes up, the Euclidean
// and / or Baca times of list i come back as (*euclid)[i] / (*baca)[i].  false, with a message and nothing filled, for an empty list,
// a vertex that is not 4-dimensional or one without a POSITION constraint (the reference reads the heading as [3] of it).
inline bool estimate_times(const char* who, const std::vector<const Vertex::Vector*>& lists, const double* L8, std::vector<std::vector<double>>* euclid,
                           std::vector<std::vector<double>>* baca) {
  std::vector<int> vtx_off(1, 0);
  std::vector<double> pos4;
  Vertex::ConstraintValue p;
  for (const Vertex::Vector* vl : lists) {
    if (vl->empty()) {
      std::printf("[%s]: a vertex list is empty\n", who);
      return false;
    }
    for (const Vertex& v : *vl) {
      if (v.D() != (size_t)kD || !v.getConstraint(derivative_order::POSITION, &p)) {
        std::printf("[%s]: every vertex needs %d dimensions (x, y, z, heading) and a POSITION constraint\n", who, kD);
        return false;
      }
      for (int d = 0; d < kD; ++d) pos4.push_back(p[d]);
    }
    vtx_off.push_back(vtx_off.back() + (int)vl->size());
  }
  const int B = (int)lists.size();
  const size_t totS = (size_t)(vtx_off[B] - B);
  std::vector<double> e(euclid ? totS : 0), b(baca ? totS : 0);
  Context& c = Context::instance();
  c.check(tg_estimate_segment_times_batch(c.get(), B, vtx_off.data(), pos4.data(), L8, euclid ? e.data() : nullptr, baca ? b.data() : nullptr),
          "tg_estimate_segment_times_batch");
  if (euclid) euclid->resize(B);
  if (baca) baca->resize(B);
  for (int i = 0; i < B; ++i) {
    const size_t s0 = (size_t)(vtx_off[i] - i), s1 = (size_t)(vtx_off[i + 1] - i - 1);
    if (euclid) (*euclid)[i].assign(e.begin() + s0, e.begin() + s1);
    if (baca) (*baca)[i].assign(b.begin() + s0, b.begin() + s1);
  }
  return true;
}
}  // namespace b200

// ---- initial segment times (eth/vertex.cpp:301-565) --------------------------------------------------------------------------
// estimateSegmentTimes (the Euclidean estimate, eth/vertex.cpp:491-565) and estimateSegmentTimesBaca (301-485) with the reference's
// argument list, as findTrajectory calls them (node.cpp:1045-1056); one device call each, the kernels of the optimisation pipeline.
// A list that is empty, not 4-dimensional or has a vertex without a POSITION constraint prints a message and gives an empty vector.
inline std::vector<double> estimateSegmentTimes(const Vertex::Vector& vertices, double v_max_horizontal, double v_max_vertical, double a_max_horizontal,
                                                double a_max_vertical, double j_max_horizontal, double j_max_vertical, double v_max_heading,
                                                double a_max_heading) {
  const double L8[8] = {v_max_horizontal, v_max_vertical, a_max_horizontal, a_max_vertical, j_max_horizontal, j_max_vertical, v_max_heading, a_max_heading};
  std::vector<std::vector<double>> out;
  if (!b200::estimate_times("estimateSegmentTimes", {&vertices}, L8, &out, nullptr)) return {};
  return out[0];
}
// the name SURVEY.md §8a gives the Euclidean estimate
inline std::vector<double> estimateSegmentTimesEuclidean(const Vertex::Vector& vertices, double v_max_horizontal, double v_max_vertical,
                                                         double a_max_horizontal, double a_max_vertical, double j_max_horizontal, double j_max_vertical,
                                                         double v_max_heading, double a_max_heading) {
  return estimateSegmentTimes(vertices, v_max_horizontal, v_max_vertical, a_max_horizontal, a_max_vertical, j_max_horizontal, j_max_vertical,
                              v_max_heading, a_max_heading);
}
inline std::vector<double> estimateSegmentTimesBaca(const Vertex::Vector& vertices, double v_max_horizontal, double v_max_vertical, double a_max_horizontal,
                                                    double a_max_vertical, double j_max_horizontal, double j_max_vertical, double v_max_heading,
                                                    double a_max_heading) {
  const double L8[8] = {v_max_horizontal, v_max_vertical, a_max_horizontal, a_max_vertical, j_max_horizontal, j_max_vertical, v_max_heading, a_max_heading};
  std::vector<std::vector<double>> out;
  if (!b200::estimate_times("estimateSegmentTimesBaca", {&vertices}, L8, nullptr, &out)) return {};
  return out[0];
}
// Not a reference name: both estimates for many vertex lists in one device call; (*euclidean)[i] / (*baca)[i] are the times of
// vertex_lists[i], either pointer may be null.  false, with a message and nothing filled, for no list, both pointers null, or what
// estimateSegmentTimes refuses for any list.
inline bool estimateSegmentTimesBatch(const std::vector<Vertex::Vector>& vertex_lists, double v_max_horizontal, double v_max_vertical,
                                      double a_max_horizontal, double a_max_vertical, double j_max_horizontal, double j_max_vertical, double v_max_heading,
                                      double a_max_heading, std::vector<std::vector<double>>* euclidean, std::vector<std::vector<double>>* baca) {
  if (vertex_lists.empty() || (!euclidean && !baca)) {
    std::printf("[estimateSegmentTimesBatch]: no vertex list or no output\n");
    return false;
  }
  const double L8[8] = {v_max_horizontal, v_max_vertical, a_max_horizontal, a_max_vertical, j_max_horizontal, j_max_vertical, v_max_heading, a_max_heading};
  std::vector<const Vertex::Vector*> lists;
  for (const Vertex::Vector& vl : vertex_lists) lists.push_back(&vl);
  return b200::estimate_times("estimateSegmentTimesBatch", lists, L8, euclidean, baca);
}

// ---- PolynomialOptimization<N> (lin.h:60-233) -----------------------------------------------------------------------------
// N = 10 on 4 dimensions with derivative_to_optimize 2..4 (the node's shape, node.cpp:902, 907-921, 1063) runs on the tuned kernels;
// every other shape the reference's template allows up to Polynomial::kMaxN = 12 -- N in {6, 8, 10, 12}, 1..4 dimensions,
// derivative_to_optimize 0 .. N/2-1 -- on the general-shape kernels (tg_solve_linear_batch_nd), bit-identical where both apply.
template <int _N = 10>
class PolynomialOptimization {
  static_assert(_N == 6 || _N == 8 || _N == 10 || _N == 12, "the B200 path is built for N = 6, 8, 10 or 12 coefficients (lin.h:46-55, kMaxN = 12)");

 public:
  enum { N = _N };
  static constexpr int kHighestDerivativeToOptimize = N / 2 - 1;  // lin.h:55
  explicit PolynomialOptimization(size_t dimension) : dimension_(dimension), derivative_to_optimize_(derivative_order::INVALID), cost_(0.0), solved_(false) {}

  // lin_impl.h:61-106
  bool setupFromVertices(const Vertex::Vector& vertices, const std::vector<double>& segment_times, int derivative_to_optimize) {
    if (!(derivative_to_optimize >= 0 && derivative_to_optimize <= kHighestDerivativeToOptimize)) {
      std::printf("[PolynomialOptimization]: you tried to optimize a derivative that is not possible\n");  // lin_impl.h:63-66
      return false;
    }
    if (dimension_ < 1 || dimension_ > (size_t)b200::kD) {
      std::printf("[PolynomialOptimization]: the B200 path carries 1 to 4 dimensions\n");
      return false;
    }
    if (vertices.size() < 2 || segment_times.size() != vertices.size() - 1) {
      std::printf("[PolynomialOptimization]: size of times must be one less than positions\n");
      return false;
    }
    derivative_to_optimize_ = derivative_to_optimize;
    vertices_ = vertices;
    segment_times_ = segment_times;
    solved_ = false;
    free_state_ = kFreeNone;
    return b200::pack_vertices(vertices_, &mask_, &vals_, N / 2, (int)dimension_);
  }
  // the node's shape: tuned kernels
  bool tunedShape() const {
    return N == b200::kN && dimension_ == (size_t)b200::kD && derivative_to_optimize_ >= derivative_order::ACCELERATION;
  }
  // lin_impl.h:288-304
  void updateSegmentTimes(const std::vector<double>& segment_times) {
    if (segment_times.size() != segment_times_.size()) {
      std::printf("[PolynomialOptimization]: number of segment times does not match\n");
      return;
    }
    segment_times_ = segment_times;
    solved_ = false;
    free_state_ = kFreeNone;
  }
  // lin_impl.h:340-373 (+ updateSegmentsFromCompactConstraints 263-282)
  bool solveLinear() {
    if (vertices_.empty()) return false;
    const int V = (int)vertices_.size();
    const int vtx_off[2] = {0, V};
    coef_.resize((size_t)(V - 1) * dimension_ * N);
    b200::Context& c = b200::Context::instance();
    const int r = derivative_to_optimize_;
    const int rc = tunedShape() ? tg_solve_linear_batch(c.get(), 1, vtx_off, mask_.data(), vals_.data(), segment_times_.data(), r, coef_.data(), &cost_)
                                : tg_solve_linear_batch_nd(c.get(), N, (int)dimension_, 1, vtx_off, mask_.data(), vals_.data(), segment_times_.data(), r,
                                                           coef_.data(), &cost_);
    if (rc != TG_OK) {
      std::printf("[PolynomialOptimization]: solveLinear failed: %s\n", tg_last_error(c.get()));
      return false;
    }
    solved_ = true;
    free_state_ = kFreeFromSolve;
    return true;
  }
  // ---- free and fixed constraints (lin_impl.h:183-257, 513-522) ----------------------------------------------------------
  // Both are dimension-major: getDimension() vectors; within a vector vertex-major with the derivative ascending.
  size_t getNumberFreeConstraints() const { return (size_t)countFree(); }
  size_t getNumberFixedConstraints() const { return mask_.size() * (size_t)(N / 2) - (size_t)countFree(); }
  size_t getNumberAllConstraints() const { return segment_times_.size() * (size_t)N; }  // N/2 start and N/2 end rows per segment
  void getFixedConstraints(std::vector<Vector>* fixed_constraints) const {
    if (!fixed_constraints) return;
    constexpr int H = N / 2;
    const size_t dims = dimension_;
    fixed_constraints->assign(dims, b200::make_vector(getNumberFixedConstraints(), 0.0));
    size_t i = 0;
    for (size_t v = 0; v < mask_.size(); ++v)
      for (int k = 0; k < H; ++k) {
        if (!((mask_[v] >> k) & 1u)) continue;
        for (size_t d = 0; d < dims; ++d) (*fixed_constraints)[d][i] = vals_[(v * H + k) * dims + d];
        ++i;
      }
  }
  // After solveLinear(): the free derivatives d_p the solve found (fetched from the device on the first request at the current times
  // and kept).  After setFreeConstraints(): what was set.  Otherwise (no solve yet, or updateSegmentTimes / a nonlinear optimisation
  // since) there is no linear solution to read: a message, and zero vectors.
  void getFreeConstraints(std::vector<Vector>* free_constraints) const {
    if (!free_constraints) return;
    const size_t dims = dimension_, nf = getNumberFreeConstraints();
    if (free_state_ == kFreeFromSolve) {
      b200::Context& c = b200::Context::instance();
      const int vtx_off[2] = {0, (int)vertices_.size()};
      free_.assign(std::max<size_t>(dims * nf, 1), 0.0);
      c.check(tg_solve_linear_free_batch_nd(c.get(), N, (int)dims, 1, vtx_off, mask_.data(), vals_.data(), segment_times_.data(),
                                            derivative_to_optimize_, nullptr, nullptr, free_.data()),
              "tg_solve_linear_free_batch_nd");
      free_state_ = kFreeKnown;
    }
    if (free_state_ == kFreeNone) {
      std::printf("[PolynomialOptimization]: getFreeConstraints: no linear solution (call solveLinear or setFreeConstraints first)\n");
      free_constraints->assign(dims, b200::make_vector(nf, 0.0));
      return;
    }
    free_constraints->assign(dims, b200::make_vector(nf, 0.0));
    for (size_t d = 0; d < dims; ++d)
      for (size_t i = 0; i < nf; ++i) (*free_constraints)[d][i] = free_[d * nf + i];
  }
  // lin_impl.h:519-522: the segments (and the cost) become A^-1 [fixed ; free] at the current times.  The wrong number of vectors or
  // of entries is refused with a message and leaves the state as it was (the reference's CHECK prints and goes on with the sizes given).
  void setFreeConstraints(const std::vector<Vector>& free_constraints) {
    const size_t dims = dimension_, nf = getNumberFreeConstraints();
    if (vertices_.empty()) {
      std::printf("[PolynomialOptimization]: setFreeConstraints before setupFromVertices\n");
      return;
    }
    bool ok = free_constraints.size() == dims;
    for (size_t d = 0; ok && d < dims; ++d) ok = (size_t)free_constraints[d].size() == nf;
    if (!ok) {
      std::printf("[PolynomialOptimization]: setFreeConstraints needs %zu vectors of %zu free derivatives\n", dims, nf);
      return;
    }
    std::vector<double> flat(std::max<size_t>(dims * nf, 1), 0.0);
    for (size_t d = 0; d < dims; ++d)
      for (size_t i = 0; i < nf; ++i) flat[d * nf + i] = free_constraints[d][i];
    const int V = (int)vertices_.size();
    const int vtx_off[2] = {0, V};
    std::vector<double> coef((size_t)(V - 1) * dims * N);
    double cost = 0.0;
    b200::Context& c = b200::Context::instance();
    c.check(tg_set_free_constraints_batch_nd(c.get(), N, (int)dims, 1, vtx_off, mask_.data(), vals_.data(), segment_times_.data(),
                                             derivative_to_optimize_, flat.data(), coef.data(), &cost),
            "tg_set_free_constraints_batch_nd");
    coef_ = std::move(coef);
    cost_ = cost;
    free_ = std::move(flat);
    solved_ = true;
    free_state_ = kFreeKnown;
  }
  double computeCost() const { return cost_; }  // lin_impl.h:127-141
  void getSegmentTimes(std::vector<double>* segment_times) const {
    if (segment_times) *segment_times = segment_times_;
  }
  void getVertices(Vertex::Vector* vertices) const {
    if (vertices) *vertices = vertices_;
  }
  void getSegments(Segment::Vector* segments) const {  // lin.h:177
    Trajectory t;
    getTrajectory(&t);
    t.getSegments(segments);
  }
  void getTrajectory(Trajectory* trajectory) const {  // lin.h:153-160
    if (!trajectory) return;
    trajectory->clear();
    if (solved_) trajectory->unpack(coef_, segment_times_, N, (int)dimension_);
  }
  // lin_impl.h:477-508 (the reference's optional list of all candidates is not produced)
  Extremum computeMaximumOfMagnitude(int derivative, std::vector<Extremum>* candidates = nullptr) const {
    if (candidates) candidates->clear();
    Extremum e;
    if (!solved_ || segment_times_.empty()) return e;
    b200::Context& c = b200::Context::instance();
    const int off[2] = {0, (int)segment_times_.size()};
    if (N != b200::kN) {  // the general-shape kernels take [S][D][N] as it is
      c.check(tg_max_magnitude_batch_nd(c.get(), N, (int)dimension_, 1, off, coef_.data(), segment_times_.data(), derivative, &e.value, &e.time,
                                        &e.segment_idx),
              "tg_max_magnitude_batch_nd");
      return e;
    }
    Trajectory t;
    getTrajectory(&t);
    std::vector<double> c4, times;
    t.pack4(&c4, &times);  // missing dimensions as zero polynomials: they add exact zeros to the squared magnitude
    c.check(tg_max_magnitude_batch(c.get(), 1, off, c4.data(), times.data(), derivative, &e.value, &e.time, &e.segment_idx), "tg_max_magnitude_batch");
    return e;
  }
  template <int Derivative>
  Extremum computeMaximumOfMagnitude(std::vector<Extremum>* candidates = nullptr) const {
    return computeMaximumOfMagnitude(Derivative, candidates);
  }
  size_t getDimension() const { return dimension_; }
  size_t getNumberSegments() const { return segment_times_.size(); }
  int getDerivativeToOptimize() const { return derivative_to_optimize_; }

  // used by PolynomialOptimizationNonLinear
  const std::vector<uint8_t>& vertexMasks() const { return mask_; }
  const std::vector<double>& vertexValues() const { return vals_; }
  void adopt(const std::vector<double>& times, const std::vector<double>& coef, double cost) {
    segment_times_ = times;
    coef_ = coef;
    cost_ = cost;
    solved_ = true;
    free_state_ = kFreeNone;
  }
  // used by optimizeTimeDerivativeFreeBatch: the state after updateSegmentTimes(times) + solveLinear() (free null: getFreeConstraints
  // fetches the solve's d_p on request), or + setFreeConstraints(free) (free [D][n_free]); coef [S][D][N]
  void adoptDerivativeFree(const std::vector<double>& times, const std::vector<double>& coef, double cost, const std::vector<double>* free) {
    adopt(times, coef, cost);
    free_state_ = free ? kFreeKnown : kFreeFromSolve;
    if (free) free_ = *free;
  }

 private:
  int countFree() const {
    int n = 0;
    for (uint8_t m : mask_)
      for (int k = 0; k < N / 2; ++k) n += ((m >> k) & 1u) ? 0 : 1;
    return n;
  }
  // where getFreeConstraints reads from: nothing, the solve of solveLinear (not fetched yet), or free_
  enum FreeState { kFreeNone, kFreeFromSolve, kFreeKnown };
  mutable FreeState free_state_ = kFreeNone;
  mutable std::vector<double> free_;  // [D][n_free]
  size_t dimension_;
  int derivative_to_optimize_;
  Vertex::Vector vertices_;
  std::vector<double> segment_times_;
  std::vector<uint8_t> mask_;
  std::vector<double> vals_;
  std::vector<double> coef_;
  double cost_;
  bool solved_;
};

// ---- NonlinearOptimizationParameters (nl.h:35-110): the fields the production path reads ---------------------------------
struct NonlinearOptimizationParameters {
  enum TimeAllocMethod { kSquaredTime, kRichterTime, kMellingerOuterLoop, kSquaredTimeAndConstraints, kRichterTimeAndConstraints, kUnknown };
  double f_abs = -1, f_rel = 0.05, x_rel = 0.1, x_abs = -1;  // node.cpp:884-887
  int max_iterations = 10;                                   // NLopt maxeval (config/private/trajectory_generation.yaml:10)
  TimeAllocMethod time_alloc_method = kMellingerOuterLoop;   // config/private/trajectory_generation.yaml:7
  double initial_stepsize_rel = 0.1;                         // nl.h:58
  double time_penalty = 500.0;                               // nl.h:73
  bool use_soft_constraints = true;                          // nl.h:88
  double soft_constraint_weight = 100.0;                     // nl.h:91
  bool print_debug_info = false, print_debug_info_time_allocation = false;
};

struct OptimizationInfo {  // nl.h:112-130
  int n_iterations = 0;
  int stopping_reason = -1;  // NLopt-style code
  double cost_trajectory = 0.0;
  double cost_time = 0.0;
  double cost_soft_constraints = 0.0;
  int n_scale_passes = 0;
};

// ---- PolynomialOptimizationNonLinear<N> (nl.h:147-197) -------------------------------------------------------------------
template <int _N = 10>
class PolynomialOptimizationNonLinear {
 public:
  enum { N = _N };
  PolynomialOptimizationNonLinear(size_t dimension, const NonlinearOptimizationParameters& parameters)
      : poly_opt_(dimension), optimization_parameters_(parameters) {
    for (double& l : limits_) l = 3.40282346638528859812e+38;  // "no constraint"
  }
  // nl_impl.h:51-82
  bool setupFromVertices(const Vertex::Vector& vertices, const std::vector<double>& segment_times, int derivative_to_optimize) {
    // The Mellinger method runs for N in {6, 8, 10, 12} on 1..4 dimensions: N = 10 on the tuned kernels (the node's shape, node.cpp:902,
    // 907-921, 1063), fewer than four dimensions carried as zero dimensions (a zero polynomial adds exact zeros to the cost, to its
    // gradient and to every squared magnitude); the other N on the general-shape kernels (tg_time_alloc_batch_nd).  derivative_to_optimize
    // starts at 2 either way.  The derivative-free methods optimise D x n_free variables on the tuned kernels: N = 10, 4 dimensions.
    const size_t dims = poly_opt_.getDimension();
    const bool mellinger = optimization_parameters_.time_alloc_method == NonlinearOptimizationParameters::kMellingerOuterLoop;
    if (derivative_to_optimize < derivative_order::ACCELERATION || dims < 1 || dims > (size_t)b200::kD ||
        (!mellinger && (N != b200::kN || dims != (size_t)b200::kD))) {
      std::printf("[PolynomialOptimizationNonLinear]: the B200 time allocation is built for derivative_to_optimize >= 2 with kMellingerOuterLoop "
                  "(N = 6, 8, 10, 12 on 1..4 dimensions), and for N = 10 on 4 dimensions with the other methods\n");
      return false;
    }
    return poly_opt_.setupFromVertices(vertices, segment_times, derivative_to_optimize);
  }
  // nl_impl.h:538-565; the (dimension, derivative) -> limit mapping of scaleSegmentTimesWithViolation (355-381):
  // dimensions 0,1 -> horizontal, 2 -> vertical, 3 -> heading; a later call overwrites an earlier one
  bool addMaximumMagnitudeConstraint(int dimension, int derivative, double maximum_value) {
    if (derivative < derivative_order::VELOCITY || derivative > derivative_order::SNAP || dimension < 0 || dimension > 3) {
      std::printf("[PolynomialOptimizationNonLinear]: constraint (dimension %d, derivative %d) has no effect on this path\n", dimension, derivative);
      return false;
    }
    if (derivative <= derivative_order::JERK) {  // snap limits only enter the soft-constraint objectives
      const int d = derivative - 1;  // 0 v, 1 a, 2 j
      int idx;                       // tg_params::limits order: v_h v_v a_h a_v j_h j_v v_hdg a_hdg j_hdg
      if (dimension <= 1) idx = 2 * d;
      else if (dimension == 2) idx = 2 * d + 1;
      else idx = 6 + d;
      limits_[idx] = maximum_value;
    }
    constraint_dimension_.push_back(dimension);
    constraint_derivative_.push_back(derivative);
    constraint_value_.push_back(maximum_value);
    return true;
  }
  // The objective of the derivative-free methods at K candidate vectors in ONE batched call: objectiveFunctionTime
  // (nl_impl.h:567-614; kSquaredTime, kRichterTime: x = the S segment times) / objectiveFunctionTimeAndConstraints
  // (nl_impl.h:651-722; the ...AndConstraints methods: x = S times, then the free derivatives dimension-major), with
  // evaluateMaximumMagnitudeAsSoftConstraint (740-762) over the constraints added so far.  The reference evaluates one x per
  // NLopt callback; a derivative-free optimiser on the B200 evaluates a whole iteration's trial points here.
  // parts (optional): K x {cost_trajectory, cost_time, cost_soft_constraints}.
  bool evaluateObjectives(const std::vector<std::vector<double>>& x, std::vector<double>* total, std::vector<double>* parts = nullptr) const {
    const int method = (int)optimization_parameters_.time_alloc_method;
    if (!total || x.empty() || method == NonlinearOptimizationParameters::kMellingerOuterLoop || method > 4) return false;
    const size_t nvar = x.front().size();
    std::vector<double> flat;
    flat.reserve(x.size() * nvar);
    for (const std::vector<double>& xi : x) {
      if (xi.size() != nvar) return false;
      flat.insert(flat.end(), xi.begin(), xi.end());
    }
    total->assign(x.size(), 0.0);
    if (parts) parts->assign(3 * x.size(), 0.0);
    const int V = (int)poly_opt_.vertexMasks().size();
    b200::Context& c = b200::Context::instance();
    const int r = poly_opt_.getDerivativeToOptimize();
    const int rc = tg_objective_batch(c.get(), V, poly_opt_.vertexMasks().data(), poly_opt_.vertexValues().data(), r, method, (long long)x.size(),
                                      flat.data(), (int)nvar, optimization_parameters_.time_penalty, optimization_parameters_.use_soft_constraints ? 1 : 0,
                                      optimization_parameters_.soft_constraint_weight, (int)constraint_derivative_.size(),
                                      constraint_derivative_.data(), constraint_value_.data(), total->data(), parts ? parts->data() : nullptr, nullptr);
    if (rc != TG_OK) {
      std::printf("[PolynomialOptimizationNonLinear]: evaluateObjectives failed: %s\n", tg_last_error(c.get()));
      return false;
    }
    return true;
  }
  // nl_impl.h:89-118: returns the NLopt-style result code (the node accepts >= 1 except 6, and -1; node.cpp:1138-1149)
  int optimize() {
    if (optimization_parameters_.time_alloc_method != NonlinearOptimizationParameters::kMellingerOuterLoop) return optimizeDerivativeFree();
    std::vector<double> times;
    poly_opt_.getSegmentTimes(&times);
    const int S = (int)times.size(), V = S + 1;
    if (S < 1) return -1;
    tg_params P;
    tg_default_params(&P);
    P.derivative_to_optimize = poly_opt_.getDerivativeToOptimize();
    P.max_evals = optimization_parameters_.max_iterations;
    P.f_rel = optimization_parameters_.f_rel;
    P.x_rel = optimization_parameters_.x_rel;
    for (int i = 0; i < 9; ++i) P.limits[i] = limits_[i];
    const int vtx_off[2] = {0, V};
    int code = -1, evals = 0, passes = 0;
    double cost = 0.0;
    b200::Context& c = b200::Context::instance();
    const int dims = (int)poly_opt_.getDimension();
    if (N != b200::kN) {  // [V][N/2][dims] in, [S][dims][N] out
      std::vector<double> coef((size_t)S * dims * N);
      const int rc = tg_time_alloc_batch_nd(c.get(), N, dims, 1, vtx_off, poly_opt_.vertexMasks().data(), poly_opt_.vertexValues().data(), times.data(),
                                            &P, coef.data(), &code, &evals, &passes, &cost);
      if (rc != TG_OK) {
        std::printf("[PolynomialOptimizationNonLinear]: optimize failed: %s\n", tg_last_error(c.get()));
        return -1;  // nlopt::FAILURE
      }
      poly_opt_.adopt(times, coef, cost);
      optimization_info_.n_iterations = evals;
      optimization_info_.stopping_reason = code;
      optimization_info_.cost_trajectory = cost;
      optimization_info_.n_scale_passes = passes;
      return code;
    }
    std::vector<double> coef((size_t)S * b200::kD * b200::kN);
    std::vector<double> vals4;  // [V][5][4]: the vertex values with the missing dimensions zero
    const double* vals = poly_opt_.vertexValues().data();
    if (dims != b200::kD) {
      vals4.assign((size_t)V * b200::kHalf * b200::kD, 0.0);
      for (size_t i = 0; i < (size_t)V * b200::kHalf; ++i)
        for (int d = 0; d < dims; ++d) vals4[i * b200::kD + d] = vals[i * dims + d];
      vals = vals4.data();
    }
    const int rc = tg_time_alloc_batch(c.get(), 1, vtx_off, poly_opt_.vertexMasks().data(), vals, times.data(), &P, coef.data(), &code, &evals,
                                       &passes, &cost);
    if (rc != TG_OK) {
      std::printf("[PolynomialOptimizationNonLinear]: optimize failed: %s\n", tg_last_error(c.get()));
      return -1;  // nlopt::FAILURE
    }
    if (dims != b200::kD) {  // [S][4][10] -> [S][dims][10]
      std::vector<double> cd((size_t)S * dims * b200::kN);
      for (int i = 0; i < S; ++i)
        for (int d = 0; d < dims; ++d)
          for (int k = 0; k < b200::kN; ++k) cd[((size_t)i * dims + d) * b200::kN + k] = coef[((size_t)i * b200::kD + d) * b200::kN + k];
      coef.swap(cd);
    }
    poly_opt_.adopt(times, coef, cost);
    optimization_info_.n_iterations = evals;
    optimization_info_.stopping_reason = code;
    optimization_info_.cost_trajectory = cost;
    optimization_info_.n_scale_passes = passes;
    return code;
  }
  // optimizeTime / optimizeTimeAndFreeConstraints (nl_impl.h:120-157, 429-536) for kSquaredTime, kRichterTime and the two
  // ...AndConstraints methods.  The reference hands the objective to NLopt's LN_BOBYQA, which is not vendored and not restated:
  // the objective (evaluateObjectives above), the bounds (kOptimizationTimeLowerBound; setFreeEndpointDerivativeHardConstraints,
  // nl_impl.h:764-805, including its free_deriv_counter that only advances for derivatives <= derivative_to_optimize), the
  // initial steps (initial_stepsize_rel |x|, 1e-13 for zeros) and the stopping rules (ftol_rel -> 3, xtol_rel -> 4, maxeval -> 5)
  // are the reference's; the search is a bound-constrained coordinate pattern search whose 2n trial points per iteration are
  // evaluated together on the device (tg_time_alloc_dfo_batch).  max_iterations counts those iterations.  PARITY UNPINNED against
  // BOBYQA's iterates.
  int optimizeDerivativeFree() {
    std::vector<PolynomialOptimizationNonLinear*> one(1, this);
    std::vector<int> codes;
    return optimizeBatch(one, &codes) ? codes[0] : -1;
  }
  // optimize() of many problems with the same derivative-free method, parameters and constraint list in ONE device call.
  // Returns false, touching nothing, when the list is empty or the problems differ in parameters, derivative_to_optimize or
  // constraints, when a method is kMellingerOuterLoop or unknown, or when the call fails; codes (optional) gets each problem's code.
  static bool optimizeBatch(std::vector<PolynomialOptimizationNonLinear*>& problems, std::vector<int>* codes) {
    if (problems.empty()) return false;
    const PolynomialOptimizationNonLinear& f = *problems[0];
    const NonlinearOptimizationParameters& q = f.optimization_parameters_;
    const int method = (int)q.time_alloc_method;
    if (!(method == 0 || method == 1 || method == 3 || method == 4)) return false;
    for (const PolynomialOptimizationNonLinear* o : problems) {
      if (!o) return false;
      const NonlinearOptimizationParameters& r = o->optimization_parameters_;
      if (r.time_alloc_method != q.time_alloc_method || r.max_iterations != q.max_iterations || r.f_rel != q.f_rel || r.x_rel != q.x_rel ||
          r.initial_stepsize_rel != q.initial_stepsize_rel || r.time_penalty != q.time_penalty || r.use_soft_constraints != q.use_soft_constraints ||
          r.soft_constraint_weight != q.soft_constraint_weight || o->poly_opt_.getDerivativeToOptimize() != f.poly_opt_.getDerivativeToOptimize() ||
          o->constraint_dimension_ != f.constraint_dimension_ || o->constraint_derivative_ != f.constraint_derivative_ ||
          o->constraint_value_ != f.constraint_value_)
        return false;
    }
    const int B = (int)problems.size();
    std::vector<int> vtx_off(1, 0);
    std::vector<uint8_t> mask;
    std::vector<double> vals, times;
    for (const PolynomialOptimizationNonLinear* o : problems) {
      std::vector<double> t;
      o->poly_opt_.getSegmentTimes(&t);
      if (t.empty()) return false;
      mask.insert(mask.end(), o->poly_opt_.vertexMasks().begin(), o->poly_opt_.vertexMasks().end());
      vals.insert(vals.end(), o->poly_opt_.vertexValues().begin(), o->poly_opt_.vertexValues().end());
      times.insert(times.end(), t.begin(), t.end());
      vtx_off.push_back((int)mask.size());
    }
    tg_dfo_params P;
    tg_default_dfo_params(&P);
    P.time_alloc_method = method;
    P.derivative_to_optimize = f.poly_opt_.getDerivativeToOptimize();
    P.max_iterations = q.max_iterations;
    P.f_rel = q.f_rel;
    P.x_rel = q.x_rel;
    P.initial_stepsize_rel = q.initial_stepsize_rel;
    P.time_penalty = q.time_penalty;
    P.use_soft_constraints = q.use_soft_constraints ? 1 : 0;
    P.soft_constraint_weight = q.soft_constraint_weight;
    std::vector<double> coef(times.size() * b200::kD * b200::kN), total(B), parts(3 * (size_t)B);
    std::vector<int> code(B), iters(B);
    b200::Context& c = b200::Context::instance();
    const int rc = tg_time_alloc_dfo_batch(c.get(), B, vtx_off.data(), mask.data(), vals.data(), times.data(), &P, (int)f.constraint_derivative_.size(),
                                           f.constraint_dimension_.data(), f.constraint_derivative_.data(), f.constraint_value_.data(), coef.data(),
                                           nullptr, code.data(), iters.data(), total.data(), parts.data());
    if (rc != TG_OK) {
      std::printf("[PolynomialOptimizationNonLinear]: optimize failed: %s\n", tg_last_error(c.get()));
      return false;
    }
    size_t s0 = 0;
    for (int p = 0; p < B; ++p) {
      PolynomialOptimizationNonLinear& o = *problems[p];
      const size_t S = (size_t)(vtx_off[p + 1] - vtx_off[p] - 1);
      o.poly_opt_.adopt(std::vector<double>(times.begin() + s0, times.begin() + s0 + S),
                        std::vector<double>(coef.begin() + s0 * b200::kD * b200::kN, coef.begin() + (s0 + S) * b200::kD * b200::kN), parts[3 * p]);
      o.optimization_info_.cost_trajectory = parts[3 * p];
      o.optimization_info_.cost_time = parts[3 * p + 1];
      o.optimization_info_.cost_soft_constraints = parts[3 * p + 2];
      o.optimization_info_.n_iterations = iters[p];
      o.optimization_info_.stopping_reason = code[p];
      s0 += S;
    }
    if (codes) codes->assign(code.begin(), code.end());
    return true;
  }
  void getTrajectory(Trajectory* trajectory) const { poly_opt_.getTrajectory(trajectory); }
  const PolynomialOptimization<_N>& getPolynomialOptimizationRef() const { return poly_opt_; }
  PolynomialOptimization<_N>& getPolynomialOptimizationRef() { return poly_opt_; }
  OptimizationInfo getOptimizationInfo() const { return optimization_info_; }

 private:
  PolynomialOptimization<_N> poly_opt_;
  NonlinearOptimizationParameters optimization_parameters_;
  OptimizationInfo optimization_info_;
  double limits_[9];
  std::vector<int> constraint_dimension_;
  std::vector<int> constraint_derivative_;   // in the order the constraints were added (inequality_constraints_, nl.h:223)
  std::vector<double> constraint_value_;
};

// ---- the derivative-free time allocation on PolynomialOptimization<N> of every shape --------------------------------------
// A maximum-magnitude constraint as addMaximumMagnitudeConstraint takes it (nl_impl.h:538-565).
struct MagnitudeConstraint {
  int dimension;
  int derivative;
  double maximum_value;
};
namespace b200 {
inline void split_constraints(const std::vector<MagnitudeConstraint>& constraints, std::vector<int>* dim, std::vector<int>* deriv, std::vector<double>* value) {
  for (const MagnitudeConstraint& c : constraints) {
    dim->push_back(c.dimension);
    deriv->push_back(c.derivative);
    value->push_back(c.maximum_value);
  }
}
inline bool dfo_method(const NonlinearOptimizationParameters& q) {
  const int m = (int)q.time_alloc_method;
  return m == 0 || m == 1 || m == 3 || m == 4;
}
}  // namespace b200

// objectiveFunctionTime / objectiveFunctionTimeAndConstraints (nl_impl.h:567-722) of the problem set up in `problem` at K candidate
// vectors in one call (tg_objective_batch_nd): x = the S segment times (kSquaredTime, kRichterTime), then for the ...AndConstraints
// methods the free derivatives, getDimension() x n_free dimension-major as getFreeConstraints lists them.  parts (optional):
// K x {cost_trajectory, cost_time, cost_soft_constraints}.  Returns false, with a message, when the call is refused.
template <int N>
bool evaluateObjectives(const PolynomialOptimization<N>& problem, const NonlinearOptimizationParameters& parameters,
                        const std::vector<MagnitudeConstraint>& constraints, const std::vector<std::vector<double>>& x, std::vector<double>* total,
                        std::vector<double>* parts = nullptr) {
  if (!total || x.empty() || !b200::dfo_method(parameters)) return false;
  const size_t nvar = x.front().size();
  std::vector<double> flat;
  flat.reserve(x.size() * nvar);
  for (const std::vector<double>& xi : x) {
    if (xi.size() != nvar) return false;
    flat.insert(flat.end(), xi.begin(), xi.end());
  }
  std::vector<int> cdim, cder;
  std::vector<double> cval;
  b200::split_constraints(constraints, &cdim, &cder, &cval);
  std::vector<double> tot(x.size()), pa(3 * x.size());
  b200::Context& c = b200::Context::instance();
  const int rc = tg_objective_batch_nd(c.get(), N, (int)problem.getDimension(), (int)problem.vertexMasks().size(), problem.vertexMasks().data(),
                                       problem.vertexValues().data(), problem.getDerivativeToOptimize(), (int)parameters.time_alloc_method,
                                       (long long)x.size(), flat.data(), (int)nvar, parameters.time_penalty, parameters.use_soft_constraints ? 1 : 0,
                                       parameters.soft_constraint_weight, (int)cder.size(), cder.data(), cval.data(), tot.data(), pa.data(), nullptr);
  if (rc != TG_OK) {
    std::printf("[evaluateObjectives]: %s\n", tg_last_error(c.get()));
    return false;
  }
  *total = tot;
  if (parts) *parts = pa;
  return true;
}

// PolynomialOptimizationNonLinear<N>::optimize() with a derivative-free method (optimizeTime / optimizeTimeAndFreeConstraints,
// nl_impl.h:120-157, 429-536; the search of PolynomialOptimizationNonLinear<10>::optimizeBatch) for many problems set up with
// setupFromVertices, of one shape N, one dimension and one derivative_to_optimize, in ONE device call (tg_time_alloc_dfo_batch_nd;
// N = 10 on 4 dimensions with derivative_to_optimize >= 2 on the tuned tg_time_alloc_dfo_batch, which gives the same bits).  Not a
// reference name.  Afterwards every problem is in the state the reference's poly_opt_ is in: kSquaredTime / kRichterTime
// updateSegmentTimes(final) + solveLinear() (getFreeConstraints returns that solve's d_p), the ...AndConstraints methods
// updateSegmentTimes(final) + setFreeConstraints(final free derivatives).  codes / infos (optional) get each problem's code and
// OptimizationInfo.  Returns false, touching nothing, for an empty list, a problem not set up, mixed shapes, the Mellinger method or
// a refused call.
template <int N>
bool optimizeTimeDerivativeFreeBatch(std::vector<PolynomialOptimization<N>*>& problems, const NonlinearOptimizationParameters& parameters,
                                     const std::vector<MagnitudeConstraint>& constraints, std::vector<int>* codes,
                                     std::vector<OptimizationInfo>* infos) {
  if (problems.empty() || !b200::dfo_method(parameters) || !problems[0]) return false;
  const PolynomialOptimization<N>& f = *problems[0];
  const int dims = (int)f.getDimension(), r = f.getDerivativeToOptimize(), H = N / 2;
  const int B = (int)problems.size();
  std::vector<int> vtx_off(1, 0);
  std::vector<uint8_t> mask;
  std::vector<double> vals, times;
  for (const PolynomialOptimization<N>* o : problems) {
    if (!o || (int)o->getDimension() != dims || o->getDerivativeToOptimize() != r || o->vertexMasks().size() < 2) return false;
    std::vector<double> t;
    o->getSegmentTimes(&t);
    mask.insert(mask.end(), o->vertexMasks().begin(), o->vertexMasks().end());
    vals.insert(vals.end(), o->vertexValues().begin(), o->vertexValues().end());
    times.insert(times.end(), t.begin(), t.end());
    vtx_off.push_back((int)mask.size());
  }
  std::vector<int> cdim, cder;
  std::vector<double> cval;
  b200::split_constraints(constraints, &cdim, &cder, &cval);
  tg_dfo_params P;
  tg_default_dfo_params(&P);
  P.time_alloc_method = (int)parameters.time_alloc_method;
  P.derivative_to_optimize = r;
  P.max_iterations = parameters.max_iterations;
  P.f_rel = parameters.f_rel;
  P.x_rel = parameters.x_rel;
  P.initial_stepsize_rel = parameters.initial_stepsize_rel;
  P.time_penalty = parameters.time_penalty;
  P.use_soft_constraints = parameters.use_soft_constraints ? 1 : 0;
  P.soft_constraint_weight = parameters.soft_constraint_weight;
  const bool with_free = P.time_alloc_method >= 3;
  std::vector<double> coef(times.size() * dims * N), vv(with_free ? vals.size() : 0), total(B), parts(3 * (size_t)B);
  std::vector<int> code(B), iters(B);
  b200::Context& c = b200::Context::instance();
  const bool tuned = N == b200::kN && dims == b200::kD && r >= derivative_order::ACCELERATION;
  const int rc = tuned ? tg_time_alloc_dfo_batch(c.get(), B, vtx_off.data(), mask.data(), vals.data(), times.data(), &P, (int)cder.size(), cdim.data(),
                                                 cder.data(), cval.data(), coef.data(), with_free ? vv.data() : nullptr, code.data(), iters.data(),
                                                 total.data(), parts.data())
                       : tg_time_alloc_dfo_batch_nd(c.get(), N, dims, B, vtx_off.data(), mask.data(), vals.data(), times.data(), &P, (int)cder.size(),
                                                    cdim.data(), cder.data(), cval.data(), coef.data(), with_free ? vv.data() : nullptr, code.data(),
                                                    iters.data(), total.data(), parts.data());
  if (rc != TG_OK) {
    std::printf("[optimizeTimeDerivativeFreeBatch]: %s\n", tg_last_error(c.get()));
    return false;
  }
  if (codes) codes->assign(code.begin(), code.end());
  if (infos) infos->assign(B, OptimizationInfo());
  size_t s0 = 0;
  for (int p = 0; p < B; ++p) {
    PolynomialOptimization<N>& o = *problems[p];
    const int v0 = vtx_off[p], V = vtx_off[p + 1] - v0;
    const size_t S = (size_t)V - 1;
    std::vector<double> free;
    if (with_free) {  // the free slots of vval_out, dimension-major (getFreeConstraints' layout)
      const size_t nf = o.getNumberFreeConstraints();
      free.assign(std::max<size_t>((size_t)dims * nf, 1), 0.0);
      size_t j = 0;
      for (int v = 0; v < V; ++v)
        for (int k = 0; k < H; ++k) {
          if ((mask[v0 + v] >> k) & 1u) continue;
          for (int d = 0; d < dims; ++d) free[(size_t)d * nf + j] = vv[(((size_t)v0 + v) * H + k) * dims + d];
          ++j;
        }
    }
    o.adoptDerivativeFree(std::vector<double>(times.begin() + s0, times.begin() + s0 + S),
                          std::vector<double>(coef.begin() + s0 * dims * N, coef.begin() + (s0 + S) * dims * N), parts[3 * p], with_free ? &free : nullptr);
    if (infos) {
      OptimizationInfo& info = (*infos)[p];
      info.cost_trajectory = parts[3 * p];
      info.cost_time = parts[3 * p + 1];
      info.cost_soft_constraints = parts[3 * p + 2];
      info.n_iterations = iters[p];
      info.stopping_reason = code[p];
    }
    s0 += S;
  }
  return true;
}

// ---- batch entry: the numeric core of optimize() / findTrajectory for many paths (node.cpp:620-851, 857-1209) -------------
struct Waypoint {
  double x, y, z, heading;
  bool stop_at;
};
struct InitialState {  // the TrackerCommand fields findTrajectory reads (node.cpp:925-957)
  double heading;
  double velocity[4], acceleration[4], jerk[4];  // x y z heading-rate
};
// The DynamicsConstraints fields findTrajectory / findTrajectoryFallback read (node.cpp:972-994, 1256-1280)
struct DynamicsConstraints {
  double horizontal_speed, vertical_ascending_speed, vertical_descending_speed;
  double horizontal_acceleration, vertical_ascending_acceleration, vertical_descending_acceleration;
  double horizontal_jerk, vertical_ascending_jerk, vertical_descending_jerk;
  double heading_speed, heading_acceleration, heading_jerk;
};
// The mrs_msgs::Path fields callbackPath / callbackPathSrv / callbackGetPathSrv act on (node.cpp:1847-1902, 2061-2118, 2294-2351).
// use_heading and fly_now only travel into the outgoing TrajectoryReference (node.cpp:1573-1575) and are carried along unchanged.
struct PathRequest {
  struct Point { double x, y, z, heading; };
  std::vector<Point> points;
  bool use_heading = true, fly_now = false, stop_at_waypoints = false, loop = false;
  bool override_constraints = false;
  double override_max_velocity_horizontal = 0, override_max_acceleration_horizontal = 0, override_max_jerk_horizontal = 0;
  double override_max_velocity_vertical = 0, override_max_acceleration_vertical = 0, override_max_jerk_vertical = 0;
  bool relax_heading = false;
  double max_deviation_from_path = 0;   // <= 0: the configured max_deviation
  bool dont_prepend_current_state = false;
  double max_execution_time = 0;        // wall-clock budget of the node's retry loop; not a numeric input of the path
};
struct ResolvedRequest {
  std::vector<Waypoint> waypoints;
  tg_params params;
  bool prepend_state;
  bool constraints_overridden;  // false when the override was refused (node.cpp:1002-1026)
};
struct PathResult {
  tg_result info;
  std::vector<Waypoint> waypoints;    // after subdivision
  Trajectory trajectory;              // final segments
  std::vector<double> samples_xyzh;   // [M][4] as getTrajectoryReference emits them (node.cpp:1578-1602)
};

class TrajectoryGeneratorBatch {
 public:
  explicit TrajectoryGeneratorBatch(int device = 0) : device_(device), devices_(1, device) { tg_default_params(&params); }
  // several GPUs of one box: the paths of a call are sharded by index over the devices (contiguous blocks, one context and one
  // host thread per device, no exchange between them -- SURVEY.md 8e)
  explicit TrajectoryGeneratorBatch(const std::vector<int>& devices) : device_(devices.empty() ? 0 : devices[0]), devices_(devices.empty() ? std::vector<int>(1, 0) : devices) {
    tg_default_params(&params);
  }
  tg_params params;  // production defaults (SURVEY.md section 5); edit before optimize()
  const std::vector<int>& devices() const { return devices_; }

  // initial_states: empty (no prepended state, node.cpp:508-510) or one per path
  bool optimize(const std::vector<std::vector<Waypoint>>& paths, const std::vector<InitialState>& initial_states, std::vector<PathResult>* out) {
    if (!out) return false;
    const int B = (int)paths.size();
    if (B < 1 || (!initial_states.empty() && (int)initial_states.size() != B)) return false;
    const int G = (int)std::min<size_t>(devices_.size(), (size_t)B);
    if (G <= 1) return optimize_on(device_, paths, initial_states, 0, B, out, true);
    std::vector<int> slot(G, 0);  // a device listed twice gets two contexts (two host threads on one GPU)
    for (int g = 0; g < G; ++g) {
      for (int h = 0; h < g; ++h)
        if (devices_[h] == devices_[g]) ++slot[g];
      b200::Context::instance(devices_[g], slot[g]);  // create the contexts before the threads start
    }
    out->assign(B, PathResult());
    std::vector<int> ok(G, 0);
    std::vector<std::thread> workers;
    for (int g = 0; g < G; ++g) {
      const int p0 = (int)((long long)B * g / G), p1 = (int)((long long)B * (g + 1) / G);
      workers.emplace_back([this, &paths, &initial_states, out, &ok, &slot, g, p0, p1]() {
        ok[g] = optimize_on(devices_[g], paths, initial_states, p0, p1, out, false, slot[g]) ? 1 : 0;
      });
    }
    for (std::thread& t : workers) t.join();
    for (int g = 0; g < G; ++g)
      if (!ok[g]) return false;
    return true;
  }

  // What the path callback turns one message into before optimize() runs: the waypoint list (stop_at on every point, the first
  // point appended again for a loop, node.cpp:1885-1906), the limits findTrajectory will use (node.cpp:972-1040) and the deviation
  // bound (node.cpp:1875-1879).  `base` carries everything the message does not touch.  The caller applies checkNaN itself.
  static ResolvedRequest resolveRequest(const PathRequest& req, const DynamicsConstraints& constraints, const tg_params& base, const InitialState* state) {
    ResolvedRequest out;
    out.params = base;
    out.prepend_state = state != nullptr && !req.dont_prepend_current_state;  // node.cpp:508-510
    out.constraints_overridden = false;
    for (const PathRequest::Point& q : req.points) out.waypoints.push_back(Waypoint{q.x, q.y, q.z, q.heading, req.stop_at_waypoints});
    if (req.loop && !out.waypoints.empty()) out.waypoints.push_back(out.waypoints.front());
    double* L = out.params.limits;  // v_h, v_v, a_h, a_v, j_h, j_v, v_hdg, a_hdg, j_hdg
    L[0] = constraints.horizontal_speed;
    L[1] = std::min(constraints.vertical_ascending_speed, constraints.vertical_descending_speed);
    L[2] = constraints.horizontal_acceleration;
    L[3] = std::min(constraints.vertical_ascending_acceleration, constraints.vertical_descending_acceleration);
    L[4] = constraints.horizontal_jerk;
    L[5] = std::min(constraints.vertical_ascending_jerk, constraints.vertical_descending_jerk);
    if (req.override_constraints) {
      // the callbacks store override_max_jerk_HORIZONTAL into the vertical slot (node.cpp:1856, 2070, 2303); the message's own
      // override_max_jerk_vertical is never read
      const double o_jv = req.override_max_jerk_horizontal;
      bool can_change = true;
      if (out.prepend_state) {  // findTrajectory's initial_state is the prepended one (node.cpp:1002-1009)
        const InitialState& s = *state;
        can_change = (std::hypot(s.velocity[0], s.velocity[1]) < req.override_max_velocity_horizontal) &&
                     (std::hypot(s.acceleration[0], s.acceleration[1]) < req.override_max_acceleration_horizontal) &&
                     (std::hypot(s.jerk[0], s.jerk[1]) < req.override_max_jerk_horizontal) && (std::fabs(s.velocity[2]) < req.override_max_velocity_vertical) &&
                     (std::fabs(s.acceleration[2]) < req.override_max_acceleration_vertical) && (std::fabs(s.jerk[2]) < o_jv);
      }
      if (can_change) {
        L[0] = req.override_max_velocity_horizontal; L[2] = req.override_max_acceleration_horizontal; L[4] = req.override_max_jerk_horizontal;
        L[1] = req.override_max_velocity_vertical;   L[3] = req.override_max_acceleration_vertical;   L[5] = o_jv;
        out.constraints_overridden = true;
      }
    }
    if (req.relax_heading) {
      L[6] = L[7] = L[8] = (double)std::numeric_limits<float>::max();  // node.cpp:1030-1034
    } else {
      L[6] = constraints.heading_speed; L[7] = constraints.heading_acceleration; L[8] = constraints.heading_jerk;
    }
    if (req.max_deviation_from_path > 0) out.params.max_deviation = req.max_deviation_from_path;
    return out;
  }
  // Many path messages in one go: requests whose resolved parameters agree share one batch call (one call when no message overrides
  // anything).  states: empty, or the current tracker state per request (ignored where dont_prepend_current_state is set).
  bool optimizeRequests(const std::vector<PathRequest>& requests, const DynamicsConstraints& constraints, const std::vector<InitialState>& states,
                        std::vector<PathResult>* out, std::vector<ResolvedRequest>* resolved_out = nullptr) {
    if (!out) return false;
    const int R = (int)requests.size();
    if (R < 1 || (!states.empty() && (int)states.size() != R)) return false;
    std::vector<ResolvedRequest> resolved;
    for (int i = 0; i < R; ++i) resolved.push_back(resolveRequest(requests[i], constraints, params, states.empty() ? nullptr : &states[i]));
    out->assign(R, PathResult());
    std::vector<char> done(R, 0);
    const tg_params saved = params;
    bool ok = true;
    for (int i = 0; i < R && ok; ++i) {
      if (done[i]) continue;
      std::vector<int> members;
      for (int j = i; j < R; ++j)
        if (!done[j] && resolved[j].prepend_state == resolved[i].prepend_state && same_params(resolved[j].params, resolved[i].params)) members.push_back(j);
      std::vector<std::vector<Waypoint>> paths;
      std::vector<InitialState> group_states;
      for (int j : members) {
        done[j] = 1;
        paths.push_back(resolved[j].waypoints);
        if (resolved[i].prepend_state) group_states.push_back(states[j]);
      }
      std::vector<PathResult> part;
      params = resolved[i].params;
      ok = optimize(paths, group_states, &part);
      params = saved;
      if (ok)
        for (size_t k = 0; k < members.size(); ++k) (*out)[members[k]] = std::move(part[k]);
    }
    if (resolved_out) *resolved_out = std::move(resolved);
    return ok;
  }

 private:
  static bool same_params(const tg_params& a, const tg_params& b) {
    bool same = a.derivative_to_optimize == b.derivative_to_optimize && a.max_evals == b.max_evals && a.f_rel == b.f_rel && a.x_rel == b.x_rel && a.dt == b.dt &&
                a.check_deviation == b.check_deviation && a.max_deviation == b.max_deviation && a.max_deviation_iters == b.max_deviation_iters &&
                a.first_segment_checked == b.first_segment_checked && a.max_len_factor == b.max_len_factor && a.min_len_factor == b.min_len_factor &&
                a.run_time_alloc == b.run_time_alloc && a.override_heading_atan2 == b.override_heading_atan2;
    for (int k = 0; k < 9; ++k) same = same && a.limits[k] == b.limits[k];
    return same;
  }
  // paths [p0, p1) on one device; results into (*out)[p0 .. p1)
  bool optimize_on(int device, const std::vector<std::vector<Waypoint>>& all_paths, const std::vector<InitialState>& all_states, int p0, int p1,
                   std::vector<PathResult>* out_all, bool resize_out, int slot = 0) {
    const std::vector<std::vector<Waypoint>> paths(all_paths.begin() + p0, all_paths.begin() + p1);
    const std::vector<InitialState> initial_states(all_states.empty() ? all_states.begin() : all_states.begin() + p0,
                                                   all_states.empty() ? all_states.begin() : all_states.begin() + p1);
    std::vector<PathResult> local;
    std::vector<PathResult>* out = &local;
    const int B = (int)paths.size();
    std::vector<int> wp_off(B + 1, 0);
    for (int p = 0; p < B; ++p) wp_off[p + 1] = wp_off[p] + (int)paths[p].size();
    std::vector<double> wp((size_t)wp_off[B] * 4);
    std::vector<uint8_t> stop(wp_off[B]);
    for (int p = 0; p < B; ++p)
      for (size_t i = 0; i < paths[p].size(); ++i) {
        const Waypoint& w = paths[p][i];
        double* dst = &wp[((size_t)wp_off[p] + i) * 4];
        dst[0] = w.x; dst[1] = w.y; dst[2] = w.z; dst[3] = w.heading;
        stop[wp_off[p] + i] = w.stop_at ? 1 : 0;
      }
    std::vector<double> init14;
    if (!initial_states.empty()) {
      init14.resize((size_t)B * 14);
      for (int p = 0; p < B; ++p) {
        double* d = &init14[(size_t)p * 14];
        d[0] = 1.0;
        d[1] = initial_states[p].heading;
        for (int k = 0; k < 4; ++k) { d[2 + k] = initial_states[p].velocity[k]; d[6 + k] = initial_states[p].acceleration[k]; d[10 + k] = initial_states[p].jerk[k]; }
      }
    }
    b200::Context& c = b200::Context::instance(device, slot);
    std::vector<tg_result> res(B);
    long long totals[2] = {0, 0};
    int rc = tg_optimize_batch(c.get(), B, wp_off.data(), wp.data(), stop.data(), init14.empty() ? nullptr : init14.data(), &params, 0, res.data(), totals);
    if (rc != TG_OK) {
      std::printf("[TrajectoryGeneratorBatch]: %s\n", tg_last_error(c.get()));
      return false;
    }
    std::vector<int> seg_off(B + 1), smp_off(B + 1);
    std::vector<double> o_wp((size_t)(totals[0] + B) * 4), times((size_t)totals[0]), coef((size_t)totals[0] * 40), samples((size_t)totals[1] * 4);
    rc = tg_fetch_outputs(c.get(), seg_off.data(), o_wp.data(), times.data(), coef.data(), smp_off.data(), samples.data());
    if (rc != TG_OK) return false;
    out->assign(B, PathResult());
    for (int p = 0; p < B; ++p) {
      PathResult& r = (*out)[p];
      r.info = res[p];
      const int s0 = seg_off[p], s1 = seg_off[p + 1];
      if (s1 > s0) {
        for (int v = s0 + p; v <= s1 + p; ++v) r.waypoints.push_back(Waypoint{o_wp[(size_t)v * 4], o_wp[(size_t)v * 4 + 1], o_wp[(size_t)v * 4 + 2], o_wp[(size_t)v * 4 + 3], false});
        r.trajectory.unpack(std::vector<double>(coef.begin() + (size_t)s0 * 40, coef.begin() + (size_t)s1 * 40),
                            std::vector<double>(times.begin() + s0, times.begin() + s1));
      }
      r.samples_xyzh.assign(samples.begin() + (size_t)smp_off[p] * 4, samples.begin() + (size_t)smp_off[p + 1] * 4);
    }
    if (resize_out) out_all->assign(all_paths.size(), PathResult());
    for (int p = 0; p < B; ++p) (*out_all)[p0 + p] = std::move(local[p]);
    return true;
  }

 public:
  // MrsTrajectoryGeneration::preprocessPath (node.cpp:431-500) for one path
  std::vector<Waypoint> preprocessPath(const std::vector<Waypoint>& in, double min_waypoint_distance = 0.05, bool straightener = false,
                                       double max_deviation = 0.05, double max_hdg_deviation = 0.1) const {
    std::vector<Waypoint> out;
    const int V = (int)in.size();
    if (V < 1) return out;
    const int wp_off[2] = {0, V};
    std::vector<double> wp((size_t)V * 4), owp((size_t)V * 4);
    std::vector<uint8_t> stop(V), ostop(V);
    for (int i = 0; i < V; ++i) {
      wp[4 * i] = in[i].x; wp[4 * i + 1] = in[i].y; wp[4 * i + 2] = in[i].z; wp[4 * i + 3] = in[i].heading;
      stop[i] = in[i].stop_at ? 1 : 0;
    }
    int count = 0;
    b200::Context& c = b200::Context::instance(device_);
    c.check(tg_preprocess_paths(c.get(), 1, wp_off, wp.data(), stop.data(), min_waypoint_distance, straightener ? 1 : 0, max_deviation, max_hdg_deviation,
                                &count, owp.data(), ostop.data()), "tg_preprocess_paths");
    for (int i = 0; i < count; ++i) out.push_back(Waypoint{owp[4 * i], owp[4 * i + 1], owp[4 * i + 2], owp[4 * i + 3], ostop[i] != 0});
    return out;
  }
  // MrsTrajectoryGeneration::findTrajectoryFallback (node.cpp:1215-1395) for one path: samples x y z heading, [M][4].
  // speed_factor / accel_factor / stopping_time: config/public/trajectory_generation.yaml:47-54
  std::vector<double> findTrajectoryFallback(const std::vector<Waypoint>& in, double speed_factor = 1.0, double accel_factor = 1.0,
                                             double stopping_time = 2.0) const {
    const int V = (int)in.size();
    std::vector<double> samples;
    if (V < 2) return samples;
    const int wp_off[2] = {0, V};
    std::vector<double> wp((size_t)V * 4);
    std::vector<uint8_t> stop(V);
    for (int i = 0; i < V; ++i) {
      wp[4 * i] = in[i].x; wp[4 * i + 1] = in[i].y; wp[4 * i + 2] = in[i].z; wp[4 * i + 3] = in[i].heading;
      stop[i] = in[i].stop_at ? 1 : 0;
    }
    double L[9];
    for (int i = 0; i < 9; ++i) L[i] = params.limits[i];
    L[0] *= speed_factor; L[1] *= speed_factor; L[2] *= accel_factor; L[3] *= accel_factor;  // node.cpp:1296-1300
    int count = 0;
    b200::Context& c = b200::Context::instance(device_);
    c.check(tg_fallback_sample_batch(c.get(), 1, wp_off, wp.data(), stop.data(), L, params.dt, stopping_time, &count, nullptr), "tg_fallback_sample_batch");
    samples.resize((size_t)count * 4);
    if (count > 0)
      c.check(tg_fallback_sample_batch(c.get(), 1, wp_off, wp.data(), stop.data(), L, params.dt, stopping_time, &count, samples.data()), "tg_fallback_sample_batch");
    return samples;
  }
  // MrsTrajectoryGeneration::getWaypointInTrajectoryIdxs (node.cpp:1461-1499) for one path
  std::vector<int> getWaypointInTrajectoryIdxs(const std::vector<double>& samples_xyzh, const std::vector<Waypoint>& waypoints) const {
    const int V = (int)waypoints.size(), M = (int)(samples_xyzh.size() / 4);
    std::vector<int> idxs(V > 0 ? V : 1);
    if (V < 1 || M < 1) return std::vector<int>();
    const int wp_off[2] = {0, V}, smp_off[2] = {0, M};
    std::vector<double> wp((size_t)V * 4);
    for (int i = 0; i < V; ++i) { wp[4 * i] = waypoints[i].x; wp[4 * i + 1] = waypoints[i].y; wp[4 * i + 2] = waypoints[i].z; wp[4 * i + 3] = waypoints[i].heading; }
    int count = 0;
    b200::Context& c = b200::Context::instance(device_);
    c.check(tg_waypoint_idxs_batch(c.get(), 1, smp_off, samples_xyzh.data(), wp_off, wp.data(), &count, idxs.data()), "tg_waypoint_idxs_batch");
    idxs.resize(count);
    return idxs;
  }

 private:
  int device_;
  std::vector<int> devices_;
};

}  // namespace eth_trajectory_generation

#endif  // ETH_TRAJECTORY_GENERATION_B200_HPP_
