// tests/cpp/test_shim_sample_range.cpp -- sampleTrajectoryInRange / sampleTrajectoryStartDuration / sampleTrajectoriesInRange and
// evaluateRange of the drop-in header, for PolynomialOptimization<10>(4) and <8>(3) trajectories.  Built twice by
// tests/test_sample_range.py: with the header's TrajectoryPoint (no Eigen), and with -DTG_TEST_EIGEN_POINT against the Eigen stand-in of
// oracle/ref_shim/ and an EigenTrajectoryPoint-shaped point (the reference's own eth_mav_msgs/eigen_mav_msgs.h where a checkout of the
// reference is present).  Dumps hex floats, which the test compares bit for bit with the oracle.
#if defined(TG_TEST_EIGEN_POINT)
#include <Eigen/Core>
#include <Eigen/Geometry>
#endif
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

#if defined(TG_TEST_EIGEN_POINT) && defined(__has_include) && __has_include(<eth_mav_msgs/eigen_mav_msgs.h>)
#include <eth_mav_msgs/eigen_mav_msgs.h>
typedef eth_mav_msgs::EigenTrajectoryPoint PointT;
#elif defined(TG_TEST_EIGEN_POINT)
struct PointT {  // the fields and accessors of eth_mav_msgs::EigenTrajectoryPoint that the sampler touches
  typedef std::vector<PointT> Vector;
  int64_t time_from_start_ns = 0;
  Eigen::Vector3d position_W, velocity_W, acceleration_W, jerk_W, snap_W, angular_velocity_W, angular_acceleration_W;
  Eigen::Quaterniond orientation_W_B;
  void setFromYaw(double yaw) { orientation_W_B = Eigen::Quaterniond(Eigen::AngleAxisd(yaw, Eigen::Vector3d::UnitZ())); }
  void setFromYawRate(double r) { angular_velocity_W = Eigen::Vector3d(0.0, 0.0, r); }
  void setFromYawAcc(double a) { angular_acceleration_W = Eigen::Vector3d(0.0, 0.0, a); }
};
#endif

#include "../../include/eth_trajectory_generation_b200.hpp"

using namespace eth_trajectory_generation;
#if !defined(TG_TEST_EIGEN_POINT)
typedef TrajectoryPoint PointT;
#endif

static void dump(FILE* f, const std::string& key, const double* v, size_t n) {
  std::fprintf(f, "%s %zu", key.c_str(), n);
  for (size_t i = 0; i < n; ++i) std::fprintf(f, " %a", v[i]);
  std::fprintf(f, "\n");
}

// per state: t_ns, p3 v3 a3 j3 s3, yaw rate, yaw acceleration (zero for a 3-dimensional trajectory, which sets no yaw)
#if defined(TG_TEST_EIGEN_POINT)
static double yaw_rate(const PointT& s) { return s.angular_velocity_W[2]; }
static double yaw_acc(const PointT& s) { return s.angular_acceleration_W[2]; }
#else
static double yaw_rate(const PointT& s) { return s.yaw_rate; }
static double yaw_acc(const PointT& s) { return s.yaw_acc; }
#endif
static void dump_states(FILE* f, const std::string& key, const std::vector<PointT>& states) {
  std::vector<double> v;
  for (const PointT& s : states) {
    v.push_back((double)s.time_from_start_ns);
    for (int k = 0; k < 3; ++k) v.push_back(s.position_W[k]);
    for (int k = 0; k < 3; ++k) v.push_back(s.velocity_W[k]);
    for (int k = 0; k < 3; ++k) v.push_back(s.acceleration_W[k]);
    for (int k = 0; k < 3; ++k) v.push_back(s.jerk_W[k]);
    for (int k = 0; k < 3; ++k) v.push_back(s.snap_W[k]);
    v.push_back(yaw_rate(s));
    v.push_back(yaw_acc(s));
  }
  dump(f, key, v.data(), v.size());
}

template <int N>
static bool make(int dims, double t0, Trajectory* t) {
  Vertex::Vector vertices;
  for (int i = 0; i < 6; ++i) {
    const double w[4] = {1.7 * i, (i % 2 == 0) ? 0.6 : -0.4, 3.0 + 0.25 * i, 0.15 * i};
    Vector p = b200::make_vector((size_t)dims, 0.0);
    for (int d = 0; d < dims; ++d) p[d] = w[d];
    Vertex v(dims);
    if (i == 0 || i == 5) v.makeStartOrEnd(p, 2);
    else v.addConstraint(derivative_order::POSITION, p);
    vertices.push_back(v);
  }
  std::vector<double> times;
  for (int i = 0; i < 5; ++i) times.push_back(t0 + 0.3 * (double)(i % 3));
  PolynomialOptimization<N> opt(dims);
  if (!opt.setupFromVertices(vertices, times, 2) || !opt.solveLinear()) return false;
  opt.getTrajectory(t);
  return true;
}

int main(int argc, char** argv) {
  if (argc < 2) return 1;
  FILE* f = std::fopen(argv[1], "w");
  if (!f) return 2;
  std::vector<Trajectory> trajs(3);
  if (!make<10>(4, 0.8, &trajs[0]) || !make<10>(4, 1.1, &trajs[1]) || !make<8>(3, 0.9, &trajs[2])) return 3;
  for (size_t i = 0; i < trajs.size(); ++i) {
    std::vector<double> coef, times;
    trajs[i].pack(&coef, &times);
    dump(f, "coef" + std::to_string(i), coef.data(), coef.size());
    dump(f, "times" + std::to_string(i), times.data(), times.size());
  }
  for (size_t i = 0; i < trajs.size(); ++i) {
    const Trajectory& t = trajs[i];
    const double end = t.getMaxTime(), mid = 0.5 * t.getSegmentTimes()[0];
    const std::string k = std::to_string(i);
    std::vector<PointT> states;
    double ok[6];
    ok[0] = sampleTrajectoryInRange(t, mid, 0.7 * end, 0.05, &states);
    dump_states(f, "in_range" + k, states);
    ok[1] = sampleTrajectoryStartDuration(t, mid, 0.3 * end, 0.07, &states);
    dump_states(f, "start_duration" + k, states);
    ok[2] = sampleTrajectoryInRange(t, 0.0, end, 0.2, &states);  // = sampleWholeTrajectory
    dump_states(f, "whole_range" + k, states);
    ok[3] = sampleWholeTrajectory(t, 0.2, &states);
    dump_states(f, "whole" + k, states);
    ok[4] = sampleTrajectoryInRange(t, mid, end + 0.5, 0.05, &states);  // outside [getMinTime(), getMaxTime()]: refused as upstream
    ok[5] = sampleTrajectoryInRange(t, -0.1, end, 0.05, &states) || !states.empty();
    dump(f, "ok" + k, ok, 6);
    std::vector<Vector> range;
    std::vector<double> st, flat;
    t.evaluateRange(mid, end + 1.0, 0.09, derivative_order::ACCELERATION, &range, &st);
    for (const Vector& v : range)
      for (int d = 0; d < t.D(); ++d) flat.push_back(v[d]);
    dump(f, "range" + k, flat.data(), flat.size());
    dump(f, "range_t" + k, st.data(), st.size());
  }
  // the batch: the two N = 10 trajectories with windows past their ends, one call
  std::vector<Trajectory> two(trajs.begin(), trajs.begin() + 2);
  const std::vector<std::pair<double, double>> windows = {{0.3, 1e9}, {0.5 * two[1].getMaxTime(), 2.0 * two[1].getMaxTime()}};
  std::vector<std::vector<PointT>> per;
  double batch_ok = sampleTrajectoriesInRange(two, windows, 0.04, &per) ? 1.0 : 0.0;
  dump(f, "batch_ok", &batch_ok, 1);
  for (size_t i = 0; i < per.size(); ++i) dump_states(f, "batch" + std::to_string(i), per[i]);
  // mixed shapes are refused
  std::vector<std::vector<PointT>> none;
  const double mixed = sampleTrajectoriesInRange(trajs, {{0, 1}, {0, 1}, {0, 1}}, 0.1, &none) ? 1.0 : 0.0;
  dump(f, "mixed_ok", &mixed, 1);
  std::fclose(f);
  return 0;
}
