// tests/cpp/test_shim_eigen.cpp -- the drop-in header with REFERENCE-TYPED call sites: Eigen::Vector4d / Eigen::VectorXd
// arguments and results and an EigenTrajectoryPoint result type, written the way MrsTrajectoryGeneration::findTrajectory
// writes them (src/mrs_trajectory_generation.cpp:923-977, 1063-1169).  Eigen itself is absent from this image: the test
// compiles against the stand-in of oracle/ref_shim/ (TEST INFRASTRUCTURE), and -- where a checkout of the reference is present -- against
// the reference's own eth_mav_msgs/eigen_mav_msgs.h for the point type.  Also: optimize() for a derivative-free time
// allocation method and the multi-context TrajectoryGeneratorBatch.  Dumps hex floats for tests/test_cpp_shim.py.
#include <Eigen/Core>
#include <Eigen/Geometry>
#include <cstdio>

#if defined(__has_include) && __has_include(<eth_mav_msgs/eigen_mav_msgs.h>)
#include <eth_mav_msgs/eigen_mav_msgs.h>
typedef eth_mav_msgs::EigenTrajectoryPoint PointT;
#define TG_TEST_POINT "reference eth_mav_msgs::EigenTrajectoryPoint"
#else
// the fields and accessors of eth_mav_msgs::EigenTrajectoryPoint that the sampler and the node touch
struct PointT {
  typedef std::vector<PointT> Vector;
  int64_t time_from_start_ns = 0;
  Eigen::Vector3d position_W, velocity_W, acceleration_W, jerk_W, snap_W, angular_velocity_W, angular_acceleration_W;
  Eigen::Quaterniond orientation_W_B;
  void setFromYaw(double yaw) { orientation_W_B = Eigen::Quaterniond(Eigen::AngleAxisd(yaw, Eigen::Vector3d::UnitZ())); }
  void setFromYawRate(double r) { angular_velocity_W = Eigen::Vector3d(0.0, 0.0, r); }
  void setFromYawAcc(double a) { angular_acceleration_W = Eigen::Vector3d(0.0, 0.0, a); }
};
#define TG_TEST_POINT "local EigenTrajectoryPoint look-alike"
#endif

#include "../../include/eth_trajectory_generation_b200.hpp"

using namespace eth_trajectory_generation;

static void dump(FILE* f, const char* key, const double* v, size_t n) {
  std::fprintf(f, "%s %zu", key, n);
  for (size_t i = 0; i < n; ++i) std::fprintf(f, " %a", v[i]);
  std::fprintf(f, "\n");
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  FILE* f = std::fopen(argv[1], "w");
  if (!f) return 2;
  static_assert(std::is_same<Vector, Eigen::VectorXd>::value, "with Eigen on the include path the header's Vector is Eigen::VectorXd");
  const int derivative_to_optimize = derivative_order::ACCELERATION;
  const int dimension = 4;
  // node.cpp:931-977, verbatim shapes: Eigen::Vector4d temporaries into makeStartOrEnd / addConstraint
  Vertex::Vector vertices;
  const int n_wp = 7;
  for (int i = 0; i < n_wp; i++) {
    const double x = 1.5 * i, y = (i % 2 == 0) ? 0.4 : -0.6, z = 4.0 + 0.1 * i, heading = 0.2 * i;
    Vertex vertex(dimension);
    if (i == 0) {
      vertex.makeStartOrEnd(Eigen::Vector4d(x, y, z, heading), derivative_to_optimize);
      vertex.addConstraint(derivative_order::POSITION, Eigen::Vector4d(x, y, z, heading));
      vertex.addConstraint(derivative_order::VELOCITY, Eigen::Vector4d(0.3, -0.1, 0.05, 0.02));
      vertex.addConstraint(derivative_order::ACCELERATION, Eigen::Vector4d(0.0, 0.1, 0.0, 0.0));
      vertex.addConstraint(derivative_order::JERK, Eigen::Vector4d(0, 0, 0, 0));
    } else if (i == n_wp - 1) {
      vertex.makeStartOrEnd(Eigen::Vector4d(x, y, z, heading), derivative_to_optimize);
      vertex.addConstraint(derivative_order::POSITION, Eigen::Vector4d(x, y, z, heading));
    } else {
      vertex.addConstraint(derivative_order::POSITION, Eigen::Vector4d(x, y, z, heading));
    }
    vertices.push_back(vertex);
  }
  std::vector<double> times;
  for (int i = 0; i + 1 < n_wp; ++i) times.push_back(0.9 + 0.2 * (i % 3));
  // an Eigen::VectorXd read back out of a vertex
  Eigen::VectorXd c0;
  if (!vertices[0].getConstraint(derivative_order::VELOCITY, &c0) || c0.size() != 4) return 3;
  dump(f, "vtx0_vel", c0.data(), 4);

  NonlinearOptimizationParameters parameters;
  parameters.f_rel = 0.05;
  parameters.x_rel = 0.1;
  parameters.max_iterations = 10;
  parameters.time_alloc_method = NonlinearOptimizationParameters::kMellingerOuterLoop;
  PolynomialOptimizationNonLinear<10> opt(dimension, parameters);
  opt.setupFromVertices(vertices, times, derivative_to_optimize);
  const double L[9] = {4.0, 2.0, 2.0, 1.0, 20.0, 20.0, 1.0, 2.0, 10.0};
  for (int dim = 0; dim < 4; ++dim) {
    const int g = dim <= 1 ? 0 : (dim == 2 ? 1 : -1);
    opt.addMaximumMagnitudeConstraint(dim, derivative_order::VELOCITY, g >= 0 ? L[g] : L[6]);
    opt.addMaximumMagnitudeConstraint(dim, derivative_order::ACCELERATION, g >= 0 ? L[2 + g] : L[7]);
    opt.addMaximumMagnitudeConstraint(dim, derivative_order::JERK, g >= 0 ? L[4 + g] : L[8]);
  }
  opt.optimize();
  const double meta[3] = {(double)opt.getOptimizationInfo().stopping_reason, (double)opt.getOptimizationInfo().n_iterations, opt.getOptimizationInfo().cost_trajectory};
  dump(f, "nl_meta", meta, 3);
  Segment::Vector segments;
  opt.getPolynomialOptimizationRef().getSegments(&segments);
  Trajectory trajectory;
  opt.getTrajectory(&trajectory);
  std::vector<double> coef, ts;
  trajectory.pack(&coef, &ts);
  dump(f, "nl_times", ts.data(), ts.size());
  dump(f, "nl_coef", coef.data(), coef.size());
  // Eigen::VectorXd results
  const Eigen::VectorXd pos = trajectory.evaluate(0.37 * trajectory.getMaxTime(), derivative_order::POSITION);
  const Eigen::VectorXd snap = trajectory.evaluate(0.37 * trajectory.getMaxTime(), derivative_order::SNAP);
  dump(f, "eval_p", pos.data(), 4);
  dump(f, "eval_s", snap.data(), 4);
  // the reference's point type through sampleWholeTrajectory (node.cpp:1162-1166)
  PointT::Vector states;
  const bool success = sampleWholeTrajectory(trajectory, 0.2, &states);
  if (!success) return 4;
  std::vector<double> flat;
  for (const PointT& s : states) {
    flat.push_back(s.position_W[0]); flat.push_back(s.position_W[1]); flat.push_back(s.position_W[2]);
    flat.push_back(s.orientation_W_B.w()); flat.push_back(s.orientation_W_B.z());
    flat.push_back(s.angular_velocity_W.z()); flat.push_back(s.snap_W[1]); flat.push_back((double)s.time_from_start_ns);
  }
  dump(f, "samples", flat.data(), flat.size());
  // evaluateRange: every dimension, jerk, a start time inside the second segment, sampling times returned
  std::vector<Eigen::VectorXd> range;
  std::vector<double> range_t;
  trajectory.evaluateRange(ts[0] + 0.05, trajectory.getMaxTime(), 0.3, derivative_order::JERK, &range, &range_t);
  std::vector<double> rf;
  for (const Eigen::VectorXd& v : range) for (int d = 0; d < 4; ++d) rf.push_back(v[d]);
  dump(f, "range_jerk", rf.data(), rf.size());
  dump(f, "range_t", range_t.data(), range_t.size());

  // optimize() with a derivative-free method (kSquaredTime; the node's time_allocation = 0)
  {
    NonlinearOptimizationParameters po;
    po.time_alloc_method = NonlinearOptimizationParameters::kSquaredTime;
    po.max_iterations = 6;
    PolynomialOptimizationNonLinear<10> oo(dimension, po);
    oo.setupFromVertices(vertices, times, derivative_to_optimize);
    oo.addMaximumMagnitudeConstraint(0, derivative_order::VELOCITY, 4.0);
    oo.addMaximumMagnitudeConstraint(0, derivative_order::ACCELERATION, 2.0);
    const int code = oo.optimize();
    Trajectory t0;
    oo.getTrajectory(&t0);
    std::vector<double> c2, t2;
    t0.pack(&c2, &t2);
    const OptimizationInfo oi = oo.getOptimizationInfo();
    const double m[5] = {(double)code, (double)oi.n_iterations, oi.cost_trajectory, oi.cost_time, oi.cost_soft_constraints};
    dump(f, "df_meta", m, 5);
    dump(f, "df_times", t2.data(), t2.size());
    dump(f, "df_coef", c2.data(), c2.size());
  }
  {
    NonlinearOptimizationParameters po;
    po.time_alloc_method = NonlinearOptimizationParameters::kRichterTimeAndConstraints;
    po.max_iterations = 3;
    PolynomialOptimizationNonLinear<10> oo(dimension, po);
    oo.setupFromVertices(vertices, times, derivative_to_optimize);
    oo.addMaximumMagnitudeConstraint(0, derivative_order::VELOCITY, 4.0);
    oo.addMaximumMagnitudeConstraint(2, derivative_order::ACCELERATION, 1.0);
    const int code = oo.optimize();
    Trajectory t0;
    oo.getTrajectory(&t0);
    std::vector<double> c2, t2;
    t0.pack(&c2, &t2);
    const OptimizationInfo oi = oo.getOptimizationInfo();
    const double m[5] = {(double)code, (double)oi.n_iterations, oi.cost_trajectory, oi.cost_time, oi.cost_soft_constraints};
    dump(f, "df4_meta", m, 5);
    dump(f, "df4_times", t2.data(), t2.size());
    dump(f, "df4_coef", c2.data(), c2.size());
  }
  // derivative_to_optimize below 2: the linear optimisation takes it (general-shape kernels, lin_impl.h:61-70 accepts 0 .. N/2-1);
  // the time allocation, built for the node's three choices, refuses it loudly
  {
    PolynomialOptimization<10> lin(dimension);
    if (!lin.setupFromVertices(vertices, times, derivative_order::VELOCITY) || !lin.solveLinear()) return 4;
    Trajectory t1;
    lin.getTrajectory(&t1);
    std::vector<double> c1, tt1;
    t1.pack(&c1, &tt1);
    c1.push_back(lin.computeCost());
    dump(f, "r1_coef_cost", c1.data(), c1.size());
    NonlinearOptimizationParameters prm;
    PolynomialOptimizationNonLinear<10> nl1(dimension, prm);
    const double refused = nl1.setupFromVertices(vertices, times, derivative_order::VELOCITY) ? 0.0 : 1.0;
    dump(f, "r1_refused", &refused, 1);
  }
  // TrajectoryGeneratorBatch over two contexts (two host threads): same results as one context
  {
    std::vector<std::vector<Waypoint>> paths(5);
    for (int p = 0; p < 5; ++p)
      for (int i = 0; i < 6 + p; ++i) paths[p].push_back(Waypoint{1.2 * i, 0.5 * ((i + p) % 3) - 0.4, 5.0 + 0.05 * p, 0.1 * i, false});
    TrajectoryGeneratorBatch one(0), two(std::vector<int>{0, 0});
    std::vector<PathResult> r1, r2;
    if (!one.optimize(paths, std::vector<InitialState>(), &r1) || !two.optimize(paths, std::vector<InitialState>(), &r2)) return 5;
    double same = 1.0;
    for (int p = 0; p < 5; ++p) {
      std::vector<double> ca, ta, cb, tb;
      r1[p].trajectory.pack(&ca, &ta);
      r2[p].trajectory.pack(&cb, &tb);
      if (ca != cb || ta != tb || r1[p].samples_xyzh != r2[p].samples_xyzh || r1[p].info.n_samples != r2[p].info.n_samples) same = 0.0;
    }
    dump(f, "multi_ctx_same", &same, 1);
    std::vector<double> c1, t1;
    r2[4].trajectory.pack(&c1, &t1);
    dump(f, "multi_ctx_times4", t1.data(), t1.size());
  }
  std::fclose(f);
  std::printf("eigen-typed shim test wrote %s (%s; point type: %s)\n", argv[1], tg_version(), TG_TEST_POINT);
  return 0;
}
