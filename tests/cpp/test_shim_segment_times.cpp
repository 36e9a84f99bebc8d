// tests/cpp/test_shim_segment_times.cpp -- the initial segment times of the drop-in header written as findTrajectory writes them
// (src/mrs_trajectory_generation.cpp:923-1083): the vertex recipe with the heading unwrapped from the previous vertex, estimateSegmentTimes
// and estimateSegmentTimesBaca with the reference's argument list, the Baca sum of the length check, then setupFromVertices + optimize().
// Also estimateSegmentTimesEuclidean, estimateSegmentTimesBatch and the refusals.  Built against the Eigen stand-in of oracle/ref_shim by
// tests/test_segment_times.py, which compares the hex dump bit for bit with the oracle.
#include <Eigen/Core>
#include <cstdio>
#include <vector>

#include "../../include/eth_trajectory_generation_b200.hpp"

using namespace eth_trajectory_generation;

static void dump(FILE* f, const char* key, const double* v, size_t n) {
  std::fprintf(f, "%s %zu", key, n);
  for (size_t i = 0; i < n; ++i) std::fprintf(f, " %a", v[i]);
  std::fprintf(f, "\n");
}
static void dump(FILE* f, const char* key, const std::vector<double>& v) { dump(f, key, v.data(), v.size()); }

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  FILE* f = std::fopen(argv[1], "w");
  if (!f) return 2;
  // a path whose headings cross +-pi, so that the unwrapped headings of the vertices leave [-pi, pi)
  const double wp[7][4] = {{0.0, 0.0, 3.0, 3.0},  {2.0, 0.5, 4.0, -3.0}, {4.0, -0.5, 5.0, 2.9}, {4.0, -0.5, 7.5, -3.1},
                           {6.0, 0.5, 5.0, 0.5},  {8.0, -0.5, 5.0, 3.1},  {10.0, 0.5, 5.0, -2.0}};
  const int n_wp = 7;
  const int derivative_to_optimize = derivative_order::ACCELERATION;
  const double max_vel_horizontal = 4.0, max_vel_vertical = 2.0, max_acc_horizontal = 2.0, max_acc_vertical = 1.0, max_jerk_horizontal = 20.0,
               max_jerk_vertical = 20.0, max_heading_rate = 1.0, max_heading_acc = 2.0, max_heading_jerk = 10.0;

  // node.cpp:923-977 without an initial state: the heading of each vertex unwrapped from the one before
  Vertex::Vector vertices;
  double last_heading = wp[0][3];
  for (int i = 0; i < n_wp; ++i) {
    double d = wp[i][3] - last_heading;  // radians::diff
    if (d < -M_PI) d += 2.0 * M_PI;
    else if (d >= M_PI) d -= 2.0 * M_PI;
    const double heading = last_heading + d;
    last_heading = heading;
    Vertex vertex(4);
    const Eigen::Vector4d p(wp[i][0], wp[i][1], wp[i][2], heading);
    if (i == 0 || i == n_wp - 1) vertex.makeStartOrEnd(p, derivative_to_optimize);
    else vertex.addConstraint(derivative_order::POSITION, p);
    vertices.push_back(vertex);
  }

  // node.cpp:1045-1056
  std::vector<double> segment_times, segment_times_baca;
  segment_times = estimateSegmentTimes(vertices, max_vel_horizontal, max_vel_vertical, max_acc_horizontal, max_acc_vertical, max_jerk_horizontal,
                                       max_jerk_vertical, max_heading_rate, max_heading_acc);
  segment_times_baca = estimateSegmentTimesBaca(vertices, max_vel_horizontal, max_vel_vertical, max_acc_horizontal, max_acc_vertical,
                                                max_jerk_horizontal, max_jerk_vertical, max_heading_rate, max_heading_acc);
  double initial_cutoff_time = 0;
  for (size_t i = 0; i < segment_times_baca.size(); i++) initial_cutoff_time += segment_times_baca[i];
  dump(f, "times", segment_times);
  dump(f, "baca", segment_times_baca);
  dump(f, "baca_sum", &initial_cutoff_time, 1);

  // node.cpp:1063-1083
  NonlinearOptimizationParameters parameters;
  parameters.f_rel = 0.05;
  parameters.x_rel = 0.1;
  parameters.max_iterations = 10;
  parameters.time_alloc_method = NonlinearOptimizationParameters::kMellingerOuterLoop;
  PolynomialOptimizationNonLinear<10> opt(4, parameters);
  opt.setupFromVertices(vertices, segment_times, derivative_to_optimize);
  opt.addMaximumMagnitudeConstraint(0, derivative_order::VELOCITY, max_vel_horizontal);
  opt.addMaximumMagnitudeConstraint(0, derivative_order::ACCELERATION, max_acc_horizontal);
  opt.addMaximumMagnitudeConstraint(0, derivative_order::JERK, max_jerk_horizontal);
  opt.addMaximumMagnitudeConstraint(1, derivative_order::VELOCITY, max_vel_horizontal);
  opt.addMaximumMagnitudeConstraint(1, derivative_order::ACCELERATION, max_acc_horizontal);
  opt.addMaximumMagnitudeConstraint(1, derivative_order::JERK, max_jerk_horizontal);
  opt.addMaximumMagnitudeConstraint(2, derivative_order::VELOCITY, max_vel_vertical);
  opt.addMaximumMagnitudeConstraint(2, derivative_order::ACCELERATION, max_acc_vertical);
  opt.addMaximumMagnitudeConstraint(2, derivative_order::JERK, max_jerk_vertical);
  opt.addMaximumMagnitudeConstraint(3, derivative_order::VELOCITY, max_heading_rate);
  opt.addMaximumMagnitudeConstraint(3, derivative_order::ACCELERATION, max_heading_acc);
  opt.addMaximumMagnitudeConstraint(3, derivative_order::JERK, max_heading_jerk);
  const int code = opt.optimize();
  const double meta[2] = {(double)code, (double)opt.getOptimizationInfo().n_iterations};
  dump(f, "nl_meta", meta, 2);
  Trajectory trajectory;
  opt.getTrajectory(&trajectory);
  std::vector<double> coef, times;
  trajectory.pack(&coef, &times);
  dump(f, "nl_times", times);
  dump(f, "nl_coef", coef);

  // the other names, and one call for several lists: the path, a list of one vertex, the first two vertices
  dump(f, "euclidean", estimateSegmentTimesEuclidean(vertices, max_vel_horizontal, max_vel_vertical, max_acc_horizontal, max_acc_vertical,
                                                      max_jerk_horizontal, max_jerk_vertical, max_heading_rate, max_heading_acc));
  const std::vector<Vertex::Vector> lists = {vertices, Vertex::Vector(vertices.begin(), vertices.begin() + 1),
                                             Vertex::Vector(vertices.begin(), vertices.begin() + 2)};
  std::vector<std::vector<double>> e, b, b_only;
  const bool ok = estimateSegmentTimesBatch(lists, max_vel_horizontal, max_vel_vertical, max_acc_horizontal, max_acc_vertical, max_jerk_horizontal,
                                            max_jerk_vertical, max_heading_rate, max_heading_acc, &e, &b);
  const bool ok_b = estimateSegmentTimesBatch(lists, max_vel_horizontal, max_vel_vertical, max_acc_horizontal, max_acc_vertical, max_jerk_horizontal,
                                              max_jerk_vertical, max_heading_rate, max_heading_acc, nullptr, &b_only);
  const double oks[2] = {ok ? 1.0 : 0.0, ok_b ? 1.0 : 0.0};
  dump(f, "batch_ok", oks, 2);
  for (size_t i = 0; i < e.size(); ++i) {
    dump(f, "batch_e", e[i]);
    dump(f, "batch_b", b[i]);
    dump(f, "batch_b_only", b_only[i]);
  }

  // refusals: a 3-dimensional list, a vertex without a POSITION constraint, an empty list (print, return empty / false, fill nothing)
  Vertex::Vector three;
  for (int i = 0; i < 3; ++i) {
    Vertex v(3);
    v.addConstraint(derivative_order::POSITION, Eigen::Vector3d(1.0 * i, 0.0, 5.0));
    three.push_back(v);
  }
  Vertex::Vector no_position = vertices;
  no_position[3].removeConstraint(derivative_order::POSITION);
  no_position[3].addConstraint(derivative_order::VELOCITY, Eigen::Vector4d(0.1, 0.0, 0.0, 0.0));
  std::vector<std::vector<double>> untouched(1, std::vector<double>(1, -7.25));
  const bool batch_refused = !estimateSegmentTimesBatch({vertices, no_position}, max_vel_horizontal, max_vel_vertical, max_acc_horizontal,
                                                        max_acc_vertical, max_jerk_horizontal, max_jerk_vertical, max_heading_rate, max_heading_acc,
                                                        &untouched, nullptr) &&
                             untouched.size() == 1 && untouched[0].size() == 1 && untouched[0][0] == -7.25;
  const double refused[5] = {
      estimateSegmentTimes(three, 4, 2, 2, 1, 20, 20, 1, 2).empty() ? 1.0 : 0.0,
      estimateSegmentTimesBaca(no_position, 4, 2, 2, 1, 20, 20, 1, 2).empty() ? 1.0 : 0.0,
      estimateSegmentTimes(Vertex::Vector(), 4, 2, 2, 1, 20, 20, 1, 2).empty() ? 1.0 : 0.0,
      batch_refused ? 1.0 : 0.0,
      estimateSegmentTimesBatch(lists, 4, 2, 2, 1, 20, 20, 1, 2, nullptr, nullptr) ? 0.0 : 1.0,
  };
  dump(f, "refused", refused, 5);
  std::fclose(f);
  return 0;
}
