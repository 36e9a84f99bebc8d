// tests/cpp/test_shim_nonlinear_general.cpp -- the drop-in header's nonlinear half on the other shapes the reference's templates
// allow: PolynomialOptimizationNonLinear<8>(3), <12>(4) and <6>(2) with the Mellinger outer loop (setupFromVertices /
// addMaximumMagnitudeConstraint / optimize / getTrajectory), and PolynomialOptimization<12>(4)::computeMaximumOfMagnitude.  Dumps hex
// floats for tests/test_general_shape_nonlinear.py, which compares them bit for bit with the oracle compiled for that N.
#include <cstdio>
#include <cstdlib>

#include "../../include/eth_trajectory_generation_b200.hpp"

using namespace eth_trajectory_generation;

static void dump(FILE* f, const std::string& key, const double* v, size_t n) {
  std::fprintf(f, "%s %zu", key.c_str(), n);
  for (size_t i = 0; i < n; ++i) std::fprintf(f, " %a", v[i]);
  std::fprintf(f, "\n");
}

// waypoint i of the test path in `dims` dimensions
static Vector waypoint(int i, int dims) {
  const double full[4] = {1.9 * i, (i % 2 == 0) ? 0.8 : -0.5, 2.0 + 0.4 * i, 0.2 * i};
  Vector v = b200::make_vector((size_t)dims, 0.0);
  for (int d = 0; d < dims; ++d) v[d] = full[d];
  return v;
}

static Vertex::Vector path(int dims, int derivative_to_optimize) {
  Vertex::Vector vertices;
  for (int i = 0; i < 7; ++i) {
    Vertex v(dims);
    if (i == 0 || i == 6) v.makeStartOrEnd(waypoint(i, dims), derivative_to_optimize);
    else v.addConstraint(derivative_order::POSITION, waypoint(i, dims));
    vertices.push_back(v);
  }
  return vertices;
}

static std::vector<double> initial_times() {
  std::vector<double> t;
  for (int i = 0; i < 6; ++i) t.push_back(0.9 + 0.2 * (double)(i % 3));
  return t;
}

template <int N>
static int run(FILE* f, const std::string& key, int dims, int derivative_to_optimize) {
  NonlinearOptimizationParameters prm;
  prm.time_alloc_method = NonlinearOptimizationParameters::kMellingerOuterLoop;
  PolynomialOptimizationNonLinear<N> nl(dims, prm);
  if (!nl.setupFromVertices(path(dims, derivative_to_optimize), initial_times(), derivative_to_optimize)) return 1;
  nl.addMaximumMagnitudeConstraint(0, derivative_order::VELOCITY, 2.5);
  nl.addMaximumMagnitudeConstraint(0, derivative_order::ACCELERATION, 1.5);
  if (dims >= 3) nl.addMaximumMagnitudeConstraint(2, derivative_order::VELOCITY, 1.0);
  const int code = nl.optimize();
  Trajectory t;
  nl.getTrajectory(&t);
  if (t.N() != N || t.D() != dims || t.K() != 6) return 2;
  std::vector<double> coef, times;
  t.pack(&coef, &times);
  times.push_back((double)code);
  dump(f, key + "_times_code", times.data(), times.size());
  dump(f, key + "_coef", coef.data(), coef.size());
  // the derivative-free methods stay on N = 10, 4 dimensions
  prm.time_alloc_method = NonlinearOptimizationParameters::kSquaredTime;
  PolynomialOptimizationNonLinear<N> dfo(dims, prm);
  const double refused = dfo.setupFromVertices(path(dims, derivative_to_optimize), initial_times(), derivative_to_optimize) ? 0.0 : 1.0;
  dump(f, key + "_dfo_refused", &refused, 1);
  return 0;
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  FILE* f = std::fopen(argv[1], "w");
  if (!f) return 2;
  int rc = 0;
  if ((rc = run<8>(f, "n8d3", 3, derivative_order::JERK))) return 10 + rc;
  if ((rc = run<12>(f, "n12d4", 4, derivative_order::SNAP))) return 20 + rc;
  if ((rc = run<6>(f, "n6d2", 2, derivative_order::ACCELERATION))) return 30 + rc;
  {
    PolynomialOptimization<12> opt(4);
    if (!opt.setupFromVertices(path(4, derivative_order::JERK), initial_times(), derivative_order::JERK) || !opt.solveLinear()) return 40;
    for (int k = 1; k <= 4; ++k) {
      const Extremum e = opt.computeMaximumOfMagnitude(k);
      const double ev[3] = {e.time, e.value, (double)e.segment_idx};
      dump(f, "n12d4_maxmag", ev, 3);
    }
  }
  std::fclose(f);
  return 0;
}
