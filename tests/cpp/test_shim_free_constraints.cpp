// tests/cpp/test_shim_free_constraints.cpp -- the free and fixed constraints of PolynomialOptimization<N> through the drop-in header
// (lin_impl.h:513-522): for N = 6, 8, 10, 12 on 3 and 4 dimensions, getFreeConstraints after solveLinear, one slot changed,
// setFreeConstraints, then getSegments / computeCost / computeMaximumOfMagnitude, the counts and getFixedConstraints.  Dumps hex
// floats for tests/test_free_constraints.py, which compares them bit for bit with the C ABI and the oracle.  Built once as it is and
// once against an Eigen (the stand-in of the tests), where the arguments are std::vector<Eigen::VectorXd> as in the reference.
#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../include/eth_trajectory_generation_b200.hpp"

using namespace eth_trajectory_generation;

#if defined(TG_B200_HAVE_EIGEN)
typedef std::vector<Eigen::VectorXd> Constraints;
static_assert(std::is_same<Vector, Eigen::VectorXd>::value, "with Eigen on the include path the header's Vector is Eigen::VectorXd");
#else
typedef std::vector<Vector> Constraints;
#endif

static void dump(FILE* f, const std::string& key, const double* v, size_t n) {
  std::fprintf(f, "%s %zu", key.c_str(), n);
  for (size_t i = 0; i < n; ++i) std::fprintf(f, " %a", v[i]);
  std::fprintf(f, "\n");
}
static void dump_constraints(FILE* f, const std::string& key, const Constraints& c) {
  std::vector<double> flat;
  for (const auto& v : c)
    for (size_t i = 0; i < (size_t)v.size(); ++i) flat.push_back(v[i]);
  dump(f, key, flat.data(), flat.size());
}
static Vector waypoint(int i, int dims) {
  const double full[4] = {1.1 * i, (i % 2 == 0) ? 0.7 : -0.5, 2.0 + 0.3 * i, 0.2 * i};
  Vector v = b200::make_vector((size_t)dims, 0.0);
  for (int d = 0; d < dims; ++d) v[d] = full[d];
  return v;
}

template <int N>
static int run(FILE* f, int dims) {
  const std::string key = "n" + std::to_string(N) + "d" + std::to_string(dims);
  const int n_wp = 6, r = N / 2 - 1 < 2 ? N / 2 - 1 : 2;
  Vertex::Vector vertices;
  for (int i = 0; i < n_wp; ++i) {
    Vertex v(dims);
    if (i == 0 || i == n_wp - 1) v.makeStartOrEnd(waypoint(i, dims), r);
    else v.addConstraint(derivative_order::POSITION, waypoint(i, dims));
    if (i == 2) v.addConstraint(derivative_order::VELOCITY, b200::make_vector((size_t)dims, 0.4));
    vertices.push_back(v);
  }
  std::vector<double> times;
  for (int i = 0; i + 1 < n_wp; ++i) times.push_back(0.9 + 0.25 * (double)(i % 3));
  PolynomialOptimization<N> opt(dims);
  if (!opt.setupFromVertices(vertices, times, r)) return 3;
  const double counts[3] = {(double)opt.getNumberFreeConstraints(), (double)opt.getNumberFixedConstraints(), (double)opt.getNumberAllConstraints()};
  dump(f, key + "_counts", counts, 3);
  Constraints c;
  opt.getFreeConstraints(&c);  // no solution yet: zeros
  if ((int)c.size() != dims) return 4;
  dump_constraints(f, key + "_free_before", c);
  opt.getFixedConstraints(&c);
  dump_constraints(f, key + "_fixed", c);
  if (!opt.solveLinear()) return 5;
  Constraints free;
  opt.getFreeConstraints(&free);
  if ((int)free.size() != dims || (size_t)free[0].size() != opt.getNumberFreeConstraints()) return 6;
  dump_constraints(f, key + "_free", free);
  Constraints again;
  opt.getFreeConstraints(&again);  // the cached copy
  dump_constraints(f, key + "_free_again", again);
  // a wrong size is refused and changes nothing
  const double cost0 = opt.computeCost();
  Constraints bad(free.begin(), free.end() - 1);
  opt.setFreeConstraints(bad);
  const double cost_bad = opt.computeCost();
  dump(f, key + "_cost_solve", &cost0, 1);
  dump(f, key + "_cost_after_bad", &cost_bad, 1);
  // one slot changed
  free[dims - 1][0] = free[dims - 1][0] + 0.75;
  opt.setFreeConstraints(free);
  Constraints got;
  opt.getFreeConstraints(&got);
  dump_constraints(f, key + "_free_set", got);
  Segment::Vector segs;
  opt.getSegments(&segs);
  Trajectory t;
  opt.getTrajectory(&t);
  std::vector<double> coef, tt;
  t.pack(&coef, &tt);
  if ((int)segs.size() != n_wp - 1) return 7;
  dump(f, key + "_coef", coef.data(), coef.size());
  const double cost = opt.computeCost();
  dump(f, key + "_cost", &cost, 1);
  const Extremum e = opt.computeMaximumOfMagnitude(derivative_order::ACCELERATION);
  const double m[3] = {e.time, e.value, (double)e.segment_idx};
  dump(f, key + "_maxacc", m, 3);
  // updateSegmentTimes leaves no linear solution to read: zeros again
  opt.updateSegmentTimes(times);
  opt.getFreeConstraints(&got);
  dump_constraints(f, key + "_free_after_times", got);
  return 0;
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  FILE* f = std::fopen(argv[1], "w");
  if (!f) return 2;
  int rc = 0;
  for (int dims = 3; dims <= 4 && rc == 0; ++dims) {
    if (rc == 0) rc = run<6>(f, dims);
    if (rc == 0) rc = run<8>(f, dims);
    if (rc == 0) rc = run<10>(f, dims);
    if (rc == 0) rc = run<12>(f, dims);
  }
  std::fclose(f);
  return rc;
}
