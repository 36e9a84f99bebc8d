// tests/cpp/test_shim_dfo_batch.cpp -- PolynomialOptimizationNonLinear<10>::optimizeBatch: five problems with a derivative-free
// method (kSquaredTime, kRichterTimeAndConstraints) in one call equal five separate optimize() calls bit for bit; problems with
// different parameters, or with the Mellinger method, are refused and left untouched.  Dumps flags for
// tests/test_derivative_free_batch.py.
#include <cstdio>
#include <cstring>

#include "../../include/eth_trajectory_generation_b200.hpp"

using namespace eth_trajectory_generation;

static void dump(FILE* f, const char* key, const double* v, size_t n) {
  std::fprintf(f, "%s %zu", key, n);
  for (size_t i = 0; i < n; ++i) std::fprintf(f, " %a", v[i]);
  std::fprintf(f, "\n");
}

typedef PolynomialOptimizationNonLinear<10> Opt;

// problem k: 3 + k waypoints of a zig-zag, ends fixed up to acceleration, a stop at the middle vertex for odd k
static void setup(Opt& o, int k) {
  const int V = 3 + k, r = derivative_order::ACCELERATION;
  Vertex::Vector vertices;
  std::vector<double> times;
  for (int i = 0; i < V; ++i) {
    const Vector w{1.3 * i + 0.1 * k, (i % 2 == 0) ? 0.4 : -0.5, 2.0 + 0.2 * i, 0.1 * i};
    Vertex v(4);
    if (i == 0 || i + 1 == V) v.makeStartOrEnd(w, r);
    else if (k % 2 == 1 && i == V / 2) v.makeStartOrEnd(w, derivative_order::JERK);
    else v.addConstraint(derivative_order::POSITION, w);
    vertices.push_back(v);
    if (i + 1 < V) times.push_back(0.7 + 0.3 * ((i + k) % 3));
  }
  o.setupFromVertices(vertices, times, r);
  o.addMaximumMagnitudeConstraint(0, derivative_order::VELOCITY, 3.0);
  o.addMaximumMagnitudeConstraint(1, derivative_order::ACCELERATION, 0.8);
  o.addMaximumMagnitudeConstraint(2, derivative_order::JERK, 0.5);
  o.addMaximumMagnitudeConstraint(3, derivative_order::VELOCITY, 0.3);
}

static bool same_result(const Opt& a, const Opt& b) {
  Trajectory ta, tb;
  a.getTrajectory(&ta);
  b.getTrajectory(&tb);
  std::vector<double> ca, sa, cb, sb;
  ta.pack(&ca, &sa);
  tb.pack(&cb, &sb);
  const OptimizationInfo ia = a.getOptimizationInfo(), ib = b.getOptimizationInfo();
  return ca == cb && sa == sb && ia.n_iterations == ib.n_iterations && ia.stopping_reason == ib.stopping_reason &&
         ia.cost_trajectory == ib.cost_trajectory && ia.cost_time == ib.cost_time && ia.cost_soft_constraints == ib.cost_soft_constraints;
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  FILE* f = std::fopen(argv[1], "w");
  if (!f) return 2;
  bool all_same = true;
  for (const NonlinearOptimizationParameters::TimeAllocMethod m :
       {NonlinearOptimizationParameters::kSquaredTime, NonlinearOptimizationParameters::kRichterTimeAndConstraints}) {
    NonlinearOptimizationParameters po;
    po.time_alloc_method = m;
    po.max_iterations = 8;
    po.f_rel = 1e-4;
    std::vector<Opt> batch(5, Opt(4, po)), single(5, Opt(4, po));
    std::vector<Opt*> ptrs;
    for (int k = 0; k < 5; ++k) {
      setup(batch[k], k);
      setup(single[k], k);
      ptrs.push_back(&batch[k]);
    }
    std::vector<int> codes;
    if (!Opt::optimizeBatch(ptrs, &codes) || codes.size() != 5) all_same = false;
    for (int k = 0; k < 5 && all_same; ++k) {
      const int code = single[k].optimize();
      all_same = code == codes[k] && code >= 3 && same_result(batch[k], single[k]);
    }
  }
  const double same = all_same ? 1.0 : 0.0;
  dump(f, "batch_equals_single", &same, 1);

  // mixed parameters: refused, nothing touched
  NonlinearOptimizationParameters p0, p1;
  p0.time_alloc_method = p1.time_alloc_method = NonlinearOptimizationParameters::kSquaredTime;
  p1.time_penalty = 400.0;
  Opt a(4, p0), b(4, p1);
  setup(a, 0);
  setup(b, 1);
  std::vector<Opt*> mixed{&a, &b};
  std::vector<int> codes(1, 42);
  const bool mixed_ok = Opt::optimizeBatch(mixed, &codes);
  Trajectory ta;
  a.getTrajectory(&ta);
  const double refused = (!mixed_ok && codes.size() == 1 && codes[0] == 42 && ta.K() == 0 && a.getOptimizationInfo().stopping_reason == -1) ? 1.0 : 0.0;
  dump(f, "mixed_refused", &refused, 1);

  NonlinearOptimizationParameters pm;
  pm.time_alloc_method = NonlinearOptimizationParameters::kMellingerOuterLoop;
  Opt c(4, pm);
  setup(c, 2);
  std::vector<Opt*> mel{&c};
  const double mrefused = Opt::optimizeBatch(mel, nullptr) ? 0.0 : 1.0;
  dump(f, "mellinger_refused", &mrefused, 1);
  std::fclose(f);
  return 0;
}
