// tests/cpp/test_shim_dfo_general.cpp -- optimizeTimeDerivativeFreeBatch and evaluateObjectives on PolynomialOptimization<N> for
// N = 6, 8, 10, 12: four problems per shape and method (kSquaredTime, kRichterTime, kSquaredTimeAndConstraints,
// kRichterTimeAndConstraints) in one call.  Each is checked against the C ABI call on the same inputs, and each object afterwards
// against a separate PolynomialOptimization<N> set up as the reference's poly_opt_ would be (updateSegmentTimes + solveLinear, or +
// setFreeConstraints): coefficients, cost and getFreeConstraints, bit for bit.  Mixed shapes and the Mellinger method are refused.
// Dumps one flag per check for tests/test_derivative_free_general.py; built as it is and against an Eigen.
#include <cstdio>
#include <string>

#include "../../include/eth_trajectory_generation_b200.hpp"

using namespace eth_trajectory_generation;

static FILE* out_file = nullptr;
static void flag(const std::string& key, bool ok) { std::fprintf(out_file, "%s 1 %a\n", key.c_str(), ok ? 1.0 : 0.0); }

// problem k: 3 + k waypoints of a zig-zag, ends fixed up to r, a stop at the middle vertex for odd k (where N/2 > 3)
template <int N>
static bool setup(PolynomialOptimization<N>& o, int k, int dims, int r) {
  const int V = 3 + k;
  Vertex::Vector vertices;
  std::vector<double> times;
  for (int i = 0; i < V; ++i) {
    std::vector<double> w{1.3 * i + 0.1 * k, (i % 2 == 0) ? 0.4 : -0.5, 2.0 + 0.2 * i, 0.1 * i};
    w.resize(dims);
    Vertex v(dims);
    if (i == 0 || i + 1 == V) v.makeStartOrEnd(b200::to_vector(w), r);
    else if (k % 2 == 1 && i == V / 2 && N / 2 > 3) v.makeStartOrEnd(b200::to_vector(w), derivative_order::JERK);
    else v.addConstraint(derivative_order::POSITION, b200::to_vector(w));
    vertices.push_back(v);
    if (i + 1 < V) times.push_back(0.7 + 0.3 * ((i + k) % 3));
  }
  return o.setupFromVertices(vertices, times, r);
}

template <int N>
static std::vector<double> coef_of(const PolynomialOptimization<N>& o) {
  Trajectory t;
  o.getTrajectory(&t);
  std::vector<double> c, s;
  t.pack(&c, &s);
  c.insert(c.end(), s.begin(), s.end());
  return c;
}
static std::vector<double> flat(const std::vector<Vector>& v) {
  std::vector<double> f;
  for (const auto& x : v)
    for (size_t i = 0; i < (size_t)x.size(); ++i) f.push_back(x[i]);
  return f;
}

template <int N>
static void run_shape(int dims) {
  const int r = 1, B = 4;
  const std::string tag = "N" + std::to_string(N) + "_D" + std::to_string(dims);
  const std::vector<MagnitudeConstraint> cons{{0, 1, 3.0}, {1, 2, 0.8}, {2, 3, 0.5}, {3, 1, 0.3}};
  for (const NonlinearOptimizationParameters::TimeAllocMethod m :
       {NonlinearOptimizationParameters::kSquaredTime, NonlinearOptimizationParameters::kRichterTime,
        NonlinearOptimizationParameters::kSquaredTimeAndConstraints, NonlinearOptimizationParameters::kRichterTimeAndConstraints}) {
    const std::string key = tag + "_m" + std::to_string((int)m);
    NonlinearOptimizationParameters po;
    po.time_alloc_method = m;
    po.max_iterations = 10;
    std::vector<PolynomialOptimization<N>> objs(B, PolynomialOptimization<N>(dims));
    std::vector<PolynomialOptimization<N>*> ptrs;
    bool ok = true;
    for (int k = 0; k < B; ++k) {
      ok = ok && setup(objs[k], k, dims, r);
      ptrs.push_back(&objs[k]);
    }
    // the C call on the same inputs
    std::vector<int> vtx_off(1, 0);
    std::vector<uint8_t> mask;
    std::vector<double> vals, times;
    for (const auto& o : objs) {
      std::vector<double> t;
      o.getSegmentTimes(&t);
      mask.insert(mask.end(), o.vertexMasks().begin(), o.vertexMasks().end());
      vals.insert(vals.end(), o.vertexValues().begin(), o.vertexValues().end());
      times.insert(times.end(), t.begin(), t.end());
      vtx_off.push_back((int)mask.size());
    }
    tg_dfo_params P;
    tg_default_dfo_params(&P);
    P.time_alloc_method = (int)m;
    P.derivative_to_optimize = r;
    const int cdim[4] = {0, 1, 2, 3}, cder[4] = {1, 2, 3, 1};
    const double cval[4] = {3.0, 0.8, 0.5, 0.3};
    std::vector<double> coef(times.size() * dims * N), vv(vals.size()), total(B), parts(3 * B);
    std::vector<int> code(B), iters(B);
    b200::Context& c = b200::Context::instance();
    ok = ok && tg_time_alloc_dfo_batch_nd(c.get(), N, dims, B, vtx_off.data(), mask.data(), vals.data(), times.data(), &P, 4, cdim, cder, cval,
                                          coef.data(), vv.data(), code.data(), iters.data(), total.data(), parts.data()) == TG_OK;
    // evaluateObjectives at the initial times (methods 0, 1) equals tg_objective_batch_nd
    if ((int)m < 3) {
      std::vector<double> t0, tot, pa, tot2(1), pa2(3);
      objs[1].getSegmentTimes(&t0);
      ok = ok && evaluateObjectives(objs[1], po, cons, {t0}, &tot, &pa);
      ok = ok && tg_objective_batch_nd(c.get(), N, dims, (int)objs[1].vertexMasks().size(), objs[1].vertexMasks().data(), objs[1].vertexValues().data(),
                                       r, (int)m, 1, t0.data(), (int)t0.size(), 500.0, 1, 100.0, 4, cder, cval, tot2.data(), pa2.data(), nullptr) == TG_OK;
      ok = ok && tot == tot2 && pa == pa2;
    }
    std::vector<int> codes;
    std::vector<OptimizationInfo> infos;
    ok = ok && optimizeTimeDerivativeFreeBatch(ptrs, po, cons, &codes, &infos);
    size_t s0 = 0;
    for (int k = 0; ok && k < B; ++k) {
      const size_t S = objs[k].getNumberSegments();
      std::vector<double> t, want_c(coef.begin() + s0 * dims * N, coef.begin() + (s0 + S) * dims * N);
      objs[k].getSegmentTimes(&t);
      ok = ok && codes[k] == code[k] && infos[k].n_iterations == iters[k] && infos[k].cost_trajectory == parts[3 * k] &&
           infos[k].cost_time == parts[3 * k + 1] && infos[k].cost_soft_constraints == parts[3 * k + 2];
      ok = ok && t == std::vector<double>(times.begin() + s0, times.begin() + s0 + S) && objs[k].computeCost() == parts[3 * k];
      // the reference's state: a fresh object at the final times, solved or set
      PolynomialOptimization<N> ref(dims);
      setup(ref, k, dims, r);
      ref.updateSegmentTimes(t);
      std::vector<Vector> fa, fb;
      if ((int)m >= 3) {
        objs[k].getFreeConstraints(&fa);
        ref.setFreeConstraints(fa);
      } else {
        ref.solveLinear();
        objs[k].getFreeConstraints(&fa);
      }
      ref.getFreeConstraints(&fb);
      std::vector<double> ca = coef_of(objs[k]), cb = coef_of(ref);
      ok = ok && ca == cb && objs[k].computeCost() == ref.computeCost() && flat(fa) == flat(fb);
      // and the C call's coefficients
      ok = ok && std::vector<double>(ca.begin(), ca.begin() + S * dims * N) == want_c;
      s0 += S;
    }
    flag(key, ok);
  }
  // refusals: the Mellinger method, mixed dimensions
  NonlinearOptimizationParameters pm;
  PolynomialOptimization<N> a(dims), b(dims == 1 ? 2 : dims - 1);
  setup(a, 0, dims, r);
  setup(b, 0, dims == 1 ? 2 : dims - 1, r);
  std::vector<double> ta;
  a.getSegmentTimes(&ta);
  std::vector<PolynomialOptimization<N>*> one{&a}, mixed{&a, &b};
  bool refused = !optimizeTimeDerivativeFreeBatch(one, pm, {}, nullptr, nullptr);
  pm.time_alloc_method = NonlinearOptimizationParameters::kSquaredTime;
  refused = refused && !optimizeTimeDerivativeFreeBatch(mixed, pm, {}, nullptr, nullptr);
  std::vector<double> tb;
  a.getSegmentTimes(&tb);
  flag(tag + "_refused", refused && ta == tb);
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  out_file = std::fopen(argv[1], "w");
  if (!out_file) return 2;
  run_shape<6>(3);
  run_shape<8>(1);
  run_shape<10>(4);
  run_shape<12>(2);
  std::fclose(out_file);
  return 0;
}
