// tests/cpp/oracle_set_free.cpp -- TEST INFRASTRUCTURE ONLY: setFreeConstraints + getSegments + computeCost on the oracle's restatement
// (oracle/linear.cpp), for tests/test_free_constraints.py.  Compiled with -DORC_N=N and linked against the oracle library built for
// that N (liboracle.so for N = 10, liboracle_n{6,8,12}.so otherwise), whose LinearSolver it calls: setup (lin_impl.h:61-106), then
// d_p assigned as setFreeConstraints does (lin_impl.h:519-522), segments_from_compact (263-282) and cost (127-141).
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../oracle/oracle.h"

using namespace orc;

// vals [V][N/2][4], dp [4][n_free] (dimension-major), coeffs out [S][4][N]; returns n_free, or -1 when the setup refuses
extern "C" int orc_set_free_constraints(int V, const uint8_t* mask, const double* vals, const double* times, int r, const double* dp,
                                        double* coeffs, double* cost) {
  std::vector<Vertex> vs(V);
  for (int v = 0; v < V; ++v) {
    vs[v].mask = mask[v];
    for (int k = 0; k < kHalf; ++k)
      for (int d = 0; d < kD; ++d) vs[v].val[k][d] = vals[((size_t)v * kHalf + k) * kD + d];
  }
  LinearSolver ls;
  if (!ls.setup(vs, std::vector<double>(times, times + (V - 1)), r)) return -1;
  for (size_t i = 0; i < ls.d_p.size(); ++i) ls.d_p[i] = dp[i];
  ls.segments_from_compact();
  for (int i = 0; i < ls.S; ++i)
    for (int d = 0; d < kD; ++d) std::memcpy(coeffs + ((size_t)i * kD + d) * kN, ls.seg[i].c[d], sizeof(double) * kN);
  *cost = ls.cost();
  return ls.n_free;
}
