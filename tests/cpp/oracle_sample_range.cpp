// tests/cpp/oracle_sample_range.cpp -- TEST INFRASTRUCTURE ONLY: the windowed walk of sampleTrajectoryInRange / evaluateRange
// (eth/trajectory_sampling.cpp:49-104, eth/trajectory.cpp:93-151) on the oracle's restatement, for tests/test_sample_range.py.
// Compiled with -DORC_N=N and linked against the oracle library built for that N (liboracle.so for N = 10, liboracle_n{6,8,12}.so
// otherwise), whose poly_eval and yaw functions it calls.  This is oracle/trajectory.cpp's sample_whole with the window as
// arguments; tests/test_sample_range.py checks that [0, end] gives orc_sample's rows bit for bit.
#include <cstdint>
#include <vector>

#include "../../oracle/oracle.h"

using namespace orc;

namespace {
struct WalkPoint {
  int seg;
  double tin, acc;  // time in segment, accumulated time (evaluateRange's sampling_times)
};
std::vector<Segment> make_segments(int S, const double* coeffs, const double* times) {
  std::vector<Segment> seg(S);
  for (int i = 0; i < S; ++i) {
    seg[i].T = times[i];
    for (int d = 0; d < kD; ++d)
      for (int n = 0; n < kN; ++n) seg[i].c[d][n] = coeffs[((size_t)i * kD + d) * kN + n];
  }
  return seg;
}
// accumulated_time starts at the start of the segment holding t_start; no such segment (t_start at or past the end, a NaN t_start):
// nothing, as evaluateRange logs and returns
std::vector<WalkPoint> range_walk(const std::vector<Segment>& seg, double t_start, double t_end, double dt) {
  std::vector<WalkPoint> out;
  double acc = 0.0;
  size_t i = 0;
  for (i = 0; i < seg.size(); ++i) {
    acc += seg[i].T;
    if (acc > t_start) break;
  }
  if (t_start > acc) return out;
  if (i >= seg.size()) return out;
  acc -= seg[i].T;
  double tin = t_start - acc;
  while (acc < t_end) {
    if (tin > seg[i].T) {
      tin = tin - seg[i].T;
      i++;
      if (i >= seg.size()) break;
      continue;
    }
    out.push_back(WalkPoint{(int)i, tin, acc});
    tin += dt;
    acc += dt;
  }
  return out;
}
}  // namespace

// rows of 19 doubles [p4 v4 a4 j3 s3 yaw_out] as orc_sample, t_ns = int64((t_start + dt k) 1e9); returns the count, -count if cap is small
extern "C" int orc_sample_range(int S, const double* coeffs, const double* times, double t_start, double t_end, double dt, int cap, double* out19,
                                int64_t* t_ns) {
  const std::vector<Segment> seg = make_segments(S, coeffs, times);
  const std::vector<WalkPoint> w = range_walk(seg, t_start, t_end, dt);
  if ((int)w.size() > cap) return -(int)w.size();
  for (size_t k = 0; k < w.size(); ++k) {
    const Segment& g = seg[w[k].seg];
    const double tin = w[k].tin;
    double* o = out19 + 19 * k;
    for (int d = 0; d < kD; ++d) {
      o[d] = poly_eval(g.c[d], tin, 0);
      o[4 + d] = poly_eval(g.c[d], tin, 1);
      o[8 + d] = poly_eval(g.c[d], tin, 2);
    }
    for (int d = 0; d < 3; ++d) {
      o[12 + d] = poly_eval(g.c[d], tin, 3);
      o[15 + d] = poly_eval(g.c[d], tin, 4);
    }
    // yawFromQuaternion(quaternionFromYaw(p[3])) (eth_mav_msgs/common.h:130-140)
    const double ha = 0.5 * o[3];
    const double qw = m_cos_k(ha), qz = m_sin_k(ha);
    o[18] = m_atan2_k(2.0 * (qw * qz + 0.0 * 0.0), 1.0 - 2.0 * (0.0 * 0.0 + qz * qz));
    if (t_ns) t_ns[k] = (int64_t)((t_start + dt * (double)k) * 1.e9);  // trajectory_sampling.cpp:98
  }
  return (int)w.size();
}

// Trajectory::evaluateRange: out4 [count][4] = derivative `deriv` of the four dimensions, sampling_times [count]; returns the count,
// -count if cap is small
extern "C" int orc_evaluate_range(int S, const double* coeffs, const double* times, double t_start, double t_end, double dt, int deriv, int cap,
                                  double* out4, double* sampling_times) {
  const std::vector<Segment> seg = make_segments(S, coeffs, times);
  const std::vector<WalkPoint> w = range_walk(seg, t_start, t_end, dt);
  if ((int)w.size() > cap) return -(int)w.size();
  for (size_t k = 0; k < w.size(); ++k) {
    for (int d = 0; d < kD; ++d) out4[4 * k + d] = poly_eval(seg[w[k].seg].c[d], w[k].tin, deriv);
    if (sampling_times) sampling_times[k] = w[k].acc;
  }
  return (int)w.size();
}
