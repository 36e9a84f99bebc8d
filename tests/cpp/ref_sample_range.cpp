// tests/cpp/ref_sample_range.cpp -- TEST INFRASTRUCTURE ONLY: the REFERENCE's own sampleTrajectoryInRange and Trajectory::evaluateRange
// (eth/trajectory_sampling.cpp:49-104, eth/trajectory.cpp:93-151) for tests/test_sample_range.py, built only where a checkout of the
// reference is present: compiled against its headers and the stand-ins of oracle/ref_shim/, linked against oracle/_ref/libref_eth.so
// (the reference's library, N = 10).  Marshals plain arrays only; the signatures mirror tests/cpp/oracle_sample_range.cpp.
#include <cstdint>
#include <vector>

#include <eth_trajectory_generation/trajectory.h>
#include <eth_trajectory_generation/trajectory_sampling.h>

namespace etg = eth_trajectory_generation;
static const int kN = 10, kD = 4;

static etg::Segment::Vector make_segments(int S, const double* coeffs, const double* times) {
  etg::Segment::Vector segs;
  for (int i = 0; i < S; ++i) {
    etg::Segment s(kN, kD);
    s.setTime(times[i]);
    for (int d = 0; d < kD; ++d) {
      Eigen::VectorXd c(kN);
      for (int k = 0; k < kN; ++k) c[k] = coeffs[((size_t)i * kD + d) * kN + k];
      s[d] = etg::Polynomial(kN, c);
    }
    segs.push_back(s);
  }
  return segs;
}

// sampleTrajectoryInRange(trajectory, t_start, t_end, dt, &states): *ok = what it returns; rows of 19 doubles as orc_sample_range, the
// 4th components of p from evaluateRange over the same window, the heading rate / acceleration and yaw as the node reads them back
extern "C" int ref_sample_range(int S, const double* coeffs, const double* times, double t_start, double t_end, double dt, int cap, double* out19,
                                int64_t* t_ns, int* ok) {
  etg::Trajectory traj;
  traj.setSegments(make_segments(S, coeffs, times));
  eth_mav_msgs::EigenTrajectoryPoint::Vector states;
  *ok = etg::sampleTrajectoryInRange(traj, t_start, t_end, dt, &states) ? 1 : 0;
  if (!*ok) return 0;
  if ((int)states.size() > cap) return -(int)states.size();
  std::vector<Eigen::VectorXd> p;
  traj.evaluateRange(t_start, t_end, dt, etg::derivative_order::POSITION, &p);
  for (size_t i = 0; i < states.size(); ++i) {
    const eth_mav_msgs::EigenTrajectoryPoint& s = states[i];
    double* o = out19 + 19 * i;
    for (int k = 0; k < 19; ++k) o[k] = 0.0;
    for (int d = 0; d < 3; ++d) {
      o[d] = s.position_W[d];
      o[4 + d] = s.velocity_W[d];
      o[8 + d] = s.acceleration_W[d];
      o[12 + d] = s.jerk_W[d];
      o[15 + d] = s.snap_W[d];
    }
    o[3] = p[i][3];
    o[7] = s.getYawRate();
    o[11] = s.getYawAcc();
    o[18] = s.getYaw();
    if (t_ns) t_ns[i] = s.time_from_start_ns;
  }
  return (int)states.size();
}

// Trajectory::evaluateRange(t_start, t_end, dt, deriv, &result, &sampling_times): out4 [count][4], sampling_times [count]
extern "C" int ref_evaluate_range(int S, const double* coeffs, const double* times, double t_start, double t_end, double dt, int deriv, int cap,
                                  double* out4, double* sampling_times) {
  etg::Trajectory traj;
  traj.setSegments(make_segments(S, coeffs, times));
  std::vector<Eigen::VectorXd> v;
  std::vector<double> st;
  traj.evaluateRange(t_start, t_end, dt, deriv, &v, &st);
  if ((int)v.size() > cap) return -(int)v.size();
  for (size_t k = 0; k < v.size(); ++k) {
    for (int d = 0; d < kD; ++d) out4[4 * k + d] = v[k][d];
    sampling_times[k] = st[k];
  }
  return (int)v.size();
}
