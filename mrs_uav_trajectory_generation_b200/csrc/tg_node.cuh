// tg_node.cuh -- the node-side numerics of findTrajectory / optimize(): vertex recipe + heading unwrap,
// initial segment times, time scaling, dt-sampling, spatial validation and midpoint subdivision.
// Reference: src/mrs_trajectory_generation.cpp:923-977, 1401-1455, 729-785, 1533-1554, 1612-1625;
// eth/vertex.cpp:491-565, 301-485; eth/trajectory.cpp:93-151, 598-692; eth/trajectory_sampling.cpp:49-104.
#ifndef TG_NODE_CUH_
#define TG_NODE_CUH_

#include "tg_common.cuh"
#include "tg_poly.cuh"

namespace tg {

// ---- mrs_lib::geometry cyclic helpers (not vendored by the reference; semantics per SURVEY.md 8c(3)) ------
TG_HD double dfmod(double x, double y) {
  // exact IEEE remainder with the sign of x, by long division on the exponent difference (|x/y| small here)
  const double ax = dabs(x), ay = dabs(y);
  if (!(ay > 0.0) || !dfinite(x)) return tgdm::bitsd(0x7ff8000000000000LL);
  if (ax < ay) return x;
  double r = ax;
  // subtract y * 2^k from the top; each subtraction is exact because r and y*2^k share an exponent window
  while (r >= ay) {
    int k = (int)((tgdm::dbits(r) >> 52) & 0x7ff) - (int)((tgdm::dbits(ay) >> 52) & 0x7ff);
    double ys = tgdm::scalb(ay, k);
    if (ys > r) ys = ys * 0.5;
    r = r - ys;
  }
  return (tgdm::dbits(x) < 0) ? -r : r;
}
TG_HD double wrap_range(double val, double minimum, double supremum) {
  const double range = supremum - minimum;
  if (val >= minimum) {
    if (val < supremum) return val;
    if (val < supremum + range) return val - range;
  } else {
    if (val >= minimum - range) return val + range;
  }
  const double rem = dfmod(val - minimum, range);
  return rem + minimum + ((tgdm::dbits(rem) < 0) ? range : 0.0);
}
TG_HD double rad_wrap(double a) { return wrap_range(a, 0.0, 2.0 * TG_PI); }
TG_HD double rad_diff(double a, double b) {
  const double d = a - b;
  if (d < -TG_PI) return d + 2.0 * TG_PI;
  if (d >= TG_PI) return d - 2.0 * TG_PI;
  return d;
}
TG_HD double rad_dist(double a, double b) { return dabs(rad_diff(a, b)); }
TG_HD double rad_interp(double a, double b, double c) { return rad_wrap(a + c * rad_diff(b, a)); }
TG_HD double srad_unwrap(double what, double from) { return from + rad_diff(what, from); }

// ---- vertex recipe (node.cpp:923-977): one thread per problem (the heading unwrap is a serial chain) -------
// wp: [V][4], stop_at: [V] ; init14: {present, heading, vel4, acc4, jerk4} or null
// writes vmask[V], vval[V][5][4], vfree[V+1]; returns np; *hbw_out = half bandwidth of Rpp
TG_HD_NOINLINE int build_vertices(int V, const double* __restrict__ wp, const uint8_t* __restrict__ stop_at, const double* __restrict__ init14, int r,
                         uint8_t* __restrict__ vmask, double* __restrict__ vval, int* __restrict__ vfree, int* hbw_out) {
  const bool have_init = init14 && init14[0] != 0.0;
  double last_heading = have_init ? init14[1] : wp[3];
  int nfree = 0, hbw = 0, prev_cnt = 0;
  for (int i = 0; i < V; ++i) {
    const double heading = srad_unwrap(wp[4 * i + 3], last_heading);
    last_heading = heading;
    double* val = vval + (size_t)i * TG_HALF * TG_D;
    for (int e = 0; e < TG_HALF * TG_D; ++e) val[e] = 0.0;
    val[0] = wp[4 * i + 0];
    val[1] = wp[4 * i + 1];
    val[2] = wp[4 * i + 2];
    val[3] = heading;
    uint32_t m = 1u;
    if (i == 0) {
      m = (1u << (r + 1)) - 1u;  // makeStartOrEnd: derivatives 0..r fixed (1..r to zero)
      if (have_init) {
        m |= 0xEu;  // velocity, acceleration, jerk from the initial state
        for (int d = 0; d < TG_D; ++d) {
          val[1 * TG_D + d] = init14[2 + d];
          val[2 * TG_D + d] = init14[6 + d];
          val[3 * TG_D + d] = init14[10 + d];
        }
      }
    } else if (i == V - 1) {
      m = (1u << (r + 1)) - 1u;
    } else if (stop_at && stop_at[i]) {
      m = 0xFu;  // position + zero velocity, acceleration, jerk
    }
    vmask[i] = (uint8_t)m;
    vfree[i] = nfree;
    const int cnt = TG_HALF - (int)((m & 1u) + ((m >> 1) & 1u) + ((m >> 2) & 1u) + ((m >> 3) & 1u) + ((m >> 4) & 1u));
    // a free slot of vertex i-1 reaches at most the last free slot of vertex i
    if (i > 0 && prev_cnt > 0) hbw = imax(hbw, prev_cnt + cnt - 1);
    if (cnt > 0) hbw = imax(hbw, cnt - 1);
    prev_cnt = cnt;
    nfree += cnt;
  }
  vfree[V] = nfree;
  *hbw_out = hbw;
  return nfree;
}

// Same bookkeeping for caller-supplied masks (the PolynomialOptimization::setupFromVertices path).
TG_HD_NOINLINE int index_vertices(int V, const uint8_t* __restrict__ vmask, int* __restrict__ vfree, int* hbw_out) {
  int nfree = 0, hbw = 0, prev_cnt = 0;
  for (int i = 0; i < V; ++i) {
    const uint32_t m = vmask[i];
    vfree[i] = nfree;
    const int cnt = TG_HALF - (int)((m & 1u) + ((m >> 1) & 1u) + ((m >> 2) & 1u) + ((m >> 3) & 1u) + ((m >> 4) & 1u));
    if (i > 0 && prev_cnt > 0) hbw = imax(hbw, prev_cnt + cnt - 1);
    if (cnt > 0) hbw = imax(hbw, cnt - 1);
    prev_cnt = cnt;
    nfree += cnt;
  }
  vfree[V] = nfree;
  *hbw_out = hbw;
  return nfree;
}

// ---- initial segment times: one thread per segment ---------------------------------------------------
// pos: vertex positions as stored in vval (stride 20 doubles per vertex, first 4 = x y z heading)
TG_HD double vmax_incl(double incl, double lim_v, double lim_h) {
  const double lim = tgdm::datan2(lim_v, lim_h);
  if (incl > lim || incl < -lim) return dabs(lim_v / tgdm::dsin(incl));
  return dabs(lim_h / tgdm::dcos(incl));
}
TG_HD double heading_fix_time(double hs, double he, const double* L, double acc_factor) {
  const double ang = dabs(rad_dist(hs, he));
  double hv = 0.0, ha = 0.0;
  const double w = L[6], al = L[7];
  if (w < TG_FLT_MAX && al < TG_FLT_MAX) {
    if (((ang - (acc_factor * (w * w) / al)) / w) < 0) hv = ang / w;
    else hv = (ang - (acc_factor * (w * w) / al)) / w;
    if (ang > TG_PI / 4) ha = 2 * (w / al);
  }
  return 1.5 * (hv + ha);
}
// eth/vertex.cpp:491-565
TG_HD double segment_time_euclidean(const double* __restrict__ s, const double* __restrict__ e, const double* __restrict__ L) {
  const double dx = e[0] - s[0], dy = e[1] - s[1], dz = e[2] - s[2];
  const double incl = tgdm::datan2(dz, dsqrt(dx * dx + dy * dy));
  const double v_max = vmax_incl(incl, L[1], L[0]);
  const double distance = dsqrt(dx * dx + dy * dy + dz * dz);
  double t = distance / v_max;
  if (t < 0.01) t = 0.01;
  // Euclidean variant uses w^2/alpha (vertex.cpp:543-546): factor 1.  (1 * x is exact.)
  const double fix = heading_fix_time(s[3], e[3], L, 1.0);
  if (fix > t) t = fix;
  return t;
}
TG_HD void normalize3(double* a) {
  const double n = dsqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
  if (n > 0.0) {
    a[0] = a[0] / n;
    a[1] = a[1] / n;
    a[2] = a[2] / n;
  }
}
// eth/vertex.cpp:301-485 ; i = segment index, nv = number of vertices, stride = doubles between vertices
TG_HD_NOINLINE double segment_time_baca(const double* __restrict__ vpos, int stride, int i, int nv, const double* __restrict__ L) {
  const double* s = vpos + (size_t)i * stride;
  const double* e = vpos + (size_t)(i + 1) * stride;
  const double dx = e[0] - s[0], dy = e[1] - s[1], dz = e[2] - s[2];
  double at1 = 0, at2 = 0;
  const double distance = dsqrt(dx * dx + dy * dy + dz * dz);
  const double incl = tgdm::datan2(dz, dsqrt(dx * dx + dy * dy));
  const double v_max = vmax_incl(incl, L[1], L[0]);
  const double a_max = vmax_incl(incl, L[3], L[2]);
  const double j_max = vmax_incl(incl, L[5], L[4]);
  if (i >= 1) {
    const double* p = vpos + (size_t)(i - 1) * stride;
    double v1[3] = {s[0] - p[0], s[1] - p[1], s[2] - p[2]};
    double v2[3] = {dx, dy, dz};
    normalize3(v1);
    normalize3(v2);
    const double dot = v1[0] * v2[0] + v1[1] * v2[1] + v1[2] * v2[2];
    const double scalar = dot < 0 ? 0.0 : dot;
    at1 = (1 - scalar) * ((v_max / a_max) + (a_max / j_max));
  }
  if (i == 0) at1 = (v_max / a_max) + (a_max / j_max);
  if (i == nv - 2) at2 = (v_max / a_max) + (a_max / j_max);
  if (i < nv - 2) {
    const double* q = vpos + (size_t)(i + 2) * stride;
    double v1[3] = {dx, dy, dz};
    double v2[3] = {q[0] - e[0], q[1] - e[1], q[2] - e[2]};
    normalize3(v1);
    normalize3(v2);
    const double dot = v1[0] * v2[0] + v1[1] * v2[1] + v1[2] * v2[2];
    const double scalar = dot < 0 ? 0.0 : dot;
    at2 = (1 - scalar) * ((v_max / a_max) + (a_max / j_max));
  }
  if (at1 > dsqrt(2 * distance / a_max)) at1 = dsqrt(2 * distance / a_max);
  if (at2 > dsqrt(2 * distance / a_max)) at2 = dsqrt(2 * distance / a_max);
  const double max_velocity_time = distance / v_max;  // vertex.cpp:442 overwrites the branch above it
  double t = max_velocity_time + at1 + at2;
  if (t < 0.01) t = 0.01;
  const double fix = heading_fix_time(s[3], e[3], L, 2.0);  // Baca variant: 2 w^2/alpha (vertex.cpp:464-467)
  if (fix > t) t = fix;
  return t;
}

// ---- time scaling of one segment from its nine maxima (eth/trajectory.cpp:625-657) -----------------------------
TG_HD double violation_scaling(const double* __restrict__ m, const double* __restrict__ L) {
  const double vv = dmax(dmax(m[0] / L[0], m[3] / L[1]), m[6] / L[6]);
  const double av = dmax(dmax(m[1] / L[2], m[4] / L[3]), m[7] / L[7]);
  const double jv = dmax(dmax(m[2] / L[4], m[5] / L[5]), m[8] / L[8]);
  return dmax(1.0, dmax(dmax(vv, dsqrt(av)), tgdm::dcbrt(jv)));
}
TG_HD bool violation_within(const double* __restrict__ g, const double* __restrict__ L, double tol = 1e-3) {
  const double vv = dmax(dmax(g[0] / L[0], g[3] / L[1]), g[6] / L[6]);
  const double av = dmax(dmax(g[1] / L[2], g[4] / L[3]), g[7] / L[7]);
  const double jv = dmax(dmax(g[2] / L[4], g[5] / L[5]), g[8] / L[8]);
  return vv <= 1.0 + tol && av <= 1.0 + tol && jv <= 1.0 + tol;  // tol = 1e-3 (eth/trajectory.cpp:604)
}
// scalePolynomialInTime(1/s) on the 4 polynomials of a segment + T *= s (polynomial.cpp:218-224); N coefficients each
template <int N = TG_N>
TG_HD void scale_segment(double* __restrict__ coef, double* __restrict__ T, double scaling) {
  const double inv = 1.0 / scaling;
  for (int d = 0; d < TG_D; ++d) {
    double scale = 1.0;
    for (int n = 0; n < N; ++n) {
      coef[d * N + n] = coef[d * N + n] * scale;
      scale = scale * inv;
    }
  }
  *T = *T * scaling;
}

// ---- dt-sampling (eth/trajectory.cpp:93-151): the serial walk.  One thread per problem. ------------------------
// Writes (segment index, time in segment) per sample when seg_idx != null; returns the sample count.
TG_HD_NOINLINE int sample_walk(int S, const double* __restrict__ T, double dt, int cap, int* __restrict__ seg_idx, double* __restrict__ t_in) {
  double t_end = 0.0;
  for (int i = 0; i < S; ++i) t_end = t_end + T[i];
  const double t_start = 0.0;
  double acc = 0.0;
  int i = 0;
  for (i = 0; i < S; ++i) {
    acc = acc + T[i];
    if (acc > t_start) break;
  }
  if (t_start > acc) return 0;
  if (i >= S) return 0;
  acc = acc - T[i];
  double tin = t_start - acc;
  int m = 0;
  while (acc < t_end) {
    if (tin > T[i]) {
      tin = tin - T[i];
      i++;
      if (i >= S) break;
      continue;
    }
    if (seg_idx && m < cap) {
      seg_idx[m] = i;
      t_in[m] = tin;
    }
    ++m;
    tin = tin + dt;
    acc = acc + dt;
  }
  return m;
}
// upper bound on the sample count, used to size the sample arrays before the walk
TG_HD int sample_cap(int S, const double* __restrict__ T, double dt) {
  double t_end = 0.0;
  for (int i = 0; i < S; ++i) t_end = t_end + T[i];
  const double n = t_end / dt;
  if (!(n < 1.0e9)) return 8;
  return (int)n + 4;
}
// One sample -> the 4 values getTrajectoryReference emits (node.cpp:1578-1602): x, y, z, yawFromQuaternion(...)
// full != null additionally receives p4 v4 a4 j3 s3 (19 doubles = the EigenTrajectoryPoint payload).
TG_HD void sample_eval(const double* __restrict__ coef, double tin, double* __restrict__ xyzh, double* __restrict__ full) {
  const double px = poly_eval(coef + 0 * TG_N, tin, 0), py = poly_eval(coef + 1 * TG_N, tin, 0);
  const double pz = poly_eval(coef + 2 * TG_N, tin, 0), ph = poly_eval(coef + 3 * TG_N, tin, 0);
  const double ha = 0.5 * ph;
  const double qw = tgdm::dcos_k(ha), qz = tgdm::dsin_k(ha);
  const double yaw = tgdm::datan2_k(2.0 * (qw * qz + 0.0 * 0.0), 1.0 - 2.0 * (0.0 * 0.0 + qz * qz));
  xyzh[0] = px;
  xyzh[1] = py;
  xyzh[2] = pz;
  xyzh[3] = yaw;
  if (full) {
    full[0] = px; full[1] = py; full[2] = pz; full[3] = ph;
    for (int d = 0; d < TG_D; ++d) {
      full[4 + d] = poly_eval(coef + d * TG_N, tin, 1);
      full[8 + d] = poly_eval(coef + d * TG_N, tin, 2);
    }
    for (int d = 0; d < 3; ++d) {
      full[12 + d] = poly_eval(coef + d * TG_N, tin, 3);
      full[15 + d] = poly_eval(coef + d * TG_N, tin, 4);
    }
    full[18] = yaw;
  }
}

// ---- spatial validation (node.cpp:1401-1455, 1533-1554) ---------------------------------------------------------
TG_HD double norm3(const double* a) { return dsqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]); }
TG_HD double dist_from_segment(const double* p, const double* s1, const double* s2) {
  const double sv[3] = {s2[0] - s1[0], s2[1] - s1[1], s2[2] - s1[2]};
  const double len = norm3(sv);
  double u[3] = {sv[0], sv[1], sv[2]};
  if (len > 0.0) {
    u[0] = u[0] / len;
    u[1] = u[1] / len;
    u[2] = u[2] / len;
  }
  const double w[3] = {p[0] - s1[0], p[1] - s1[1], p[2] - s1[2]};
  const double coord = u[0] * w[0] + u[1] * w[1] + u[2] * w[2];
  if (coord < 0) return norm3(w);
  if (coord > len) {
    const double q[3] = {p[0] - s2[0], p[1] - s2[1], p[2] - s2[2]};
    return norm3(q);
  }
  double dd[3];
  for (int i = 0; i < 3; ++i) {
    const double m0 = u[i] * u[0], m1 = u[i] * u[1], m2 = u[i] * u[2];
    const double proj = s1[i] + ((m0 * w[0] + m1 * w[1]) + m2 * w[2]);
    dd[i] = p[i] - proj;
  }
  return norm3(dd);
}
// One thread per problem.  samples: [M][4] (x y z heading), wp: [V][4].  seg_ok: [V-1] bytes.
// Returns 1 when safe.
TG_HD_NOINLINE int validate_spatial(int M, const double* __restrict__ samples, int V, const double* __restrict__ wp, double max_deviation,
                           int first_segment_checked, uint8_t* __restrict__ seg_ok, double* max_dev_out) {
  for (int i = 0; i < V - 1; ++i) seg_ok[i] = 1;
  int widx = 0, safe = 1;
  double max_dev = 0.0;
  for (int i = 0; i + 1 < M; ++i) {
    const double* sample = samples + 4 * (size_t)i;
    const double* next = samples + 4 * (size_t)(i + 1);
    const double* s0 = wp + 4 * (size_t)widx;
    const double* s1 = wp + 4 * (size_t)(widx + 1);
    const double dist = dist_from_segment(sample, s0, s1);
    const double end_dist = dist_from_segment(s1, sample, next);
    if (widx > 0 || first_segment_checked || V <= 2) {
      if (dist > max_dev) max_dev = dist;
      if (dist > max_deviation) {
        seg_ok[widx] = 0;
        safe = 0;
      }
    }
    if (end_dist < 0.05 && widx < (V - 2)) widx++;
  }
  *max_dev_out = max_dev;
  return safe;
}
// midpoint insertion (node.cpp:739-753, 1612-1625).  Returns the new vertex count; writes when wp_out != null.
TG_HD_NOINLINE int subdivide(int V, const double* __restrict__ wp, const uint8_t* __restrict__ stop_at, const uint8_t* __restrict__ seg_ok,
                    int first_segment_checked, double* __restrict__ wp_out, uint8_t* __restrict__ stop_out) {
  int n = 0;
  for (int i = 0; i + 1 < V; ++i) {
    if (wp_out) {
      for (int d = 0; d < 4; ++d) wp_out[4 * (size_t)n + d] = wp[4 * (size_t)i + d];
      stop_out[n] = stop_at ? stop_at[i] : 0;
    }
    ++n;
    if (!seg_ok[i] && (i > 0 || first_segment_checked || V <= 2)) {
      if (wp_out) {
        const double* a = wp + 4 * (size_t)i;
        const double* b = wp + 4 * (size_t)(i + 1);
        wp_out[4 * (size_t)n + 0] = a[0] + 0.5 * (b[0] - a[0]);
        wp_out[4 * (size_t)n + 1] = a[1] + 0.5 * (b[1] - a[1]);
        wp_out[4 * (size_t)n + 2] = a[2] + 0.5 * (b[2] - a[2]);
        wp_out[4 * (size_t)n + 3] = rad_interp(a[3], b[3], 0.5);
        stop_out[n] = 0;
      }
      ++n;
    }
  }
  if (wp_out) {
    for (int d = 0; d < 4; ++d) wp_out[4 * (size_t)n + d] = wp[4 * (size_t)(V - 1) + d];
    stop_out[n] = stop_at ? stop_at[V - 1] : 0;
  }
  ++n;
  return n;
}

// ---- the steps either side of the path (SURVEY.md 8f ranks 1-2); one thread per path ----------------------------------
// preprocessPath (node.cpp:431-500): optional straightener, then the min-distance filter.  The reference's expression
// `fabs(radians::diff(a, b) > limit)` (fabs of a bool) is kept as written: it is true iff the SIGNED difference exceeds the limit.
TG_HD_NOINLINE int preprocess_path(int V, const double* __restrict__ wp, const uint8_t* __restrict__ stop, double min_dist, int straighten,
                                   double max_dev, double max_hdg_dev, double* __restrict__ out_wp, uint8_t* __restrict__ out_stop) {
  int n = 0, last_added = 0;
  for (int i = 0; i < V; ++i) {
    if (straighten && V >= 3 && i > 0 && i < V - 1) {
      const double* first = wp + 4 * (size_t)last_added;
      const double* last = wp + 4 * (size_t)(i + 1);
      bool segment_is_ok = true;
      for (int j = last_added + 1; j < i + 1; ++j) {
        const double* mid = wp + 4 * (size_t)j;
        const double d = dist_from_segment(mid, first, last);
        if (d > max_dev || (rad_diff(first[3], mid[3]) > max_hdg_dev) || (rad_diff(last[3], mid[3]) > max_hdg_dev)) {
          segment_is_ok = false;
          break;
        }
      }
      if (segment_is_ok) continue;
    }
    if (i > 0 && i < V - 1) {
      const double* first = wp + 4 * (size_t)last_added;
      const double* last = wp + 4 * (size_t)i;
      const double dx = first[0] - last[0], dy = first[1] - last[1], dz = first[2] - last[2];
      if (dsqrt(dx * dx + dy * dy + dz * dz) < min_dist) continue;
    }
    for (int d = 0; d < 4; ++d) out_wp[4 * (size_t)n + d] = wp[4 * (size_t)i + d];
    out_stop[n] = stop ? stop[i] : 0;
    ++n;
    last_added = i;
  }
  return n;
}

// findTrajectoryFallback (node.cpp:1215-1395): constant-velocity samples along the polyline with Baca segment times.
// vpos: scratch [V][4] for the vertex positions with the heading unwrapped (node.cpp:1236-1248).  out == null: count only.
TG_HD_NOINLINE int fallback_samples(int V, const double* __restrict__ wp, const uint8_t* __restrict__ stop, const double* __restrict__ L, double dt,
                                    double stopping_time, double* __restrict__ vpos, double* __restrict__ out) {
  if (V < 2) return 0;
  double last_heading = wp[3];
  for (int i = 0; i < V; ++i) {
    const double heading = srad_unwrap(wp[4 * (size_t)i + 3], last_heading);
    last_heading = heading;
    vpos[4 * (size_t)i + 0] = wp[4 * (size_t)i + 0];
    vpos[4 * (size_t)i + 1] = wp[4 * (size_t)i + 1];
    vpos[4 * (size_t)i + 2] = wp[4 * (size_t)i + 2];
    vpos[4 * (size_t)i + 3] = heading;
  }
  int n = 0;
  for (int i = 0; i + 1 < V; ++i) {
    const double segment_time = segment_time_baca(vpos, 4, i, V, L);
    int n_samples;
    double interp_step;
    if (segment_time > 1e-1) {
      n_samples = (int)::ceil(segment_time / dt);
      interp_step = (n_samples > 0) ? 1.0 / (double)n_samples : 0.5;
    } else {
      n_samples = 0;
      interp_step = 0;
    }
    if (n_samples > 0 && i == V - 2) n_samples++;
    const double* a = wp + 4 * (size_t)i;
    const double* b = wp + 4 * (size_t)(i + 1);
    for (int j = 0; j < n_samples; ++j) {
      int reps = 1;
      if (j == 0 && i > 0 && stop && stop[i]) reps += (int)::round(stopping_time / dt);
      if (out) {
        const double c = (double)j * interp_step;
        const double x = a[0] + c * (b[0] - a[0]), y = a[1] + c * (b[1] - a[1]), z = a[2] + c * (b[2] - a[2]);
        const double h = rad_interp(a[3], b[3], c);
        const double ha = 0.5 * h;
        const double qw = tgdm::dcos_k(ha), qz = tgdm::dsin_k(ha);
        const double yaw = tgdm::datan2_k(2.0 * (qw * qz + 0.0 * 0.0), 1.0 - 2.0 * (0.0 * 0.0 + qz * qz));
        for (int k = 0; k < reps; ++k) {
          double* o = out + 4 * (size_t)(n + k);
          o[0] = x;
          o[1] = y;
          o[2] = z;
          o[3] = yaw;
        }
      }
      n += reps;
    }
  }
  return n;
}

// getWaypointInTrajectoryIdxs (node.cpp:1461-1499)
TG_HD_NOINLINE int waypoint_idxs(int M, const double* __restrict__ samples, int V, const double* __restrict__ wp, int* __restrict__ idxs) {
  int n = 0, waypoint_idx = 0;
  if (M < 1 || V < 1) return 0;
  for (int i = 0; i + 1 < M; ++i) {
    const double d = dist_from_segment(wp + 4 * (size_t)waypoint_idx, samples + 4 * (size_t)i, samples + 4 * (size_t)(i + 1));
    if (d < 0.1) {
      idxs[n++] = i;
      waypoint_idx++;
    }
    if (waypoint_idx == V) break;
  }
  return n;
}

}  // namespace tg

#endif  // TG_NODE_CUH_
