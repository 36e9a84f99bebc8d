// tg_generic.cuh -- the linear optimisation, evaluation and sampling for ANY even number of coefficients N <= 12.
//
// The reference's classes are templates over N ("_N = Number of coefficients", lin.h:46-55; Polynomial::kMaxN = 12,
// eth/polynomial.h:45-48) and take the dimension D at run time; its node instantiates N = 10, D = 4 only (node.cpp:902, 1063),
// and that shape is what the tuned kernels of tg_segment / tg_solve* / tg_kernels are built for (register-resident 10x10
// products, 4x4 vertex blocks).  This file is the general-shape path behind tg_solve_linear_batch_nd / tg_evaluate_batch_nd /
// tg_sample_batch_nd: the same algorithm with N a template parameter, written for correctness at any shape rather than for
// the last percent of one shape:
//   record_head<N>   one thread per segment            A (eth/polynomial.h:208-226), A^-1 by the Schur form (lin_impl.h:147-177),
//                                                      Q (lin_impl.h:605-618)  -> dense N x N each
//   record_hrow<N>   one thread per (segment, row a)   row a of H = (A^-T Q) A^-1 (lin_impl.h:320)
//   solve_warp<N>    one warp per problem              reduced banded system, LU without pivoting, coefficients, cost
//                                                      (lin_impl.h:310-373, 263-282, 127-141) -- the phases of tg_solve.cuh
//   SolveFreeFn<N>                                     solve_warp<N> that also writes the free derivatives d_p (getFreeConstraints)
//   SetFreeFn<N>, SetFreeCostFn                        setFreeConstraints: coefficients and cost from given d_p, one thread per
//                                                      (segment, dimension), with solve_warp's coef_from_endpoints / cost_partial
//   poly_eval_n<N>, sample_eval_n<N>                   Trajectory::evaluate / sampleWholeTrajectory (eth/trajectory.cpp:55-151,
//                                                      eth/trajectory_sampling.cpp:49-124)
//   RangeWalkFn, EvaluateRangeFn<N>                    sampleTrajectoryInRange / evaluateRange over a window per trajectory
//   ExtremaFn<N, Q>, MaxMagnitudeSegFn<N, K>           per-segment maxima (tg_poly.cuh over N), one thread per segment
//   ScaleFn<N>                                         scaleSegmentTimesToMeetConstraints' stretch (eth/trajectory.cpp:610-658)
//   MellingerHeadFn / HrowFn / SolveFn<N>              one Mellinger evaluation: S+1 solves per running problem (nl_impl.h:282-323);
//                                                      the optimiser state machine (tg_plis.cuh) does not depend on N
//   candidate_rec<N>                                   the record rule of a derivative-free candidate's solve (tg_dfo_generic.cuh)
// Every sum is the DENSE sum over ascending index, exactly as the reference-order restatement writes it (the tuned path skips structural
// zeros, which is the same IEEE result); for N = 10 this path and the tuned one are compared bit for bit in the tests.
// D: the device works on 4 right-hand sides; tg_*_nd pad D < 4 with zero dimensions (a zero dimension adds exact zeros to the
// cost and nothing to the other dimensions) and strip them from the outputs.
#ifndef TG_GENERIC_CUH_
#define TG_GENERIC_CUH_

#include "tg_common.cuh"
#include "tg_kernels.cuh"  // BatchPtrs, the PLIS and scaling functors that do not depend on N
#include "tg_node.cuh"     // sample_cap, sample_walk
#include "tg_poly.cuh"     // segment maxima and Jenkins-Traub over N coefficients
#include "tg_solve.cuh"    // TG_PHASE

namespace tg {
namespace gen {

template <int N>
struct Rec {
  static constexpr int kAinv = 0;        // N x N, row major
  static constexpr int kQ = N * N;       // N x N
  static constexpr int kH = 2 * N * N;   // N x N
  static constexpr int kSize = 3 * N * N;
};

// n x n inverse, n = N/2: LU with first-maximum row pivoting, multipliers by division, identity columns by forward and back
// substitution -- the contract of inverse5 (tg_segment.cuh) for any n.  Eigen's fixed-size inverse() is this algorithm
// (PartialPivLU) for n > 4; for n <= 4 Eigen uses cofactor formulas, which are not restated (DESIGN.md).
template <int H>
TG_HD void inverse_lu(const double* Din, double* out) {
  double lu[H][H];
  int perm[H];
  for (int i = 0; i < H; ++i) {
    perm[i] = i;
    for (int j = 0; j < H; ++j) lu[i][j] = Din[i * H + j];
  }
  for (int k = 0; k < H; ++k) {
    int piv = k;
    double best = dabs(lu[k][k]);
    for (int i = k + 1; i < H; ++i) {
      const double a = dabs(lu[i][k]);
      if (a > best) { best = a; piv = i; }
    }
    if (piv != k) {
      for (int j = 0; j < H; ++j) { const double t = lu[k][j]; lu[k][j] = lu[piv][j]; lu[piv][j] = t; }
      const int t = perm[k]; perm[k] = perm[piv]; perm[piv] = t;
    }
    for (int i = k + 1; i < H; ++i) lu[i][k] = lu[i][k] / lu[k][k];
    for (int i = k + 1; i < H; ++i)
      for (int j = k + 1; j < H; ++j) lu[i][j] = lu[i][j] - lu[i][k] * lu[k][j];
  }
  for (int c = 0; c < H; ++c) {
    double y[H];
    for (int i = 0; i < H; ++i) {
      double s = (perm[i] == c) ? 1.0 : 0.0;
      for (int j = 0; j < i; ++j) s = s - lu[i][j] * y[j];
      y[i] = s;
    }
    for (int i = H - 1; i >= 0; --i) {
      double s = y[i];
      for (int j = i + 1; j < H; ++j) s = s - lu[i][j] * y[j];
      y[i] = s / lu[i][i];
    }
    for (int i = 0; i < H; ++i) out[i * H + c] = y[i];
  }
}

// A^-1 and Q of one segment time (dense, zeros written).  r = derivative whose squared integral is minimised, 2 <= r <= N/2 - 1.
template <int N>
TG_HD void record_head(double T, int r, double* __restrict__ rec) {
  constexpr int H = N / 2;
  double* __restrict__ Ainv = rec + Rec<N>::kAinv;
  double* __restrict__ Q = rec + Rec<N>::kQ;
  for (int e = 0; e < N * N; ++e) {
    Ainv[e] = 0.0;
    Q[e] = 0.0;
  }
  // Q[i][j] = B[r][i] B[r][j] pow(T, e) 2/e, e = i + j - 2r + 1, left to right (lin_impl.h:605-618)
  {
    double pw[2 * N];
    const int emax = (N - 1 - r) * 2 + 1;
    tgdm::powers(T, emax, pw);
    for (int i = r; i < N; ++i)
      for (int j = r; j < N; ++j) {
        const int e = i + j - 2 * r + 1;
        Q[i * N + j] = bcoef(r, i) * bcoef(r, j) * pw[e - 1] * 2.0 / (double)e;
      }
  }
  // rows k + H of A: derivative k at t = T, entry j = B[k][j] tp with tp = T, T*T, ... restarted per row (eth/polynomial.h:208-226)
  const bool tzero = dabs(T) < TG_DBL_EPSILON;
  double C[H * H], D[H * H], Dinv[H * H], a_inv[H];
  for (int k = 0; k < H; ++k) {
    a_inv[k] = 1.0 / bcoef(k, k);  // cwiseInverse of the diagonal of the upper-left block (lin_impl.h:166-167)
    double row[N];
    for (int j = 0; j < N; ++j) row[j] = 0.0;
    row[k] = bcoef(k, k);
    if (!tzero) {
      double tp = T;
      for (int j = k + 1; j < N; ++j) {
        row[j] = bcoef(k, j) * tp;
        tp = tp * T;
      }
    }
    for (int j = 0; j < H; ++j) {
      C[k * H + j] = row[j];
      D[k * H + j] = row[H + j];
    }
  }
  inverse_lu<H>(D, Dinv);
  for (int k = 0; k < H; ++k) Ainv[k * N + k] = a_inv[k];
  for (int i = 0; i < H; ++i)
    for (int j = 0; j < H; ++j) {
      // ((-Dinv) C) diag(a_inv), inner index ascending (lin_impl.h:173-176)
      double m = (-Dinv[i * H + 0]) * C[0 * H + j];
      for (int k = 1; k < H; ++k) m = m + (-Dinv[i * H + k]) * C[k * H + j];
      Ainv[(i + H) * N + j] = m * a_inv[j];
      Ainv[(i + H) * N + (j + H)] = Dinv[i * H + j];
    }
}

// row a of H = (A^-T Q) A^-1 from the head of the record; both products accumulate over ascending k starting from the k = 0 term
template <int N>
TG_HD void record_hrow(double* __restrict__ rec, int a) {
  const double* __restrict__ Ainv = rec + Rec<N>::kAinv;
  const double* __restrict__ Q = rec + Rec<N>::kQ;
  double W[N];
#pragma unroll
  for (int b = 0; b < N; ++b) {
    double s = Ainv[0 * N + a] * Q[0 * N + b];
#pragma unroll
    for (int k = 1; k < N; ++k) s = s + Ainv[k * N + a] * Q[k * N + b];
    W[b] = s;
  }
  double* __restrict__ Hrow = rec + Rec<N>::kH + a * N;
#pragma unroll
  for (int b = 0; b < N; ++b) {
    double s = W[0] * Ainv[0 * N + b];
#pragma unroll
    for (int k = 1; k < N; ++k) s = s + W[k] * Ainv[k * N + b];
    Hrow[b] = s;
  }
}

// ---- one problem per warp ---------------------------------------------------------------------------------------------
struct Problem {
  int S, np, hbw, r;
  int rec_stride;        // records per segment: 1 (one time per segment) or 3 (the time variants of a Mellinger evaluation)
  int variant;           // with 3 records: 0 the point itself, n >= 1 the point perturbed along segment n-1
  const uint8_t* vmask;  // [V]
  const int* vfree;      // [V+1]
  const double* vval;    // [V][N/2][4]
  const double* recs;    // [S][rec_stride][Rec<N>::kSize]
  double* coef;          // [S][4][N], or null
  double* cost;          // scalar
  double* ws;            // solve_ws_doubles<N>(S, np, hbw) doubles
  double* dp = nullptr;  // [4][np]: the free derivatives d_p, dimension-major (getFreeConstraints, lin_impl.h:513-516), or null
};
// the record segment s is solved with: variant 0 for every segment of the point itself; for the point perturbed along segment
// n-1, variant 1 (T + 0.1) on that segment and variant 2 (T - 0.1/(S-1)) on the others (nl_impl.h:282-323)
template <int N>
TG_HD const double* problem_rec(const Problem& P, int s) {
  const int which = (P.rec_stride == 1 || P.variant == 0) ? 0 : (s == P.variant - 1 ? 1 : 2);
  return P.recs + ((size_t)s * P.rec_stride + which) * Rec<N>::kSize;
}
// the record segment s is solved with by a derivative-free candidate (tg_dfo_generic.cuh), the rule of solve_rec (tg_solve.cuh) for
// variant <= 0: variant 0 the point itself (record 0 everywhere); variant -(2 i + dir + 1) the point with segment i moved by +step
// (dir 0) or -step (dir 1): record 1 + dir on segment i and record 0 on every other segment (DESIGN.md 4.4)
template <int N>
TG_HD const double* candidate_rec(const Problem& P, int s) {
  int which = 0;
  if (P.variant < 0) {
    const int c = -P.variant - 1;
    which = (s == (c >> 1)) ? 1 + (c & 1) : 0;
  }
  return P.recs + ((size_t)s * P.rec_stride + which) * Rec<N>::kSize;
}
template <int N, bool kCandidate>
TG_HD const double* warp_rec(const Problem& P, int s) {
  if (kCandidate) return candidate_rec<N>(P, s);
  return problem_rec<N>(P, s);
}
TG_HD int row_stride(int hbw) { return 2 * hbw + 1 + TG_D + 1; }  // band, 4 right-hand sides, reciprocal pivot
template <int N>
TG_HD size_t ws_doubles(int S, int np, int hbw) {
  const size_t V = (size_t)S + 1;
  return (size_t)np * row_stride(hbw) + 4 * (size_t)np + (size_t)S * TG_D * N + (size_t)S * TG_D + (V * (N / 2) + 1) / 2 + 2;
}

// coefficient a of one (segment, dimension) = row a of A^-1 against the N end-point derivatives (derivatives 0 .. N/2-1 at
// vertex s, then at vertex s+1; nd(k) returns derivative k), a dense sum over ascending k (lin_impl.h:271-280)
template <int N, class Endpoint>
TG_HD double coef_from_endpoints(const double* Ai_row, const Endpoint& nd) {
  double c = 0.0;
  for (int k = 0; k < N; ++k) {
    const double e = nd(k);  // before the load of A^-1 and without __restrict__: solve_warp's phase 4 compiles as it did inline
    const double t = Ai_row[k] * e;
    c = (k == 0) ? t : c + t;
  }
  return c;
}
// (c^T Q) c of one (segment, dimension), dense (lin_impl.h:135-137)
template <int N>
TG_HD double cost_partial(const double* __restrict__ Q, const double* __restrict__ c) {
  double partial = 0.0;
  for (int b = 0; b < N; ++b) {
    double sum = c[0] * Q[0 * N + b];
    for (int k = 1; k < N; ++k) sum = sum + c[k] * Q[k * N + b];
    partial = (b == 0) ? sum * c[b] : partial + sum * c[b];
  }
  return partial;
}
// rank of derivative a among the free (clear) bits of a vertex mask: the slot's offset from the vertex's first free unknown
TG_HD int free_rank(uint32_t mask, int a) {
  int rank = 0;
  for (int q = 0; q < a; ++q) rank += ((mask >> q) & 1u) ? 0 : 1;
  return rank;
}

// kCandidate: the records are selected by candidate_rec (a derivative-free candidate) instead of problem_rec
template <int N, bool kCandidate = false>
TG_HD void solve_warp(const Problem& P, int lane) {
  constexpr int H = N / 2;
  (void)lane;
  const int S = P.S, V = S + 1, np = P.np, hbw = P.hbw, W = row_stride(hbw), RB = 2 * hbw + 1;
  double* __restrict__ rows = P.ws;
  double* __restrict__ xs = rows + (size_t)np * W;          // [np][4]
  double* __restrict__ cf = xs + 4 * (size_t)np;             // [S][4][N]
  double* __restrict__ part = cf + (size_t)S * TG_D * N;     // [S][4]
  int* __restrict__ slot = (int*)(part + (size_t)S * TG_D);  // [V][H]: index of the free unknown, -1 when fixed
  // ---- phase 0: slot table, zero the banded rows
  TG_PHASE(lane) {
    for (int it = lane; it < V * H; it += 32) {
      const int v = it / H, a = it - v * H;
      const uint32_t m = P.vmask[v];
      slot[it] = ((m >> a) & 1u) ? -1 : P.vfree[v] + free_rank(m, a);
    }
    for (int e = lane; e < np * W; e += 32) rows[e] = 0.0;
  }
  if (np > 0) {
    // ---- phase 1: rows of Rpp and rhs = (-Rpf) d_f, one lane per free (vertex, derivative); columns in ascending order
    // (vertex v-1, v, v+1); the entry shared by two segments adds segment v-1 first (lin_impl.h:317-333)
    TG_PHASE(lane) {
      for (int it = lane; it < V * H; it += 32) {
        const int i = slot[it];
        if (i < 0) continue;
        const int v = it / H, a = it - v * H;
        const bool has_p = v > 0, has_c = v < S;
        const double* hp = has_p ? warp_rec<N, kCandidate>(P, v - 1) + Rec<N>::kH + (H + a) * N : nullptr;
        const double* hc = has_c ? warp_rec<N, kCandidate>(P, v) + Rec<N>::kH + a * N : nullptr;
        double* row = rows + (size_t)i * W;
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
        for (int g = 0; g < 3; ++g) {
          const int w = v - 1 + g;
          if (w < 0 || w > S) continue;
          for (int b = 0; b < H; ++b) {
            double rv;
            if (g == 0) rv = hp[b];
            else if (g == 2) rv = hc[H + b];
            else rv = has_p ? (has_c ? hp[H + b] + hc[b] : hp[H + b]) : hc[b];
            const int j = slot[w * H + b];
            if (j >= 0) {
              row[j - i + hbw] = rv;
            } else {
              const double* f = P.vval + ((size_t)w * H + b) * TG_D;
              const double nr = -rv;
              acc0 = acc0 + nr * f[0];
              acc1 = acc1 + nr * f[1];
              acc2 = acc2 + nr * f[2];
              acc3 = acc3 + nr * f[3];
            }
          }
        }
        row[RB + 0] = acc0;
        row[RB + 1] = acc1;
        row[RB + 2] = acc2;
        row[RB + 3] = acc3;
      }
    }
    // ---- phase 2: LU without pivoting on the full band, multipliers through the reciprocal pivot; lane -> (row, column group)
    for (int k = 0; k < np; ++k) {
      TG_PHASE(lane) {
        const int iend = imin(np - 1, k + hbw);
        const int nr = iend - k;
        double* rk = rows + (size_t)k * W;
        const double rinv = 1.0 / rk[hbw];
        const int ri = lane >> 2, cg = lane & 3;
        if (lane == 0) rk[RB + TG_D] = rinv;
        for (int i = k + 1 + ri; i <= iend; i += 8) {
          double* rw = rows + (size_t)i * W;
          const double l = rw[k - i + hbw] * rinv;
          const int sh = i - k;
          for (int c = cg; c < nr; c += 4) {
            const int pk = c + 1 + hbw;
            rw[pk - sh] = rw[pk - sh] - l * rk[pk];
          }
          rw[RB + cg] = rw[RB + cg] - l * rk[RB + cg];
        }
      }
    }
    // ---- phase 3: back substitution, column oriented: far columns are subtracted first
    for (int j = np - 1; j >= 0; --j) {
      TG_PHASE(lane) {
        const int d = lane & 3, ri = lane >> 2;
        const double* rj = rows + (size_t)j * W;
        const double xj = rj[RB + d] * rj[RB + TG_D];
        if (ri == 0) xs[j * 4 + d] = xj;
        if (ri == 0 && P.dp) P.dp[(size_t)d * np + j] = xj;
        const int i0 = imax(0, j - hbw);
        for (int i = j - 1 - ri; i >= i0; i -= 8) {
          double* rw = rows + (size_t)i * W;
          rw[RB + d] = rw[RB + d] - rw[j - i + hbw] * xj;
        }
      }
    }
  }
  // ---- phase 4: coefficients c = A^-1 [derivatives of vertex s ; of vertex s+1], dense row sums (lin_impl.h:271-280)
  TG_PHASE(lane) {
    for (int it = lane; it < S * TG_D * N; it += 32) {
      const int s = it / (TG_D * N), rem = it - s * (TG_D * N), d = rem / N, a = rem - d * N;
      const double* Ai = warp_rec<N, kCandidate>(P, s) + Rec<N>::kAinv + a * N;
      const double c = coef_from_endpoints<N>(Ai, [&](int k) {
        const int j = slot[s * H + k];  // the slots of vertex s and of vertex s+1 are contiguous in the table
        return (j >= 0) ? xs[j * 4 + d] : P.vval[((size_t)s * H + k) * TG_D + d];
      });
      cf[it] = c;
      if (P.coef) P.coef[it] = c;
    }
  }
  // ---- phase 5: (c^T Q) c per (segment, dimension), dense (lin_impl.h:135-137)
  TG_PHASE(lane) {
    for (int it = lane; it < S * TG_D; it += 32) {
      const int s = it / TG_D;
      part[it] = cost_partial<N>(warp_rec<N, kCandidate>(P, s) + Rec<N>::kQ, cf + (size_t)it * N);
    }
  }
  // ---- phase 6: total in (segment, dimension) order (lin_impl.h:131-140)
  TG_PHASE(lane) {
    if (lane == 0) {
      double total = 0.0;
      for (int it = 0; it < S * TG_D; ++it) total += part[it];
      *P.cost = 0.5 * total;
    }
  }
}

// ---- evaluation ---------------------------------------------------------------------------------------------------------
// Polynomial::evaluate(t, derivative) (eth/polynomial.h:115-150): Horner over the base coefficients, multiply then add
template <int N>
TG_HD double poly_eval_n(const double* __restrict__ c, double t, int deriv) {
  if (deriv >= N) return 0.0;
  double acc = bcoef(deriv, N - 1) * c[N - 1];
  for (int j = N - 2; j >= deriv; --j) {
    acc = acc * t;
    acc = acc + bcoef(deriv, j) * c[j];
  }
  return acc;
}
// one sample: x y z yaw as getTrajectoryReference emits them, and p4 v4 a4 j3 s3 yaw (the layout of sample_eval, tg_node.cuh)
template <int N>
TG_HD void sample_eval_n(const double* __restrict__ coef, double tin, double* __restrict__ xyzh, double* __restrict__ full) {
  const double px = poly_eval_n<N>(coef + 0 * N, tin, 0), py = poly_eval_n<N>(coef + 1 * N, tin, 0);
  const double pz = poly_eval_n<N>(coef + 2 * N, tin, 0), ph = poly_eval_n<N>(coef + 3 * N, tin, 0);
  const double ha = 0.5 * ph;
  const double qw = tgdm::dcos_k(ha), qz = tgdm::dsin_k(ha);
  const double yaw = tgdm::datan2_k(2.0 * (qw * qz + 0.0 * 0.0), 1.0 - 2.0 * (0.0 * 0.0 + qz * qz));
  if (xyzh) {
    xyzh[0] = px;
    xyzh[1] = py;
    xyzh[2] = pz;
    xyzh[3] = yaw;
  }
  if (full) {
    full[0] = px; full[1] = py; full[2] = pz; full[3] = ph;
    for (int d = 0; d < TG_D; ++d) {
      full[4 + d] = poly_eval_n<N>(coef + d * N, tin, 1);
      full[8 + d] = poly_eval_n<N>(coef + d * N, tin, 2);
    }
    for (int d = 0; d < 3; ++d) {
      full[12 + d] = poly_eval_n<N>(coef + d * N, tin, 3);
      full[15 + d] = poly_eval_n<N>(coef + d * N, tin, 4);
    }
    full[18] = yaw;
  }
}

// ---- kernels (functors for the backends' for_each / for_each_warp) -----------------------------------------------------------
template <int N>
struct RecordHeadFn {  // one thread per segment
  int r;
  const double* times;
  double* recs;
  TG_HD void operator()(size_t s) const { record_head<N>(times[s], r, recs + s * Rec<N>::kSize); }
};
template <int N>
struct RecordHrowFn {  // one thread per (segment, row)
  double* recs;
  TG_HD void operator()(size_t it) const {
    const size_t s = it / N;
    record_hrow<N>(recs + s * Rec<N>::kSize, (int)(it - s * N));
  }
};
template <int N>
struct SolveFn {  // one warp per problem
  int r;
  const int* vtx_off;       // [B+1]
  const uint8_t* vmask;     // [totV]
  const int* vfree;         // [totV + B]: V+1 entries per problem, problem p's at vtx_off[p] + p
  const double* vval;       // [totV][N/2][4]
  const int* np;            // [B]
  const int* hbw;           // [B]
  const double* recs;       // [totS][Rec<N>::kSize]
  const long long* ws_off;  // [B] offsets into ws (doubles)
  double* ws;
  double* coef;             // [totS][4][N]
  double* cost;             // [B]
  TG_HD void operator()(size_t p, int lane) const { solve_warp<N>(problem(p), lane); }
  TG_HD Problem problem(size_t p) const {
    const int v0 = vtx_off[p], s0 = v0 - (int)p;
    Problem P;
    P.S = vtx_off[p + 1] - v0 - 1;
    P.np = np[p];
    P.hbw = hbw[p];
    P.r = r;
    P.rec_stride = 1;
    P.variant = 0;
    P.vmask = vmask + v0;
    P.vfree = vfree + v0 + p;
    P.vval = vval + (size_t)v0 * (N / 2) * TG_D;
    P.recs = recs + (size_t)s0 * Rec<N>::kSize;
    P.coef = coef + (size_t)s0 * TG_D * N;
    P.cost = cost + p;
    P.ws = ws + ws_off[p];
    return P;
  }
};
// SolveFn that also writes every problem's free derivatives d_p (getFreeConstraints after solveLinear, lin_impl.h:340-373, 513-516)
template <int N>
struct SolveFreeFn {
  SolveFn<N> solve;
  const long long* dp_off;  // [B]: offset of problem p's [4][np] block in dp
  double* dp;
  TG_HD void operator()(size_t p, int lane) const {
    Problem P = solve.problem(p);
    P.dp = dp + dp_off[p];
    solve_warp<N>(P, lane);
  }
};
// setFreeConstraints + getSegments (lin_impl.h:519-522 -> updateSegmentsFromCompactConstraints 263-282): one thread per (segment,
// dimension) computes the coefficients from the fixed values and the caller's free vector, with the functions phases 4 and 5 of
// solve_warp use, and the cost partial; SetFreeCostFn then adds the partials as phase 6 does.  Reads A^-1 and Q of the record heads
// only (RecordHeadFn): no row of H is needed without a solve.
template <int N>
struct SetFreeFn {
  const int* prob_of_seg;   // [totS]
  const uint8_t* vmask;     // [totV]
  const int* vfree;         // [totV + B], as in SolveFn
  const double* vval;       // [totV][N/2][4]
  const long long* dp_off;  // [B]
  const int* np;            // [B]
  const double* dp;         // problem p: [4][np[p]] at dp_off[p]
  const double* recs;       // [totS][Rec<N>::kSize]
  double* coef;             // [totS][4][N]
  double* part;             // [totS][4]
  TG_HD void operator()(size_t it) const {
    constexpr int H = N / 2;
    const size_t gs = it / TG_D;
    const int d = (int)(it - gs * TG_D), p = prob_of_seg[gs];
    const int v = (int)gs + p;  // first vertex of the segment: segment s of problem p joins vertices vtx_off[p] + s and + s + 1
    const int* vf = vfree + v + p;  // problem p's table starts at vtx_off[p] + p
    const double* x = dp + dp_off[p] + (size_t)d * np[p];
    const double* rec = recs + gs * Rec<N>::kSize;
    double c[N];
    for (int a = 0; a < N; ++a)
      c[a] = coef_from_endpoints<N>(rec + Rec<N>::kAinv + a * N, [&](int k) {
        const int w = k / H, b = k - w * H;
        const uint32_t m = vmask[v + w];
        return ((m >> b) & 1u) ? vval[((size_t)(v + w) * H + b) * TG_D + d] : x[vf[w] + free_rank(m, b)];
      });
    for (int a = 0; a < N; ++a) coef[it * N + a] = c[a];
    part[it] = cost_partial<N>(rec + Rec<N>::kQ, c);
  }
};
struct SetFreeCostFn {  // one thread per problem: the total in (segment, dimension) order (lin_impl.h:131-140)
  const int* vtx_off;
  const double* part;
  double* cost;
  TG_HD void operator()(size_t p) const {
    const int s0 = vtx_off[p] - (int)p, S = vtx_off[p + 1] - vtx_off[p] - 1;
    double total = 0.0;
    for (int it = 0; it < S * TG_D; ++it) total += part[(size_t)s0 * TG_D + it];
    cost[p] = 0.5 * total;
  }
};
// Trajectory::evaluate(t, derivative) (eth/trajectory.cpp:55-87): one thread per query time
template <int N>
struct EvaluateFn {
  int S, deriv;
  const double* coef;
  const double* T;
  const double* tq;
  double* out;
  uint8_t* ok;
  TG_HD void operator()(size_t qi) const {
    const double t = tq[qi];
    double acc = 0.0;
    int i = 0;
    for (i = 0; i < S; ++i) {
      acc = acc + T[i];
      if (acc > t) break;
    }
    if (t > acc) {
      for (int d = 0; d < TG_D; ++d) out[4 * qi + d] = 0.0;
      if (ok) ok[qi] = 0;
      return;
    }
    if (i >= S) i = S - 1;
    acc = acc - T[i];
    for (int d = 0; d < TG_D; ++d) out[4 * qi + d] = poly_eval_n<N>(coef + ((size_t)i * TG_D + d) * N, t - acc, deriv);
    if (ok) ok[qi] = 1;
  }
};
template <int N>
struct SampleEvalFn {  // one thread per sample slot; slots beyond a trajectory's count are skipped
  const int* seg_off;   // [B+1]
  const int* smp_off;   // [B+1] slot offsets (capacity scan)
  const int* smp_prob;  // slot -> trajectory
  const int* count;     // [B]
  const int* seg_idx;
  const double* t_in;
  const double* coef;
  double* xyzh;  // [slots][4] or null
  double* full;  // [slots][19] or null
  TG_HD void operator()(size_t slot) const {
    const int p = smp_prob[slot];
    if ((int)slot - smp_off[p] >= count[p]) return;
    const int gs = seg_off[p] + seg_idx[slot];
    sample_eval_n<N>(coef + (size_t)gs * TG_D * N, t_in[slot], xyzh ? xyzh + 4 * slot : nullptr, full ? full + 19 * slot : nullptr);
  }
};

// ---- maxima, time scaling and the Mellinger evaluation ----------------------------------------------------------------------
// Per-segment maximum of quantity Q (tg_poly.cuh over N coefficients): one thread per work item (every segment, or the entries of a
// device work list), one launch per quantity so that a kernel has one polynomial degree.  Every (segment, quantity) goes through
// exact root finding: the Bernstein certificates of tg_bound.cuh are built for N = 10, and since they never change a result,
// leaving them out only costs time.
template <int N, int Q>
struct ExtremaFn {
  const double* coef;  // [totS][4][N]
  const double* times;
  double* maxima;      // [totS][9]
  const int* work;     // optional work list
  const int* n_dev;    // optional length of the work list (device memory)
  static constexpr int kScratch = JtScratch<QuantityDegree<Q, N>::value>::kShared;
  TG_HD void operator()(size_t item, double* scratch, int stride) const {
    if (n_dev && item >= (size_t)*n_dev) return;
    const size_t gs = work ? (size_t)work[item] : item;
    maxima[gs * 9 + Q] = segment_max_impl<Q, N>(coef + gs * TG_D * N, times[gs], scratch, stride, nullptr);
  }
};
// computeMaximumOfMagnitude (lin_impl.h:477-508), step 1 over N coefficients; step 2 is MaxMagnitudeReduceFn
template <int N, int K>
struct MaxMagnitudeSegFn {
  const double* coef;
  const double* times;
  double* seg_value;
  double* seg_time;
  static constexpr int kScratch = JtScratch<MaxAllDegree<K, N>::value>::kShared;
  TG_HD void operator()(size_t gs, double* scratch, int stride) const {
    segment_max_all_dims<K, N>(coef + gs * TG_D * N, times[gs], scratch, stride, seg_value + gs, seg_time + gs);
  }
};
template <int N>
struct ScaleFn {  // one thread per segment (eth/trajectory.cpp:610-658); b.coef is [totS][4][N]
  BatchPtrs b;
  double L[9];
  uint8_t* changed;  // [totS]: 1 when the segment was stretched by a factor other than exactly 1
  TG_HD void operator()(size_t gs) const {
    const int p = b.prob_of_seg[gs];
    if (b.ps[p].scale_done) return;
    const double s = violation_scaling(b.maxima + gs * 9, L);
    scale_segment<N>(b.coef + gs * TG_D * N, b.times + gs, s);
    changed[gs] = (s != 1.0) ? 1 : 0;
  }
};

// One Mellinger evaluation (nl_impl.h:282-323): records of every segment at three times, item = 3 * segment + variant, the times
// computed exactly as SetupMellingerFn computes them; nothing for a problem whose optimiser has finished, nor for the perturbed
// variants of a one-segment problem (its gradient needs the point only).  b.recs: [totS][3][Rec<N>::kSize].
TG_HD bool mellinger_item_live(const BatchPtrs& b, size_t gs, int which, int* S) {
  const int p = b.prob_of_seg[gs];
  if (b.opt[p].done) return false;
  *S = b.seg_off[p + 1] - b.seg_off[p];
  return !(*S == 1 && which != 0);
}
template <int N>
struct MellingerHeadFn {  // one thread per (segment, variant)
  BatchPtrs b;
  TG_HD void operator()(size_t item) const {
    const size_t gs = item / 3;
    const int which = (int)(item - gs * 3);
    int S;
    if (!mellinger_item_live(b, gs, which, &S)) return;
    double T = b.xeval[gs];
    if (which == 1) {
      T = T + 0.1;
      T = dmax(kTimeLowerBound, T);
    } else if (which == 2) {
      const double corr = 0.1 / ((double)S - 1.0);  // nl_impl.h:288
      T = T - corr;
      T = dmax(kTimeLowerBound, T);
    }
    record_head<N>(T, b.r, b.recs + item * Rec<N>::kSize);
  }
};
template <int N>
struct MellingerHrowFn {  // one thread per (segment, variant, row)
  BatchPtrs b;
  TG_HD void operator()(size_t it) const {
    const size_t item = it / N, gs = item / 3;
    int S;
    if (!mellinger_item_live(b, gs, (int)(item - gs * 3), &S)) return;
    record_hrow<N>(b.recs + item * Rec<N>::kSize, (int)(it - item * N));
  }
};
// one warp per solve instance = vertex index: instance (p, n) is vertex n of problem p, n = 0 the point, n >= 1 the point perturbed
// along segment n-1 (the numbering of SolveProblemDesc mode 1).  Cost to b.costs[first vertex of p + n]; coefficients for n = 0 only.
template <int N>
struct MellingerSolveFn {
  BatchPtrs b;
  const long long* ws_off;  // [totV] workspace offset of every instance (doubles)
  double* ws;
  TG_HD void operator()(size_t inst, int lane) const {
    const int p = b.prob_of_vtx[inst], v0 = vtx_off(b, p), n = (int)inst - v0;
    if (b.opt[p].done) return;
    const int s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0;
    if (S == 1 && n > 0) return;
    Problem P;
    P.S = S;
    P.np = b.np[p];
    P.hbw = b.hbw[p];
    P.r = b.r;
    P.rec_stride = 3;
    P.variant = n;
    P.vmask = b.vmask + v0;
    P.vfree = b.vfree + v0 + p;
    P.vval = b.vval + (size_t)v0 * (N / 2) * TG_D;
    P.recs = b.recs + (size_t)s0 * 3 * Rec<N>::kSize;
    P.coef = (n == 0) ? b.coef + (size_t)s0 * TG_D * N : nullptr;
    P.cost = b.costs + v0 + n;
    P.ws = ws + ws_off[inst];
    solve_warp<N>(P, lane);
  }
};

}  // namespace gen

// the dt walk of evaluateRange (eth/trajectory.cpp:93-151) without the per-problem state of the optimisation pipeline
struct GenSampleCapFn {
  const int* seg_off;
  const double* times;
  double dt;
  int* cap;
  TG_HD void operator()(size_t p) const { cap[p] = sample_cap(seg_off[p + 1] - seg_off[p], times + seg_off[p], dt); }
};
struct GenSampleWalkFn {
  const int* seg_off;
  const double* times;
  double dt;
  const int* smp_off;  // [B+1] exclusive scan of cap
  int* seg_idx;
  double* t_in;
  int* count;
  TG_HD void operator()(size_t p) const {
    const int cap = smp_off[p + 1] - smp_off[p];
    const int S = seg_off[p + 1] - seg_off[p];
    const int m = sample_walk(S, times + seg_off[p], 0.0, total_time(S, times + seg_off[p]), dt, cap, seg_idx + smp_off[p], t_in + smp_off[p], nullptr);
    count[p] = m > cap ? cap : m;
  }
};
// sampleTrajectoryInRange / evaluateRange (eth/trajectory_sampling.cpp:49-104, eth/trajectory.cpp:93-151): the walk over the window
// [t_range[2p], t_range[2p+1]] of trajectory p, capped by sample_range_cap.  Without row_off it only counts; with row_off (the
// exclusive scan of those counts) it writes every sample's segment, time in segment, accumulated time and time_from_start_ns at its
// compacted row.  A count past the cap raises *overflow: the call fails instead of returning a short window.
struct RangeWalkFn {
  const int* seg_off;
  const double* times;
  const double* t_range;  // [B][2]
  double dt;
  const int* row_off;  // [B+1] or null
  int* count;          // [B], written by the counting pass
  int* seg_idx;        // [rows]
  double* t_in;        // [rows]
  double* acc;         // [rows]
  long long* t_ns;     // [rows] or null
  int* overflow;
  TG_HD void operator()(size_t p) const {
    const int s0 = seg_off[p], S = seg_off[p + 1] - s0;
    const double t_start = t_range[2 * p], t_end = t_range[2 * p + 1];
    const int cap = sample_range_cap(S, times + s0, t_start, t_end, dt);
    int m = cap + 1;
    if (cap >= 0) {
      const int r = row_off ? row_off[p] : 0;
      m = sample_walk(S, times + s0, t_start, t_end, dt, cap, row_off ? seg_idx + r : nullptr, t_in + r, acc + r);
      if (row_off && t_ns)
        for (int k = 0; k < m && k < cap; ++k) t_ns[r + k] = (long long)((t_start + dt * (double)k) * 1.e9);  // trajectory_sampling.cpp:98
    }
    if (m > cap) TG_ATOMIC_ADD(overflow, 1);
    if (!row_off) count[p] = m > cap ? 0 : m;
  }
};
namespace gen {
// Trajectory::evaluateRange's values: derivative `deriv` of the D dimensions at every compacted row, zeros for deriv >= N
template <int N>
struct EvaluateRangeFn {  // one thread per row
  const int* seg_off;
  const int* row_prob;  // row -> trajectory
  const int* seg_idx;
  const double* t_in;
  const double* coef;  // [totS][4][N]
  int deriv, D;
  double* out;  // [rows][D]
  TG_HD void operator()(size_t row) const {
    const size_t gs = (size_t)seg_off[row_prob[row]] + seg_idx[row];
    for (int d = 0; d < D; ++d) out[row * D + d] = poly_eval_n<N>(coef + (gs * TG_D + d) * N, t_in[row], deriv);
  }
};
}  // namespace gen

}  // namespace tg

#endif  // TG_GENERIC_CUH_
