// tg_solve.cuh -- one warp solves one unconstrained QP instance (one problem at one segment-time vector).
// Replaces PolynomialOptimization<10>::constructR + solveLinear + updateSegmentsFromCompactConstraints +
// computeCost (reference: lin_impl.h:310-334, 340-373, 263-282, 127-141).
//
// The reduced matrix Rpp is block tridiagonal (a free derivative of vertex v couples only to v-1, v, v+1), so it is
// assembled directly into banded rows in shared memory -- each row carries its 2*hbw+1 band entries followed by the
// four right-hand sides (x, y, z, heading) -- and factorised by LU without pivoting on the FULL non-symmetric band
// (DESIGN.md: why not Cholesky), multipliers through the reciprocal pivot (as LAPACK dgetf2 does).
//
// The routine is a sequence of PHASES (TG_PHASE): inside a phase every lane owns disjoint outputs and reads only data
// written in earlier phases; on the device a phase ends with __syncwarp(), tests/host_emu runs the lanes of a phase
// one after the other.  Round-1 profile of the first version (ncu in session 1 of round 1, DESIGN.md 4.1): 19 k warp instructions per
// solve, most of them index arithmetic and phase dispatch; this version precomputes the slot table once per solve,
// loads whole 10-entry rows of H with independent loads, and runs the factorisation as a tight loop.
#ifndef TG_SOLVE_CUH_
#define TG_SOLVE_CUH_

#include "tg_common.cuh"

#if defined(__CUDA_ARCH__)
#define TG_PHASE(lane) for (int tg_once_ = 0; tg_once_ < 1; ++tg_once_, __syncwarp())
#else
#define TG_PHASE(lane) for (int lane = 0; lane < 32; ++lane)
#endif

namespace tg {

struct SolveInst {
  int S;                  // segments
  int np;                 // free unknowns per dimension
  int hbw;                // half bandwidth of Rpp
  int fmax;               // largest number of free derivatives at one vertex (<= 4: the thread-per-instance kernel can take it)
  int variant;            // 0: base times; n >= 1: Mellinger perturbation of segment n-1 (nl_impl.h:282-311); n < 0: solve_rec
  int rec_stride;         // records per segment (1: base only, 3: base / +0.1 / -corr)
  int r;                  // derivative whose squared integral is minimised
  const uint8_t* vmask;   // [V] fixed-derivative bit masks
  const int* vfree;       // [V+1] index of the first free unknown of each vertex
  const double* vval;     // [V][5][4] fixed values
  const double* recs;     // [S*rec_stride][TG_REC_SIZE]
  double* coef_out;       // [S][4][10] or null
  double* cost_out;       // or null
  double* dp_out;         // [4][np] or null
  double* x_out;          // [np][4] or null: when set the routine stops after the back substitution and writes the solution here
                          // (coefficients and cost are then computed by CoefCostFn / CostSumFn, one thread per (segment, dimension))
  // workspace (shared or global memory)
  int W;                  // row stride: 2*hbw+1 band entries + 4 right-hand sides + the reciprocal pivot
  double* rows;           // max(np*W, 40*S): banded rows; later the coefficient scratch
  double* xs;             // np*4 solution, [row][dim]
  double* part;           // 4*S partial costs
  int16_t* slot;          // V*5: index of the free unknown of (vertex, derivative), -1 when fixed
  int16_t* rowva;         // np: (vertex, derivative) of each free unknown (octet kernel only)
};

TG_HD int solve_row_stride(int hbw) { return 2 * hbw + 1 + TG_D + 1; }  // band, 4 right-hand sides, reciprocal pivot
TG_HD int solve_ws_doubles(int S, int np, int hbw) {
  const int W = solve_row_stride(hbw);
  return imax(np * W, 40 * S) + 4 * np + 4 * S + (5 * (S + 1) + 3) / 4 + 1;
}
TG_HD void solve_ws_bind(SolveInst& I, double* ws) {
  I.W = solve_row_stride(I.hbw);
  I.rows = ws;
  I.xs = ws + imax(I.np * I.W, 40 * I.S);
  I.part = I.xs + 4 * I.np;
  I.slot = (int16_t*)(I.part + 4 * I.S);
}

// variant -(2 i + dir + 1): a one-coordinate candidate of the derivative-free search (tg_dfo.cuh), record 1 + dir on segment i
// and record 0 on every other segment
TG_HD const double* solve_rec(const SolveInst& I, int s) {
  const int which = (I.variant >= 0) ? ((I.variant == 0) ? 0 : ((s == I.variant - 1) ? 1 : 2))
                                     : ((s == ((-I.variant - 1) >> 1)) ? 1 + ((-I.variant - 1) & 1) : 0);
  return I.recs + (size_t)(s * I.rec_stride + (I.rec_stride == 1 ? 0 : which)) * TG_REC_SIZE;
}

// rank of slot a among the free slots of a vertex with mask m
TG_HD int free_rank(uint32_t m, int a) {
  const uint32_t below = (~m) & ((1u << a) - 1u) & 31u;
  return (int)((below & 1u) + ((below >> 1) & 1u) + ((below >> 2) & 1u) + ((below >> 3) & 1u) + ((below >> 4) & 1u));
}

// `lane` is the calling thread's lane on the device; the host emulation ignores it (TG_PHASE loops over the lanes).
TG_HD void solve_warp(const SolveInst& I, int lane) {
  const int S = I.S, V = S + 1, np = I.np, hbw = I.hbw, W = I.W, RB = 2 * hbw + 1;
  (void)lane;
  // ---- phase 0: slot table, zero the banded rows ---------------------------------------------------------------
  TG_PHASE(lane) {
    for (int it = lane; it < V * TG_HALF; it += 32) {
      const int v = it / TG_HALF, a = it - v * TG_HALF;
      const uint32_t m = I.vmask[v];
      I.slot[it] = ((m >> a) & 1u) ? (int16_t)-1 : (int16_t)(I.vfree[v] + free_rank(m, a));
    }
    for (int e = lane; e < np * W; e += 32) I.rows[e] = 0.0;
  }
  if (np > 0) {
    // ---- phase 1: assemble Rpp and rhs = (-Rpf) d_f.  One lane per (vertex, slot) row. ---------------------------
    TG_PHASE(lane) {
      for (int it = lane; it < V * TG_HALF; it += 32) {
        const int i = I.slot[it];
        if (i < 0) continue;
        const int v = it / TG_HALF, a = it - v * TG_HALF;
        // row (5+a) of H_{v-1} and row a of H_v hold every entry this row of R needs (lin_impl.h:317-333)
        double hp[TG_N], hc[TG_N];
        const bool has_p = v > 0, has_c = v < S;
        if (has_p) {
          const double* src = solve_rec(I, v - 1) + TG_REC_H + (TG_HALF + a) * TG_N;
#pragma unroll
          for (int q = 0; q < TG_N; ++q) hp[q] = src[q];
        }
        if (has_c) {
          const double* src = solve_rec(I, v) + TG_REC_H + a * TG_N;
#pragma unroll
          for (int q = 0; q < TG_N; ++q) hc[q] = src[q];
        }
        double* row = I.rows + (size_t)i * W;
        double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
        // columns in ascending order: vertex v-1, v, v+1 (the order of the fixed columns, lin_impl.h:235-254, 367)
#pragma unroll
        for (int g = 0; g < 3; ++g) {
          const int w = v - 1 + g;
          if (w < 0 || w > S) continue;
#pragma unroll
          for (int b = 0; b < TG_HALF; ++b) {
            double rv;
            if (g == 0) rv = hp[b];
            else if (g == 2) rv = hc[TG_HALF + b];
            else rv = has_p ? (has_c ? hp[TG_HALF + b] + hc[b] : hp[TG_HALF + b]) : hc[b];
            const int j = I.slot[w * TG_HALF + b];
            if (j >= 0) {
              row[j - i + hbw] = rv;
            } else {
              const double* f = I.vval + ((size_t)w * TG_HALF + b) * TG_D;
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
    // ---- phase 2: LU without pivoting, right-looking; lane -> (row group, column group) ----------------------------
    for (int k = 0; k < np; ++k) {
      TG_PHASE(lane) {
        const int iend = imin(np - 1, k + hbw);
        const int nr = iend - k;
        double* rk = I.rows + (size_t)k * W;
        const double rinv = 1.0 / rk[hbw];
        const int ri = lane >> 2, cg = lane & 3;
        if (lane == 0) rk[RB + TG_D] = rinv;  // kept for the back substitution (nobody reads this slot in this phase)
        for (int i = k + 1 + ri; i <= iend; i += 8) {
          double* rw = I.rows + (size_t)i * W;
          const double l = rw[k - i + hbw] * rinv;
          const int sh = i - k;  // column j sits at rk[j-k+hbw] and rw[j-i+hbw]
          for (int c = cg; c < nr; c += 4) {
            const int pk = c + 1 + hbw;
            rw[pk - sh] = rw[pk - sh] - l * rk[pk];
          }
          rw[RB + cg] = rw[RB + cg] - l * rk[RB + cg];
        }
      }
    }
    // ---- phase 3: back substitution, column oriented (far columns are subtracted first, the contract's order) ----
    for (int j = np - 1; j >= 0; --j) {
      TG_PHASE(lane) {
        const int d = lane & 3, ri = lane >> 2;
        const double* rj = I.rows + (size_t)j * W;
        const double xj = rj[RB + d] * rj[RB + TG_D];
        if (ri == 0) I.xs[j * 4 + d] = xj;
        const int i0 = imax(0, j - hbw);
        for (int i = j - 1 - ri; i >= i0; i -= 8) {
          double* rw = I.rows + (size_t)i * W;
          rw[RB + d] = rw[RB + d] - rw[j - i + hbw] * xj;
        }
      }
    }
  }
  if (I.x_out) {
    TG_PHASE(lane) {
      for (int e = lane; e < TG_D * np; e += 32) I.x_out[e] = I.xs[e];
    }
    return;
  }
  // ---- phase 4: coefficients c = A^-1 [slots of vertex s ; slots of vertex s+1]  (lin_impl.h:271-280) -----------------
  TG_PHASE(lane) {
    for (int it = lane; it < S * TG_D * TG_N; it += 32) {
      const int s = it / (TG_D * TG_N), rem = it - s * (TG_D * TG_N), d = rem / TG_N, a = rem - d * TG_N;
      double c;
      if (a < TG_HALF) {
        // rows 0..4 of A^-1 are diag(1/k!)
        const int j = I.slot[s * TG_HALF + a];
        const double nd = (j >= 0) ? I.xs[j * 4 + d] : I.vval[((size_t)s * TG_HALF + a) * TG_D + d];
        const double ai = (a < 2) ? 1.0 : ((a == 2) ? 1.0 / 2.0 : ((a == 3) ? 1.0 / 6.0 : 1.0 / 24.0));
        c = ai * nd;
      } else {
        const double* rec = solve_rec(I, s);
        const double* xr = rec + TG_REC_X + (a - TG_HALF) * 5;
        const double* dr = rec + TG_REC_DINV + (a - TG_HALF) * 5;
        double nd[TG_N];
#pragma unroll
        for (int k = 0; k < TG_N; ++k) {
          const int j = I.slot[s * TG_HALF + k];  // slots of vertex s then vertex s+1 are contiguous in the table
          nd[k] = (j >= 0) ? I.xs[j * 4 + d] : I.vval[((size_t)s * TG_HALF + k) * TG_D + d];
        }
        c = xr[0] * nd[0];
#pragma unroll
        for (int k = 1; k < 5; ++k) c = c + xr[k] * nd[k];
#pragma unroll
        for (int k = 0; k < 5; ++k) c = c + dr[k] * nd[5 + k];
      }
      I.rows[it] = c;  // scratch for the cost (the band is dead now)
      if (I.coef_out) I.coef_out[it] = c;
    }
    if (I.dp_out)
      for (int e = lane; e < TG_D * np; e += 32) I.dp_out[(e & 3) * np + (e >> 2)] = I.xs[e];
  }
  if (!I.cost_out) return;
  // ---- phase 5: partial cost of (segment, dimension): (c^T Q) c over the non-zero block (lin_impl.h:135-137) ---------
  TG_PHASE(lane) {
    const int r = I.r, nq = TG_N - r;
    for (int it = lane; it < S * TG_D; it += 32) {
      const int s = it / TG_D;
      const double* Q = solve_rec(I, s) + TG_REC_Q;
      const double* c = I.rows + it * TG_N;
      double partial = 0.0;
      for (int b = 0; b < nq; ++b) {
        double sum = c[r] * Q[tg_qsym(0, b)];
        for (int k = 1; k < nq; ++k) sum = sum + c[r + k] * Q[tg_qsym(k, b)];
        partial = (b == 0) ? sum * c[r + b] : partial + sum * c[r + b];
      }
      I.part[it] = partial;
    }
  }
  // ---- phase 6: total in (segment, dimension) order (lin_impl.h:131-140) -------------------------------------------------
  TG_PHASE(lane) {
    if (lane == 0) {
      double total = 0.0;
      for (int it = 0; it < S * TG_D; ++it) total += I.part[it];
      *I.cost_out = 0.5 * total;
    }
  }
}

}  // namespace tg

#endif  // TG_SOLVE_CUH_
