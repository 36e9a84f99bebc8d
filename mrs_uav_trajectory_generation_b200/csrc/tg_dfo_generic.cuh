// tg_dfo_generic.cuh -- the derivative-free time allocation of tg_dfo.cuh (methods 0, 1, 3, 4; nl_impl.h:120-157, 429-536) for
// PolynomialOptimization<N>, N = 6, 8, 10, 12, on 4 (zero-padded) dimensions: tg_time_alloc_dfo_batch_nd.
//
// The search, its per-problem state (DfoBatch, DfoProb), the candidate reuse and the N-independent functors (DfoMapFn, DfoBeginFn,
// DfoTotalFn, DfoBaseTotalFn, DfoAdvanceFn, DfoTimesOutFn) are those of tg_dfo.cuh.  What depends on N is here, written with the
// functions of the general-shape linear path (tg_generic.cuh), so that every objective value is the one tg_objective_batch_nd
// computes for that x, bit for bit:
//   records          record_head<N> (A^-1, Q) per (segment, variant); record_hrow<N> for methods 0, 1, whose solves read H
//   methods 0, 1     solve_warp<N> with candidate_rec: candidate (i, dir) reads record 1 + dir on segment i, record 0 elsewhere
//   methods 3, 4     coef_from_endpoints<N> / cost_partial<N> per (segment, dimension), as SetFreeFn<N> computes them
//   maxima           segment_max_all_dims<K, N> (MaxMagnitudeSegFn<N, K>)
// b.vval: [totV][N/2][4]; b.coef, ccoef: [.][4][N]; b.recs: [totS][3][Rec<N>::kSize].  Variables exist for the dimensions d < D
// only (n = S + D * n_free for methods 3, 4); a dimension d >= D is carried with zero values, which adds exact zeros to the cost
// and nothing to a magnitude, as the zero-padded objective computes it.
#ifndef TG_DFO_GENERIC_CUH_
#define TG_DFO_GENERIC_CUH_

#include "tg_dfo.cuh"
#include "tg_generic.cuh"

namespace tg {
namespace gen {

// dfo_endpoints over N coefficients: the N end-point derivatives of dimension `dim` of segment s at the point x, free slot j_over
// of dimension dim_over replaced by v_over; the free slots of a dimension dim >= D are zero
template <int N>
TG_HD void dfo_endpoints_n(const DfoBatch& d, const DfoProb& P, int p, int s, int D, int dim, int dim_over, int j_over, double v_over,
                           double (&nd)[N]) {
  constexpr int H = N / 2;
  const int v0 = P.s0 + p;
  const int* vf = d.b.vfree + P.s0 + 2 * p;
  const double* xf = d.x + (size_t)P.x0 + P.S + (size_t)dim * P.n_free;
  for (int k = 0; k < N; ++k) {
    const int v = s + (k >= H ? 1 : 0), sl = k - (k >= H ? H : 0);
    const uint32_t m = d.b.vmask[v0 + v];
    if ((m >> sl) & 1u) {
      nd[k] = d.b.vval[((size_t)(v0 + v) * H + sl) * TG_D + dim];
    } else {
      const int u = vf[v] + free_rank(m, sl);
      nd[k] = dim >= D ? 0.0 : ((dim == dim_over && u == j_over) ? v_over : xf[u]);
    }
  }
}
// coefficients and cost partial of one (segment, dimension) from its end-point derivatives (SetFreeFn<N>)
template <int N>
TG_HD double dfo_coef_part(const double* rec, const double (&nd)[N], double* co) {
  double c[N];
  for (int a = 0; a < N; ++a) c[a] = coef_from_endpoints<N>(rec + Rec<N>::kAinv + a * N, [&](int k) { return nd[k]; });
  for (int a = 0; a < N; ++a) co[a] = c[a];
  return cost_partial<N>(rec + Rec<N>::kQ, c);
}

// methods 3, 4, one thread per vertex: x0 of its free slots = derivative k of the linear solution at the initial times (b.coef),
// Trajectory::evaluate on segment v at t = 0, or on the last segment at its end for the last vertex (nl_impl.h:436-462)
template <int N>
struct DfoFreeInitFn {
  DfoBatch d;
  int D;
  TG_HD void operator()(size_t gv) const {
    const int p = d.b.prob_of_vtx[gv];
    const DfoProb& P = d.prob[p];
    const int v = (int)gv - (P.s0 + p);
    const uint32_t m = d.b.vmask[gv];
    const int seg = v < P.S ? v : P.S - 1;
    const double t = v < P.S ? 0.0 : d.b.times[P.s0 + seg];
    const double* c = d.b.coef + (size_t)(P.s0 + seg) * TG_D * N;
    const int j0 = d.b.vfree[P.s0 + 2 * p + v];
    for (int k = 0; k < N / 2; ++k) {
      if ((m >> k) & 1u) continue;
      const int j = j0 + free_rank(m, k);
      for (int dim = 0; dim < D; ++dim) d.x[(size_t)P.x0 + P.S + (size_t)dim * P.n_free + j] = poly_eval_n<N>(c + dim * N, t, k);
    }
  }
};
// records of segment items (segment, variant) as DfoRecsFn takes them: variant 0 at x_s, 1 at min(x_s + step_s, hi_s), 2 at
// max(x_s - step_s, lo_s); the head (A^-1, Q) one thread per item, the rows of H (methods 0, 1) one thread per (item, row)
TG_HD bool dfo_rec_item(const DfoBatch& d, const int* seg_list, int variants, int all, size_t item, size_t* gs, int* w, double* T) {
  const size_t k = item / (size_t)variants;
  *w = (int)(item - k * (size_t)variants);
  *gs = seg_list ? (size_t)seg_list[k] : k;
  const int p = d.b.prob_of_seg[*gs];
  const DfoProb& P = d.prob[p];
  if (!all && P.done) return false;
  const size_t q = (size_t)P.x0 + (*gs - (size_t)P.s0);
  *T = *w == 0 ? d.x[q] : (*w == 1 ? dfo_up(d.x[q], d.step[q], d.hi[q]) : dfo_dn(d.x[q], d.step[q], d.lo[q]));
  return true;
}
template <int N>
struct DfoHeadFn {
  DfoBatch d;
  const int* seg_list;  // null: every segment
  int variants;         // 1 (base point only) or 3
  int all;              // 1: also the problems whose search has stopped
  TG_HD void operator()(size_t item) const {
    size_t gs;
    int w;
    double T;
    if (!dfo_rec_item(d, seg_list, variants, all, item, &gs, &w, &T)) return;
    record_head<N>(T, d.b.r, d.b.recs + (gs * 3 + w) * Rec<N>::kSize);
  }
};
template <int N>
struct DfoHrowFn {
  DfoBatch d;
  const int* seg_list;
  int variants, all;
  TG_HD void operator()(size_t it) const {
    const size_t item = it / N;
    size_t gs;
    int w;
    double T;
    if (!dfo_rec_item(d, seg_list, variants, all, item, &gs, &w, &T)) return;
    record_hrow<N>(d.b.recs + (gs * 3 + w) * Rec<N>::kSize, (int)(it - item * N));
  }
};
// methods 0, 1, one warp per solve: base: instance = problem at x; else instance = candidate.  Problem p's candidates own
// consecutive workspaces of ws_size[p] doubles from ws_off[p]; the base solve uses the first.
template <int N>
struct DfoSolveFn {
  DfoBatch d;
  int base;
  const int* list;           // null: every instance
  const long long* ws_off;   // [G]
  const long long* ws_size;  // [G]
  double* ws;
  TG_HD void operator()(size_t k, int lane) const {
    int p, c = 0, variant = 0, kk = 0;
    if (base) {
      p = list ? list[k] : (int)k;
    } else {
      c = list ? list[k] : (int)k;
      p = d.cand_prob[c];
      if (d.prob[p].done) return;
      kk = c - d.prob[p].c0;
      const int dir = kk >= d.prob[p].n ? 1 : 0;
      variant = -(2 * (kk - dir * d.prob[p].n) + dir + 1);
    }
    const DfoProb& Q = d.prob[p];
    const int v0 = Q.s0 + p;
    Problem P;
    P.S = Q.S;
    P.np = d.b.np[p];
    P.hbw = d.b.hbw[p];
    P.r = d.b.r;
    P.rec_stride = 3;
    P.variant = variant;
    P.vmask = d.b.vmask + v0;
    P.vfree = d.b.vfree + v0 + p;
    P.vval = d.b.vval + (size_t)v0 * (N / 2) * TG_D;
    P.recs = d.b.recs + (size_t)Q.s0 * 3 * Rec<N>::kSize;
    P.coef = base ? d.b.coef + (size_t)Q.s0 * TG_D * N : d.ccoef + ((size_t)Q.i0 + (size_t)kk * Q.S) * TG_D * N;
    P.cost = base ? d.bcost + p : d.ccost + c;
    P.ws = ws + ws_off[p] + (long long)kk * ws_size[p];
    solve_warp<N, true>(P, lane);
  }
};
// methods 3, 4, one thread per (segment, dimension) of the base point: coefficients and cost partial
template <int N>
struct DfoBaseCoefFn {
  DfoBatch d;
  const int* seg_list;
  int all, D;
  TG_HD void operator()(size_t item) const {
    const size_t k = item >> 2;
    const int dim = (int)(item & 3);
    const size_t gs = seg_list ? (size_t)seg_list[k] : k;
    const int p = d.b.prob_of_seg[gs];
    const DfoProb& P = d.prob[p];
    if (!all && P.done) return;
    double nd[N];
    dfo_endpoints_n<N>(d, P, p, (int)(gs - (size_t)P.s0), D, dim, -1, -1, 0.0, nd);
    d.bpart[gs * 4 + dim] = dfo_coef_part<N>(d.b.recs + gs * 3 * Rec<N>::kSize, nd, d.b.coef + (gs * TG_D + dim) * N);
  }
};
// methods 3, 4, one thread per candidate item (DfoItemFn): the four dimensions of the one segment the item recomputes
template <int N>
struct DfoItemFn {
  DfoBatch d;
  const int* item_list;
  int D;
  TG_HD void operator()(size_t k) const {
    const size_t item = item_list ? (size_t)item_list[k] : k;
    const int c = (int)(item / (size_t)d.ipc_free), slot = (int)(item - (size_t)c * d.ipc_free);
    int i, dir;
    double val;
    const int p = dfo_cand(d, c, &i, &dir, &val);
    const DfoProb& P = d.prob[p];
    if (P.done) return;
    int dd, jj;
    const int s = dfo_item_seg(d, P, p, i, slot, &dd, &jj);
    if (s < 0) return;
    const size_t gs = (size_t)P.s0 + s;
    const double* rec = d.b.recs + (gs * 3 + (dd < 0 ? 1 + dir : 0)) * Rec<N>::kSize;
    double* co = d.ccoef + item * TG_D * N;
    for (int dim = 0; dim < TG_D; ++dim) {
      if (dd >= 0 && dim != dd) {
        for (int a = 0; a < N; ++a) co[dim * N + a] = d.b.coef[(gs * TG_D + dim) * N + a];
        d.cpart[item * 4 + dim] = d.bpart[gs * 4 + dim];
        continue;
      }
      double nd[N];
      dfo_endpoints_n<N>(d, P, p, s, D, dim, dd, jj, val, nd);
      d.cpart[item * 4 + dim] = dfo_coef_part<N>(rec, nd, co + dim * N);
    }
  }
};
// computeMaximumOfMagnitude<K> per segment (DfoMaxFn over N coefficients)
template <int N, int K>
struct DfoMaxFn {
  DfoBatch d;
  const int* list;
  int base, all;
  static constexpr int kScratch = MaxMagnitudeSegFn<N, K>::kScratch;
  TG_HD void operator()(size_t k, double* scratch, int stride) const {
    const size_t item = list ? (size_t)list[k] : k;
    double T, t_at;
    const double* co;
    double* out;
    if (base) {
      const int p = d.b.prob_of_seg[item];
      const DfoProb& P = d.prob[p];
      if (!all && P.done) return;
      T = d.x[(size_t)P.x0 + (item - (size_t)P.s0)];
      co = d.b.coef + item * TG_D * N;
      out = d.bsv + (size_t)(K - 1) * d.totS + item;
    } else {
      const int c = d.method < 3 ? d.item_cand[item] : (int)(item / (size_t)d.ipc_free);
      int i, dir, s;
      double val;
      const int p = dfo_cand(d, c, &i, &dir, &val);
      const DfoProb& P = d.prob[p];
      if (P.done) return;
      if (d.method < 3) {
        s = (int)(item - (size_t)P.i0 - (size_t)(c - P.c0) * P.S);
      } else {
        int dd, jj;
        s = dfo_item_seg(d, P, p, i, (int)(item - (size_t)c * d.ipc_free), &dd, &jj);
        if (s < 0) return;
      }
      T = s == i ? val : d.x[(size_t)P.x0 + s];
      co = d.ccoef + item * TG_D * N;
      out = d.csv + (size_t)(K - 1) * d.totItems + item;
    }
    segment_max_all_dims<K, N>(co, T, scratch, stride, out, &t_at);
  }
};
// output: the vertex values with the free slots at their final variables (methods 3, 4), one thread per vertex
template <int N>
struct DfoVvalOutFn {
  DfoBatch d;
  int D;
  double* vval;
  TG_HD void operator()(size_t gv) const {
    constexpr int H = N / 2;
    const int p = d.b.prob_of_vtx[gv];
    const DfoProb& P = d.prob[p];
    const int v = (int)gv - (P.s0 + p);
    const uint32_t m = d.b.vmask[gv];
    const int j0 = d.b.vfree[P.s0 + 2 * p + v];
    for (int k = 0; k < H; ++k)
      for (int dim = 0; dim < TG_D; ++dim) {
        const size_t o = (gv * H + k) * TG_D + dim;
        if ((m >> k) & 1u) vval[o] = d.b.vval[o];
        else vval[o] = dim < D ? d.x[(size_t)P.x0 + P.S + (size_t)dim * P.n_free + j0 + free_rank(m, k)] : 0.0;
      }
  }
};

}  // namespace gen
}  // namespace tg

#endif  // TG_DFO_GENERIC_CUH_
