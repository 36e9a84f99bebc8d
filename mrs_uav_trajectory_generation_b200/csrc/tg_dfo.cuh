// tg_dfo.cuh -- the derivative-free time allocation of PolynomialOptimizationNonLinear<10> (methods 0 kSquaredTime, 1 kRichterTime,
// 3 kSquaredTimeAndConstraints, 4 kRichterTimeAndConstraints; nl_impl.h:120-157, 429-536) for many problems per call.
//
// The search is a bound-constrained coordinate pattern search: 2n candidates per iteration, each x with one coordinate moved by
// +-step (clamped to the bounds); the first strictly smallest total is accepted when it improves f, otherwise every step halves.
// One state per problem lives in device memory and advances once per batched iteration (DfoAdvanceFn), like PlisAdvanceFn does
// for the Mellinger method.  Every objective value is the one tg_objective_batch computes for that x, bit for bit: the records,
// the coefficients (coef_from_endpoints / the solve kernels), the cost partials summed in (segment, dimension) order, the
// per-segment maxima (segment_max_all_dims) reduced in segment order and ObjTerms::combine are the same functions.
//
// A candidate recomputes only what its coordinate changes:
//   methods 0, 1 (x = the segment times): candidate (i, dir) changes T_i, i.e. one record; its linear solve reads record 1 + dir
//     on segment i and record 0 elsewhere (solve_rec, variant < 0), then coefficients, partials and maxima of all its segments.
//   methods 3, 4 (x = the times, then the free derivatives dimension-major; no linear solve): a time candidate changes segment i
//     only; a free derivative (dimension d, slot j) at vertex v changes dimension d of segments v-1 and v.  The base point's
//     per-(segment, dimension) partials and per-segment maxima are computed once per iteration and every candidate substitutes its
//     (at most two) recomputed segments into them, in the same summation and reduction order.
#ifndef TG_DFO_CUH_
#define TG_DFO_CUH_

#include "tg_kernels.cuh"

namespace tg {

// tg_dfo_params (include/tg_b200.h)
struct DfoParams {
  int time_alloc_method, derivative_to_optimize, max_iterations;
  double f_rel, x_rel, initial_stepsize_rel, time_penalty;
  int use_soft_constraints;
  double soft_constraint_weight;
};

struct DfoProb {
  int S, n, n_free;    // segments, variables, free slots per dimension
  int s0, x0, c0, i0;  // first segment, variable, candidate (2 n per problem) and candidate item of the problem
  int iterations, code, done;
  double f;
};

TG_HD double dfo_up(double x, double step, double hi) {  // std::min(x + step, hi)
  const double a = x + step;
  return (hi < a) ? hi : a;
}
TG_HD double dfo_dn(double x, double step, double lo) {  // std::max(x - step, lo)
  const double a = x - step;
  return (a < lo) ? lo : a;
}

struct DfoBatch {
  BatchPtrs b;  // vertices; b.recs [totS][3] records at x, x + step, x - step; b.coef the base point's coefficients; b.xs / b.part
  DfoProb* prob;
  int method, max_iter, ipc_free;  // ipc_free: candidate items per candidate of methods 3, 4 (2)
  double f_rel, x_rel, step_rel;
  ObjTerms obj;
  int con_dim[16];
  double *x, *lo, *hi, *step;      // [sum n]
  int* cand_prob;                  // [totCand] problem of each candidate
  int* item_cand;                  // [totItems] candidate of each item (methods 0, 1: S items per candidate)
  double *ctot, *ccost, *ccoef, *cpart, *csv;  // per candidate: total, cost (0, 1); per item: [4][10], [4] partials (3, 4), [4][totItems] maxima
  double *bcost, *bpart, *bsv, *btot, *bparts;  // base point: cost (0, 1), [totS][4] partials (3, 4), [4][totS] maxima, total, [B][3] parts
  size_t totS, totItems;
  int* lists[2][4];                // running problems, their segments, candidates and items (two alternating buffers)
  int* cnt;                        // [0] problems still running, [1 + 4 * buf + k] lengths of lists[buf][k]
};

// candidate c -> problem, variable, direction (0: +step, 1: -step) and the value of the moved variable
TG_HD int dfo_cand(const DfoBatch& d, int c, int* i, int* dir, double* val) {
  const int p = d.cand_prob[c];
  const DfoProb& P = d.prob[p];
  const int k = c - P.c0;
  *dir = k >= P.n ? 1 : 0;
  *i = k - *dir * P.n;
  const size_t q = (size_t)P.x0 + *i;
  *val = *dir ? dfo_dn(d.x[q], d.step[q], d.lo[q]) : dfo_up(d.x[q], d.step[q], d.hi[q]);
  return p;
}
// methods 3, 4: the segment recomputed by item `slot` of variable i (-1: none); a free variable also gives its dimension and slot
TG_HD int dfo_item_seg(const DfoBatch& d, const DfoProb& P, int p, int i, int slot, int* dim, int* j) {
  *dim = -1;
  *j = -1;
  if (i < P.S) return slot == 0 ? i : -1;
  const int q = i - P.S;
  *dim = q / P.n_free;
  *j = q - *dim * P.n_free;
  const int* vf = d.b.vfree + P.s0 + 2 * p;  // V + 1 entries: first free slot of each vertex
  int a = 0, e = P.S + 1;                      // vf[a] <= j < vf[e]
  while (e - a > 1) {
    const int mid = (a + e) >> 1;
    if (vf[mid] <= *j) a = mid;
    else e = mid;
  }
  const int s = a - 1 + slot;  // vertex a ends segment a - 1 and starts segment a
  return (s >= 0 && s < P.S) ? s : -1;
}
// the ten end-point derivatives of dimension `dim` of segment s (local) at the point x, free slot j_over of dimension dim_over
// replaced by v_over (setFreeConstraints, lin_impl.h:513-522, as CoefCostFn reads them)
TG_HD void dfo_endpoints(const DfoBatch& d, const DfoProb& P, int p, int s, int dim, int dim_over, int j_over, double v_over, double (&nd)[TG_N]) {
  const int v0 = P.s0 + p;
  const int* vf = d.b.vfree + P.s0 + 2 * p;
  const double* xf = d.x + (size_t)P.x0 + P.S + (size_t)dim * P.n_free;
#pragma unroll
  for (int k = 0; k < TG_N; ++k) {
    const int v = s + (k >= TG_HALF ? 1 : 0), sl = k - (k >= TG_HALF ? TG_HALF : 0);
    const uint32_t m = d.b.vmask[v0 + v];
    if ((m >> sl) & 1u) {
      nd[k] = d.b.vval[((size_t)(v0 + v) * TG_HALF + sl) * TG_D + dim];
    } else {
      const int u = vf[v] + free_rank(m, sl);
      nd[k] = (dim == dim_over && u == j_over) ? v_over : xf[u];
    }
  }
}
// appends a running problem and its work to the lists of buffer `buf`
TG_HD void dfo_enlist(const DfoBatch& d, int p, int buf) {
  const DfoProb& P = d.prob[p];
  const int ipc = d.method >= 3 ? d.ipc_free : P.S;
  int* c = d.cnt + 1 + 4 * buf;
  TG_ATOMIC_ADD(d.cnt, 1);
  d.lists[buf][0][TG_ATOMIC_ADD_RET(c + 0, 1)] = p;
  const int a = TG_ATOMIC_ADD_RET(c + 1, P.S);
  for (int s = 0; s < P.S; ++s) d.lists[buf][1][a + s] = P.s0 + s;
  const int e = TG_ATOMIC_ADD_RET(c + 2, 2 * P.n);
  for (int k = 0; k < 2 * P.n; ++k) d.lists[buf][2][e + k] = P.c0 + k;
  const int g = TG_ATOMIC_ADD_RET(c + 3, 2 * P.n * ipc);
  for (int k = 0; k < 2 * P.n * ipc; ++k) d.lists[buf][3][g + k] = P.i0 + k;
}

// ---- set-up -------------------------------------------------------------------------------------------------------------------
struct DfoMapFn {  // one thread per problem: candidate -> problem, item -> candidate
  DfoBatch d;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi;
    const DfoProb& P = d.prob[p];
    for (int k = 0; k < 2 * P.n; ++k) d.cand_prob[P.c0 + k] = p;
    if (d.method < 3)
      for (int k = 0; k < 2 * P.n; ++k)
        for (int s = 0; s < P.S; ++s) d.item_cand[P.i0 + k * P.S + s] = P.c0 + k;
  }
};
// methods 3, 4, one thread per vertex: x0 of its free slots = derivative k of the linear solution at the initial times, evaluated
// as Trajectory::evaluate does on segment v at t = 0, or on the last segment at its end for the last vertex (nl_impl.h:436-462)
struct DfoFreeInitFn {
  DfoBatch d;
  TG_HD void operator()(size_t gv) const {
    const int p = d.b.prob_of_vtx[gv];
    const DfoProb& P = d.prob[p];
    const int v = (int)gv - (P.s0 + p);
    const uint32_t m = d.b.vmask[gv];
    const int seg = v < P.S ? v : P.S - 1;
    const double t = v < P.S ? 0.0 : d.b.times[P.s0 + seg];
    const double* c = d.b.coef + (size_t)(P.s0 + seg) * TG_D * TG_N;
    const int j0 = d.b.vfree[P.s0 + 2 * p + v];
    for (int k = 0; k < TG_HALF; ++k) {
      if ((m >> k) & 1u) continue;
      const int j = j0 + free_rank(m, k);
      for (int dim = 0; dim < TG_D; ++dim) d.x[(size_t)P.x0 + P.S + (size_t)dim * P.n_free + j] = poly_eval(c + dim * TG_N, t, k);
    }
  }
};
// one thread per problem: times into x, bounds (kOptimizationTimeLowerBound; setFreeEndpointDerivativeHardConstraints,
// nl_impl.h:764-805, whose counter advances only for derivatives <= derivative_to_optimize), steps (nl_impl.h:488-495) and the
// bounds widened to an x0 outside them (nl_impl.h:497-503)
struct DfoBeginFn {
  DfoBatch d;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi;
    DfoProb& P = d.prob[p];
    double* x = d.x + P.x0;
    double* lo = d.lo + P.x0;
    double* hi = d.hi + P.x0;
    for (int s = 0; s < P.S; ++s) x[s] = d.b.times[P.s0 + s];
    for (int i = 0; i < P.n; ++i) {
      lo[i] = i < P.S ? kTimeLowerBound : -1.7976931348623157e308;
      hi[i] = 1.7976931348623157e308;
    }
    if (d.method >= 3) {
      const int v0 = P.s0 + p;
      for (int c = 0; c < d.obj.ncon; ++c) {
        int counter = 0;
        const double a = fabs(d.obj.con_value[c]);
        for (int v = 0; v <= P.S; ++v)
          for (int deriv = 0; deriv <= d.b.r; ++deriv)
            if (!((d.b.vmask[v0 + v] >> deriv) & 1u)) {
              if (deriv == d.obj.con_deriv[c]) {
                const long long at = (long long)P.S + (long long)d.con_dim[c] * P.n_free + counter;
                if (at < P.n) {
                  lo[at] = -a;
                  hi[at] = a;
                }
              }
              ++counter;
            }
      }
    }
    for (int i = 0; i < P.n; ++i) {
      const double ax = fabs(x[i]);
      d.step[P.x0 + i] = (ax <= 2.220446049250313e-16) ? 1e-13 : d.step_rel * ax;
      if (x[i] < lo[i]) lo[i] = x[i];
      else if (x[i] > hi[i]) hi[i] = x[i];
    }
    P.iterations = 0;
    P.code = 5;
    P.done = d.max_iter <= 0 ? 1 : 0;
  }
};

// ---- evaluation ---------------------------------------------------------------------------------------------------------------
// records of segment items (segment, variant): variant 0 at x_s, 1 at min(x_s + step_s, hi_s), 2 at max(x_s - step_s, lo_s).
// Methods 3, 4 only read Q, Dinv and X (setup_record_head: the same bits as setup_segment_record).
struct DfoRecsFn {
  DfoBatch d;
  const int* seg_list;  // null: every segment
  int variants;         // 1 (base point only) or 3
  int all;              // 1: also the problems whose search has stopped
  TG_HD void operator()(size_t item) const {
    const size_t k = item / (size_t)variants;
    const int w = (int)(item - k * (size_t)variants);
    const size_t gs = seg_list ? (size_t)seg_list[k] : k;
    const int p = d.b.prob_of_seg[gs];
    const DfoProb& P = d.prob[p];
    if (!all && P.done) return;
    const size_t q = (size_t)P.x0 + (gs - (size_t)P.s0);
    const double T = w == 0 ? d.x[q] : (w == 1 ? dfo_up(d.x[q], d.step[q], d.hi[q]) : dfo_dn(d.x[q], d.step[q], d.lo[q]));
    double* rec = d.b.recs + (gs * 3 + w) * TG_REC_SIZE;
    if (d.method >= 3) setup_record_head(T, d.b.r, rec);
    else setup_segment_record(T, d.b.r, rec);
  }
};
// methods 0, 1: the linear solves.  base: instance = problem at x (final / initial evaluation); else instance = candidate.
struct DfoSolveDesc {
  DfoBatch d;
  int base;
  const int* list;  // null: every instance
  TG_HD bool instance(size_t k, SolveInst& I) const {
    const BatchPtrs& b = d.b;
    int p, c = 0, variant = 0, kk = 0;
    if (base) {
      p = list ? list[k] : (int)k;
    } else {
      c = list ? list[k] : (int)k;
      p = d.cand_prob[c];
      if (d.prob[p].done) return false;
      kk = c - d.prob[p].c0;
      const int dir = kk >= d.prob[p].n ? 1 : 0;
      variant = -(2 * (kk - dir * d.prob[p].n) + dir + 1);
    }
    const DfoProb& P = d.prob[p];
    const int s0 = P.s0, v0 = s0 + p;
    I.S = P.S;
    I.np = b.np[p];
    I.hbw = b.hbw[p];
    I.fmax = b.fmax[p];
    I.variant = variant;
    I.rec_stride = 3;
    I.r = b.r;
    I.vmask = b.vmask + v0;
    I.vfree = b.vfree + v0 + p;
    I.vval = b.vval + (size_t)v0 * TG_HALF * TG_D;
    I.recs = b.recs + (size_t)s0 * 3 * TG_REC_SIZE;
    I.coef_out = base ? b.coef + (size_t)s0 * TG_D * TG_N : d.ccoef + ((size_t)P.i0 + (size_t)kk * P.S) * TG_D * TG_N;
    I.cost_out = base ? d.bcost + p : d.ccost + c;
    I.dp_out = nullptr;
    I.x_out = b.xs + (size_t)(base ? p : c) * (size_t)b.xstride;
    return true;
  }
};
// methods 3, 4, one thread per (segment, dimension) of the base point: coefficients and cost partial
struct DfoBaseCoefFn {
  DfoBatch d;
  const int* seg_list;
  int all;
  TG_HD void operator()(size_t item) const {
    const size_t k = item >> 2;
    const int dim = (int)(item & 3);
    const size_t gs = seg_list ? (size_t)seg_list[k] : k;
    const int p = d.b.prob_of_seg[gs];
    const DfoProb& P = d.prob[p];
    if (!all && P.done) return;
    double nd[TG_N], c[TG_N];
    dfo_endpoints(d, P, p, (int)(gs - (size_t)P.s0), dim, -1, -1, 0.0, nd);
    const double* rec = d.b.recs + gs * 3 * TG_REC_SIZE;
    coef_from_endpoints(rec, nd, c);
    double* co = d.b.coef + (gs * TG_D + dim) * TG_N;
    for (int a = 0; a < TG_N; ++a) co[a] = c[a];
    d.bpart[gs * 4 + dim] = cost_partial_rec(d.b.r, c, rec);
  }
};
// methods 3, 4, one thread per candidate item: the four dimensions of the one segment the item recomputes.  A time candidate
// reads its moved record; a free-derivative candidate recomputes its dimension and copies the base point's other three.
struct DfoItemFn {
  DfoBatch d;
  const int* item_list;
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
    const double* rec = d.b.recs + (gs * 3 + (dd < 0 ? 1 + dir : 0)) * TG_REC_SIZE;
    double* co = d.ccoef + item * TG_D * TG_N;
    for (int dim = 0; dim < TG_D; ++dim) {
      if (dd >= 0 && dim != dd) {
        for (int a = 0; a < TG_N; ++a) co[dim * TG_N + a] = d.b.coef[(gs * TG_D + dim) * TG_N + a];
        d.cpart[item * 4 + dim] = d.bpart[gs * 4 + dim];
        continue;
      }
      double nd[TG_N], cc[TG_N];
      dfo_endpoints(d, P, p, s, dim, dd, jj, val, nd);
      coef_from_endpoints(rec, nd, cc);
      for (int a = 0; a < TG_N; ++a) co[dim * TG_N + a] = cc[a];
      d.cpart[item * 4 + dim] = cost_partial_rec(d.b.r, cc, rec);
    }
  }
};
// computeMaximumOfMagnitude<K> per segment (MaxMagnitudeSegFn): of the base point's segments (items = segments), or of the
// candidate items (methods 0, 1: every segment of a candidate; 3, 4: its recomputed segments)
template <int K>
struct DfoMaxFn {
  DfoBatch d;
  const int* list;
  int base, all;
  static constexpr int kScratch = MaxMagnitudeSegFn<K>::kScratch;
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
      co = d.b.coef + item * TG_D * TG_N;
      out = d.bsv + (size_t)(K - 1) * d.totS + item;
    } else {
      int c, s;
      if (d.method < 3) {
        c = d.item_cand[item];
      } else {
        c = (int)(item / (size_t)d.ipc_free);
      }
      int i, dir;
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
      co = d.ccoef + item * TG_D * TG_N;
      out = d.csv + (size_t)(K - 1) * d.totItems + item;
    }
    segment_max_all_dims<K>(co, T, scratch, stride, out, &t_at);
  }
};
// one thread per candidate: total = cost + time cost + soft constraints, the base point's values with the candidate's substituted
struct DfoTotalFn {
  DfoBatch d;
  const int* cand_list;
  TG_HD void operator()(size_t k) const {
    const int c = cand_list ? cand_list[k] : (int)k;
    int i, dir;
    double val;
    const int p = dfo_cand(d, c, &i, &dir, &val);
    const DfoProb& P = d.prob[p];
    if (P.done) return;
    const double* x = d.x + P.x0;
    double total_time = 0.0;
    for (int s = 0; s < P.S; ++s) total_time = total_time + (s == i ? val : x[s]);
    const size_t ci = (size_t)P.i0 + (size_t)(c - P.c0) * (d.method < 3 ? P.S : d.ipc_free);  // the candidate's first item
    int sa = -1, sb = -1;
    double cost;
    if (d.method < 3) {
      cost = d.ccost[c];
    } else {
      int dd, jj;
      sa = dfo_item_seg(d, P, p, i, 0, &dd, &jj);
      sb = dfo_item_seg(d, P, p, i, 1, &dd, &jj);
      double tot = 0.0;
      for (int s = 0; s < P.S; ++s) {
        const double* pp = s == sa ? d.cpart + ci * 4 : (s == sb ? d.cpart + (ci + 1) * 4 : d.bpart + (size_t)(P.s0 + s) * 4);
        for (int dim = 0; dim < TG_D; ++dim) tot += pp[dim];
      }
      cost = 0.5 * tot;
    }
    double mv[4] = {0.0, 0.0, 0.0, 0.0};
    if (d.obj.use_soft)
      for (int K = 1; K <= 4; ++K) {
        bool need = false;
        for (int q = 0; q < d.obj.ncon; ++q) need = need || d.obj.con_deriv[q] == K;
        if (!need) continue;
        const double* cs = d.csv + (size_t)(K - 1) * d.totItems;
        const double* bs = d.bsv + (size_t)(K - 1) * d.totS + P.s0;
        double best = 0.0;  // MaxMagnitudeReduceFn: the running Extremum starts at 0
        for (int s = 0; s < P.S; ++s) {
          const double sv = d.method < 3 ? cs[ci + s] : (s == sa ? cs[ci] : (s == sb ? cs[ci + 1] : bs[s]));
          if (best < sv) best = sv;
        }
        mv[K - 1] = best;
      }
    d.ctot[c] = d.obj.combine(cost, total_time, mv, 1, nullptr);
  }
};
// one thread per problem: the base point's total (before the first iteration: f = objective(x0); after the last: the outputs)
struct DfoBaseTotalFn {
  DfoBatch d;
  int start;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi;
    DfoProb& P = d.prob[p];
    const double* x = d.x + P.x0;
    double total_time = 0.0;
    for (int s = 0; s < P.S; ++s) total_time = total_time + x[s];
    double cost;
    if (d.method < 3) {
      cost = d.bcost[p];
    } else {
      double tot = 0.0;
      for (int it = 0; it < P.S * TG_D; ++it) tot += d.bpart[(size_t)P.s0 * 4 + it];
      cost = 0.5 * tot;
    }
    double mv[4] = {0.0, 0.0, 0.0, 0.0};
    if (d.obj.use_soft)
      for (int K = 1; K <= 4; ++K) {
        bool need = false;
        for (int q = 0; q < d.obj.ncon; ++q) need = need || d.obj.con_deriv[q] == K;
        if (!need) continue;
        const double* bs = d.bsv + (size_t)(K - 1) * d.totS + P.s0;
        double best = 0.0;
        for (int s = 0; s < P.S; ++s)
          if (best < bs[s]) best = bs[s];
        mv[K - 1] = best;
      }
    const double tot = d.obj.combine(cost, total_time, mv, 1, d.bparts + 3 * (size_t)p);
    d.btot[p] = tot;
    if (start) {
      P.f = tot;
      if (!P.done) dfo_enlist(d, p, 0);
    }
  }
};
// one thread per running problem: the first strictly smallest total, then accept (ftol_rel -> 3) or halve the steps
// (xtol_rel -> 4); maxeval -> 5 once max_iterations iterations have run
struct DfoAdvanceFn {
  DfoBatch d;
  const int* prob_list;
  int nbuf;
  TG_HD void operator()(size_t k) const {
    const int p = prob_list ? prob_list[k] : (int)k;
    DfoProb& P = d.prob[p];
    if (P.done) return;
    ++P.iterations;
    const double* tot = d.ctot + P.c0;
    int kb = 0;
    for (int q = 1; q < 2 * P.n; ++q)
      if (tot[q] < tot[kb]) kb = q;
    double* x = d.x + P.x0;
    double* step = d.step + P.x0;
    if (tot[kb] < P.f) {
      const double f_old = P.f;
      P.f = tot[kb];
      const int dir = kb >= P.n ? 1 : 0, i = kb - dir * P.n;
      x[i] = dir ? dfo_dn(x[i], step[i], d.lo[P.x0 + i]) : dfo_up(x[i], step[i], d.hi[P.x0 + i]);
      if (fabs(f_old - P.f) <= d.f_rel * fabs(P.f)) {
        P.code = 3;
        P.done = 1;
      }
    } else {
      bool small = true;
      for (int i = 0; i < P.n; ++i) {
        step[i] *= 0.5;
        if (!(step[i] <= d.x_rel * fabs(x[i]))) small = false;
      }
      if (small) {
        P.code = 4;
        P.done = 1;
      }
    }
    if (!P.done && P.iterations >= d.max_iter) P.done = 1;
    if (!P.done) dfo_enlist(d, p, nbuf);
  }
};
// outputs: the final times (one thread per segment) and the vertex values with the free slots at their final variables (one
// thread per vertex, methods 3, 4)
struct DfoTimesOutFn {
  DfoBatch d;
  double* times;
  TG_HD void operator()(size_t gs) const {
    const int p = d.b.prob_of_seg[gs];
    times[gs] = d.x[(size_t)d.prob[p].x0 + (gs - (size_t)d.prob[p].s0)];
  }
};
struct DfoVvalOutFn {
  DfoBatch d;
  double* vval;
  TG_HD void operator()(size_t gv) const {
    const int p = d.b.prob_of_vtx[gv];
    const DfoProb& P = d.prob[p];
    const int v = (int)gv - (P.s0 + p);
    const uint32_t m = d.b.vmask[gv];
    const int j0 = d.b.vfree[P.s0 + 2 * p + v];
    for (int k = 0; k < TG_HALF; ++k)
      for (int dim = 0; dim < TG_D; ++dim) {
        const size_t o = (gv * TG_HALF + k) * TG_D + dim;
        vval[o] = ((m >> k) & 1u) ? d.b.vval[o] : d.x[(size_t)P.x0 + P.S + (size_t)dim * P.n_free + j0 + free_rank(m, k)];
      }
  }
};

}  // namespace tg

#endif  // TG_DFO_CUH_
