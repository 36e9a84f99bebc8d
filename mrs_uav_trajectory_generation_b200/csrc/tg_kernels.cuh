// tg_kernels.cuh -- the per-thread / per-warp work items of every kernel, as TG_HD functors over raw device
// pointers.  cuda_backend.cu wraps them in __global__ kernels; tests/host_emu runs the same functors in loops.
//
// Ragged batch layout (all arrays in HBM, struct-of-arrays, problem p owns contiguous slices):
//   seg_off[B+1]             first segment of problem p; vertices start at seg_off[p] + p (V = S + 1)
//   wp[totV][4], stop[totV]  waypoints x y z heading, stop_at flags
//   vmask[totV], vval[totV][5][4], vfree[totV + B]   vertex constraints and free-unknown index (V+1 per problem)
//   times/xeval/x/g/d[totS], ix[totS], hist_s/hist_y[mf][totS], coef[totS][4][10], recs[totS*{1,3}][186], maxima[totS][9]
//   costs[totV]              cost of solve instance (p, n): n = 0 base, n >= 1 perturbed segment n-1
#ifndef TG_KERNELS_CUH_
#define TG_KERNELS_CUH_

#include "tg_common.cuh"
#include "tg_bound.cuh"
#include "tg_plis.cuh"
#include "tg_node.cuh"
#include "tg_poly.cuh"
#include "tg_segment.cuh"
#include "tg_solve.cuh"
#include "tg_solve_octet.cuh"
#include "tg_solve_thread.cuh"

#if defined(__CUDA_ARCH__)
#define TG_ATOMIC_MAX(p, v) atomicMax((p), (v))
#define TG_ATOMIC_ADD(p, v) atomicAdd((p), (v))
#define TG_ATOMIC_ADD_RET(p, v) atomicAdd((p), (v))
#elif defined(__CUDACC__)
// host pass of nvcc over TG_HD code: never executed (the library has no CPU path)
#define TG_ATOMIC_MAX(p, v) ((void)0)
#define TG_ATOMIC_ADD(p, v) ((void)0)
#define TG_ATOMIC_ADD_RET(p, v) (0)
#else
// tests/host_emu only (g++): the emulator runs work items on several host threads
static inline void tg_host_atomic_max(int* p, int v) {
  int cur = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (cur < v && !__atomic_compare_exchange_n(p, &cur, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
}
#define TG_ATOMIC_MAX(p, v) tg_host_atomic_max((p), (v))
#define TG_ATOMIC_ADD(p, v) __atomic_fetch_add((p), (v), __ATOMIC_RELAXED)
#define TG_ATOMIC_ADD_RET(p, v) __atomic_fetch_add((p), (v), __ATOMIC_RELAXED)
#endif

namespace tg {

enum FindStatus { kFindOk = 0, kFindNloptRejected = 1, kFindTooLong = 2, kFindTooShort = 3, kFindSampleFail = 4, kFindEmptyPath = 5, kFindNotFinite = 6 };

// per-problem record of one findTrajectory pass (device side)
struct ProbState {
  int status;          // FindStatus
  int nlopt_code;
  int n_evals;
  int n_scale_passes;
  int scale_done;
  int n_samples;
  int sample_cap;
  int safe;
  int next_V;          // vertex count after subdivision (0: no re-solve needed)
  int n_grads;         // Mellinger evaluations whose gradient was computed (PLIS consumes every one: == n_evals)
  double final_cost;   // OptimizationInfo::cost_trajectory: the cost at the last point the optimiser evaluated
  double cost;         // cost of the final linear solve
  double baca_total;
  double max_dev;
};

struct BatchPtrs {
  int B, totS, totV, r;
  const int* seg_off;
  const int* prob_of_vtx;
  const int* prob_of_seg;
  const double* wp;
  const uint8_t* stop;
  const double* init14;  // [B][14] or null
  uint8_t* vmask;
  double* vval;
  int* vfree;
  int* np;
  int* hbw;
  int* fmax;             // [B] largest number of free derivatives at one vertex
  int* stats;            // [16]: [0] max solve workspace doubles, [1] problems still to scale, [2] max octet-solve workspace doubles, [3] max np, [4] max S,
                         // [5] root findings executed, [6] problems the octet routine cannot take, [7] problems whose optimiser still runs,
                         // [8] problems the thread-per-instance solve cannot take
  double *times, *baca, *xeval, *x, *g, *d, *hist_s, *hist_y;
  PlisScalars* opt;      // [B] optimiser state (tg_plis.cuh)
  int* ix;               // [totS] PLIS bound codes / active set
  // work lists of the problems whose optimiser still runs, appended by PlisBeginFn / PlisAdvanceFn for the NEXT evaluation
  // (two alternating buffers; lengths in stats[9 + 3 * buf .. 11 + 3 * buf]: problems, vertices = solve instances, segments)
  int* act_prob[2];
  int* act_vtx[2];
  int* act_seg[2];
  double* recs;
  double* costs;
  double* coef;
  double* maxima;
  ProbState* ps;
  double* xs;            // [instances][xstride] solutions of the reduced systems (solve kernels -> CoefCostFn)
  double* part;          // [instances][4 * smax] partial costs
  int xstride, smax;
};

TG_HD int vtx_off(const BatchPtrs& b, int p) { return b.seg_off[p] + p; }

// ---- 1. vertex recipe + unknown indexing: one thread per problem ----------------------------------------------
struct PrepareFn {
  BatchPtrs b;
  int from_waypoints;  // 1: node recipe from wp/stop/init ; 0: masks/values supplied by the caller
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0, V = S + 1, v0 = s0 + p;
    int hbw = 0, np;
    if (from_waypoints)
      np = build_vertices(V, b.wp + 4 * (size_t)v0, b.stop ? b.stop + v0 : nullptr, b.init14 ? b.init14 + 14 * (size_t)p : nullptr, b.r,
                          b.vmask + v0, b.vval + (size_t)v0 * TG_HALF * TG_D, b.vfree + v0 + p, &hbw);
    else
      np = index_vertices(V, b.vmask + v0, b.vfree + v0 + p, &hbw);
    b.np[p] = np;
    b.hbw[p] = hbw;
    int fmax = 0;
    for (int v = 0; v < V; ++v) {
      const uint32_t m = b.vmask[v0 + v];
      fmax = imax(fmax, TG_HALF - (int)((m & 1u) + ((m >> 1) & 1u) + ((m >> 2) & 1u) + ((m >> 3) & 1u) + ((m >> 4) & 1u)));
    }
    b.fmax[p] = fmax;
    if (fmax > kThrB || np == 0) TG_ATOMIC_ADD(&b.stats[8], 1);
    TG_ATOMIC_MAX(&b.stats[0], solve_ws_doubles(S, np, hbw));
    TG_ATOMIC_MAX(&b.stats[3], np);
    TG_ATOMIC_MAX(&b.stats[4], S);
    if (hbw == kOctHbw && np >= kOctMinNp) TG_ATOMIC_MAX(&b.stats[2], octet_ws_doubles(S, np));
    else TG_ATOMIC_ADD(&b.stats[6], 1);  // problems the octet routine cannot take
    ProbState& ps = b.ps[p];
    ps.status = kFindOk;
    ps.nlopt_code = 1;
    ps.n_evals = 0;
    ps.n_grads = 0;
    ps.n_scale_passes = 0;
    ps.scale_done = 0;
    ps.n_samples = 0;
    ps.sample_cap = 0;
    ps.safe = 0;
    ps.next_V = 0;
    ps.final_cost = 0.0;
    ps.cost = 0.0;
    ps.baca_total = 0.0;
    ps.max_dev = 0.0;
  }
};

// ---- 2. initial segment times: one thread per segment, then one per problem for the Baca total ------------------
struct TimesFn {
  BatchPtrs b;
  double L[9];
  TG_HD void operator()(size_t gs) const {
    const int p = b.prob_of_seg[gs];
    const int s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0, i = (int)gs - s0, v0 = s0 + p;
    const double* vpos = b.vval + (size_t)v0 * TG_HALF * TG_D;
    const int stride = TG_HALF * TG_D;
    b.times[gs] = segment_time_euclidean(vpos + (size_t)i * stride, vpos + (size_t)(i + 1) * stride, L);
    b.baca[gs] = segment_time_baca(vpos, stride, i, S + 1, L);
  }
};
struct BacaTotalFn {
  BatchPtrs b;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0;
    double tot = 0.0;
    for (int i = 0; i < S; ++i) tot = tot + b.baca[s0 + i];  // node.cpp:1053-1056
    b.ps[p].baca_total = tot;
  }
};

// ---- 3. per-segment records ------------------------------------------------------------------------------------------
// base: one record per segment at times[]; Mellinger: three per segment at xeval, xeval+0.1, max(lb, xeval-corr)
struct SetupBaseFn {
  BatchPtrs b;
  const double* T;
  TG_HD void operator()(size_t gs) const { setup_segment_record(T[gs], b.r, b.recs + gs * TG_REC_SIZE); }
};
// Two launches (tg_segment.cuh, "two stages"): SetupMellingerFn<0> over the records writes Q, Dinv, X; SetupMellingerFn<1>
// over (record, row) writes the ten rows of H.
template <int STAGE>  // 0: heads, one item per record; 1: rows of H, ten items per record
struct SetupMellingerFn {
  BatchPtrs b;
  const int* seg_list;  // null: item = 3 * segment + which over all segments; else over the listed segments
  static constexpr int stage = STAGE;
#ifndef TG_SETUP_ROW_BLOCKS
#define TG_SETUP_ROW_BLOCKS 8
#endif
  static constexpr int kMinBlocks = STAGE ? TG_SETUP_ROW_BLOCKS : 2;  // the row stage is small: resident warps instead of registers
  TG_HD void operator()(size_t item00) const {
    const size_t item0 = stage ? item00 / TG_N : item00;
    const size_t k = item0 / 3;
    const int which = (int)(item0 - k * 3);
    const size_t gs = seg_list ? (size_t)seg_list[k] : k;
    const size_t item = gs * 3 + which;
    const int p = b.prob_of_seg[gs];
    double T = stage ? 0.0 : b.xeval[gs];  // issued next to the problem lookup, not behind the two early-outs that depend on it
    if (b.opt[p].done) return;
    const int S = b.seg_off[p + 1] - b.seg_off[p];
    if (S == 1 && which != 0) return;
    double* rec = b.recs + item * TG_REC_SIZE;
    if (stage) {
      setup_record_hrow(b.r, rec, (int)(item00 - item0 * TG_N));
      return;
    }
    if (which == 1) {
      T = T + 0.1;
      T = dmax(kTimeLowerBound, T);
    } else if (which == 2) {
      const double corr = 0.1 / ((double)S - 1.0);  // nl_impl.h:288
      T = T - corr;
      T = dmax(kTimeLowerBound, T);
    }
    setup_record_head(T, b.r, rec);
  }
};

// ---- 4. warp solves ----------------------------------------------------------------------------------------------------
struct SolveProblemDesc {
  BatchPtrs b;
  // 0: instance = problem, base times, one record per segment (final solve, linear batch)
  // 1: instance = vertex index = (problem, variant), every variant of every running problem (one Mellinger evaluation:
  //    variant 0 the point itself, variant n >= 1 the point perturbed along segment n-1; three records per segment)
  int mellinger;
  double* dp_out; // optional [sum np][4]-> per problem offset by 4*vfree base (only base mode), may be null
  const int* dp_off;
  TG_HD bool instance(size_t inst, SolveInst& I) const {
    int p, n;
    if (mellinger == 1) {
      p = b.prob_of_vtx[inst];
      n = (int)inst - vtx_off(b, p);
      if (b.opt[p].done) return false;
    } else {
      p = (int)inst;
      n = 0;
    }
    const int s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0, v0 = s0 + p;
    if (mellinger && S == 1 && n > 0) return false;
    I.S = S;
    I.np = b.np[p];
    I.hbw = b.hbw[p];
    I.fmax = b.fmax[p];
    I.variant = n;
    I.rec_stride = mellinger ? 3 : 1;
    I.r = b.r;
    I.vmask = b.vmask + v0;
    I.vfree = b.vfree + v0 + p;
    I.vval = b.vval + (size_t)v0 * TG_HALF * TG_D;
    I.recs = b.recs + (size_t)s0 * I.rec_stride * TG_REC_SIZE;
    I.coef_out = (n == 0) ? b.coef + (size_t)s0 * TG_D * TG_N : nullptr;
    I.cost_out = mellinger ? b.costs + v0 + n : &b.ps[p].cost;
    I.dp_out = (dp_out && !mellinger) ? dp_out + (size_t)TG_D * dp_off[p] : nullptr;
    // the solution slot of (problem, variant) is the same whichever way the instance was numbered
    I.x_out = b.xs ? b.xs + (mellinger ? (size_t)(v0 + n) : inst) * (size_t)b.xstride : nullptr;
    return true;
  }
};
// the same instances taken from a work list (instance k of the launch = list[k])
struct SolveProblemListDesc {
  SolveProblemDesc d;
  const int* list;
  TG_HD bool instance(size_t k, SolveInst& I) const { return d.instance((size_t)list[k], I); }
};
// time-vector sweep (BASELINE config 5): K candidates for ONE problem, records laid out [candidate][segment]
struct SolveSweepDesc {
  BatchPtrs b;  // a batch holding the single problem
  const double* recs;
  double* costs;
  double* coefs = nullptr;  // optional [K][S][4][10]
  TG_HD bool instance(size_t k, SolveInst& I) const {
    const int S = b.seg_off[1] - b.seg_off[0];
    I.S = S;
    I.np = b.np[0];
    I.hbw = b.hbw[0];
    I.fmax = b.fmax[0];
    I.variant = 0;
    I.rec_stride = 1;
    I.r = b.r;
    I.vmask = b.vmask;
    I.vfree = b.vfree;
    I.vval = b.vval;
    I.recs = recs + k * (size_t)S * TG_REC_SIZE;
    I.coef_out = coefs ? coefs + k * (size_t)S * TG_D * TG_N : nullptr;
    I.cost_out = costs + k;
    I.dp_out = nullptr;
    I.x_out = b.xs ? b.xs + k * (size_t)b.xstride : nullptr;
    return true;
  }
};
struct SetupSweepFn {
  int S, r;
  const double* cand;  // [K][S]
  double* recs;
  TG_HD void operator()(size_t item) const { setup_segment_record(cand[item], r, recs + item * TG_REC_SIZE); }
};

// objective functions of the time-allocation methods 0/1/3/4 (nl_impl.h:567-722), K candidates x[K][nvar] of one problem:
// records and contiguous segment times from the first S entries of every candidate
struct SetupObjFn {
  int S, r, nvar;
  const double* x;
  double* recs;   // [K][S]
  double* times;  // [K][S]
  TG_HD void operator()(size_t item) const {
    const size_t k = item / (size_t)S;
    const int s = (int)(item - k * (size_t)S);
    const double T = x[k * (size_t)nvar + s];
    times[item] = T;
    setup_segment_record(T, r, recs + item * TG_REC_SIZE);
  }
};
// setFreeConstraints (lin_impl.h:513-522): the free derivatives of candidate k, x[k][S + d * n_free + j], into the solution
// layout [j][d] that CoefCostFn reads
struct FillFreeFn {
  int S, nvar, n_free, xstride;
  const double* x;
  double* xs;
  TG_HD void operator()(size_t item) const {
    const size_t k = item / (size_t)(n_free * TG_D);
    const int rem = (int)(item - k * (size_t)(n_free * TG_D)), j = rem / TG_D, d = rem - j * TG_D;
    xs[k * (size_t)xstride + j * TG_D + d] = x[k * (size_t)nvar + S + (size_t)d * n_free + j];
  }
};
// total = cost_trajectory + cost_time + cost_soft_constraints (nl_impl.h:613, 721); soft constraints as
// min(maximum_cost, exp(relative_violation * weight)) summed in constraint order (nl_impl.h:740-762), the maxima of the
// distinct derivatives precomputed per candidate (maxval[derivative - 1][k])
struct ObjTerms {
  int method, ncon;
  double time_penalty, soft_weight;
  int use_soft;
  int con_deriv[16];
  double con_value[16];
  // maxval[(derivative - 1) * stride] = computeMaximumOfMagnitude(derivative).value of the candidate; parts optional [3]
  TG_HD double combine(double cost_traj, double total_time, const double* maxval, size_t stride, double* parts) const {
    const double cost_time = (method == 1 || method == 4) ? total_time * time_penalty : total_time * total_time * time_penalty;
    double cost_con = 0.0;
    if (use_soft)
      for (int c = 0; c < ncon; ++c) {
        const double abs_violation = maxval[(size_t)(con_deriv[c] - 1) * stride] - con_value[c];
        const double relative_violation = abs_violation / con_value[c];
        cost_con = cost_con + dmin(1.0e12, tgdm::dexp(relative_violation * soft_weight));
      }
    if (parts) {
      parts[0] = cost_traj;
      parts[1] = cost_time;
      parts[2] = cost_con;
    }
    return cost_traj + cost_time + cost_con;
  }
};
struct ObjCombineFn {
  int S;
  ObjTerms terms;
  const double* times;   // [K][S]
  const double* costs;   // [K] trajectory cost
  const double* maxval;  // [4][K]
  size_t K;
  double* total;
  double* parts;  // optional [K][3]
  TG_HD void operator()(size_t k) const {
    double total_time = 0.0;
    for (int s = 0; s < S; ++s) total_time = total_time + times[k * (size_t)S + s];
    total[k] = terms.combine(costs[k], total_time, maxval + k, K, parts ? parts + 3 * k : nullptr);
  }
};

// ---- 4b. coefficients and cost from the solutions of the reduced systems ---------------------------------------------
// One thread per (instance, segment, dimension): c = A^-1 [derivatives of vertex s ; vertex s+1] (lin_impl.h:271-280) and
// the partial cost (c^T Q) c (lin_impl.h:135-137); then one thread per instance adds the partials in (segment, dimension)
// order (lin_impl.h:131-140).  Same sums as the in-kernel versions (tg_solve.cuh phase 4-6).
template <int R>
TG_HD double cost_partial(const double (&c)[TG_N], const double* __restrict__ Qg) {
  constexpr int nq = TG_N - R;
  double qt[36];  // the packed Q block of the record (tg_qtri), fetched with 16-byte loads
#pragma unroll
  for (int e = 0; e < 36; e += 2) {
    const Dbl2 t = *reinterpret_cast<const Dbl2*>(Qg + e);
    qt[e] = t.x;
    qt[e + 1] = t.y;
  }
  double partial = 0.0;
#pragma unroll
  for (int b = 0; b < nq; ++b) {
    double sum = c[R] * qt[tg_qsym(0, b)];
#pragma unroll
    for (int k = 1; k < nq; ++k) sum = sum + c[R + k] * qt[tg_qsym(k, b)];
    partial = (b == 0) ? sum * c[R + b] : partial + sum * c[R + b];
  }
  return partial;
}
TG_HD double cost_partial_rec(int r, const double (&c)[TG_N], const double* __restrict__ rec) {
  const double* Q = rec + TG_REC_Q;
  return (r == 2) ? cost_partial<2>(c, Q) : ((r == 3) ? cost_partial<3>(c, Q) : cost_partial<4>(c, Q));
}
// c = A^-1 nd from the segment's record, nd = the ten end-point derivatives of one dimension (0..4 at the start, 0..4 at the end)
TG_HD void coef_from_endpoints(const double* __restrict__ rec, const double (&nd)[TG_N], double (&c)[TG_N]) {
  c[0] = 1.0 * nd[0];
  c[1] = 1.0 * nd[1];
  c[2] = (1.0 / 2.0) * nd[2];
  c[3] = (1.0 / 6.0) * nd[3];
  c[4] = (1.0 / 24.0) * nd[4];
  double blk[50];  // Dinv (25) then X (25): the first 400 bytes of the record, fetched with 16-byte loads
#pragma unroll
  for (int e = 0; e < 50; e += 2) {
    const Dbl2 t = *reinterpret_cast<const Dbl2*>(rec + e);
    blk[e] = t.x;
    blk[e + 1] = t.y;
  }
#pragma unroll
  for (int a = 0; a < TG_HALF; ++a) {
    double acc = blk[TG_REC_X + a * 5] * nd[0];
#pragma unroll
    for (int k = 1; k < 5; ++k) acc = acc + blk[TG_REC_X + a * 5 + k] * nd[k];
#pragma unroll
    for (int k = 0; k < 5; ++k) acc = acc + blk[TG_REC_DINV + a * 5 + k] * nd[5 + k];
    c[TG_HALF + a] = acc;
  }
}
template <class D>
struct CoefCostFn {
  D desc;
  int per_inst;   // 4 * smax: stride of `part` per instance
  double* part;   // [instances][per_inst]
  size_t inst0;   // this launch covers instances inst0 .. with per_items (<= per_inst) items each: 4 * (largest S among them)
  int per_items;
  TG_HD void operator()(size_t item0) const {
    const size_t inst = inst0 + item0 / (size_t)per_items;
    const int it = (int)(item0 % (size_t)per_items);
    run(inst, it);
  }
  TG_HD void run(size_t inst, int it) const {
    SolveInst I;
    if (!desc.instance(inst, I)) return;
    if (it >= I.S * TG_D) return;
    run_instance(I, inst * (size_t)per_inst + it, it);
  }
  // item `it` = (segment, dimension) of the prepared instance I; `item` = its slot in `part`
  TG_HD void run_instance(const SolveInst& I, size_t item, int it) const {
    const int s = it >> 2, d = it & 3;
    const double* rec = solve_rec(I, s);
    double nd[TG_N], c[TG_N];
#pragma unroll
    for (int k = 0; k < TG_N; ++k) {
      const int v = s + (k >= TG_HALF ? 1 : 0), sl = k - (k >= TG_HALF ? TG_HALF : 0);
      const uint32_t m = I.vmask[v];
      nd[k] = ((m >> sl) & 1u) ? I.vval[((size_t)v * TG_HALF + sl) * TG_D + d] : I.x_out[(size_t)(I.vfree[v] + free_rank(m, sl)) * 4 + d];
    }
    coef_from_endpoints(rec, nd, c);
    if (I.coef_out) {
#pragma unroll
      for (int a = 0; a < TG_N; a += 2) store2(I.coef_out + it * TG_N + a, c[a], c[a + 1]);
    }
    if (I.cost_out) part[item] = cost_partial_rec(I.r, c, rec);
  }
};
// The same for all points of a Mellinger evaluation (SolveProblemDesc mode 1), organised by PROBLEM: 128 consecutive items
// (one CTA of k_for_each) belong to one problem and share its (variant, segment, dimension) items among them, so that a
// problem whose optimiser has finished costs one flag test per thread instead of a scan of all its items -- late
// evaluations run for a few per cent of the problems.
struct CoefCostGradFn {
#ifndef TG_COEF_MIN_BLOCKS
#define TG_COEF_MIN_BLOCKS 5
#endif
  static constexpr int kMinBlocks = TG_COEF_MIN_BLOCKS;  // 96 registers: measured 20.3 ms per step against 23.1 at 158
  CoefCostFn<SolveProblemDesc> f;
  int p0;  // first problem of this launch
  const int* prob_list;  // or the listed problems
  TG_HD void operator()(size_t item0) const {
    const BatchPtrs& b = f.desc.b;
    const int p = prob_list ? prob_list[item0 >> 7] : p0 + (int)(item0 >> 7), t = (int)(item0 & 127);
    if (b.opt[p].done) return;
    const int s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0, v0 = s0 + p;
    const int per = S * TG_D, total = (S == 1) ? per : (S + 1) * per;  // variants 0..S
    // the instance of (problem, variant) built from what this thread already holds: SolveProblemDesc::instance would walk
    // prob_of_vtx -> seg_off -> opt again for every item, three dependent loads in front of 420 flop (ncu: 13.7 stall cycles per
    // issued instruction on the long scoreboard)
    SolveInst I;
    I.S = S;
    I.np = 0;  // np, hbw, fmax: not read by the coefficient stage
    I.hbw = 0;
    I.fmax = 0;
    I.rec_stride = 3;
    I.r = b.r;
    I.vmask = b.vmask + v0;
    I.vfree = b.vfree + v0 + p;
    I.vval = b.vval + (size_t)v0 * TG_HALF * TG_D;
    I.recs = b.recs + (size_t)s0 * 3 * TG_REC_SIZE;
    I.dp_out = nullptr;
    for (int k = t; k < total; k += 128) {
      const int n = k / per, it = k - n * per;
      I.variant = n;
      I.coef_out = (n == 0) ? b.coef + (size_t)s0 * TG_D * TG_N : nullptr;
      I.cost_out = b.costs + v0 + n;
      I.x_out = b.xs + (size_t)(v0 + n) * (size_t)b.xstride;
      f.run_instance(I, (size_t)(v0 + n) * (size_t)f.per_inst + it, it);
    }
  }
};
template <class D>
struct CostSumFn {
  D desc;
  int per_inst;
  const double* part;
  const int* inst_list = nullptr;  // null: every instance; else the listed ones
  TG_HD void operator()(size_t k) const {
    const size_t inst = inst_list ? (size_t)inst_list[k] : k;
    SolveInst I;
    if (!desc.instance(inst, I)) return;
    if (!I.cost_out) return;
    const double* pp = part + inst * (size_t)per_inst;
    double total = 0.0;
    for (int it = 0; it < I.S * TG_D; ++it) total += pp[it];
    *I.cost_out = 0.5 * total;
  }
};

// ---- 5. PLIS state machine (tg_plis.cuh): one thread per problem ---------------------------------------------------------
TG_HD PlisVectors plis_vectors(const BatchPtrs& b, int p) {
  PlisVectors v;
  const int s0 = b.seg_off[p];
  v.x = b.x + s0;
  v.gf = b.g + s0;
  v.s = b.d + s0;
  v.xeval = b.xeval + s0;
  v.xo = b.hist_s + s0;
  v.go = b.hist_y + s0;
  v.ix = b.ix + s0;
  v.hstride = (size_t)b.totS;
  return v;
}
// a running problem enters the work lists of the next evaluation (buffer `buf`)
TG_HD void plis_enlist(const BatchPtrs& b, int p, int buf) {
  const int s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0, v0 = s0 + p;
  int* cnt = b.stats + 9 + 3 * buf;
  const int jp = TG_ATOMIC_ADD_RET(&cnt[0], 1);
  b.act_prob[buf][jp] = p;
  const int jv = TG_ATOMIC_ADD_RET(&cnt[1], S + 1);
  for (int n = 0; n <= S; ++n) b.act_vtx[buf][jv + n] = v0 + n;
  const int js = TG_ATOMIC_ADD_RET(&cnt[2], S);
  for (int i = 0; i < S; ++i) b.act_seg[buf][js + i] = s0 + i;
}
struct PlisBeginFn {
  BatchPtrs b;
  int max_evals;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0;
    if (plis_begin(S, b.opt[p], plis_vectors(b, p), b.times + s0, max_evals)) plis_enlist(b, p, 0);
  }
};
// after the S+1 solves of one evaluation; stats[7] counts the problems that still run
struct PlisAdvanceFn {
  BatchPtrs b;
  int max_evals;
  double f_rel, x_rel;
  const int* prob_list;  // null: every problem; else the listed ones
  int next_buf;          // work-list buffer of the next evaluation
  TG_HD void operator()(size_t k) const {
    const int p = prob_list ? prob_list[k] : (int)k, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0;
    PlisScalars& st = b.opt[p];
    if (st.done) return;
    plis_advance(S, st, plis_vectors(b, p), b.costs + vtx_off(b, p), max_evals, f_rel, x_rel, -1.0);
    if (!st.done) {
      TG_ATOMIC_ADD(&b.stats[7], 1);
      plis_enlist(b, p, next_buf);
    }
  }
};
// after the loop: times <- last evaluated point (what poly_opt_ holds when nlopt returns, nl_impl.h:210-215)
struct PlisFinishFn {
  BatchPtrs b;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0;
    for (int i = 0; i < S; ++i) b.times[s0 + i] = b.xeval[s0 + i];
    ProbState& ps = b.ps[p];
    const PlisScalars& st = b.opt[p];
    ps.nlopt_code = st.code;
    ps.n_evals = st.n_evals;
    ps.n_grads = st.n_evals;
    ps.final_cost = st.f_last;
    if (st.n_evals == 0) ps.scale_done = 1;  // start point outside the bounds: nlopt throws before any evaluation, no scaling (nl_impl.h:192-194)
    const int code = ps.nlopt_code;
    if (!((code >= 1 && code != 6) || code == -1)) ps.status = kFindNloptRejected;  // node.cpp:1138-1149
  }
};

// ---- 6. extrema + time scaling ------------------------------------------------------------------------------------------------
template <int Q>
struct ExtremaFn {  // one thread per segment for quantity Q (one launch per quantity: uniform polynomial degree per kernel)
  BatchPtrs b;
  int* shift_count;  // optional counter of fixed-shift stages (flop accounting)
  static constexpr int kScratch = JtScratch<QuantityDegree<Q>::value>::kShared;  // doubles of strided scratch per thread
  TG_HD void operator()(size_t gs, double* scratch, int stride) const {
    const int p = b.prob_of_seg[gs];
    if (b.ps[p].scale_done) return;
    int shifts = 0;
    b.maxima[gs * 9 + Q] = segment_max_impl<Q>(b.coef + gs * TG_D * TG_N, b.times[gs], scratch, stride, &shifts);
    if (shift_count) TG_ATOMIC_ADD(shift_count, shifts);
  }
};
// work list of the segments whose maxima must be recomputed after a scaling pass: the problem is still being scaled
// and the segment was stretched by a factor other than exactly 1 (a factor of 1 leaves every coefficient bit-identical,
// eth/polynomial.cpp:218-224, so its zeros and maxima are unchanged)
struct ExtremaWorkFn {
  const int* prob_of_seg;
  const ProbState* ps;
  const uint8_t* changed;  // [totS] written by ScaleFn
  uint8_t* flag;           // [totS] 1: recompute (the ordered work list is built from the flags by the backend's select)
  TG_HD void operator()(size_t gs) const { flag[gs] = (!ps[prob_of_seg[gs]].scale_done && changed[gs]) ? 1 : 0; }
};

// Certificates for the global check (tg_bound.cuh): one thread per entry of the changed-segment work list.  A quantity
// whose Bernstein bound already passes the 1.001 x limit test gets the bound stored and flagged; the others are appended
// to the per-quantity work lists for exact root finding.
struct ExtremaBoundFn {
  const double* coef;
  const double* times;
  double* maxima;
  uint8_t* is_bound;   // [totS * 9]
  const int* work;     // changed segments
  const int* n_work;   // device count
  uint8_t* need;       // [9][list_stride] 1: (segment, quantity) needs exact root finding
  int list_stride;
  double L[9];
  double tol;
  TG_HD void operator()(size_t item) const {
    if (item >= (size_t)*n_work) return;
    const size_t gs = (size_t)work[item];
    for (int q = 0; q < 9; ++q) {
      // a value v with v / L <= 1 + tol passes the check (eth/trajectory.cpp:676-681); thr is such a value with a margin
      const double thr = L[limit_index(q)] * (1.0 + tol) * (1.0 - 1e-12);
      const bool passes = (thr / L[limit_index(q)] <= 1.0 + tol) && certify_quantity_le(coef + gs * TG_D * TG_N, times[gs], q, thr);
      if (passes) {
        maxima[gs * 9 + q] = thr;
        is_bound[gs * 9 + q] = 1;
      } else {
        is_bound[gs * 9 + q] = 0;
        need[(size_t)q * list_stride + gs] = 1;
      }
    }
  }
};
// ---- pruned maxima for the per-segment stretch factor ----------------------------------------------------------------
// The stretch factor of a segment (eth/trajectory.cpp:640-655) is s = max(1, V, sqrt(A), cbrt(J)) over the nine maxima:
// only the largest transformed ratio matters.  With rigorous upper bounds u_q (tg_bound.cuh) and r_q = g_q(u_q / L_q)
// (g = identity / sqrt / cbrt, inflated by 1e-9 so that cbrt needs no monotonicity at the ulp level):
//   A. r_max <= 1  => no quantity can exceed its limit, s = 1 exactly, nothing to compute;
//      otherwise the quantity q* with the largest r is computed exactly (Jenkins-Traub);
//   C. M = max(1, g(exact ratio of q*)); every q with r_q <= M cannot raise the maximum and is dropped (its slot gets 0,
//      which never binds); the others are computed exactly.
// s is then evaluated by the reference's expression over the exact values -- bit-identical to evaluating it over all
// nine (the dropped transformed values are <= M <= s).
TG_HD double prune_transform(int q, double ratio) {
  const int d = q % 3;  // 0 velocity, 1 acceleration, 2 jerk
  return d == 0 ? ratio : (d == 1 ? dsqrt(ratio) : tgdm::dcbrt(ratio));
}
struct ExtremaPruneAFn {
  BatchPtrs b;
  double L[9];
  double* rq;          // [totS][9] transformed bounds
  uint8_t* qstar;      // [totS] quantity computed first, 0xff: none needed, 0xfe: all nine (bounds unusable)
  uint8_t* need;       // [9][list_stride] 1: (segment, quantity) needs exact root finding
  int list_stride;
  TG_HD void operator()(size_t gs) const {
    const double* coef = b.coef + gs * TG_D * TG_N;
    const double T = b.times[gs];
    double bnd[9];
    segment_bounds(coef, T, bnd);
    double rmax = -1.0;
    int qs = -1;
    bool usable = true;
    for (int q = 0; q < 9; ++q) {
      const double lim = L[limit_index(q)];
      const double ratio = bnd[q] / lim;
      double r = prune_transform(q, ratio) * (1.0 + 1e-9);
      if (!(r >= 0.0) || tgdm::disinf(r) || !(lim > 0.0)) usable = false;  // NaN, non-positive limits, overflow: no pruning here
      // a quantity that provably stays within its limit can never raise s above 1 (s = max(1, ...)): drop it
      if (usable && (r <= 1.0 || certify_quantity_le(coef, T, q, lim * (1.0 - 1e-9)))) r = 0.0;
      rq[gs * 9 + q] = r;
      if (r > rmax) rmax = r;
    }
    double best = -1.0;
    if (usable && rmax > 1.0) {
      // which of the remaining quantities to compute first: the one that most likely binds, judged by curve values at five
      // points (a LOWER estimate of each maximum); the choice affects only how much is pruned afterwards, never the result
      for (int q = 0; q < 9; ++q) {
        if (!(rq[gs * 9 + q] > 1.0)) continue;
        const int group = q / 3, deriv = q % 3 + 1;
        const int d0 = (group == 0) ? 0 : (group == 1 ? 2 : 3), nd = (group == 0) ? 2 : 1;
        double lo = 0.0;
        for (int k = 0; k <= 4; ++k) {
          const double t = 0.25 * (double)k * T;
          double mag = 0.0;
          for (int dim = d0; dim < d0 + nd; ++dim) {
            const double v = poly_eval(coef + dim * TG_N, t, deriv);
            mag = mag + v * v;
          }
          if (mag > lo) lo = mag;
        }
        const double est = prune_transform(q, dsqrt(lo) / L[limit_index(q)]);
        if (est > best) { best = est; qs = q; }
      }
    }
    if (!usable) {
      qstar[gs] = 0xfe;
      for (int q = 0; q < 9; ++q) need[(size_t)q * list_stride + gs] = 1;
      return;
    }
    if (rmax <= 1.0) {
      qstar[gs] = 0xff;
      for (int q = 0; q < 9; ++q) b.maxima[gs * 9 + q] = 0.0;
      return;
    }
    qstar[gs] = (uint8_t)qs;
    need[(size_t)qs * list_stride + gs] = 1;
    // The other quantities are decided after the exact maximum of qs is known (ExtremaPruneCFn): certified below it, or
    // computed exactly in a SECOND launch -- which holds a handful of polynomials and lasts as long as the slowest of them
    // (a Jenkins-Traub launch is bound by its slowest warp: profiles/r01_final_ncu_launches_step.csv).  `best` is a LOWER
    // estimate of what that exact maximum will be; a quantity that cannot be certified even against it would not be
    // certified against the exact value in most cases either, so its root finding joins this first launch.  Marked with a
    // negative rq; computing a maximum exactly instead of certifying it never changes a stretch factor.
    const double Mlo = (1.0 < best) ? best : 1.0;
    for (int q = 0; q < 9; ++q) {
      if (q == qs || !(rq[gs * 9 + q] > Mlo)) continue;
      const int d = q % 3;
      const double lim = L[limit_index(q)];
      const double thr = (d == 0 ? lim * Mlo : (d == 1 ? lim * Mlo * Mlo : lim * Mlo * Mlo * Mlo)) * (1.0 - 1e-9);
      if (!certify_quantity_le(coef, T, q, thr)) {
        rq[gs * 9 + q] = -1.0;
        need[(size_t)q * list_stride + gs] = 1;
      }
    }
  }
};
struct ExtremaPruneCFn {
  BatchPtrs b;
  double L[9];
  const double* rq;
  const uint8_t* qstar;
  uint8_t* need;
  int list_stride;
  TG_HD void operator()(size_t gs) const {
    const int qs = qstar[gs];
    if (qs >= 9) return;
    const double m = prune_transform(qs, b.maxima[gs * 9 + qs] / L[limit_index(qs)]);
    const double M = (1.0 < m) ? m : 1.0;
    for (int q = 0; q < 9; ++q) {
      if (q == qs) continue;
      if (rq[gs * 9 + q] < 0.0) continue;  // already exact (first launch)
      bool drop = rq[gs * 9 + q] <= M;
      if (!drop) {
        // largest maximum of q whose transformed ratio stays below M: L*M, L*M^2, L*M^3 (with a margin)
        const int d = q % 3;
        const double lim = L[limit_index(q)];
        const double thr = (d == 0 ? lim * M : (d == 1 ? lim * M * M : lim * M * M * M)) * (1.0 - 1e-9);
        drop = certify_quantity_le(b.coef + gs * TG_D * TG_N, b.times[gs], q, thr);
      }
      if (drop) b.maxima[gs * 9 + q] = 0.0;
      else need[(size_t)q * list_stride + gs] = 1;
    }
  }
};

struct AccumCountsFn {  // adds the nine work-list lengths into a running total (Jenkins-Traub runs launched)
  const int* counts;
  int* total;
  TG_HD void operator()(size_t) const {
    int t = 0;
    for (int q = 0; q < 9; ++q) t += counts[q];
    *total += t;
  }
};
// Before another scaling pass reads the maxima of a problem that failed the check: its flagged entries become exact.
struct ExtremaCompleteFn {
  const int* prob_of_seg;
  const ProbState* ps;
  uint8_t* is_bound;
  uint8_t* need;
  int list_stride;
  TG_HD void operator()(size_t gs) const {
    if (ps[prob_of_seg[gs]].scale_done) return;
    for (int q = 0; q < 9; ++q)
      if (is_bound[gs * 9 + q]) {
        is_bound[gs * 9 + q] = 0;
        need[(size_t)q * list_stride + gs] = 1;
      }
  }
};

struct ScaleFn {  // one thread per segment (eth/trajectory.cpp:610-658)
  BatchPtrs b;
  double L[9];
  uint8_t* changed;  // optional [totS]: 1 when the segment was stretched by a factor other than exactly 1
  TG_HD void operator()(size_t gs) const {
    const int p = b.prob_of_seg[gs];
    if (b.ps[p].scale_done) return;
    const double s = violation_scaling(b.maxima + gs * 9, L);
    scale_segment(b.coef + gs * TG_D * TG_N, b.times + gs, s);
    if (changed) changed[gs] = (s != 1.0) ? 1 : 0;
  }
};
struct ScaleCheckFn {  // one thread per problem: the global re-check (eth/trajectory.cpp:660-689)
  BatchPtrs b;
  double L[9];
  double tol;  // 1e-3 (eth/trajectory.cpp:604)
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0;
    ProbState& ps = b.ps[p];
    if (ps.scale_done) return;
    ps.n_scale_passes += 1;
    double g[9];
    for (int q = 0; q < 9; ++q) g[q] = TG_DBL_LOWEST;
    for (int i = 0; i < S; ++i)
      for (int q = 0; q < 9; ++q) {
        const double m = b.maxima[(size_t)(s0 + i) * 9 + q];
        if (m > g[q]) g[q] = m;
      }
    if (violation_within(g, L, tol) || ps.n_scale_passes >= 20) ps.scale_done = 1;
    else TG_ATOMIC_ADD(&b.stats[1], 1);
  }
};

// ---- 7. sampling ----------------------------------------------------------------------------------------------------------------
struct SampleCapFn {
  BatchPtrs b;
  double dt;
  int* cap;  // [B]
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0;
    cap[p] = (b.ps[p].status == kFindOk) ? sample_cap(S, b.times + s0, dt) : 0;
  }
};
struct SampleWalkFn {
  BatchPtrs b;
  double dt;
  const int* smp_off;  // [B+1] exclusive scan of cap
  int* seg_idx;
  double* t_in;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0;
    ProbState& ps = b.ps[p];
    const int cap = smp_off[p + 1] - smp_off[p];
    ps.sample_cap = cap;
    if (ps.status != kFindOk) { ps.n_samples = 0; return; }
    const int m = sample_walk(S, b.times + s0, dt, cap, seg_idx + smp_off[p], t_in + smp_off[p]);
    ps.n_samples = m;
    if (m > cap) { ps.n_samples = cap; ps.status = kFindSampleFail; }
  }
};
struct SampleEvalFn {  // one thread per sample slot
  BatchPtrs b;
  const int* smp_off;
  const int* smp_prob;  // slot -> problem
  const int* seg_idx;
  const double* t_in;
  double* xyzh;  // [slots][4]
  double* full;  // [slots][19] or null
  TG_HD void operator()(size_t slot) const {
    const int p = smp_prob[slot];
    if ((int)slot - smp_off[p] >= b.ps[p].n_samples) return;
    const int gs = b.seg_off[p] + seg_idx[slot];
    sample_eval(b.coef + (size_t)gs * TG_D * TG_N, t_in[slot], xyzh + 4 * slot, full ? full + 19 * slot : nullptr);
  }
};
struct SlotProblemFn {  // fills slot -> problem map: one thread per problem
  int B;
  const int* smp_off;
  int* smp_prob;
  TG_HD void operator()(size_t pi) const {
    for (int s = smp_off[pi]; s < smp_off[pi + 1]; ++s) smp_prob[s] = (int)pi;
  }
};
struct LengthCheckFn {  // node.cpp:1178-1199
  BatchPtrs b;
  double dt, max_factor, min_factor;
  TG_HD void operator()(size_t pi) const {
    ProbState& ps = b.ps[pi];
    if (ps.status != kFindOk) return;
    const double len = (double)ps.n_samples * dt;
    if (len > 1.0 && len > (max_factor * ps.baca_total)) ps.status = kFindTooLong;
    else if (len > 1.0 && len < (min_factor * ps.baca_total)) ps.status = kFindTooShort;
  }
};

// ---- 8. validation + subdivision: one thread per problem -------------------------------------------------------------------
struct ValidateFn {
  BatchPtrs b;
  const int* smp_off;
  const double* xyzh;
  uint8_t* seg_ok;  // [totS]
  double max_deviation;
  int first_segment_checked, check_deviation;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = b.seg_off[p], S = b.seg_off[p + 1] - s0, V = S + 1, v0 = s0 + p;
    ProbState& ps = b.ps[p];
    ps.next_V = 0;
    if (ps.status != kFindOk) return;
    double md = 0.0;
    const int safe = validate_spatial(ps.n_samples, xyzh + 4 * (size_t)smp_off[p], V, b.wp + 4 * (size_t)v0, max_deviation,
                                      first_segment_checked, seg_ok + s0, &md);
    ps.max_dev = md;
    ps.safe = safe;
    if (check_deviation && !safe)
      ps.next_V = subdivide(V, b.wp + 4 * (size_t)v0, nullptr, seg_ok + s0, first_segment_checked, nullptr, nullptr);
  }
};
struct SubdivideFillFn {  // one thread per problem of the NEXT batch
  BatchPtrs old_b;
  const uint8_t* seg_ok;
  const int* src;          // next-batch problem -> old-batch problem
  const int* new_seg_off;  // next batch
  double* new_wp;
  uint8_t* new_stop;
  double* new_init14;      // or null
  int first_segment_checked;
  TG_HD void operator()(size_t qi) const {
    const int q = (int)qi, p = src[q];
    const int s0 = old_b.seg_off[p], V = old_b.seg_off[p + 1] - s0 + 1, v0 = s0 + p;
    const int nv0 = new_seg_off[q] + q;
    subdivide(V, old_b.wp + 4 * (size_t)v0, old_b.stop ? old_b.stop + v0 : nullptr, seg_ok + s0, first_segment_checked,
              new_wp + 4 * (size_t)nv0, new_stop + nv0);
    if (new_init14)
      for (int e = 0; e < 14; ++e) new_init14[14 * (size_t)q + e] = old_b.init14[14 * (size_t)p + e];
  }
};

// ---- 9. stand-alone pieces behind the class-level entry points ---------------------------------------------------------------
struct InitStateFn {  // ProbState reset for bare batches (no vertex recipe)
  ProbState* ps;
  TG_HD void operator()(size_t p) const {
    ProbState z;
    z.status = kFindOk; z.nlopt_code = 1; z.n_evals = 0; z.n_scale_passes = 0; z.scale_done = 0; z.n_samples = 0;
    z.sample_cap = 0; z.safe = 0; z.next_V = 0; z.n_grads = 0; z.final_cost = 0.0; z.cost = 0.0; z.baca_total = 0.0; z.max_dev = 0.0;
    ps[p] = z;
  }
};
struct CostOutFn {
  const ProbState* ps;
  double* cost;
  TG_HD void operator()(size_t p) const { cost[p] = ps[p].cost; }
};
struct CountOutFn {
  const ProbState* ps;
  int* counts;
  TG_HD void operator()(size_t p) const { counts[p] = ps[p].n_samples; }
};
struct ScaleOutFn {
  const ProbState* ps;
  const double* maxima;
  const int* seg_off;
  double L[9];
  int* passes;
  uint8_t* within;
  double tol;
  TG_HD void operator()(size_t p) const {
    passes[p] = ps[p].n_scale_passes;
    double g[9];
    for (int q = 0; q < 9; ++q) g[q] = TG_DBL_LOWEST;
    for (int i = seg_off[p]; i < seg_off[p + 1]; ++i)
      for (int q = 0; q < 9; ++q)
        if (maxima[(size_t)i * 9 + q] > g[q]) g[q] = maxima[(size_t)i * 9 + q];
    within[p] = violation_within(g, L, tol) ? 1 : 0;
  }
};
// Trajectory::evaluate(t, derivative) (eth/trajectory.cpp:55-87): one thread per query time
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
    for (int d = 0; d < TG_D; ++d) out[4 * qi + d] = (deriv >= TG_N) ? 0.0 : poly_eval(coef + ((size_t)i * TG_D + d) * TG_N, t - acc, deriv);
    if (ok) ok[qi] = 1;
  }
};
template <int Q>
struct ExtremaRawFn {  // one thread per work item (segment, or entry of a device work list) for quantity Q
  const double* coef;
  const double* times;
  double* maxima;
  const int* work;   // optional work list
  const int* n_dev;  // optional length of the work list (device memory)
  static constexpr int kScratch = JtScratch<QuantityDegree<Q>::value>::kShared;
  TG_HD void operator()(size_t item, double* scratch, int stride) const {
    if (n_dev && item >= (size_t)*n_dev) return;
    const size_t gs = work ? (size_t)work[item] : item;
    maxima[gs * 9 + Q] = segment_max_impl<Q>(coef + gs * TG_D * TG_N, times[gs], scratch, stride, nullptr);
  }
};
// The same launch with the operations of the executed stage-machine blocks added up (bench.py's per-kernel profile step only)
template <int Q>
struct ExtremaRawCountFn {
  ExtremaRawFn<Q> f;
  unsigned long long* flops;
  static constexpr int kScratch = ExtremaRawFn<Q>::kScratch;
  TG_HD void operator()(size_t item, double* scratch, int stride) const {
    if (f.n_dev && item >= (size_t)*f.n_dev) return;
    const size_t gs = f.work ? (size_t)f.work[item] : item;
    int fl = 0;
    f.maxima[gs * 9 + Q] = segment_max_impl<Q>(f.coef + gs * TG_D * TG_N, f.times[gs], scratch, stride, nullptr, &fl);
    TG_ATOMIC_ADD(flops, (unsigned long long)fl);
  }
};
// getTrajectoryReference with override_heading_atan2 (node.cpp:1586-1599): the heading of sample i becomes the direction towards
// sample i+1, or the previous sample's (already overridden) heading when that step is shorter than 0.05 m; the last sample
// keeps getYaw().  Sequential in the previous heading: one thread per problem.
struct HeadingAtan2Fn {
  const int* smp_off;
  const ProbState* ps;
  double* xyzh;
  TG_HD void operator()(size_t p) const {
    const int n = ps[p].n_samples;
    double* s = xyzh + (size_t)smp_off[p] * 4;
    for (int it = 0; it + 1 < n; ++it) {
      const double dy = s[4 * (it + 1) + 1] - s[4 * it + 1], dx = s[4 * (it + 1)] - s[4 * it];
      const double dist = tgdm::dhypot(dy, dx);
      if (dist < 0.05 && it > 0) s[4 * it + 3] = s[4 * (it - 1) + 3];
      else s[4 * it + 3] = tgdm::datan2(dy, dx);
    }
  }
};
// Test hook (tg_test_find_roots_batch): findRootsJenkinsTraub (rpoly_ak1.cpp:76-120) on arbitrary polynomials of up to 16
// coefficients, zeros written in the order the reference stores them (zeros at the origin, then as found)
struct RootSink {
  double* re;
  double* im;
  int n;
  TG_HD void operator()(double r, double i) {
    re[n] = r;
    im[n] = i;
    ++n;
  }
};
struct FindRootsFn {
  const double* coeffs;  // [n][16] increasing powers, zero padded
  const int* ncoef;
  double* re;            // [n][16]
  double* im;
  int* nroots;
  static constexpr int kScratch = 4 * 16;
  TG_HD void operator()(size_t i, double* scratch, int stride) const {
    double ci[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) ci[k] = (k < ncoef[i]) ? coeffs[i * 16 + k] : 0.0;
    RootSink sink{re + i * 16, im + i * 16, 0};
    find_roots_jt<15>(ci, scratch, stride, sink, nullptr);
    nroots[i] = sink.n;
  }
};
// computeMaximumOfMagnitude (lin_impl.h:477-508), step 1: one thread per segment -> the segment's first-largest candidate
template <int DERIV>
struct MaxMagnitudeSegFn {
  const double* coef;
  const double* times;
  double* seg_value;
  double* seg_time;
  static constexpr int kScratch = 4 * (MaxAllDegree<DERIV>::value + 1);  // always the stage machine of tg_poly.cuh
  TG_HD void operator()(size_t gs, double* scratch, int stride) const {
    segment_max_all_dims<DERIV>(coef + gs * TG_D * TG_N, times[gs], scratch, stride, seg_value + gs, seg_time + gs);
  }
};
// step 2: one thread per trajectory walks its segments in order; the running Extremum starts at (0, 0, 0) (lin_impl.h:483)
struct MaxMagnitudeReduceFn {
  const int* seg_off;
  const double* seg_value;
  const double* seg_time;
  double* value;
  double* time;
  int* segment_idx;
  TG_HD void operator()(size_t p) const {
    double best = 0.0, best_t = 0.0;
    int best_i = 0;
    const int s0 = seg_off[p], s1 = seg_off[p + 1];
    for (int s = s0; s < s1; ++s)
      if (best < seg_value[s]) {
        best = seg_value[s];
        best_t = seg_time[s];
        best_i = s - s0;
      }
    value[p] = best;
    time[p] = best_t;
    segment_idx[p] = best_i;
  }
};
struct CompactSamplesFn {  // one thread per sample slot: slot arrays (with per-problem slack) -> contiguous outputs
  const int* smp_off;
  const int* smp_prob;
  const int* dst_off;  // [B] exclusive scan of the true counts
  const ProbState* ps;
  const double* xyzh;
  const double* full;
  double* o_xyzh;
  double* o_full;
  TG_HD void operator()(size_t slot) const {
    const int p = smp_prob[slot], k = (int)slot - smp_off[p];
    if (k >= ps[p].n_samples) return;
    const size_t dst = (size_t)dst_off[p] + k;
    if (o_xyzh)
      for (int e = 0; e < 4; ++e) o_xyzh[4 * dst + e] = xyzh[4 * slot + e];
    if (o_full)
      for (int e = 0; e < 19; ++e) o_full[19 * dst + e] = full[19 * slot + e];
  }
};
// first-minimum argmin over chunks of 1024 candidates (the host finishes over the chunk results)
struct ArgminChunkFn {
  long long K;
  const double* costs;
  double* cmin;
  long long* cidx;
  TG_HD void operator()(size_t c) const {
    const long long k0 = (long long)c * 1024, k1 = (k0 + 1024 < K) ? k0 + 1024 : K;
    double best = costs[k0];
    long long bi = k0;
    for (long long k = k0 + 1; k < k1; ++k)
      if (costs[k] < best) { best = costs[k]; bi = k; }
    cmin[c] = best;
    cidx[c] = bi;
  }
};

// final gather: 32 consecutive items (one warp) copy the outputs of one group member into the contiguous result arrays
struct GatherFn {
  const int* seg_off;
  const int* smp_off;
  const ProbState* ps;
  const int* dst_seg;  // [B] destination segment offset, or -1 when this group does not hold the member's final result
  const int* dst_vtx;
  const int* dst_smp;
  const double *wp, *times, *coef, *xyzh;
  double *o_wp, *o_times, *o_coef, *o_xyzh;
  TG_HD void operator()(size_t item) const {
    const int m = (int)(item >> 5), lane = (int)(item & 31);
    const int ds = dst_seg[m];
    if (ds < 0) return;
    const int s0 = seg_off[m], S = seg_off[m + 1] - s0, v0 = s0 + m;
    if (o_times)
      for (int i = lane; i < S; i += 32) o_times[ds + i] = times[s0 + i];
    if (o_coef)
      for (int i = lane; i < S * TG_D * TG_N; i += 32) o_coef[(size_t)ds * TG_D * TG_N + i] = coef[(size_t)s0 * TG_D * TG_N + i];
    if (o_wp)
      for (int i = lane; i < (S + 1) * 4; i += 32) o_wp[4 * (size_t)dst_vtx[m] + i] = wp[4 * (size_t)v0 + i];
    if (o_xyzh) {
      const int n = ps[m].n_samples * 4;
      for (int i = lane; i < n; i += 32) o_xyzh[4 * (size_t)dst_smp[m] + i] = xyzh[4 * (size_t)smp_off[m] + i];
    }
  }
};

// any non-finite waypoint or initial-state entry among the uploaded inputs (checkNaN of the path callbacks, node.cpp:1896-1900): one
// thread per path; the count only says whether the host has to find out which paths to leave out
struct FiniteInputsFn {
  const int* seg_off;
  const double* wp;      // [totV][4]
  const double* init14;  // [B][14] or null
  int* bad;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, v0 = seg_off[p] + p, V = seg_off[p + 1] - seg_off[p] + 1;
    bool finite = true;
    for (int i = 0; i < V * 4; ++i) finite = finite && dfinite(wp[(size_t)v0 * 4 + i]);
    if (init14 && init14[(size_t)p * 14] != 0.0)
      for (int k = 1; k < 14; ++k) finite = finite && dfinite(init14[(size_t)p * 14 + k]);
    if (!finite) TG_ATOMIC_ADD(bad, 1);
  }
};

// samples of the members whose result is final, compacted in member order: one warp per member (dst_row < 0: not final yet)
struct GatherSamplesFn {
  const int* smp_off;
  const ProbState* ps;
  const int* dst_row;
  const double* xyzh;
  double* out;
  TG_HD void operator()(size_t item) const {
    const int m = (int)(item >> 5), lane = (int)(item & 31);
    const int d = dst_row[m];
    if (d < 0) return;
    const int n = ps[m].n_samples * 4;
    for (int i = lane; i < n; i += 32) out[4 * (size_t)d + i] = xyzh[4 * (size_t)smp_off[m] + i];
  }
};

// vertex -> problem map: one thread per problem
struct VtxProblemFn {
  const int* seg_off;
  int* prob_of_vtx;
  int* prob_of_seg;
  TG_HD void operator()(size_t pi) const {
    const int p = (int)pi, s0 = seg_off[p], v0 = s0 + p, S = seg_off[p + 1] - s0;
    for (int v = 0; v < S + 1; ++v) prob_of_vtx[v0 + v] = p;
    for (int i = 0; i < S; ++i) prob_of_seg[s0 + i] = p;
  }
};

// ---- 10. the steps either side of the path: one thread per path ----------------------------------------------------------
struct PreprocessFn {
  const int* wp_off;
  const double* wp;
  const uint8_t* stop;  // or null
  double min_dist, max_dev, max_hdg_dev;
  int straighten;
  double* out_wp;       // [totV][4], problem p writes from wp_off[p]
  uint8_t* out_stop;
  int* out_count;
  TG_HD void operator()(size_t p) const {
    const int v0 = wp_off[p], V = wp_off[p + 1] - v0;
    out_count[p] = preprocess_path(V, wp + 4 * (size_t)v0, stop ? stop + v0 : nullptr, min_dist, straighten, max_dev, max_hdg_dev, out_wp + 4 * (size_t)v0,
                                   out_stop + v0);
  }
};
struct FallbackFn {
  const int* wp_off;
  const double* wp;
  const uint8_t* stop;
  double L[9];
  double dt, stopping_time;
  double* vpos;          // scratch [totV][4]
  int* count;            // [B]
  const int* smp_off;    // null in the counting pass
  double* samples;       // null in the counting pass
  TG_HD void operator()(size_t p) const {
    const int v0 = wp_off[p], V = wp_off[p + 1] - v0;
    const int n = fallback_samples(V, wp + 4 * (size_t)v0, stop ? stop + v0 : nullptr, L, dt, stopping_time, vpos + 4 * (size_t)v0,
                                   samples ? samples + 4 * (size_t)smp_off[p] : nullptr);
    if (!samples) count[p] = n;
  }
};
struct WaypointIdxFn {
  const int* smp_off;
  const double* samples;
  const int* wp_off;
  const double* wp;
  int* idxs;    // [totV], problem p writes from wp_off[p]
  int* count;   // [B]
  TG_HD void operator()(size_t p) const {
    const int m0 = smp_off[p], M = smp_off[p + 1] - m0, v0 = wp_off[p], V = wp_off[p + 1] - v0;
    count[p] = waypoint_idxs(M, samples + 4 * (size_t)m0, V, wp + 4 * (size_t)v0, idxs + v0);
  }
};

}  // namespace tg

#endif  // TG_KERNELS_CUH_
