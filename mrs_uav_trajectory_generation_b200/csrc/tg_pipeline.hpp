// tg_pipeline.hpp -- host-side orchestration of the batched trajectory pipeline, templated on a Backend that knows
// how to allocate device memory, copy, and launch the functors of tg_kernels.cuh (CudaBackend in cuda_backend.cu;
// tests/host_emu/EmuBackend runs the same code on the CPU for GPU-less bit-parity tests).
//
// find_batch()     = MrsTrajectoryGeneration::findTrajectory for every problem of a ragged batch (node.cpp:857-1209)
// optimize_batch() = the validation / midpoint-subdivision loop of optimize() around it (node.cpp:729-785)
#ifndef TG_PIPELINE_HPP_
#define TG_PIPELINE_HPP_

#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <functional>
#include <memory>
#include <string>
#include <vector>

#include "tg_kernels.cuh"
#include "tg_dfo.cuh"
#include "tg_dfo_generic.cuh"
#include "tg_generic.cuh"

namespace tg {

// bump allocator over backend device memory; chunks are kept and reused across calls
template <class BE>
class Arena {
 public:
  explicit Arena(BE& be, size_t chunk = (size_t)256 << 20) : be_(be), chunk_(chunk) {}
  ~Arena() {
    for (auto& c : chunks_) be_.dev_free(c.ptr);
  }
  void* alloc_bytes(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes == 0) bytes = 256;
    while (cur_ < chunks_.size()) {
      Chunk& c = chunks_[cur_];
      if (c.used + bytes <= c.size) {
        void* p = (char*)c.ptr + c.used;
        c.used += bytes;
        return p;
      }
      ++cur_;
    }
    Chunk c;
    c.size = std::max(chunk_, bytes);
    c.ptr = be_.dev_alloc(c.size);
    c.used = bytes;
    chunks_.push_back(c);
    cur_ = chunks_.size() - 1;
    return c.ptr;
  }
  template <class T>
  T* alloc(size_t n) { return (T*)alloc_bytes(n * sizeof(T)); }
  void reset() {
    for (auto& c : chunks_) c.used = 0;
    cur_ = 0;
  }
  size_t bytes_reserved() const {
    size_t t = 0;
    for (auto& c : chunks_) t += c.size;
    return t;
  }

 private:
  struct Chunk { void* ptr; size_t size, used; };
  BE& be_;
  size_t chunk_;
  std::vector<Chunk> chunks_;
  size_t cur_ = 0;
};

// host-visible per-problem result (mirrors tg_result in include/tg_b200.h)
struct Result {
  int status, success, nlopt_code, n_evals, rounds, safe, n_waypoints, n_samples, n_scale_passes, overflow;
  double max_dev, final_cost, baca_total;
  long long total_solves, total_root_calls, total_evals;
};

// a typed view of host memory owned by the backend's page-locked arena
template <class T>
struct HostView {
  T* p = nullptr;
  size_t n = 0;
  T& operator[](size_t i) { return p[i]; }
  const T& operator[](size_t i) const { return p[i]; }
  T* data() { return p; }
  size_t size() const { return n; }
};

// One processed group of problems whose outputs stay on the device until gathered.
struct Group {
  int B = 0, totS = 0, totV = 0, totSlots = 0;
  std::vector<int> seg_off, smp_off;       // host copies
  HostView<ProbState> ps;                  // host copy after find (page-locked arena of the backend, valid until the next batch call)
  std::vector<int> orig;                   // original problem index of each member
  std::vector<int> h_np, h_hbw;            // host copies of the unknown counts / half bandwidths (work accounting)
  // device (persistent arena)
  int* d_seg_off = nullptr;
  double* d_wp = nullptr;
  uint8_t* d_stop = nullptr;
  double* d_init14 = nullptr;
  double* d_times = nullptr;
  double* d_coef = nullptr;
  double* d_xyzh = nullptr;
  int* d_smp_off = nullptr;
  uint8_t* d_seg_ok = nullptr;
  ProbState* d_ps = nullptr;
  BatchPtrs bp;
};

struct Counters {
  long long launches = 0, solves = 0, evals = 0, root_finds = 0, segment_setups = 0, samples = 0;
  // algorithmic flops (SURVEY.md 8(d) formula, DESIGN.md) of the work actually launched, per kernel family
  double flops_solve = 0, flops_setup = 0, flops_sample = 0, flops_coef = 0;
  long long root_finds_executed = 0;  // Jenkins-Traub runs actually launched (root_finds counts what the reference would run)
  long long mellinger_solves = 0, mellinger_launches = 0;
};

template <class BE>
class Pipeline {
 public:
  explicit Pipeline(BE& be) : be_(be), persist_(be), scratch_(be) {}

  BE& backend() { return be_; }
  Counters counters;
  bool prune_extrema = true;            // tg_bound.cuh certificates (exact); off only for A/B measurements (TG_NO_PRUNE)
  bool use_thread_solve = std::getenv("TG_NO_THREAD_SOLVE") == nullptr;  // tg_solve_thread.cuh; off only for A/B measurements
  // The thread-per-instance solve is a throughput kernel: one thread walks a whole system (50 us at S = 10, 1.3 ms at S = 264), so it
  // only pays when the instances fill the machine (148 SMs x 256 threads).  Smaller launches -- single paths, the 200-waypoint path
  // of BASELINE config 4 -- go to the lane-parallel kernels (8 lanes or a warp per system), whose results are bit-identical.
  size_t thread_min_inst = std::getenv("TG_THREAD_MIN_INST") ? (size_t)std::atoll(std::getenv("TG_THREAD_MIN_INST")) : (size_t)16384;
  bool thread_solve_for(size_t n_inst) const { return use_thread_solve && n_inst >= thread_min_inst; }
  // the same rule inside the evaluation tail: a work list shorter than this goes to the lane-parallel kernels (measured: list
  // launches 13.1 -> 9.5 ms per step; default = thread_min_inst)
  size_t list_octet_below = std::getenv("TG_LIST_OCTET_BELOW") ? (size_t)std::atoll(std::getenv("TG_LIST_OCTET_BELOW")) : thread_min_inst;
  double scale_tolerance = 1e-3;        // eth/trajectory.cpp:604; tg_test_set_scale_tolerance changes it (tests only)
  // max segments per group (bounds scratch memory: ~5.6 kB per segment); TG_SEG_BUDGET lowers it so that tests can drive the
  // several-groups path of a huge batch with a small one
  size_t seg_budget = std::getenv("TG_SEG_BUDGET") ? (size_t)std::max(1LL, std::atoll(std::getenv("TG_SEG_BUDGET"))) : ((size_t)1 << 21);

  // ---------------------------------------------------------------------------------------------------------------
  // findTrajectory over one group.  Inputs (wp/stop/init14) already in device memory inside `g`.
  void find_group(Group& g, const Params& P, bool validate) {
    const int B = g.B, totS = g.totS, totV = g.totV;
    HostTrace tf0 = trace_mark();
    BatchPtrs& b = g.bp;
    std::memset(&b, 0, sizeof(b));
    b.B = B; b.totS = totS; b.totV = totV; b.r = P.derivative_to_optimize;
    b.seg_off = g.d_seg_off;
    b.wp = g.d_wp; b.stop = g.d_stop; b.init14 = g.d_init14;
    int* pov = scratch_.template alloc<int>(totV);
    int* pos = scratch_.template alloc<int>(totS);
    b.prob_of_vtx = pov; b.prob_of_seg = pos;
    b.vmask = scratch_.template alloc<uint8_t>(totV);
    b.vval = scratch_.template alloc<double>((size_t)totV * TG_HALF * TG_D);
    b.vfree = scratch_.template alloc<int>((size_t)totV + B);
    b.np = scratch_.template alloc<int>(B);
    b.hbw = scratch_.template alloc<int>(B);
    b.fmax = scratch_.template alloc<int>(B);
    b.stats = scratch_.template alloc<int>(16);
    b.times = g.d_times;
    b.baca = scratch_.template alloc<double>(totS);
    b.coef = g.d_coef;
    b.ps = g.d_ps;
    be_.dev_memset(b.stats, 0, 16 * sizeof(int));
    be_.for_each(B, VtxProblemFn{g.d_seg_off, pov, pos}); launches(1);
    be_.for_each(B, PrepareFn{b, 1}); launches(1);
    TimesFn tf{b, {}};
    for (int i = 0; i < 9; ++i) tf.L[i] = P.limits[i];
    be_.for_each(totS, tf); launches(1);
    be_.for_each(B, BacaTotalFn{b}); launches(1);
    int stats[16];
    be_.d2h(stats, b.stats, sizeof(stats));
    const int ws = stats[0], ows = stats[2];
    alloc_solution_buffers(b, (size_t)(P.run_time_alloc ? totV : B), stats);
    std::vector<int>& h_np = g.h_np;
    std::vector<int>& h_hbw = g.h_hbw;
    h_np.resize(B);
    h_hbw.resize(B);
    be_.d2h(h_np.data(), b.np, sizeof(int) * B);
    be_.d2h(h_hbw.data(), b.hbw, sizeof(int) * B);
    const std::vector<SolveBucket> buckets = make_buckets(B, g.seg_off.data(), h_np.data(), h_hbw.data(), ws, ows, stats[3]);
    trace_report(" find: prepare + buckets", -1, tf0);
    tf0 = trace_mark();
    if (P.run_time_alloc) {
      time_alloc_core(b, P, stats, &buckets);
      trace_report(" find: time allocation", -1, tf0);
      tf0 = trace_mark();
    } else {
      b.recs = scratch_.template alloc<double>((size_t)totS * TG_REC_SIZE);
    }
    // final linear solve at the (scaled) times (nl_impl.h:405-408 / lin_impl.h:340-373)
    be_.for_each(totS, SetupBaseFn{b, b.times});
    solve_with_outputs((size_t)B, stats, SolveProblemDesc{b, 0, nullptr, nullptr}, b, &buckets, false);
    launches(2);
    // sampling (eth/trajectory_sampling.cpp:49-104)
    int* cap = scratch_.template alloc<int>((size_t)B + 1);
    g.d_smp_off = persist_.template alloc<int>((size_t)B + 1);
    be_.for_each(B, SampleCapFn{b, P.dt, cap}); launches(1);
    be_.exclusive_scan(cap, g.d_smp_off, B); launches(1);
    g.smp_off.resize(B + 1);
    be_.d2h(g.smp_off.data(), g.d_smp_off, sizeof(int) * (B + 1));
    g.totSlots = g.smp_off[B];
    const size_t slots = (size_t)std::max(g.totSlots, 1);
    int* seg_idx = scratch_.template alloc<int>(slots);
    int* smp_prob = scratch_.template alloc<int>(slots);
    double* t_in = scratch_.template alloc<double>(slots);
    g.d_xyzh = persist_.template alloc<double>(slots * 4);
    be_.for_each(B, SampleWalkFn{b, P.dt, g.d_smp_off, seg_idx, t_in});
    be_.for_each(B, SlotProblemFn{B, g.d_smp_off, smp_prob});
    be_.for_each((size_t)g.totSlots, SampleEvalFn{b, g.d_smp_off, smp_prob, seg_idx, t_in, g.d_xyzh, nullptr});
    be_.for_each(B, LengthCheckFn{b, P.dt, P.max_len_factor, P.min_len_factor});
    launches(4);
    if (P.override_heading_atan2) {  // validation reads positions only, so the override may happen here
      be_.for_each(B, HeadingAtan2Fn{g.d_smp_off, g.d_ps, g.d_xyzh});
      launches(1);
    }
    if (validate) {  // validateTrajectorySpatial (node.cpp:1401-1455) before the one read-back of the per-problem state
      be_.for_each(B, ValidateFn{g.bp, g.d_smp_off, g.d_xyzh, g.d_seg_ok, P.max_deviation, P.first_segment_checked, P.check_deviation});
      launches(1);
    }
    g.ps = HostView<ProbState>{static_cast<ProbState*>(be_.pinned_alloc(sizeof(ProbState) * (size_t)B)), (size_t)B};
    be_.d2h_pinned(g.ps.data(), g.d_ps, sizeof(ProbState) * B);
    trace_report(" find: solve .. state read", -1, tf0);
    if (P.run_time_alloc) {
      int executed = 0;
      be_.d2h(&executed, b.stats + 5, sizeof(int));
      counters.root_finds_executed += executed;
    }
  }
  // work accounting of one processed group (SURVEY.md 8(d) formulas x what was launched); pure host arithmetic over the per-problem
  // state, deferred like fill_results
  void account_group(const Group& g, const Params& P) {
    const int B = g.B;
    const std::vector<int>& h_np = g.h_np;
    const std::vector<int>& h_hbw = g.h_hbw;
    for (int p = 0; p < B; ++p) {
      const int S = g.seg_off[p + 1] - g.seg_off[p];
      const int ev = g.ps[p].n_evals;
      const int ng = g.ps[p].n_grads;  // evaluations whose S perturbed solves were run
      const long long nsolve = (long long)ev + (S == 1 ? 0 : (long long)ng * S) + 1;
      const long long nsetup = (long long)ev * S + (S == 1 ? 0 : (long long)ng * 2 * S) + S;
      const double np_ = h_np[p], bw = h_hbw[p];
      // SURVEY.md 8(d) formula, split by kernel: banded factorisation + right-hand sides + back substitution (solve kernel),
      // coefficients + cost (CoefCostFn)
      const double f_solve = np_ * (bw * bw + 3.0 * bw) + 4.0 * (2.0 * np_ * 15.0 + 4.0 * np_ * bw);
      const double f_coef = 4.0 * (S * 200.0 + S * 220.0);
      const double nq = TG_N - P.derivative_to_optimize;
      const double f_setup = 3.0 * nq * nq + 525.0 + 4.0 * TG_N * TG_N * TG_N;
      counters.flops_solve += f_solve * (double)nsolve;
      counters.flops_coef += f_coef * (double)nsolve;
      counters.flops_setup += f_setup * (double)nsetup;
      counters.flops_sample += 340.0 * g.ps[p].n_samples;
      counters.mellinger_solves += nsolve - 1;
      counters.evals += ev;
      counters.solves += nsolve;
      counters.segment_setups += nsetup;
      counters.root_finds += (long long)(P.run_time_alloc ? (g.ps[p].n_scale_passes + 1) * 9 * S : 0);
      counters.samples += g.ps[p].n_samples;
    }
  }

  // ---------------------------------------------------------------------------------------------------------------
  // Builds a group on the device from host inputs (problem subset [p0, p1) of a host batch).
  Group* make_group_from_host(const std::vector<int>& members, const int* wp_off, const double* wp, const uint8_t* stop,
                              const double* init14, bool on_device_inputs) {
    groups_.emplace_back(new Group());
    Group& g = *groups_.back();
    const int B = (int)members.size();
    g.B = B;
    g.orig = members;
    g.seg_off.resize(B + 1);
    g.seg_off[0] = 0;
    for (int i = 0; i < B; ++i) g.seg_off[i + 1] = g.seg_off[i] + (wp_off[members[i] + 1] - wp_off[members[i]] - 1);
    g.totS = g.seg_off[B];
    g.totV = g.totS + B;
    alloc_group_outputs(g, init14 != nullptr);
    // members are a contiguous range of the host batch: copy straight through
    const int first = members.front();
    const size_t v0 = (size_t)wp_off[first];
    if (on_device_inputs) {
      be_.d2d(g.d_wp, wp + 4 * v0, sizeof(double) * 4 * g.totV);
      if (stop) be_.d2d(g.d_stop, stop + v0, g.totV);
      if (init14) be_.d2d(g.d_init14, init14 + 14 * (size_t)first, sizeof(double) * 14 * B);
    } else {
      be_.h2d(g.d_wp, wp + 4 * v0, sizeof(double) * 4 * g.totV);
      if (stop) be_.h2d(g.d_stop, stop + v0, g.totV);
      if (init14) be_.h2d(g.d_init14, init14 + 14 * (size_t)first, sizeof(double) * 14 * B);
    }
    if (!stop) be_.dev_memset(g.d_stop, 0, g.totV);
    return &g;
  }

  void alloc_group_outputs(Group& g, bool with_init) {
    const int B = g.B;
    g.d_seg_off = persist_.template alloc<int>((size_t)B + 1);
    be_.h2d(g.d_seg_off, g.seg_off.data(), sizeof(int) * (B + 1));
    g.d_wp = persist_.template alloc<double>((size_t)g.totV * 4);
    g.d_stop = persist_.template alloc<uint8_t>(g.totV);
    g.d_init14 = with_init ? persist_.template alloc<double>((size_t)B * 14) : nullptr;
    g.d_times = persist_.template alloc<double>(g.totS);
    g.d_coef = persist_.template alloc<double>((size_t)g.totS * TG_D * TG_N);
    g.d_seg_ok = persist_.template alloc<uint8_t>(g.totS);
    g.d_ps = persist_.template alloc<ProbState>(B);
  }

  // ---------------------------------------------------------------------------------------------------------------
  // Samples streamed to the host while later rounds still run (tg_optimize_batch_streamed).  A path's samples are final as soon as
  // its validation passes (or it fails); most paths finish in the first rounds, so their device-to-host copy -- 120 MB per 65 536
  // paths, the largest cost outside the kernels -- overlaps the rounds that follow.  Paths land in COMPLETION order: begin[p] is
  // the first row of path p.  Too small a buffer sets `overflow` and stops the copies (the results stay fetchable).
  // TG_TRACE_HOST: host time outside device waits, per phase of a round (the device may be idle during it)
  struct HostTrace {
    std::chrono::steady_clock::time_point t;
    double w;
  };
  HostTrace trace_mark() const { return HostTrace{std::chrono::steady_clock::now(), be_.wait_s}; }
  void trace_report(const char* what, int round, const HostTrace& m) const {
    if (!be_.trace_host) return;
    const double tot = std::chrono::duration<double>(std::chrono::steady_clock::now() - m.t).count();
    std::fprintf(stderr, "[tg]   round %d %-28s %7.2f ms, host work %6.2f ms\n", round, what, 1e3 * tot, 1e3 * (tot - (be_.wait_s - m.w)));
  }
  struct EarlySamples {
    double* host = nullptr;
    long long cap = 0, used = 0;
    long long* begin = nullptr;  // [B]
    bool overflow = false;
  };
  EarlySamples early;
  // host bookkeeping of a finished round that the device does not wait for (see optimize_batch)
  std::function<void()> deferred_;
  bool defer_bookkeeping = std::getenv("TG_DEFER") ? std::atoi(std::getenv("TG_DEFER")) != 0 : true;  // off only for A/B measurements
  void run_deferred() {
    if (!deferred_) return;
    std::function<void()> f = std::move(deferred_);
    deferred_ = nullptr;
    f();
  }
  void fill_results(const Group& g, int gi, int round, bool last_round, const Params& P, Result* results) {
    for (int m = 0; m < g.B; ++m) {
      const int p = g.orig[m];
      // from round 1 on the members are ordered by their new size, not by path: results[] is walked at random
      if (m + 16 < g.B) __builtin_prefetch(&results[g.orig[m + 16]], 1);
      const ProbState& ps = g.ps[m];
      Result& R = results[p];
      final_group_[p] = gi;
      final_index_[p] = m;
      const int S = g.seg_off[m + 1] - g.seg_off[m];
      R.status = ps.status;
      R.nlopt_code = ps.nlopt_code;
      R.n_evals = ps.n_evals;
      R.rounds = round;
      R.n_waypoints = S + 1;
      R.n_samples = ps.n_samples;
      R.n_scale_passes = ps.n_scale_passes;
      R.final_cost = P.run_time_alloc ? ps.final_cost : ps.cost;
      R.baca_total = ps.baca_total;
      R.total_evals += ps.n_evals;
      R.total_solves += (long long)ps.n_evals * (S == 1 ? 1 : S + 2) + 1;  // reference count: S+2 solves per evaluation
      R.total_root_calls += P.run_time_alloc ? (long long)ps.n_scale_passes * 18 * S : 0;
      if (ps.status != kFindOk) { R.success = 0; continue; }
      R.success = 1;
      if (last_round) { R.safe = 0; continue; }  // returned without re-validation (node.cpp:729-785)
      R.max_dev = ps.max_dev;
      if (ps.next_V <= 0) R.safe = 1;
    }
  }
  void stream_finished_samples(Group& g, const std::vector<int>& finals) {
    if (!early.host || early.overflow || finals.empty()) return;
    std::vector<int> dst((size_t)g.B, -1);
    long long rows = 0;
    for (int m : finals) {
      dst[m] = (int)rows;
      early.begin[g.orig[m]] = early.used + rows;
      rows += g.ps[m].n_samples;
    }
    if (rows == 0) return;
    if (early.used + rows > early.cap) {
      early.overflow = true;
      return;
    }
    // the compact copy and the offsets live in the persistent arena: the copy engine reads them after scratch_ has been reset
    int* d_dst = persist_.template alloc<int>((size_t)g.B);
    double* d_rows = persist_.template alloc<double>((size_t)rows * 4);
    be_.h2d(d_dst, dst.data(), sizeof(int) * (size_t)g.B);
    be_.for_each((size_t)g.B * 32, GatherSamplesFn{g.d_smp_off, g.d_ps, d_dst, g.d_xyzh, d_rows});
    launches(1);
    be_.d2h_overlapped(early.host + 4 * early.used, d_rows, sizeof(double) * 4 * (size_t)rows);
    early.used += rows;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // optimize(): findTrajectory + validation + subdivision rounds for a whole host batch.
  // wp_off: [B+1] vertex offsets (host).  wp/stop/init14: host pointers, or device pointers when on_device_inputs.
  void optimize_batch(int B, const int* wp_off, const double* wp, const uint8_t* stop, const double* init14, const Params& P,
                      bool on_device_inputs, Result* results) {
    // round 0: consecutive groups within the segment budget.  Non-finite host inputs are looked for on the device first (one small
    // launch per group over data that is being uploaded anyway); only a batch that has one pays for the host scan, which is what
    // tells the groups which paths to leave out (2.9 M isfinite tests per 65 536 paths: ~2 ms of every host-buffer call otherwise).
    std::vector<Group*> current;
    deferred_ = nullptr;
    for (int attempt = 0;; ++attempt) {
      const bool host_scan = attempt > 0;
      persist_.reset();
      scratch_.reset();
      groups_.clear();
      be_.pinned_reset();
      current.clear();
      final_group_.assign(B, -1);
      final_index_.assign(B, -1);
      B_ = B;
      for (int p = 0; p < B; ++p) {
        std::memset(&results[p], 0, sizeof(Result));
        results[p].nlopt_code = -1;
      }
      std::vector<int> members;
      size_t segs = 0;
      for (int p = 0; p < B; ++p) {
        const int S = wp_off[p + 1] - wp_off[p] - 1;
        // the path callbacks drop a message with a non-finite waypoint before optimize() runs (checkNaN, node.cpp:1896-1900); a batch
        // cannot drop its caller's message, so the path is excluded and flagged (host inputs only: device-resident inputs are the
        // caller's contract)
        bool finite = true;
        if (host_scan && S >= 1) {
          for (int v = wp_off[p]; v < wp_off[p + 1] && finite; ++v)
            for (int k = 0; k < 4; ++k) finite = finite && std::isfinite(wp[(size_t)v * 4 + k]);
          if (finite && init14 && init14[(size_t)p * 14] != 0.0)
            for (int k = 1; k < 14; ++k) finite = finite && std::isfinite(init14[(size_t)p * 14 + k]);
        }
        if (!finite) {
          if (!members.empty()) { current.push_back(make_group_from_host(members, wp_off, wp, stop, init14, on_device_inputs)); members.clear(); segs = 0; }
          results[p].status = kFindNotFinite;
          continue;
        }
        if (S < 1) {  // "the path is empty (after postprocessing)" (node.cpp:676-681)
          if (!members.empty()) { current.push_back(make_group_from_host(members, wp_off, wp, stop, init14, on_device_inputs)); members.clear(); segs = 0; }
          results[p].status = kFindEmptyPath;
          continue;
        }
        if (!members.empty() && segs + S > seg_budget) {
          current.push_back(make_group_from_host(members, wp_off, wp, stop, init14, on_device_inputs));
          members.clear();
          segs = 0;
        }
        members.push_back(p);
        segs += S;
      }
      if (!members.empty()) current.push_back(make_group_from_host(members, wp_off, wp, stop, init14, on_device_inputs));
      if (on_device_inputs || host_scan || current.empty()) break;  // device-resident inputs are the caller's contract
      int* d_bad = scratch_.template alloc<int>(1);
      be_.dev_memset(d_bad, 0, sizeof(int));
      for (Group* g : current) be_.for_each(g->B, FiniteInputsFn{g->d_seg_off, g->d_wp, g->d_init14, d_bad});
      launches((int)current.size());
      int bad = 0;
      be_.d2h(&bad, d_bad, sizeof(int));
      if (bad == 0) break;
    }
    for (int round = 0;; ++round) {
      // run findTrajectory on every group of this round, then validate
      std::vector<std::pair<Group*, int>> pending;  // (group, member) that need another round
      for (Group* g : current) {
        scratch_.reset();
        const bool last_round = (round >= P.max_deviation_iters);
        HostTrace tm = trace_mark();
        find_group(*g, P, !last_round);
        trace_report("find_group", round, tm);
        tm = trace_mark();
        // What the next round needs (which members go on) and which members are final: one light pass over the per-problem state.
        // The result records and the work accounting -- ~1.5 ms of host stores per round that nothing on the device depends on -- are
        // deferred: they run while the device works on the first evaluation of the next round (run_deferred in time_alloc_core).
        std::vector<int> finals;  // members whose result is final after this round
        if (early.host) finals.reserve((size_t)g->B);
        for (int m = 0; m < g->B; ++m) {
          const ProbState& ps = g->ps[m];
          if (ps.status == kFindOk && !last_round && ps.next_V > 0) pending.emplace_back(g, m);
          else if (early.host) finals.push_back(m);
        }
        stream_finished_samples(*g, finals);
        run_deferred();
        {
          const int gi = group_index(g);
          deferred_ = [this, g, gi, round, last_round, results, &P]() {
            fill_results(*g, gi, round, last_round, P, results);
            account_group(*g, P);
          };
          if (!defer_bookkeeping) run_deferred();
        }
        trace_report("next-round scan + streamed samples", round, tm);
      }
      if (pending.empty()) break;
      const HostTrace tn = trace_mark();
      // members of a next-round group in order of their new segment count (the order inside a group is free: results
      // go back through `orig`), so that problems of one workspace class are consecutive -> SolveBucket runs
      {
        size_t a = 0;
        while (a < pending.size()) {
          size_t e = a;
          while (e < pending.size() && pending[e].first == pending[a].first) ++e;
          // stable counting sort on the new vertex count (a few hundred distinct values at most): the device waits for this loop, and a
          // comparison sort of ~40 000 entries cost it milliseconds per round
          int kmin = pending[a].first->ps[pending[a].second].next_V, kmax = kmin;
          for (size_t i = a; i < e; ++i) {
            const int k = pending[i].first->ps[pending[i].second].next_V;
            kmin = std::min(kmin, k);
            kmax = std::max(kmax, k);
          }
          if ((size_t)(kmax - kmin) <= (e - a) + 1024) {
            std::vector<size_t> start((size_t)(kmax - kmin) + 2, 0);
            for (size_t i = a; i < e; ++i) ++start[(size_t)(pending[i].first->ps[pending[i].second].next_V - kmin) + 1];
            for (size_t k = 1; k < start.size(); ++k) start[k] += start[k - 1];
            std::vector<std::pair<Group*, int>> sorted(e - a);
            for (size_t i = a; i < e; ++i) sorted[start[(size_t)(pending[i].first->ps[pending[i].second].next_V - kmin)]++] = pending[i];
            std::copy(sorted.begin(), sorted.end(), pending.begin() + a);
          } else {
            std::stable_sort(pending.begin() + a, pending.begin() + e, [](const std::pair<Group*, int>& x, const std::pair<Group*, int>& y) {
              return x.first->ps[x.second].next_V < y.first->ps[y.second].next_V;
            });
          }
          a = e;
        }
      }
      // build the next round's groups by midpoint insertion on the device
      std::vector<Group*> next;
      size_t i = 0;
      while (i < pending.size()) {
        Group* src = pending[i].first;
        groups_.emplace_back(new Group());
        Group& ng = *groups_.back();
        std::vector<int> srcm;
        size_t segs = 0;
        srcm.reserve(pending.size() - i);
        ng.orig.reserve(pending.size() - i);
        ng.seg_off.reserve(pending.size() - i + 1);
        ng.seg_off.push_back(0);
        while (i < pending.size() && pending[i].first == src) {
          const int m = pending[i].second;
          const int newS = src->ps[m].next_V - 1;
          if (!srcm.empty() && segs + newS > seg_budget) break;
          srcm.push_back(m);
          ng.orig.push_back(src->orig[m]);
          ng.seg_off.push_back(ng.seg_off.back() + newS);
          segs += newS;
          ++i;
        }
        ng.B = (int)srcm.size();
        ng.totS = ng.seg_off.back();
        ng.totV = ng.totS + ng.B;
        alloc_group_outputs(ng, src->d_init14 != nullptr);
        int* d_src = scratch_.template alloc<int>(ng.B);
        be_.h2d(d_src, srcm.data(), sizeof(int) * ng.B);
        be_.for_each(ng.B, SubdivideFillFn{src->bp, src->d_seg_ok, d_src, ng.d_seg_off, ng.d_wp, ng.d_stop, ng.d_init14, P.first_segment_checked});
        launches(1);
        be_.sync();  // d_src lives in scratch, which the next find_group resets
        next.push_back(&ng);
      }
      current.swap(next);
      trace_report("sort + next groups", round, tn);
    }
    run_deferred();
    if (early.host) be_.copy_join();
  }

  // sizes of the ragged outputs of the last optimize_batch: totals[0] = segments, totals[1] = samples
  void output_sizes(long long* totals, const Result* results) const {
    long long s = 0, m = 0;
    for (int p = 0; p < B_; ++p) {
      if (final_group_[p] < 0) continue;
      s += results[p].n_waypoints - 1;
      m += results[p].n_samples;
    }
    totals[0] = s;
    totals[1] = m;
  }

  // Gathers the final outputs into contiguous ragged arrays and copies them to host buffers (any may be null).
  void fetch_outputs(const Result* results, int* seg_off_out, double* wp_out, double* times_out, double* coef_out, int* smp_off_out,
                     double* samples_out) {
    const int B = B_;
    std::vector<int> so(B + 1, 0), mo(B + 1, 0);
    for (int p = 0; p < B; ++p) {
      const bool have = final_group_[p] >= 0;
      so[p + 1] = so[p] + (have ? results[p].n_waypoints - 1 : 0);
      mo[p + 1] = mo[p] + (have ? results[p].n_samples : 0);
    }
    if (seg_off_out) std::memcpy(seg_off_out, so.data(), sizeof(int) * (B + 1));
    if (smp_off_out) std::memcpy(smp_off_out, mo.data(), sizeof(int) * (B + 1));
    const long long totS = so[B], totM = mo[B];
    scratch_.reset();
    double* o_wp = wp_out ? scratch_.template alloc<double>((size_t)(totS + B) * 4) : nullptr;
    double* o_times = times_out ? scratch_.template alloc<double>((size_t)std::max<long long>(totS, 1)) : nullptr;
    double* o_coef = coef_out ? scratch_.template alloc<double>((size_t)std::max<long long>(totS, 1) * TG_D * TG_N) : nullptr;
    double* o_xyzh = samples_out ? scratch_.template alloc<double>((size_t)std::max<long long>(totM, 1) * 4) : nullptr;
    // problems without any result (S < 1) still own one vertex slot in the output numbering: vertex offset = so[p] + p
    for (size_t gi = 0; gi < groups_.size(); ++gi) {
      Group& g = *groups_[gi];
      std::vector<int> dst(3 * (size_t)g.B);
      bool any = false;
      for (int m = 0; m < g.B; ++m) {
        const int p = g.orig[m];
        const bool fin = final_group_[p] == (int)gi;
        dst[m] = fin ? so[p] : -1;
        dst[g.B + m] = fin ? so[p] + p : -1;
        dst[2 * g.B + m] = fin ? mo[p] : -1;
        any = any || fin;
      }
      if (!any) continue;
      int* d_dst = scratch_.template alloc<int>(dst.size());
      be_.h2d(d_dst, dst.data(), sizeof(int) * dst.size());
      be_.for_each((size_t)g.B * 32, GatherFn{g.d_seg_off, g.d_smp_off, g.d_ps, d_dst, d_dst + g.B, d_dst + 2 * g.B, g.d_wp, g.d_times, g.d_coef,
                                               g.d_xyzh, o_wp, o_times, o_coef, o_xyzh});
      launches(1);
    }
    if (wp_out) be_.d2h(wp_out, o_wp, sizeof(double) * 4 * (size_t)(totS + B));
    if (times_out && totS) be_.d2h(times_out, o_times, sizeof(double) * (size_t)totS);
    if (coef_out && totS) be_.d2h(coef_out, o_coef, sizeof(double) * (size_t)totS * TG_D * TG_N);
    if (samples_out && totM) be_.d2h(samples_out, o_xyzh, sizeof(double) * 4 * (size_t)totM);
  }


  // ===============================================================================================================
  // Class-level pieces (PolynomialOptimization / Trajectory / sampling) on caller-supplied data
  // ===============================================================================================================
  struct Bare {
    BatchPtrs b;
    int* d_seg_off;
  };
  // device batch skeleton from host segment offsets (scratch arena)
  Bare bare_batch(int B, const int* seg_off, int r) {
    Bare o;
    BatchPtrs& b = o.b;
    std::memset(&b, 0, sizeof(b));
    b.B = B; b.totS = seg_off[B]; b.totV = b.totS + B; b.r = r;
    o.d_seg_off = scratch_.template alloc<int>((size_t)B + 1);
    be_.h2d(o.d_seg_off, seg_off, sizeof(int) * (B + 1));
    b.seg_off = o.d_seg_off;
    int* pov = scratch_.template alloc<int>(b.totV);
    int* pos = scratch_.template alloc<int>(std::max(b.totS, 1));
    b.prob_of_vtx = pov; b.prob_of_seg = pos;
    b.ps = scratch_.template alloc<ProbState>(B);
    b.stats = scratch_.template alloc<int>(16);
    be_.dev_memset(b.stats, 0, 16 * sizeof(int));
    be_.for_each(B, VtxProblemFn{o.d_seg_off, pov, pos});
    be_.for_each(B, InitStateFn{b.ps});
    launches(2);
    return o;
  }

  // PolynomialOptimization<10>::setupFromVertices + solveLinear + getSegments + computeCost for B problems
  bool linear_batch(int B, const int* vtx_off, const uint8_t* vmask, const double* vval, const double* times, int r, double* coef, double* cost) {
    scratch_.reset();
    std::vector<int> so(B + 1);
    for (int p = 0; p <= B; ++p) so[p] = vtx_off[p] - p;
    for (int p = 0; p < B; ++p)
      if (so[p + 1] - so[p] < 1) return false;
    Bare bb = bare_batch(B, so.data(), r);
    BatchPtrs& b = bb.b;
    b.vmask = scratch_.template alloc<uint8_t>(b.totV);
    b.vval = scratch_.template alloc<double>((size_t)b.totV * TG_HALF * TG_D);
    b.vfree = scratch_.template alloc<int>((size_t)b.totV + B);
    b.np = scratch_.template alloc<int>(B);
    b.hbw = scratch_.template alloc<int>(B);
    b.fmax = scratch_.template alloc<int>(B);
    b.times = scratch_.template alloc<double>(b.totS);
    b.coef = scratch_.template alloc<double>((size_t)b.totS * TG_D * TG_N);
    b.recs = scratch_.template alloc<double>((size_t)b.totS * TG_REC_SIZE);
    double* d_cost = scratch_.template alloc<double>(B);
    be_.h2d(b.vmask, vmask, b.totV);
    be_.h2d(b.vval, vval, sizeof(double) * (size_t)b.totV * TG_HALF * TG_D);
    be_.h2d(b.times, times, sizeof(double) * b.totS);
    be_.for_each(B, PrepareFn{b, 0});
    int stats[16];
    be_.d2h(stats, b.stats, sizeof(stats));
    alloc_solution_buffers(b, (size_t)B, stats);
    be_.for_each(b.totS, SetupBaseFn{b, b.times});
    solve_with_outputs((size_t)B, stats, SolveProblemDesc{b, 0, nullptr, nullptr}, b);
    be_.for_each(B, CostOutFn{b.ps, d_cost});
    launches(4);
    counters.solves += B;
    counters.segment_setups += b.totS;
    if (coef) be_.d2h(coef, b.coef, sizeof(double) * (size_t)b.totS * TG_D * TG_N);
    if (cost) be_.d2h(cost, d_cost, sizeof(double) * B);
    return true;
  }

  // Solutions of the reduced systems and partial costs travel from the solve kernels to CoefCostFn / CostSumFn through
  // these buffers (per instance: 4 * max n_p doubles and 4 * max S doubles).
  void alloc_solution_buffers(BatchPtrs& b, size_t n_inst_max, const int* stats) {
    b.xstride = 4 * std::max(stats[3], 1);
    b.smax = std::max(stats[4], 1);
    b.xs = scratch_.template alloc<double>(std::max<size_t>(n_inst_max, 1) * (size_t)b.xstride);
    b.part = scratch_.template alloc<double>(std::max<size_t>(n_inst_max, 1) * 4 * (size_t)b.smax);
  }
  // A run of consecutive problems whose solve workspaces fall into the same occupancy class of the backend
  // (BE::solve_class): each run is launched with its own shared-memory size, so that a few long paths in a group do
  // not take the resident warps away from all the short ones (profiles/r01_solve_octet_s3.md).
  struct SolveBucket {
    int p0, p1;      // problems [p0, p1)
    size_t v0, v1;   // their vertices = Mellinger instances
    int ws, ows;     // workspace sizes (doubles): warp-per-instance routine, octet routine (0: not eligible)
    int np_cap;      // largest number of unknowns in the run
    int s_cap;       // largest number of segments in the run
    int kernel_cls;  // BE::solve_class of its members: consecutive runs of one class share a solve launch
  };
  std::vector<SolveBucket> make_buckets(int B, const int* seg_off, const int* np, const int* hbw, int ws_all, int ows_all, int np_all) const {
    std::vector<SolveBucket> out;
    int cls_prev = 0;
    for (int p = 0; p < B; ++p) {
      const int S = seg_off[p + 1] - seg_off[p];
      const int ws = solve_ws_doubles(S, np[p], hbw[p]);
      const int ows = (hbw[p] == kOctHbw && np[p] >= kOctMinNp) ? octet_ws_doubles(S, np[p]) : 0;
      // same kernel and resident warps (solve_class), and segment counts within one group of four: the U slab and the
      // coefficient kernel's thread count are sized by the largest member of a run
      const int cls = be_.solve_class(ws, ows) * 4096 + (S + 3) / 4;
      if (out.empty() || cls != cls_prev) {
        if (out.size() >= 32) {  // ragged input in no particular order: one launch pair for everything, sized by the batch maxima
          out.assign(1, SolveBucket{0, B, 0, (size_t)seg_off[B] + B, ws_all, ows_all, np_all, 0, 0});
          mixed_single_ = true;
          return out;
        }
        out.push_back(SolveBucket{p, p, (size_t)seg_off[p] + p, 0, 0, 0, 0, 0, cls / 4096});
        cls_prev = cls;
      }
      SolveBucket& k = out.back();
      k.p1 = p + 1;
      k.v1 = (size_t)seg_off[p + 1] + p + 1;
      k.ws = std::max(k.ws, ws);
      k.ows = std::max(k.ows, ows);
      k.np_cap = std::max(k.np_cap, np[p]);
      k.s_cap = std::max(k.s_cap, S);
    }
    mixed_single_ = false;
    return out;
  }
  mutable bool mixed_single_ = false;
  // stats: b.stats read back (0: ws, 2: octet ws, 3: max np, 6: problems the octet routine cannot take)
  template <class D>
  void solve_with_outputs(size_t n_inst, const int* stats, const D& desc, const BatchPtrs& b, const std::vector<SolveBucket>* buckets = nullptr,
                          bool per_vertex = false) {
    // thread-per-instance kernel for every instance it can take (at most four free derivatives per vertex: the node's
    // recipe always); the older kernels below then only see the rest (stats[8] = how many problems that is)
    const bool use_thr = thread_solve_for(n_inst);
    const bool thread_all = use_thr && stats[8] == 0;
    if (use_thr) {
      be_.solve_thread(0, n_inst, kThrB * (std::max(b.smax, 1) + 1), desc);
      launches(1);
    }
    be_.skip_thread_eligible = use_thr;
    if (thread_all) {
      // nothing left for the lane-parallel kernels
    } else if (buckets && !buckets->empty()) {
      // one solve launch per stretch of runs that go to the same kernel at the same residency (many small launches cost more
      // in tails than tighter slabs gain: measured); a run is homogeneous by construction unless it is the collapsed one
      const bool mixed = mixed_single_;
      size_t a = 0;
      int n_launch = 0;
      while (a < buckets->size()) {
        SolveBucket m = (*buckets)[a];
        size_t e = a + 1;
        while (e < buckets->size() && (*buckets)[e].kernel_cls == m.kernel_cls) {
          const SolveBucket& k = (*buckets)[e];
          m.p1 = k.p1;
          m.v1 = k.v1;
          m.ws = std::max(m.ws, k.ws);
          m.ows = std::max(m.ows, k.ows);
          m.np_cap = std::max(m.np_cap, k.np_cap);
          ++e;
        }
        if (per_vertex) be_.solve(m.v0, m.v1, m.ws, m.ows, m.np_cap, mixed, desc);
        else be_.solve((size_t)m.p0, (size_t)m.p1, m.ws, m.ows, m.np_cap, mixed, desc);
        ++n_launch;
        a = e;
      }
      launches(n_launch - 1);
    } else {
      be_.solve(0, n_inst, stats[0], stats[2], stats[3], stats[6] > 0, desc);
    }
    // coefficients + partial costs: one thread per (instance, segment, dimension); with runs, each run is launched over
    // its own largest segment count instead of the group's
    const int per = 4 * b.smax;
    if (coef_cost_by_problem(n_inst, desc, b, buckets, per)) {
      // all points of a Mellinger evaluation: one CTA per problem (CoefCostGradFn)
    } else if (buckets && buckets->size() > 1) {
      for (const SolveBucket& k : *buckets) {
        const size_t i0 = per_vertex ? k.v0 : (size_t)k.p0, i1 = per_vertex ? k.v1 : (size_t)k.p1;
        const int items = 4 * std::max(k.s_cap, 1);
        be_.for_each((i1 - i0) * (size_t)items, CoefCostFn<D>{desc, per, b.part, i0, items});
      }
      launches((int)buckets->size() - 1);
    } else {
      be_.for_each(n_inst * (size_t)per, CoefCostFn<D>{desc, per, b.part, 0, per});
    }
    be_.for_each(n_inst, CostSumFn<D>{desc, per, b.part, nullptr});
    launches(2);
  }

  template <class D>
  bool coef_cost_by_problem(size_t, const D&, const BatchPtrs&, const std::vector<SolveBucket>*, int) { return false; }
  bool coef_cost_by_problem(size_t, const SolveProblemDesc& desc, const BatchPtrs& b, const std::vector<SolveBucket>*, int per) {
    if (desc.mellinger != 1) return false;
    be_.for_each((size_t)b.B * 128, CoefCostGradFn{CoefCostFn<SolveProblemDesc>{desc, per, b.part, 0, per}, 0, nullptr});
    return true;
  }

  // PolynomialOptimizationNonLinear<10>::optimize() for every problem of the batch: Mellinger outer loop (nl_impl.h:159-234,
  // objective + forward-difference gradient 256-333 as S+1 batched solves per evaluation) then the time scaling of
  // scaleSegmentTimesWithViolation (335-427).  Needs b.times (initial), vmask/vval/vfree/np/hbw, coef, ps; leaves the
  // stretched times in b.times (the caller runs the final solve).
  void time_alloc_core(BatchPtrs& b, const Params& P, const int* stats, const std::vector<SolveBucket>* buckets = nullptr) {
    const int B = b.B, totS = b.totS, totV = b.totV;
    const int mf = (P.max_evals > 0) ? std::min(std::max(P.max_evals, 1), kPlisMfMax) : kPlisMfMax;
    b.xeval = scratch_.template alloc<double>(totS);
    b.x = scratch_.template alloc<double>(totS);
    b.g = scratch_.template alloc<double>(totS);
    b.d = scratch_.template alloc<double>(totS);
    b.ix = scratch_.template alloc<int>(totS);
    b.hist_s = scratch_.template alloc<double>((size_t)mf * totS);
    b.hist_y = scratch_.template alloc<double>((size_t)mf * totS);
    b.opt = scratch_.template alloc<PlisScalars>(B);
    b.recs = scratch_.template alloc<double>((size_t)totS * 3 * TG_REC_SIZE);
    b.costs = scratch_.template alloc<double>(totV);
    b.maxima = scratch_.template alloc<double>((size_t)totS * 9);
    for (int k = 0; k < 2; ++k) {
      b.act_prob[k] = scratch_.template alloc<int>(B);
      b.act_vtx[k] = scratch_.template alloc<int>(totV);
      b.act_seg[k] = scratch_.template alloc<int>(totS);
    }
    be_.dev_memset(b.stats + 9, 0, 6 * sizeof(int));
    be_.for_each(B, PlisBeginFn{b, P.max_evals}); launches(1);
    // One evaluation = S+1 linear solves per running problem: the point itself and its S perturbed neighbours
    // (nl_impl.h:282-323).  PLIS consumes the gradient of EVERY evaluation (the directional derivative at each line-search
    // trial decides between acceptance, extrapolation and interpolation), so all of them are computed.  maxeval is tested
    // between iterations only, so a line search may overrun it: loop until no problem is left running.
    // Most problems stop after three or four evaluations; the tail runs for up to ~30.  Once fewer than half of the
    // problems are left, the launches walk the work lists that PlisAdvanceFn wrote for them (problems, solve instances,
    // segments still running) instead of scanning the whole batch for the few that are.
    const int eval_cap = (P.max_evals > 0 ? P.max_evals : 1000) + 64;
    int cnt[3] = {B, totV, totS};
    const bool lists_ok = thread_solve_for((size_t)totV) && stats[8] == 0;  // the lane-parallel kernels scan (done problems drop out at once)
    for (int e = 0; e < eval_cap; ++e) {
      const int buf = e & 1, nbuf = buf ^ 1;
      const bool sparse = lists_ok && e > 0 && (size_t)cnt[0] * 2 < (size_t)B;
      be_.dev_memset(b.stats + 7, 0, sizeof(int));
      be_.dev_memset(b.stats + 9 + 3 * nbuf, 0, 3 * sizeof(int));
      if (sparse) {
        const SolveProblemDesc desc{b, 1, nullptr, nullptr};
        const int per = 4 * b.smax;
        be_.for_each((size_t)cnt[2] * 3, SetupMellingerFn<0>{b, b.act_seg[buf]});
        be_.for_each((size_t)cnt[2] * 3 * TG_N, SetupMellingerFn<1>{b, b.act_seg[buf]});
        if ((size_t)cnt[1] >= list_octet_below) {
          be_.solve_thread(0, (size_t)cnt[1], kThrB * (std::max(b.smax, 1) + 1), SolveProblemListDesc{desc, b.act_vtx[buf]});
        } else {
          // a short list is latency bound: eight lanes per system finish sooner than one thread per system
          be_.skip_thread_eligible = false;
          be_.solve(0, (size_t)cnt[1], stats[0], stats[2], stats[3], stats[6] > 0, SolveProblemListDesc{desc, b.act_vtx[buf]});
        }
        be_.for_each((size_t)cnt[0] * 128, CoefCostGradFn{CoefCostFn<SolveProblemDesc>{desc, per, b.part, 0, per}, 0, b.act_prob[buf]});
        be_.for_each((size_t)cnt[1], CostSumFn<SolveProblemDesc>{desc, per, b.part, b.act_vtx[buf]});
        be_.for_each((size_t)cnt[0], PlisAdvanceFn{b, P.max_evals, P.f_rel, P.x_rel, b.act_prob[buf], nbuf});
        launches(6);
      } else {
        be_.for_each((size_t)totS * 3, SetupMellingerFn<0>{b, nullptr});
        be_.for_each((size_t)totS * 3 * TG_N, SetupMellingerFn<1>{b, nullptr});
        solve_with_outputs((size_t)totV, stats, SolveProblemDesc{b, 1, nullptr, nullptr}, b, buckets, true);
        be_.for_each(B, PlisAdvanceFn{b, P.max_evals, P.f_rel, P.x_rel, nullptr, nbuf});
        launches(4);
      }
      counters.mellinger_launches += 1;
      run_deferred();  // the previous round's result records: host stores while the device runs this evaluation
      int back[8];  // stats[7 .. 14]
      be_.d2h(back, b.stats + 7, sizeof(back));
      if (back[0] == 0) break;
      cnt[0] = back[2 + 3 * nbuf];
      cnt[1] = back[3 + 3 * nbuf];
      cnt[2] = back[4 + 3 * nbuf];
    }
    be_.for_each(B, PlisFinishFn{b}); launches(1);
    // time scaling (nl_impl.h:335-427 -> eth/trajectory.cpp:598-692)
    scale_loop(b, P.limits);
  }

  // PolynomialOptimizationNonLinear<10>::setupFromVertices + addMaximumMagnitudeConstraint + optimize() + getTrajectory
  // for B problems given as vertices (masks / fixed values) and initial segment times.
  bool time_alloc_batch(int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times, const Params& P, double* coef,
                        int* nlopt_code, int* n_evals, int* n_scale_passes, double* final_cost) {
    scratch_.reset();
    std::vector<int> so(B + 1);
    for (int p = 0; p <= B; ++p) so[p] = vtx_off[p] - p;
    for (int p = 0; p < B; ++p)
      if (so[p + 1] - so[p] < 1) return false;
    Bare bb = bare_batch(B, so.data(), P.derivative_to_optimize);
    BatchPtrs& b = bb.b;
    b.vmask = scratch_.template alloc<uint8_t>(b.totV);
    b.vval = scratch_.template alloc<double>((size_t)b.totV * TG_HALF * TG_D);
    b.vfree = scratch_.template alloc<int>((size_t)b.totV + B);
    b.np = scratch_.template alloc<int>(B);
    b.hbw = scratch_.template alloc<int>(B);
    b.fmax = scratch_.template alloc<int>(B);
    b.times = scratch_.template alloc<double>(b.totS);
    b.coef = scratch_.template alloc<double>((size_t)b.totS * TG_D * TG_N);
    be_.h2d(b.vmask, vmask, b.totV);
    be_.h2d(b.vval, vval, sizeof(double) * (size_t)b.totV * TG_HALF * TG_D);
    be_.h2d(b.times, times, sizeof(double) * b.totS);
    be_.for_each(B, PrepareFn{b, 0}); launches(1);
    int stats[16];
    be_.d2h(stats, b.stats, sizeof(stats));
    alloc_solution_buffers(b, (size_t)b.totV, stats);
    time_alloc_core(b, P, stats);
    be_.for_each(b.totS, SetupBaseFn{b, b.times});
    solve_with_outputs((size_t)B, stats, SolveProblemDesc{b, 0, nullptr, nullptr}, b);
    launches(2);
    std::vector<ProbState> ps(B);
    be_.d2h(ps.data(), b.ps, sizeof(ProbState) * B);
    for (int p = 0; p < B; ++p) {
      if (nlopt_code) nlopt_code[p] = ps[p].nlopt_code;
      if (n_evals) n_evals[p] = ps[p].n_evals;
      if (n_scale_passes) n_scale_passes[p] = ps[p].n_scale_passes;
      if (final_cost) final_cost[p] = ps[p].final_cost;
      const int S = so[p + 1] - so[p];
      counters.evals += ps[p].n_evals;
      counters.solves += (long long)ps[p].n_evals * (S == 1 ? 1 : S + 1) + 1;
    }
    be_.d2h(times, b.times, sizeof(double) * b.totS);
    if (coef) be_.d2h(coef, b.coef, sizeof(double) * (size_t)b.totS * TG_D * TG_N);
    return true;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // The steps either side of the path (SURVEY.md 8f): preprocessPath, findTrajectoryFallback, getWaypointInTrajectoryIdxs
  void preprocess_batch(int B, const int* wp_off, const double* wp, const uint8_t* stop, double min_dist, int straighten, double max_dev,
                        double max_hdg_dev, int* out_count, double* out_wp, uint8_t* out_stop) {
    scratch_.reset();
    const int totV = wp_off[B];
    int* d_off = scratch_.template alloc<int>((size_t)B + 1);
    double* d_wp = scratch_.template alloc<double>((size_t)std::max(totV, 1) * 4);
    uint8_t* d_stop = stop ? scratch_.template alloc<uint8_t>(std::max(totV, 1)) : nullptr;
    double* d_owp = scratch_.template alloc<double>((size_t)std::max(totV, 1) * 4);
    uint8_t* d_ostop = scratch_.template alloc<uint8_t>(std::max(totV, 1));
    int* d_cnt = scratch_.template alloc<int>(B);
    be_.h2d(d_off, wp_off, sizeof(int) * (B + 1));
    be_.h2d(d_wp, wp, sizeof(double) * 4 * (size_t)totV);
    if (stop) be_.h2d(d_stop, stop, totV);
    be_.for_each(B, PreprocessFn{d_off, d_wp, d_stop, min_dist, max_dev, max_hdg_dev, straighten, d_owp, d_ostop, d_cnt});
    launches(1);
    be_.d2h(out_count, d_cnt, sizeof(int) * B);
    if (out_wp) be_.d2h(out_wp, d_owp, sizeof(double) * 4 * (size_t)totV);
    if (out_stop) be_.d2h(out_stop, d_ostop, totV);
  }
  void fallback_batch(int B, const int* wp_off, const double* wp, const uint8_t* stop, const double* L9, double dt, double stopping_time, int* counts,
                      double* samples) {
    scratch_.reset();
    const int totV = wp_off[B];
    int* d_off = scratch_.template alloc<int>((size_t)B + 1);
    double* d_wp = scratch_.template alloc<double>((size_t)std::max(totV, 1) * 4);
    uint8_t* d_stop = stop ? scratch_.template alloc<uint8_t>(std::max(totV, 1)) : nullptr;
    double* d_vpos = scratch_.template alloc<double>((size_t)std::max(totV, 1) * 4);
    int* d_cnt = scratch_.template alloc<int>((size_t)B + 1);
    int* d_smp_off = scratch_.template alloc<int>((size_t)B + 1);
    be_.h2d(d_off, wp_off, sizeof(int) * (B + 1));
    be_.h2d(d_wp, wp, sizeof(double) * 4 * (size_t)totV);
    if (stop) be_.h2d(d_stop, stop, totV);
    FallbackFn f{d_off, d_wp, d_stop, {}, dt, stopping_time, d_vpos, d_cnt, nullptr, nullptr};
    for (int i = 0; i < 9; ++i) f.L[i] = L9[i];
    be_.for_each(B, f);
    be_.exclusive_scan(d_cnt, d_smp_off, B);
    launches(2);
    std::vector<int> off(B + 1);
    be_.d2h(off.data(), d_smp_off, sizeof(int) * (B + 1));
    for (int p = 0; p < B; ++p) counts[p] = off[p + 1] - off[p];
    if (!samples || off[B] == 0) return;
    double* d_smp = scratch_.template alloc<double>((size_t)off[B] * 4);
    f.smp_off = d_smp_off;
    f.samples = d_smp;
    be_.for_each(B, f);
    launches(1);
    be_.d2h(samples, d_smp, sizeof(double) * 4 * (size_t)off[B]);
    counters.samples += off[B];
  }
  void waypoint_idxs_batch(int B, const int* smp_off, const double* samples, const int* wp_off, const double* wp, int* counts, int* idxs) {
    scratch_.reset();
    const int totV = wp_off[B], totM = smp_off[B];
    int* d_soff = scratch_.template alloc<int>((size_t)B + 1);
    int* d_woff = scratch_.template alloc<int>((size_t)B + 1);
    double* d_smp = scratch_.template alloc<double>((size_t)std::max(totM, 1) * 4);
    double* d_wp = scratch_.template alloc<double>((size_t)std::max(totV, 1) * 4);
    int* d_idx = scratch_.template alloc<int>(std::max(totV, 1));
    int* d_cnt = scratch_.template alloc<int>(B);
    be_.h2d(d_soff, smp_off, sizeof(int) * (B + 1));
    be_.h2d(d_woff, wp_off, sizeof(int) * (B + 1));
    be_.h2d(d_smp, samples, sizeof(double) * 4 * (size_t)totM);
    be_.h2d(d_wp, wp, sizeof(double) * 4 * (size_t)totV);
    be_.for_each(B, WaypointIdxFn{d_soff, d_smp, d_woff, d_wp, d_idx, d_cnt});
    launches(1);
    be_.d2h(counts, d_cnt, sizeof(int) * B);
    be_.d2h(idxs, d_idx, sizeof(int) * totV);
  }

  // sampleWholeTrajectory for B trajectories
  void sample_batch(int B, const int* seg_off, const double* coef, const double* times, double dt, int* counts, double* samples, double* full) {
    scratch_.reset();
    Bare bb = bare_batch(B, seg_off, 2);
    BatchPtrs& b = bb.b;
    b.times = scratch_.template alloc<double>(std::max(b.totS, 1));
    b.coef = scratch_.template alloc<double>((size_t)std::max(b.totS, 1) * TG_D * TG_N);
    be_.h2d(b.times, times, sizeof(double) * b.totS);
    be_.h2d(b.coef, coef, sizeof(double) * (size_t)b.totS * TG_D * TG_N);
    int* cap = scratch_.template alloc<int>((size_t)B + 1);
    int* d_smp_off = scratch_.template alloc<int>((size_t)B + 1);
    be_.for_each(B, SampleCapFn{b, dt, cap});
    be_.exclusive_scan(cap, d_smp_off, B);
    std::vector<int> smp_off(B + 1);
    be_.d2h(smp_off.data(), d_smp_off, sizeof(int) * (B + 1));
    const size_t slots = (size_t)std::max(smp_off[B], 1);
    int* seg_idx = scratch_.template alloc<int>(slots);
    int* smp_prob = scratch_.template alloc<int>(slots);
    double* t_in = scratch_.template alloc<double>(slots);
    be_.for_each(B, SampleWalkFn{b, dt, d_smp_off, seg_idx, t_in});
    launches(3);
    std::vector<ProbState> ps(B);
    be_.d2h(ps.data(), b.ps, sizeof(ProbState) * B);
    std::vector<int> dst(B + 1, 0);
    for (int p = 0; p < B; ++p) {
      counts[p] = ps[p].n_samples;
      dst[p + 1] = dst[p] + ps[p].n_samples;
    }
    counters.samples += dst[B];
    if (!samples && !full) return;
    double* d_xyzh = scratch_.template alloc<double>(slots * 4);
    double* d_full = full ? scratch_.template alloc<double>(slots * 19) : nullptr;
    const size_t tot = (size_t)std::max(dst[B], 1);
    double* o_xyzh = samples ? scratch_.template alloc<double>(tot * 4) : nullptr;
    double* o_full = full ? scratch_.template alloc<double>(tot * 19) : nullptr;
    int* d_dst = scratch_.template alloc<int>((size_t)B + 1);
    be_.h2d(d_dst, dst.data(), sizeof(int) * (B + 1));
    be_.for_each(B, SlotProblemFn{B, d_smp_off, smp_prob});
    be_.for_each((size_t)smp_off[B], SampleEvalFn{b, d_smp_off, smp_prob, seg_idx, t_in, d_xyzh, d_full});
    be_.for_each((size_t)smp_off[B], CompactSamplesFn{d_smp_off, smp_prob, d_dst, b.ps, d_xyzh, d_full, o_xyzh, o_full});
    launches(3);
    if (samples && dst[B]) be_.d2h(samples, o_xyzh, sizeof(double) * 4 * (size_t)dst[B]);
    if (full && dst[B]) be_.d2h(full, o_full, sizeof(double) * 19 * (size_t)dst[B]);
  }

  // Trajectory::evaluate at n times of one trajectory
  void evaluate_batch(int S, const double* coef, const double* times, int n, const double* t, int deriv, double* out, uint8_t* ok) {
    scratch_.reset();
    double* d_coef = scratch_.template alloc<double>((size_t)S * TG_D * TG_N);
    double* d_T = scratch_.template alloc<double>(S);
    double* d_t = scratch_.template alloc<double>(std::max(n, 1));
    double* d_out = scratch_.template alloc<double>((size_t)std::max(n, 1) * 4);
    uint8_t* d_ok = scratch_.template alloc<uint8_t>(std::max(n, 1));
    be_.h2d(d_coef, coef, sizeof(double) * (size_t)S * TG_D * TG_N);
    be_.h2d(d_T, times, sizeof(double) * S);
    be_.h2d(d_t, t, sizeof(double) * n);
    be_.for_each(n, EvaluateFn{S, deriv, d_coef, d_T, d_t, d_out, d_ok});
    launches(1);
    be_.d2h(out, d_out, sizeof(double) * 4 * (size_t)n);
    if (ok) be_.d2h(ok, d_ok, n);
  }

  // per-segment maxima of |v|,|a|,|j| for the three dimension groups
  void extrema_batch(int totS, const double* coef, const double* times, double* maxima) {
    scratch_.reset();
    double* d_coef = scratch_.template alloc<double>((size_t)totS * TG_D * TG_N);
    double* d_T = scratch_.template alloc<double>(totS);
    double* d_m = scratch_.template alloc<double>((size_t)totS * 9);
    be_.h2d(d_coef, coef, sizeof(double) * (size_t)totS * TG_D * TG_N);
    be_.h2d(d_T, times, sizeof(double) * totS);
    ExtremaScratch es = extrema_scratch((size_t)totS);
    extrema_segments(d_coef, d_T, d_m, (size_t)totS, nullptr, nullptr, es);
    counters.root_finds += (long long)totS * 9;
    be_.d2h(maxima, d_m, sizeof(double) * (size_t)totS * 9);
  }

  // test hook: the device Jenkins-Traub on n arbitrary polynomials (<= 16 coefficients each, increasing powers)
  void find_roots_batch(int n, const double* coeffs, const int* ncoef, double* re, double* im, int* nroots) {
    scratch_.reset();
    double* d_c = scratch_.template alloc<double>((size_t)n * 16);
    int* d_n = scratch_.template alloc<int>(n);
    double* d_re = scratch_.template alloc<double>((size_t)n * 16);
    double* d_im = scratch_.template alloc<double>((size_t)n * 16);
    int* d_nr = scratch_.template alloc<int>(n);
    be_.h2d(d_c, coeffs, sizeof(double) * (size_t)n * 16);
    be_.h2d(d_n, ncoef, sizeof(int) * n);
    be_.dev_memset(d_re, 0, sizeof(double) * (size_t)n * 16);
    be_.dev_memset(d_im, 0, sizeof(double) * (size_t)n * 16);
    be_.for_each_scratch((size_t)n, FindRootsFn{d_c, d_n, d_re, d_im, d_nr});
    launches(1);
    be_.d2h(re, d_re, sizeof(double) * (size_t)n * 16);
    be_.d2h(im, d_im, sizeof(double) * (size_t)n * 16);
    be_.d2h(nroots, d_nr, sizeof(int) * n);
  }

  // PolynomialOptimization<10>::computeMaximumOfMagnitude(derivative) for B trajectories (lin_impl.h:477-508)
  bool max_magnitude_batch(int B, const int* seg_off, const double* coef, const double* times, int derivative, double* value, double* time,
                           int* segment_idx) {
    if (derivative < 1 || derivative > 4) return false;
    scratch_.reset();
    const int totS = seg_off[B];
    int* d_off = scratch_.template alloc<int>((size_t)B + 1);
    double* d_coef = scratch_.template alloc<double>((size_t)totS * TG_D * TG_N);
    double* d_T = scratch_.template alloc<double>(totS);
    double* d_sv = scratch_.template alloc<double>(totS);
    double* d_st = scratch_.template alloc<double>(totS);
    double* d_v = scratch_.template alloc<double>(B);
    double* d_t = scratch_.template alloc<double>(B);
    int* d_i = scratch_.template alloc<int>(B);
    be_.h2d(d_off, seg_off, sizeof(int) * ((size_t)B + 1));
    be_.h2d(d_coef, coef, sizeof(double) * (size_t)totS * TG_D * TG_N);
    be_.h2d(d_T, times, sizeof(double) * totS);
    switch (derivative) {
      case 1: be_.for_each_scratch((size_t)totS, MaxMagnitudeSegFn<1>{d_coef, d_T, d_sv, d_st}); break;
      case 2: be_.for_each_scratch((size_t)totS, MaxMagnitudeSegFn<2>{d_coef, d_T, d_sv, d_st}); break;
      case 3: be_.for_each_scratch((size_t)totS, MaxMagnitudeSegFn<3>{d_coef, d_T, d_sv, d_st}); break;
      default: be_.for_each_scratch((size_t)totS, MaxMagnitudeSegFn<4>{d_coef, d_T, d_sv, d_st}); break;
    }
    be_.for_each((size_t)B, MaxMagnitudeReduceFn{d_off, d_sv, d_st, d_v, d_t, d_i});
    launches(2);
    counters.root_finds += totS;
    counters.root_finds_executed += totS;
    be_.d2h(value, d_v, sizeof(double) * B);
    be_.d2h(time, d_t, sizeof(double) * B);
    be_.d2h(segment_idx, d_i, sizeof(int) * B);
    return true;
  }

  // Trajectory::scaleSegmentTimesToMeetConstraints in place
  void scale_times_batch(int B, const int* seg_off, double* coef, double* times, const double* L9, int* passes, uint8_t* within) {
    scratch_.reset();
    Bare bb = bare_batch(B, seg_off, 2);
    BatchPtrs& b = bb.b;
    b.times = scratch_.template alloc<double>(b.totS);
    b.coef = scratch_.template alloc<double>((size_t)b.totS * TG_D * TG_N);
    b.maxima = scratch_.template alloc<double>((size_t)b.totS * 9);
    be_.h2d(b.times, times, sizeof(double) * b.totS);
    be_.h2d(b.coef, coef, sizeof(double) * (size_t)b.totS * TG_D * TG_N);
    ScaleOutFn of{b.ps, b.maxima, bb.d_seg_off, {}, nullptr, nullptr, scale_tolerance};
    for (int i = 0; i < 9; ++i) of.L[i] = L9[i];
    scale_loop(b, L9);
    int* d_passes = scratch_.template alloc<int>(B);
    uint8_t* d_within = scratch_.template alloc<uint8_t>(B);
    of.passes = d_passes;
    of.within = d_within;
    be_.for_each(B, of); launches(1);
    be_.d2h(coef, b.coef, sizeof(double) * (size_t)b.totS * TG_D * TG_N);
    be_.d2h(times, b.times, sizeof(double) * b.totS);
    if (passes) be_.d2h(passes, d_passes, sizeof(int) * B);
    if (within) be_.d2h(within, d_within, B);
  }

  // cost of ONE problem at K candidate segment-time vectors + first-minimum argmin
  bool sweep_costs(int V, const uint8_t* vmask, const double* vval, int r, long long K, const double* cand, bool cand_on_device, double* costs,
                   long long* best_index, double* best_cost) {
    scratch_.reset();
    const int S = V - 1;
    if (S < 1 || K < 1) return false;
    const int so[2] = {0, S};
    Bare bb = bare_batch(1, so, r);
    BatchPtrs& b = bb.b;
    b.vmask = scratch_.template alloc<uint8_t>(V);
    b.vval = scratch_.template alloc<double>((size_t)V * TG_HALF * TG_D);
    b.vfree = scratch_.template alloc<int>((size_t)V + 1);
    b.np = scratch_.template alloc<int>(1);
    b.hbw = scratch_.template alloc<int>(1);
    b.fmax = scratch_.template alloc<int>(1);
    be_.h2d(b.vmask, vmask, V);
    be_.h2d(b.vval, vval, sizeof(double) * (size_t)V * TG_HALF * TG_D);
    be_.for_each(1, PrepareFn{b, 0}); launches(1);
    int stats[16];
    be_.d2h(stats, b.stats, sizeof(stats));
    const long long chunk = std::min<long long>(K, (long long)sweep_chunk);
    alloc_solution_buffers(b, (size_t)chunk, stats);
    double* d_recs = scratch_.template alloc<double>((size_t)chunk * S * TG_REC_SIZE);
    double* d_costs = scratch_.template alloc<double>((size_t)K);
    const double* d_cand = cand;
    if (!cand_on_device) {
      double* dc = scratch_.template alloc<double>((size_t)K * S);
      be_.h2d(dc, cand, sizeof(double) * (size_t)K * S);
      d_cand = dc;
    }
    for (long long k0 = 0; k0 < K; k0 += chunk) {
      const long long kc = std::min(chunk, K - k0);
      be_.for_each((size_t)kc * S, SetupSweepFn{S, r, d_cand + (size_t)k0 * S, d_recs});
      solve_with_outputs((size_t)kc, stats, SolveSweepDesc{b, d_recs, d_costs + k0}, b);
      launches(2);
    }
    counters.solves += K;
    counters.segment_setups += K * S;
    const long long nchunks = (K + 1023) / 1024;
    double* d_cmin = scratch_.template alloc<double>((size_t)nchunks);
    long long* d_cidx = scratch_.template alloc<long long>((size_t)nchunks);
    be_.for_each((size_t)nchunks, ArgminChunkFn{K, d_costs, d_cmin, d_cidx}); launches(1);
    std::vector<double> cmin(nchunks);
    std::vector<long long> cidx(nchunks);
    be_.d2h(cmin.data(), d_cmin, sizeof(double) * nchunks);
    be_.d2h(cidx.data(), d_cidx, sizeof(long long) * nchunks);
    long long bi = cidx[0];
    double bc = cmin[0];
    for (long long c = 1; c < nchunks; ++c)
      if (cmin[c] < bc) { bc = cmin[c]; bi = cidx[c]; }
    if (best_index) *best_index = bi;
    if (best_cost) *best_cost = bc;
    if (costs) be_.d2h(costs, d_costs, sizeof(double) * (size_t)K);
    return true;
  }
  // objectiveFunctionTime / objectiveFunctionTimeAndConstraints (nl_impl.h:567-722) of ONE problem at K candidate vectors.
  // method 0/1: x = S times (update + solve); 3/4: x = S times + 4 * n_free free derivatives (update + setFreeConstraints).
  // Returns 0, or a negative value: -1 bad sizes / method, -2 nvar does not match the problem, -3 too many / bad constraints.
  int objective_batch(int V, const uint8_t* vmask, const double* vval, int r, int method, long long K, const double* x, int nvar,
                      double time_penalty, int use_soft, double soft_weight, int ncon, const int* con_deriv, const double* con_value,
                      double* total, double* parts, double* coef) {
    scratch_.reset();
    const int S = V - 1;
    if (S < 1 || K < 1 || !(method == 0 || method == 1 || method == 3 || method == 4)) return -1;
    if (ncon < 0 || ncon > 16) return -3;
    bool need[4] = {false, false, false, false};
    for (int c = 0; c < ncon; ++c) {
      if (con_deriv[c] < 1 || con_deriv[c] > 4 || !(con_value[c] != 0.0)) return -3;
      need[con_deriv[c] - 1] = true;
    }
    const int so[2] = {0, S};
    Bare bb = bare_batch(1, so, r);
    BatchPtrs& b = bb.b;
    b.vmask = scratch_.template alloc<uint8_t>(V);
    b.vval = scratch_.template alloc<double>((size_t)V * TG_HALF * TG_D);
    b.vfree = scratch_.template alloc<int>((size_t)V + 1);
    b.np = scratch_.template alloc<int>(1);
    b.hbw = scratch_.template alloc<int>(1);
    b.fmax = scratch_.template alloc<int>(1);
    be_.h2d(b.vmask, vmask, V);
    be_.h2d(b.vval, vval, sizeof(double) * (size_t)V * TG_HALF * TG_D);
    be_.for_each(1, PrepareFn{b, 0}); launches(1);
    int stats[16];
    be_.d2h(stats, b.stats, sizeof(stats));
    const int n_free = stats[3];
    if (nvar != ((method >= 3) ? S + TG_D * n_free : S)) return -2;
    const long long chunk = std::min<long long>(K, (long long)objective_chunk);
    alloc_solution_buffers(b, (size_t)chunk, stats);
    double* d_recs = scratch_.template alloc<double>((size_t)chunk * S * TG_REC_SIZE);
    double* d_T = scratch_.template alloc<double>((size_t)chunk * S);
    double* d_coef = scratch_.template alloc<double>((size_t)chunk * S * TG_D * TG_N);
    double* d_x = scratch_.template alloc<double>((size_t)chunk * nvar);
    double* d_costs = scratch_.template alloc<double>((size_t)chunk);
    double* d_sv = scratch_.template alloc<double>((size_t)chunk * S);
    double* d_st = scratch_.template alloc<double>((size_t)chunk * S);
    double* d_max = scratch_.template alloc<double>((size_t)4 * chunk);
    double* d_mt = scratch_.template alloc<double>((size_t)chunk);
    int* d_mi = scratch_.template alloc<int>((size_t)chunk);
    int* d_off = scratch_.template alloc<int>((size_t)chunk + 1);
    double* d_total = scratch_.template alloc<double>((size_t)chunk);
    double* d_parts = parts ? scratch_.template alloc<double>((size_t)chunk * 3) : nullptr;
    {
      std::vector<int> off((size_t)chunk + 1);
      for (long long k = 0; k <= chunk; ++k) off[(size_t)k] = (int)(k * S);
      be_.h2d(d_off, off.data(), sizeof(int) * ((size_t)chunk + 1));
    }
    for (long long k0 = 0; k0 < K; k0 += chunk) {
      const long long kc = std::min(chunk, K - k0);
      be_.h2d(d_x, x + (size_t)k0 * nvar, sizeof(double) * (size_t)kc * nvar);
      be_.for_each((size_t)kc * S, SetupObjFn{S, r, nvar, d_x, d_recs, d_T});
      launches(1);
      SolveSweepDesc desc{b, d_recs, d_costs, d_coef};
      if (method >= 3) {
        if (n_free > 0) be_.for_each((size_t)kc * n_free * TG_D, FillFreeFn{S, nvar, n_free, b.xstride, d_x, b.xs});
        const int per = 4 * b.smax;
        be_.for_each((size_t)kc * (size_t)per, CoefCostFn<SolveSweepDesc>{desc, per, b.part, 0, per});
        be_.for_each((size_t)kc, CostSumFn<SolveSweepDesc>{desc, per, b.part});
        launches(3);
      } else {
        solve_with_outputs((size_t)kc, stats, desc, b);
        launches(1);
        counters.solves += kc;
      }
      counters.segment_setups += kc * S;
      if (use_soft)
        for (int kd = 1; kd <= 4; ++kd) {
          if (!need[kd - 1]) continue;
          const size_t n = (size_t)kc * S;
          switch (kd) {
            case 1: be_.for_each_scratch(n, MaxMagnitudeSegFn<1>{d_coef, d_T, d_sv, d_st}); break;
            case 2: be_.for_each_scratch(n, MaxMagnitudeSegFn<2>{d_coef, d_T, d_sv, d_st}); break;
            case 3: be_.for_each_scratch(n, MaxMagnitudeSegFn<3>{d_coef, d_T, d_sv, d_st}); break;
            default: be_.for_each_scratch(n, MaxMagnitudeSegFn<4>{d_coef, d_T, d_sv, d_st}); break;
          }
          be_.for_each((size_t)kc, MaxMagnitudeReduceFn{d_off, d_sv, d_st, d_max + (size_t)(kd - 1) * chunk, d_mt, d_mi});
          launches(2);
          counters.root_finds += (long long)n;
          counters.root_finds_executed += (long long)n;
        }
      const ObjCombineFn cf{S, obj_terms(method, time_penalty, use_soft, soft_weight, ncon, con_deriv, con_value), d_T, d_costs, d_max, (size_t)chunk,
                            d_total, d_parts};
      be_.for_each((size_t)kc, cf);
      launches(1);
      be_.d2h(total + k0, d_total, sizeof(double) * (size_t)kc);
      if (parts) be_.d2h(parts + 3 * (size_t)k0, d_parts, sizeof(double) * 3 * (size_t)kc);
      if (coef) be_.d2h(coef + (size_t)k0 * S * TG_D * TG_N, d_coef, sizeof(double) * (size_t)kc * S * TG_D * TG_N);
    }
    return 0;
  }
  static ObjTerms obj_terms(int method, double time_penalty, int use_soft, double soft_weight, int ncon, const int* con_deriv, const double* con_value) {
    ObjTerms t{method, ncon, time_penalty, soft_weight, use_soft, {}, {}};
    for (int c = 0; c < ncon; ++c) {
      t.con_deriv[c] = con_deriv[c];
      t.con_value[c] = con_value[c];
    }
    return t;
  }

  // The derivative-free time allocation (tg_dfo.cuh) for B problems given as vertices; the caller has validated the inputs.
  // Problems are cut into groups of consecutive problems of at most seg_budget candidate segments (the segments the candidates of
  // one iteration recompute: S per candidate for methods 0, 1, two for 3, 4); a group runs its whole search before the next starts.
  void dfo_batch(int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times, const DfoParams& Q, int ncon, const int* con_dim,
                 const int* con_deriv, const double* con_value, double* coef, double* vval_out, int* code, int* n_iter, double* total, double* parts) {
    dfo_groups(B, vtx_off, vmask, TG_HALF, TG_D, Q.time_alloc_method >= 3, [&](int p0, int p1) {
      dfo_group(p0, p1, vtx_off, vmask, vval, times, Q, ncon, con_dim, con_deriv, con_value, coef, vval_out, code, n_iter, total, parts);
    });
  }
  // the groups of dfo_batch / dfo_batch_n: run(p0, p1) for consecutive problems [p0, p1) of at most seg_budget candidate segments
  // (a problem over its budget alone forms a group); half = N/2 derivatives per vertex, dims = D dimensions with variables
  template <class Run>
  void dfo_groups(int B, const int* vtx_off, const uint8_t* vmask, int half, int dims, bool with_free, const Run& run) {
    std::vector<size_t> units(B);
    for (int p = 0; p < B; ++p) {
      const int V = vtx_off[p + 1] - vtx_off[p], S = V - 1;
      int nf = 0;
      for (int v = vtx_off[p]; v < vtx_off[p + 1]; ++v)
        for (int k = 0; k < half; ++k) nf += ((vmask[v] >> k) & 1u) ? 0 : 1;
      const size_t n = (size_t)(with_free ? S + dims * nf : S);
      units[p] = 2 * n * (size_t)(with_free ? 2 : S);
    }
    for (int p0 = 0; p0 < B;) {
      int p1 = p0 + 1;
      size_t u = units[p0];
      while (p1 < B && u + units[p1] <= seg_budget) u += units[p1++];
      run(p0, p1);
      p0 = p1;
    }
  }
  void dfo_group(int p0, int p1, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times, const DfoParams& Q, int ncon,
                 const int* con_dim, const int* con_deriv, const double* con_value, double* coef, double* vval_out, int* code, int* n_iter,
                 double* total, double* parts) {
    scratch_.reset();
    const int G = p1 - p0, method = Q.time_alloc_method;
    const bool with_free = method >= 3;
    const size_t gv0 = (size_t)vtx_off[p0], gs0 = gv0 - (size_t)p0;
    std::vector<int> so(G + 1);
    for (int i = 0; i <= G; ++i) so[i] = vtx_off[p0 + i] - (int)gv0 - i;
    Bare bb = bare_batch(G, so.data(), Q.derivative_to_optimize);
    BatchPtrs& b = bb.b;
    const int totS = b.totS, totV = b.totV;
    b.vmask = scratch_.template alloc<uint8_t>(totV);
    b.vval = scratch_.template alloc<double>((size_t)totV * TG_HALF * TG_D);
    b.vfree = scratch_.template alloc<int>((size_t)totV + G);
    b.np = scratch_.template alloc<int>(G);
    b.hbw = scratch_.template alloc<int>(G);
    b.fmax = scratch_.template alloc<int>(G);
    b.times = scratch_.template alloc<double>(totS);
    b.coef = scratch_.template alloc<double>((size_t)totS * TG_D * TG_N);
    b.recs = scratch_.template alloc<double>((size_t)totS * 3 * TG_REC_SIZE);
    be_.h2d(b.vmask, vmask + gv0, totV);
    be_.h2d(b.vval, vval + gv0 * TG_HALF * TG_D, sizeof(double) * (size_t)totV * TG_HALF * TG_D);
    be_.h2d(b.times, times + gs0, sizeof(double) * totS);
    be_.for_each(G, PrepareFn{b, 0});
    launches(1);
    int stats[16];
    be_.d2h(stats, b.stats, sizeof(stats));
    std::vector<int> np(G);
    be_.d2h(np.data(), b.np, sizeof(int) * G);
    // per-problem layout of the variables, candidates (2 n) and candidate items
    std::vector<DfoProb> hp(G);
    size_t totN = 0, totCand = 0, totItems = 0;
    for (int i = 0; i < G; ++i) {
      DfoProb& P = hp[i];
      std::memset(&P, 0, sizeof(P));
      P.S = so[i + 1] - so[i];
      P.n_free = np[i];
      P.n = with_free ? P.S + TG_D * P.n_free : P.S;
      P.s0 = so[i];
      P.x0 = (int)totN;
      P.c0 = (int)totCand;
      P.i0 = (int)totItems;
      totN += (size_t)P.n;
      totCand += 2 * (size_t)P.n;
      totItems += 2 * (size_t)P.n * (size_t)(with_free ? 2 : P.S);
    }
    DfoBatch d;
    std::memset(&d, 0, sizeof(d));
    d.prob = scratch_.template alloc<DfoProb>(G);
    be_.h2d(d.prob, hp.data(), sizeof(DfoProb) * G);
    d.method = method;
    d.max_iter = Q.max_iterations;
    d.ipc_free = 2;
    d.f_rel = Q.f_rel;
    d.x_rel = Q.x_rel;
    d.step_rel = Q.initial_stepsize_rel;
    d.obj = obj_terms(method, Q.time_penalty, Q.use_soft_constraints, Q.soft_constraint_weight, ncon, con_deriv, con_value);
    for (int c = 0; c < ncon; ++c) d.con_dim[c] = con_dim[c];
    d.x = scratch_.template alloc<double>(totN);
    d.lo = scratch_.template alloc<double>(totN);
    d.hi = scratch_.template alloc<double>(totN);
    d.step = scratch_.template alloc<double>(totN);
    d.cand_prob = scratch_.template alloc<int>(totCand);
    d.item_cand = with_free ? nullptr : scratch_.template alloc<int>(totItems);
    d.ctot = scratch_.template alloc<double>(totCand);
    d.ccost = with_free ? nullptr : scratch_.template alloc<double>(totCand);
    d.ccoef = scratch_.template alloc<double>(totItems * TG_D * TG_N);
    d.cpart = with_free ? scratch_.template alloc<double>(totItems * 4) : nullptr;
    bool need[4] = {false, false, false, false};
    for (int c = 0; c < ncon; ++c) need[con_deriv[c] - 1] = Q.use_soft_constraints != 0;
    d.csv = scratch_.template alloc<double>(4 * totItems);
    d.bcost = scratch_.template alloc<double>(G);
    d.bpart = scratch_.template alloc<double>((size_t)totS * 4);
    d.bsv = scratch_.template alloc<double>((size_t)4 * totS);
    d.btot = scratch_.template alloc<double>(G);
    d.bparts = scratch_.template alloc<double>((size_t)3 * G);
    d.totS = (size_t)totS;
    d.totItems = totItems;
    for (int k = 0; k < 2; ++k) {
      d.lists[k][0] = scratch_.template alloc<int>(G);
      d.lists[k][1] = scratch_.template alloc<int>(totS);
      d.lists[k][2] = scratch_.template alloc<int>(totCand);
      d.lists[k][3] = scratch_.template alloc<int>(totItems);
    }
    d.cnt = scratch_.template alloc<int>(9);
    alloc_solution_buffers(b, with_free ? (size_t)G : totCand, stats);
    d.b = b;
    be_.for_each(G, DfoMapFn{d});
    launches(1);
    if (with_free) {  // x0 of the free derivatives: the linear solution at the initial times (solveLinear + getFreeConstraints)
      be_.for_each(totS, SetupBaseFn{b, b.times});
      solve_with_outputs((size_t)G, stats, SolveProblemDesc{b, 0, nullptr, nullptr}, b);
      be_.for_each(totV, DfoFreeInitFn{d});
      launches(3);
      counters.solves += G;
      counters.segment_setups += totS;
    }
    be_.for_each(G, DfoBeginFn{d});
    be_.dev_memset(d.cnt, 0, 9 * sizeof(int));
    launches(1);
    dfo_base_eval(d, stats, need, 1);
    int back[5];
    be_.d2h(back, d.cnt, sizeof(back));
    for (int it = 0; it < Q.max_iterations && back[0] > 0; ++it) {
      const int buf = it & 1, nbuf = buf ^ 1;
      const bool sparse = (size_t)back[0] * 2 < (size_t)G;
      const int* const* L = sparse ? d.lists[buf] : nullptr;
      const size_t nprob = sparse ? (size_t)back[1] : (size_t)G, nseg = sparse ? (size_t)back[2] : (size_t)totS;
      const size_t ncand = sparse ? (size_t)back[3] : totCand, nitem = sparse ? (size_t)back[4] : totItems;
      be_.dev_memset(d.cnt, 0, sizeof(int));
      be_.dev_memset(d.cnt + 1 + 4 * nbuf, 0, 4 * sizeof(int));
      be_.for_each(nseg * 3, DfoRecsFn{d, L ? L[1] : nullptr, 3, 0});
      launches(1);
      if (with_free) {
        be_.for_each(nseg * 4, DfoBaseCoefFn{d, L ? L[1] : nullptr, 0});
        dfo_maxima(d, need, L ? L[1] : nullptr, nseg, 1, 0);
        be_.for_each(nitem, DfoItemFn{d, L ? L[3] : nullptr});
        launches(2);
      } else {
        solve_with_outputs(ncand, stats, DfoSolveDesc{d, 0, L ? L[2] : nullptr}, b);
        launches(1);
      }
      dfo_maxima(d, need, L ? L[3] : nullptr, nitem, 0, 0);
      be_.for_each(ncand, DfoTotalFn{d, L ? L[2] : nullptr});
      be_.for_each(nprob, DfoAdvanceFn{d, L ? L[0] : nullptr, nbuf});
      launches(2);
      // work of the running problems (the lists hold exactly them, dense launches or not)
      counters.segment_setups += (long long)back[2] * 3;
      counters.evals += (long long)back[3];
      if (!with_free) counters.solves += back[3];
      for (int k = 0; k < 4; ++k)
        if (need[k]) {
          counters.root_finds += (long long)back[4] + (with_free ? back[2] : 0);
          counters.root_finds_executed += (long long)back[4] + (with_free ? back[2] : 0);
        }
      int nb[5];
      be_.d2h(nb, d.cnt, sizeof(int));
      be_.d2h(nb + 1, d.cnt + 1 + 4 * nbuf, 4 * sizeof(int));
      std::memcpy(back, nb, sizeof(back));
    }
    dfo_base_eval(d, stats, need, 0);  // the final point, with coefficients and the three terms
    double* d_times = scratch_.template alloc<double>(totS);
    be_.for_each(totS, DfoTimesOutFn{d, d_times});
    launches(1);
    be_.d2h(times + gs0, d_times, sizeof(double) * totS);
    if (coef) be_.d2h(coef + gs0 * TG_D * TG_N, b.coef, sizeof(double) * (size_t)totS * TG_D * TG_N);
    if (vval_out && with_free) {
      double* d_vv = scratch_.template alloc<double>((size_t)totV * TG_HALF * TG_D);
      be_.for_each(totV, DfoVvalOutFn{d, d_vv});
      launches(1);
      be_.d2h(vval_out + gv0 * TG_HALF * TG_D, d_vv, sizeof(double) * (size_t)totV * TG_HALF * TG_D);
    }
    be_.d2h(hp.data(), d.prob, sizeof(DfoProb) * G);
    for (int i = 0; i < G; ++i) {
      if (code) code[p0 + i] = hp[i].code;
      if (n_iter) n_iter[p0 + i] = hp[i].iterations;
      if (total) total[p0 + i] = hp[i].f;
    }
    if (parts) be_.d2h(parts + 3 * (size_t)p0, d.bparts, sizeof(double) * 3 * G);
  }
  // the objective at every problem's current x: records, coefficients (a linear solve for methods 0, 1), maxima, total
  void dfo_base_eval(const DfoBatch& d, const int* stats, const bool* need, int start) {
    const int G = d.b.B, totS = d.b.totS;
    be_.for_each((size_t)totS, DfoRecsFn{d, nullptr, 1, 1});
    if (d.method >= 3) {
      be_.for_each((size_t)totS * 4, DfoBaseCoefFn{d, nullptr, 1});
    } else {
      solve_with_outputs((size_t)G, stats, DfoSolveDesc{d, 1, nullptr}, d.b);
      counters.solves += G;
    }
    dfo_maxima(d, need, nullptr, (size_t)totS, 1, 1);
    be_.for_each((size_t)G, DfoBaseTotalFn{d, start});
    launches(3);
    counters.segment_setups += totS;
    counters.evals += G;
  }
  void dfo_maxima(const DfoBatch& d, const bool* need, const int* list, size_t n, int base, int all) {
    for (int k = 0; k < 4; ++k) {
      if (!need[k] || n == 0) continue;
      switch (k + 1) {
        case 1: be_.for_each_scratch(n, DfoMaxFn<1>{d, list, base, all}); break;
        case 2: be_.for_each_scratch(n, DfoMaxFn<2>{d, list, base, all}); break;
        case 3: be_.for_each_scratch(n, DfoMaxFn<3>{d, list, base, all}); break;
        default: be_.for_each_scratch(n, DfoMaxFn<4>{d, list, base, all}); break;
      }
      launches(1);
      if (base && all) {
        counters.root_finds += (long long)n;
        counters.root_finds_executed += (long long)n;
      }
    }
  }
  // ---- general-shape path (tg_generic.cuh): PolynomialOptimization<N> for N = 6, 8, 10, 12 on 4 (zero-padded) dimensions ----------
  // setupFromVertices + solveLinear + getSegments + computeCost for B problems.  The vertex bookkeeping (first free unknown per
  // vertex, half bandwidth, workspace offsets) is host logic here: the inputs arrive from the host and this path is not the
  // benchmarked one.  vval: [totV][N/2][4]; coef out: [totS][4][N].
  struct GenVertices {
    std::vector<int> vfree, np, hbw;  // first free unknown per vertex (V + 1 entries per problem, at vtx_off[p] + p); per problem
  };
  template <int N>
  static GenVertices gen_vertices(int B, const int* vtx_off, const uint8_t* vmask) {
    constexpr int H = N / 2;
    GenVertices g;
    g.vfree.resize((size_t)vtx_off[B] + B);
    g.np.resize(B);
    g.hbw.resize(B);
    for (int p = 0; p < B; ++p) {
      const int v0 = vtx_off[p], V = vtx_off[p + 1] - v0;
      int* ff = g.vfree.data() + v0 + p;
      ff[0] = 0;
      for (int v = 0; v < V; ++v) {
        int cnt = 0;
        for (int k = 0; k < H; ++k) cnt += ((vmask[v0 + v] >> k) & 1u) ? 0 : 1;
        ff[v + 1] = ff[v] + cnt;
      }
      int hb = 0;  // a free slot of vertex v couples to the free slots of v-1 .. v+1 (lin_impl.h:317-333)
      for (int v = 0; v < V; ++v)
        if (ff[v + 1] > ff[v]) hb = std::max(hb, ff[std::min(v + 2, V)] - 1 - ff[v]);
      g.np[p] = ff[V];
      g.hbw[p] = hb;
    }
    return g;
  }
  // offset of every problem's [4][n_free] block of free derivatives (dimension-major, problems in order); the total at [B]
  static std::vector<long long> gen_dp_offsets(const std::vector<int>& np) {
    std::vector<long long> off(np.size() + 1, 0);
    for (size_t p = 0; p < np.size(); ++p) off[p + 1] = off[p] + (long long)TG_D * np[p];
    return off;
  }
  // dp (optional): the free derivatives d_p of every problem after the solve, [4][n_free] per problem (gen_dp_offsets)
  template <int N>
  bool linear_batch_n(int B, const int* vtx_off, const uint8_t* vmask, const double* vval, const double* times, int r, double* coef, double* cost,
                      double* dp = nullptr) {
    constexpr int H = N / 2;
    scratch_.reset();
    const int totV = vtx_off[B], totS = totV - B;
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] - vtx_off[p] < 2) return false;
    const GenVertices gv = gen_vertices<N>(B, vtx_off, vmask);
    const std::vector<int>&vfree = gv.vfree, &np = gv.np, &hbw = gv.hbw;
    std::vector<long long> ws_off(B);
    long long ws_tot = 0;
    for (int p = 0; p < B; ++p) {
      ws_off[p] = ws_tot;
      ws_tot += (long long)gen::ws_doubles<N>(vtx_off[p + 1] - vtx_off[p] - 1, np[p], hbw[p]);
    }
    int* d_vtx_off = scratch_.template alloc<int>((size_t)B + 1);
    uint8_t* d_vmask = scratch_.template alloc<uint8_t>(totV);
    int* d_vfree = scratch_.template alloc<int>(vfree.size());
    double* d_vval = scratch_.template alloc<double>((size_t)totV * H * TG_D);
    int* d_np = scratch_.template alloc<int>(B);
    int* d_hbw = scratch_.template alloc<int>(B);
    double* d_times = scratch_.template alloc<double>(totS);
    double* d_recs = scratch_.template alloc<double>((size_t)totS * gen::Rec<N>::kSize);
    long long* d_ws_off = scratch_.template alloc<long long>(B);
    double* d_ws = scratch_.template alloc<double>((size_t)std::max<long long>(ws_tot, 1));
    double* d_coef = scratch_.template alloc<double>((size_t)totS * TG_D * N);
    double* d_cost = scratch_.template alloc<double>(B);
    be_.h2d(d_vtx_off, vtx_off, sizeof(int) * ((size_t)B + 1));
    be_.h2d(d_vmask, vmask, totV);
    be_.h2d(d_vfree, vfree.data(), sizeof(int) * vfree.size());
    be_.h2d(d_vval, vval, sizeof(double) * (size_t)totV * H * TG_D);
    be_.h2d(d_np, np.data(), sizeof(int) * B);
    be_.h2d(d_hbw, hbw.data(), sizeof(int) * B);
    be_.h2d(d_times, times, sizeof(double) * totS);
    be_.h2d(d_ws_off, ws_off.data(), sizeof(long long) * B);
    be_.for_each((size_t)totS, gen::RecordHeadFn<N>{r, d_times, d_recs});
    be_.for_each((size_t)totS * N, gen::RecordHrowFn<N>{d_recs});
    const gen::SolveFn<N> solve{r, d_vtx_off, d_vmask, d_vfree, d_vval, d_np, d_hbw, d_recs, d_ws_off, d_ws, d_coef, d_cost};
    std::vector<long long> dp_off;
    double* d_dp = nullptr;
    if (dp) {
      dp_off = gen_dp_offsets(np);
      long long* d_dp_off = scratch_.template alloc<long long>(B);
      d_dp = scratch_.template alloc<double>((size_t)std::max<long long>(dp_off[B], 1));
      be_.h2d(d_dp_off, dp_off.data(), sizeof(long long) * B);
      be_.for_each_warp((size_t)B, gen::SolveFreeFn<N>{solve, d_dp_off, d_dp});
    } else {
      be_.for_each_warp((size_t)B, solve);
    }
    launches(3);
    counters.solves += B;
    counters.segment_setups += totS;
    if (coef) be_.d2h(coef, d_coef, sizeof(double) * (size_t)totS * TG_D * N);
    if (cost) be_.d2h(cost, d_cost, sizeof(double) * B);
    if (dp) be_.d2h(dp, d_dp, sizeof(double) * (size_t)dp_off[B]);
    return true;
  }
  // setFreeConstraints + getSegments + computeCost (lin_impl.h:519-522, 263-282, 127-141) for B problems: the coefficients from the
  // fixed values and the given free derivatives dp ([4][n_free] per problem, gen_dp_offsets), without a solve.
  template <int N>
  bool set_free_batch_n(int B, const int* vtx_off, const uint8_t* vmask, const double* vval, const double* times, int r, const double* dp,
                        double* coef, double* cost) {
    constexpr int H = N / 2;
    scratch_.reset();
    const int totV = vtx_off[B], totS = totV - B;
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] - vtx_off[p] < 2) return false;
    const GenVertices gv = gen_vertices<N>(B, vtx_off, vmask);
    const std::vector<long long> dp_off = gen_dp_offsets(gv.np);
    std::vector<int> prob_of_seg(totS);
    for (int p = 0; p < B; ++p)
      for (int s = vtx_off[p] - p; s < vtx_off[p + 1] - p - 1; ++s) prob_of_seg[s] = p;
    int* d_vtx_off = scratch_.template alloc<int>((size_t)B + 1);
    int* d_prob_of_seg = scratch_.template alloc<int>(totS);
    uint8_t* d_vmask = scratch_.template alloc<uint8_t>(totV);
    int* d_vfree = scratch_.template alloc<int>(gv.vfree.size());
    double* d_vval = scratch_.template alloc<double>((size_t)totV * H * TG_D);
    long long* d_dp_off = scratch_.template alloc<long long>(B);
    int* d_np = scratch_.template alloc<int>(B);
    double* d_dp = scratch_.template alloc<double>((size_t)std::max<long long>(dp_off[B], 1));
    double* d_times = scratch_.template alloc<double>(totS);
    double* d_recs = scratch_.template alloc<double>((size_t)totS * gen::Rec<N>::kSize);
    double* d_coef = scratch_.template alloc<double>((size_t)totS * TG_D * N);
    double* d_part = scratch_.template alloc<double>((size_t)totS * TG_D);
    double* d_cost = scratch_.template alloc<double>(B);
    be_.h2d(d_vtx_off, vtx_off, sizeof(int) * ((size_t)B + 1));
    be_.h2d(d_prob_of_seg, prob_of_seg.data(), sizeof(int) * (size_t)totS);
    be_.h2d(d_vmask, vmask, totV);
    be_.h2d(d_vfree, gv.vfree.data(), sizeof(int) * gv.vfree.size());
    be_.h2d(d_vval, vval, sizeof(double) * (size_t)totV * H * TG_D);
    be_.h2d(d_dp_off, dp_off.data(), sizeof(long long) * B);
    be_.h2d(d_np, gv.np.data(), sizeof(int) * B);
    be_.h2d(d_dp, dp, sizeof(double) * (size_t)dp_off[B]);
    be_.h2d(d_times, times, sizeof(double) * totS);
    be_.for_each((size_t)totS, gen::RecordHeadFn<N>{r, d_times, d_recs});
    be_.for_each((size_t)totS * TG_D, gen::SetFreeFn<N>{d_prob_of_seg, d_vmask, d_vfree, d_vval, d_dp_off, d_np, d_dp, d_recs, d_coef, d_part});
    be_.for_each((size_t)B, gen::SetFreeCostFn{d_vtx_off, d_part, d_cost});
    launches(3);
    counters.segment_setups += totS;
    if (coef) be_.d2h(coef, d_coef, sizeof(double) * (size_t)totS * TG_D * N);
    if (cost) be_.d2h(cost, d_cost, sizeof(double) * B);
    return true;
  }
  // Trajectory::evaluate at n times of one trajectory of N-coefficient segments
  template <int N>
  void evaluate_batch_n(int S, const double* coef, const double* times, int n, const double* t, int deriv, double* out, uint8_t* ok) {
    scratch_.reset();
    double* d_coef = scratch_.template alloc<double>((size_t)S * TG_D * N);
    double* d_T = scratch_.template alloc<double>(S);
    double* d_t = scratch_.template alloc<double>(std::max(n, 1));
    double* d_out = scratch_.template alloc<double>((size_t)std::max(n, 1) * 4);
    uint8_t* d_ok = scratch_.template alloc<uint8_t>(std::max(n, 1));
    be_.h2d(d_coef, coef, sizeof(double) * (size_t)S * TG_D * N);
    be_.h2d(d_T, times, sizeof(double) * S);
    be_.h2d(d_t, t, sizeof(double) * n);
    be_.for_each(n, gen::EvaluateFn<N>{S, deriv, d_coef, d_T, d_t, d_out, d_ok});
    launches(1);
    be_.d2h(out, d_out, sizeof(double) * 4 * (size_t)n);
    if (ok) be_.d2h(ok, d_ok, n);
  }
  // sampleWholeTrajectory for B trajectories of N-coefficient segments (the dt walk does not depend on N)
  template <int N>
  void sample_batch_n(int B, const int* seg_off, const double* coef, const double* times, double dt, int* counts, double* samples, double* full) {
    scratch_.reset();
    const int totS = seg_off[B];
    int* d_seg_off = scratch_.template alloc<int>((size_t)B + 1);
    double* d_times = scratch_.template alloc<double>(std::max(totS, 1));
    double* d_coef = scratch_.template alloc<double>((size_t)std::max(totS, 1) * TG_D * N);
    be_.h2d(d_seg_off, seg_off, sizeof(int) * ((size_t)B + 1));
    be_.h2d(d_times, times, sizeof(double) * totS);
    be_.h2d(d_coef, coef, sizeof(double) * (size_t)totS * TG_D * N);
    int* cap = scratch_.template alloc<int>((size_t)B + 1);
    int* d_smp_off = scratch_.template alloc<int>((size_t)B + 1);
    int* d_count = scratch_.template alloc<int>(B);
    be_.for_each(B, GenSampleCapFn{d_seg_off, d_times, dt, cap});
    be_.exclusive_scan(cap, d_smp_off, B);
    std::vector<int> smp_off(B + 1);
    be_.d2h(smp_off.data(), d_smp_off, sizeof(int) * (B + 1));
    const size_t slots = (size_t)std::max(smp_off[B], 1);
    int* seg_idx = scratch_.template alloc<int>(slots);
    int* smp_prob = scratch_.template alloc<int>(slots);
    double* t_in = scratch_.template alloc<double>(slots);
    be_.for_each(B, GenSampleWalkFn{d_seg_off, d_times, dt, d_smp_off, seg_idx, t_in, d_count});
    launches(3);
    be_.d2h(counts, d_count, sizeof(int) * B);
    std::vector<int> dst(B + 1, 0);
    for (int p = 0; p < B; ++p) dst[p + 1] = dst[p] + counts[p];
    counters.samples += dst[B];
    if ((!samples && !full) || dst[B] == 0) return;
    double* d_xyzh = samples ? scratch_.template alloc<double>(slots * 4) : nullptr;
    double* d_full = full ? scratch_.template alloc<double>(slots * 19) : nullptr;
    be_.for_each(B, SlotProblemFn{B, d_smp_off, smp_prob});
    be_.for_each((size_t)smp_off[B], gen::SampleEvalFn<N>{d_seg_off, d_smp_off, smp_prob, d_count, seg_idx, t_in, d_coef, d_xyzh, d_full});
    launches(2);
    // a trajectory's samples are contiguous from its slot offset; the unused tail of each capacity range is skipped here
    for (int p = 0; p < B; ++p) {
      if (counts[p] == 0) continue;
      if (samples) be_.d2h(samples + 4 * (size_t)dst[p], d_xyzh + 4 * (size_t)smp_off[p], sizeof(double) * 4 * (size_t)counts[p]);
      if (full) be_.d2h(full + 19 * (size_t)dst[p], d_full + 19 * (size_t)smp_off[p], sizeof(double) * 19 * (size_t)counts[p]);
    }
  }
  // The windowed dt walk of sampleTrajectoryInRange / evaluateRange for B trajectories of N-coefficient segments, window
  // p = [t_range[2p], t_range[2p+1]]: the trajectories go up, a counting walk gives counts[B]; when rows are wanted, the device
  // scans the counts and walks again, writing each sample at its compacted row, and row_prob maps rows to trajectories.
  // false: some window's count passed its bound (sample_range_cap); counts is then not written.
  struct RangeRows {
    int* seg_off;
    double* coef;
    int* count;
    int* row_off;
    int* row_prob;
    int* seg_idx;
    double* t_in;
    double* acc;
    long long* t_ns;
    size_t rows;
  };
  template <int N>
  bool range_walk(int B, const int* seg_off, const double* coef, const double* times, const double* t_range, double dt, int* counts,
                  bool rows_wanted, bool want_tns, RangeRows* w) {
    scratch_.reset();
    const int totS = seg_off[B];
    w->seg_off = scratch_.template alloc<int>((size_t)B + 1);
    double* d_times = scratch_.template alloc<double>(std::max(totS, 1));
    double* d_range = scratch_.template alloc<double>((size_t)B * 2);
    int* d_count = w->count = scratch_.template alloc<int>((size_t)B + 1);
    int* d_overflow = scratch_.template alloc<int>(1);
    be_.h2d(w->seg_off, seg_off, sizeof(int) * ((size_t)B + 1));
    be_.h2d(d_times, times, sizeof(double) * totS);
    be_.h2d(d_range, t_range, sizeof(double) * 2 * (size_t)B);
    be_.dev_memset(d_overflow, 0, sizeof(int));
    be_.for_each(B, RangeWalkFn{w->seg_off, d_times, d_range, dt, nullptr, d_count, nullptr, nullptr, nullptr, nullptr, d_overflow});
    launches(1);
    int overflow = 0;
    std::vector<int> cnt(B);
    be_.d2h(&overflow, d_overflow, sizeof(int));
    if (overflow) return false;
    be_.d2h(cnt.data(), d_count, sizeof(int) * B);
    long long rows = 0;
    for (int p = 0; p < B; ++p) rows += cnt[p];
    if (rows > (long long)INT_MAX) return false;
    std::copy(cnt.begin(), cnt.end(), counts);
    counters.samples += rows;
    w->rows = (size_t)rows;
    if (!rows_wanted || rows == 0) return true;
    w->coef = scratch_.template alloc<double>((size_t)std::max(totS, 1) * TG_D * N);
    be_.h2d(w->coef, coef, sizeof(double) * (size_t)totS * TG_D * N);
    w->row_off = scratch_.template alloc<int>((size_t)B + 1);
    w->row_prob = scratch_.template alloc<int>(w->rows);
    w->seg_idx = scratch_.template alloc<int>(w->rows);
    w->t_in = scratch_.template alloc<double>(w->rows);
    w->acc = scratch_.template alloc<double>(w->rows);
    w->t_ns = want_tns ? scratch_.template alloc<long long>(w->rows) : nullptr;
    be_.exclusive_scan(d_count, w->row_off, B);
    be_.for_each(B, RangeWalkFn{w->seg_off, d_times, d_range, dt, w->row_off, d_count, w->seg_idx, w->t_in, w->acc, w->t_ns, d_overflow});
    be_.for_each(B, SlotProblemFn{B, w->row_off, w->row_prob});
    launches(3);
    return true;
  }
  // sampleTrajectoryInRange: the sample record of every row (gen::SampleEvalFn over the compacted rows) and time_from_start_ns;
  // each output array comes back in one copy
  template <int N>
  bool sample_range_batch_n(int B, const int* seg_off, const double* coef, const double* times, const double* t_range, double dt, int* counts,
                            double* samples, double* full, long long* t_ns) {
    RangeRows w;
    if (!range_walk<N>(B, seg_off, coef, times, t_range, dt, counts, samples || full || t_ns, t_ns != nullptr, &w)) return false;
    if ((!samples && !full && !t_ns) || w.rows == 0) return true;
    double* d_xyzh = samples ? scratch_.template alloc<double>(w.rows * 4) : nullptr;
    double* d_full = full ? scratch_.template alloc<double>(w.rows * 19) : nullptr;
    if (samples || full) {
      be_.for_each(w.rows, gen::SampleEvalFn<N>{w.seg_off, w.row_off, w.row_prob, w.count, w.seg_idx, w.t_in, w.coef, d_xyzh, d_full});
      launches(1);
    }
    if (samples) be_.d2h(samples, d_xyzh, sizeof(double) * 4 * w.rows);
    if (full) be_.d2h(full, d_full, sizeof(double) * 19 * w.rows);
    if (t_ns) be_.d2h(t_ns, w.t_ns, sizeof(long long) * w.rows);
    return true;
  }
  // Trajectory::evaluateRange: derivative `deriv` of the D dimensions at every row ([rows][D]) and the accumulated sampling times
  template <int N>
  bool evaluate_range_batch_n(int B, int D, const int* seg_off, const double* coef, const double* times, const double* t_range, double dt, int deriv,
                              int* counts, double* out, double* sampling_times) {
    RangeRows w;
    if (!range_walk<N>(B, seg_off, coef, times, t_range, dt, counts, out || sampling_times, false, &w)) return false;
    if ((!out && !sampling_times) || w.rows == 0) return true;
    if (out) {
      double* d_out = scratch_.template alloc<double>(w.rows * D);
      be_.for_each(w.rows, gen::EvaluateRangeFn<N>{w.seg_off, w.row_prob, w.seg_idx, w.t_in, w.coef, deriv, D, d_out});
      launches(1);
      be_.d2h(out, d_out, sizeof(double) * D * w.rows);
    }
    if (sampling_times) be_.d2h(sampling_times, w.acc, sizeof(double) * w.rows);
    return true;
  }
  // per-segment maxima of |v|,|a|,|j| for the three dimension groups, N-coefficient segments
  template <int N>
  void extrema_batch_n(int totS, const double* coef, const double* times, double* maxima) {
    scratch_.reset();
    double* d_coef = scratch_.template alloc<double>((size_t)totS * TG_D * N);
    double* d_T = scratch_.template alloc<double>(totS);
    double* d_m = scratch_.template alloc<double>((size_t)totS * 9);
    be_.h2d(d_coef, coef, sizeof(double) * (size_t)totS * TG_D * N);
    be_.h2d(d_T, times, sizeof(double) * totS);
    extrema_segments_n<N>(d_coef, d_T, d_m, (size_t)totS, nullptr, nullptr);
    counters.root_finds += (long long)totS * 9;
    counters.root_finds_executed += (long long)totS * 9;
    be_.d2h(maxima, d_m, sizeof(double) * (size_t)totS * 9);
  }
  // PolynomialOptimization<N>::computeMaximumOfMagnitude(derivative) for B trajectories (lin_impl.h:477-508)
  template <int N>
  void max_magnitude_batch_n(int B, const int* seg_off, const double* coef, const double* times, int derivative, double* value, double* time,
                             int* segment_idx) {
    scratch_.reset();
    const int totS = seg_off[B];
    int* d_off = scratch_.template alloc<int>((size_t)B + 1);
    double* d_coef = scratch_.template alloc<double>((size_t)totS * TG_D * N);
    double* d_T = scratch_.template alloc<double>(totS);
    double* d_sv = scratch_.template alloc<double>(totS);
    double* d_st = scratch_.template alloc<double>(totS);
    double* d_v = scratch_.template alloc<double>(B);
    double* d_t = scratch_.template alloc<double>(B);
    int* d_i = scratch_.template alloc<int>(B);
    be_.h2d(d_off, seg_off, sizeof(int) * ((size_t)B + 1));
    be_.h2d(d_coef, coef, sizeof(double) * (size_t)totS * TG_D * N);
    be_.h2d(d_T, times, sizeof(double) * totS);
    switch (derivative) {
      case 1: be_.for_each_scratch((size_t)totS, gen::MaxMagnitudeSegFn<N, 1>{d_coef, d_T, d_sv, d_st}); break;
      case 2: be_.for_each_scratch((size_t)totS, gen::MaxMagnitudeSegFn<N, 2>{d_coef, d_T, d_sv, d_st}); break;
      case 3: be_.for_each_scratch((size_t)totS, gen::MaxMagnitudeSegFn<N, 3>{d_coef, d_T, d_sv, d_st}); break;
      default: be_.for_each_scratch((size_t)totS, gen::MaxMagnitudeSegFn<N, 4>{d_coef, d_T, d_sv, d_st}); break;
    }
    be_.for_each((size_t)B, MaxMagnitudeReduceFn{d_off, d_sv, d_st, d_v, d_t, d_i});
    launches(2);
    counters.root_finds += totS;
    counters.root_finds_executed += totS;
    be_.d2h(value, d_v, sizeof(double) * B);
    be_.d2h(time, d_t, sizeof(double) * B);
    be_.d2h(segment_idx, d_i, sizeof(int) * B);
  }
  // Trajectory::scaleSegmentTimesToMeetConstraints in place, N-coefficient segments
  template <int N>
  void scale_times_batch_n(int B, const int* seg_off, double* coef, double* times, const double* L9, int* passes, uint8_t* within) {
    scratch_.reset();
    Bare bb = bare_batch(B, seg_off, 2);
    BatchPtrs& b = bb.b;
    b.times = scratch_.template alloc<double>(b.totS);
    b.coef = scratch_.template alloc<double>((size_t)b.totS * TG_D * N);
    b.maxima = scratch_.template alloc<double>((size_t)b.totS * 9);
    be_.h2d(b.times, times, sizeof(double) * b.totS);
    be_.h2d(b.coef, coef, sizeof(double) * (size_t)b.totS * TG_D * N);
    scale_loop_n<N>(b, L9);
    ScaleOutFn of{b.ps, b.maxima, bb.d_seg_off, {}, nullptr, nullptr, scale_tolerance};
    for (int i = 0; i < 9; ++i) of.L[i] = L9[i];
    of.passes = scratch_.template alloc<int>(B);
    of.within = scratch_.template alloc<uint8_t>(B);
    be_.for_each(B, of); launches(1);
    be_.d2h(coef, b.coef, sizeof(double) * (size_t)b.totS * TG_D * N);
    be_.d2h(times, b.times, sizeof(double) * b.totS);
    if (passes) be_.d2h(passes, of.passes, sizeof(int) * B);
    if (within) be_.d2h(within, of.within, B);
  }
  // estimateSegmentTimes / estimateSegmentTimesBaca (eth/vertex.cpp:491-565, 301-485) for B vertex lists given as positions
  // pos4[totV][4]: euclid / baca [totS] (either null), segment s of problem p at vtx_off[p] - p + s
  void estimate_times_batch(int B, const int* vtx_off, const double* pos4, const double* L8, double* euclid, double* baca) {
    scratch_.reset();
    const int totV = vtx_off[B], totS = totV - B;
    if (totS == 0) return;
    int* d_off = scratch_.template alloc<int>((size_t)B + 1);
    double* d_pos = scratch_.template alloc<double>((size_t)totV * 4);
    be_.h2d(d_off, vtx_off, sizeof(int) * ((size_t)B + 1));
    be_.h2d(d_pos, pos4, sizeof(double) * 4 * (size_t)totV);
    EstimateTimesFn f{B, d_off, d_pos, {}, euclid ? scratch_.template alloc<double>(totS) : nullptr,
                      baca ? scratch_.template alloc<double>(totS) : nullptr};
    for (int k = 0; k < 8; ++k) f.L[k] = L8[k];
    be_.for_each((size_t)totS, f);
    launches(1);
    if (euclid) be_.d2h(euclid, f.euclid, sizeof(double) * totS);
    if (baca) be_.d2h(baca, f.baca, sizeof(double) * totS);
  }
  // PolynomialOptimizationNonLinear<N>::setupFromVertices + optimize() (Mellinger outer loop, nl_impl.h:159-234, then the time
  // scaling of scaleSegmentTimesWithViolation, 335-427) + getTrajectory for B problems given as vertices.  The evaluation runs S+1
  // solves per running problem with dense launches (a finished problem costs an early exit); the optimiser state machine is the one
  // of time_alloc_core.  vval: [totV][N/2][4]; coef out: [totS][4][N].
  template <int N>
  bool time_alloc_batch_n(int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times, const Params& P, double* coef,
                          int* nlopt_code, int* n_evals, int* n_scale_passes, double* final_cost) {
    constexpr int H = N / 2;
    scratch_.reset();
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] - vtx_off[p] < 2) return false;
    const GenVertices gv = gen_vertices<N>(B, vtx_off, vmask);
    std::vector<int> so(B + 1);
    for (int p = 0; p <= B; ++p) so[p] = vtx_off[p] - p;
    Bare bb = bare_batch(B, so.data(), P.derivative_to_optimize);
    BatchPtrs& b = bb.b;
    const int totS = b.totS, totV = b.totV;
    // a workspace per solve instance (p, n) = vertex v0 + n; the final solve of problem p reuses that of instance (p, 0)
    std::vector<long long> ws_inst(totV), ws_prob(B);
    long long ws_tot = 0;
    for (int p = 0; p < B; ++p) {
      const int S = so[p + 1] - so[p];
      const long long w = (long long)gen::ws_doubles<N>(S, gv.np[p], gv.hbw[p]);
      ws_prob[p] = ws_tot;
      for (int n = 0; n <= S; ++n, ws_tot += w) ws_inst[(size_t)vtx_off[p] + n] = ws_tot;
    }
    const int mf = (P.max_evals > 0) ? std::min(std::max(P.max_evals, 1), kPlisMfMax) : kPlisMfMax;
    int* d_vtx_off = scratch_.template alloc<int>((size_t)B + 1);
    long long* d_ws_inst = scratch_.template alloc<long long>(totV);
    long long* d_ws_prob = scratch_.template alloc<long long>(B);
    double* d_ws = scratch_.template alloc<double>((size_t)std::max<long long>(ws_tot, 1));
    double* d_cost = scratch_.template alloc<double>(B);
    b.vmask = scratch_.template alloc<uint8_t>(totV);
    b.vval = scratch_.template alloc<double>((size_t)totV * H * TG_D);
    b.vfree = scratch_.template alloc<int>(gv.vfree.size());
    b.np = scratch_.template alloc<int>(B);
    b.hbw = scratch_.template alloc<int>(B);
    b.times = scratch_.template alloc<double>(totS);
    b.coef = scratch_.template alloc<double>((size_t)totS * TG_D * N);
    b.recs = scratch_.template alloc<double>((size_t)totS * 3 * gen::Rec<N>::kSize);
    b.costs = scratch_.template alloc<double>(totV);
    b.maxima = scratch_.template alloc<double>((size_t)totS * 9);
    b.xeval = scratch_.template alloc<double>(totS);
    b.x = scratch_.template alloc<double>(totS);
    b.g = scratch_.template alloc<double>(totS);
    b.d = scratch_.template alloc<double>(totS);
    b.ix = scratch_.template alloc<int>(totS);
    b.hist_s = scratch_.template alloc<double>((size_t)mf * totS);
    b.hist_y = scratch_.template alloc<double>((size_t)mf * totS);
    b.opt = scratch_.template alloc<PlisScalars>(B);
    for (int k = 0; k < 2; ++k) {
      b.act_prob[k] = scratch_.template alloc<int>(B);
      b.act_vtx[k] = scratch_.template alloc<int>(totV);
      b.act_seg[k] = scratch_.template alloc<int>(totS);
    }
    be_.h2d(d_vtx_off, vtx_off, sizeof(int) * ((size_t)B + 1));
    be_.h2d(d_ws_inst, ws_inst.data(), sizeof(long long) * totV);
    be_.h2d(d_ws_prob, ws_prob.data(), sizeof(long long) * B);
    be_.h2d(b.vmask, vmask, totV);
    be_.h2d(b.vval, vval, sizeof(double) * (size_t)totV * H * TG_D);
    be_.h2d(b.vfree, gv.vfree.data(), sizeof(int) * gv.vfree.size());
    be_.h2d(b.np, gv.np.data(), sizeof(int) * B);
    be_.h2d(b.hbw, gv.hbw.data(), sizeof(int) * B);
    be_.h2d(b.times, times, sizeof(double) * totS);
    be_.dev_memset(b.stats + 9, 0, 6 * sizeof(int));
    be_.for_each(B, PlisBeginFn{b, P.max_evals}); launches(1);
    // maxeval is tested between iterations only, so a line search may overrun it: loop until no problem is left running
    const int eval_cap = (P.max_evals > 0 ? P.max_evals : 1000) + 64;
    for (int e = 0; e < eval_cap; ++e) {
      const int nbuf = (e & 1) ^ 1;
      be_.dev_memset(b.stats + 7, 0, sizeof(int));
      be_.dev_memset(b.stats + 9 + 3 * nbuf, 0, 3 * sizeof(int));
      be_.for_each((size_t)totS * 3, gen::MellingerHeadFn<N>{b});
      be_.for_each((size_t)totS * 3 * N, gen::MellingerHrowFn<N>{b});
      be_.for_each_warp((size_t)totV, gen::MellingerSolveFn<N>{b, d_ws_inst, d_ws});
      be_.for_each(B, PlisAdvanceFn{b, P.max_evals, P.f_rel, P.x_rel, nullptr, nbuf});
      launches(4);
      counters.mellinger_launches += 1;
      int running = 0;
      be_.d2h(&running, b.stats + 7, sizeof(int));
      if (running == 0) break;
    }
    be_.for_each(B, PlisFinishFn{b}); launches(1);
    scale_loop_n<N>(b, P.limits);
    // the final solve at the stretched times
    be_.for_each((size_t)totS, gen::RecordHeadFn<N>{b.r, b.times, b.recs});
    be_.for_each((size_t)totS * N, gen::RecordHrowFn<N>{b.recs});
    be_.for_each_warp((size_t)B, gen::SolveFn<N>{b.r, d_vtx_off, b.vmask, b.vfree, b.vval, b.np, b.hbw, b.recs, d_ws_prob, d_ws, b.coef, d_cost});
    launches(3);
    std::vector<ProbState> ps(B);
    be_.d2h(ps.data(), b.ps, sizeof(ProbState) * B);
    for (int p = 0; p < B; ++p) {
      if (nlopt_code) nlopt_code[p] = ps[p].nlopt_code;
      if (n_evals) n_evals[p] = ps[p].n_evals;
      if (n_scale_passes) n_scale_passes[p] = ps[p].n_scale_passes;
      if (final_cost) final_cost[p] = ps[p].final_cost;
      const int S = so[p + 1] - so[p];
      counters.evals += ps[p].n_evals;
      counters.solves += (long long)ps[p].n_evals * (S == 1 ? 1 : S + 1) + 1;
      if (ps[p].n_evals > 0) counters.root_finds += (long long)(ps[p].n_scale_passes + 1) * 9 * S;
    }
    counters.segment_setups += totS;
    be_.d2h(times, b.times, sizeof(double) * totS);
    if (coef) be_.d2h(coef, b.coef, sizeof(double) * (size_t)totS * TG_D * N);
    return true;
  }

  // objectiveFunctionTime / objectiveFunctionTimeAndConstraints (objective_batch) of ONE problem of N-coefficient segments at K
  // candidate vectors; the caller has validated the inputs.  The K candidates are solved as K copies of the problem: methods 0, 1
  // with linear_batch_n's kernels, 3, 4 with set_free_batch_n's (the free derivatives are read from x in place).  vval: [V][N/2][4];
  // x: [K][nvar], nvar = S or S + 4 * n_free; coef out: [K][S][4][N].
  template <int N>
  void objective_batch_n(int V, const uint8_t* vmask, const double* vval, int r, int method, long long K, const double* x, int nvar,
                         double time_penalty, int use_soft, double soft_weight, int ncon, const int* con_deriv, const double* con_value,
                         double* total, double* parts, double* coef) {
    constexpr int H = N / 2;
    scratch_.reset();
    const int S = V - 1;
    bool need[4] = {false, false, false, false};
    for (int c = 0; c < ncon; ++c) need[con_deriv[c] - 1] = use_soft != 0;
    const int one[2] = {0, V};
    const GenVertices g1 = gen_vertices<N>(1, one, vmask);
    const long long w = (long long)gen::ws_doubles<N>(S, g1.np[0], g1.hbw[0]);
    const long long chunk = std::min<long long>(K, (long long)objective_chunk);
    const size_t C = (size_t)chunk;
    std::vector<int> vo(C + 1), so(C + 1), vfree(C * (V + 1)), np(C, g1.np[0]), hbw(C, g1.hbw[0]), pos(C * S);
    std::vector<long long> ws_off(C), dp_off(C);
    std::vector<uint8_t> vm(C * V);
    std::vector<double> vv(C * V * H * TG_D);
    for (size_t k = 0; k <= C; ++k) {
      vo[k] = (int)(k * V);
      so[k] = (int)(k * S);
    }
    for (size_t k = 0; k < C; ++k) {
      std::memcpy(&vfree[k * (V + 1)], g1.vfree.data(), sizeof(int) * (V + 1));
      std::memcpy(&vm[k * V], vmask, V);
      std::memcpy(&vv[k * V * H * TG_D], vval, sizeof(double) * V * H * TG_D);
      for (int s = 0; s < S; ++s) pos[k * S + s] = (int)k;
      ws_off[k] = (long long)k * w;
      dp_off[k] = (long long)k * nvar + S;
    }
    int* d_vo = scratch_.template alloc<int>(C + 1);
    int* d_so = scratch_.template alloc<int>(C + 1);
    int* d_pos = scratch_.template alloc<int>(C * S);
    uint8_t* d_vm = scratch_.template alloc<uint8_t>(C * V);
    int* d_vfree = scratch_.template alloc<int>(vfree.size());
    double* d_vv = scratch_.template alloc<double>(vv.size());
    int* d_np = scratch_.template alloc<int>(C);
    int* d_hbw = scratch_.template alloc<int>(C);
    long long* d_ws_off = scratch_.template alloc<long long>(C);
    long long* d_dp_off = scratch_.template alloc<long long>(C);
    double* d_ws = method < 3 ? scratch_.template alloc<double>((size_t)std::max<long long>(w * chunk, 1)) : nullptr;
    double* d_x = scratch_.template alloc<double>(C * nvar);
    double* d_T = scratch_.template alloc<double>(C * S);
    double* d_recs = scratch_.template alloc<double>(C * S * gen::Rec<N>::kSize);
    double* d_coef = scratch_.template alloc<double>(C * S * TG_D * N);
    double* d_part = scratch_.template alloc<double>(C * S * TG_D);
    double* d_costs = scratch_.template alloc<double>(C);
    double* d_sv = scratch_.template alloc<double>(C * S);
    double* d_st = scratch_.template alloc<double>(C * S);
    double* d_max = scratch_.template alloc<double>(4 * C);
    double* d_mt = scratch_.template alloc<double>(C);
    int* d_mi = scratch_.template alloc<int>(C);
    double* d_total = scratch_.template alloc<double>(C);
    double* d_parts = scratch_.template alloc<double>(3 * C);
    be_.h2d(d_vo, vo.data(), sizeof(int) * (C + 1));
    be_.h2d(d_so, so.data(), sizeof(int) * (C + 1));
    be_.h2d(d_pos, pos.data(), sizeof(int) * C * S);
    be_.h2d(d_vm, vm.data(), C * V);
    be_.h2d(d_vfree, vfree.data(), sizeof(int) * vfree.size());
    be_.h2d(d_vv, vv.data(), sizeof(double) * vv.size());
    be_.h2d(d_np, np.data(), sizeof(int) * C);
    be_.h2d(d_hbw, hbw.data(), sizeof(int) * C);
    be_.h2d(d_ws_off, ws_off.data(), sizeof(long long) * C);
    be_.h2d(d_dp_off, dp_off.data(), sizeof(long long) * C);
    const ObjTerms terms = obj_terms(method, time_penalty, use_soft, soft_weight, ncon, con_deriv, con_value);
    std::vector<double> T(C * S);
    for (long long k0 = 0; k0 < K; k0 += chunk) {
      const long long kc = std::min(chunk, K - k0);
      for (long long k = 0; k < kc; ++k) std::memcpy(&T[(size_t)k * S], x + (size_t)(k0 + k) * nvar, sizeof(double) * S);
      be_.h2d(d_x, x + (size_t)k0 * nvar, sizeof(double) * (size_t)kc * nvar);
      be_.h2d(d_T, T.data(), sizeof(double) * (size_t)kc * S);
      const size_t nS = (size_t)kc * S;
      be_.for_each(nS, gen::RecordHeadFn<N>{r, d_T, d_recs});
      if (method >= 3) {
        be_.for_each(nS * TG_D, gen::SetFreeFn<N>{d_pos, d_vm, d_vfree, d_vv, d_dp_off, d_np, d_x, d_recs, d_coef, d_part});
        be_.for_each((size_t)kc, gen::SetFreeCostFn{d_vo, d_part, d_costs});
      } else {
        be_.for_each(nS * N, gen::RecordHrowFn<N>{d_recs});
        be_.for_each_warp((size_t)kc, gen::SolveFn<N>{r, d_vo, d_vm, d_vfree, d_vv, d_np, d_hbw, d_recs, d_ws_off, d_ws, d_coef, d_costs});
        counters.solves += kc;
      }
      launches(3);
      counters.segment_setups += (long long)nS;
      for (int kd = 1; kd <= 4; ++kd) {
        if (!need[kd - 1]) continue;
        switch (kd) {
          case 1: be_.for_each_scratch(nS, gen::MaxMagnitudeSegFn<N, 1>{d_coef, d_T, d_sv, d_st}); break;
          case 2: be_.for_each_scratch(nS, gen::MaxMagnitudeSegFn<N, 2>{d_coef, d_T, d_sv, d_st}); break;
          case 3: be_.for_each_scratch(nS, gen::MaxMagnitudeSegFn<N, 3>{d_coef, d_T, d_sv, d_st}); break;
          default: be_.for_each_scratch(nS, gen::MaxMagnitudeSegFn<N, 4>{d_coef, d_T, d_sv, d_st}); break;
        }
        be_.for_each((size_t)kc, MaxMagnitudeReduceFn{d_so, d_sv, d_st, d_max + (size_t)(kd - 1) * C, d_mt, d_mi});
        launches(2);
        counters.root_finds += (long long)nS;
        counters.root_finds_executed += (long long)nS;
      }
      be_.for_each((size_t)kc, ObjCombineFn{S, terms, d_T, d_costs, d_max, C, d_total, d_parts});
      launches(1);
      be_.d2h(total + k0, d_total, sizeof(double) * (size_t)kc);
      if (parts) be_.d2h(parts + 3 * (size_t)k0, d_parts, sizeof(double) * 3 * (size_t)kc);
      if (coef) be_.d2h(coef + (size_t)k0 * S * TG_D * N, d_coef, sizeof(double) * nS * TG_D * N);
    }
  }

  // dfo_batch for N-coefficient segments (tg_dfo_generic.cuh): the same search, state, groups and candidate reuse; the caller has
  // validated the inputs.  The free derivatives of dimensions d < D are variables.  vval, vval_out: [totV][N/2][4] (dimensions
  // d >= D zero); coef out: [totS][4][N].
  template <int N>
  void dfo_batch_n(int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times, const DfoParams& Q, int ncon,
                   const int* con_dim, const int* con_deriv, const double* con_value, double* coef, double* vval_out, int* code, int* n_iter,
                   double* total, double* parts) {
    dfo_groups(B, vtx_off, vmask, N / 2, D, Q.time_alloc_method >= 3, [&](int p0, int p1) {
      dfo_group_n<N>(D, p0, p1, vtx_off, vmask, vval, times, Q, ncon, con_dim, con_deriv, con_value, coef, vval_out, code, n_iter, total, parts);
    });
  }
  // the workspaces of the linear solves of one group: methods 0, 1 one per candidate, 3, 4 one per problem (the initial solve)
  struct DfoWorkspace {
    const long long* off;
    const long long* size;
    double* ws;
  };
  template <int N>
  void dfo_group_n(int D, int p0, int p1, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times, const DfoParams& Q, int ncon,
                   const int* con_dim, const int* con_deriv, const double* con_value, double* coef, double* vval_out, int* code, int* n_iter,
                   double* total, double* parts) {
    constexpr int H = N / 2, RS = gen::Rec<N>::kSize;
    scratch_.reset();
    const int G = p1 - p0, method = Q.time_alloc_method;
    const bool with_free = method >= 3;
    const size_t gv0 = (size_t)vtx_off[p0], gs0 = gv0 - (size_t)p0;
    std::vector<int> vo(G + 1), so(G + 1);
    for (int i = 0; i <= G; ++i) {
      vo[i] = vtx_off[p0 + i] - (int)gv0;
      so[i] = vo[i] - i;
    }
    const GenVertices gv = gen_vertices<N>(G, vo.data(), vmask + gv0);
    Bare bb = bare_batch(G, so.data(), Q.derivative_to_optimize);
    BatchPtrs& b = bb.b;
    const int totS = b.totS, totV = b.totV;
    b.vmask = scratch_.template alloc<uint8_t>(totV);
    b.vval = scratch_.template alloc<double>((size_t)totV * H * TG_D);
    b.vfree = scratch_.template alloc<int>(gv.vfree.size());
    b.np = scratch_.template alloc<int>(G);
    b.hbw = scratch_.template alloc<int>(G);
    b.times = scratch_.template alloc<double>(totS);
    b.coef = scratch_.template alloc<double>((size_t)totS * TG_D * N);
    b.recs = scratch_.template alloc<double>((size_t)totS * 3 * RS);
    be_.h2d(b.vmask, vmask + gv0, totV);
    be_.h2d(b.vval, vval + gv0 * H * TG_D, sizeof(double) * (size_t)totV * H * TG_D);
    be_.h2d(b.vfree, gv.vfree.data(), sizeof(int) * gv.vfree.size());
    be_.h2d(b.np, gv.np.data(), sizeof(int) * G);
    be_.h2d(b.hbw, gv.hbw.data(), sizeof(int) * G);
    be_.h2d(b.times, times + gs0, sizeof(double) * totS);
    // per-problem layout of the variables, candidates (2 n), candidate items and solve workspaces
    std::vector<DfoProb> hp(G);
    std::vector<long long> ws_off(G), ws_size(G);
    size_t totN = 0, totCand = 0, totItems = 0;
    long long ws_tot = 0;
    for (int i = 0; i < G; ++i) {
      DfoProb& P = hp[i];
      std::memset(&P, 0, sizeof(P));
      P.S = so[i + 1] - so[i];
      P.n_free = gv.np[i];
      P.n = with_free ? P.S + D * P.n_free : P.S;
      P.s0 = so[i];
      P.x0 = (int)totN;
      P.c0 = (int)totCand;
      P.i0 = (int)totItems;
      totN += (size_t)P.n;
      totCand += 2 * (size_t)P.n;
      totItems += 2 * (size_t)P.n * (size_t)(with_free ? 2 : P.S);
      ws_size[i] = (long long)gen::ws_doubles<N>(P.S, gv.np[i], gv.hbw[i]);
      ws_off[i] = ws_tot;
      ws_tot += ws_size[i] * (with_free ? 1 : 2 * P.n);
    }
    DfoBatch d;
    std::memset(&d, 0, sizeof(d));
    d.prob = scratch_.template alloc<DfoProb>(G);
    be_.h2d(d.prob, hp.data(), sizeof(DfoProb) * G);
    d.method = method;
    d.max_iter = Q.max_iterations;
    d.ipc_free = 2;
    d.f_rel = Q.f_rel;
    d.x_rel = Q.x_rel;
    d.step_rel = Q.initial_stepsize_rel;
    d.obj = obj_terms(method, Q.time_penalty, Q.use_soft_constraints, Q.soft_constraint_weight, ncon, con_deriv, con_value);
    for (int c = 0; c < ncon; ++c) d.con_dim[c] = con_dim[c];
    d.x = scratch_.template alloc<double>(totN);
    d.lo = scratch_.template alloc<double>(totN);
    d.hi = scratch_.template alloc<double>(totN);
    d.step = scratch_.template alloc<double>(totN);
    d.cand_prob = scratch_.template alloc<int>(totCand);
    d.item_cand = with_free ? nullptr : scratch_.template alloc<int>(totItems);
    d.ctot = scratch_.template alloc<double>(totCand);
    d.ccost = with_free ? nullptr : scratch_.template alloc<double>(totCand);
    d.ccoef = scratch_.template alloc<double>(totItems * TG_D * N);
    d.cpart = with_free ? scratch_.template alloc<double>(totItems * 4) : nullptr;
    bool need[4] = {false, false, false, false};
    for (int c = 0; c < ncon; ++c) need[con_deriv[c] - 1] = Q.use_soft_constraints != 0;
    d.csv = scratch_.template alloc<double>(4 * totItems);
    d.bcost = scratch_.template alloc<double>(G);
    d.bpart = scratch_.template alloc<double>((size_t)totS * 4);
    d.bsv = scratch_.template alloc<double>((size_t)4 * totS);
    d.btot = scratch_.template alloc<double>(G);
    d.bparts = scratch_.template alloc<double>((size_t)3 * G);
    d.totS = (size_t)totS;
    d.totItems = totItems;
    for (int k = 0; k < 2; ++k) {
      d.lists[k][0] = scratch_.template alloc<int>(G);
      d.lists[k][1] = scratch_.template alloc<int>(totS);
      d.lists[k][2] = scratch_.template alloc<int>(totCand);
      d.lists[k][3] = scratch_.template alloc<int>(totItems);
    }
    d.cnt = scratch_.template alloc<int>(9);
    d.b = b;
    long long* d_ws_off = scratch_.template alloc<long long>(G);
    long long* d_ws_size = scratch_.template alloc<long long>(G);
    be_.h2d(d_ws_off, ws_off.data(), sizeof(long long) * G);
    be_.h2d(d_ws_size, ws_size.data(), sizeof(long long) * G);
    const DfoWorkspace ws{d_ws_off, d_ws_size, scratch_.template alloc<double>((size_t)std::max<long long>(ws_tot, 1))};
    be_.for_each(G, DfoMapFn{d});
    launches(1);
    if (with_free) {  // x0 of the free derivatives: the linear solution at the initial times (solveLinear + getFreeConstraints)
      int* d_vo = scratch_.template alloc<int>((size_t)G + 1);
      be_.h2d(d_vo, vo.data(), sizeof(int) * ((size_t)G + 1));
      double* recs0 = scratch_.template alloc<double>((size_t)totS * RS);
      be_.for_each((size_t)totS, gen::RecordHeadFn<N>{b.r, b.times, recs0});
      be_.for_each((size_t)totS * N, gen::RecordHrowFn<N>{recs0});
      be_.for_each_warp((size_t)G, gen::SolveFn<N>{b.r, d_vo, b.vmask, b.vfree, b.vval, b.np, b.hbw, recs0, ws.off, ws.ws, b.coef, d.bcost});
      be_.for_each(totV, gen::DfoFreeInitFn<N>{d, D});
      launches(4);
      counters.solves += G;
      counters.segment_setups += totS;
    }
    be_.for_each(G, DfoBeginFn{d});
    be_.dev_memset(d.cnt, 0, 9 * sizeof(int));
    launches(1);
    dfo_base_eval_n<N>(d, D, ws, need, 1);
    int back[5];
    be_.d2h(back, d.cnt, sizeof(back));
    for (int it = 0; it < Q.max_iterations && back[0] > 0; ++it) {
      const int buf = it & 1, nbuf = buf ^ 1;
      const bool sparse = (size_t)back[0] * 2 < (size_t)G;
      const int* const* L = sparse ? d.lists[buf] : nullptr;
      const size_t nprob = sparse ? (size_t)back[1] : (size_t)G, nseg = sparse ? (size_t)back[2] : (size_t)totS;
      const size_t ncand = sparse ? (size_t)back[3] : totCand, nitem = sparse ? (size_t)back[4] : totItems;
      be_.dev_memset(d.cnt, 0, sizeof(int));
      be_.dev_memset(d.cnt + 1 + 4 * nbuf, 0, 4 * sizeof(int));
      be_.for_each(nseg * 3, gen::DfoHeadFn<N>{d, L ? L[1] : nullptr, 3, 0});
      launches(1);
      if (with_free) {
        be_.for_each(nseg * 4, gen::DfoBaseCoefFn<N>{d, L ? L[1] : nullptr, 0, D});
        dfo_maxima_n<N>(d, need, L ? L[1] : nullptr, nseg, 1, 0);
        be_.for_each(nitem, gen::DfoItemFn<N>{d, L ? L[3] : nullptr, D});
        launches(2);
      } else {
        be_.for_each(nseg * 3 * N, gen::DfoHrowFn<N>{d, L ? L[1] : nullptr, 3, 0});
        be_.for_each_warp(ncand, gen::DfoSolveFn<N>{d, 0, L ? L[2] : nullptr, ws.off, ws.size, ws.ws});
        launches(2);
      }
      dfo_maxima_n<N>(d, need, L ? L[3] : nullptr, nitem, 0, 0);
      be_.for_each(ncand, DfoTotalFn{d, L ? L[2] : nullptr});
      be_.for_each(nprob, DfoAdvanceFn{d, L ? L[0] : nullptr, nbuf});
      launches(2);
      counters.segment_setups += (long long)back[2] * 3;
      counters.evals += (long long)back[3];
      if (!with_free) counters.solves += back[3];
      for (int k = 0; k < 4; ++k)
        if (need[k]) {
          counters.root_finds += (long long)back[4] + (with_free ? back[2] : 0);
          counters.root_finds_executed += (long long)back[4] + (with_free ? back[2] : 0);
        }
      int nb[5];
      be_.d2h(nb, d.cnt, sizeof(int));
      be_.d2h(nb + 1, d.cnt + 1 + 4 * nbuf, 4 * sizeof(int));
      std::memcpy(back, nb, sizeof(back));
    }
    dfo_base_eval_n<N>(d, D, ws, need, 0);  // the final point, with coefficients and the three terms
    double* d_times = scratch_.template alloc<double>(totS);
    be_.for_each(totS, DfoTimesOutFn{d, d_times});
    launches(1);
    be_.d2h(times + gs0, d_times, sizeof(double) * totS);
    if (coef) be_.d2h(coef + gs0 * TG_D * N, b.coef, sizeof(double) * (size_t)totS * TG_D * N);
    if (vval_out && with_free) {
      double* d_vv = scratch_.template alloc<double>((size_t)totV * H * TG_D);
      be_.for_each(totV, gen::DfoVvalOutFn<N>{d, D, d_vv});
      launches(1);
      be_.d2h(vval_out + gv0 * H * TG_D, d_vv, sizeof(double) * (size_t)totV * H * TG_D);
    }
    be_.d2h(hp.data(), d.prob, sizeof(DfoProb) * G);
    for (int i = 0; i < G; ++i) {
      if (code) code[p0 + i] = hp[i].code;
      if (n_iter) n_iter[p0 + i] = hp[i].iterations;
      if (total) total[p0 + i] = hp[i].f;
    }
    if (parts) be_.d2h(parts + 3 * (size_t)p0, d.bparts, sizeof(double) * 3 * G);
  }
  // dfo_base_eval over N coefficients
  template <int N>
  void dfo_base_eval_n(const DfoBatch& d, int D, const DfoWorkspace& ws, const bool* need, int start) {
    const int G = d.b.B, totS = d.b.totS;
    be_.for_each((size_t)totS, gen::DfoHeadFn<N>{d, nullptr, 1, 1});
    if (d.method >= 3) {
      be_.for_each((size_t)totS * 4, gen::DfoBaseCoefFn<N>{d, nullptr, 1, D});
    } else {
      be_.for_each((size_t)totS * N, gen::DfoHrowFn<N>{d, nullptr, 1, 1});
      be_.for_each_warp((size_t)G, gen::DfoSolveFn<N>{d, 1, nullptr, ws.off, ws.size, ws.ws});
      launches(1);
      counters.solves += G;
    }
    dfo_maxima_n<N>(d, need, nullptr, (size_t)totS, 1, 1);
    be_.for_each((size_t)G, DfoBaseTotalFn{d, start});
    launches(3);
    counters.segment_setups += totS;
    counters.evals += G;
  }
  template <int N>
  void dfo_maxima_n(const DfoBatch& d, const bool* need, const int* list, size_t n, int base, int all) {
    for (int k = 0; k < 4; ++k) {
      if (!need[k] || n == 0) continue;
      switch (k + 1) {
        case 1: be_.for_each_scratch(n, gen::DfoMaxFn<N, 1>{d, list, base, all}); break;
        case 2: be_.for_each_scratch(n, gen::DfoMaxFn<N, 2>{d, list, base, all}); break;
        case 3: be_.for_each_scratch(n, gen::DfoMaxFn<N, 3>{d, list, base, all}); break;
        default: be_.for_each_scratch(n, gen::DfoMaxFn<N, 4>{d, list, base, all}); break;
      }
      launches(1);
      if (base && all) {
        counters.root_finds += (long long)n;
        counters.root_finds_executed += (long long)n;
      }
    }
  }

  size_t objective_chunk = (size_t)1 << 15;
  size_t sweep_chunk = (size_t)1 << 17;

 private:
  struct ExtremaScratch {
    double* polys = nullptr;
    int* degree = nullptr;
    int* counters = nullptr;
  };
  ExtremaScratch extrema_scratch(size_t n_max) {
    ExtremaScratch es;
    (void)n_max;
    es.counters = scratch_.template alloc<int>(16);  // work-item counters of the persistent extrema kernels
    return es;
  }
  // Trajectory::scaleSegmentTimesToMeetConstraints over a batch (eth/trajectory.cpp:598-692): maxima of every segment,
  // then up to 20 passes of { stretch every segment, recompute the maxima of the segments that changed, global check }.
  void scale_loop(BatchPtrs& b, const double* L9) {
    const size_t totS = (size_t)b.totS;
    ScaleFn sf{b, {}, nullptr};
    ScaleCheckFn cf{b, {}, scale_tolerance};
    for (int i = 0; i < 9; ++i) { sf.L[i] = L9[i]; cf.L[i] = L9[i]; }
    uint8_t* changed = scratch_.template alloc<uint8_t>(totS);
    uint8_t* is_bound = scratch_.template alloc<uint8_t>(totS * 9);
    uint8_t* need = scratch_.template alloc<uint8_t>(totS * 9);   // [9][totS] flags -> ordered work lists
    uint8_t* wflag = scratch_.template alloc<uint8_t>(totS);
    int* work = scratch_.template alloc<int>(totS);
    int* lists = scratch_.template alloc<int>(totS * 9);
    int* counts = scratch_.template alloc<int>(16);  // [0..8] per-quantity list lengths, [9] changed segments
    sf.changed = changed;
    be_.dev_memset(is_bound, 0, totS * 9);
    ExtremaScratch es = extrema_scratch(totS);
    // work lists are built by an order-preserving select (deterministic order; measured no faster than atomic append)
    auto run_lists = [&](const char* what) {
      for (int q = 0; q < 9; ++q) be_.select_flagged(need + (size_t)q * totS, lists + (size_t)q * totS, counts + q, (int)totS);
      be_.for_each(1, AccumCountsFn{counts, b.stats + 5});
      trace_counts(what, counts, totS);
      extrema_lists(b.coef, b.times, b.maxima, totS, lists, counts, es);
    };
    if (prune_extrema) {
      // maxima for the first pass' stretch factors: bounds, then the one quantity that can bind, then whatever is left
      double* rq = scratch_.template alloc<double>(totS * 9);
      uint8_t* qstar = scratch_.template alloc<uint8_t>(totS);
      ExtremaPruneAFn pa{b, {}, rq, qstar, need, (int)totS};
      ExtremaPruneCFn pc{b, {}, rq, qstar, need, (int)totS};
      for (int i = 0; i < 9; ++i) { pa.L[i] = L9[i]; pc.L[i] = L9[i]; }
      be_.dev_memset(need, 0, totS * 9);
      be_.for_each(totS, pa);
      run_lists("prune A (first quantity)");
      be_.dev_memset(need, 0, totS * 9);
      be_.for_each(totS, pc);
      run_lists("prune C (not certified)");
      launches(2);
    } else {
      extrema_segments(b.coef, b.times, b.maxima, totS, nullptr, nullptr, es);
      counters.root_finds_executed += (long long)totS * 9;
    }
    for (int pass = 0; pass < 20; ++pass) {
      be_.dev_memset(b.stats + 1, 0, sizeof(int));
      be_.for_each(totS, sf);
      be_.for_each(totS, ExtremaWorkFn{b.prob_of_seg, b.ps, changed, wflag});
      be_.select_flagged(wflag, work, counts + 9, (int)totS);
      // global check (eth/trajectory.cpp:660-689): certificates first, exact root finding only where they do not decide
      be_.dev_memset(need, 0, totS * 9);
      ExtremaBoundFn bf{b.coef, b.times, b.maxima, is_bound, work, counts + 9, need, (int)totS, {}, scale_tolerance};
      for (int i = 0; i < 9; ++i) bf.L[i] = L9[i];
      be_.for_each(totS, bf);
      run_lists("global check (not certified)");
      be_.for_each((size_t)b.B, cf);
      launches(4);
      int pending = 0;
      be_.d2h(&pending, b.stats + 1, sizeof(int));
      if (pending == 0) break;
      // another pass follows for `pending` problems: their certified entries must be exact before ScaleFn reads them
      be_.dev_memset(need, 0, totS * 9);
      be_.for_each(totS, ExtremaCompleteFn{b.prob_of_seg, b.ps, is_bound, need, (int)totS});
      run_lists("completion");
      launches(1);
    }
  }

  // scale_loop for N-coefficient segments: the same passes, with exact maxima for every segment that changed (no certificates)
  template <int N>
  void scale_loop_n(BatchPtrs& b, const double* L9) {
    const size_t totS = (size_t)b.totS;
    gen::ScaleFn<N> sf{b, {}, scratch_.template alloc<uint8_t>(totS)};
    ScaleCheckFn cf{b, {}, scale_tolerance};
    for (int i = 0; i < 9; ++i) { sf.L[i] = L9[i]; cf.L[i] = L9[i]; }
    uint8_t* wflag = scratch_.template alloc<uint8_t>(totS);
    int* work = scratch_.template alloc<int>(totS);
    int* n_work = scratch_.template alloc<int>(1);
    extrema_segments_n<N>(b.coef, b.times, b.maxima, totS, nullptr, nullptr);
    counters.root_finds_executed += (long long)totS * 9;
    for (int pass = 0; pass < 20; ++pass) {
      be_.dev_memset(b.stats + 1, 0, sizeof(int));
      be_.for_each(totS, sf);
      be_.for_each(totS, ExtremaWorkFn{b.prob_of_seg, b.ps, sf.changed, wflag});
      be_.select_flagged(wflag, work, n_work, (int)totS);
      extrema_segments_n<N>(b.coef, b.times, b.maxima, totS, work, n_work);
      be_.for_each((size_t)b.B, cf);
      launches(3);
      int st[2];  // stats[1]: problems still to scale
      be_.d2h(st, b.stats, sizeof(st));
      int nw = 0;
      be_.d2h(&nw, n_work, sizeof(int));
      counters.root_finds_executed += (long long)nw * 9;
      if (st[1] == 0) break;
    }
  }
  template <int N>
  void extrema_segments_n(const double* coef, const double* times, double* maxima, size_t n_max, const int* work, const int* n_dev) {
    if (n_max == 0) return;
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 0>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 1>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 2>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 3>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 4>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 5>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 6>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 7>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, gen::ExtremaFn<N, 8>{coef, times, maxima, work, n_dev});
    launches(9);
  }

  // TG_TRACE_PRUNE=1: prints how many (segment, quantity) pairs still need root finding after each certificate stage
  void trace_counts(const char* what, const int* d_counts, size_t totS) {
    static const bool on = std::getenv("TG_TRACE_PRUNE") != nullptr;
    if (!on) return;
    int c[16];
    be_.d2h(c, d_counts, sizeof(c));
    std::fprintf(stderr, "[prune] %-30s segments %zu  per quantity:", what, totS);
    for (int q = 0; q < 9; ++q) std::fprintf(stderr, " %d", c[q]);
    std::fprintf(stderr, "\n");
  }

  // exact maxima for per-quantity work lists: lists[q * n_max ..], lengths counts[q] in device memory
  void extrema_lists(const double* coef, const double* times, double* maxima, size_t n_max, const int* lists, const int* counts,
                     const ExtremaScratch& es) {
    if (n_max == 0) return;
    // the nine quantities are independent: one side stream each, so that the long tails of the root finder overlap
    be_.dev_memset(es.counters, 0, 16 * sizeof(int));
    be_.fork(9);
    be_.template extrema_refill<0>(0, n_max, coef, times, maxima, lists + 0 * n_max, counts + 0, es.counters + 0);
    be_.template extrema_refill<1>(1, n_max, coef, times, maxima, lists + 1 * n_max, counts + 1, es.counters + 1);
    be_.template extrema_refill<2>(2, n_max, coef, times, maxima, lists + 2 * n_max, counts + 2, es.counters + 2);
    be_.template extrema_refill<3>(3, n_max, coef, times, maxima, lists + 3 * n_max, counts + 3, es.counters + 3);
    be_.template extrema_refill<4>(4, n_max, coef, times, maxima, lists + 4 * n_max, counts + 4, es.counters + 4);
    be_.template extrema_refill<5>(5, n_max, coef, times, maxima, lists + 5 * n_max, counts + 5, es.counters + 5);
    be_.template extrema_refill<6>(6, n_max, coef, times, maxima, lists + 6 * n_max, counts + 6, es.counters + 6);
    be_.template extrema_refill<7>(7, n_max, coef, times, maxima, lists + 7 * n_max, counts + 7, es.counters + 7);
    be_.template extrema_refill<8>(8, n_max, coef, times, maxima, lists + 8 * n_max, counts + 8, es.counters + 8);
    be_.join(9);
    launches(9);
  }

  // per-segment maxima of the nine quantities for n_max work items (all segments, or the entries of a device work
  // list whose length lives in device memory); one launch pair per quantity so that every kernel has one degree
  void extrema_segments(const double* coef, const double* times, double* maxima, size_t n_max, const int* work, const int* n_dev,
                        const ExtremaScratch& es) {
    if (n_max == 0) return;
    (void)es;
    be_.for_each_scratch(n_max, ExtremaRawFn<0>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, ExtremaRawFn<1>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, ExtremaRawFn<2>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, ExtremaRawFn<3>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, ExtremaRawFn<4>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, ExtremaRawFn<5>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, ExtremaRawFn<6>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, ExtremaRawFn<7>{coef, times, maxima, work, n_dev});
    be_.for_each_scratch(n_max, ExtremaRawFn<8>{coef, times, maxima, work, n_dev});
    launches(9);
  }
  int group_index(const Group* g) const {
    for (size_t i = 0; i < groups_.size(); ++i)
      if (groups_[i].get() == g) return (int)i;
    return -1;
  }
  void launches(int n) { counters.launches += n; }

  BE& be_;
  Arena<BE> persist_, scratch_;
  std::vector<std::unique_ptr<Group>> groups_;
  std::vector<int> final_group_, final_index_;
  int B_ = 0;
};

}  // namespace tg

#endif  // TG_PIPELINE_HPP_
