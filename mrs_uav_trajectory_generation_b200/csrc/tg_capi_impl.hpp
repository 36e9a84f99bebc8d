// tg_capi_impl.hpp -- the extern "C" functions of include/tg_b200.h, written once over a Backend type.
// cuda_backend.cu defines TG_BACKEND = CudaBackend and includes this file (the product, libtg_b200.so);
// tests/host_emu/emu.cpp defines TG_BACKEND = EmuBackend (test-only CPU emulation of the same code).
#ifndef TG_CAPI_IMPL_HPP_
#define TG_CAPI_IMPL_HPP_

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <exception>
#include <memory>
#include <stdexcept>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/tg_b200.h"
#include "tg_pipeline.hpp"

// A context owns one backend + pipeline ("lane 0", which serves every entry point) and, created on first use, a second
// pair ("lane 1") with its own streams and arenas.  With TG_LANES=2, tg_optimize_batch gives the two halves of a large batch
// to the two lanes on two host threads, so that one half's solves could fill the GPU while the other half sits in the tail
// of a Jenkins-Traub launch.  MEASURED on the bench workload (profiles/r01_lanes_sweep.md): no gain -- 137.0 k vs 141.7 k
// trajectories/s, at every residency cap of the solve kernel -- because the halves' launches are half as large and their tails
// relatively longer.  OFF by default; kept because the results are identical however the batch is cut (tests: two lanes, batch
// independence) and a caller with two unrelated batches can use it.
struct tg_ctx {
  TG_BACKEND be;
  tg::Pipeline<TG_BACKEND> pipe;
  std::unique_ptr<TG_BACKEND> be2;
  std::unique_ptr<tg::Pipeline<TG_BACKEND>> pipe2;
  int device;
  int lanes = 1;               // TG_LANES=2 switches the second lane on
  int lane_min_batch = 4096;   // smaller batches stay on one lane (TG_LANE_MIN_BATCH)
  bool profiling = false;      // per-kernel timing keeps everything on lane 0
  int split = 0;               // last tg_optimize_batch: problems [0, split) on lane 0, [split, B) on lane 1; 0 = one lane
  std::string err;
  std::vector<tg::Result> last;
  int last_B = 0;
  double last_ms = 0.0;
  explicit tg_ctx(int dev) : be(dev), pipe(be), device(dev) {
    if (std::getenv("TG_NO_PRUNE")) pipe.prune_extrema = false;
    if (const char* e = std::getenv("TG_LANES")) lanes = std::atoi(e);
    if (const char* e = std::getenv("TG_LANE_MIN_BATCH")) lane_min_batch = std::atoi(e);
  }
  tg::Pipeline<TG_BACKEND>& lane1() {
    if (!pipe2) {
      be2.reset(new TG_BACKEND(device));
      pipe2.reset(new tg::Pipeline<TG_BACKEND>(*be2));
      pipe2->prune_extrema = pipe.prune_extrema;
    }
    pipe2->scale_tolerance = pipe.scale_tolerance;
    return *pipe2;
  }
};

static_assert(sizeof(tg_params) == sizeof(tg::Params), "tg_params / tg::Params layout mismatch");
static_assert(sizeof(tg_result) == sizeof(tg::Result), "tg_result / tg::Result layout mismatch");

namespace {
template <class F>
int tg_guard(tg_ctx* ctx, F&& f) {
  if (!ctx) return TG_ERR_INVALID;
  try {
    ctx->err.clear();
    ctx->be.bind();
    return f();
  } catch (const std::exception& e) {
    ctx->err = e.what();
    return TG_ERR_CUDA;
  } catch (...) {
    ctx->err = "unknown error";
    return TG_ERR_CUDA;
  }
}
}  // namespace

extern "C" {

const char* tg_version(void) { return TG_VERSION_STRING; }

void tg_default_params(tg_params* p) {
  if (!p) return;
  p->derivative_to_optimize = 2;
  p->max_evals = 10;
  p->f_rel = 0.05;
  p->x_rel = 0.1;
  const double lim[9] = {4.0, 2.0, 2.0, 1.0, 20.0, 20.0, 1.0, 2.0, 10.0};  // SURVEY.md 8(d) synthetic dynamics limits
  for (int i = 0; i < 9; ++i) p->limits[i] = lim[i];
  p->dt = 0.2;
  p->check_deviation = 1;
  p->max_deviation = 0.05;
  p->max_deviation_iters = 6;
  p->first_segment_checked = 1;
  p->max_len_factor = 3.0;
  p->min_len_factor = 0.33;
  p->run_time_alloc = 1;
  p->override_heading_atan2 = 0;
}

int tg_ctx_create(int device, tg_ctx** out) {
  if (!out) return TG_ERR_INVALID;
  *out = nullptr;
  try {
    *out = new tg_ctx(device);
    return TG_OK;
  } catch (const std::exception& e) {
    std::fprintf(stderr, "tg_ctx_create: %s\n", e.what());
    return TG_ERR_NO_DEVICE;
  }
}

void tg_ctx_destroy(tg_ctx* ctx) { delete ctx; }

const char* tg_last_error(const tg_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int tg_get_counters(const tg_ctx* ctx, long long* c) {
  if (!ctx || !c) return TG_ERR_INVALID;
  const tg::Counters& k = ctx->pipe.counters;
  c[0] = k.launches; c[1] = k.solves; c[2] = k.evals; c[3] = k.root_finds; c[4] = k.segment_setups; c[5] = k.samples; c[6] = k.mellinger_solves; c[7] = k.mellinger_launches; c[8] = k.root_finds_executed;
  if (ctx->pipe2) {
    const tg::Counters& q = ctx->pipe2->counters;
    c[0] += q.launches; c[1] += q.solves; c[2] += q.evals; c[3] += q.root_finds; c[4] += q.segment_setups; c[5] += q.samples; c[6] += q.mellinger_solves; c[7] += q.mellinger_launches; c[8] += q.root_finds_executed;
  }
  return TG_OK;
}

double tg_last_device_ms(const tg_ctx* ctx) { return ctx ? ctx->last_ms : 0.0; }

int tg_get_flop_counters(const tg_ctx* ctx, double* f) {
  if (!ctx || !f) return TG_ERR_INVALID;
  const tg::Counters& k = ctx->pipe.counters;
  f[0] = k.flops_solve; f[1] = k.flops_setup; f[2] = k.flops_sample; f[3] = k.flops_coef;
  if (ctx->pipe2) {
    const tg::Counters& q = ctx->pipe2->counters;
    f[0] += q.flops_solve; f[1] += q.flops_setup; f[2] += q.flops_sample; f[3] += q.flops_coef;
  }
  return TG_OK;
}

static bool tg_params_valid(const tg_params* P) {
  if (!P) return false;
  if (P->derivative_to_optimize < 2 || P->derivative_to_optimize > 4) return false;
  if (P->max_evals < 1 || !(P->dt > 0.0) || P->max_deviation_iters < 0) return false;
  for (int i = 0; i < 9; ++i)
    if (!(P->limits[i] > 0.0)) return false;
  return true;
}

int tg_optimize_batch(tg_ctx* ctx, int B, const int* wp_off, const double* wp, const uint8_t* stop_at, const double* init14,
                      const tg_params* params, int inputs_on_device, tg_result* results, long long* totals) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 0 || !wp_off || !wp || !results || !tg_params_valid(params)) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    tg::Params P;
    std::memcpy(&P, params, sizeof(P));
    ctx->last.assign(B, tg::Result());
    ctx->last_B = B;
    ctx->split = 0;
    if (ctx->lanes >= 2 && !ctx->profiling && B >= ctx->lane_min_batch && B >= 2) ctx->split = B / 2;
    ctx->be.timer_start();
    if (ctx->split > 0) {
      const int B0 = ctx->split, B1 = B - B0;
      tg::Pipeline<TG_BACKEND>& p1 = ctx->lane1();
      std::vector<int> off1((size_t)B1 + 1);
      for (int i = 0; i <= B1; ++i) off1[i] = wp_off[B0 + i] - wp_off[B0];
      const size_t v0 = (size_t)wp_off[B0];
      std::string err1;
      std::thread t([&]() {
        try {
          ctx->be2->bind();
          p1.optimize_batch(B1, off1.data(), wp + 4 * v0, stop_at ? stop_at + v0 : nullptr, init14 ? init14 + 14 * (size_t)B0 : nullptr, P,
                            inputs_on_device != 0, ctx->last.data() + B0);
        } catch (const std::exception& e) {
          err1 = e.what();
        } catch (...) {
          err1 = "unknown error";
        }
      });
      std::string err0;
      try {
        ctx->pipe.optimize_batch(B0, wp_off, wp, stop_at, init14, P, inputs_on_device != 0, ctx->last.data());
      } catch (const std::exception& e) {
        err0 = e.what();
      }
      t.join();
      if (!err0.empty() || !err1.empty()) throw std::runtime_error(err0.empty() ? err1 : err0);
    } else if (B > 0) {
#if defined(__CUDACC__)
      const auto t0 = std::chrono::steady_clock::now();
      const double w0 = ctx->be.wait_s;
      const long long n0 = ctx->be.waits;
#endif
      ctx->pipe.optimize_batch(B, wp_off, wp, stop_at, init14, P, inputs_on_device != 0, ctx->last.data());
#if defined(__CUDACC__)
      if (ctx->be.trace_host) {
        const double tot = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        std::fprintf(stderr, "[tg] optimize_batch B=%d: %.2f ms, of which %.2f ms waiting for the device in %lld waits, %.2f ms host work\n", B,
                     1e3 * tot, 1e3 * (ctx->be.wait_s - w0), ctx->be.waits - n0, 1e3 * (tot - (ctx->be.wait_s - w0)));
      }
#endif
    }
    ctx->last_ms = ctx->be.timer_stop();  // both lanes have drained (their last calls were synchronous read-backs)
    std::memcpy(results, ctx->last.data(), sizeof(tg_result) * (size_t)B);
    if (totals) {
      ctx->pipe.output_sizes(totals, ctx->last.data());
      if (ctx->split > 0) {
        long long t1[2];
        ctx->pipe2->output_sizes(t1, ctx->last.data() + ctx->split);
        totals[0] += t1[0];
        totals[1] += t1[1];
      }
    }
    return TG_OK;
  });
}

int tg_optimize_batch_streamed(tg_ctx* ctx, int B, const int* wp_off, const double* wp, const uint8_t* stop_at, const double* init14,
                               const tg_params* params, int inputs_on_device, tg_result* results, long long* totals, double* samples_out,
                               long long samples_cap, long long* smp_begin) {
  if (!ctx) return TG_ERR_INVALID;
  if (!samples_out || samples_cap < 0 || !smp_begin || B < 0) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
  for (int p = 0; p < B; ++p) smp_begin[p] = 0;
  tg::Pipeline<TG_BACKEND>::EarlySamples& e = ctx->pipe.early;
  e.host = samples_out;
  e.cap = samples_cap;
  e.used = 0;
  e.begin = smp_begin;
  e.overflow = false;
  const int lanes = ctx->lanes;
  ctx->lanes = 1;  // one pipeline owns the stream of finished samples
  const int rc = tg_optimize_batch(ctx, B, wp_off, wp, stop_at, init14, params, inputs_on_device, results, totals);
  ctx->lanes = lanes;
  const bool overflow = e.overflow;
  e = tg::Pipeline<TG_BACKEND>::EarlySamples();
  if (rc != TG_OK) return rc;
  if (overflow) { ctx->err = "samples_out is too small (totals[1] rows are needed); the results can still be read with tg_fetch_outputs"; return TG_ERR_CAPACITY; }
  return TG_OK;
}

int tg_fetch_outputs(tg_ctx* ctx, int* seg_off, double* wp, double* times, double* coef, int* smp_off, double* samples) {
  return tg_guard(ctx, [&]() -> int {
    if (ctx->last_B <= 0) { ctx->err = "no batch result to fetch"; return TG_ERR_NO_RESULT; }
    if (ctx->split <= 0) {
      ctx->pipe.fetch_outputs(ctx->last.data(), seg_off, wp, times, coef, smp_off, samples);
      return TG_OK;
    }
    // two lanes: lane 1's ragged outputs follow lane 0's; its offsets are shifted by lane 0's totals
    const int B0 = ctx->split, B1 = ctx->last_B - B0;
    long long t0[2];
    ctx->pipe.output_sizes(t0, ctx->last.data());
    const size_t S0 = (size_t)t0[0], M0 = (size_t)t0[1];
    std::vector<int> so1, mo1;
    if (seg_off) so1.resize((size_t)B1 + 1);
    if (smp_off) mo1.resize((size_t)B1 + 1);
    std::string err1;
    std::thread t([&]() {
      try {
        ctx->be2->bind();
        ctx->pipe2->fetch_outputs(ctx->last.data() + B0, seg_off ? so1.data() : nullptr, wp ? wp + 4 * (S0 + (size_t)B0) : nullptr,
                                  times ? times + S0 : nullptr, coef ? coef + S0 * TG_D * TG_N : nullptr, smp_off ? mo1.data() : nullptr,
                                  samples ? samples + 4 * M0 : nullptr);
      } catch (const std::exception& e) {
        err1 = e.what();
      } catch (...) {
        err1 = "unknown error";
      }
    });
    std::string err0;
    try {
      ctx->pipe.fetch_outputs(ctx->last.data(), seg_off, wp, times, coef, smp_off, samples);
    } catch (const std::exception& e) {
      err0 = e.what();
    }
    t.join();
    if (!err0.empty() || !err1.empty()) throw std::runtime_error(err0.empty() ? err1 : err0);
    if (seg_off)
      for (int i = 0; i <= B1; ++i) seg_off[B0 + i] = so1[i] + (int)S0;
    if (smp_off)
      for (int i = 0; i <= B1; ++i) smp_off[B0 + i] = mo1[i] + (int)M0;
    return TG_OK;
  });
}

int tg_solve_linear_batch(tg_ctx* ctx, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, const double* times, int r,
                          double* coef, double* cost) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !vtx_off || !vmask || !vval || !times || r < 2 || r > 4) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    const bool ok = ctx->pipe.linear_batch(B, vtx_off, vmask, vval, times, r, coef, cost);
    ctx->last_ms = ctx->be.timer_stop();
    if (!ok) { ctx->err = "every problem needs at least two vertices"; return TG_ERR_INVALID; }
    return TG_OK;
  });
}

// ---- general shape (N in {6, 8, 10, 12}, D in 1..4): zero-padded to the 4 dimensions the kernels carry ------------------------
extern "C++" {
namespace {
inline bool tg_shape_ok(int N, int D) { return (N == 6 || N == 8 || N == 10 || N == 12) && D >= 1 && D <= TG_D; }
// [rows][D] -> [rows][4], missing dimensions zero
inline std::vector<double> tg_pad_dims(const double* src, size_t rows, int D) {
  std::vector<double> out(rows * TG_D, 0.0);
  for (size_t i = 0; i < rows; ++i)
    for (int d = 0; d < D; ++d) out[i * TG_D + d] = src[i * D + d];
  return out;
}
// [S][D][N] -> [S][4][N]
inline std::vector<double> tg_pad_coef(const double* coef, size_t S, int N, int D) {
  std::vector<double> out(S * TG_D * N, 0.0);
  for (size_t s = 0; s < S; ++s)
    for (int d = 0; d < D; ++d) std::memcpy(&out[(s * TG_D + d) * N], coef + (s * D + d) * N, sizeof(double) * N);
  return out;
}
// [S][4][N] -> [S][D][N]
inline void tg_strip_coef(const double* c4, size_t S, int N, int D, double* coef) {
  for (size_t s = 0; s < S; ++s)
    for (int d = 0; d < D; ++d) std::memcpy(coef + (s * D + d) * N, c4 + (s * TG_D + d) * N, sizeof(double) * N);
}
inline bool tg_segments_ok(int B, const int* seg_off) {
  for (int p = 0; p < B; ++p)
    if (seg_off[p + 1] - seg_off[p] < 1) return false;
  return true;
}
// n_free of every problem: the clear mask bits below N/2 over its vertices
inline std::vector<int> tg_free_counts(int N, int B, const int* vtx_off, const uint8_t* vmask) {
  std::vector<int> nf(B, 0);
  for (int p = 0; p < B; ++p)
    for (int v = vtx_off[p]; v < vtx_off[p + 1]; ++v)
      for (int k = 0; k < N / 2; ++k) nf[p] += ((vmask[v] >> k) & 1u) ? 0 : 1;
  return nf;
}
// free derivatives, D x n_free per problem <-> 4 x n_free per problem (dimension-major; missing dimensions zero)
inline size_t tg_free_total(const std::vector<int>& nf, int D) {
  size_t tot = 0;
  for (int n : nf) tot += (size_t)D * n;
  return tot;
}
inline std::vector<double> tg_pad_free(const double* free, const std::vector<int>& nf, int D) {
  std::vector<double> out(std::max<size_t>(tg_free_total(nf, TG_D), 1), 0.0);
  size_t i = 0, o = 0;
  for (int n : nf) {
    std::memcpy(out.data() + o, free + i, sizeof(double) * (size_t)D * n);
    i += (size_t)D * n;
    o += (size_t)TG_D * n;
  }
  return out;
}
inline void tg_strip_free(const double* f4, const std::vector<int>& nf, int D, double* free) {
  size_t i = 0, o = 0;
  for (int n : nf) {
    std::memcpy(free + o, f4 + i, sizeof(double) * (size_t)D * n);
    i += (size_t)TG_D * n;
    o += (size_t)D * n;
  }
}
template <class F>
inline void tg_dispatch_n(int N, F&& f) {
  switch (N) {
    case 6: f(std::integral_constant<int, 6>()); break;
    case 8: f(std::integral_constant<int, 8>()); break;
    case 10: f(std::integral_constant<int, 10>()); break;
    default: f(std::integral_constant<int, 12>()); break;
  }
}
}  // namespace
}  // extern "C++"

int tg_solve_linear_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, const double* times,
                             int r, double* coef, double* cost) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (B < 1 || !vtx_off || !vmask || !vval || !times || r < 0 || r > N / 2 - 1) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    const size_t totV = (size_t)vtx_off[B], totS = totV - (size_t)B;
    const std::vector<double> vv = tg_pad_dims(vval, totV * (size_t)(N / 2), D);
    std::vector<double> c4(coef ? totS * TG_D * N : 0);
    bool ok = false;
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto n) { ok = ctx->pipe.template linear_batch_n<decltype(n)::value>(B, vtx_off, vmask, vv.data(), times, r, coef ? c4.data() : nullptr, cost); });
    ctx->last_ms = ctx->be.timer_stop();
    if (!ok) { ctx->err = "every problem needs at least two vertices"; return TG_ERR_INVALID; }
    if (coef)
      for (size_t s = 0; s < totS; ++s)
        for (int d = 0; d < D; ++d) std::memcpy(coef + (s * D + d) * N, &c4[(s * TG_D + d) * N], sizeof(double) * N);
    return TG_OK;
  });
}

int tg_solve_linear_free_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval,
                                  const double* times, int r, double* coef, double* cost, double* free) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (B < 1 || !vtx_off || !vmask || !vval || !times || r < 0 || r > N / 2 - 1) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] - vtx_off[p] < 2) { ctx->err = "every problem needs at least two vertices"; return TG_ERR_INVALID; }
    const size_t totV = (size_t)vtx_off[B], totS = totV - (size_t)B;
    const std::vector<int> nf = tg_free_counts(N, B, vtx_off, vmask);
    const std::vector<double> vv = tg_pad_dims(vval, totV * (size_t)(N / 2), D);
    std::vector<double> c4(coef ? totS * TG_D * N : 0), f4(free ? std::max<size_t>(tg_free_total(nf, TG_D), 1) : 0);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto n) {
      ctx->pipe.template linear_batch_n<decltype(n)::value>(B, vtx_off, vmask, vv.data(), times, r, coef ? c4.data() : nullptr, cost,
                                                            free ? f4.data() : nullptr);
    });
    ctx->last_ms = ctx->be.timer_stop();
    if (coef) tg_strip_coef(c4.data(), totS, N, D, coef);
    if (free) tg_strip_free(f4.data(), nf, D, free);
    return TG_OK;
  });
}

int tg_set_free_constraints_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval,
                                     const double* times, int r, const double* free, double* coef, double* cost) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (B < 1 || !vtx_off || !vmask || !vval || !times || !free || r < 0 || r > N / 2 - 1) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] - vtx_off[p] < 2) { ctx->err = "every problem needs at least two vertices"; return TG_ERR_INVALID; }
    const size_t totV = (size_t)vtx_off[B], totS = totV - (size_t)B;
    const std::vector<int> nf = tg_free_counts(N, B, vtx_off, vmask);
    const std::vector<double> vv = tg_pad_dims(vval, totV * (size_t)(N / 2), D);
    const std::vector<double> f4 = tg_pad_free(free, nf, D);
    std::vector<double> c4(coef ? totS * TG_D * N : 0);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto n) {
      ctx->pipe.template set_free_batch_n<decltype(n)::value>(B, vtx_off, vmask, vv.data(), times, r, f4.data(), coef ? c4.data() : nullptr, cost);
    });
    ctx->last_ms = ctx->be.timer_stop();
    if (coef) tg_strip_coef(c4.data(), totS, N, D, coef);
    return TG_OK;
  });
}

int tg_evaluate_batch_nd(tg_ctx* ctx, int N, int D, int S, const double* coef, const double* times, int n, const double* t, int derivative,
                         double* out, uint8_t* ok) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (S < 1 || n < 0 || !coef || !times || !t || !out || derivative < 0) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    if (n == 0) return TG_OK;
    const std::vector<double> c4 = tg_pad_coef(coef, (size_t)S, N, D);
    std::vector<double> o4((size_t)n * TG_D);
    tg_dispatch_n(N, [&](auto nn) { ctx->pipe.template evaluate_batch_n<decltype(nn)::value>(S, c4.data(), times, n, t, derivative, o4.data(), ok); });
    for (size_t i = 0; i < (size_t)n; ++i)
      for (int d = 0; d < D; ++d) out[i * D + d] = o4[i * TG_D + d];
    return TG_OK;
  });
}

int tg_sample_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* seg_off, const double* coef, const double* times, double dt, int* counts,
                       double* samples, double* full) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (D < 3) { ctx->err = "Dimension has to be at least 3"; return TG_ERR_INVALID; }  // eth/trajectory_sampling.cpp:58-61
    if (B < 1 || !seg_off || !coef || !times || !counts || !(dt > 0.0)) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    const std::vector<double> c4 = tg_pad_coef(coef, (size_t)seg_off[B], N, D);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto nn) { ctx->pipe.template sample_batch_n<decltype(nn)::value>(B, seg_off, c4.data(), times, dt, counts, samples, full); });
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

namespace {
// the refusals shared by the windowed entry points; an empty string accepts
inline const char* tg_range_refusal(int N, int D, int B, const int* seg_off, const double* coef, const double* times, const double* t_range,
                                    double dt, const int* counts) {
  if (!tg_shape_ok(N, D)) return "supported shapes: N in {6, 8, 10, 12}, D in 1..4";
  if (B < 1 || !seg_off || !coef || !times || !t_range || !counts || !(dt > 0.0)) return "invalid argument";
  if (seg_off[0] != 0) return "seg_off[0] must be 0";
  for (int p = 0; p < B; ++p)
    if (seg_off[p + 1] < seg_off[p]) return "seg_off must not decrease";
  return "";
}
}  // namespace

int tg_sample_range_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* seg_off, const double* coef, const double* times,
                             const double* t_range, double dt, int* counts, double* samples, double* full, long long* t_ns) {
  return tg_guard(ctx, [&]() -> int {
    const char* why = tg_range_refusal(N, D, B, seg_off, coef, times, t_range, dt, counts);
    if (!*why && D < 3) why = "Dimension has to be at least 3";  // eth/trajectory_sampling.cpp:58-61
    if (*why) { ctx->err = why; return TG_ERR_INVALID; }
    const std::vector<double> c4 = tg_pad_coef(coef, (size_t)seg_off[B], N, D);
    bool ok = false;
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto nn) {
      ok = ctx->pipe.template sample_range_batch_n<decltype(nn)::value>(B, seg_off, c4.data(), times, t_range, dt, counts, samples, full, t_ns);
    });
    ctx->last_ms = ctx->be.timer_stop();
    if (!ok) { ctx->err = "a window's sample count passed its bound"; return TG_ERR_CAPACITY; }
    return TG_OK;
  });
}

int tg_evaluate_range_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* seg_off, const double* coef, const double* times,
                               const double* t_range, double dt, int derivative, int* counts, double* out, double* sampling_times) {
  return tg_guard(ctx, [&]() -> int {
    const char* why = tg_range_refusal(N, D, B, seg_off, coef, times, t_range, dt, counts);
    if (!*why && derivative < 0) why = "derivative must not be negative";
    if (*why) { ctx->err = why; return TG_ERR_INVALID; }
    const std::vector<double> c4 = tg_pad_coef(coef, (size_t)seg_off[B], N, D);
    bool ok = false;
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto nn) {
      ok = ctx->pipe.template evaluate_range_batch_n<decltype(nn)::value>(B, D, seg_off, c4.data(), times, t_range, dt, derivative, counts, out,
                                                                        sampling_times);
    });
    ctx->last_ms = ctx->be.timer_stop();
    if (!ok) { ctx->err = "a window's sample count passed its bound"; return TG_ERR_CAPACITY; }
    return TG_OK;
  });
}

int tg_extrema_batch_nd(tg_ctx* ctx, int N, int D, int totS, const double* coef, const double* times, double* maxima) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (totS < 1 || !coef || !times || !maxima) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    const std::vector<double> c4 = tg_pad_coef(coef, (size_t)totS, N, D);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto nn) { ctx->pipe.template extrema_batch_n<decltype(nn)::value>(totS, c4.data(), times, maxima); });
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

int tg_max_magnitude_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* seg_off, const double* coef, const double* times, int derivative,
                              double* value, double* time, int* segment_idx) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (B < 1 || !seg_off || !coef || !times || !value || !time || !segment_idx) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    if (derivative < 1 || derivative > 4) { ctx->err = "derivative must be 1..4"; return TG_ERR_INVALID; }
    if (!tg_segments_ok(B, seg_off)) { ctx->err = "every trajectory needs at least one segment"; return TG_ERR_INVALID; }
    const std::vector<double> c4 = tg_pad_coef(coef, (size_t)seg_off[B], N, D);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto nn) {
      ctx->pipe.template max_magnitude_batch_n<decltype(nn)::value>(B, seg_off, c4.data(), times, derivative, value, time, segment_idx);
    });
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

int tg_scale_times_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* seg_off, double* coef, double* times, const double* limits9,
                            int* passes, uint8_t* within) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (B < 1 || !seg_off || !coef || !times || !limits9) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    if (!tg_segments_ok(B, seg_off)) { ctx->err = "every trajectory needs at least one segment"; return TG_ERR_INVALID; }
    const size_t totS = (size_t)seg_off[B];
    std::vector<double> c4 = tg_pad_coef(coef, totS, N, D);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto nn) { ctx->pipe.template scale_times_batch_n<decltype(nn)::value>(B, seg_off, c4.data(), times, limits9, passes, within); });
    ctx->last_ms = ctx->be.timer_stop();
    tg_strip_coef(c4.data(), totS, N, D, coef);
    return TG_OK;
  });
}

int tg_time_alloc_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times,
                           const tg_params* params, double* coef, int* nlopt_code, int* n_evals, int* n_scale_passes, double* final_cost) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (B < 1 || !vtx_off || !vmask || !vval || !times || !params || params->derivative_to_optimize < 0 ||
        params->derivative_to_optimize > N / 2 - 1 || params->max_evals < 1) {
      ctx->err = "invalid argument";
      return TG_ERR_INVALID;
    }
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] - vtx_off[p] < 2) { ctx->err = "every problem needs at least two vertices"; return TG_ERR_INVALID; }
    tg::Params P;
    std::memcpy(&P, params, sizeof(P));
    const size_t totV = (size_t)vtx_off[B], totS = totV - (size_t)B;
    const std::vector<double> vv = tg_pad_dims(vval, totV * (size_t)(N / 2), D);
    std::vector<double> c4(coef ? totS * TG_D * N : 0);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto nn) {
      ctx->pipe.template time_alloc_batch_n<decltype(nn)::value>(B, vtx_off, vmask, vv.data(), times, P, coef ? c4.data() : nullptr, nlopt_code,
                                                                 n_evals, n_scale_passes, final_cost);
    });
    ctx->last_ms = ctx->be.timer_stop();
    if (coef) tg_strip_coef(c4.data(), totS, N, D, coef);
    return TG_OK;
  });
}

int tg_time_alloc_batch(tg_ctx* ctx, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times,
                        const tg_params* params, double* coef, int* nlopt_code, int* n_evals, int* n_scale_passes, double* final_cost) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !vtx_off || !vmask || !vval || !times || !params || params->derivative_to_optimize < 2 || params->derivative_to_optimize > 4 ||
        params->max_evals < 1) {
      ctx->err = "invalid argument";
      return TG_ERR_INVALID;
    }
    tg::Params P;
    std::memcpy(&P, params, sizeof(P));
    ctx->be.timer_start();
    const bool ok = ctx->pipe.time_alloc_batch(B, vtx_off, vmask, vval, times, P, coef, nlopt_code, n_evals, n_scale_passes, final_cost);
    ctx->last_ms = ctx->be.timer_stop();
    if (!ok) { ctx->err = "every problem needs at least two vertices"; return TG_ERR_INVALID; }
    return TG_OK;
  });
}

int tg_test_set_scale_tolerance(tg_ctx* ctx, double tolerance) {
  if (!ctx) return TG_ERR_INVALID;
  ctx->pipe.scale_tolerance = tolerance;
  return TG_OK;
}

int tg_test_find_roots_batch(tg_ctx* ctx, int n, const double* coeffs, const int* ncoef, double* re, double* im, int* nroots) {
  return tg_guard(ctx, [&]() -> int {
    if (n < 1 || !coeffs || !ncoef || !re || !im || !nroots) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    for (int i = 0; i < n; ++i)
      if (ncoef[i] < 0 || ncoef[i] > 16) { ctx->err = "at most 16 coefficients per polynomial"; return TG_ERR_INVALID; }
    ctx->pipe.find_roots_batch(n, coeffs, ncoef, re, im, nroots);
    return TG_OK;
  });
}

int tg_preprocess_paths(tg_ctx* ctx, int B, const int* wp_off, const double* wp, const uint8_t* stop_at, double min_waypoint_distance, int straightener_enabled,
                        double straightener_max_deviation, double straightener_max_hdg_deviation, int* out_count, double* out_wp, uint8_t* out_stop_at) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !wp_off || !wp || !out_count) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    ctx->pipe.preprocess_batch(B, wp_off, wp, stop_at, min_waypoint_distance, straightener_enabled, straightener_max_deviation,
                               straightener_max_hdg_deviation, out_count, out_wp, out_stop_at);
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

int tg_fallback_sample_batch(tg_ctx* ctx, int B, const int* wp_off, const double* wp, const uint8_t* stop_at, const double* limits9, double dt,
                             double stopping_time, int* counts, double* samples) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !wp_off || !wp || !limits9 || !counts || !(dt > 0.0)) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    ctx->pipe.fallback_batch(B, wp_off, wp, stop_at, limits9, dt, stopping_time, counts, samples);
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

int tg_waypoint_idxs_batch(tg_ctx* ctx, int B, const int* smp_off, const double* samples, const int* wp_off, const double* wp, int* counts, int* idxs) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !smp_off || !samples || !wp_off || !wp || !counts || !idxs) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    ctx->pipe.waypoint_idxs_batch(B, smp_off, samples, wp_off, wp, counts, idxs);
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

int tg_sample_batch(tg_ctx* ctx, int B, const int* seg_off, const double* coef, const double* times, double dt, int* counts,
                    double* samples, double* full) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !seg_off || !coef || !times || !counts || !(dt > 0.0)) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    ctx->pipe.sample_batch(B, seg_off, coef, times, dt, counts, samples, full);
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

int tg_evaluate_batch(tg_ctx* ctx, int S, const double* coef, const double* times, int n, const double* t, int derivative, double* out,
                      uint8_t* ok) {
  return tg_guard(ctx, [&]() -> int {
    if (S < 1 || n < 0 || !coef || !times || !t || !out || derivative < 0) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    if (n > 0) ctx->pipe.evaluate_batch(S, coef, times, n, t, derivative, out, ok);
    return TG_OK;
  });
}

int tg_extrema_batch(tg_ctx* ctx, int totS, const double* coef, const double* times, double* maxima) {
  return tg_guard(ctx, [&]() -> int {
    if (totS < 1 || !coef || !times || !maxima) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    ctx->pipe.extrema_batch(totS, coef, times, maxima);
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

int tg_max_magnitude_batch(tg_ctx* ctx, int B, const int* seg_off, const double* coef, const double* times, int derivative, double* value,
                           double* time, int* segment_idx) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !seg_off || !coef || !times || !value || !time || !segment_idx) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    for (int p = 0; p < B; ++p)
      if (seg_off[p + 1] - seg_off[p] < 1) { ctx->err = "every trajectory needs at least one segment"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    const bool ok = ctx->pipe.max_magnitude_batch(B, seg_off, coef, times, derivative, value, time, segment_idx);
    ctx->last_ms = ctx->be.timer_stop();
    if (!ok) { ctx->err = "derivative must be 1..4"; return TG_ERR_INVALID; }
    return TG_OK;
  });
}

int tg_objective_batch(tg_ctx* ctx, int V, const uint8_t* vmask, const double* vval, int r, int time_alloc_method, long long K, const double* x,
                       int nvar, double time_penalty, int use_soft_constraints, double soft_constraint_weight, int n_constraints,
                       const int* con_derivative, const double* con_value, double* total, double* parts, double* coef) {
  return tg_guard(ctx, [&]() -> int {
    if (V < 2 || !vmask || !vval || r < 2 || r > 4 || K < 1 || !x || !total || (n_constraints > 0 && (!con_derivative || !con_value))) {
      ctx->err = "invalid argument";
      return TG_ERR_INVALID;
    }
    ctx->be.timer_start();
    const int rc = ctx->pipe.objective_batch(V, vmask, vval, r, time_alloc_method, K, x, nvar, time_penalty, use_soft_constraints,
                                             soft_constraint_weight, n_constraints, con_derivative, con_value, total, parts, coef);
    ctx->last_ms = ctx->be.timer_stop();
    if (rc != 0) {
      ctx->err = rc == -2 ? "nvar must be S (methods 0, 1) or S + 4 * n_free (methods 3, 4)"
                          : (rc == -3 ? "at most 16 constraints, derivatives 1..4, non-zero values" : "time_alloc_method must be 0, 1, 3 or 4");
      return TG_ERR_INVALID;
    }
    return TG_OK;
  });
}

void tg_default_dfo_params(tg_dfo_params* p) {
  if (!p) return;
  p->time_alloc_method = 0;
  p->derivative_to_optimize = 2;
  p->max_iterations = 10;
  p->f_rel = 0.05;
  p->x_rel = 0.1;
  p->initial_stepsize_rel = 0.1;
  p->time_penalty = 500.0;
  p->use_soft_constraints = 1;
  p->soft_constraint_weight = 100.0;
}

int tg_time_alloc_dfo_batch(tg_ctx* ctx, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times,
                            const tg_dfo_params* params, int n_constraints, const int* con_dimension, const int* con_derivative,
                            const double* con_value, double* coef, double* vval_out, int* code, int* n_iterations, double* total, double* parts) {
  static_assert(sizeof(tg_dfo_params) == sizeof(tg::DfoParams), "tg_dfo_params / tg::DfoParams layout mismatch");
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !vtx_off || !vmask || !vval || !times || !params || n_constraints < 0 ||
        (n_constraints > 0 && (!con_dimension || !con_derivative || !con_value))) {
      ctx->err = "invalid argument";
      return TG_ERR_INVALID;
    }
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] - vtx_off[p] < 2) { ctx->err = "every problem needs at least two vertices"; return TG_ERR_INVALID; }
    const int m = params->time_alloc_method;
    if (!(m == 0 || m == 1 || m == 3 || m == 4)) { ctx->err = "time_alloc_method must be 0, 1, 3 or 4"; return TG_ERR_INVALID; }
    if (params->derivative_to_optimize < 2 || params->derivative_to_optimize > 4) { ctx->err = "derivative_to_optimize must be 2..4"; return TG_ERR_INVALID; }
    if (n_constraints > 16) { ctx->err = "at most 16 constraints"; return TG_ERR_INVALID; }
    for (int c = 0; c < n_constraints; ++c)
      if (con_derivative[c] < 1 || con_derivative[c] > 4 || con_dimension[c] < 0 || con_dimension[c] > 3 || !(con_value[c] != 0.0)) {
        ctx->err = "constraints need dimension 0..3, derivative 1..4 and a non-zero value";
        return TG_ERR_INVALID;
      }
    tg::DfoParams P;
    std::memcpy(&P, params, sizeof(P));
    ctx->be.timer_start();
    ctx->pipe.dfo_batch(B, vtx_off, vmask, vval, times, P, n_constraints, con_dimension, con_derivative, con_value, coef, vval_out, code,
                        n_iterations, total, parts);
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

namespace {
// the constraint rules of tg_time_alloc_dfo_batch (con_dimension may be null: tg_objective_batch_nd has no dimensions)
inline bool tg_dfo_constraints_ok(int n, const int* dim, const int* deriv, const double* value) {
  if (n < 0 || n > 16 || (n > 0 && (!deriv || !value))) return false;
  for (int c = 0; c < n; ++c)
    if (deriv[c] < 1 || deriv[c] > 4 || (dim && (dim[c] < 0 || dim[c] > 3)) || !(value[c] != 0.0)) return false;
  return true;
}
inline bool tg_dfo_method_ok(int m) { return m == 0 || m == 1 || m == 3 || m == 4; }
}  // namespace

int tg_objective_batch_nd(tg_ctx* ctx, int N, int D, int V, const uint8_t* vmask, const double* vval, int r, int time_alloc_method, long long K,
                          const double* x, int nvar, double time_penalty, int use_soft_constraints, double soft_constraint_weight,
                          int n_constraints, const int* con_derivative, const double* con_value, double* total, double* parts, double* coef) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (V < 2 || !vmask || !vval || r < 0 || r > N / 2 - 1 || K < 1 || !x || !total) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    if (!tg_dfo_method_ok(time_alloc_method)) { ctx->err = "time_alloc_method must be 0, 1, 3 or 4"; return TG_ERR_INVALID; }
    if (!tg_dfo_constraints_ok(n_constraints, nullptr, con_derivative, con_value)) {
      ctx->err = "at most 16 constraints, derivatives 1..4, non-zero values";
      return TG_ERR_INVALID;
    }
    const int S = V - 1, nf = tg_free_counts(N, 1, std::vector<int>{0, V}.data(), vmask)[0];
    const bool with_free = time_alloc_method >= 3;
    if (nvar != (with_free ? S + D * nf : S)) { ctx->err = "nvar must be S (methods 0, 1) or S + D * n_free (methods 3, 4)"; return TG_ERR_INVALID; }
    const std::vector<double> vv = tg_pad_dims(vval, (size_t)V * (N / 2), D);
    // x with the free derivatives of the missing dimensions zero: [K][S + 4 * n_free]
    const int nvar4 = with_free ? S + TG_D * nf : S;
    std::vector<double> x4;
    if (with_free && D < TG_D) {
      x4.assign((size_t)K * nvar4, 0.0);
      for (long long k = 0; k < K; ++k) std::memcpy(&x4[(size_t)k * nvar4], x + (size_t)k * nvar, sizeof(double) * nvar);
    }
    std::vector<double> c4(coef ? (size_t)K * S * TG_D * N : 0);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto n) {
      ctx->pipe.template objective_batch_n<decltype(n)::value>(V, vmask, vv.data(), r, time_alloc_method, K, x4.empty() ? x : x4.data(), nvar4,
                                                               time_penalty, use_soft_constraints, soft_constraint_weight, n_constraints,
                                                               con_derivative, con_value, total, parts, coef ? c4.data() : nullptr);
    });
    ctx->last_ms = ctx->be.timer_stop();
    if (coef) tg_strip_coef(c4.data(), (size_t)K * S, N, D, coef);
    return TG_OK;
  });
}

int tg_time_alloc_dfo_batch_nd(tg_ctx* ctx, int N, int D, int B, const int* vtx_off, const uint8_t* vmask, const double* vval, double* times,
                               const tg_dfo_params* params, int n_constraints, const int* con_dimension, const int* con_derivative,
                               const double* con_value, double* coef, double* vval_out, int* code, int* n_iterations, double* total,
                               double* parts) {
  return tg_guard(ctx, [&]() -> int {
    if (!tg_shape_ok(N, D)) { ctx->err = "supported shapes: N in {6, 8, 10, 12}, D in 1..4"; return TG_ERR_INVALID; }
    if (B < 1 || !vtx_off || !vmask || !vval || !times || !params) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] - vtx_off[p] < 2) { ctx->err = "every problem needs at least two vertices"; return TG_ERR_INVALID; }
    if (!tg_dfo_method_ok(params->time_alloc_method)) { ctx->err = "time_alloc_method must be 0, 1, 3 or 4"; return TG_ERR_INVALID; }
    if (params->derivative_to_optimize < 0 || params->derivative_to_optimize > N / 2 - 1) {
      ctx->err = "derivative_to_optimize must be 0 .. N/2-1";
      return TG_ERR_INVALID;
    }
    if (!tg_dfo_constraints_ok(n_constraints, con_dimension, con_derivative, con_value) || (n_constraints > 0 && !con_dimension)) {
      ctx->err = "at most 16 constraints, with dimension 0..3, derivative 1..4 and a non-zero value";
      return TG_ERR_INVALID;
    }
    tg::DfoParams P;
    std::memcpy(&P, params, sizeof(P));
    const size_t totV = (size_t)vtx_off[B], totS = totV - (size_t)B, H = (size_t)(N / 2);
    const std::vector<double> vv = tg_pad_dims(vval, totV * H, D);
    std::vector<double> c4(coef ? totS * TG_D * N : 0), v4(vval_out ? totV * H * TG_D : 0);
    ctx->be.timer_start();
    tg_dispatch_n(N, [&](auto n) {
      ctx->pipe.template dfo_batch_n<decltype(n)::value>(D, B, vtx_off, vmask, vv.data(), times, P, n_constraints, con_dimension, con_derivative,
                                                         con_value, coef ? c4.data() : nullptr, vval_out ? v4.data() : nullptr, code,
                                                         n_iterations, total, parts);
    });
    ctx->last_ms = ctx->be.timer_stop();
    if (coef) tg_strip_coef(c4.data(), totS, N, D, coef);
    if (vval_out) {
      if (P.time_alloc_method >= 3) {
        for (size_t i = 0; i < totV * H; ++i)
          for (int d = 0; d < D; ++d) vval_out[i * D + d] = v4[i * TG_D + d];
      }
    }
    return TG_OK;
  });
}

int tg_scale_times_batch(tg_ctx* ctx, int B, const int* seg_off, double* coef, double* times, const double* limits9, int* passes,
                         uint8_t* within) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !seg_off || !coef || !times || !limits9) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    ctx->pipe.scale_times_batch(B, seg_off, coef, times, limits9, passes, within);
    return TG_OK;
  });
}

int tg_estimate_segment_times_batch(tg_ctx* ctx, int B, const int* vtx_off, const double* pos4, const double* limits8, double* euclid,
                                    double* baca) {
  return tg_guard(ctx, [&]() -> int {
    if (B < 1 || !vtx_off || !pos4 || !limits8 || (!euclid && !baca)) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    if (vtx_off[0] != 0) { ctx->err = "vtx_off[0] must be 0"; return TG_ERR_INVALID; }
    for (int p = 0; p < B; ++p)
      if (vtx_off[p + 1] <= vtx_off[p]) { ctx->err = "every vertex list needs at least one vertex"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    ctx->pipe.estimate_times_batch(B, vtx_off, pos4, limits8, euclid, baca);
    ctx->last_ms = ctx->be.timer_stop();
    return TG_OK;
  });
}

int tg_sweep_costs(tg_ctx* ctx, int V, const uint8_t* vmask, const double* vval, int r, long long K, const double* cand, int cand_on_device,
                   double* costs, long long* best_index, double* best_cost) {
  return tg_guard(ctx, [&]() -> int {
    if (V < 2 || !vmask || !vval || !cand || K < 1 || r < 2 || r > 4) { ctx->err = "invalid argument"; return TG_ERR_INVALID; }
    ctx->be.timer_start();
    const bool ok = ctx->pipe.sweep_costs(V, vmask, vval, r, K, cand, cand_on_device != 0, costs, best_index, best_cost);
    ctx->last_ms = ctx->be.timer_stop();
    return ok ? TG_OK : TG_ERR_INVALID;
  });
}

int tg_sweep_best(tg_ctx* const* ctxs, int n_ctx, int V, const uint8_t* vmask, const double* vval, int r, long long K, const double* cand,
                  long long* best_index, double* best_cost, double* best_times) {
  if (!ctxs || n_ctx < 1 || !ctxs[0]) return TG_ERR_INVALID;
  for (int g = 0; g < n_ctx; ++g)
    if (!ctxs[g]) return TG_ERR_INVALID;
  if (V < 2 || !vmask || !vval || !cand || K < 1 || r < 2 || r > 4 || !best_index || !best_cost) {
    ctxs[0]->err = "invalid argument";
    return TG_ERR_INVALID;
  }
  const int S = V - 1;
  const int G = (int)std::min<long long>(n_ctx, K);
  std::vector<int> rc(G, TG_OK);
  std::vector<long long> idx(G, 0);
  std::vector<double> cost(G, 0.0);
  // contiguous shards of the candidate list, one host thread per context (each context owns its device and stream); the only
  // exchange is the (cost, index) pair each shard returns
  auto shard = [&](int g) {
    const long long k0 = K * g / G, k1 = K * (g + 1) / G;
    long long bi = 0;
    rc[g] = tg_sweep_costs(ctxs[g], V, vmask, vval, r, k1 - k0, cand + (size_t)k0 * S, 0, nullptr, &bi, &cost[g]);
    idx[g] = k0 + bi;
  };
  if (G == 1) {
    shard(0);
  } else {
    std::vector<std::thread> workers;
    for (int g = 0; g < G; ++g) workers.emplace_back(shard, g);
    for (std::thread& t : workers) t.join();
  }
  int best = -1;
  for (int g = 0; g < G; ++g) {
    if (rc[g] != TG_OK) {
      if (g != 0) ctxs[0]->err = ctxs[g]->err;
      return rc[g];
    }
    // first minimum of the whole list: shards are in index order, so a strictly smaller cost is required to move on;
    // a NaN cost never wins against a number (a serial `cost < best` scan behaves the same)
    if (best < 0 || cost[g] < cost[best] || (cost[best] != cost[best] && cost[g] == cost[g])) best = g;
  }
  *best_index = idx[best];
  *best_cost = cost[best];
  if (best_times)
    for (int i = 0; i < S; ++i) best_times[i] = cand[(size_t)idx[best] * S + i];
  return TG_OK;
}

double tg_detmath_eval(int fn, double x, double y) {
  switch (fn) {
    case 0: return tgdm::dlog(x);
    case 1: return tgdm::dexp(x);
    case 2: return tgdm::dsin(x);
    case 3: return tgdm::dcos(x);
    case 4: return tgdm::datan2(x, y);
    case 5: return tgdm::dcbrt(x);
    case 6: {
      double pw[64];
      const int e = (int)y;
      if (e < 1 || e > 64) return 0.0;
      tgdm::powers(x, e, pw);
      return pw[e - 1];
    }
  }
  return 0.0;
}

}  // extern "C"

#endif  // TG_CAPI_IMPL_HPP_
