// tests/cpp/oracle_estimate_times.cpp -- TEST INFRASTRUCTURE ONLY.
// The oracle's estimateSegmentTimes / estimateSegmentTimesBaca (orc_estimate_times, oracle/capi.cpp) over a ragged batch of vertex
// lists in the layout of tg_estimate_segment_times_batch, on `nthreads` host threads (problems dealt out in contiguous ranges).
// Linked against the unchanged oracle library by tests/test_segment_times.py and tools/bench_segment_times.py.
#include <algorithm>
#include <thread>
#include <vector>

extern "C" void orc_estimate_times(int V, const double* pos4, const double* limits, double* euclid, double* baca);

extern "C" void orc_estimate_times_batch(int B, const int* vtx_off, const double* pos4, const double* limits9, double* euclid, double* baca,
                                         int nthreads) {
  auto run = [&](int p0, int p1) {
    for (int p = p0; p < p1; ++p) {
      const int v0 = vtx_off[p], V = vtx_off[p + 1] - v0, s0 = v0 - p;
      orc_estimate_times(V, pos4 + 4 * (size_t)v0, limits9, euclid + s0, baca + s0);
    }
  };
  nthreads = std::max(1, std::min(nthreads, B));
  std::vector<std::thread> th;
  for (int t = 0; t < nthreads; ++t) th.emplace_back(run, (int)((long long)B * t / nthreads), (int)((long long)B * (t + 1) / nthreads));
  for (auto& t : th) t.join();
}
