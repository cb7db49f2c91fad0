// topolow_b200/csrc/batch.cu
//
// topolow_fit_batch: the fork-parallel fan-out of independent fits of the reference
// (parallel::mclapply over parameter samples and folds, R/adaptive_sampling.R:645-672, :1301-1320,
// :2670-2693) as ONE call.  Jobs that point at the same edge arrays share one EdgeStore; fits that run
// on one CTA are launched many per kernel (tile_batch_kernel), grouped by (ndim, precision, warps, tile).
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <string>
#include <thread>
#include <tuple>

#include "plan.h"

using namespace tl;

namespace {

// One launch for the next chunk of many single-CTA fits with 64-point tiles and equal (D, precision, W).
template <class real>
void launch_group(const std::vector<topolow_plan*>& members, const std::vector<int>& n_iters, cudaStream_t stream) {
  std::vector<BatchJob<real>> jobs(members.size());
  const topolow_plan& first = *members[0];
  const size_t base = tile_smem_bytes(first.D, first.geo.W, sizeof(real), first.geo.P);
  size_t smem = base;
  for (size_t i = 0; i < members.size(); ++i) {
    topolow_plan& pl = *members[i];
    jobs[i] = BatchJob<real>{device_view<real>(pl), pl.geo, pl.prm, n_iters[i], 0, pl.d_flag};
    smem = std::max(smem, with_perm_table(jobs[i].geo, base));
    pl.launches++;
  }
  AsyncBuf<BatchJob<real>> d_jobs(jobs.size(), stream);
  // (pageable source: the call returns once the source has been staged, so `jobs` may go out of scope)
  TL_CUDA(cudaMemcpyAsync(d_jobs, jobs.data(), jobs.size() * sizeof(BatchJob<real>), cudaMemcpyHostToDevice, stream));
  const topolow_plan& p0 = *members[0];
  if constexpr (sizeof(real) == 8) launch_tile_batch_f64(p0.D, p0.geo.P, d_jobs, (int)jobs.size(), p0.geo.W, smem, stream);
  else launch_tile_batch_f32(p0.D, p0.geo.P, d_jobs, (int)jobs.size(), p0.geo.W, smem, stream);
}
// Tile size of the one-CTA-per-fit path (TOPOLOW_BATCH_TILE overrides: measurement aid).
int batch_tile_points() {
  if (const char* e = std::getenv("TOPOLOW_BATCH_TILE")) { const int v = std::atoi(e); if (v == 32 || v == 64 || v == 96) return v; }
  return 64;
}

// Result of a job the batch stopped before it ran: the starting positions, no iteration.
void result_not_run(const topolow_problem& pb, topolow_result& r) {
  double* pos = r.positions;
  double* trace = r.trace_mae;
  std::memset(&r, 0, sizeof r);
  r.positions = pos; r.trace_mae = trace;
  if (pb.n < 2) {
    r.status = TOPOLOW_ERR_TOO_FEW_POINTS;
    set_msg(r.message, sizeof r.message, "Need at least 2 points for embedding");
    return;
  }
  if (pos && pb.initial_positions) std::memcpy(pos, pb.initial_positions, sizeof(double) * (size_t)pb.n * (size_t)pb.ndim);
  r.status = TOPOLOW_ERR_INTERRUPTED;
  set_msg(r.message, sizeof r.message, "interrupted");
}

}  // namespace

extern "C" int topolow_fit_batch(int32_t n_jobs, const topolow_problem* problems, const topolow_params* params,
                      topolow_result* results, int32_t device) {
  return topolow_fit_batch_interruptible(n_jobs, problems, params, results, device, nullptr, nullptr);
}

extern "C" int topolow_fit_batch_interruptible(int32_t n_jobs, const topolow_problem* problems, const topolow_params* params,
                                               topolow_result* results, int32_t device, topolow_interrupt_fn poll,
                                               void* user) {
  if (n_jobs < 0 || (n_jobs > 0 && (!problems || !params || !results))) return TOPOLOW_ERR_BAD_ARG;
  if (poll && poll(user)) {
    for (int j = 0; j < n_jobs; ++j) result_not_run(problems[j], results[j]);
    return TOPOLOW_ERR_INTERRUPTED;
  }
  // Independent fits: every job gets its own plan and stream; chunks of all jobs are issued
  // round-robin so that the device always has several fits in flight.
  std::unique_ptr<PinnedBuf<int>> flags;   // declared before the plans: outlives them
  // The abort word (when the batch can be interrupted): mapped, and 16 aligned bytes, the unit the kernels copy.
  std::unique_ptr<PinnedBuf<int>> abort_block;
  volatile int* abort_word = nullptr;
  const int* d_abort = nullptr;            // its device address
  std::vector<std::unique_ptr<topolow_plan>> plans(n_jobs);
  std::vector<int> left(n_jobs, 0);
  const bool dbg = std::getenv("TOPOLOW_DEBUG") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  auto since = [&]() { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count(); };
  // Many independent fits: one CTA per fit (no grid barrier, plain launches that run side by side on
  // different SMs) keeps every SM busy; a lone large fit still gets the whole chip.
  auto job_params = [&](int j) {
    topolow_params pr = params[j];
    pr.device = device;
    if (n_jobs >= 16 && pr.max_ctas == 0) {
      pr.max_ctas = 1;
      if (pr.tile_points == 0) pr.tile_points = batch_tile_points();
    }
    return pr;
  };
  // Jobs that point at the same edge arrays (the parameter samples of a CV grid evaluated on the same
  // fold, R/adaptive_sampling.R:2605-2667) share one relabelling and one set of bucketed records.
  struct StoreKey {
    const void *ei, *ej, *ed, *et; int64_t E, n; int P;
    bool operator<(const StoreKey& o) const {
      return std::tie(ei, ej, ed, et, E, n, P) < std::tie(o.ei, o.ej, o.ed, o.et, o.E, o.n, o.P);
    }
  };
  struct StoreSlot { std::shared_ptr<EdgeStore> store; int first_job = -1; int status = TOPOLOW_OK; std::string error; };
  std::map<StoreKey, int> key_index;
  std::vector<StoreSlot> slots;
  std::vector<int> slot_of_job(n_jobs, -1);
  for (int j = 0; j < n_jobs; ++j) {
    const topolow_problem& pb = problems[j];
    if (pb.n < 2 || pb.n > 1000000 || params[j].mode != TOPOLOW_MODE_COLOURED || params[j].n_shards > 1) continue;
    const topolow_params pr = job_params(j);
    const StoreKey key{pb.edge_i, pb.edge_j, pb.edge_dist, pb.edge_thresh, pb.n_edges, pb.n, choose_tile_points(pb.n, pr.tile_points)};
    auto it = key_index.find(key);
    if (it == key_index.end()) {
      it = key_index.emplace(key, (int)slots.size()).first;
      slots.emplace_back();
      slots.back().first_job = j;
    }
    slot_of_job[j] = it->second;
  }
  auto run_pool = [&](int count, const std::function<void(int)>& fn) {
    const int n_threads = std::max(1, std::min<int>({(int)std::thread::hardware_concurrency(), 16, count}));
    std::atomic<int> next{0};
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; ++t)
      pool.emplace_back([&] { for (int i = next.fetch_add(1); i < count; i = next.fetch_add(1)) fn(i); });
    for (auto& th : pool) th.join();
  };
  run_pool((int)slots.size(), [&](int k) {
    StoreSlot& sl = slots[k];
    const topolow_problem& pb = problems[sl.first_job];
    try {
      const topolow_params pr = job_params(sl.first_job);
      validate(pb, pr);
      const int P = choose_tile_points(pb.n, pr.tile_points);
      sl.store = make_store(pb, (int)((pb.n + 32 * P - 1) / (32 * P)), P, device);
    } catch (const CudaError& e) {
      sl.status = TOPOLOW_ERR_CUDA; sl.error = e.what(); cudaGetLastError();
    } catch (const std::exception& e) {
      sl.status = TOPOLOW_ERR_BAD_ARG; sl.error = e.what();
    }
  });
  if (dbg) std::fprintf(stderr, "[topolow] batch: %zu edge stores for %d jobs: %.3f s\n", slots.size(), n_jobs, since());
  // Per-job set-up (point upload, state) is independent: spread it over the host cores, as the reference
  // spreads whole fits with mclapply.
  auto setup_one = [&](int j) {
    topolow_result& r = results[j];
    r.status = TOPOLOW_OK; r.message[0] = 0;
    try {
      if (problems[j].n < 2) {
        r.status = TOPOLOW_ERR_TOO_FEW_POINTS;
        set_msg(r.message, sizeof r.message, "Need at least 2 points for embedding");
        return;
      }
      if (!r.positions) throw BadArg("result->positions must be caller-allocated");
      if (params[j].mode != TOPOLOW_MODE_COLOURED) throw BadArg("batch supports the coloured mode only");
      const topolow_params pr = job_params(j);
      std::shared_ptr<EdgeStore> store;
      if (slot_of_job[j] >= 0) {
        const StoreSlot& sl = slots[slot_of_job[j]];
        if (sl.status != TOPOLOW_OK) { r.status = sl.status; set_msg(r.message, sizeof r.message, sl.error.c_str()); return; }
        store = sl.store;
      }
      plans[j] = make_plan(problems[j], pr, store, flags ? (int*)*flags + 2 * j : nullptr);
      plans[j]->d_abort = d_abort;
      left[j] = pr.n_iter;
    } catch (const CudaError& e) {
      r.status = TOPOLOW_ERR_CUDA; set_msg(r.message, sizeof r.message, e.what()); cudaGetLastError();
    } catch (const std::exception& e) {
      r.status = TOPOLOW_ERR_BAD_ARG; set_msg(r.message, sizeof r.message, e.what());
    }
  };
  try {
    if (n_jobs > 0) {
      TL_CUDA(cudaSetDevice(device));
      flags.reset(new PinnedBuf<int>(2 * (size_t)n_jobs, cudaHostAllocMapped));
    }
  } catch (const CudaError&) { cudaGetLastError(); flags.reset(); }   // plans then allocate their own
  if (poll && n_jobs > 0) {
    try {
      abort_block.reset(new PinnedBuf<int>(4, cudaHostAllocMapped));   // (page-aligned)
      abort_word = *abort_block;
      abort_word[0] = abort_word[1] = abort_word[2] = abort_word[3] = 0;
      TL_CUDA(cudaHostGetDevicePointer((void**)&d_abort, (void*)*abort_block, 0));
    } catch (const CudaError&) {   // the fits then cannot see a stop request; the host still stops issuing launches
      cudaGetLastError();
      abort_block.reset(); abort_word = nullptr; d_abort = nullptr;
    }
  }
  run_pool(n_jobs, setup_one);
  if (dbg) std::fprintf(stderr, "[topolow] batch set-up of %d jobs: %.3f s\n", n_jobs, since());
  // Interrupt: from the calling thread only (R is single-threaded).  Once it fires, the abort word tells every fit on
  // the device to stop at its next decision point and no further launch is issued.
  bool aborted = false;
  auto last_poll = std::chrono::steady_clock::now();
  auto poll_now = [&]() {
    last_poll = std::chrono::steady_clock::now();
    if (poll(user)) {
      aborted = true;
      if (abort_word) { *abort_word = 1; std::atomic_thread_fence(std::memory_order_seq_cst); }
    }
    return aborted;
  };
  constexpr auto kPollPeriod = std::chrono::milliseconds(20);
  try {
    // Single-CTA fits with 64-point tiles are launched many per kernel (one CTA each), grouped by
    // (ndim, precision, warps): the device runs at most 128 kernels side by side, fewer than it has SMs.
    struct Group { std::vector<int> jobs; std::unique_ptr<StreamGuard> stream; std::unique_ptr<EventGuard> ev0, ev1; };
    std::map<std::tuple<int, int, int, int>, Group> groups;   // (ndim, precision, warps, points per lane)
    std::vector<char> grouped(n_jobs, 0);
    for (int j = 0; j < n_jobs; ++j) {
      if (!plans[j] || plans[j]->geo.G != 1 || plans[j]->geo.P > 2) continue;
      groups[std::make_tuple(plans[j]->D, plans[j]->precision, plans[j]->geo.W, plans[j]->geo.P)].jobs.push_back(j);
      grouped[j] = 1;
    }
    for (auto& kv : groups) {   // load every kernel the batch needs before the first one starts
      const int gd = std::get<0>(kv.first), gw = std::get<2>(kv.first), gp = std::get<3>(kv.first);
      if (std::get<1>(kv.first) == TOPOLOW_PREC_F64_EXACT) launch_tile_batch_f64(gd, gp, nullptr, 0, gw, 0, nullptr);
      else launch_tile_batch_f32(gd, gp, nullptr, 0, gw, 0, nullptr);
    }
    for (auto& kv : groups) {
      Group& g = kv.second;
      g.stream.reset(new StreamGuard()); g.ev0.reset(new EventGuard()); g.ev1.reset(new EventGuard());
      TL_CUDA(cudaEventRecord(*g.ev0, *g.stream));
    }
    for (int j = 0; j < n_jobs; ++j)
      if (plans[j] && !grouped[j]) TL_CUDA(cudaEventRecord(plans[j]->ev0, plans[j]->stream));
    if (poll) poll_now();   // after set-up, before the first launch
    bool any = !aborted;
    while (any) {
      any = false;
      // (reverse key order = highest ndim first: the longest fits are handed to the SMs first.  Every fit
      // of a group runs to its own stop in one launch - no chunk boundaries at which a group would have to
      // wait for its slowest member; an interrupt reaches the fits through the abort word instead.)
      for (auto it = groups.rbegin(); it != groups.rend(); ++it) {
        auto& kv = *it;
        Group& g = kv.second;
        std::vector<topolow_plan*> members; std::vector<int> iters;
        for (int j : g.jobs) {
          if (left[j] <= 0 || plans[j]->h_flag[0]) continue;
          const int c = left[j];
          members.push_back(plans[j].get()); iters.push_back(c);
          left[j] -= c;
        }
        if (members.empty()) continue;
        if (std::get<1>(kv.first) == TOPOLOW_PREC_F64_EXACT) launch_group<double>(members, iters, *g.stream);
        else launch_group<float>(members, iters, *g.stream);
        any = true;
      }
      for (int j = 0; j < n_jobs; ++j) {
        if (!plans[j] || grouped[j] || left[j] <= 0 || plans[j]->h_flag[0]) continue;
        if (poll && std::chrono::steady_clock::now() - last_poll >= kPollPeriod && poll_now()) { any = false; break; }
        const int c = std::min(left[j], plans[j]->chunk_iters);
        launch_chunk(*plans[j], c, plans[j]->stream);
        left[j] -= c;
        any = true;
      }
    }
    if (dbg) std::fprintf(stderr, "[topolow] batch launches issued: %.3f s\n", since());
    for (auto& kv : groups) TL_CUDA(cudaEventRecord(*kv.second.ev1, *kv.second.stream));
    for (int j = 0; j < n_jobs; ++j)
      if (plans[j] && !grouped[j]) TL_CUDA(cudaEventRecord(plans[j]->ev1, plans[j]->stream));
    if (poll && !aborted) {   // wait with event queries, polling, until every fit has ended or the poll fires
      std::vector<cudaEvent_t> pending;
      for (auto& kv : groups) pending.push_back(*kv.second.ev1);
      for (int j = 0; j < n_jobs; ++j)
        if (plans[j] && !grouped[j]) pending.push_back(plans[j]->ev1);
      while (true) {
        for (size_t i = 0; i < pending.size();) {
          const cudaError_t q = cudaEventQuery(pending[i]);
          if (q == cudaErrorNotReady) { ++i; continue; }
          TL_CUDA(q);
          pending[i] = pending.back();
          pending.pop_back();
        }
        if (pending.empty()) break;
        if (std::chrono::steady_clock::now() - last_poll >= kPollPeriod) {
          if (poll_now()) break;
        } else {
          std::this_thread::sleep_for(std::chrono::microseconds(200));
        }
      }
      if (cudaPeekAtLastError() == cudaErrorNotReady) cudaGetLastError();
      if (dbg) std::fprintf(stderr, "[topolow] batch %s: %.3f s\n", aborted ? "interrupted" : "fits ended", since());
    }
    for (auto& kv : groups) {
      Group& g = kv.second;
      TL_CUDA(cudaEventSynchronize(*g.ev1));
      float ms = 0.f;
      TL_CUDA(cudaEventElapsedTime(&ms, *g.ev0, *g.ev1));
      for (int j : g.jobs) plans[j]->total_ms = ms;   // the fits of a group share its launches
    }
    for (int j = 0; j < n_jobs; ++j) {
      if (!plans[j]) continue;
      if (!grouped[j]) {
        TL_CUDA(cudaEventSynchronize(plans[j]->ev1));
        float ms = 0.f;
        TL_CUDA(cudaEventElapsedTime(&ms, plans[j]->ev0, plans[j]->ev1));
        plans[j]->total_ms = ms;
      }
      // After an interrupt, a fit that neither stopped (converged, non-finite, or stopped by the abort word: that
      // one carries kStatusStopped) nor ran all its iterations was cut short on the host: it is interrupted too.
      const bool cut = aborted && !plans[j]->h_flag[0] && plans[j]->h_flag[1] < plans[j]->prm.n_iter;
      fill_result(*plans[j], results[j], cut);
    }
    if (dbg) std::fprintf(stderr, "[topolow] batch results read: %.3f s\n", since());
    plans.clear();
    if (dbg) std::fprintf(stderr, "[topolow] batch plans destroyed: %.3f s\n", since());
  } catch (const CudaError& e) {
    for (int j = 0; j < n_jobs; ++j)
      if (plans[j]) { results[j].status = TOPOLOW_ERR_CUDA; set_msg(results[j].message, sizeof results[j].message, e.what()); }
    cudaGetLastError();
    return TOPOLOW_ERR_CUDA;
  }
  return aborted ? TOPOLOW_ERR_INTERRUPTED : TOPOLOW_OK;
}

