// topolow_b200/csrc/batch.cu
//
// topolow_fit_batch: the fork-parallel fan-out of independent fits of the reference
// (parallel::mclapply over parameter samples and folds, R/adaptive_sampling.R:645-672, :1301-1320,
// :2670-2693) as ONE call.  Jobs that point at the same edge arrays share one EdgeStore; fits that run
// on one CTA are launched many per kernel (tile_batch_kernel), grouped by (ndim, precision, warps, tile).
// topolow_fit_batch_devices deals the jobs over several devices and runs each device's share on a host thread of
// its own with the same code (run_share).  Row-block jobs (large maps, ndim up to 32) run after a share's coloured
// fits have ended, one at a time, each exactly the single fit of topolow_fit.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "plan.h"
#include "rowblock.h"

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


// How the share of a batch that runs on one device learns that the batch is stopped.  A batch on one device runs its
// only share on the calling thread, which polls the caller's callback itself.  The shares of a multi-device batch run
// on worker threads that never call it (R's API is single-threaded): the calling thread waits until every share has
// been set up, polls, and when the poll fires it raises the abort word of every share at once.
class StopSource {
 public:
  // workers = 0: one share on the calling thread; otherwise the number of worker threads.
  StopSource(topolow_interrupt_fn poll, void* user, int workers)
      : poll_(poll), user_(user), workers_(workers), pending_(workers), arrived_(workers, 0) {}
  bool armed() const { return poll_ != nullptr; }
  bool fired() const { return fired_.load(); }
  // A share's abort word (mapped host memory its fits read); raised at once if the batch is already stopped.
  void attach(volatile int* w) {
    std::lock_guard<std::mutex> l(m_);
    words_.push_back(w);
    if (fired_) raise(w);
  }
  void detach(volatile int* w) {
    std::lock_guard<std::mutex> l(m_);
    words_.erase(std::remove(words_.begin(), words_.end(), w), words_.end());
  }
  // The periodic check of a share: polls (one share, on the calling thread) or reads the calling thread's decision.
  bool check() {
    if (!workers_ && poll_ && !fired_ && poll_(user_)) fire();
    return fired_;
  }
  // A share has been set up and is about to launch.  With workers: waits until every share got here (or ended) and
  // the calling thread has polled, so that no device launches before every device has loaded its kernels.
  bool ready(int share) {
    if (!workers_) return check();
    std::unique_lock<std::mutex> l(m_);
    arrived_[share] = 1;
    --pending_;
    cv_.notify_all();
    cv_.wait(l, [&] { return go_; });
    return fired_;
  }
  // A worker has returned (whether or not it reached ready()).
  void done(int share) {
    std::lock_guard<std::mutex> l(m_);
    if (!arrived_[share]) { arrived_[share] = 1; --pending_; }
    ++finished_;
    cv_.notify_all();
  }
  // The calling thread of a multi-device batch: the poll after set-up, then every kPeriod until every worker returned.
  void watch() {
    std::unique_lock<std::mutex> l(m_);
    cv_.wait(l, [&] { return pending_ == 0; });
    l.unlock();
    if (poll_ && poll_(user_)) fire();
    l.lock();
    go_ = true;
    cv_.notify_all();
    auto last = std::chrono::steady_clock::now();
    while (finished_ < workers_) {
      if (!poll_ || fired_) { cv_.wait(l, [&] { return finished_ == workers_; }); break; }
      if (cv_.wait_until(l, last + kPeriod, [&] { return finished_ == workers_; })) break;
      l.unlock();
      if (poll_(user_)) fire();
      l.lock();
      last = std::chrono::steady_clock::now();
    }
  }
  static constexpr auto kPeriod = std::chrono::milliseconds(20);

 private:
  static void raise(volatile int* w) { *w = 1; std::atomic_thread_fence(std::memory_order_seq_cst); }
  void fire() {
    std::lock_guard<std::mutex> l(m_);
    fired_ = true;
    for (volatile int* w : words_) raise(w);
  }
  topolow_interrupt_fn poll_;
  void* user_;
  const int workers_;
  std::mutex m_;
  std::condition_variable cv_;
  int pending_, finished_ = 0;
  bool go_ = false;
  std::vector<char> arrived_;
  std::vector<volatile int*> words_;
  std::atomic<bool> fired_{false};
};

// Keeps a share's abort word known to the StopSource while the block that holds it is alive.
struct AbortAttach {
  StopSource& stop;
  volatile int* word = nullptr;
  explicit AbortAttach(StopSource& s) : stop(s) {}
  void set(volatile int* w) { word = w; stop.attach(w); }
  ~AbortAttach() { if (word) stop.detach(word); }
};

// Jobs of a call that are not row-block jobs: the count the one-CTA rule is taken on, so that adding or removing
// row-block jobs never changes a coloured job's result.
int coloured_count(int n_jobs, const topolow_params* params) {
  int c = 0;
  for (int j = 0; j < n_jobs; ++j) c += params[j].mode != TOPOLOW_MODE_ROWBLOCK;
  return c;
}

// One device's share of a batch: jobs `ids` (indices into the caller's arrays) of a call with n_coloured jobs that are
// not row-block jobs, run on `device` from the current host thread; `shares` host threads run shares at the same time
// (they split the set-up threads).  Returns TOPOLOW_OK, TOPOLOW_ERR_INTERRUPTED when this share saw the stop request,
// or TOPOLOW_ERR_CUDA.
int run_share(const std::vector<int>& ids, int n_coloured, const topolow_problem* problems_in,
              const topolow_params* params_in, topolow_result* results_in, int device, int share, int shares,
              StopSource& stop) {
  const int n_jobs = (int)ids.size();
  std::vector<topolow_problem> problems(n_jobs);
  std::vector<topolow_params> params(n_jobs);
  std::vector<topolow_result*> results(n_jobs);
  for (int j = 0; j < n_jobs; ++j) {
    problems[j] = problems_in[ids[j]];
    params[j] = params_in[ids[j]];
    results[j] = &results_in[ids[j]];
  }
  // Independent fits: every job gets its own plan and stream; chunks of all jobs are issued
  // round-robin so that the device always has several fits in flight.
  std::unique_ptr<PinnedBuf<int>> flags;   // declared before the plans: outlives them
  // The abort word (when the batch can be interrupted): mapped, and 16 aligned bytes, the unit the kernels copy.
  // Each share allocates its own on its device, so the address the kernels read is valid there.
  std::unique_ptr<PinnedBuf<int>> abort_block;
  AbortAttach abort_attach(stop);
  const int* d_abort = nullptr;            // its device address
  std::vector<std::unique_ptr<topolow_plan>> plans(n_jobs);
  std::vector<int> left(n_jobs, 0);
  std::vector<char> rowblock(n_jobs, 0);   // row-block jobs still to run (one at a time, after the coloured launches)
  int rowblock_running = -1;
  const bool dbg = std::getenv("TOPOLOW_DEBUG") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  auto since = [&]() { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count(); };
  // Many independent fits: one CTA per fit (no grid barrier, plain launches that run side by side on
  // different SMs) keeps every SM busy; a lone large fit still gets the whole chip.  Decided on the coloured job count
  // of the whole call, so that a job's result does not depend on how the call was split over devices.
  auto job_params = [&](int j) {
    topolow_params pr = params[j];
    pr.device = device;
    if (n_coloured >= 16 && pr.max_ctas == 0) {
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
  // (the current device is per host thread: every set-up thread selects the share's device)
  auto run_pool = [&](int count, const std::function<void(int)>& fn) {
    const int n_threads = std::max(1, std::min<int>({(int)std::thread::hardware_concurrency() / shares, 16, count}));
    std::atomic<int> next{0};
    std::vector<std::thread> pool;
    for (int t = 0; t < n_threads; ++t)
      pool.emplace_back([&] {
        cudaSetDevice(device);
        for (int i = next.fetch_add(1); i < count; i = next.fetch_add(1)) fn(i);
      });
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
  if (dbg) std::fprintf(stderr, "[topolow] batch (device %d): %zu edge stores for %d jobs: %.3f s\n", device, slots.size(), n_jobs, since());
  // Per-job set-up (point upload, state) is independent: spread it over the host cores, as the reference
  // spreads whole fits with mclapply.
  auto setup_one = [&](int j) {
    topolow_result& r = *results[j];
    r.status = TOPOLOW_OK; r.message[0] = 0;
    try {
      if (problems[j].n < 2) {
        r.status = TOPOLOW_ERR_TOO_FEW_POINTS;
        set_msg(r.message, sizeof r.message, "Need at least 2 points for embedding");
        return;
      }
      if (params[j].mode == TOPOLOW_MODE_ROWBLOCK) { rowblock[j] = 1; return; }   // set up when its turn comes
      if (params[j].mode != TOPOLOW_MODE_COLOURED) throw BadArg("batch supports the coloured and row-block modes only");
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
  if (stop.armed() && n_jobs > 0) {
    try {
      abort_block.reset(new PinnedBuf<int>(4, cudaHostAllocMapped));   // (page-aligned)
      volatile int* w = *abort_block;
      w[0] = w[1] = w[2] = w[3] = 0;
      TL_CUDA(cudaHostGetDevicePointer((void**)&d_abort, (void*)*abort_block, 0));
      abort_attach.set(w);
    } catch (const CudaError&) {   // the fits then cannot see a stop request; the host still stops issuing launches
      cudaGetLastError();
      abort_block.reset(); d_abort = nullptr;
    }
  }
  run_pool(n_jobs, setup_one);
  if (dbg) std::fprintf(stderr, "[topolow] batch set-up of %d jobs (device %d): %.3f s\n", n_jobs, device, since());
  // Interrupt: once it fires, the abort word tells every fit on the device to stop at its next decision point and no
  // further launch is issued.
  bool aborted = false;
  auto last_poll = std::chrono::steady_clock::now();
  auto poll_now = [&]() {
    last_poll = std::chrono::steady_clock::now();
    if (stop.check()) aborted = true;
    return aborted;
  };
  constexpr auto kPollPeriod = StopSource::kPeriod;
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
    // after set-up, before the first launch (on any device of the batch)
    last_poll = std::chrono::steady_clock::now();
    if (stop.ready(share)) aborted = true;
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
        if (stop.armed() && std::chrono::steady_clock::now() - last_poll >= kPollPeriod && poll_now()) { any = false; break; }
        const int c = std::min(left[j], plans[j]->chunk_iters);
        launch_chunk(*plans[j], c, plans[j]->stream);
        left[j] -= c;
        any = true;
      }
    }
    if (dbg) std::fprintf(stderr, "[topolow] batch launches issued (device %d): %.3f s\n", device, since());
    for (auto& kv : groups) TL_CUDA(cudaEventRecord(*kv.second.ev1, *kv.second.stream));
    for (int j = 0; j < n_jobs; ++j)
      if (plans[j] && !grouped[j]) TL_CUDA(cudaEventRecord(plans[j]->ev1, plans[j]->stream));
    if (stop.armed() && !aborted) {   // wait with event queries, polling, until every fit has ended or the poll fires
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
      if (dbg) std::fprintf(stderr, "[topolow] batch %s (device %d): %.3f s\n", aborted ? "interrupted" : "fits ended", device, since());
    }
    // Row-block jobs, once the coloured fits have ended (waited for above with the poll running: row_create
    // synchronises the device, which would otherwise wait for them without a poll): one at a time in job-index order,
    // each created, run, read back and destroyed before the next (device memory is bounded by the largest job), each
    // exactly what topolow_fit returns.  The poll runs before and after each set-up; the set-up itself is not
    // interrupted.
    auto stop_requested = [&]() {
      if (!stop.armed()) return false;
      if (aborted || stop.fired()) return aborted = true;
      return std::chrono::steady_clock::now() - last_poll >= kPollPeriod && poll_now();
    };
    for (int j = 0; j < n_jobs; ++j) {
      if (!rowblock[j]) continue;
      topolow_result& r = *results[j];
      rowblock[j] = 0;
      if (stop.armed() && (aborted || poll_now())) { result_not_run(problems[j], r); continue; }
      std::unique_ptr<RowPlan, void (*)(RowPlan*)> rp(nullptr, row_destroy);
      try {
        topolow_params pr = params[j];
        pr.device = device;
        rp.reset(row_create(problems[j], pr, 0, 1));
      } catch (const CudaError& e) {   // (out of device memory): this job fails, the share goes on
        r.status = TOPOLOW_ERR_CUDA; set_msg(r.message, sizeof r.message, e.what()); cudaGetLastError();
        continue;
      } catch (const std::exception& e) {
        r.status = TOPOLOW_ERR_BAD_ARG; set_msg(r.message, sizeof r.message, e.what());
        continue;
      }
      if (stop.armed() && poll_now()) { rp.reset(); result_not_run(problems[j], r); continue; }
      rowblock_running = j;
      const bool cut = row_run_windows(*rp, stop_requested);
      // without positions to return, the hold-out cells are scored on a host copy of them
      double* const pos = r.positions;
      std::vector<double> scratch;
      if (!pos && problems[j].n_holdout > 0) {
        scratch.resize((size_t)problems[j].n * (size_t)problems[j].ndim);
        r.positions = scratch.data();
      }
      try {
        row_result(*rp, r, cut);
      } catch (const BadArg& e) {   // (hold-out cells out of range: what topolow_fit reports)
        r.status = TOPOLOW_ERR_BAD_ARG; set_msg(r.message, sizeof r.message, e.what());
      } catch (...) {
        r.positions = pos;
        throw;
      }
      r.positions = pos;
      rowblock_running = -1;
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
      fill_result(*plans[j], *results[j], cut);
    }
    if (dbg) std::fprintf(stderr, "[topolow] batch results read (device %d): %.3f s\n", device, since());
    plans.clear();
    if (dbg) std::fprintf(stderr, "[topolow] batch plans destroyed (device %d): %.3f s\n", device, since());
  } catch (const CudaError& e) {
    for (int j = 0; j < n_jobs; ++j)
      if (plans[j] || rowblock[j] || j == rowblock_running) {
        results[j]->status = TOPOLOW_ERR_CUDA; set_msg(results[j]->message, sizeof results[j]->message, e.what());
      }
    cudaGetLastError();
    return TOPOLOW_ERR_CUDA;
  }
  return aborted ? TOPOLOW_ERR_INTERRUPTED : TOPOLOW_OK;
}

// Longest first by n(n-1)/2 x n_iter (the pair updates a job may execute), each job to the share with the least work so
// far; ties to the lower job index, then to the lower list position (topolow_b200/shard.py::partition).  Each share
// keeps its jobs in index order.
std::vector<std::vector<int>> deal_jobs(int n_jobs, const topolow_problem* problems, const topolow_params* params,
                                        int n_shares) {
  std::vector<double> cost(n_jobs);
  for (int j = 0; j < n_jobs; ++j) cost[j] = 0.5 * (double)problems[j].n * (double)(problems[j].n - 1) * (double)params[j].n_iter;
  std::vector<int> order(n_jobs);
  for (int j = 0; j < n_jobs; ++j) order[j] = j;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });
  std::vector<double> load(n_shares, 0.0);
  std::vector<std::vector<int>> parts(n_shares);
  for (int j : order) {
    const int s = (int)(std::min_element(load.begin(), load.end()) - load.begin());   // (first of equal loads)
    parts[s].push_back(j);
    load[s] += cost[j];
  }
  for (auto& p : parts) std::sort(p.begin(), p.end());
  return parts;
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
  std::vector<int> all(n_jobs);
  for (int j = 0; j < n_jobs; ++j) all[j] = j;
  StopSource stop(poll, user, 0);
  return run_share(all, coloured_count(n_jobs, params), problems, params, results, device, 0, 1, stop);
}

extern "C" int topolow_fit_batch_devices(int32_t n_jobs, const topolow_problem* problems, const topolow_params* params,
                                         topolow_result* results, const int32_t* devices, int32_t n_devices,
                                         topolow_interrupt_fn poll, void* user) {
  if (n_jobs < 0 || (n_jobs > 0 && (!problems || !params || !results))) return TOPOLOW_ERR_BAD_ARG;
  auto refuse = [&](int status, const char* why) {
    if (n_jobs > 0) set_msg(results[0].message, sizeof results[0].message, why);
    return status;
  };
  if (!devices || n_devices < 1) return refuse(TOPOLOW_ERR_BAD_ARG, "devices must list at least one CUDA ordinal");
  for (int i = 0; i < n_devices; ++i)
    if (devices[i] < 0) return refuse(TOPOLOW_ERR_BAD_ARG, "device ordinal out of range");
  int count = 0;
  const cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count < 1) {
    cudaGetLastError();
    return refuse(TOPOLOW_ERR_CUDA, e != cudaSuccess ? cudaGetErrorString(e) : "no CUDA device");
  }
  for (int i = 0; i < n_devices; ++i)
    if (devices[i] >= count) return refuse(TOPOLOW_ERR_BAD_ARG, "device ordinal out of range");
  if (n_devices == 1) return topolow_fit_batch_interruptible(n_jobs, problems, params, results, devices[0], poll, user);
  if (poll && poll(user)) {
    for (int j = 0; j < n_jobs; ++j) result_not_run(problems[j], results[j]);
    return TOPOLOW_ERR_INTERRUPTED;
  }
  const std::vector<std::vector<int>> parts = deal_jobs(n_jobs, problems, params, n_devices);
  const int n_coloured = coloured_count(n_jobs, params);
  StopSource stop(poll, user, n_devices);
  std::vector<int> status(n_devices, TOPOLOW_OK);
  std::vector<std::thread> workers;
  for (int s = 0; s < n_devices; ++s)
    workers.emplace_back([&, s] {
      try {
        status[s] = run_share(parts[s], n_coloured, problems, params, results, devices[s], s, n_devices, stop);
      } catch (const std::exception& ex) {   // (host memory exhausted): the share's jobs fail, the others do not
        for (int j : parts[s]) { results[j].status = TOPOLOW_ERR_CUDA; set_msg(results[j].message, sizeof results[j].message, ex.what()); }
        status[s] = TOPOLOW_ERR_CUDA;
      }
      stop.done(s);
    });
  stop.watch();   // on the calling thread: the only caller of `poll`
  for (auto& w : workers) w.join();
  for (int s : status)
    if (s == TOPOLOW_ERR_CUDA) return TOPOLOW_ERR_CUDA;
  return stop.fired() ? TOPOLOW_ERR_INTERRUPTED : TOPOLOW_OK;
}
