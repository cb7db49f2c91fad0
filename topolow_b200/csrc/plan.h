// topolow_b200/csrc/plan.h - the host-side state of one fit and the helpers plan.cu and batch.cu share.
#pragma once

#include <memory>
#include <stdexcept>
#include <vector>
#include <cstdio>

#include "../../include/topolow_b200.h"
#include "edges.h"
#include "replay.h"
#include "tilepass_launch.h"

namespace tl {
// The part of a plan that depends only on the edge list and the tile geometry: the relabelling of the
// points into slots and the bucketed edge records on the device.  The fits of a CV grid that run on the
// same fold (same edge arrays) share one store (topolow_fit_batch).
struct EdgeStore {
  std::vector<int32_t> point_of_slot;  // -1 = phantom
  std::vector<int32_t> slot_of_point;
  EdgeRec* edges = nullptr;
  uint32_t* bucket_off = nullptr;
  int device = 0;
  ~EdgeStore() { DeviceScope on(device); pool_free(edges); pool_free(bucket_off); }
};

}  // namespace tl

// (global namespace: the opaque type of include/topolow_b200.h)
struct topolow_plan {
  int device = 0;
  int precision = 0;
  int64_t n = 0, E = 0;
  int D = 0;
  tl::Geometry geo{};
  tl::FitParams prm{};
  std::shared_ptr<tl::EdgeStore> store;
  // device
  void* pos = nullptr; void* best = nullptr; void* dp1 = nullptr;
  tl::FitState* state = nullptr; double* partials = nullptr; unsigned* barrier = nullptr; double* trace = nullptr;
  int64_t n_holdout = 0; int32_t* hold_si = nullptr; int32_t* hold_sj = nullptr; double* hold_truth = nullptr;   // slots of the hold-out cells
  volatile int* h_flag = nullptr; int* d_flag = nullptr; bool owns_flag = true;   // mapped host words: stop flag, iterations done
  const int* d_abort = nullptr;   // the abort word of the batch the plan runs in (mapped, owned by the batch), or null
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int chunk_iters = 1;
  int64_t launches = 0;
  int wmax = 1, ctas = 1, n_shards = 0;
  double total_ms = 0.0;
  size_t smem = 0;

  ~topolow_plan() {
    tl::DeviceScope on(device);
    if (stream) cudaStreamSynchronize(stream);   // the buffers go back to the pool in another stream's order
    tl::pool_free(pos); tl::pool_free(best); tl::pool_free(dp1);
    tl::pool_free(state); tl::pool_free(partials); tl::pool_free(barrier); tl::pool_free(trace);
    tl::pool_free(hold_si); tl::pool_free(hold_sj); tl::pool_free(hold_truth);
    if (h_flag && owns_flag) cudaFreeHost((void*)h_flag);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace tl {

struct BadArg : std::runtime_error {
  using std::runtime_error::runtime_error;
};
inline void set_msg(char* dst, int len, const char* src) {
  if (dst && len > 0) std::snprintf(dst, len, "%s", src);
}

void validate(const topolow_problem& pb, const topolow_params& pr);
int choose_tile_points(int64_t n, int requested);
// Relabelling + bucketed records of one edge list for T tiles of 32 P points.
std::shared_ptr<EdgeStore> make_store(const topolow_problem& pb, int T, int P, int device);
// shared: a store built for this edge list by the caller; shared_flag: two mapped host words the caller owns.
std::unique_ptr<topolow_plan> make_plan(const topolow_problem& pb, const topolow_params& pr,
                                        std::shared_ptr<EdgeStore> shared = nullptr, int* shared_flag = nullptr);
template <class real>
TileDev<real> device_view(const topolow_plan& pl) {
  const unsigned long long ppi = (unsigned long long)pl.n * (unsigned long long)(pl.n - 1) / 2ull;
  return TileDev<real>{(real*)pl.pos, (real*)pl.best, (const real*)pl.dp1, pl.store->edges, pl.store->bucket_off, pl.state,
                       pl.partials, pl.barrier, pl.trace, (long long)pl.E, ppi, pl.d_abort};
}
void launch_chunk(topolow_plan& pl, int n_iters, cudaStream_t stream);
void fill_result(topolow_plan& pl, topolow_result& res, bool interrupted);
void holdout_resident(const void* best, bool is_f64, int dim, int64_t n_cells, const int32_t* d_slot_i,
                      const int32_t* d_slot_j, const double* d_truth, cudaStream_t stream, double* sum_abs,
                      int64_t* count);   // post.cu

}  // namespace tl
