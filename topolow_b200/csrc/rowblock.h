// topolow_b200/csrc/rowblock.h - host interface of the row-block ("owner computes") mode, rowblock.cu.
#pragma once
#include <cstdint>
#include <functional>
#include <vector>

#include "../../include/topolow_b200.h"
#include "common.cuh"

namespace tl {

constexpr int kMaxShards = 16;          // replicas of one map (GPUs of one NVSwitch domain)
constexpr int kRowTile = 256;           // rows of one repulsion work item; slot count and shard bounds are multiples of it
constexpr int kChunk = 2048;            // partner slots of one repulsion work item (fixed: the summation tree of a
                                        // point's repulsion must not depend on the number of shards)
constexpr int kBlockRows = 128;         // rows of one spring / MAE CTA = rows behind one reduction entry

struct RowPlan;

RowPlan* row_create(const topolow_problem& pb, const topolow_params& pr, int rank, int n_ranks);   // throws BadArg / CudaError
void row_destroy(RowPlan* rp);
// Up to n_iters further iterations (stops on convergence); returns CUDA-event milliseconds.
double row_run(RowPlan& rp, int n_iters, cudaStream_t stream, topolow_interrupt_fn poll, void* user, bool* interrupted);
// The loop of a row-block job of a fit batch (single rank): every remaining iteration, in windows of 5 on the plan's
// stream with an event after each and at most two windows queued; waits with event queries, calling `stop` (the
// batch's stop check, which rate-limits its own poll) every 200 us.  When `stop` returns true no further window is
// issued and the queued ones finish (at most 10 iterations).  Returns true when that cut the fit short (it had not
// converged, failed or issued all its iterations); the CUDA-event time is added to the plan's device time.
bool row_run_windows(RowPlan& rp, const std::function<bool()>& stop);
// All replicas of a map that live in this process: same device = lock-step emulation on one stream (every
// wait is already satisfied when its kernel starts), distinct devices = concurrent.
double row_run_local(RowPlan* const* plans, int n, int n_iters);
void row_result(RowPlan& rp, topolow_result& res, bool interrupted);
// {slots, ndim, stride, shards, rank, row0, own_rows, chunks, records, mae_records, launches, iterations_done,
//  stopped, exchange_bytes_per_iter, repulse_items, repulse_ctas}
void row_info(const RowPlan& rp, int64_t* out, int cap);
// Average milliseconds per kernel over n_iters iterations, events around every launch:
// {repulse, spring, mae, controller, snapshot, mae_launches}
void row_time_kernels(RowPlan& rp, int n_iters, double* out, int cap);

size_t row_handle_bytes();
void row_export(RowPlan& rp, void* blob);                              // this replica's shared block (CUDA IPC)
void row_attach(RowPlan& rp, const void* blobs, int n_blobs);          // blobs of all ranks, rank order
void row_attach_local(RowPlan* const* plans, int n);                   // all replicas in this process

}  // namespace tl
