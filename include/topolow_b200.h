/* include/topolow_b200.h
 *
 * C ABI of libtopolow_b200.so: the B200 (sm_100a) drop-in for topolow's native
 * hot path.  Plain pointers and sizes only.  Citations are relative to the
 * reference tree (/root/reference).
 *
 * What each entry point replaces:
 *
 *   topolow_optimize_layout_exact()   the body behind the .Call symbol
 *       _topolow_optimize_layout_exact_cpp (src/RcppExports.cpp:16-39, arity 16,
 *       registered at :41-49), i.e. optimize_layout_exact_cpp
 *       (src/optimization.cpp:108-126): same 16 arguments in the same order and
 *       meaning, R objects flattened to (pointer, size); same five results
 *       (src/optimization.cpp:375-381).
 *   topolow_fit()                     the same call in struct form, plus the
 *       B200 extensions (mode, precision, seed, explicit pair order, trace).
 *   topolow_fit_batch()               the fork-parallel fan-out of independent
 *       fits: parallel::mclapply over parameter samples / folds
 *       (R/adaptive_sampling.R:645-672, :1301-1320, :2670-2693).  One call, many
 *       fits, per-job status instead of exceptions (:2657-2666).
 *       topolow_fit_batch_interruptible() is the same call with a user-interrupt callback.
 *   topolow_plan_*()                  device-resident form of one fit for callers
 *       that keep inputs in HBM and step the loop themselves (bench, sharded map).
 *   topolow_est_distances()           as.matrix(stats::dist(positions)), R/core.R:474.
 *   topolow_holdout_errors()          the OutSampleError reduction of
 *       error_calculator_comparison (R/error_metrics.R:95-114) as consumed by
 *       likelihood_function (R/adaptive_sampling.R:2639-2647).
 *
 * Error behaviour mirrors Rcpp::stop (src/optimization.cpp:131,359-361): status
 * TOPOLOW_ERR_TOO_FEW_POINTS / TOPOLOW_ERR_NONFINITE carry the reference's two
 * messages in result->message; the R shim turns them into Rf_error.
 * No CPU fallback exists: without a usable CUDA device every compute entry
 * returns TOPOLOW_ERR_CUDA.
 */
#ifndef TOPOLOW_B200_H
#define TOPOLOW_B200_H

#include <stdint.h>

#if defined(__GNUC__)
#define TOPOLOW_API __attribute__((visibility("default")))
#else
#define TOPOLOW_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

enum {
  TOPOLOW_OK = 0,
  TOPOLOW_ERR_BAD_ARG = 1,        /* message says which */
  TOPOLOW_ERR_NONFINITE = 2,      /* "Numerical instability at iteration %d. Reduce k0 or c_repulsion." */
  TOPOLOW_ERR_CUDA = 3,           /* CUDA runtime / no device; message holds cudaGetErrorString */
  TOPOLOW_ERR_TOO_FEW_POINTS = 4, /* "Need at least 2 points for embedding" */
  TOPOLOW_ERR_INTERRUPTED = 5     /* interrupt callback returned non-zero */
};

/* mode */
enum {
  TOPOLOW_MODE_COLOURED = 0, /* production: hierarchical tournament of matchings (every pair once
                                per iteration, updates within a matching commute); ndim 1..16 */
  TOPOLOW_MODE_REPLAY = 1,   /* FP64, consumes a given / seeded std::mt19937 pair permutation and
                                executes it by dependency levels: exactly the sequential loop; any ndim */
  TOPOLOW_MODE_ROWBLOCK = 2  /* relaxed, for large maps: every point's update is computed by the owner of its row
                                against a replica of all positions (Gauss-Seidel along a row, Jacobi across
                                rows); FP32; the scheme topolow_shard_* spreads over several GPUs.  ndim 1..32:
                                1..16 with the tensor-core repulsion pass, 17..32 with the FP32 difference form
                                only (TOPOLOW_ERR_BAD_ARG beyond 32 and for another form asked for by name) */
};
/* precision (coloured mode) */
enum {
  TOPOLOW_PREC_F32 = 0,      /* FP32 FMA forces and positions, FP64 error sums and controller */
  TOPOLOW_PREC_F64_EXACT = 1 /* IEEE double, one rounding per reference operation (bit-comparable
                                with the CPU loop run on the same pair order) */
};

typedef struct {
  int64_t n;                        /* points (rows of initial_positions) */
  int32_t ndim;                     /* columns of initial_positions */
  int64_t n_edges;                  /* measured upper-triangle pairs (R/core.R:383-402) */
  const int32_t* edge_i;            /* 0-based */
  const int32_t* edge_j;            /* 0-based, edge_i[e] != edge_j[e] */
  const double* edge_dist;          /* target distance */
  const int32_t* edge_thresh;       /* 0 exact, +1 '>' , -1 '<'  (R/core.R:346,358-359) */
  const int32_t* degrees;           /* rowSums(!is.na), diagonal included (R/core.R:340-341) */
  const double* initial_positions;  /* n x ndim, column-major like an R matrix */
  /* ---- optional: cells held out of this fit, scored on the final (best) positions before they leave
   * the device (the OutSampleError reduction of R/error_metrics.R:95-114 as pooled by
   * R/adaptive_sampling.R:2642-2647; same numbers as topolow_holdout_errors on the returned positions).
   * n_holdout = 0 (all-zero tail) = none. ---- */
  int64_t n_holdout;
  const int32_t* holdout_i;         /* 0-based rows */
  const int32_t* holdout_j;
  const double* holdout_truth;      /* true dissimilarity of the cell; NaN = dropped */
} topolow_problem;

typedef struct {
  int32_t n_iter;                   /* mapping_max_iter */
  double k0;
  double cooling_rate;
  double c_repulsion;
  double relative_epsilon;
  int32_t convergence_window;       /* convergence_counter */
  int32_t convergence_check_freq;   /* < 1 means 10 (src/optimization.cpp:181) */
  int32_t verbose;                  /* print "Iter a/b, MAE=..., k=..." lines to stderr */
  /* ---- B200 extensions (all-zero = production defaults) ---- */
  int32_t mode;                     /* TOPOLOW_MODE_* */
  int32_t precision;                /* TOPOLOW_PREC_* */
  uint64_t seed;                    /* schedule seed (coloured) / std::mt19937 seed (replay) */
  const int32_t* pair_order;        /* replay only, optional: [n_iter][pairs_per_iter][2]; i<0 = skip */
  int64_t pairs_per_iter;
  int32_t device;                   /* CUDA device ordinal */
  int32_t max_ctas;                 /* 0 = all SMs; cap on the persistent grid (tests / sharing) */
  int32_t max_warps;                /* 0 = policy default; cap on warps (tiles) per CTA - lets an FP32 run use
                                       the schedule an FP64 run of the same problem gets */
  int32_t tile_points;              /* 0 = auto; 32, 64 or 96: points per tile (1, 2 or 3 per lane) */
  int32_t n_shards;                 /* > 1: the map will be stepped job by job by that many ranks (see
                                       topolow_plan_run_job); pads the tile count to a multiple of 2 * n_shards */
} topolow_params;

typedef struct {
  double* positions;                /* caller-allocated n x ndim, column-major; best state */
  int32_t converged;
  int32_t iterations;               /* best_iter (src/optimization.cpp:378) */
  double final_mae;                 /* best_mae */
  double final_k;                   /* best_k */
  int32_t status;                   /* TOPOLOW_* */
  int32_t fail_iter;                /* iteration for TOPOLOW_ERR_NONFINITE */
  int32_t iterations_run;           /* iterations actually executed */
  int64_t pair_updates;             /* pair visits executed */
  double device_ms;                 /* CUDA-event time of the optimisation kernels */
  double* trace_mae;                /* optional, length n_iter; NaN where no check ran */
  double holdout_sum_abs;           /* sum |truth - ||x_i - x_j||| over the problem's hold-out cells (0 if none) */
  int64_t holdout_count;            /* cells that entered the sum */
  char message[256];
} topolow_result;

/* R_CheckUserInterrupt equivalent; non-zero aborts.  Polled between device chunks by topolow_fit_interruptible,
 * while the fits run by topolow_fit_batch_interruptible. */
typedef int (*topolow_interrupt_fn)(void* user);

/* ---- single fit ------------------------------------------------------- */
TOPOLOW_API int topolow_fit(const topolow_problem* problem, const topolow_params* params, topolow_result* result);

TOPOLOW_API int topolow_fit_interruptible(const topolow_problem* problem, const topolow_params* params,
                              topolow_result* result, topolow_interrupt_fn poll, void* user);

/* The reference's 16 arguments, flattened.  dissimilarity_matrix and
 * threshold_matrix (n x n, column-major, Inf = unmeasured) may be NULL: they
 * are redundant with the edge list (both come from the same upper triangle,
 * R/core.R:383-402,429-436) and are only validated when given. */
TOPOLOW_API int topolow_optimize_layout_exact(
    const double* initial_positions, int32_t n, int32_t ndim, const double* dissimilarity_matrix,
    const int32_t* threshold_matrix, const int32_t* degrees, const int32_t* edge_i,
    const int32_t* edge_j, const double* edge_dist, const int32_t* edge_thresh, int64_t n_edges,
    int32_t n_iter, double k0, double cooling_rate, double c_repulsion, double relative_epsilon,
    int32_t convergence_window, int32_t convergence_check_freq, int32_t verbose,
    double* positions_out, int32_t* converged_out, int32_t* iterations_out, double* final_mae_out,
    double* final_k_out, char* message, int32_t message_len);

/* ---- batch of independent fits ----------------------------------------- */
/* Jobs run concurrently on `device` (params[j].device is ignored); results[j].status is
 * per job and the call itself only fails for argument / CUDA set-up errors.
 * Modes: params[j].mode is TOPOLOW_MODE_COLOURED or TOPOLOW_MODE_ROWBLOCK; a TOPOLOW_MODE_REPLAY job fails alone with
 * TOPOLOW_ERR_BAD_ARG.
 *   - Coloured jobs run first.  With 16 or more coloured jobs in the call (every job that is not a row-block job
 *     counts) every coloured fit runs on one CTA (64-point tiles unless tile_points is set) and the fits are launched
 *     many per kernel.  Jobs whose edge_i / edge_j / edge_dist / edge_thresh POINTERS (and n, n_edges) are equal share
 *     one set of device records: hand the parameter samples of a CV grid the same arrays per fold.
 *   - Row-block jobs (large maps, ndim 1..32) run after the coloured fits of the call (of the share, for
 *     topolow_fit_batch_devices) have ended, one at a time in job order, each created, run, read back and destroyed before the next: device memory is bounded by the largest job.
 *     Each result is bit for bit what topolow_fit returns for the same problem and params on `device` (positions,
 *     MAE, k, iterations, iterations_run, pair_updates, hold-out sums, trace, status and message, including the
 *     single fit's argument checks); device_ms is the job's own CUDA-event time.  No records are shared between them.
 *   - results[j].positions may be NULL (not topolow_fit's): the positions are then not returned, and the hold-out
 *     sums are the same as with positions.
 * topolow_fit_batch is topolow_fit_batch_interruptible with poll = NULL. */
TOPOLOW_API int topolow_fit_batch(int32_t n_jobs, const topolow_problem* problems, const topolow_params* params,
                      topolow_result* results, int32_t device);

/* The same batch, stoppable.  `poll` is called from the calling thread only: once before set-up, once after set-up
 * (before the first launch), before and after the set-up of each row-block job, then at least every 100 ms (every
 * 20 ms today) while any fit of the batch is on the device, and not again once every fit has ended.  When it returns non-zero the library raises the batch's abort
 * word (mapped host memory the kernels read), issues no further launch, waits for every stream and returns
 * TOPOLOW_ERR_INTERRUPTED with every result filled in:
 *   - a job that had already ended (converged, ran all its iterations, non-finite) keeps the result it has without
 *     the interrupt (positions, MAE, iterations and hold-out sums bit for bit);
 *   - a job that was stopped has status TOPOLOW_ERR_INTERRUPTED, message "interrupted", iterations_run = the
 *     iterations it completed, and the best state, trace, pair count and hold-out sums as of its last completed
 *     iteration (before set-up: the starting positions and no iteration);
 *   - a job that failed set-up (or has n < 2) keeps its status.
 * How soon a fit stops: a fit on one CTA (every fit of a batch of 16 or more jobs) at the end of the iteration
 * it is running; a fit on several CTAs at its next convergence check or finite check, i.e. after at most
 * min(convergence_check_freq, 10) more iterations; a row-block job at an iteration boundary within 10 iterations (the
 * host keeps at most 10 of its iterations queued); a fit or chunk that had not started yet does not start.  The
 * set-up of a row-block job (record build and uploads) is not interrupted mid-way.
 * Everything the batch allocated is released before the call returns, the abort word included. */
TOPOLOW_API int topolow_fit_batch_interruptible(int32_t n_jobs, const topolow_problem* problems,
                                                const topolow_params* params, topolow_result* results, int32_t device,
                                                topolow_interrupt_fn poll, void* user);

/* The same batch spread over several GPUs from one process (R runs in one process, and a forked child cannot use a
 * CUDA context its parent holds).  `devices` holds n_devices >= 1 CUDA ordinals; one host thread runs the share of
 * each entry.  An ordinal may repeat: its shares then run on the same device from separate host threads (how one GPU
 * runs this path).
 *   - Results: every job's result (positions, MAE, k, iterations, iterations_run, pair_updates, hold-out sums,
 *     trace, status, message) is bit for bit what topolow_fit_batch_interruptible(..., devices[0], ...) returns for
 *     the same arrays, whatever the list.  The one-CTA rule above (16 or more coloured jobs) is taken on the jobs of the
 *     whole call, never on one share.  params[j].device is ignored.  Row-block jobs are dealt like the others; a share
 *     runs its own one at a time, and a single-rank row-block fit waits on no peer, so the shares of one device (an
 *     ordinal that repeats) run their row-block fits side by side.
 *   - Arguments: a null `devices`, n_devices < 1 or an ordinal outside [0, cudaGetDeviceCount()) returns
 *     TOPOLOW_ERR_BAD_ARG before anything is allocated, with the reason in results[0].message when n_jobs > 0
 *     (TOPOLOW_ERR_CUDA when the device count cannot be read).  n_devices == 1 is
 *     topolow_fit_batch_interruptible on devices[0].
 *   - Placement: jobs are dealt longest first by n(n-1)/2 x n_iter to the entry with the least work so far; ties go
 *     to the lower job index, then to the lower list position.  The placement is a pure function of the inputs.
 *     Jobs that share edge arrays share one set of device records per device.
 *   - Interrupt: `poll` is called from the calling thread only (never from a worker thread): once before set-up,
 *     once after the set-up of every share and before the first launch on any device, then at least every 100 ms
 *     while any fit on any device runs.  When it fires, the abort word of every share is raised, no device issues
 *     another launch, and every result is filled in by the rules of topolow_fit_batch_interruptible.
 *   - Errors: a CUDA error in one share marks that share's jobs TOPOLOW_ERR_CUDA and the call returns
 *     TOPOLOW_ERR_CUDA (also when the batch was interrupted); jobs of the other shares keep their full results.
 *     Everything allocated on every device, and every mapped host block, is released before the call returns. */
TOPOLOW_API int topolow_fit_batch_devices(int32_t n_jobs, const topolow_problem* problems, const topolow_params* params,
                                          topolow_result* results, const int32_t* devices, int32_t n_devices,
                                          topolow_interrupt_fn poll, void* user);

/* ---- device-resident plan ----------------------------------------------- */
typedef struct topolow_plan topolow_plan;

TOPOLOW_API int topolow_plan_create(const topolow_problem* problem, const topolow_params* params,
                        topolow_plan** plan_out, char* message, int32_t message_len);
/* Run up to n_iters further iterations (stops early on convergence).  `stream`
 * is a cudaStream_t (NULL = the plan's own).  ms_out = CUDA-event time on that stream. */
TOPOLOW_API int topolow_plan_run(topolow_plan* plan, int32_t n_iters, void* stream, double* ms_out);
TOPOLOW_API int topolow_plan_result(topolow_plan* plan, topolow_result* result);
/* Geometry of the schedule: fills up to `cap` int64 values
 * {tiles, super_blocks, warps_per_cta, ctas, tasks_per_cta, rounds, pairs_per_iter, smem_bytes,
 * iterations_per_launch, kernel_launches_so_far, tile_points, iterations_done, stopped} (the last two as of
 * the last FINISHED launch: synchronise the stream first). */
TOPOLOW_API int topolow_plan_info(const topolow_plan* plan, int64_t* out, int32_t cap);
TOPOLOW_API void topolow_plan_destroy(topolow_plan* plan);

/* ---- one large map across several GPUs (every rank holds a plan of the SAME problem and seed) ----
 * An iteration is a tournament over 2R mega-blocks of tiles (R = n_shards): in each of the 2R-1
 * rounds rank r runs ONE bipartite job (kind 1: every pair between tile ranges [t0,t0+tc) and
 * [y0,y0+yc)), in the last round the kind-0 jobs (every pair inside a range) of its two mega-blocks;
 * between rounds the caller all-gathers the position array (topolow_plan_positions: [slots][ndim],
 * element size and slot count from topolow_plan_layout) so that every replica is current; then every
 * rank calls topolow_plan_end_iteration (cooling, edge MAE, controller) on its identical replica.
 * topolow_b200/sharded.py drives this with torch.distributed (NCCL). */
TOPOLOW_API int topolow_plan_run_job(topolow_plan* plan, int32_t kind, int32_t t0, int32_t tc, int32_t y0, int32_t yc,
                                     void* stream);
TOPOLOW_API int topolow_plan_end_iteration(topolow_plan* plan, void* stream);
/* out (up to 6 values): {total_tiles, tile_points, ndim, element_bytes, n_shards, total_slots}. */
TOPOLOW_API int topolow_plan_layout(const topolow_plan* plan, int64_t* out, int32_t cap);
TOPOLOW_API void* topolow_plan_positions(topolow_plan* plan);
/* The sequential pair order one job is equivalent to (cf. topolow_plan_enumerate). */
TOPOLOW_API int64_t topolow_plan_enumerate_job(const topolow_plan* plan, int32_t iter, int32_t kind, int32_t t0,
                                               int32_t tc, int32_t y0, int32_t yc, int32_t* out, int64_t cap_pairs);

/* ---- one large map, row-block sharded (mode TOPOLOW_MODE_ROWBLOCK; SURVEY section 8e) ----------------
 * Rank r of n_ranks (one process per GPU, or several shards in one process) owns a contiguous block of
 * rows and a replica of all positions.  Per iteration it computes the one-sided updates of its rows
 * (src/optimization.cpp:199-282 seen from the row's endpoint), stores the new rows straight into every
 * replica over NVLink and raises one flag per peer; nothing goes through the host.  Protocol:
 *   every rank: topolow_shard_create(same problem, same params, rank, n_ranks)  -> topolow_shard_export(handle)
 *   all-gather the handles (topolow_shard_handle_bytes() each; any transport: torch.distributed, MPI, a file)
 *   every rank: topolow_shard_attach(all handles in rank order)     [CUDA IPC; or topolow_shard_attach_local
 *                                                                    for shards that live in one process]
 *   every rank: topolow_shard_run(n_iters) with the same n_iters, as often as wanted; topolow_shard_result
 *   on any rank returns the whole map (replicas are identical).  Synchronise the ranks (a host barrier)
 *   before topolow_shard_destroy: peers store into a shard's memory until their last iteration ends.
 * The result does not depend on n_ranks (fixed summation trees), n_ranks = 1 is topolow_fit with
 * mode = TOPOLOW_MODE_ROWBLOCK.  A peer that does not arrive within 20 s ends the fit with TOPOLOW_ERR_CUDA. */
typedef struct topolow_shard topolow_shard;
TOPOLOW_API int topolow_shard_create(const topolow_problem* problem, const topolow_params* params, int32_t rank,
                                     int32_t n_ranks, topolow_shard** shard_out, char* message, int32_t message_len);
TOPOLOW_API int64_t topolow_shard_handle_bytes(void);
TOPOLOW_API int topolow_shard_export(topolow_shard* shard, void* handle_out);
TOPOLOW_API int topolow_shard_attach(topolow_shard* shard, const void* handles, int32_t n_handles, char* message,
                                     int32_t message_len);
TOPOLOW_API int topolow_shard_attach_local(topolow_shard* const* shards, int32_t n, char* message, int32_t message_len);
/* Up to n_iters further iterations on `stream` (cudaStream_t, NULL = the shard's own); ms_out = CUDA-event time. */
TOPOLOW_API int topolow_shard_run(topolow_shard* shard, int32_t n_iters, void* stream, double* ms_out);
/* All shards of a map that live in this process.  Shards on one device run in lock step on one stream
 * (how a single GPU checks the multi-GPU path: every wait finds its flag already raised), shards on
 * distinct devices run concurrently. */
TOPOLOW_API int topolow_shard_run_local(topolow_shard* const* shards, int32_t n, int32_t n_iters, double* ms_out);
/* Runs n_iters iterations with every kernel in order on one stream and CUDA events around every launch (the
 * production path overlaps the spring walk with the repulsion pass); out (up to 7 values) = average milliseconds
 * of {repulsion, springs, edge MAE, controller, snapshot}, the number of MAE launches seen, {combine}. */
TOPOLOW_API int topolow_shard_time_kernels(topolow_shard* shard, int32_t n_iters, double* out, int32_t cap);
TOPOLOW_API int topolow_shard_result(topolow_shard* shard, topolow_result* result);
/* out (up to 18 values): {slots, ndim, stride, n_ranks, rank, row0, own_rows, partner_chunks, spring_records,
 * mae_records, kernel_launches, iterations_done, stopped, peer_store_bytes_per_iteration, repulsion_items (work items
 * of one pass of repulsion_form: 256 own rows x one chunk of 2048 partners in form 5, x a group of chunks in form 11),
 * repulsion_ctas, repulsion_form (5: FP32 difference form, 11: distances and accumulation on tcgen05),
 * tensor_form_iterations (form 11 chosen by the policy runs adaptively: the device picks the form of every iteration;
 * the count is read back by topolow_shard_result, -1 before that or when the form is not adaptive)}. */
TOPOLOW_API int topolow_shard_info(const topolow_shard* shard, int64_t* out, int32_t cap);
/* slot_of_point of the row-block layout (a pure function of n). */
TOPOLOW_API int topolow_shard_slot_order(int64_t n, int32_t* slot_of_point_out);
TOPOLOW_API void topolow_shard_destroy(topolow_shard* shard);

/* The sequential pair order that is equivalent to iteration `iter` of a coloured-mode plan
 * (host-side walk of the same schedule functions the kernel executes).  out = [pairs][2]
 * original point ids; returns the number of pairs written (n(n-1)/2) or <0 on error. */
TOPOLOW_API int64_t topolow_plan_enumerate(const topolow_plan* plan, int32_t iter, int32_t* out, int64_t cap_pairs);

/* The same walk without a device or a plan: geometry and relabelling are pure functions of
 * (n, ndim, precision, sm_count, max_ctas, seed).  out may be NULL (geometry only). */
TOPOLOW_API int64_t topolow_schedule_enumerate(int64_t n, int32_t ndim, int32_t precision, int32_t sm_count,
                                   int32_t max_ctas, uint64_t seed, int32_t iter, int32_t* out,
                                   int64_t cap_pairs, int64_t* geometry_out, int32_t tile_points);

/* ---- post-processing kernels --------------------------------------------- */
/* est_distances[n x n] (column-major == row-major, symmetric) from positions[n x ndim col-major]. */
TOPOLOW_API int topolow_est_distances(const double* positions, int64_t n, int32_t ndim, double* est_distances,
                          int32_t device);
/* sum |truth - ||x_i - x_j||| and count over held-out cells (cell_i, cell_j may repeat a pair in
 * both orientations, as the flattened R matrices do). */
TOPOLOW_API int topolow_holdout_errors(const double* positions, int64_t n, int32_t ndim, int64_t n_cells,
                           const int32_t* cell_i, const int32_t* cell_j, const double* truth,
                           double* sum_abs_out, int64_t* count_out, int32_t device);

/* ---- measurement graph ------------------------------------------------------ */
/* Connected components of the graph whose edges are the non-NA off-diagonal cells (adjacency = !is.na,
 * R/diagnostics.R:444-446), i.e. what check_matrix_connectivity gets from igraph::components()$no
 * (R/utils.R:223-229) - for n_masks candidate point subsets at once: masks[m * n + v] != 0 selects point v in
 * candidate m (the attempts of subsample_dissimilarity_matrix, R/utils.R:371-440); masks == NULL means one
 * candidate with every point.  Per candidate: components among the selected points, selected points, and edges with
 * both ends selected (n_measurements of R/diagnostics.R:462).  points_out / edges_out may be NULL. */
TOPOLOW_API int topolow_components(int64_t n, int64_t n_edges, const int32_t* edge_i, const int32_t* edge_j, int32_t n_masks,
                                   const uint8_t* masks, int64_t* components_out, int64_t* points_out, int64_t* edges_out,
                                   int32_t device);

/* ---- measurement helpers --------------------------------------------------- */
/* which: 0 FFMA (FP32 flop/s), 1 packed fma.f32x2, 2 DFMA, 3 SHFL (warp-instr/s), 4 MUFU.RSQ,
 * 5 device copy (bytes/s read+write), 6/7/8 = milliseconds of a loop of 8 FFMA2 / 4 SHFL / both per trip
 * (do the FMA pipe and the shuffle unit overlap?).  value_out in the unit named. */
TOPOLOW_API int topolow_microbench(int32_t which, int32_t device, double* value_out);
TOPOLOW_API int topolow_device_info(int32_t device, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor,
                        int64_t* global_mem);
TOPOLOW_API const char* topolow_version(void);
/* sizeof(topolow_problem), sizeof(topolow_params), sizeof(topolow_result): lets a binding check its own
 * struct declarations against the library it loaded. */
TOPOLOW_API void topolow_abi_sizes(int64_t out[3]);

#ifdef __cplusplus
}
#endif
#endif /* TOPOLOW_B200_H */
