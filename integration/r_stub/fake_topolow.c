/* integration/r_stub/fake_topolow.c - a recording fake of the library entries the shim calls, for the CPU-only
 * marshalling test (no GPU, no fit): it checks what arrives and answers with values that are functions of the
 * inputs, so that the harness can tell whether every field crossed the boundary in the right place. */
#include <stdio.h>
#include <string.h>
#include "topolow_b200.h"

static void answer(const topolow_problem* pb, const topolow_params* pr, topolow_result* rs) {
  memset(rs->message, 0, sizeof rs->message);
  if (pb->n < 2) {
    rs->status = TOPOLOW_ERR_TOO_FEW_POINTS;
    snprintf(rs->message, sizeof rs->message, "Need at least 2 points for embedding");
    return;
  }
  double s = 0.0;
  for (int64_t e = 0; e < pb->n_edges; ++e) s += pb->edge_dist[e] * (double)(1 + pb->edge_thresh[e]) + pb->edge_i[e] - pb->edge_j[e];
  if (rs->positions)
    for (int64_t x = 0; x < pb->n * pb->ndim; ++x) rs->positions[x] = 2.0 * pb->initial_positions[x] + (double)pb->degrees[x % pb->n];
  rs->converged = pr->convergence_window == 5;
  rs->iterations = pr->n_iter - pr->convergence_check_freq;
  rs->final_mae = s;
  rs->final_k = pr->k0 * (1.0 - pr->cooling_rate) + pr->c_repulsion + pr->relative_epsilon;
  rs->holdout_count = pb->n_holdout;
  rs->holdout_sum_abs = 0.0;
  for (int64_t h = 0; h < pb->n_holdout; ++h) rs->holdout_sum_abs += pb->holdout_truth[h] + pb->holdout_i[h] + 2 * pb->holdout_j[h];
  rs->status = TOPOLOW_OK;
  snprintf(rs->message, sizeof rs->message, "mode=%d seed=%llu verbose=%d", pr->mode, (unsigned long long)pr->seed, pr->verbose);
}

int topolow_fit_interruptible(const topolow_problem* pb, const topolow_params* pr, topolow_result* rs,
                              topolow_interrupt_fn poll, void* user) {
  for (int chunk = 0; chunk < 4; ++chunk)          /* the library polls between device chunks */
    if (poll && poll(user)) {
      rs->status = TOPOLOW_ERR_INTERRUPTED;
      snprintf(rs->message, sizeof rs->message, "interrupted");
      return rs->status;                           /* a normal return: everything the library holds is released */
    }
  answer(pb, pr, rs);
  return rs->status;
}

int topolow_fit_batch(int32_t n_jobs, const topolow_problem* pb, const topolow_params* pr, topolow_result* rs, int32_t device) {
  if (device < 0) return TOPOLOW_ERR_CUDA;
  int shared = 0;
  for (int32_t j = 0; j < n_jobs; ++j) {
    answer(&pb[j], &pr[j], &rs[j]);
    if (j > 0 && pb[j].edge_i == pb[0].edge_i && pb[j].edge_dist == pb[0].edge_dist) ++shared;
  }
  if (n_jobs > 0 && rs[0].status == TOPOLOW_OK) {
    const size_t at = strlen(rs[0].message);
    snprintf(rs[0].message + at, sizeof rs[0].message - at, " shared=%d", shared);
  }
  return TOPOLOW_OK;
}

/* Polls once before each job; without an interrupt it answers what topolow_fit_batch answers. */
int topolow_fit_batch_interruptible(int32_t n_jobs, const topolow_problem* pb, const topolow_params* pr, topolow_result* rs,
                                    int32_t device, topolow_interrupt_fn poll, void* user) {
  if (device < 0) return TOPOLOW_ERR_CUDA;
  for (int32_t j = 0; j < n_jobs; ++j)
    if (poll && poll(user)) {
      for (int32_t k = j; k < n_jobs; ++k) {
        rs[k].status = TOPOLOW_ERR_INTERRUPTED;
        snprintf(rs[k].message, sizeof rs[k].message, "interrupted");
      }
      return TOPOLOW_ERR_INTERRUPTED;
    }
  return topolow_fit_batch(n_jobs, pb, pr, rs, device);
}

/* Records the device list it was handed at the end of the first job's message (" devices=0,0"); polls and answers
 * as topolow_fit_batch_interruptible does. */
int topolow_fit_batch_devices(int32_t n_jobs, const topolow_problem* pb, const topolow_params* pr, topolow_result* rs,
                              const int32_t* devices, int32_t n_devices, topolow_interrupt_fn poll, void* user) {
  if (!devices || n_devices < 1) return TOPOLOW_ERR_BAD_ARG;
  for (int32_t i = 0; i < n_devices; ++i)
    if (devices[i] < 0) return TOPOLOW_ERR_BAD_ARG;
  const int rc = topolow_fit_batch_interruptible(n_jobs, pb, pr, rs, devices[0], poll, user);
  if (rc == TOPOLOW_OK && n_jobs > 0) {
    size_t at = strlen(rs[0].message);
    at += (size_t)snprintf(rs[0].message + at, sizeof rs[0].message - at, " devices=");
    for (int32_t i = 0; i < n_devices && at < sizeof rs[0].message; ++i)
      at += (size_t)snprintf(rs[0].message + at, sizeof rs[0].message - at, "%s%d", i ? "," : "", devices[i]);
  }
  return rc;
}
