/* integration/r_shim.c - the .Call wrappers around libtopolow_b200.so (INTEGRATION.md sections 2 and 4).
 *
 *   _topolow_optimize_layout_b200   same 16 SEXPs, same order, same named list back as
 *                                   _topolow_optimize_layout_exact_cpp (src/RcppExports.cpp:16-39,
 *                                   src/optimization.cpp:375-381)
 *   _topolow_fit_batch_b200         one call for a whole batch of independent fits (what the launchers do with
 *                                   parallel::mclapply today: R/adaptive_sampling.R:645-672, :2670-2693), every
 *                                   job with its own hold-out cells (R/adaptive_sampling.R:2639-2647); Ctrl-C stops it
 *
 * No R exists in the build image.  The file is compiled and RUN there against the stand-in headers of
 * integration/r_stub/ (tests/test_host.py::test_r_shim_*: marshalling, error, interrupt and registration paths
 * against a recording fake of the library on CPU; against the real library in the GPU tests).  With R:
 *   R CMD SHLIB r_shim.c -I<repo>/include -L<repo>/topolow_b200/lib -ltopolow_b200
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>
#include <stdint.h>
#include <string.h>
#include "topolow_b200.h"

/* Rcpp::checkUserInterrupt() (src/optimization.cpp:364) without a longjmp through the library: the check runs
 * inside R_ToplevelExec, which returns FALSE when R_CheckUserInterrupt jumped; the callback then only REPORTS the
 * interrupt, the library unwinds normally (streams, device buffers and events are released), returns
 * TOPOLOW_ERR_INTERRUPTED, and the R condition is raised afterwards from the shim's own frame. */
static void check_interrupt(void* unused) { (void)unused; R_CheckUserInterrupt(); }
static int poll_interrupt(void* unused) { (void)unused; return R_ToplevelExec(check_interrupt, NULL) == FALSE; }

/* The schedule seed comes from R's RNG, so set.seed() fixes a run (the reference's std::random_device,
 * src/optimization.cpp:153, does not).  unif_rand() is only valid between GetRNGstate() and PutRNGstate(). */
static uint64_t seed_from_r(void) {
  GetRNGstate();
  const double hi = unif_rand(), lo = unif_rand();
  PutRNGstate();
  return ((uint64_t)(hi * 4294967296.0) << 32) | (uint64_t)(lo * 4294967296.0);
}

static int backend_mode(void) {          /* options(topolow.b200.mode = "coloured" | "rowblock" | "replay") */
  SEXP opt = Rf_GetOption1(Rf_install("topolow.b200.mode"));
  if (TYPEOF(opt) != STRSXP || XLENGTH(opt) < 1) return TOPOLOW_MODE_COLOURED;
  const char* s = CHAR(STRING_ELT(opt, 0));
  if (strcmp(s, "rowblock") == 0) return TOPOLOW_MODE_ROWBLOCK;
  if (strcmp(s, "replay") == 0) return TOPOLOW_MODE_REPLAY;
  return TOPOLOW_MODE_COLOURED;
}

static void fill_params(topolow_params* pr, int n_iter, double k0, double cooling, double c_rep, double rel_eps,
                        int window, int freq, int verbose) {
  memset(pr, 0, sizeof *pr);
  pr->n_iter = n_iter; pr->k0 = k0; pr->cooling_rate = cooling; pr->c_repulsion = c_rep;
  pr->relative_epsilon = rel_eps; pr->convergence_window = window; pr->convergence_check_freq = freq;
  pr->verbose = verbose;
}

SEXP _topolow_optimize_layout_b200(SEXP init, SEXP dmat, SEXP tmat, SEXP degrees, SEXP edge_i, SEXP edge_j,
                                   SEXP edge_dist, SEXP edge_thresh, SEXP n_iter, SEXP k0, SEXP cooling,
                                   SEXP c_rep, SEXP rel_eps, SEXP window, SEXP freq, SEXP verbose) {
  (void)dmat; (void)tmat;   /* the dense matrices repeat the edge list (R/core.R:383-402 vs :429-436) */
  const int n = Rf_nrows(init), d = Rf_ncols(init);
  if (XLENGTH(edge_j) != XLENGTH(edge_i) || XLENGTH(edge_dist) != XLENGTH(edge_i) || XLENGTH(edge_thresh) != XLENGTH(edge_i))
    Rf_error("edge_i, edge_j, edge_dist and edge_thresh must have the same length");
  if (XLENGTH(degrees) != n) Rf_error("degrees must have one entry per point");
  topolow_problem pb;
  memset(&pb, 0, sizeof pb);
  pb.n = n; pb.ndim = d; pb.n_edges = XLENGTH(edge_i);
  pb.edge_i = INTEGER(edge_i); pb.edge_j = INTEGER(edge_j); pb.edge_dist = REAL(edge_dist);
  pb.edge_thresh = INTEGER(edge_thresh); pb.degrees = INTEGER(degrees); pb.initial_positions = REAL(init);   /* read only */
  topolow_params pr;
  fill_params(&pr, Rf_asInteger(n_iter), Rf_asReal(k0), Rf_asReal(cooling), Rf_asReal(c_rep), Rf_asReal(rel_eps),
              Rf_asInteger(window), Rf_asInteger(freq), Rf_asLogical(verbose) == TRUE);
  pr.mode = backend_mode();
  pr.seed = seed_from_r();
  SEXP pos = PROTECT(Rf_allocMatrix(REALSXP, n, d));
  topolow_result rs;
  memset(&rs, 0, sizeof rs);
  rs.positions = REAL(pos);
  const int rc = topolow_fit_interruptible(&pb, &pr, &rs, poll_interrupt, NULL);
  if (rc == TOPOLOW_ERR_INTERRUPTED) { UNPROTECT(1); Rf_onintr(); Rf_error("interrupted"); }   /* the library has unwound */
  if (rc != TOPOLOW_OK) { UNPROTECT(1); Rf_error("%s", rs.message); }   /* the two Rcpp::stop strings, :131 / :360 */
  const char* names[] = {"positions", "converged", "iterations", "final_mae", "final_k", ""};
  SEXP out = PROTECT(Rf_mkNamed(VECSXP, names));                 /* src/optimization.cpp:375-381 */
  SET_VECTOR_ELT(out, 0, pos);
  SET_VECTOR_ELT(out, 1, Rf_ScalarLogical(rs.converged));
  SET_VECTOR_ELT(out, 2, Rf_ScalarInteger(rs.iterations));
  SET_VECTOR_ELT(out, 3, Rf_ScalarReal(rs.final_mae));
  SET_VECTOR_ELT(out, 4, Rf_ScalarReal(rs.final_k));
  UNPROTECT(2);
  return out;
}

/* The optional 11th element of a batch job: "coloured" or "rowblock" (a character scalar). */
static int job_mode(SEXP job, int number) {
  if (XLENGTH(job) < 11) return TOPOLOW_MODE_COLOURED;
  SEXP m = VECTOR_ELT(job, 10);
  if (TYPEOF(m) == STRSXP && XLENGTH(m) == 1) {   /* (NA_character_ is the string "NA" here: refused below) */
    const char* s = CHAR(STRING_ELT(m, 0));
    if (strcmp(s, "coloured") == 0) return TOPOLOW_MODE_COLOURED;
    if (strcmp(s, "rowblock") == 0) return TOPOLOW_MODE_ROWBLOCK;
  }
  Rf_error("job %d: element 11 (mode) must be 'coloured' or 'rowblock'", number);
}

/* One batch of independent fits.  `jobs` is a list; job j is a named-by-position list of
 *   [[1]] initial_positions (n x ndim double)   [[2]] degrees (int)   [[3]] edge_i  [[4]] edge_j (int, 0-based)
 *   [[5]] edge_dist (double)  [[6]] edge_thresh (int)   [[7]] holdout_i  [[8]] holdout_j (int, 0-based; may be
 *   length 0)  [[9]] holdout_truth (double)   [[10]] c(mapping_max_iter, k0, cooling_rate, c_repulsion,
 *   relative_epsilon, convergence_counter, convergence_check_freq) (double)   [[11]] optional: the mode, "coloured"
 *   (the default when the job has 10 elements) or "rowblock" (large maps, ndim up to 32; the fit is exactly the
 *   single row-block fit); anything else is an R error raised before the library is called
 * Jobs that carry the SAME R vectors for [[3]]..[[6]] (the parameter samples evaluated on one fold) share one set
 * of device records - R lists hold references, so `job$edge_i <- fold$edge_i` is enough.  Returns a list of
 * per-job lists {converged, iterations, final_mae, final_k, holdout_sum_abs, holdout_count, status, message,
 * positions (only when keep_positions; a 0 x 0 matrix otherwise)}: a failed fit is a status + message, never an R error
 * (R/adaptive_sampling.R:2657-2666 turns failures into NA rows).  Ctrl-C stops the batch as it stops a single fit: the
 * library is polled while the fits run, stops them, releases what it holds and returns TOPOLOW_ERR_INTERRUPTED, and
 * the R condition is raised from this frame.
 * keep_positions = FALSE is the call for a CV grid: only the hold-out sums are needed, and they are the same as with
 * TRUE; no positions cross back (a 100 000-point map would be 12.8 MB per fold fit).
 * `device` is one CUDA ordinal, or an integer or double vector of them (e.g. 0:7): the batch is then dealt over those
 * GPUs from this one process (topolow_fit_batch_devices), with the same results as on the first of them. */
SEXP _topolow_fit_batch_b200(SEXP jobs, SEXP keep_positions, SEXP device) {
  if (TYPEOF(jobs) != VECSXP) Rf_error("jobs must be a list");
  const R_xlen_t nj = XLENGTH(jobs);
  const int keep = Rf_asLogical(keep_positions) == TRUE;
  const R_xlen_t n_dev = XLENGTH(device);
  if (n_dev < 1) Rf_error("device must name at least one CUDA ordinal");
  if (n_dev > 1024) Rf_error("device: too many ordinals");   /* (the count crosses the C ABI as int32) */
  SEXP dev_int = PROTECT(Rf_coerceVector(device, INTSXP));   /* (device itself when it is already integer) */
  for (R_xlen_t i = 0; i < n_dev; ++i)
    if (INTEGER(dev_int)[i] == NA_INTEGER) { UNPROTECT(1); Rf_error("device must not be NA"); }
  const int dev = INTEGER(dev_int)[0];
  topolow_problem* pb = (topolow_problem*)R_alloc((size_t)(nj > 0 ? nj : 1), sizeof(topolow_problem));   /* freed by R at .Call exit */
  topolow_params* pr = (topolow_params*)R_alloc((size_t)(nj > 0 ? nj : 1), sizeof(topolow_params));
  topolow_result* rs = (topolow_result*)R_alloc((size_t)(nj > 0 ? nj : 1), sizeof(topolow_result));
  SEXP out = PROTECT(Rf_allocVector(VECSXP, nj));
  const uint64_t seed = seed_from_r();
  const char* names[] = {"converged", "iterations", "final_mae", "final_k", "holdout_sum_abs", "holdout_count", "status",
                         "message", "positions", ""};
  for (R_xlen_t j = 0; j < nj; ++j) {
    SEXP job = VECTOR_ELT(jobs, j);
    if (TYPEOF(job) != VECSXP || XLENGTH(job) < 10) Rf_error("job %d: expected a list of 10 elements", (int)j + 1);
    const int mode = job_mode(job, (int)j + 1);
    SEXP init = VECTOR_ELT(job, 0), hp = VECTOR_ELT(job, 9);
    if (TYPEOF(init) != REALSXP || TYPEOF(hp) != REALSXP || XLENGTH(hp) < 7) Rf_error("job %d: malformed", (int)j + 1);
    const R_xlen_t E = XLENGTH(VECTOR_ELT(job, 2)), Hn = XLENGTH(VECTOR_ELT(job, 6));
    if (XLENGTH(VECTOR_ELT(job, 3)) != E || XLENGTH(VECTOR_ELT(job, 4)) != E || XLENGTH(VECTOR_ELT(job, 5)) != E ||
        XLENGTH(VECTOR_ELT(job, 7)) != Hn || XLENGTH(VECTOR_ELT(job, 8)) != Hn || XLENGTH(VECTOR_ELT(job, 1)) != Rf_nrows(init))
      Rf_error("job %d: array lengths disagree", (int)j + 1);
    memset(&pb[j], 0, sizeof pb[j]);
    pb[j].n = Rf_nrows(init); pb[j].ndim = Rf_ncols(init); pb[j].n_edges = E;
    pb[j].initial_positions = REAL(init); pb[j].degrees = INTEGER(VECTOR_ELT(job, 1));
    pb[j].edge_i = INTEGER(VECTOR_ELT(job, 2)); pb[j].edge_j = INTEGER(VECTOR_ELT(job, 3));
    pb[j].edge_dist = REAL(VECTOR_ELT(job, 4)); pb[j].edge_thresh = INTEGER(VECTOR_ELT(job, 5));
    pb[j].n_holdout = Hn;
    if (Hn > 0) {
      pb[j].holdout_i = INTEGER(VECTOR_ELT(job, 6)); pb[j].holdout_j = INTEGER(VECTOR_ELT(job, 7));
      pb[j].holdout_truth = REAL(VECTOR_ELT(job, 8));
    }
    const double* h = REAL(hp);
    fill_params(&pr[j], (int)h[0], h[1], h[2], h[3], h[4], (int)h[5], (int)h[6], 0);
    pr[j].mode = mode;
    pr[j].seed = seed + (uint64_t)j;
    memset(&rs[j], 0, sizeof rs[j]);
    SEXP res = PROTECT(Rf_mkNamed(VECSXP, names));
    SET_VECTOR_ELT(out, j, res);
    UNPROTECT(1);                                   /* reachable from `out` now */
    SEXP pos = Rf_allocMatrix(REALSXP, keep ? (int)pb[j].n : 0, keep ? pb[j].ndim : 0);
    SET_VECTOR_ELT(res, 8, pos);
    rs[j].positions = keep ? REAL(pos) : NULL;
  }
  const int rc = n_dev == 1 ? topolow_fit_batch_interruptible((int32_t)nj, pb, pr, rs, dev, poll_interrupt, NULL)
                            : topolow_fit_batch_devices((int32_t)nj, pb, pr, rs, INTEGER(dev_int), (int32_t)n_dev,
                                                        poll_interrupt, NULL);
  if (rc == TOPOLOW_ERR_INTERRUPTED) { UNPROTECT(2); Rf_onintr(); Rf_error("interrupted"); }   /* the library has unwound */
  if (rc != TOPOLOW_OK) { UNPROTECT(2); Rf_error("topolow_fit_batch failed with status %d%s%s", rc, nj > 0 ? ": " : "", nj > 0 ? rs[0].message : ""); }
  for (R_xlen_t j = 0; j < nj; ++j) {
    SEXP res = VECTOR_ELT(out, j);
    SET_VECTOR_ELT(res, 0, Rf_ScalarLogical(rs[j].converged));
    SET_VECTOR_ELT(res, 1, Rf_ScalarInteger(rs[j].iterations));
    SET_VECTOR_ELT(res, 2, Rf_ScalarReal(rs[j].final_mae));
    SET_VECTOR_ELT(res, 3, Rf_ScalarReal(rs[j].final_k));
    SET_VECTOR_ELT(res, 4, Rf_ScalarReal(rs[j].holdout_sum_abs));
    SET_VECTOR_ELT(res, 5, Rf_ScalarReal((double)rs[j].holdout_count));
    SET_VECTOR_ELT(res, 6, Rf_ScalarInteger(rs[j].status));
    SET_VECTOR_ELT(res, 7, Rf_mkString(rs[j].message));
  }
  UNPROTECT(2);
  return out;
}

static const R_CallMethodDef CallEntries[] = {
  {"_topolow_optimize_layout_b200", (DL_FUNC)&_topolow_optimize_layout_b200, 16},
  {"_topolow_fit_batch_b200", (DL_FUNC)&_topolow_fit_batch_b200, 3},
  {NULL, NULL, 0}};
void R_init_topolowb200(DllInfo* dll) {
  R_registerRoutines(dll, NULL, CallEntries, NULL, NULL);
  R_useDynamicSymbols(dll, FALSE);
}
