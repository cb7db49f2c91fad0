/* integration/r_stub/harness.c - drives integration/r_shim.c the way R would: builds the SEXPs, makes the .Call,
 * prints what came back as one JSON object per line.  Linked with fake_topolow.c on a CPU-only box (marshalling,
 * errors, interrupt, registration) and with libtopolow_b200.so on the GPU box (a real fit through the shim).
 *
 *   harness register
 *   harness too_few
 *   harness single    problem.bin out.bin n_iter k0 cooling c_rep rel_eps window freq [mode]
 *   harness interrupt problem.bin at_check
 *   harness batch     problem.bin out.bin n_jobs n_iter k0 cooling c_rep rel_eps window freq keep
 *   harness batch_interrupt problem.bin out.bin n_jobs n_iter k0 cooling c_rep rel_eps window freq keep at_check
 *                     (the batch call with R_CheckUserInterrupt firing at its at_check-th call; 0 = never)
 *   harness batch_devices problem.bin out.bin n_jobs n_iter k0 cooling c_rep rel_eps window freq keep int|double d...
 *                     (the batch call with `device` an integer or double vector of the ordinals d...; NA = NA, none =
 *                     a vector of length 0)
 *   harness batch_modes problem.bin out.bin n_jobs n_iter k0 cooling c_rep rel_eps window freq keep m...
 *                     (the batch call with one mode token per job: "-" = a job of 10 elements, "@int" / "@real" = an
 *                     11th element of that type, anything else = that string as the 11th element)
 *
 * problem.bin: int64 n, d, E, H | init[n*d] f64 (column-major) | degrees[n] i32 | edge_i[E] edge_j[E] i32 | edge_dist[E]
 * f64 | edge_thresh[E] i32 | holdout_i[H] holdout_j[H] i32 | holdout_truth[H] f64.  out.bin: the doubles named in the
 * JSON line, in order.  Test infrastructure only. */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "r_stub.h"

SEXP _topolow_optimize_layout_b200(SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP);
SEXP _topolow_fit_batch_b200(SEXP, SEXP, SEXP);
void R_init_topolowb200(DllInfo*);

struct problem { long long n, d, E, H; SEXP init, deg, ei, ej, ed, et, hi, hj, ht; };

static void* slurp(FILE* f, size_t bytes) {
  void* p = malloc(bytes ? bytes : 1);
  if (bytes && fread(p, 1, bytes, f) != bytes) { fprintf(stderr, "short problem file\n"); exit(2); }
  return p;
}
static struct problem load(const char* path) {
  struct problem p;
  FILE* f = fopen(path, "rb");
  if (!f) { perror(path); exit(2); }
  int64_t hdr[4];
  if (fread(hdr, 8, 4, f) != 4) exit(2);
  p.n = hdr[0]; p.d = hdr[1]; p.E = hdr[2]; p.H = hdr[3];
  p.init = stub_matrix((int)p.n, (int)p.d, slurp(f, (size_t)(p.n * p.d) * 8));
  p.deg = stub_int(p.n, slurp(f, (size_t)p.n * 4));
  p.ei = stub_int(p.E, slurp(f, (size_t)p.E * 4));
  p.ej = stub_int(p.E, slurp(f, (size_t)p.E * 4));
  p.ed = stub_real(p.E, slurp(f, (size_t)p.E * 8));
  p.et = stub_int(p.E, slurp(f, (size_t)p.E * 4));
  p.hi = stub_int(p.H, slurp(f, (size_t)p.H * 4));
  p.hj = stub_int(p.H, slurp(f, (size_t)p.H * 4));
  p.ht = stub_real(p.H, slurp(f, (size_t)p.H * 8));
  fclose(f);
  return p;
}
static void health(void) {
  printf("\"protect_depth\": %d, \"type_errors\": %d, \"rng_violations\": %d, \"rng_open\": %d, \"raw_interrupt_jumps\": %d, "
         "\"interrupt_checks\": %d, \"onintr_calls\": %d, \"errors\": %d",
         stub.protect_depth, stub.type_errors, stub.rng_violations, stub.rng_open, stub.raw_interrupt_jumps,
         stub.interrupt_checks, stub.onintr_calls, stub.errors);
}
static SEXP call_single(struct problem* p, char** a) {   /* a: n_iter k0 cooling c_rep rel_eps window freq */
  int n_iter = atoi(a[0]), window = atoi(a[5]), freq = atoi(a[6]), verbose = 0;
  double k0 = atof(a[1]), cooling = atof(a[2]), c_rep = atof(a[3]), eps = atof(a[4]);
  SEXP v = Rf_ScalarLogical(verbose);
  return _topolow_optimize_layout_b200(p->init, R_NilValue, R_NilValue, p->deg, p->ei, p->ej, p->ed, p->et, stub_int(1, &n_iter),
                                       stub_real(1, &k0), stub_real(1, &cooling), stub_real(1, &c_rep), stub_real(1, &eps),
                                       stub_int(1, &window), stub_int(1, &freq), v);
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  memset(&stub, 0, sizeof stub);
  const char* what = argv[1];
  const int jumped = setjmp(stub.toplevel);
  if (jumped) {     /* 1 Rf_error, 2 Rf_onintr, 3 an interrupt that jumped straight out of the library */
    printf("{\"scenario\": \"%s\", \"left_by\": \"%s\", \"message\": \"%s\", ", what,
           jumped == 1 ? "Rf_error" : jumped == 2 ? "Rf_onintr" : "raw longjmp", stub.error_message);
    health();
    printf("}\n");
    return 0;
  }
  if (!strcmp(what, "register")) {
    R_init_topolowb200(NULL);
    printf("{\"scenario\": \"register\", \"dynamic_symbols\": %d, \"routines\": {", stub.dynamic_symbols);
    for (int i = 0; i < stub.n_registered && i < 8; ++i) printf("%s\"%s\": %d", i ? ", " : "", stub.registered[i].name, stub.registered[i].numArgs);
    printf("}}\n");
    return 0;
  }
  if (!strcmp(what, "too_few")) {
    struct problem p;
    double z = 0.0; int one = 1;
    p.init = stub_matrix(1, 2, NULL); p.deg = stub_int(1, &one); p.ei = stub_int(0, NULL); p.ej = stub_int(0, NULL);
    p.ed = stub_real(0, &z); p.et = stub_int(0, NULL);
    char* a[] = {"10", "1", "0.01", "0.01", "1e-4", "5", "3"};
    call_single(&p, a);
    printf("{\"scenario\": \"too_few\", \"left_by\": \"return\"}\n");
    return 1;
  }
  if (!strcmp(what, "single") && argc >= 11) {
    struct problem p = load(argv[2]);
    if (argc > 11) stub.option_mode = argv[11];
    SEXP r = call_single(&p, argv + 4);
    FILE* o = fopen(argv[3], "wb");
    const double sc[4] = {(double)Rf_asLogical(VECTOR_ELT(r, 1)), (double)Rf_asInteger(VECTOR_ELT(r, 2)), Rf_asReal(VECTOR_ELT(r, 3)),
                          Rf_asReal(VECTOR_ELT(r, 4))};
    fwrite(sc, 8, 4, o);
    fwrite(REAL(VECTOR_ELT(r, 0)), 8, (size_t)(p.n * p.d), o);
    fclose(o);
    printf("{\"scenario\": \"single\", \"names\": [");
    for (int i = 0; i < (int)XLENGTH(r); ++i) printf("%s\"%s\"", i ? ", " : "", stub_name(r, i));
    printf("], \"types\": [");
    for (int i = 0; i < (int)XLENGTH(r); ++i) printf("%s%d", i ? ", " : "", TYPEOF(VECTOR_ELT(r, i)));
    printf("], \"dim\": [%d, %d], \"converged\": %g, \"iterations\": %g, \"final_mae\": %.17g, \"final_k\": %.17g, ",
           Rf_nrows(VECTOR_ELT(r, 0)), Rf_ncols(VECTOR_ELT(r, 0)), sc[0], sc[1], sc[2], sc[3]);
    health();
    printf("}\n");
    return 0;
  }
  if (!strcmp(what, "interrupt") && argc >= 4) {
    struct problem p = load(argv[2]);
    stub.interrupt_after = atoi(argv[3]);
    char* a[] = {"1000", "5", "0.01", "0.02", "1e-12", "2000", "3"};
    call_single(&p, a);
    printf("{\"scenario\": \"interrupt\", \"left_by\": \"return\", ");
    health();
    printf("}\n");
    return 0;
  }
  const int batch_interrupt = !strcmp(what, "batch_interrupt"), batch_devices = !strcmp(what, "batch_devices");
  const int batch_modes = !strcmp(what, "batch_modes");
  if ((!strcmp(what, "batch") && argc >= 13) || ((batch_interrupt || batch_devices) && argc >= 14) ||
      (batch_modes && argc >= 13 + atoi(argv[4]))) {
    struct problem p = load(argv[2]);
    if (batch_interrupt) stub.interrupt_after = atoi(argv[13]);
    SEXP device;
    if (batch_devices) {
      const int nd = argc - 14, as_double = !strcmp(argv[13], "double");
      device = as_double ? stub_real(nd, NULL) : stub_int(nd, NULL);
      for (int i = 0; i < nd; ++i) {
        const int na = !strcmp(argv[14 + i], "NA");
        if (as_double) REAL(device)[i] = na ? NAN : atof(argv[14 + i]);
        else INTEGER(device)[i] = na ? NA_INTEGER : atoi(argv[14 + i]);
      }
    } else {
      int dev = 0;
      device = stub_int(1, &dev);
    }
    const int nj = atoi(argv[4]), keep = atoi(argv[12]);
    SEXP jobs = stub_list(nj);
    for (int j = 0; j < nj; ++j) {
      const char* m = batch_modes ? argv[13 + j] : "-";
      SEXP job = stub_list(strcmp(m, "-") ? 11 : 10);
      if (strcmp(m, "-")) {
        int one = 1; double half = 0.5;
        SET_VECTOR_ELT(job, 10, !strcmp(m, "@int") ? stub_int(1, &one) : !strcmp(m, "@real") ? stub_real(1, &half) : Rf_mkString(m));
      }
      double hp[7] = {atof(argv[5]), atof(argv[6]) * (1.0 + 0.25 * j), atof(argv[7]), atof(argv[8]), atof(argv[9]), atof(argv[10]), atof(argv[11])};
      SET_VECTOR_ELT(job, 0, p.init); SET_VECTOR_ELT(job, 1, p.deg);
      SET_VECTOR_ELT(job, 2, p.ei); SET_VECTOR_ELT(job, 3, p.ej); SET_VECTOR_ELT(job, 4, p.ed); SET_VECTOR_ELT(job, 5, p.et);   /* the same vectors in every job */
      SET_VECTOR_ELT(job, 6, p.hi); SET_VECTOR_ELT(job, 7, p.hj); SET_VECTOR_ELT(job, 8, p.ht);
      SET_VECTOR_ELT(job, 9, stub_real(7, hp));
      SET_VECTOR_ELT(jobs, j, job);
    }
    SEXP r = _topolow_fit_batch_b200(jobs, Rf_ScalarLogical(keep), device);
    FILE* o = fopen(argv[3], "wb");
    printf("{\"scenario\": \"%s\", \"left_by\": \"return\", \"n\": %d, \"names\": [", what, (int)XLENGTH(r));
    for (int i = 0; nj > 0 && i < (int)XLENGTH(VECTOR_ELT(r, 0)); ++i) printf("%s\"%s\"", i ? ", " : "", stub_name(VECTOR_ELT(r, 0), i));
    printf("], \"jobs\": [");
    for (int j = 0; j < nj; ++j) {
      SEXP res = VECTOR_ELT(r, j);
      const double sc[7] = {(double)Rf_asLogical(VECTOR_ELT(res, 0)), (double)Rf_asInteger(VECTOR_ELT(res, 1)), Rf_asReal(VECTOR_ELT(res, 2)),
                            Rf_asReal(VECTOR_ELT(res, 3)), Rf_asReal(VECTOR_ELT(res, 4)), Rf_asReal(VECTOR_ELT(res, 5)),
                            (double)Rf_asInteger(VECTOR_ELT(res, 6))};
      fwrite(sc, 8, 7, o);
      if (keep) fwrite(REAL(VECTOR_ELT(res, 8)), 8, (size_t)(p.n * p.d), o);
      printf("%s{\"status\": %g, \"message\": \"%s\", \"pos_len\": %d}", j ? ", " : "", sc[6], CHAR(STRING_ELT(VECTOR_ELT(res, 7), 0)),
             (int)XLENGTH(VECTOR_ELT(res, 8)));
    }
    fclose(o);
    printf("], ");
    health();
    printf("}\n");
    return 0;
  }
  fprintf(stderr, "unknown scenario\n");
  return 2;
}
