/* integration/r_stub/r_stub.c - a few hundred lines of "R": the objects and control flow integration/r_shim.c needs,
 * with R's semantics where they matter for the shim's correctness:
 *   - Rf_error and a pending interrupt inside R_CheckUserInterrupt leave by longjmp (to the harness's top level or
 *     to the enclosing R_ToplevelExec), exactly what makes a naive interrupt callback unsafe;
 *   - unif_rand() outside GetRNGstate()/PutRNGstate() is counted as a violation;
 *   - the protect stack is counted so that the harness can check PROTECT / UNPROTECT balance;
 *   - R_registerRoutines records what was registered.
 * Test infrastructure only. */
#include <setjmp.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "R.h"
#include "Rinternals.h"
#include "R_ext/Rdynload.h"
#include "r_stub.h"

struct SEXPREC { int type; R_xlen_t len; int nrow, ncol; void* data; const char** names; };
static struct SEXPREC nil_obj = {NILSXP, 0, 0, 0, NULL, NULL};
SEXP R_NilValue = &nil_obj;

struct stub_state stub;
static jmp_buf* toplevel_exec_jmp = NULL;

static SEXP new_obj(int type, R_xlen_t n, size_t elt) {
  SEXP x = (SEXP)calloc(1, sizeof *x);
  x->type = type; x->len = n; x->nrow = (int)n; x->ncol = 1;
  x->data = calloc((size_t)(n > 0 ? n : 1), elt);
  return x;
}
int TYPEOF(SEXP x) { return x->type; }
R_xlen_t XLENGTH(SEXP x) { return x->len; }
int Rf_nrows(SEXP x) { return x->nrow; }
int Rf_ncols(SEXP x) { return x->ncol; }
int* INTEGER(SEXP x) { if (x->type != INTSXP && x->type != LGLSXP) stub.type_errors++; return (int*)x->data; }
int* LOGICAL(SEXP x) { if (x->type != LGLSXP) stub.type_errors++; return (int*)x->data; }
double* REAL(SEXP x) { if (x->type != REALSXP) stub.type_errors++; return (double*)x->data; }
const char* CHAR(SEXP x) { return (const char*)x->data; }
SEXP STRING_ELT(SEXP x, R_xlen_t i) { return ((SEXP*)x->data)[i]; }
SEXP VECTOR_ELT(SEXP x, R_xlen_t i) {
  if (x->type != VECSXP || i < 0 || i >= x->len) { stub.type_errors++; return R_NilValue; }
  return ((SEXP*)x->data)[i];
}
SEXP SET_VECTOR_ELT(SEXP x, R_xlen_t i, SEXP v) {
  if (x->type != VECSXP || i < 0 || i >= x->len) { stub.type_errors++; return v; }
  ((SEXP*)x->data)[i] = v;
  return v;
}
int Rf_asInteger(SEXP x) { return x->type == REALSXP ? (int)((double*)x->data)[0] : ((int*)x->data)[0]; }
int Rf_asLogical(SEXP x) { return x->type == REALSXP ? ((double*)x->data)[0] != 0.0 : ((int*)x->data)[0] != 0; }
double Rf_asReal(SEXP x) { return x->type == REALSXP ? ((double*)x->data)[0] : (double)((int*)x->data)[0]; }
SEXP Rf_allocVector(unsigned type, R_xlen_t n) {
  stub.allocations++;
  switch (type) {
    case REALSXP: return new_obj(REALSXP, n, sizeof(double));
    case INTSXP: case LGLSXP: return new_obj((int)type, n, sizeof(int));
    case VECSXP: case STRSXP: {
      SEXP x = new_obj((int)type, n, sizeof(SEXP));
      for (R_xlen_t i = 0; i < n; ++i) ((SEXP*)x->data)[i] = R_NilValue;
      return x;
    }
    default: stub.type_errors++; return R_NilValue;
  }
}
/* INTSXP only (what the shim asks for): x itself when it is already integer, NA for NaN or out of range doubles */
SEXP Rf_coerceVector(SEXP x, unsigned type) {
  if (type != INTSXP || (x->type != INTSXP && x->type != LGLSXP && x->type != REALSXP)) { stub.type_errors++; return R_NilValue; }
  if (x->type == INTSXP) return x;
  SEXP y = Rf_allocVector(INTSXP, x->len);
  for (R_xlen_t i = 0; i < x->len; ++i) {
    if (x->type == LGLSXP) { ((int*)y->data)[i] = ((int*)x->data)[i]; continue; }
    const double v = ((double*)x->data)[i];
    ((int*)y->data)[i] = (v != v || v >= 2147483648.0 || v <= -2147483649.0) ? NA_INTEGER : (int)v;
  }
  return y;
}
SEXP Rf_allocMatrix(unsigned type, int nrow, int ncol) {
  SEXP x = Rf_allocVector(type, (R_xlen_t)nrow * ncol);
  x->nrow = nrow; x->ncol = ncol;
  return x;
}
SEXP Rf_mkNamed(unsigned type, const char** names) {
  R_xlen_t n = 0;
  while (names[n][0]) ++n;
  SEXP x = Rf_allocVector(type, n);
  const char** copy = (const char**)calloc((size_t)n + 1, sizeof(char*));   /* R copies the names: the caller's array may be a local */
  for (R_xlen_t i = 0; i < n; ++i) copy[i] = strdup(names[i]);
  x->names = copy;
  return x;
}
static SEXP mk_char(const char* s) {
  SEXP c = new_obj(CHARSXP, (R_xlen_t)strlen(s), 1);
  free(c->data);
  c->data = strdup(s);
  return c;
}
SEXP Rf_mkString(const char* s) { SEXP x = Rf_allocVector(STRSXP, 1); ((SEXP*)x->data)[0] = mk_char(s); return x; }
SEXP Rf_ScalarLogical(int v) { SEXP x = Rf_allocVector(LGLSXP, 1); ((int*)x->data)[0] = v != 0; return x; }
SEXP Rf_ScalarInteger(int v) { SEXP x = Rf_allocVector(INTSXP, 1); ((int*)x->data)[0] = v; return x; }
SEXP Rf_ScalarReal(double v) { SEXP x = Rf_allocVector(REALSXP, 1); ((double*)x->data)[0] = v; return x; }
SEXP Rf_install(const char* name) { SEXP c = mk_char(name); c->type = SYMSXP; return c; }
SEXP Rf_GetOption1(SEXP tag) {
  if (stub.option_mode && strcmp((const char*)tag->data, "topolow.b200.mode") == 0) return Rf_mkString(stub.option_mode);
  return R_NilValue;
}
SEXP Rf_protect(SEXP x) { stub.protect_depth++; return x; }
void Rf_unprotect(int n) { stub.protect_depth -= n; if (stub.protect_depth < 0) stub.type_errors++; }
void Rf_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(stub.error_message, sizeof stub.error_message, fmt, ap);
  va_end(ap);
  stub.errors++;
  stub.protect_depth = 0;                 /* R unwinds the protect stack to the context it jumps to */
  longjmp(stub.toplevel, 1);
}
void Rf_onintr(void) { stub.onintr_calls++; stub.protect_depth = 0; longjmp(stub.toplevel, 2); }
void R_CheckUserInterrupt(void) {
  stub.interrupt_checks++;
  if (stub.interrupt_after > 0 && stub.interrupt_checks >= stub.interrupt_after) {
    stub.interrupt_after = 0;
    if (toplevel_exec_jmp) longjmp(*toplevel_exec_jmp, 1);
    stub.raw_interrupt_jumps++;           /* jumped out of whatever called us: the unsafe path */
    longjmp(stub.toplevel, 3);
  }
}
Rboolean R_ToplevelExec(void (*fun)(void*), void* data) {
  jmp_buf here;
  jmp_buf* saved = toplevel_exec_jmp;
  volatile Rboolean ok = TRUE;
  toplevel_exec_jmp = &here;
  if (setjmp(here) == 0) fun(data); else ok = FALSE;
  toplevel_exec_jmp = saved;
  return ok;
}
char* R_alloc(size_t n, int size) { return (char*)calloc(n ? n : 1, (size_t)size); }
void GetRNGstate(void) { stub.rng_open++; }
void PutRNGstate(void) { stub.rng_open--; }
double unif_rand(void) {
  if (stub.rng_open <= 0) stub.rng_violations++;
  const double v[2] = {0.25, 0.5};        /* fixed stream: the shim's seed is then (2^30 << 32) | 2^31 */
  return v[stub.rng_draws++ & 1];
}
int R_registerRoutines(DllInfo* info, const void* c, const R_CallMethodDef* call, const void* f, const void* e) {
  (void)info; (void)c; (void)f; (void)e;
  stub.n_registered = 0;
  for (; call && call->name; ++call) {
    if (stub.n_registered < 8) stub.registered[stub.n_registered] = *call;
    stub.n_registered++;
  }
  return 1;
}
Rboolean R_useDynamicSymbols(DllInfo* info, Rboolean value) { (void)info; stub.dynamic_symbols = value; return TRUE; }

/* constructors for the harness */
SEXP stub_real(R_xlen_t n, const double* v) {
  SEXP x = Rf_allocVector(REALSXP, n);
  if (v) memcpy(x->data, v, (size_t)n * sizeof(double));
  return x;
}
SEXP stub_int(R_xlen_t n, const int* v) {
  SEXP x = Rf_allocVector(INTSXP, n);
  if (v) memcpy(x->data, v, (size_t)n * sizeof(int));
  return x;
}
SEXP stub_matrix(int nrow, int ncol, const double* v) {
  SEXP x = stub_real((R_xlen_t)nrow * ncol, v);
  x->nrow = nrow; x->ncol = ncol;
  return x;
}
SEXP stub_list(R_xlen_t n) { return Rf_allocVector(VECSXP, n); }
const char* stub_name(SEXP x, R_xlen_t i) { return x->names ? x->names[i] : ""; }
