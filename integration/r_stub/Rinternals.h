/* integration/r_stub/Rinternals.h - stand-in for R's C API, written for this repo (no R exists in the build image):
 * only the ~35 names integration/r_shim.c touches, with R's documented semantics, implemented by r_stub.c.
 * It exists so that the shim is compiled and exercised (tests/test_host.py::test_r_shim_*); it is not shipped. */
#ifndef TOPOLOW_R_STUB_RINTERNALS_H
#define TOPOLOW_R_STUB_RINTERNALS_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif
typedef ptrdiff_t R_xlen_t;
typedef enum { FALSE = 0, TRUE = 1 } Rboolean;
typedef struct SEXPREC* SEXP;
enum { NILSXP = 0, SYMSXP = 1, CHARSXP = 9, LGLSXP = 10, INTSXP = 13, REALSXP = 14, STRSXP = 16, VECSXP = 19 };
extern SEXP R_NilValue;
#define NA_INTEGER (-2147483647 - 1)   /* R_NaInt */
int TYPEOF(SEXP x);
R_xlen_t XLENGTH(SEXP x);
int Rf_nrows(SEXP x);
int Rf_ncols(SEXP x);
int* INTEGER(SEXP x);
int* LOGICAL(SEXP x);
double* REAL(SEXP x);
const char* CHAR(SEXP x);
SEXP STRING_ELT(SEXP x, R_xlen_t i);
SEXP VECTOR_ELT(SEXP x, R_xlen_t i);
SEXP SET_VECTOR_ELT(SEXP x, R_xlen_t i, SEXP v);
int Rf_asInteger(SEXP x);
int Rf_asLogical(SEXP x);
double Rf_asReal(SEXP x);
SEXP Rf_coerceVector(SEXP x, unsigned type);
SEXP Rf_allocVector(unsigned type, R_xlen_t n);
SEXP Rf_allocMatrix(unsigned type, int nrow, int ncol);
SEXP Rf_mkNamed(unsigned type, const char** names);
SEXP Rf_mkString(const char* s);
SEXP Rf_ScalarLogical(int v);
SEXP Rf_ScalarInteger(int v);
SEXP Rf_ScalarReal(double v);
SEXP Rf_install(const char* name);
SEXP Rf_GetOption1(SEXP tag);
SEXP Rf_protect(SEXP x);
void Rf_unprotect(int n);
#define PROTECT(x) Rf_protect(x)
#define UNPROTECT(n) Rf_unprotect(n)
void Rf_error(const char* fmt, ...) __attribute__((noreturn));
void Rf_onintr(void);
void R_CheckUserInterrupt(void);
Rboolean R_ToplevelExec(void (*fun)(void*), void* data);
char* R_alloc(size_t n, int size);
#ifdef __cplusplus
}
#endif
#endif
