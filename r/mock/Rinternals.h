/* MOCK of Rinternals.h: the subset of the R C API that r/shim.c uses, implemented for real (malloc-backed
 * SEXPs) in r/mock/mock_r.c so that the shim can be compiled, linked against libgpb200.so and EXECUTED in an
 * image without R (tests/test_r_shim_gpu.py).  Semantics follow R's: REAL() on a non-double is an error,
 * Rf_coerceVector(INTSXP -> REALSXP) copies and keeps the dim attribute, Rf_error does not return. */
#ifndef MOCK_RINTERNALS_H
#define MOCK_RINTERNALS_H
#include <stddef.h>
typedef struct SEXPREC *SEXP;
typedef ptrdiff_t R_xlen_t;
#define NILSXP 0
#define CHARSXP 9
#define INTSXP 13
#define REALSXP 14
#define STRSXP 16
#define VECSXP 19
extern SEXP R_NamesSymbol;
extern SEXP R_NilValue;
int LENGTH(SEXP);
R_xlen_t XLENGTH(SEXP);
double *REAL(SEXP);
int *INTEGER(SEXP);
SEXP Rf_allocMatrix(int, int, int);
SEXP Rf_allocVector(int, R_xlen_t);
SEXP Rf_duplicate(SEXP);
SEXP Rf_coerceVector(SEXP, int);
int Rf_isNull(SEXP);
int TYPEOF(SEXP);
SEXP Rf_mkChar(const char *);
SEXP Rf_setAttrib(SEXP, SEXP, SEXP);
SEXP VECTOR_ELT(SEXP, R_xlen_t);
SEXP SET_VECTOR_ELT(SEXP, R_xlen_t, SEXP);
void SET_STRING_ELT(SEXP, R_xlen_t, SEXP);
double Rf_asReal(SEXP);
int Rf_asInteger(SEXP);
int Rf_nrows(SEXP);
int Rf_ncols(SEXP);
SEXP Rf_protect(SEXP);
void Rf_unprotect(int);
#define PROTECT(s) Rf_protect(s)
#define UNPROTECT(n) Rf_unprotect(n)
void Rf_error(const char *, ...) __attribute__((noreturn));
#endif
