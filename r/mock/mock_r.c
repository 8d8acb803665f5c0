/* Functional MOCK of the R C API subset declared in r/mock/Rinternals.h (test infrastructure: lets r/shim.c
 * run without R).  SEXPs are malloc-backed records; Rf_error longjmps back into mock_call(), which is how a
 * test invokes a registered .Call entry point by name -- the same lookup R does through R_registerRoutines. */
#include <setjmp.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "R.h"
#include "Rinternals.h"
#include "R_ext/Rdynload.h"

struct SEXPREC {
  int type;
  R_xlen_t len;
  int nrow, ncol; /* -1: no dim attribute */
  void *data;
  SEXP names;
};

static struct SEXPREC nil_rec = {NILSXP, 0, -1, -1, NULL, NULL};
static struct SEXPREC names_sym = {NILSXP, 0, -1, -1, NULL, NULL};
SEXP R_NilValue = &nil_rec;
SEXP R_NamesSymbol = &names_sym;

static void **g_allocs = NULL;
static size_t g_nallocs = 0, g_cap = 0;
static int g_protect = 0;
static char g_err[1024];
static jmp_buf g_jmp;
static int g_jmp_active = 0;
static const R_CallMethodDef *g_methods = NULL;

static void *track(void *p) {
  if (g_nallocs == g_cap) {
    g_cap = g_cap ? 2 * g_cap : 256;
    g_allocs = (void **)realloc(g_allocs, g_cap * sizeof(void *));
  }
  g_allocs[g_nallocs++] = p;
  return p;
}

void Rf_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  if (g_jmp_active) longjmp(g_jmp, 1);
  fprintf(stderr, "mock R error outside mock_call: %s\n", g_err);
  abort();
}

static size_t elt_size(int type) {
  switch (type) {
    case REALSXP: return sizeof(double);
    case INTSXP: return sizeof(int);
    case VECSXP: case STRSXP: return sizeof(SEXP);
    case CHARSXP: return 1;
    default: Rf_error("mock: unsupported SEXP type %d", type);
  }
}

SEXP Rf_allocVector(int type, R_xlen_t n) {
  if (n < 0) Rf_error("negative length vectors are not allowed");
  SEXP s = (SEXP)track(calloc(1, sizeof(struct SEXPREC)));
  s->type = type;
  s->len = n;
  s->nrow = s->ncol = -1;
  s->data = track(calloc((size_t)n + 1, elt_size(type)));
  s->names = R_NilValue;
  if (type == VECSXP || type == STRSXP)
    for (R_xlen_t i = 0; i < n; i++) ((SEXP *)s->data)[i] = R_NilValue;
  return s;
}

SEXP Rf_allocMatrix(int type, int nr, int nc) {
  if (nr < 0 || nc < 0) Rf_error("negative extents to matrix");
  SEXP s = Rf_allocVector(type, (R_xlen_t)nr * nc);
  s->nrow = nr;
  s->ncol = nc;
  return s;
}

int LENGTH(SEXP s) { return (int)s->len; }
R_xlen_t XLENGTH(SEXP s) { return s->len; }
double *REAL(SEXP s) {
  if (s->type != REALSXP) Rf_error("REAL() can only be applied to a 'numeric', not a type-%d object", s->type);
  return (double *)s->data;
}
int *INTEGER(SEXP s) {
  if (s->type != INTSXP) Rf_error("INTEGER() can only be applied to a 'integer', not a type-%d object", s->type);
  return (int *)s->data;
}
int Rf_isNull(SEXP s) { return s == R_NilValue || s->type == NILSXP; }
int TYPEOF(SEXP s) { return s->type; }
int Rf_nrows(SEXP s) { return s->nrow >= 0 ? s->nrow : (int)s->len; }
int Rf_ncols(SEXP s) { return s->ncol >= 0 ? s->ncol : 1; }

SEXP Rf_duplicate(SEXP s) {
  if (Rf_isNull(s)) return s;
  SEXP d = Rf_allocVector(s->type, s->len);
  d->nrow = s->nrow;
  d->ncol = s->ncol;
  if (s->type == VECSXP) {
    for (R_xlen_t i = 0; i < s->len; i++) ((SEXP *)d->data)[i] = Rf_duplicate(((SEXP *)s->data)[i]);
  } else {
    memcpy(d->data, s->data, (size_t)s->len * elt_size(s->type));
  }
  d->names = s->names;
  return d;
}

SEXP Rf_coerceVector(SEXP s, int type) {
  if (s->type == type) return s;
  if (type == REALSXP && s->type == INTSXP) {
    SEXP d = Rf_allocVector(REALSXP, s->len);
    d->nrow = s->nrow;
    d->ncol = s->ncol;
    for (R_xlen_t i = 0; i < s->len; i++) ((double *)d->data)[i] = (double)((int *)s->data)[i];
    return d;
  }
  if (type == INTSXP && s->type == REALSXP) {
    SEXP d = Rf_allocVector(INTSXP, s->len);
    d->nrow = s->nrow;
    d->ncol = s->ncol;
    for (R_xlen_t i = 0; i < s->len; i++) ((int *)d->data)[i] = (int)((double *)s->data)[i];
    return d;
  }
  Rf_error("cannot coerce type %d to vector of type %d", s->type, type);
}

double Rf_asReal(SEXP s) {
  if (s->len < 1) Rf_error("mock Rf_asReal: empty argument");
  if (s->type == REALSXP) return ((double *)s->data)[0];
  if (s->type == INTSXP) return (double)((int *)s->data)[0];
  Rf_error("mock Rf_asReal: not a number");
}
int Rf_asInteger(SEXP s) {
  if (s->len < 1) Rf_error("mock Rf_asInteger: empty argument");
  if (s->type == INTSXP) return ((int *)s->data)[0];
  if (s->type == REALSXP) return (int)((double *)s->data)[0];
  Rf_error("mock Rf_asInteger: not a number");
}

SEXP Rf_mkChar(const char *c) {
  SEXP s = Rf_allocVector(CHARSXP, (R_xlen_t)strlen(c));
  memcpy(s->data, c, strlen(c));
  return s;
}
SEXP Rf_setAttrib(SEXP s, SEXP sym, SEXP val) {
  if (sym != R_NamesSymbol) Rf_error("mock Rf_setAttrib: only names are supported");
  s->names = val;
  return val;
}
SEXP VECTOR_ELT(SEXP s, R_xlen_t i) {
  if (s->type != VECSXP) Rf_error("VECTOR_ELT() can only be applied to a 'list', not a type-%d object", s->type);
  if (i < 0 || i >= s->len) Rf_error("mock VECTOR_ELT: index out of range");
  return ((SEXP *)s->data)[i];
}
SEXP SET_VECTOR_ELT(SEXP s, R_xlen_t i, SEXP v) {
  if (s->type != VECSXP) Rf_error("SET_VECTOR_ELT() can only be applied to a 'list'");
  if (i < 0 || i >= s->len) Rf_error("mock SET_VECTOR_ELT: index out of range");
  ((SEXP *)s->data)[i] = v;
  return v;
}
void SET_STRING_ELT(SEXP s, R_xlen_t i, SEXP v) {
  if (s->type != STRSXP) Rf_error("SET_STRING_ELT() can only be applied to a 'character vector'");
  if (i < 0 || i >= s->len) Rf_error("mock SET_STRING_ELT: index out of range");
  ((SEXP *)s->data)[i] = v;
}
SEXP Rf_protect(SEXP s) { g_protect++; return s; }
void Rf_unprotect(int n) {
  g_protect -= n;
  if (g_protect < 0) { fprintf(stderr, "mock R: protection stack underflow\n"); abort(); }
}
char *R_alloc(size_t n, int size) { return (char *)track(calloc(n + 1, (size_t)size)); }

int R_registerRoutines(DllInfo *dll, const void *c, const R_CallMethodDef *call, const void *f, const void *e) {
  (void)dll; (void)c; (void)f; (void)e;
  g_methods = call;
  return 1;
}
int R_useDynamicSymbols(DllInfo *dll, int v) { (void)dll; (void)v; return 0; }

/* ---- the test's side of the mock ------------------------------------------------------------------ */
SEXP mock_real_vector(const double *v, long n) {
  SEXP s = Rf_allocVector(REALSXP, n);
  if (n) memcpy(s->data, v, (size_t)n * sizeof(double));
  return s;
}
SEXP mock_int_vector(const int *v, long n) {
  SEXP s = Rf_allocVector(INTSXP, n);
  if (n) memcpy(s->data, v, (size_t)n * sizeof(int));
  return s;
}
SEXP mock_real_matrix(const double *v, int nr, int nc) {
  SEXP s = Rf_allocMatrix(REALSXP, nr, nc);
  if (nr > 0 && nc > 0) memcpy(s->data, v, (size_t)nr * nc * sizeof(double));
  return s;
}
SEXP mock_int_matrix(const int *v, int nr, int nc) {
  SEXP s = Rf_allocMatrix(INTSXP, nr, nc);
  if (nr > 0 && nc > 0) memcpy(s->data, v, (size_t)nr * nc * sizeof(int));
  return s;
}
SEXP mock_list(long n) { return Rf_allocVector(VECSXP, n); }
void mock_list_set(SEXP l, long i, SEXP v) { SET_VECTOR_ELT(l, i, v); }
SEXP mock_nil(void) { return R_NilValue; }
int mock_type(SEXP s) { return s->type; }
long mock_length(SEXP s) { return (long)s->len; }
int mock_nrow(SEXP s) { return s->nrow; }
int mock_ncol(SEXP s) { return s->ncol; }
void *mock_data(SEXP s) { return s->data; }
SEXP mock_list_get(SEXP l, long i) { return ((SEXP *)l->data)[i]; }
const char *mock_name(SEXP s, long i) {
  if (Rf_isNull(s->names) || i >= s->names->len) return "";
  return (const char *)((SEXP *)s->names->data)[i]->data;
}
const char *mock_last_error(void) { return g_err; }
int mock_protect_depth(void) { return g_protect; }
int mock_registered(const char *name) {
  for (const R_CallMethodDef *m = g_methods; m && m->name; m++)
    if (strcmp(m->name, name) == 0) return m->numArgs;
  return -1;
}
void mock_free_all(void) {
  for (size_t i = 0; i < g_nallocs; i++) free(g_allocs[i]);
  g_nallocs = 0;
  g_protect = 0;
}

/* .Call(name, args...): looks the entry point up in the table the shim registered, like R does.
 * Returns NULL (and leaves the message in mock_last_error) if the entry point raised an R error. */
SEXP mock_call(const char *name, int nargs, SEXP *a) {
  typedef SEXP (*f1)(SEXP); typedef SEXP (*f2)(SEXP, SEXP); typedef SEXP (*f3)(SEXP, SEXP, SEXP);
  typedef SEXP (*f4)(SEXP, SEXP, SEXP, SEXP); typedef SEXP (*f5)(SEXP, SEXP, SEXP, SEXP, SEXP);
  typedef SEXP (*f6)(SEXP, SEXP, SEXP, SEXP, SEXP, SEXP); typedef SEXP (*f7)(SEXP, SEXP, SEXP, SEXP, SEXP, SEXP, SEXP);
  g_err[0] = 0;
  const R_CallMethodDef *volatile m = g_methods;
  for (; m && m->name; m++)
    if (strcmp(m->name, name) == 0) break;
  if (!m || !m->name) { snprintf(g_err, sizeof(g_err), "mock .Call: \"%s\" not registered", name); return NULL; }
  if (m->numArgs != nargs) { snprintf(g_err, sizeof(g_err), "mock .Call: %s takes %d arguments, got %d", name, m->numArgs, nargs); return NULL; }
  const int depth = g_protect;
  g_jmp_active = 1;
  SEXP volatile out = NULL;
  if (setjmp(g_jmp) == 0) {
    switch (nargs) {
      case 1: out = ((f1)m->fun)(a[0]); break;
      case 2: out = ((f2)m->fun)(a[0], a[1]); break;
      case 3: out = ((f3)m->fun)(a[0], a[1], a[2]); break;
      case 4: out = ((f4)m->fun)(a[0], a[1], a[2], a[3]); break;
      case 5: out = ((f5)m->fun)(a[0], a[1], a[2], a[3], a[4]); break;
      case 6: out = ((f6)m->fun)(a[0], a[1], a[2], a[3], a[4], a[5]); break;
      case 7: out = ((f7)m->fun)(a[0], a[1], a[2], a[3], a[4], a[5], a[6]); break;
      default: snprintf(g_err, sizeof(g_err), "mock .Call: %d arguments unsupported", nargs); break;
    }
    if (out && g_protect != depth) {
      snprintf(g_err, sizeof(g_err), "%s: PROTECT/UNPROTECT imbalance (%d left on the stack)", name, g_protect - depth);
      out = NULL;
    }
  } else {
    out = NULL;      /* Rf_error: R unwinds the protection stack itself */
  }
  g_protect = depth;
  g_jmp_active = 0;
  return out;
}
