/* r/shim.c -- thin .Call shim between R and libgpb200.so.
 *
 * Build where R exists with
 *     R CMD SHLIB r/shim.c -I include -L gp_b200/lib -lgpb200 -o r/gpb200_r.so
 * (see r/build.sh).  In the build container (no R) the same file is compiled against the FUNCTIONAL
 * mock of the R C API in r/mock/ (malloc-backed SEXPs), linked against libgpb200.so and executed on
 * the GPU box by tests/test_r_shim_gpu.py -- so every line below runs, only not under a real R.
 *
 * Every entry point only converts SEXPs to plain pointers, calls the C ABI of include/gpb200.h and
 * turns a non-zero status into an R error -- the arithmetic is in the CUDA library.  It replaces the
 * wrapper Rcpp attributes generate for covariance.cpp:8-9
 * (`extern "C" SEXP sourceCpp_N_rbf_cov_chol(SEXP x1SEXP, SEXP l_SEXP)`) and gives the R kernel and
 * conditioning functions of R/kernels.R, derivative_kernels.R, R/ode_gp_library.R one call per
 * matrix instead of one closure call per element.
 *
 * Like Rcpp's NumericVector / NumericMatrix, every numeric argument is COERCED to double storage
 * (an integer matrix from R is fine) and every shape the C ABI relies on is checked here, so that a
 * wrong shape is an R error and never an out-of-bounds read.
 *
 * R is single-threaded: all entry points run on the main R thread and synchronise before returning
 * (host-pointer mode of the ABI).  Outputs are R-allocated and PROTECTed while being filled.
 */
#include <stdlib.h>
#include <string.h>

#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>

#include "gpb200.h"

static gpb200_handle_t g_h = NULL;

static gpb200_handle_t handle(void) {
  if (!g_h) {
    int dev = 0;
    const char *e = getenv("GPB200_DEVICE");
    if (e) dev = atoi(e);
    int rc = gpb200_create(&g_h, dev);
    if (rc != 0) Rf_error("gpb200: no usable B200 GPU (gpb200_create returned %d); there is no CPU fallback", rc);
  }
  return g_h;
}

static void check(int rc, const char *where) {
  if (rc < 0) Rf_error("%s failed (%d): %s", where, rc, gpb200_last_error(g_h));
  if (rc > 0) Rf_error("%s: matrix is not positive definite (first non-positive pivot at %d)", where, rc);
}

/* double-storage view of a numeric argument (what Rcpp::NumericVector(x) does); PROTECTs, counts in *np */
static SEXP as_real(SEXP x, int *np, const char *what) {
  if (Rf_isNull(x)) Rf_error("%s must not be NULL", what);
  SEXP r = PROTECT(Rf_coerceVector(x, REALSXP));
  (*np)++;
  return r;
}

static void need_matrix(SEXP m, int nrow, int ncol, const char *what) {
  if (Rf_nrows(m) != nrow || Rf_ncols(m) != ncol)
    Rf_error("%s must be a %d x %d matrix (got %d x %d)", what, nrow, ncol, Rf_nrows(m), Rf_ncols(m));
}

static SEXP named_list(int n, SEXP *elts, const char *const *names) {
  SEXP out = PROTECT(Rf_allocVector(VECSXP, n));
  SEXP nm = PROTECT(Rf_allocVector(STRSXP, n));
  for (int i = 0; i < n; i++) {
    SET_VECTOR_ELT(out, i, elts[i]);
    SET_STRING_ELT(nm, i, Rf_mkChar(names[i]));
  }
  Rf_setAttrib(out, R_NamesSymbol, nm);
  UNPROTECT(2);
  return out;
}

/* rbf_cov_chol(x1, l_) -> list(L =, dLdl =)          [covariance.cpp:8-47] */
SEXP gp_rbf_cov_chol(SEXP x1_, SEXP l_) {
  int np = 0;
  SEXP x1 = as_real(x1_, &np, "x1");
  const int n = LENGTH(x1);
  SEXP L = PROTECT(Rf_allocMatrix(REALSXP, n, n));
  SEXP dL = PROTECT(Rf_allocMatrix(REALSXP, n, n));
  np += 2;
  check(gpb200_rbf_cov_chol(handle(), n, REAL(x1), Rf_asReal(l_), REAL(L), REAL(dL)), "rbf_cov_chol");
  SEXP elts[2] = {L, dL};
  static const char *const names[2] = {"L", "dLdl"};
  SEXP out = named_list(2, elts, names);
  UNPROTECT(np);
  return out;
}

/* approx_L(l, lp, Ls, dLdls)                         [covariance.cpp:49-96] */
SEXP gp_approx_L(SEXP l, SEXP lp_, SEXP Ls, SEXP dLdls) {
  int np = 0;
  SEXP lp = as_real(lp_, &np, "lp");
  const int P = LENGTH(lp);
  if (P < 2) Rf_error("approx_L: need at least two grid points");
  if (LENGTH(Ls) != P || LENGTH(dLdls) != P) Rf_error("approx_L: lp, Ls, dLdls must have equal length");
  const int n = Rf_nrows(VECTOR_ELT(Ls, 0));
  const double **a = (const double **)R_alloc(P, sizeof(double *));
  const double **b = (const double **)R_alloc(P, sizeof(double *));
  for (int i = 0; i < P; i++) {
    SEXP ai = as_real(VECTOR_ELT(Ls, i), &np, "Ls[[i]]"), bi = as_real(VECTOR_ELT(dLdls, i), &np, "dLdls[[i]]");
    need_matrix(ai, n, n, "every element of Ls");
    need_matrix(bi, n, n, "every element of dLdls");
    a[i] = REAL(ai);
    b[i] = REAL(bi);
  }
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, n, n));
  np++;
  check(gpb200_approx_L(handle(), n, Rf_asReal(l), P, REAL(lp), a, b, REAL(out)), "approx_L");
  UNPROTECT(np);
  return out;
}

/* approx_Lz(l, lp, Ls, dLdls, z) -> list(vz =, dvdl_z =)   [models/cubic_interpolated_gp.hpp:38-73] */
SEXP gp_approx_Lz(SEXP l, SEXP lp_, SEXP Ls, SEXP dLdls, SEXP z_) {
  int np = 0;
  SEXP lp = as_real(lp_, &np, "lp"), z = as_real(z_, &np, "z");
  const int P = LENGTH(lp), n = LENGTH(z);
  if (P < 2) Rf_error("approx_Lz: need at least two grid points");
  if (LENGTH(Ls) != P || LENGTH(dLdls) != P) Rf_error("approx_Lz: lp, Ls, dLdls must have equal length");
  const double **a = (const double **)R_alloc(P, sizeof(double *));
  const double **b = (const double **)R_alloc(P, sizeof(double *));
  for (int i = 0; i < P; i++) {
    SEXP ai = as_real(VECTOR_ELT(Ls, i), &np, "Ls[[i]]"), bi = as_real(VECTOR_ELT(dLdls, i), &np, "dLdls[[i]]");
    need_matrix(ai, n, n, "every element of Ls");
    need_matrix(bi, n, n, "every element of dLdls");
    a[i] = REAL(ai);
    b[i] = REAL(bi);
  }
  SEXP vz = PROTECT(Rf_allocVector(REALSXP, n));
  SEXP dvz = PROTECT(Rf_allocVector(REALSXP, n));
  np += 2;
  check(gpb200_approx_Lz(handle(), n, Rf_asReal(l), P, REAL(lp), a, b, REAL(z), REAL(vz), REAL(dvz)), "approx_Lz");
  SEXP elts[2] = {vz, dvz};
  static const char *const names[2] = {"vz", "dvdl_z"};
  SEXP out = named_list(2, elts, names);
  UNPROTECT(np);
  return out;
}

/* all P tables of a length-scale grid in one batched call -> list(Ls = list(...), dLdls = list(...))
 * (data block of models/cubic_interpolated_gp.stan:11-12; interpolated_gp.stan:15-21) */
SEXP gp_rbf_cov_chol_grid(SEXP x1_, SEXP lp_) {
  int np = 0;
  SEXP x1 = as_real(x1_, &np, "x1"), lp = as_real(lp_, &np, "lp");
  const int n = LENGTH(x1), P = LENGTH(lp);
  double *L = (double *)R_alloc((size_t)P * n * n + 1, sizeof(double));
  double *dL = (double *)R_alloc((size_t)P * n * n + 1, sizeof(double));
  int *info = (int *)R_alloc((size_t)P + 1, sizeof(int));
  check(gpb200_rbf_cov_chol_batched(handle(), n, REAL(x1), P, REAL(lp), L, dL, info), "rbf_cov_chol_grid");
  for (int q = 0; q < P; q++)
    if (info[q] > 0) Rf_error("rbf_cov_chol_grid: table %d is not positive definite (pivot %d)", q + 1, info[q]);
  SEXP Ls = PROTECT(Rf_allocVector(VECSXP, P));
  SEXP dLs = PROTECT(Rf_allocVector(VECSXP, P));
  np += 2;
  for (int q = 0; q < P; q++) {
    SEXP a = PROTECT(Rf_allocMatrix(REALSXP, n, n));
    SEXP b = PROTECT(Rf_allocMatrix(REALSXP, n, n));
    memcpy(REAL(a), L + (size_t)q * n * n, sizeof(double) * (size_t)n * n);
    memcpy(REAL(b), dL + (size_t)q * n * n, sizeof(double) * (size_t)n * n);
    SET_VECTOR_ELT(Ls, q, a);
    SET_VECTOR_ELT(dLs, q, b);
    UNPROTECT(2);
  }
  SEXP elts[2] = {Ls, dLs};
  static const char *const names[2] = {"Ls", "dLdls"};
  SEXP out = named_list(2, elts, names);
  UNPROTECT(np);
  return out;
}

/* approx_L(M, scale, xt, sigma, l) of models/westbrook.stan:2-30 / bH of spectral_test.R:6-27 */
SEXP gp_approx_L_basis(SEXP M, SEXP scale, SEXP x_, SEXP sigma, SEXP l) {
  int np = 0;
  SEXP x = as_real(x_, &np, "x");
  const int n = LENGTH(x), m = Rf_asInteger(M);
  if (m < 1) Rf_error("approx_L: M must be >= 1");
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, n, m));
  np++;
  check(gpb200_approx_L_basis(handle(), n, m, Rf_asReal(scale), REAL(x), Rf_asReal(sigma), Rf_asReal(l), REAL(out),
                              n > 0 ? n : 1), "approx_L_basis");
  UNPROTECT(np);
  return out;
}

/* L = chol(cov_exp_quad(x, alpha, rho) + diag_add I) and dL/d(alpha | rho): the latent models' Cholesky
 * with its tangent (exact_gp.stan:17-25, fit_full_gp.stan:18-26) */
SEXP gp_se_chol_tangent(SEXP x_, SEXP alpha, SEXP rho, SEXP diag_add, SEXP wrt) {
  int np = 0;
  SEXP x = as_real(x_, &np, "x");
  const int n = LENGTH(x);
  SEXP L = PROTECT(Rf_allocMatrix(REALSXP, n, n));
  SEXP dL = PROTECT(Rf_allocMatrix(REALSXP, n, n));
  np += 2;
  check(gpb200_se_chol_tangent(handle(), n, REAL(x), Rf_asReal(alpha), Rf_asReal(rho), Rf_asReal(diag_add),
                               Rf_asInteger(wrt), REAL(L), REAL(dL)), "se_chol_tangent");
  SEXP elts[2] = {L, dL};
  static const char *const names[2] = {"L", "dL"};
  SEXP out = named_list(2, elts, names);
  UNPROTECT(np);
  return out;
}

/* outer(x, y, kernel) in one call: kind per include/gpb200.h  [derivative_kernels.R, R/kernels.R] */
SEXP gp_gram_outer(SEXP kind, SEXP x_, SEXP y_, SEXP amp2, SEXP l) {
  int np = 0;
  SEXP x = as_real(x_, &np, "x"), y = as_real(y_, &np, "y");
  const int n = LENGTH(x), m = LENGTH(y);
  SEXP K = PROTECT(Rf_allocMatrix(REALSXP, n, m));
  np++;
  check(gpb200_gram_outer(handle(), Rf_asInteger(kind), n, m, REAL(x), REAL(y), Rf_asReal(amp2), Rf_asReal(l),
                          REAL(K), n > 0 ? n : 1), "gram_outer");
  UNPROTECT(np);
  return K;
}

/* element-wise kernel (vectorised R closure semantics) */
SEXP gp_kernel_eval(SEXP kind, SEXP tj_, SEXP tk_, SEXP amp2, SEXP l) {
  int np = 0;
  SEXP tj = as_real(tj_, &np, "tj"), tk = as_real(tk_, &np, "tk");
  const R_xlen_t len = XLENGTH(tj);
  if (XLENGTH(tk) != len) Rf_error("kernel_eval: tj and tk must have the same length (recycle in R first)");
  SEXP out = PROTECT(Rf_allocVector(REALSXP, len));
  np++;
  check(gpb200_kernel_eval(handle(), Rf_asInteger(kind), (long long)len, REAL(tj), REAL(tk), Rf_asReal(amp2),
                           Rf_asReal(l), REAL(out)), "kernel_eval");
  UNPROTECT(np);
  return out;
}

/* QQard(X, Y, phi)                                   [R/kernels.R:19] */
SEXP gp_gram_ard(SEXP X_, SEXP Y_, SEXP alpha, SEXP rho_) {
  int np = 0;
  SEXP X = as_real(X_, &np, "X"), Y = as_real(Y_, &np, "Y"), rho = as_real(rho_, &np, "phi[[2]]");
  const int n = Rf_nrows(X), D = Rf_ncols(X), m = Rf_nrows(Y);
  if (Rf_ncols(Y) != D) Rf_error("QQard: X and Y must have the same number of columns");
  if (LENGTH(rho) != 1 && LENGTH(rho) != D) Rf_error("QQard: phi[[2]] must have length 1 or ncol(X)");
  double *r = (double *)R_alloc((size_t)D + 1, sizeof(double));
  for (int d = 0; d < D; d++) r[d] = REAL(rho)[LENGTH(rho) == 1 ? 0 : d];
  SEXP K = PROTECT(Rf_allocMatrix(REALSXP, n, m));
  np++;
  check(gpb200_gram_ard(handle(), n, m, D, REAL(X), n > 0 ? n : 1, REAL(Y), m > 0 ? m : 1, Rf_asReal(alpha), r, REAL(K),
                        n > 0 ? n : 1), "gram_ard");
  UNPROTECT(np);
  return K;
}

/* joint derivative covariance                        [R/ode_gp_library.R:29-30; design_notes.Rmd] */
SEXP gp_gram_deriv(SEXP t_, SEXP alpha, SEXP rho, SEXP nblocks, SEXP noise_, SEXP jitter, SEXP quirk) {
  int np = 0;
  SEXP t = as_real(t_, &np, "t"), noise = as_real(noise_, &np, "noise");
  const int n = LENGTH(t), nb = Rf_asInteger(nblocks), N = n * nb;
  if (nb < 1 || nb > 3) Rf_error("gram_deriv: nblocks must be 1, 2 or 3");
  if (LENGTH(noise) < nb) Rf_error("gram_deriv: noise must hold one sd per block (%d)", nb);
  SEXP K = PROTECT(Rf_allocMatrix(REALSXP, N, N));
  np++;
  check(gpb200_gram_deriv(handle(), n, REAL(t), Rf_asReal(alpha), Rf_asReal(rho), nb, REAL(noise),
                          Rf_asReal(jitter), Rf_asInteger(quirk), REAL(K), N > 0 ? N : 1), "gram_deriv");
  UNPROTECT(np);
  return K;
}

/* chol(K) lower                                      [spectral_test.R:32; cholesky_decompose] */
SEXP gp_potrf(SEXP K_) {
  int np = 0;
  SEXP K = as_real(K_, &np, "K");
  const int n = Rf_nrows(K);
  need_matrix(K, n, n, "K");
  SEXP L = PROTECT(Rf_duplicate(K));
  np++;
  check(gpb200_potrf(handle(), n, REAL(L), n > 0 ? n : 1), "cholesky_decompose");
  UNPROTECT(np);
  return L;
}

/* solve(K, B) given the lower Cholesky factor L of K (the qr-prefactorised solves of R/ode_gp_library.R:55-57,76) */
SEXP gp_potrs(SEXP L_, SEXP B_) {
  int np = 0;
  SEXP L = as_real(L_, &np, "L"), B = as_real(B_, &np, "B");
  const int n = Rf_nrows(L);
  need_matrix(L, n, n, "L");
  const int is_mat = Rf_ncols(B) > 1 || Rf_nrows(B) != LENGTH(B);
  const int nrhs = is_mat ? Rf_ncols(B) : 1;
  if ((is_mat ? Rf_nrows(B) : LENGTH(B)) != n) Rf_error("potrs: B must have nrow(L) rows");
  SEXP X = PROTECT(Rf_duplicate(B));
  np++;
  check(gpb200_potrs(handle(), n, nrhs, REAL(L), n > 0 ? n : 1, REAL(X), n > 0 ? n : 1), "potrs");
  UNPROTECT(np);
  return X;
}

/* LML + gradient for B draws: theta is a 3 x B matrix (alpha, rho, sigma per column) */
SEXP gp_lml_grad_draws(SEXP x_, SEXP y_, SEXP theta_, SEXP jitter) {
  int np = 0;
  SEXP x = as_real(x_, &np, "x"), y = as_real(y_, &np, "y"), theta = as_real(theta_, &np, "theta");
  const int n = LENGTH(x), B = Rf_ncols(theta);
  if (LENGTH(y) != n) Rf_error("gp_lml_grad_draws: length(y) = %d must equal length(x) = %d", LENGTH(y), n);
  if (Rf_nrows(theta) != 3)
    Rf_error("gp_lml_grad_draws: theta must be a 3 x B matrix, one (alpha, rho, sigma) per COLUMN (got %d x %d; "
             "transpose a draws-by-parameters matrix)", Rf_nrows(theta), B);
  SEXP lml = PROTECT(Rf_allocVector(REALSXP, B));
  SEXP grad = PROTECT(Rf_allocMatrix(REALSXP, 3, B));
  SEXP info = PROTECT(Rf_allocVector(INTSXP, B));
  np += 3;
  check(gpb200_lml_grad_batched(handle(), n, B, REAL(x), 0, REAL(y), 0, REAL(theta), Rf_asReal(jitter), 1,
                                REAL(lml), REAL(grad), INTEGER(info)), "lml_grad_draws");
  SEXP elts[3] = {lml, grad, info};
  static const char *const names[3] = {"lml", "grad", "info"};
  SEXP out = named_list(3, elts, names);
  UNPROTECT(np);
  return out;
}

/* LML + gradient of a GP observed through derivative orders order0 .. order0+nblocks-1 on the grid t
 * (gpderivs.py:62-83 is order0 = 1, nblocks = 1; design_notes.Rmd:25-46 is 0, 3); theta is a
 * (2 + nblocks) x B matrix (alpha, rho, noise[nblocks] per column), y the stacked observations */
SEXP gp_lml_grad_deriv_draws(SEXP t_, SEXP y_, SEXP theta_, SEXP order0, SEXP jitter) {
  int np = 0;
  SEXP t = as_real(t_, &np, "t"), y = as_real(y_, &np, "y"), theta = as_real(theta_, &np, "theta");
  const int n = LENGTH(t), B = Rf_ncols(theta), nb = Rf_nrows(theta) - 2;
  if (nb < 1 || nb > 3) Rf_error("gp_lml_grad_deriv_draws: theta must be a (2 + nblocks) x B matrix with nblocks in 1..3");
  if (LENGTH(y) != n * nb) Rf_error("gp_lml_grad_deriv_draws: y must hold n * (nrow(theta) - 2) = %d values", n * nb);
  SEXP lml = PROTECT(Rf_allocVector(REALSXP, B));
  SEXP grad = PROTECT(Rf_allocMatrix(REALSXP, 2 + nb, B));
  SEXP info = PROTECT(Rf_allocVector(INTSXP, B));
  np += 3;
  check(gpb200_lml_grad_deriv_batched(handle(), n, Rf_asInteger(order0), nb, B, REAL(t), 0, REAL(y), 0, REAL(theta),
                                      Rf_asReal(jitter), 1, REAL(lml), REAL(grad), INTEGER(info)), "lml_grad_deriv_draws");
  SEXP elts[3] = {lml, grad, info};
  static const char *const names[3] = {"lml", "grad", "info"};
  SEXP out = named_list(3, elts, names);
  UNPROTECT(np);
  return out;
}

/* MASS::mvrnorm(n, mu, Sigma) with the device generator (pendulum_fit.R:253): n x length(mu) matrix; mu may be NULL */
SEXP gp_mvrnorm(SEXP n_, SEXP mu_, SEXP Sigma_, SEXP seed) {
  int np = 0;
  SEXP Sigma = as_real(Sigma_, &np, "Sigma");
  const int nd = Rf_asInteger(n_), m = Rf_nrows(Sigma);
  need_matrix(Sigma, m, m, "Sigma");
  if (nd < 0) Rf_error("mvrnorm: n must be >= 0");
  const double *mu = NULL;
  if (!Rf_isNull(mu_)) {
    SEXP mur = as_real(mu_, &np, "mu");
    if (LENGTH(mur) != m) Rf_error("mvrnorm: length(mu) = %d must equal nrow(Sigma) = %d", LENGTH(mur), m);
    mu = REAL(mur);
  }
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, nd, m));
  np++;
  check(gpb200_mvrnorm(handle(), nd, m, mu, REAL(Sigma), m > 0 ? m : 1, 0.0, (unsigned long long)Rf_asReal(seed), REAL(out),
                       nd > 0 ? nd : 1), "mvrnorm");
  UNPROTECT(np);
  return out;
}

/* The mclapply body of pendulum_fit.R:259-268 for all draws at once: one sample_derivs (:227-255) draw per COLUMN
 * (l, a, sy) of the 3 x B matrix params; ynoise is a vector of length(ti) or a length(ti) x B matrix.  Normals: the
 * device stream of `seed`, or the length(ti) x B matrix z when seed is NULL.  Returns a length(ti) x B matrix. */
SEXP gp_sample_derivs_draws(SEXP params_, SEXP ynoise_, SEXP ti_, SEXP seed, SEXP z_) {
  int np = 0;
  SEXP params = as_real(params_, &np, "params"), y = as_real(ynoise_, &np, "ynoise"), ti = as_real(ti_, &np, "ti");
  const int n = LENGTH(ti), B = Rf_ncols(params);
  if (n < 1) Rf_error("sample_derivs_draws: ti must not be empty");
  if (Rf_nrows(params) != 3)
    Rf_error("sample_derivs_draws: params must be a 3 x B matrix, one (l, a, sy) per COLUMN (got %d x %d)", Rf_nrows(params), B);
  const int y_mat = LENGTH(y) != n;
  if (y_mat) need_matrix(y, n, B, "ynoise");
  const double *z = NULL;
  if (Rf_isNull(seed)) {
    SEXP zr = as_real(z_, &np, "z (normals, needed when seed is NULL)");
    need_matrix(zr, n, B, "z");
    z = REAL(zr);
  }
  SEXP theta = PROTECT(Rf_allocVector(REALSXP, 3 * (R_xlen_t)B));
  SEXP out = PROTECT(Rf_allocMatrix(REALSXP, n, B));
  SEXP info = PROTECT(Rf_allocVector(INTSXP, B));
  np += 3;
  const double *p = REAL(params);
  double *th = REAL(theta);
  for (int b = 0; b < B; b++) {  /* (l, a, sy) -> (alpha, rho, sigma) */
    th[3 * b] = p[3 * b + 1];
    th[3 * b + 1] = p[3 * b];
    th[3 * b + 2] = p[3 * b + 2];
  }
  check(gpb200_posterior_draws_batched(handle(), n, n, 1, B, REAL(ti), 0, NULL, 0, REAL(y), y_mat ? n : 0, th, 1e-8, z,
                                       z ? 0ULL : (unsigned long long)Rf_asReal(seed), REAL(out), NULL, INTEGER(info)),
        "sample_derivs_draws");
  for (int b = 0; b < B; b++)
    if (INTEGER(info)[b]) Rf_error("sample_derivs_draws: draw %d: matrix is not positive definite (first non-positive pivot at %d)",
                                   b + 1, INTEGER(info)[b]);
  UNPROTECT(np);
  return out;
}

/* mu = Ks (K + s2 I)^-1 y ; cov = Kss - Ks (K + s2 I)^-1 Ks^T + jitter I   [pendulum_fit.R:242-251] */
SEXP gp_condition(SEXP K_, SEXP Ks_, SEXP Kss_, SEXP y_, SEXP noise_var, SEXP jitter) {
  int np = 0;
  SEXP K = as_real(K_, &np, "K"), Ks = as_real(Ks_, &np, "Ks"), Kss = as_real(Kss_, &np, "Kss"), y = as_real(y_, &np, "y");
  const int n = Rf_nrows(K), m = Rf_nrows(Ks);
  need_matrix(K, n, n, "K");
  need_matrix(Ks, m, n, "Ks");
  need_matrix(Kss, m, m, "Kss");
  if (LENGTH(y) != n) Rf_error("gp_condition: length(y) = %d must equal nrow(K) = %d", LENGTH(y), n);
  SEXP mu = PROTECT(Rf_allocVector(REALSXP, m));
  SEXP cov = PROTECT(Rf_allocMatrix(REALSXP, m, m));
  np += 2;
  check(gpb200_gp_condition(handle(), n, m, REAL(K), n, REAL(Ks), m, REAL(Kss), m, REAL(y), Rf_asReal(noise_var),
                            Rf_asReal(jitter), REAL(mu), REAL(cov), m), "gp_condition");
  SEXP elts[2] = {mu, cov};
  static const char *const names[2] = {"mu", "cov"};
  SEXP out = named_list(2, elts, names);
  UNPROTECT(np);
  return out;
}

/* condMVN for the reference's block layout (given block first)   [R/ode_gp_library.R:17,32]; mean may be NULL (zeros) */
SEXP gp_cond_mvn(SEXP mean_, SEXP sigma_, SEXP ng_, SEXP x_given_) {
  int np = 0;
  SEXP sigma = as_real(sigma_, &np, "sigma"), x_given = as_real(x_given_, &np, "X.given");
  const int N = Rf_nrows(sigma), ng = Rf_asInteger(ng_), nd = N - ng;
  need_matrix(sigma, N, N, "sigma");
  if (ng < 1 || nd < 1) Rf_error("condMVN: need at least one given and one dependent index");
  if (LENGTH(x_given) != ng) Rf_error("condMVN: length(X.given) = %d must equal the number of given indices %d", LENGTH(x_given), ng);
  const double *mean = NULL;
  if (!Rf_isNull(mean_)) {
    SEXP mr = as_real(mean_, &np, "mean");
    if (LENGTH(mr) != N) Rf_error("condMVN: length(mean) = %d must equal nrow(sigma) = %d", LENGTH(mr), N);
    mean = REAL(mr);
  }
  SEXP cm = PROTECT(Rf_allocVector(REALSXP, nd));
  SEXP cv = PROTECT(Rf_allocMatrix(REALSXP, nd, nd));
  np += 2;
  check(gpb200_cond_mvn(handle(), ng, nd, mean, REAL(sigma), N, REAL(x_given), REAL(cm), REAL(cv), nd), "condMVN");
  SEXP elts[2] = {cm, cv};
  static const char *const names[2] = {"condMean", "condVar"};
  SEXP out = named_list(2, elts, names);
  UNPROTECT(np);
  return out;
}

static const R_CallMethodDef call_methods[] = {
    {"gp_rbf_cov_chol", (DL_FUNC)&gp_rbf_cov_chol, 2}, {"gp_approx_L", (DL_FUNC)&gp_approx_L, 4},
    {"gp_approx_Lz", (DL_FUNC)&gp_approx_Lz, 5},
    {"gp_gram_outer", (DL_FUNC)&gp_gram_outer, 5},     {"gp_kernel_eval", (DL_FUNC)&gp_kernel_eval, 5},
    {"gp_gram_ard", (DL_FUNC)&gp_gram_ard, 4},         {"gp_gram_deriv", (DL_FUNC)&gp_gram_deriv, 7},
    {"gp_potrf", (DL_FUNC)&gp_potrf, 1},               {"gp_potrs", (DL_FUNC)&gp_potrs, 2},
    {"gp_lml_grad_draws", (DL_FUNC)&gp_lml_grad_draws, 4},
    {"gp_condition", (DL_FUNC)&gp_condition, 6},       {"gp_cond_mvn", (DL_FUNC)&gp_cond_mvn, 4},
    {"gp_rbf_cov_chol_grid", (DL_FUNC)&gp_rbf_cov_chol_grid, 2}, {"gp_approx_L_basis", (DL_FUNC)&gp_approx_L_basis, 5},
    {"gp_se_chol_tangent", (DL_FUNC)&gp_se_chol_tangent, 5},
    {"gp_lml_grad_deriv_draws", (DL_FUNC)&gp_lml_grad_deriv_draws, 5}, {"gp_mvrnorm", (DL_FUNC)&gp_mvrnorm, 4},
    {"gp_sample_derivs_draws", (DL_FUNC)&gp_sample_derivs_draws, 5},
    {NULL, NULL, 0}};

void R_init_gpb200_r(DllInfo *dll) {
  R_registerRoutines(dll, NULL, call_methods, NULL, NULL);
  R_useDynamicSymbols(dll, FALSE);
}
