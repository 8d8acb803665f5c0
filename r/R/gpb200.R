# Core of the drop-in R layer backed by libgpb200.so (through r/shim.c).  Source this file INSTEAD of
#   sourceCpp("covariance.cpp")            (gpc_sigma.R:7)
# and then, exactly where the reference sources its own files, the same-named replacements:
#   source("r/R/kernels.R")              for  source("R/kernels.R")              QQ/QR/RR(x, y, phi), QQard
#   source("r/R/derivative_kernels.R")   for  source("derivative_kernels.R")     QQ..TT(tj, tk, l)
#   source("r/R/ode_gp_library.R")       for  source("R/ode_gp_library.R")       p_Xn, p_dotXn, create_p_dotXnS (condMVN flavour)
#   source("r/R/ode_gp.R")               for  source("R/ode_gp.R")               the same with $mn / $Kn
# (kernels.R and derivative_kernels.R define the same names with different arities in the reference too:
# source the flavour you need last, as the reference's scripts do.)
# Formals are identical to the reference's; each matrix is built by ONE .Call instead of outer().
dyn.load(file.path(Sys.getenv("GPB200_HOME", "."), "r", "gpb200_r.so"))

.gp_kind <- c(QQ = 0L, QR = 1L, RQ = 2L, RR = 3L, QT = 4L, TQ = 5L, RT = 6L, TR = 7L, TT = 8L, RR_QUIRK = 9L)

# ---- covariance.cpp -----------------------------------------------------------------------------
rbf_cov_chol <- function(x1, l_) .Call("gp_rbf_cov_chol", x1, l_)
approx_L <- function(l, lp, Ls, dLdls) .Call("gp_approx_L", l, lp, Ls, dLdls)
# models/cubic_interpolated_gp.hpp:38-73: list(vz = v(l) %*% z, dvdl_z = dv/dl %*% z), tables read once on the GPU
approx_Lz <- function(l, lp, Ls, dLdls, z) .Call("gp_approx_Lz", l, lp, Ls, dLdls, z)
# all tables of a length-scale grid in one GPU call: tabs <- rbf_cov_chol_grid(x, lp); tabs$Ls, tabs$dLdls
rbf_cov_chol_grid <- function(x1, lp) .Call("gp_rbf_cov_chol_grid", x1, lp)
# eigen-basis factor of models/westbrook.stan:2-30 (named approx_L there too; bH in spectral_test.R:6)
bH <- function(M, scale, x, sigma, l) .Call("gp_approx_L_basis", as.integer(M), scale, x, sigma, l)
# latent models: Cholesky and its tangent (wrt = 0 alpha, 1 rho)
se_chol_tangent <- function(x, alpha, rho, diag_add, wrt) .Call("gp_se_chol_tangent", x, alpha, rho, diag_add, as.integer(wrt))

# ---- whole-matrix kernel builders used by the per-file replacements -------------------------------
# outer(tj, tk, FUN = kern) in one call (pendulum_fit.R:238-240)
gp_outer <- function(kind, tj, tk, l, amp2 = 1.0) .Call("gp_gram_outer", .gp_kind[[kind]], tj, tk, amp2, l)
# the element-wise closures of derivative_kernels.R, vectorised with R's recycling rule
gp_elementwise <- function(kind, tj, tk, l) {
  n <- max(length(tj), length(tk))
  .Call("gp_kernel_eval", .gp_kind[[kind]], rep_len(as.double(tj), n), rep_len(as.double(tk), n), 1.0, l)
}
gp_chol <- function(K) .Call("gp_potrf", K)                    # lower factor (t(chol(K)) in base R)
gp_chol_solve <- function(L, B) .Call("gp_potrs", L, B)        # solve(K, B) given L
gp_condition <- function(K, Ks, Kss, y, noise_var, jitter = 0) .Call("gp_condition", K, Ks, Kss, y, noise_var, jitter)
# condMVNorm::condMVN(mean, sigma, dependent.ind, given.ind, X.given) for the block layout the reference uses
# (given block first, R/ode_gp_library.R:17,32); other layouts are permuted into it here
condMVN <- function(mean, sigma, dependent.ind, given.ind = integer(0), X.given = numeric(0)) {
  if (length(given.ind) == 0) return(list(condMean = mean[dependent.ind], condVar = sigma[dependent.ind, dependent.ind, drop = FALSE]))
  ord <- c(given.ind, dependent.ind)
  .Call("gp_cond_mvn", mean[ord], sigma[ord, ord, drop = FALSE], length(given.ind), X.given)
}

# ---- pendulum_fit.R:227-255 -----------------------------------------------------------------------
sample_derivs <- function(params, ynoise, ti, seed = NULL) {
  l <- params[1]; a <- params[2]; sy <- params[3]
  K <- gp_outer("QQ", ti, ti, l, a^2); KsK <- gp_outer("RQ", ti, ti, l, a^2); KsKs <- gp_outer("RR", ti, ti, l, a^2)
  m <- gp_condition(K, KsK, KsKs, ynoise, sy^2, 1e-8)
  if (!is.null(seed)) return(as.numeric(.Call("gp_mvrnorm", 1L, m$mu, m$cov, seed)))  # device RNG
  L <- gp_chol(m$cov)
  as.numeric(m$mu + L %*% rnorm(length(m$mu)))
}
# the mclapply loop of pendulum_fit.R:259-268 in one GPU call: params is 3 x B, one (l, a, sy) per COLUMN; ynoise a
# vector or a length(ti) x B matrix; returns a length(ti) x B matrix, column b = sample_derivs(params[, b], ...)
sample_derivs_draws <- function(params, ynoise, ti, seed = NULL) {
  params <- as.matrix(params)
  z <- if (is.null(seed)) matrix(rnorm(length(ti) * ncol(params)), length(ti), ncol(params)) else NULL
  .Call("gp_sample_derivs_draws", params, ynoise, ti, seed, z)
}
mvrnorm <- function(n = 1, mu, Sigma, seed = sample.int(.Machine$integer.max, 1)) {   # MASS::mvrnorm signature + seed
  out <- .Call("gp_mvrnorm", as.integer(n), mu, Sigma, seed)
  if (n == 1) drop(out) else out
}

# ---- batched LML + gradient over hyper-parameter draws (the mclapply axis, pendulum_fit.R:259-268) -
# theta: 3 x B matrix, one (alpha, rho, sigma) per COLUMN
gp_lml_grad_draws <- function(x, y, theta, jitter = 0) .Call("gp_lml_grad_draws", x, y, theta, jitter)

# ---- GP observed through derivatives (the Stan model inside gpderivs.py:25-133; design_notes.Rmd:25-46) ----
# theta: (2 + nblocks) x B matrix, columns (alpha, rho, noise_1..noise_nblocks); y = c(y, yp, ypp) stacked
gp_lml_grad_deriv_draws <- function(t, y, theta, order0 = 0L, jitter = 0)
  .Call("gp_lml_grad_deriv_draws", t, y, theta, as.integer(order0), jitter)
