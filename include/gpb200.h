/* gpb200.h -- C ABI of libgpb200.so: the B200-native (sm_100a) GP hot path that replaces the
 * arithmetic behind bbbales2/gp's native and R-level entry points.
 *
 * Conventions (the ones R / Rcpp / Eigen use on the reference side):
 *   - every matrix is COLUMN-MAJOR double with an explicit leading dimension;
 *   - plain pointers and sizes only -- no R, Stan, Eigen or torch types cross this boundary;
 *   - every call returns an int status: 0 = ok; k > 0 = the matrix is not positive definite and
 *     k is the 1-based index of the first non-positive pivot (LAPACK convention; Stan Math's
 *     cholesky_decompose throws std::domain_error in that case, the R shim raises an R error);
 *     k < 0 = bad argument / CUDA failure, text available from gpb200_last_error();
 *   - pointers are HOST pointers by default (R's memory); gpb200_set_pointer_mode(h, 1) makes all
 *     DATA pointers device pointers (scalars passed by value stay by value; output scalars are
 *     then device pointers too).  The library synchronises before returning in host mode; in
 *     device mode work is enqueued on the handle's stream and the caller synchronises.
 *   - theta is always (alpha, rho, sigma): amplitude, length-scale, noise sd  (the parameters of
 *     models/fit_hyperparameters.stan:12-16).
 *
 * There is no CPU fallback: every entry point runs hand-written CUDA kernels and fails with a
 * negative status if no sm_100 device is present.
 *
 * Reference citations are relative to the root of bbbales2/gp.
 */
#ifndef GPB200_H
#define GPB200_H

#if defined(__GNUC__)
#define GPB200_API __attribute__((visibility("default")))
#else
#define GPB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpb200_handle_s *gpb200_handle_t;

/* ---- handle ------------------------------------------------------------------------------- */
GPB200_API int gpb200_create(gpb200_handle_t *h, int device);          /* one handle per GPU / host thread  */
GPB200_API int gpb200_destroy(gpb200_handle_t h);
GPB200_API int gpb200_set_stream(gpb200_handle_t h, void *cuda_stream); /* cudaStream_t; NULL = default      */
/* gpb200_set_stream orders the new stream after everything the handle enqueued on the old one (one workspace per handle).
 * The _unordered form adds no such edge: for callers that overlap independent gpb200_mg_panel_* / gpb200_mg_bcast work of
 * one handle on several streams and order it with their own events (gp_b200/block_cyclic.py). */
GPB200_API int gpb200_set_stream_unordered(gpb200_handle_t h, void *cuda_stream);
GPB200_API int gpb200_set_pointer_mode(gpb200_handle_t h, int device_pointers);
GPB200_API int gpb200_synchronize(gpb200_handle_t h);
GPB200_API const char *gpb200_last_error(gpb200_handle_t h);
GPB200_API long long gpb200_launch_count(gpb200_handle_t h);            /* kernels launched by this handle   */
GPB200_API int gpb200_version(void);
/* cap on the device workspace the batched entry points may use (bytes; 0 = 85% of free memory);
 * a batch that does not fit is processed in chunks with identical results */
GPB200_API int gpb200_set_workspace_limit(gpb200_handle_t h, long long bytes);

/* Small (launch-latency-bound) lml_grad evaluations are replayed as one CUDA graph; this returns how
 * many replays the handle has done.  GPB200_NO_GRAPH=1 in the environment disables the graphs. */
GPB200_API long long gpb200_graph_replays(gpb200_handle_t h);

/* tuning/testing knob: Cholesky panel width in 128-column tiles (0 = automatic: pure left-looking
 * for batches >= 64, 8-tile panels + right-looking trailing updates for small batches) */
GPB200_API int gpb200_set_chol_panel_tiles(gpb200_handle_t h, int tiles);

/* tuning/testing knob: GEMM configuration.  0 = default (2); 1 = one 128x128 CTA per SM (8 warps of 64x32,
 * the first design); 2 = two 128x64 half-tile CTAs per SM (8 warps of 32x32 each).  GPB200_GEMM_CFG in the
 * environment sets the same knob at handle creation. */
GPB200_API int gpb200_set_gemm_config(gpb200_handle_t h, int cfg);

/* per-kernel-class timing with CUDA events on the handle's stream (used by bench.py for the
 * roofline of the dominant kernel).  Classes: 0 DMMA tile GEMM, 1 POTRF tile, 2 TRSM tile,
 * 3 Gram, 4 triangular mat-vec/solves, 5 other.  get_profile synchronises, sums and resets. */
GPB200_API int gpb200_set_profiling(gpb200_handle_t h, int on);
GPB200_API int gpb200_get_profile(gpb200_handle_t h, double *ms_out6, long long *count_out6);

/* flops the DMMA tile-GEMM launches really executed since counting was switched on: 2 x CTA tile area x contraction
 * length per CTA, after the skipping of triangular / symmetric tile parts (host-side, from the task lists) and of the
 * tiles outside an item's envelope (counted by the CTAs on the device; the getter waits for the handle's stream);
 * bench.py reports it against the algorithmic count */
GPB200_API int gpb200_set_flop_counting(gpb200_handle_t h, int on);
GPB200_API double gpb200_executed_gemm_flops(gpb200_handle_t h);

/* tuning aid (not a reference interface): times one panel kernel in isolation on `batch` synthetic
 * matrices of nt x nt 128-tiles.  what: 0 POTRF of a diagonal tile, 1 TRSM of the nt-1 tiles below it,
 * 2 inverse of the nt diagonal tiles, 3 POTRF + TRSM of the first block column the way the Cholesky issues them (one fused
 * launch on the latency path, else two).  ms_out[0] = mean device time per launch (CUDA events). */
GPB200_API int gpb200_debug_bench_panel(gpb200_handle_t h, int what, int nt, int batch, int reps, double *ms_out);
/* instrumented builds only (-DGPB_PANEL_TRACE): 2048 clock64 stamps left by CTA 0 of the panel kernels; -1 otherwise */
GPB200_API int gpb200_debug_panel_trace(gpb200_handle_t h, long long *out2048);

/* ---- a9: kernel functions ------------------------------------------------------------------ */
/* kinds of derivative_kernels.R:39-73 (Q = value, R = first derivative, T = second derivative;
 * first letter goes with tj) */
enum { GPB200_QQ = 0, GPB200_QR = 1, GPB200_RQ = 2, GPB200_RR = 3, GPB200_QT = 4,
       GPB200_TQ = 5, GPB200_RT = 6, GPB200_TR = 7, GPB200_TT = 8,
       GPB200_RR_QUIRK = 9 /* R/kernels.R:30-32: amp2 multiplies only the first term */ };

/* element-wise kernel: out[i] = amp2 * kind(tj[i], tk[i], l) -- the R closures
 * QQ..TT(tj, tk, l) of derivative_kernels.R:39-73 (amp2 = 1) and gp_derivs.py:15-40 (amp2 = a^2) */
GPB200_API int gpb200_kernel_eval(gpb200_handle_t h, int kind, long long len, const double *tj,
                       const double *tk, double amp2, double l, double *out);

/* outer(x, y, kind): K[i + j*ldk] = amp2 * kind(x[i], y[j], l), n x m.  Replaces
 * outer(ti, ti, FUN = kern) (pendulum_fit.R:238-240), QQ/QR/RR(x, y, phi) of R/kernels.R:22-32
 * (amp2 = phi1^2, l = phi2) and cov() of gp_derivs.py:76-83. */
GPB200_API int gpb200_gram_outer(gpb200_handle_t h, int kind, int n, int m, const double *x, const double *y,
                      double amp2, double l, double *K, int ldk);

/* QQard (R/kernels.R:19): K[i,j] = alpha^2 exp(-0.5 sum_d ((X[i,d]-Y[j,d])/rho[d])^2);
 * X is n x D, Y is m x D, both column-major (R matrices). */
GPB200_API int gpb200_gram_ard(gpb200_handle_t h, int n, int m, int D, const double *X, int ldx,
                    const double *Y, int ldy, double alpha, const double *rho, double *K, int ldk);

/* cov_exp_quad(x, alpha, rho) + diag_add * I in one pass (models/fit_hyperparameters.stan:19-24,
 * exact_gp.stan:17-22, covariance.cpp:15-25 with alpha = 1, diag_add = 1e-10). Full symmetric
 * n x n output. */
GPB200_API int gpb200_gram_se(gpb200_handle_t h, int n, const double *x, double alpha, double rho,
                   double diag_add, double *K, int ldk);

/* joint covariance of (y, y', y'') on one grid t (design_notes.Rmd:6-46; blocks
 * {QQ,QR,QT;RQ,RR,RT;TQ,TR,TT} * alpha^2 + diag(noise[b]^2 + jitter)); nblocks in 1..3,
 * output (nblocks*n)^2.  nblocks = 2, noise = (sigma, 0), jitter = 1e-6 is the matrix of
 * R/ode_gp_library.R:29-30 (set quirk = 1 for R/kernels.R's RR). */
GPB200_API int gpb200_gram_deriv(gpb200_handle_t h, int n, const double *t, double alpha, double rho,
                      int nblocks, const double *noise, double jitter, int quirk, double *K,
                      int ldk);

/* f-3: approx_L(M, scale, xt, sigma, l) of models/westbrook.stan:2-30 (and its six copies;
 * spectral_test.R:6-27 bH): N x M eigen-basis factor, out out^T ~ cov_exp_quad(x, sigma, l). */
GPB200_API int gpb200_approx_L_basis(gpb200_handle_t h, int n, int M, double scale, const double *x,
                                     double sigma, double l, double *out, int ldo);

/* ---- a6-a8: factorisation, solves, likelihood ------------------------------------------------ */
/* cholesky_decompose (fit_hyperparameters.stan:25; covariance.cpp:29; R chol spectral_test.R:32):
 * in place, lower; the strict upper triangle is zeroed like Eigen's matrixL(). */
GPB200_API int gpb200_potrf(gpb200_handle_t h, int n, double *A, int lda);

/* mdivide_left_tri_low (inside multi_normal_cholesky): B <- L^-1 B, n x nrhs */
GPB200_API int gpb200_trsm_lower(gpb200_handle_t h, int n, int nrhs, const double *L, int ldl, double *B,
                      int ldb);
/* B <- (L L^T)^-1 B: solve(K, y), solve(K, KKs) (pendulum_fit.R:244,250) given the factor */
GPB200_API int gpb200_potrs(gpb200_handle_t h, int n, int nrhs, const double *L, int ldl, double *B, int ldb);
/* f = L z, lower-triangular (exact_gp.stan:25, heteroscedastic.stan:31-32) */
GPB200_API int gpb200_trmv_lower(gpb200_handle_t h, int n, const double *L, int ldl, const double *z,
                      double *f);
/* f = L^T z: the adjoint of the above (zbar = L^T fbar in the reverse sweep of f = L z) */
GPB200_API int gpb200_trmv_lower_t(gpb200_handle_t h, int n, const double *L, int ldl, const double *z,
                        double *f);
/* multi_normal_cholesky_lpdf(y | mu, L) (fit_hyperparameters.stan:31); mu may be NULL (zeros);
 * drop_constants != 0 omits -0.5 n log(2 pi) like Stan's `~` statement. */
GPB200_API int gpb200_mvn_chol_lpdf(gpb200_handle_t h, int n, const double *y, const double *mu,
                         const double *L, int ldl, int drop_constants, double *lp);

/* ---- CS-A: fused Gram -> Cholesky -> LML + gradient ----------------------------------------- */
/* One evaluation of the model block of models/fit_hyperparameters.stan:18-31 and of its reverse
 * sweep: K = cov_exp_quad(x, alpha, rho) + (sigma^2 + jitter) I;
 * lml = MVN(y | 0, K) with constants; grad = d lml / d (alpha, rho, sigma). */
GPB200_API int gpb200_lml_grad(gpb200_handle_t h, int n, const double *x, const double *y,
                    const double *theta, double jitter, double *lml, double *grad);

/* B independent evaluations (hyper-parameter draws: pendulum_fit.R:259-268; per-group GPs:
 * multiple_players.stan:59-63).  x, y: B strides in doubles (0 = one shared vector);
 * theta: B x 3 row-major; outputs lml[B], grad[B*3], info[B] (per-item LAPACK-style status).
 * want_grad = 0 skips the inverse (LML only, N^3/3 flops instead of N^3). */
GPB200_API int gpb200_lml_grad_batched(gpb200_handle_t h, int n, int B, const double *x, long long x_stride,
                            const double *y, long long y_stride, const double *theta,
                            double jitter, int want_grad, double *lml, double *grad, int *info);

/* The same evaluation for a GP observed through derivatives (config C2; the dense-multi_normal LML of
 * gpderivs.py:62-83 over the covdd kernel is order0 = 1, nblocks = 1; design_notes.Rmd:25-46 is the
 * joint (y, y', y'') case order0 = 0, nblocks = 3).  On a grid t[n] the covariance is
 *   K = alpha^2 {k_pq(t_i, t_j)}_{p,q = order0 .. order0+nblocks-1} + diag(noise_b^2 + jitter)
 * with k_pq the kernels of derivative_kernels.R:39-73 (QQ..TT); it is (n*nblocks)^2, block b holding
 * derivative order order0 + b, and y is the stacked observation vector of length n*nblocks.
 * theta: B x (2 + nblocks) row-major = (alpha, rho, noise[0..nblocks)); grad has the same layout;
 * t_stride / y_stride in doubles (0 = shared); lml[B], info[B]. */
GPB200_API int gpb200_lml_grad_deriv_batched(gpb200_handle_t h, int n, int order0, int nblocks, int B,
                                             const double *t, long long t_stride, const double *y,
                                             long long y_stride, const double *theta, double jitter,
                                             int want_grad, double *lml, double *grad, int *info);

/* LML + gradient of B GPs with the ARD squared-exponential covariance (QQard, R/kernels.R:19):
 *   K = alpha^2 exp(-0.5 sum_d (X[i,d] - X[j,d])^2 / rho_d^2) + (sigma^2 + jitter) I,   1 <= D <= 8
 * X: per item an n x D column-major matrix with leading dimension n (an R matrix); x_stride in doubles between items
 * (0 = shared, else >= n*D); y, y_stride as in gpb200_lml_grad_batched; theta and grad: B x (D + 2) row-major,
 * (alpha, rho_1 .. rho_D, sigma); lml[B], info[B] with the conventions of gpb200_lml_grad_batched.
 * want_grad = 0 skips the inverse.  At D = 1 this is the model of gpb200_lml_grad_batched. */
GPB200_API int gpb200_lml_grad_ard_batched(gpb200_handle_t h, int n, int D, int B, const double *X, long long x_stride,
                                           const double *y, long long y_stride, const double *theta, double jitter,
                                           int want_grad, double *lml, double *grad, int *info);

/* B independent GPs of different sizes (per-group GPs, multiple_players.stan:59-63), the model of
 * gpb200_lml_grad_batched for each: item b owns x[offsets[b] .. offsets[b+1]) and the same slice of y,
 * n_b = offsets[b+1] - offsets[b] >= 1 (at most 65407).  offsets: HOST array of B + 1 int64, offsets[0] = 0,
 * non-decreasing (sizes are scheduling information, as ls of gpb200_rbf_cov_chol_batched).  x, y, theta (B x 3
 * row-major), lml[B], grad[B*3], info[B] follow the pointer mode; any of lml, grad, info may be NULL and is then
 * not written (grad is not written when want_grad = 0).  B has no limit beyond memory.  info[b] in 1..n_b as in gpb200_lml_grad_batched; the other items are unaffected by a failing one.
 * Item b gives, to rounding, what gpb200_lml_grad_batched(h, n_b, 1, x + offsets[b], 0, y + offsets[b], 0,
 * theta + 3b, ...) gives.  The items run as one lock-step batch per tile count ceil(n_b / 128), zero-padded to
 * 128 * that count (the padding is exact), the bucket with the most work first. */
GPB200_API int gpb200_lml_grad_ragged(gpb200_handle_t h, int B, const long long *offsets, const double *x,
                                      const double *y, const double *theta, double jitter, int want_grad,
                                      double *lml, double *grad, int *info);

/* ---- a1-a3: the reference's one native entry point ----------------------------------------- */
/* Exact twin of rbf_cov_chol (covariance.cpp:9-47): Sigma = exp(-(xi-xj)^2/(2 l^2)) + 1e-10 I,
 * L = chol(Sigma), dLdl = d L / d l (forward mode); both n x n column-major with zero strict
 * upper triangle. */
GPB200_API int gpb200_rbf_cov_chol(gpb200_handle_t h, int n, const double *x1, double l, double *L,
                        double *dLdl);

/* The same for P length-scales in one call: the tables Ls[P], dLdls[P] that approx_L / approx_Lz
 * interpolate (models/interpolated_gp.stan:15-21 builds them with P separate Choleskys;
 * test_interpolate.R:9 uses P = 10).  ls, info: HOST arrays of length P; L, dLdl: P consecutive n x n. */
GPB200_API int gpb200_rbf_cov_chol_batched(gpb200_handle_t h, int n, const double *x1, int P, const double *ls,
                                           double *L, double *dLdl, int *info);

/* Generalisation used by the non-centred latent models (exact_gp.stan:17-25 alpha = 1, diag_add =
 * 1e-10; fit_full_gp.stan:18-26; heteroscedastic.stan:23-32): L = chol(cov_exp_quad(x, alpha, rho) +
 * diag_add I) and its forward-mode tangent dL/dalpha (wrt = 0) or dL/drho (wrt = 1).  With f = L z
 * the reverse sweep through the Cholesky that Stan performs is  d lp/d theta = fbar^T (dL z). */
GPB200_API int gpb200_se_chol_tangent(gpb200_handle_t h, int n, const double *x, double alpha, double rho,
                                      double diag_add, int wrt, double *L, double *dL);

/* f-2, REVERSE mode: the non-centred latent models differentiate through cholesky_decompose (exact_gp.stan:17-25,
 * fit_full_gp.stan:18-26, westbrook_exact.stan:17-24; heteroscedastic.stan:23-32 with two mat-vecs on one L).
 * forward: f_m = L z_m, m < nvec, L = chol(cov_exp_quad(x, alpha, rho) + diag_add I) (kept on the device);
 * backward: given fbar_m = d lp / d f_m, zbar_m = L^T fbar_m and theta_bar = d lp / d (alpha, rho) through f and the
 * Cholesky (Kbar = L^-T Phi(L^T Lbar) L^-1 contracted with dK/dtheta): ONE N^3 pass for all parameters, instead of one
 * 5 N^3 / 3 forward-mode pass per parameter.  z, f, fbar, zbar: nvec consecutive vectors of length n. */
GPB200_API int gpb200_latent_forward(gpb200_handle_t h, int n, const double *x, double alpha, double rho, double diag_add,
                                     int nvec, const double *z, double *f);
GPB200_API int gpb200_latent_backward(gpb200_handle_t h, int n, const double *x, double alpha, double rho, double diag_add,
                                      int nvec, const double *z, const double *fbar, double *theta_bar, double *zbar);

/* B states of the non-centred latent model in one call (multi-chain samplers, f over a set of posterior draws).  Item b:
 *   K_b = cov_exp_quad(x_b, alpha_b, rho_b) + diag_add I,  L_b = chol(K_b),  f_{b,m} = L_b z_{b,m}  (m < nvec)
 * x: per item n doubles, x_stride in doubles (0 = shared, else >= n); theta: B x 2 row-major (alpha, rho);
 * z, f: B*nvec vectors of length n, vector m of item b at offset (b*nvec + m)*n; info[B] as in
 * gpb200_lml_grad_batched (items with info != 0 get NaN in f; the others are unaffected).
 * The handle keeps a record of this call: the B factors and device copies of x, theta and z, so the caller may
 * overwrite its buffers before the backward call.  All B factors stay on the device (B * 8 * np^2 bytes, np = 128 *
 * ceil(n / 128)); when they do not fit the call fails.  A call that fails for any reason leaves no record.
 * gpb200_latent_backward_batched uses that record. */
GPB200_API int gpb200_latent_forward_batched(gpb200_handle_t h, int n, int B, int nvec, const double *x,
                                             long long x_stride, const double *theta, double diag_add,
                                             const double *z, double *f, int *info);
/* Reverse sweep of the batch recorded by the last gpb200_latent_forward_batched on this handle:
 * zbar_{b,m} = L_b^T fbar_{b,m};  theta_bar[b] = d lp / d (alpha_b, rho_b) through f and the Cholesky.
 * n, B, nvec must equal the record's (else, or with no record, a negative status and nothing is launched).
 * fbar and zbar use the layout of z; theta_bar is B x 2.  Items whose forward info != 0 get NaN.
 * The record is left unchanged, so backward may be called again.  The single-item gpb200_latent_forward / _backward
 * neither read nor change the record.  Both batched calls follow the pointer mode; in device-pointer mode neither
 * synchronises the host. */
GPB200_API int gpb200_latent_backward_batched(gpb200_handle_t h, int n, int B, int nvec, const double *fbar,
                                              double *theta_bar, double *zbar);

/* approx_L (covariance.cpp:49-96): cubic-Hermite interpolation in l between tabulated factors;
 * Ls / dLdls are P pointers to n x n column-major tables, lp the P grid points. */
GPB200_API int gpb200_approx_L(gpb200_handle_t h, int n, double l, int P, const double *lp,
                    const double *const *Ls, const double *const *dLdls, double *out);
/* approx_Lz (models/cubic_interpolated_gp.hpp:38-73): value v(l) z and partial dv/dl z */
GPB200_API int gpb200_approx_Lz(gpb200_handle_t h, int n, double l, int P, const double *lp,
                     const double *const *Ls, const double *const *dLdls, const double *z,
                     double *vz, double *dvdl_z);

/* ---- a10: conditioning --------------------------------------------------------------------- */
/* mu = Ks (K + noise_var I)^-1 y ; cov = Kss - Ks (K + noise_var I)^-1 Ks^T + jitter I
 * (pendulum_fit.R:242-251; R/ode_gp.R:27-31; gp_derivs.py:97-113).  K n x n symmetric,
 * Ks m x n, Kss m x m; mu length m, cov m x m.  Cholesky-based. */
GPB200_API int gpb200_gp_condition(gpb200_handle_t h, int n, int m, const double *K, int ldk,
                        const double *Ks, int ldks, const double *Kss, int ldkss, const double *y,
                        double noise_var, double jitter, double *mu, double *cov, int ldcov);

/* condMVN(mean, sigma, dependent = [nd..], given = [..], X.given) (R/ode_gp_library.R:17,32) for
 * the block layout the reference uses: sigma is (ng+nd)^2 with the GIVEN block first. */
GPB200_API int gpb200_cond_mvn(gpb200_handle_t h, int ng, int nd, const double *mean, const double *sigma,
                    int lds, const double *x_given, double *cond_mean, double *cond_var, int ldv);

/* ---- f-4: posterior sampling ------------------------------------------------------------------ */
/* out[e] = standard normal number (offset + e) of the stream `seed`, e in [0, len): counter-based
 * Philox4x32-10 -> 53-bit uniforms -> Box-Muller (pairs: offset must be even).  Stateless, so any
 * slice of a stream can be regenerated anywhere; replaces rnorm / numpy.random.randn on the host
 * (ch2.py:43-45). */
GPB200_API int gpb200_normal_fill(gpb200_handle_t h, unsigned long long seed, unsigned long long offset,
                                  long long len, double *out);
/* MASS::mvrnorm(n = ndraws, mu, Sigma) (pendulum_fit.R:253; lorenz.Rmd:105; `m + L z` of ch2.py:42-45):
 * out is ndraws x m column-major (R's return layout; ldo >= ndraws), row d = mu + L z_d with
 * L = chol(Sigma + jitter I) and z_d = normals [d*m, (d+1)*m) of gpb200_normal_fill(seed).  mu may be
 * NULL (zeros).  (MASS uses an eigen-decomposition square root; both give N(mu, Sigma) draws.) */
GPB200_API int gpb200_mvrnorm(gpb200_handle_t h, int ndraws, int m, const double *mu, const double *Sigma, int lds,
                              double jitter, unsigned long long seed, double *out, int ldo);
/* B posterior draws, one per hyper-parameter draw theta_b = (alpha, rho, sigma), in one call that stays on the
 * device: the loop of pendulum_fit.R:259-268 over sample_derivs (:227-255: three Grams, conditioning, one
 * mvrnorm draw) and of lorenz.Rmd:58-68,80-107 (separate prediction grid, 1e-6 jitter).  For item b
 *   K   = alpha^2 QQ(t, t) + sigma^2 I          n x n   (training grid t, observations y)
 *   Ks  = alpha^2 k_{p,0}(s, t)                  m x n   (covariance of f^(p)(s_i) with f(t_j))
 *   Kss = alpha^2 k_{p,p}(s, s)                  m x m
 *   mu  = Ks K^-1 y,   cov = Kss - Ks K^-1 Ks^T + jitter I,   draw_b = mu + chol(cov) eps_b
 * with k_{p,q} the kernels of derivative_kernels.R:39-73 and derivative order p = `order` in {0, 1, 2}:
 * (QQ, QQ) as in ch2.py:36-45, (RQ, RR) as in pendulum_fit.R:238-240, (TQ, TT) as in gp_derivs.py on tts.
 * s == NULL predicts on t (then m == n).  t, s, y: B strides in doubles (0 = shared; s == NULL takes t's);
 * theta: B x 3 row-major.  eps_b = z + b*m when z != NULL, else the standard normals [b*m, (b+1)*m) of
 * gpb200_normal_fill(seed) (B = 1: the normals of gpb200_mvrnorm(1, ..., seed)).  Outputs: draws[B*m] (column b
 * = draw b), mu[B*m] (may be NULL), info[B]: 0 ok; k in 1..n: K is not positive definite at pivot k; n + k: cov is
 * not positive definite at pivot k.  Items with info != 0 get NaN in draws and mu; the others are unaffected.
 * Computed from one Cholesky factorisation of the joint (n+m)^2 prior covariance of (y, f^(p)(s)) per item. */
GPB200_API int gpb200_posterior_draws_batched(gpb200_handle_t h, int n, int m, int order, int B, const double *t,
                                              long long t_stride, const double *s, long long s_stride, const double *y,
                                              long long y_stride, const double *theta, double jitter, const double *z,
                                              unsigned long long seed, double *draws, double *mu, int *info);
/* The same B posterior draws for the ARD squared-exponential kernel (QQard, R/kernels.R:19) on D-column inputs,
 * 1 <= D <= 8 (the states of create_p_dotXnS, R/ode_gp_library.R:43-93).  For item b, with
 * k(p, q) = alpha^2 exp(-0.5 sum_d (p_d - q_d)^2 / rho_d^2):
 *   K = k(X, X) + sigma^2 I  (n x n),  Ks = k(Xs, X)  (m x n),  Kss = k(Xs, Xs)  (m x m)
 *   mu = Ks K^-1 y,   cov = Kss - Ks K^-1 Ks^T + jitter I,   draw_b = mu + chol(cov) eps_b
 * X: per item n x D column-major with leading dimension n (an R matrix); Xs: per item m x D with leading dimension m;
 * x_stride / xs_stride in doubles between items (0 = shared, else >= n*D / m*D); Xs == NULL predicts on X (then
 * m == n).  theta: B x (D + 2) row-major, (alpha, rho_1 .. rho_D, sigma) as in gpb200_lml_grad_ard_batched.  y, z,
 * seed, draws, mu and info as in gpb200_posterior_draws_batched.  At D = 1 this is its order-0 model. */
GPB200_API int gpb200_posterior_draws_ard_batched(gpb200_handle_t h, int n, int m, int D, int B, const double *X,
                                                  long long x_stride, const double *Xs, long long xs_stride,
                                                  const double *y, long long y_stride, const double *theta, double jitter,
                                                  const double *z, unsigned long long seed, double *draws, double *mu,
                                                  int *info);

/* ---- (e) multi-GPU block-cyclic Cholesky of ONE large matrix: per-rank building blocks ------------
 * DEVICE pointers only.  A panel is a block column of the padded matrix (np = ceil(n/128)*128)
 * stored compactly: rows [col0, np) x ncols columns, leading dimension ldp >= np - col0 (even);
 * col0 and ncols are multiples of 128.  Panels are distributed block-column-cyclically over the
 * GPUs of one box; the panel broadcast between these calls is an NCCL collective issued by the host
 * side (gp_b200/block_cyclic.py, torch.distributed).  The reference has no counterpart (SURVEY 2.2):
 * the semantics are those of cholesky_decompose / multi_normal_cholesky at sizes one GPU's time
 * budget does not allow. */
GPB200_API int gpb200_mg_gram_panel(gpb200_handle_t h, int n, const double *x, double alpha, double rho,
                                    double diag_add, int col0, int ncols, double *P, long long ldp);
/* Cholesky of the (already updated) panel in place: diagonal block + everything below it */
GPB200_API int gpb200_mg_panel_factor(gpb200_handle_t h, int n, int col0, int ncols, double *P, long long ldp,
                                      int *info_dev);
/* the same, one 128-wide tile column at a time (jl = 0 .. ncols/128 - 1, in order), so that a finished tile column
 * can travel (gpb200_mg_bcast of its ldp * 128 doubles) while the next one is being factored */
GPB200_API int gpb200_mg_panel_factor_col(gpb200_handle_t h, int n, int col0, int ncols, double *P, long long ldp, int jl,
                                          int *info_dev);
/* right-looking update of a panel to the right: C -= P(rows of C) P(cols of C)^T, lower part */
GPB200_API int gpb200_mg_panel_update(gpb200_handle_t h, int n, int pcol0, int pncols, const double *P,
                                      long long ldp, int ccol0, int cncols, double *C, long long ldc);
/* the same restricted to tile columns [jl0, jl1) of the target panel */
GPB200_API int gpb200_mg_panel_update_cols(gpb200_handle_t h, int n, int pcol0, int pncols, const double *P,
                                           long long ldp, int ccol0, int cncols, double *C, long long ldc, int jl0,
                                           int jl1);
/* forward substitution through a factored panel: z[col0..] solved, acc[below] += L z;
 * y, acc, z: length-np device vectors; wscratch: ldp x 128 doubles */
GPB200_API int gpb200_mg_panel_trsv(gpb200_handle_t h, int n, int col0, int ncols, const double *P,
                                    long long ldp, const double *y, double *acc, double *z, double *wscratch);
/* out[0] += sum of log L_ii over the panel's diagonal (device scalar) */
GPB200_API int gpb200_mg_panel_logdiag(gpb200_handle_t h, int n, int col0, int ncols, const double *P,
                                       long long ldp, double *out);


/* ---- (e) collectives of config 5, enqueued from C.  NCCL is loaded at run time (the copy the host process
 * already carries, e.g. torch's, else the system libnccl.so.2; GPB200_NCCL_LIB overrides).  The communicator lives in
 * the handle: rank 0 draws the 128-byte unique id, the caller ships it to the other ranks by whatever means it has
 * (torch.distributed, MPI, a file), every rank calls comm_init.  gpb200_mg_bcast runs ncclBroadcast on the handle's
 * own communication stream, ordered behind the compute stream by an event, and returns a ticket; gpb200_mg_wait makes
 * the compute stream wait for that ticket -- so a panel travels over NVLink while the trailing update runs. */
GPB200_API int gpb200_mg_comm_id(gpb200_handle_t h, void *id128);
GPB200_API int gpb200_mg_comm_init(gpb200_handle_t h, const void *id128, int rank, int world);
GPB200_API int gpb200_mg_comm_destroy(gpb200_handle_t h);
GPB200_API int gpb200_mg_bcast(gpb200_handle_t h, double *buf, long long count, int root, long long *ticket);
GPB200_API int gpb200_mg_wait(gpb200_handle_t h, long long ticket);
/* in-place all-reduce on the compute stream: op 0 sum, 1 max; is_int != 0 for int32 data */
GPB200_API int gpb200_mg_allreduce(gpb200_handle_t h, void *buf, long long count, int op, int is_int);

/* ---- (e) distributed GRADIENT of config 5: per-rank building blocks without communication (DEVICE pointers).
 * Every rank holds the whole factor after the factorisation (its panels and the broadcast copies).  Rank r computes
 * the columns of X = L^-T of ITS panels (= its rows of L^-1; N^3/3P flops), z_k = x_k^T y for its k, a_r = X_r z_r, and
 * feeds G_r = X_r X_r^T tile by tile to the fused trace epilogue (N^3/3P flops): since tr(K^-1 dK) = sum_k w_k dK w_k^T
 * over the rows w_k of L^-1, the partial sums of the ranks add up to the single-GPU result exactly.
 *   Lsq np x np (ld np): full lower factor; Xp np x nmine (ld np): the rank's columns of X, packed;
 *   S pc x nmine and Wd 2 * npanels * pc * pc doubles: scratch; nmine = gpb200_mg_my_columns(...). */
GPB200_API int gpb200_mg_panel_to_square(gpb200_handle_t h, int n, int col0, int ncols, const double *P, long long ldp, double *Lsq);
GPB200_API long long gpb200_mg_my_columns(int n, int pc, int rank, int world);
GPB200_API int gpb200_mg_inverse_rows(gpb200_handle_t h, int n, int pc, int rank, int world, const double *Lsq, double *Xp,
                                      double *S, double *Wd);
/* z_mine = X_r^T y, sums2 = (sum z_mine^2, log det L), a_part = X_r z_mine; ypad = y padded with zeros to np; part: 8 np scratch */
GPB200_API int gpb200_mg_solve_partials(gpb200_handle_t h, int n, int pc, int rank, int world, const double *Lsq, const double *Xp,
                                        const double *ypad, double *z_mine, double *a_part, double *sums2, double *part);
/* sums3 = (sum M e, sum M e d^2, tr G_r) over the tiles this rank's columns reach, M = avec avec^T - G_r.  Pass a ZERO
 * avec for the distributed gradient (the a a^T half comes from gpb200_mg_quadform_partials, which covers every tile);
 * theta3 = device (alpha, rho, sigma); partial: 16 * nt (nt + 1) / 2 doubles of scratch, nt = np / 128 */
GPB200_API int gpb200_mg_trace_partials(gpb200_handle_t h, int n, int pc, int rank, int world, const double *Xp, const double *x,
                                        const double *avec, const double *theta3, double *partial, double *sums3);
/* sums2 = (a^T E a, a^T (E o D^2) a) over this rank's contiguous share of the rows, E_ij = exp(-(x_i - x_j)^2 / 2 rho^2);
 * part: 2 * ceil(n / 128) doubles of scratch */
GPB200_API int gpb200_mg_quadform_partials(gpb200_handle_t h, int n, int rank, int world, const double *x, const double *a,
                                           const double *theta3, double *part, double *sums2);

#ifdef __cplusplus
}
#endif
#endif /* GPB200_H */
