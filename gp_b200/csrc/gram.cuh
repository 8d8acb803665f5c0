// Kernel-kind ids (match include/gpb200.h) and launchers of gram.cu / solve.cu.
#pragma once
#include "common.cuh"

namespace gpb {

enum { K_QQ = 0, K_QR = 1, K_RQ = 2, K_RR = 3, K_QT = 4, K_TQ = 5, K_RT = 6, K_TR = 7, K_TT = 8, K_RR_QUIRK = 9 };

int launch_kernel_eval(Handle *h, int kind, long long len, const double *tj, const double *tk, double amp2,
                       double l, double *out);
int launch_gram_outer(Handle *h, int kind, int n, int m, const double *x, const double *y, double amp2, double l,
                      double *K, long long ldk);
int launch_gram_se_batched(Handle *h, int n, int np, const double *x, long long x_stride, const double *theta,
                           double jitter, int lower_only, double *K, long long stride, int batch, int *envF = nullptr);
int launch_gram_tangent(Handle *h, int n, int np, const double *x, double alpha, const double *ls, double dadd, int mode,
                        double *S, double *Sdot, long long stride, int batch);
int launch_gram_deriv(Handle *h, int n, int nblocks, const double *t, double alpha, double rho, const double *noise,
                      double jitter, int quirk, double *K, long long ldk);
int launch_gram_deriv_batched(Handle *h, int n, int order0, int nblocks, int np, const double *t, long long t_stride,
                              const double *theta, int theta_stride, double jitter, int lower_only, double *K,
                              long long stride, int batch);
int launch_gram_cond_batched(Handle *h, int n, int m, int order, int np, const double *t, long long t_stride,
                             const double *s, long long s_stride, const double *theta, double jitter, double *K,
                             long long stride, int batch);
int launch_gram_ard(Handle *h, int n, int m, int D, const double *X, long long ldx, const double *Y, long long ldy,
                    double alpha, const double *rho, int rho_len, double *K, long long ldk);

int launch_approx_basis(Handle *h, int n, int M, double scale, const double *x, double sigma, double l, double *out,
                        long long ldo);

// solve.cu
int launch_trmv_lower_n(Handle *h, int np, const double *W, long long stride, const double *y, long long y_stride,
                        int n_valid, double *z, long long z_stride, int batch);
int trmv_split_chunks(int np, int batch);
int launch_trmv_lower_n_split(Handle *h, int np, int ks, const double *W, long long stride, const double *y, long long y_stride,
                              int n_valid, double *part, double *z, long long z_stride, int batch);
int launch_trmv_lower_t(Handle *h, int np, const double *W, long long stride, const double *z, long long z_stride,
                        double *a, long long a_stride, int batch);
int launch_trsv_blocked(Handle *h, int np, const double *L, const double *Wdiag, long long stride, const double *y,
                        long long y_stride, const double *mu, int n_valid, double *z, long long z_stride, int batch,
                        const int *env = nullptr);
int launch_trsv_diag(Handle *h, long long ldw, long long w_off, int row0, const double *Wdiag, long long stride,
                     const double *y, long long y_stride, const double *mu, int n_valid, const double *acc, double *z,
                     long long z_stride, int batch);
int launch_trsv_update(Handle *h, long long ld, long long l_off, int z_row0, int acc_row0, int ntiles, const double *L,
                       long long stride, const double *z, double *acc, long long z_stride, int batch);
int launch_gram_se_panel(Handle *h, int n, int np, const double *x, double alpha, double rho, double diag_add,
                         int col0, int ncols, double *P, long long ldp);
int launch_trsv_sweep(Handle *h, int np, const double *L, const double *Wdiag, long long stride, const double *y,
                      long long y_stride, const double *mu, int n_valid, double *z, double *acc, long long z_stride,
                      int batch);
int launch_finalize(Handle *h, int n, int np, int want_grad, const double *dvec, const double *z, const double *a,
                    const double *partial, int ntasks, int ntasks2, const double *theta, double *lml, double *grad, int batch);
int launch_finalize_deriv(Handle *h, int n_grid, int nblocks, int np, int want_grad, const double *dvec, const double *z,
                          const double *a, const double *partial, int ntasks, int ntasks2, const double *theta, double *lml,
                          double *grad, int batch);
int launch_pack(Handle *h, int rows, int cols, const double *src, long long lds, int rp, int cp, double *dst,
                int mode, double diag_add);
int launch_unpack(Handle *h, int rows, int cols, const double *src, long long lds_src, double *dst, long long ldd,
                  int mode, double diag_add);
int launch_phi_lower(Handle *h, int np, double *A, long long stride, int batch);
int launch_gemv_t(Handle *h, int rows, int cols, const double *V, long long ldv, const double *z, const double *add,
                  double *out);
int launch_hermite(Handle *h, long long len, int n, const double *y1, const double *y2, const double *k1,
                   const double *k2, double x1, double x2, double l, double *v, double *dvdl);
int hermite_matvec_chunks(int n);
int launch_hermite_matvec(Handle *h, int n, const double *y1, const double *y2, const double *k1, const double *k2, double x1,
                          double x2, double l, const double *z, double *part, double *vz, double *dvz);
int launch_sumsq_logdiag(Handle *h, int n, const double *z, const double *L, long long ldl, double *out2);

// small.cu
int small_smem_setup(Handle *h);
bool lml_small_applies(const Handle *h, int n);
int launch_lml_small(Handle *h, int n, const double *x, long long x_stride, const double *y, long long y_stride,
                     const double *theta, double jitter, int want_grad, double *lml, double *grad, int *info, int batch);

// rng.cu
int launch_normal_fill(Handle *h, unsigned long long seed, unsigned long long offset, long long len, long long rows,
                       long long ld, double *out);
int launch_add_mean_transpose(Handle *h, int m, int ndraws, const double *X, long long ldx, const double *mu,
                              double *out, long long ldo);
int launch_rows_or_nan(Handle *h, int row0, int rows, const double *src, long long src_stride, const int *info,
                       double *dst, int batch);

}  // namespace gpb
