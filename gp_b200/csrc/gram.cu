// Covariance (Gram) assembly kernels for sm_100a: coalesced 16-byte stores, inputs staged in shared
// memory, noise/jitter diagonal fused.  HBM-write bound when K is materialised (8 N^2 bytes).
//
// Reference semantics restated here (not copied):
//   cov_exp_quad + diagonal add     models/fit_hyperparameters.stan:19-24, exact_gp.stan:17-22
//   rbf Gram and its l-tangent      covariance.cpp:15-25 (value) and the fvar tangent it seeds (:13)
//   nine derivative kernels         derivative_kernels.R:39-73 ; R/kernels.R:19-32 (incl. the :31 quirk)
//   joint (y, y', y'') covariance   design_notes.Rmd:6-46 ; R/ode_gp_library.R:29-30
#include "common.cuh"
#include "fastexp.cuh"
#include "gram.cuh"

namespace gpb {

// value of one derivative kernel; operation order follows derivative_kernels.R:39-73
__device__ __forceinline__ double kern_value(int kind, double tj, double tk, double l, double amp2) {
  double d;
  int base = kind;
  if (kind == K_RQ) { d = tk - tj; base = K_QR; }
  else if (kind == K_TQ) { d = tk - tj; base = K_QT; }
  else if (kind == K_TR) { d = tk - tj; base = K_RT; }
  else d = tj - tk;
  const double l2 = l * l;
  const double e = exp(-((d * d) / (2.0 * l2)));
  const double l4 = l2 * l2;
  switch (base) {
    case K_QQ: return amp2 * e;
    case K_QR: return amp2 * ((e * d) / l2);
    case K_RR: return amp2 * (e / l2 - (e * d * d) / l4);
    case K_RR_QUIRK: return amp2 * e / l2 - (e * d * d) / l4;  // R/kernels.R:31
    case K_QT: return amp2 * (-(e / l2) + (e * d * d) / l4);
    case K_RT: { const double l6 = l4 * l2; return amp2 * ((3.0 * e * d) / l4 - (e * d * d * d) / l6); }
    case K_TT: { const double l6 = l4 * l2, l8 = l4 * l4;
                 return amp2 * ((3.0 * e) / l4 - (6.0 * e * d * d) / l6 + (e * d * d * d * d) / l8); }
    default: return 0.0;
  }
}

// ---- element-wise evaluation (the R closures) ------------------------------------------------
__global__ void kernel_eval_kernel(int kind, long long len, const double *__restrict__ tj,
                                   const double *__restrict__ tk, double amp2, double l, double *__restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < len; i += (long long)gridDim.x * blockDim.x)
    out[i] = kern_value(kind, tj[i], tk[i], l, amp2);
}

// ---- generic outer(x, y, kind): n x m, tile 128x128 per CTA, two rows per thread -------------
__global__ void __launch_bounds__(256) gram_outer_kernel(int kind, int n, int m, const double *__restrict__ x,
                                                        const double *__restrict__ y, double amp2, double l,
                                                        double *__restrict__ K, long long ldk) {
  __shared__ double xs[TILE], ys[TILE];
  const int r0 = blockIdx.x * TILE, c0 = blockIdx.y * TILE, tid = threadIdx.x;
  if (tid < TILE) xs[tid] = (r0 + tid < n) ? x[r0 + tid] : 0.0;
  else ys[tid - TILE] = (c0 + tid - TILE < m) ? y[c0 + tid - TILE] : 0.0;
  __syncthreads();
  const int rl = 2 * (tid & 63), cq = tid >> 6;
  const int i = r0 + rl;
  const bool vec_ok = ((ldk & 1) == 0) && ((reinterpret_cast<uintptr_t>(K) & 15) == 0);
  for (int s = 0; s < 32; s++) {
    const int cl = cq + 4 * s, j = c0 + cl;
    if (j >= m) break;
    const double v0 = kern_value(kind, xs[rl], ys[cl], l, amp2);
    const double v1 = kern_value(kind, xs[rl + 1], ys[cl], l, amp2);
    double *dst = K + i + (long long)j * ldk;
    if (i + 1 < n && vec_ok) *reinterpret_cast<double2 *>(dst) = make_double2(v0, v1);
    else {
      if (i < n) dst[0] = v0;
      if (i + 1 < n) dst[1] = v1;
    }
  }
}

// ---- batched padded SE Gram for the fused LML path: K = alpha^2 exp(-0.5 d^2/rho^2) + c I -------
// Internal layout: np x np (np multiple of 128) per item, identity in the padding so that the
// padded factor is [L 0; 0 I].  Only tiles with tile_row >= tile_col are produced when lower_only.
// RAGGED: item b has its own size nvec[b] <= np (gpb200_lml_grad_ragged), identity beyond it.
// Element profile for the envelope record (common.cuh, ENV_BLK) of item b: fcol / lrow are the first nonzero column
// and the last nonzero row among this thread's elements of tile (tr, tc) (INT_MAX / -1: none).  Warp w holds the rows of
// 64-row block (w & 1) of the tile row (rl = 2 (tid & 63)).
__device__ __forceinline__ void record_profile(int *rec, int nt, int tr, int tc, int fcol, int lrow) {
  const unsigned fw = __reduce_min_sync(0xffffffffu, (unsigned)fcol);
  const int lw = __reduce_max_sync(0xffffffffu, lrow);
  if ((threadIdx.x & 31) == 0) {
    if (fw != (unsigned)INT_MAX) atomicMin(reinterpret_cast<unsigned *>(rec + 2 * nt) + 2 * tr + ((threadIdx.x >> 5) & 1), fw);
    if (lw >= 0) atomicMax(rec + 4 * nt + tc, lw);
  }
}

template <bool RAGGED>
__global__ void __launch_bounds__(256) gram_se_batched_kernel(int n_all, int np, const double *__restrict__ x,
                                                             long long x_stride, const double *__restrict__ theta,
                                                             double jitter, int lower_only,
                                                             double *__restrict__ K, long long stride,
                                                             int *__restrict__ env, const int *__restrict__ nvec) {
  const int nt = np / TILE;
  const int tr = blockIdx.x % nt, tc = blockIdx.x / nt;
  if (lower_only && tr < tc) return;
  const int n = RAGGED ? nvec[blockIdx.y] : n_all;
  // env (optional, records of env_record_ints(nt) ints, fb preset to UINT_MAX and er to -1): the element profile of the
  // tile, where an element is nonzero when its exp(-d^2/2rho^2) is not exactly zero (NaN counts) or it is on the
  // diagonal.  That set holds the support of K and of dK/dtheta, and the diagonal of the identity padding.
  __shared__ double xs[TILE], ys[TILE];
  const long long b = blockIdx.y;
  const double *xb = x + b * x_stride;
  const int r0 = tr * TILE, c0 = tc * TILE, tid = threadIdx.x;
  if (tid < TILE) xs[tid] = (r0 + tid < n) ? xb[r0 + tid] : 0.0;
  else ys[tid - TILE] = (c0 + tid - TILE < n) ? xb[c0 + tid - TILE] : 0.0;
  __syncthreads();
  const double alpha = theta[b * 3 + 0], rho = theta[b * 3 + 1], sigma = theta[b * 3 + 2];
  const double a2 = alpha * alpha, nh = -0.5 / (rho * rho), dadd = sigma * sigma + jitter;
  double *Kb = K + b * stride;
  const int rl = 2 * (tid & 63), cq = tid >> 6;
  int fcol = INT_MAX, lrow = -1;
  if (tr != tc && r0 + TILE <= n && c0 + TILE <= n) {
    // interior off-diagonal tile (all but O(nt) of the nt^2/2 tiles): no masks, no diagonal
    const double x0 = xs[rl], x1 = xs[rl + 1];
    double *dst = Kb + (r0 + rl) + (long long)(c0 + cq) * np;
    int s0 = 32;  // the first column step with a nonzero
    bool nz0 = false, nz1 = false;
#pragma unroll 4
    for (int s = 0; s < 32; s++) {
      const double yc = ys[cq + 4 * s];
      const double d0 = x0 - yc, d1 = x1 - yc;
      const double e0 = exp_nonpos(d0 * d0 * nh), e1 = exp_nonpos(d1 * d1 * nh);
      nz0 |= e0 != 0.0;
      nz1 |= e1 != 0.0;
      s0 = min(s0, (e0 != 0.0 || e1 != 0.0) ? s : 32);
      *reinterpret_cast<double2 *>(dst) = make_double2(a2 * e0, a2 * e1);
      dst += 4LL * np;
    }
    if (env) {
      if (s0 < 32) fcol = c0 + cq + 4 * s0;
      lrow = nz1 ? r0 + rl + 1 : (nz0 ? r0 + rl : -1);
      record_profile(env + b * env_record_ints(nt), nt, tr, tc, fcol, lrow);
    }
    return;
  }
#pragma unroll 2
  for (int s = 0; s < 32; s++) {
    const int cl = cq + 4 * s;
    const int j = c0 + cl;
    double v[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int i = r0 + rl + e;
      bool nz = i == j;
      if (i < n && j < n) {
        const double d = xs[rl + e] - ys[cl];
        const double ek = exp_nonpos(d * d * nh);
        nz |= ek != 0.0;
        v[e] = (i == j) ? a2 + dadd : a2 * ek;
      } else {
        v[e] = (i == j) ? 1.0 : 0.0;
      }
      if (nz) {
        fcol = min(fcol, j);
        lrow = max(lrow, i);
      }
    }
    *reinterpret_cast<double2 *>(Kb + (r0 + rl) + (long long)j * np) = make_double2(v[0], v[1]);
  }
  if (env) record_profile(env + b * env_record_ints(nt), nt, tr, tc, fcol, lrow);
}

// ---- block-column panel of the padded SE Gram for the block-cyclic multi-GPU Cholesky ----------
// P holds rows [col0, np) x columns [col0, col0+ncols) compactly (leading dimension ldp = np - col0);
// tiles strictly above the diagonal are skipped.  x is replicated on every GPU: no K scatter.
__global__ void __launch_bounds__(256) gram_se_panel_kernel(int n, int np, const double *__restrict__ x, double alpha,
                                                           double rho, double dadd, int col0, double *__restrict__ P,
                                                           long long ldp) {
  const int r0 = col0 + blockIdx.x * TILE, c0 = col0 + blockIdx.y * TILE;
  if (r0 < c0) return;
  __shared__ double xs[TILE], ys[TILE];
  const int tid = threadIdx.x;
  if (tid < TILE) xs[tid] = (r0 + tid < n) ? x[r0 + tid] : 0.0;
  else ys[tid - TILE] = (c0 + tid - TILE < n) ? x[c0 + tid - TILE] : 0.0;
  __syncthreads();
  const double a2 = alpha * alpha, nh = -0.5 / (rho * rho);
  const int rl = 2 * (tid & 63), cq = tid >> 6;
#pragma unroll 4
  for (int s = 0; s < 32; s++) {
    const int cl = cq + 4 * s;
    const int j = c0 + cl;
    double v[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int i = r0 + rl + e;
      if (i < n && j < n) {
        const double d = xs[rl + e] - ys[cl];
        v[e] = (i == j) ? a2 + dadd : a2 * exp_nonpos(d * d * nh);
      } else {
        v[e] = (i == j) ? 1.0 : 0.0;
      }
    }
    *reinterpret_cast<double2 *>(P + (r0 - col0 + rl) + (long long)(j - col0) * ldp) = make_double2(v[0], v[1]);
  }
}

// ---- Gram + parameter tangent for the forward-mode Cholesky: padded, full square ----------------
// mode 0: rbf_cov_chol literal (covariance.cpp:15-25): S = exp(-d^2/(2 l^2)) + jitter I, dS/dl
// mode 1: cov_exp_quad form, tangent w.r.t. rho:   S = alpha^2 exp(-0.5 d^2/rho^2) + c I, dS/drho = S_se d^2/rho^3
// mode 2: cov_exp_quad form, tangent w.r.t. alpha: dS/dalpha = 2 alpha exp(-0.5 d^2/rho^2)
__global__ void __launch_bounds__(256) gram_tangent_kernel(int n, int np, const double *__restrict__ x, double alpha,
                                                          const double *__restrict__ ls, double dadd, int mode,
                                                          double *__restrict__ S, double *__restrict__ Sdot,
                                                          long long stride) {
  const double l = ls[blockIdx.z];
  S += (long long)blockIdx.z * stride;
  Sdot += (long long)blockIdx.z * stride;
  __shared__ double xs[TILE], ys[TILE];
  const int r0 = blockIdx.x * TILE, c0 = blockIdx.y * TILE, tid = threadIdx.x;
  if (tid < TILE) xs[tid] = (r0 + tid < n) ? x[r0 + tid] : 0.0;
  else ys[tid - TILE] = (c0 + tid - TILE < n) ? x[c0 + tid - TILE] : 0.0;
  __syncthreads();
  const double two_l2 = 2.0 * l * l, l3 = l * l * l, a2 = alpha * alpha, nh = -0.5 / (l * l);
  const int rl = 2 * (tid & 63), cq = tid >> 6;
  for (int s = 0; s < 32; s++) {
    const int cl = cq + 4 * s, j = c0 + cl;
    double v[2], dv[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int i = r0 + rl + e;
      if (i < n && j < n) {
        const double d = xs[rl + e] - ys[cl];
        if (mode == 0) {
          const double ev = exp(-(d * d) / two_l2);
          v[e] = ev + ((i == j) ? dadd : 0.0);
          dv[e] = ev * d * d / l3;
        } else {
          const double ev = (i == j) ? 1.0 : exp(d * d * nh);
          v[e] = a2 * ev + ((i == j) ? dadd : 0.0);
          dv[e] = (mode == 1) ? a2 * ev * d * d / l3 : 2.0 * alpha * ev;
        }
      } else {
        v[e] = (i == j) ? 1.0 : 0.0;
        dv[e] = 0.0;
      }
    }
    *reinterpret_cast<double2 *>(S + (r0 + rl) + (long long)j * np) = make_double2(v[0], v[1]);
    *reinterpret_cast<double2 *>(Sdot + (r0 + rl) + (long long)j * np) = make_double2(dv[0], dv[1]);
  }
}

// ---- joint derivative-observation covariance ---------------------------------------------------
__constant__ int c_joint_kind[3][3] = {{K_QQ, K_QR, K_QT}, {K_RQ, K_RR, K_RT}, {K_TQ, K_TR, K_TT}};

__global__ void __launch_bounds__(256) gram_deriv_kernel(int n, int nblocks, const double *__restrict__ t, double alpha,
                                                        double rho, double n0, double n1, double n2, double jitter,
                                                        int quirk, double *__restrict__ K, long long ldk) {
  const int N = n * nblocks;
  const int r0 = blockIdx.x * TILE, c0 = blockIdx.y * TILE, tid = threadIdx.x;
  const double amp2 = alpha * alpha;
  const double noise2[3] = {n0 * n0, n1 * n1, n2 * n2};
  const int rl = tid & 127, ch = tid >> 7;
  const int I = r0 + rl;
  if (I >= N) return;
  const int bi = I / n, i = I - bi * n;
  const double ti = t[i];
  for (int s = 0; s < 64; s++) {
    const int J = c0 + ch + 2 * s;
    if (J >= N) break;
    const int bj = J / n, j = J - bj * n;
    int kind = c_joint_kind[bi][bj];
    if (quirk && kind == K_RR) kind = K_RR_QUIRK;
    double v = kern_value(kind, ti, t[j], rho, amp2);
    if (I == J) v += noise2[bi] + jitter;
    K[I + (long long)J * ldk] = v;
  }
}

// Batched padded form of the same matrix for the fused LML path: derivative orders order0 .. order0 +
// nblocks - 1 of one grid t (n points) per item; theta = (alpha, rho, noise[nblocks]) per item; identity
// in the padding; only tiles with tile_row >= tile_col when lower_only.  Element values come from the
// same kern_value as gram_deriv_kernel, so both produce identical bits.
__global__ void __launch_bounds__(256) gram_deriv_batched_kernel(int n, int order0, int nblocks, int np,
                                                                const double *__restrict__ t, long long t_stride,
                                                                const double *__restrict__ theta, int theta_stride,
                                                                double jitter, int lower_only,
                                                                double *__restrict__ K, long long stride) {
  const int nt = np / TILE;
  const int tr = blockIdx.x % nt, tc = blockIdx.x / nt;
  if (lower_only && tr < tc) return;
  __shared__ double xs[TILE], ys[TILE];
  __shared__ int bxs[TILE], bys[TILE];
  const long long b = blockIdx.y;
  const double *tb = t + b * t_stride;
  const int N = n * nblocks;
  const int r0 = tr * TILE, c0 = tc * TILE, tid = threadIdx.x;
  {
    const int I = (tid < TILE) ? r0 + tid : c0 + tid - TILE;
    const int blk = (I < N) ? I / n : 0;
    const double v = (I < N) ? tb[I - blk * n] : 0.0;
    if (tid < TILE) { xs[tid] = v; bxs[tid] = blk; }
    else { ys[tid - TILE] = v; bys[tid - TILE] = blk; }
  }
  __syncthreads();
  const double *th = theta + b * theta_stride;
  const double alpha = th[0], rho = th[1];
  const double amp2 = alpha * alpha;
  double *Kb = K + b * stride;
  const int rl = 2 * (tid & 63), cq = tid >> 6;
  for (int s = 0; s < 32; s++) {
    const int cl = cq + 4 * s;
    const int J = c0 + cl;
    double v[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int I = r0 + rl + e;
      if (I < N && J < N) {
        const int bi = bxs[rl + e], bj = bys[cl];
        v[e] = kern_value(c_joint_kind[order0 + bi][order0 + bj], xs[rl + e], ys[cl], rho, amp2);
        if (I == J) { const double nz = th[2 + bi]; v[e] += nz * nz + jitter; }
      } else {
        v[e] = (I == J) ? 1.0 : 0.0;
      }
    }
    *reinterpret_cast<double2 *>(Kb + (r0 + rl) + (long long)J * np) = make_double2(v[0], v[1]);
  }
}

// Joint prior covariance of the noisy values f(t) + noise and the derivative f^(p)(s) of a GP, for
// conditioning and drawing in one factorisation (gpb200_posterior_draws_batched):
//   J = [[alpha^2 QQ(t, t) + sigma^2 I,  .                          ],
//        [alpha^2 k_{p,0}(s, t),        alpha^2 k_{p,p}(s, s) + jitter I]]
// rows [0, n) from t, rows [n, n+m) from s; padded np x np per item with identity in the padding, lower tiles only.
// Lower-triangle elements come from kern_value / c_joint_kind exactly as gram_outer evaluates them (row point first);
// the strict upper part of a diagonal tile mirrors them.  theta = (alpha, rho, sigma) per item.
__global__ void __launch_bounds__(256) gram_cond_batched_kernel(int n, int m, int order, int np,
                                                               const double *__restrict__ t, long long t_stride,
                                                               const double *__restrict__ s, long long s_stride,
                                                               const double *__restrict__ theta, double jitter,
                                                               double *__restrict__ K, long long stride) {
  const int nt = np / TILE;
  const int tr = blockIdx.x % nt, tc = blockIdx.x / nt;
  if (tr < tc) return;
  __shared__ double xs[TILE], ys[TILE];
  const long long b = blockIdx.y;
  const double *tb = t + b * t_stride, *sb = s + b * s_stride;
  const int N = n + m;
  const int r0 = tr * TILE, c0 = tc * TILE, tid = threadIdx.x;
  {
    const int I = (tid < TILE) ? r0 + tid : c0 + tid - TILE;
    const double v = (I < n) ? tb[I] : (I < N) ? sb[I - n] : 0.0;
    if (tid < TILE) xs[tid] = v;
    else ys[tid - TILE] = v;
  }
  __syncthreads();
  const double alpha = theta[b * 3 + 0], rho = theta[b * 3 + 1], sigma = theta[b * 3 + 2];
  const double amp2 = alpha * alpha;
  double *Kb = K + b * stride;
  const int rl = 2 * (tid & 63), cq = tid >> 6;
  for (int q = 0; q < 32; q++) {
    const int cl = cq + 4 * q;
    const int J = c0 + cl;
    double v[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int I = r0 + rl + e;
      if (I < N && J < N) {
        const bool up = I < J;  // only inside a diagonal tile
        const int Ir = up ? J : I, Jc = up ? I : J;
        const double xr = up ? ys[cl] : xs[rl + e], xc = up ? xs[rl + e] : ys[cl];
        v[e] = kern_value(c_joint_kind[Ir < n ? 0 : order][Jc < n ? 0 : order], xr, xc, rho, amp2);
        if (I == J) v[e] += (I < n) ? sigma * sigma : jitter;
      } else {
        v[e] = (I == J) ? 1.0 : 0.0;
      }
    }
    *reinterpret_cast<double2 *>(Kb + (r0 + rl) + (long long)J * np) = make_double2(v[0], v[1]);
  }
}

// ---- QQard (R/kernels.R:19) ---------------------------------------------------------------------
__global__ void __launch_bounds__(256) gram_ard_kernel(int n, int m, int D, const double *__restrict__ X, long long ldx,
                                                      const double *__restrict__ Y, long long ldy, double alpha,
                                                      const double *__restrict__ rho, int rho_len,
                                                      double *__restrict__ K, long long ldk) {
  const int i = blockIdx.x * 128 + (threadIdx.x & 127);
  const int jh = threadIdx.x >> 7;
  if (i >= n) return;
  const double a2 = alpha * alpha;
  for (int j = blockIdx.y * 64 + jh; j < min(m, (int)(blockIdx.y + 1) * 64); j += 2) {
    double s = 0.0;
    for (int d = 0; d < D; d++) {
      const double q = (X[i + d * ldx] - Y[j + d * ldy]) / rho[rho_len == 1 ? 0 : d];
      s += q * q;
    }
    K[i + (long long)j * ldk] = a2 * exp(-0.5 * s);
  }
}

// ---- batched padded ARD Grams (gpb200_lml_grad_ard_batched, gpb200_posterior_draws_ard_batched) ----
// Squared scaled distance r^2 = sum_d (xs[r] - ys[c])^2 between staged row point r and column point c (coordinates
// already divided by rho_d, one dimension every TILE doubles), accumulated over d in order.  It is symmetric to the bit
// ((a - b)^2 == (b - a)^2).  Both ARD Gram kernels turn it into alpha^2 exp(-r^2 / 2) themselves: written as one
// helper, the whole element changes the register allocation of gram_ard_batched_kernel; this part leaves its SASS as
// it was.  exp_nonpos clamps its argument with fmax, which drops a NaN: a NaN coordinate or length-scale must reach
// the factorisation (and fail its item) as it does in the reference, hence the isnan pass-through in both kernels.
__device__ __forceinline__ double ard_r2(const double *xs, const double *ys, int r, int c, int D) {
  double r2 = 0.0;
  for (int d = 0; d < D; d++) {
    const double dq = xs[d * TILE + r] - ys[d * TILE + c];
    r2 = fma(dq, dq, r2);
  }
  return r2;
}

// K = alpha^2 exp(-0.5 sum_d ((X_id - X_jd) / rho_d)^2) + c I: QQard of R/kernels.R:19 plus the noise diagonal.
// X per item is n x D column-major (leading dimension n); theta per item (alpha, rho_1 .. rho_D, sigma).  Layout as
// gram_se_batched_kernel: np x np per item, identity in the padding, lower tiles only.  The coordinates are staged
// already divided by rho_d, with the same division the ARD trace epilogue (gemm.cu) uses.
__global__ void __launch_bounds__(256) gram_ard_batched_kernel(int n, int D, int np, const double *__restrict__ X,
                                                              long long x_stride, const double *__restrict__ theta,
                                                              double jitter, double *__restrict__ K, long long stride) {
  const int nt = np / TILE;
  const int tr = blockIdx.x % nt, tc = blockIdx.x / nt;
  if (tr < tc) return;
  __shared__ double xs[ARD_MAX_D * TILE], ys[ARD_MAX_D * TILE];
  const long long b = blockIdx.y;
  const double *Xb = X + b * x_stride;
  const double *th = theta + b * (D + 2);
  const int r0 = tr * TILE, c0 = tc * TILE, tid = threadIdx.x;
  for (int q = tid; q < D * 2 * TILE; q += 256) {
    const int d = q / (2 * TILE), l = q % (2 * TILE);
    const int i = (l < TILE) ? r0 + l : c0 + l - TILE;
    const double v = (i < n) ? Xb[i + (long long)d * n] / th[1 + d] : 0.0;
    if (l < TILE) xs[d * TILE + l] = v;
    else ys[d * TILE + l - TILE] = v;
  }
  __syncthreads();
  const double alpha = th[0], sigma = th[D + 1];
  const double a2 = alpha * alpha, dadd = sigma * sigma + jitter;
  double *Kb = K + b * stride;
  const int rl = 2 * (tid & 63), cq = tid >> 6;
#pragma unroll 2
  for (int s = 0; s < 32; s++) {
    const int cl = cq + 4 * s;
    const int j = c0 + cl;
    double v[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int i = r0 + rl + e;
      if (i < n && j < n) {
        const double r2 = ard_r2(xs, ys, rl + e, cl, D);
        v[e] = (i == j) ? a2 + dadd : a2 * (isnan(r2) ? r2 : exp_nonpos(-0.5 * r2));
      } else {
        v[e] = (i == j) ? 1.0 : 0.0;
      }
    }
    *reinterpret_cast<double2 *>(Kb + (r0 + rl) + (long long)j * np) = make_double2(v[0], v[1]);
  }
}

// Joint prior covariance of the noisy values f(X) + noise and f(Xs) under the ARD kernel, for conditioning and drawing
// in one factorisation (gpb200_posterior_draws_ard_batched):
//   J = [[QQard(X, X) + sigma^2 I,  .                       ],
//        [QQard(Xs, X),             QQard(Xs, Xs) + jitter I]]
// rows [0, n) from X (n x D per item, leading dimension n), rows [n, n+m) from Xs (m x D, leading dimension m);
// theta = (alpha, rho_1 .. rho_D, sigma) per item.  Layout as gram_cond_batched_kernel: np x np per item, identity in
// the padding, lower tiles only, the strict upper part of a diagonal tile mirrored (ard_r2 is symmetric).  The
// elements are those of gram_ard_batched_kernel.
__global__ void __launch_bounds__(256) gram_cond_ard_batched_kernel(int n, int m, int D, int np,
                                                                   const double *__restrict__ X, long long x_stride,
                                                                   const double *__restrict__ Xs, long long xs_stride,
                                                                   const double *__restrict__ theta, double jitter,
                                                                   double *__restrict__ K, long long stride) {
  const int nt = np / TILE;
  const int tr = blockIdx.x % nt, tc = blockIdx.x / nt;
  if (tr < tc) return;
  __shared__ double xs[ARD_MAX_D * TILE], ys[ARD_MAX_D * TILE];
  const long long b = blockIdx.y;
  const double *Xb = X + b * x_stride, *Sb = Xs + b * xs_stride;
  const double *th = theta + b * (D + 2);
  const int N = n + m;
  const int r0 = tr * TILE, c0 = tc * TILE, tid = threadIdx.x;
  for (int q = tid; q < D * 2 * TILE; q += 256) {
    const int d = q / (2 * TILE), l = q % (2 * TILE);
    const int i = (l < TILE) ? r0 + l : c0 + l - TILE;
    const double v = (i < n) ? Xb[i + (long long)d * n] / th[1 + d] : (i < N) ? Sb[i - n + (long long)d * m] / th[1 + d] : 0.0;
    if (l < TILE) xs[d * TILE + l] = v;
    else ys[d * TILE + l - TILE] = v;
  }
  __syncthreads();
  const double alpha = th[0], sigma = th[D + 1];
  const double a2 = alpha * alpha;
  double *Kb = K + b * stride;
  const int rl = 2 * (tid & 63), cq = tid >> 6;
#pragma unroll 2
  for (int s = 0; s < 32; s++) {
    const int cl = cq + 4 * s;
    const int j = c0 + cl;
    double v[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int i = r0 + rl + e;
      if (i < N && j < N) {
        const double r2 = ard_r2(xs, ys, rl + e, cl, D);
        v[e] = (i == j) ? a2 + (i < n ? sigma * sigma : jitter) : a2 * (isnan(r2) ? r2 : exp_nonpos(-0.5 * r2));
      } else {
        v[e] = (i == j) ? 1.0 : 0.0;
      }
    }
    *reinterpret_cast<double2 *>(Kb + (r0 + rl) + (long long)j * np) = make_double2(v[0], v[1]);
  }
}

// ---- f-3: Mercer / Hermite eigen-basis factor of the SE kernel ---------------------------------
// approx_L(M, scale, x, sigma, l) of models/westbrook.stan:2-30 (copied into six other models;
// spectral_test.R:6-27 `bH`): N x M matrix whose columns are scaled Hermite functions built by a
// three-term recurrence, with L L^T ~ cov_exp_quad(x, sigma, l).  One thread per row, columns written
// coalesced; HBM-bound (8 N M bytes).
__global__ void approx_basis_kernel(int n, int M, double scale, const double *__restrict__ x, double sigma, double l,
                                    double *__restrict__ out, long long ldo) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double a = 1.0 / (4.0 * scale * scale);
  const double b = 1.0 / (2.0 * l * l);
  const double epsilon = sqrt(b);
  const double alpha = sqrt(2.0 * a);
  const double r = 2.0 * epsilon / alpha;
  const double beta = sqrt(sqrt(1.0 + r * r));
  const double delta = sqrt(alpha * alpha * (beta * beta - 1.0) / 2.0);
  const double denom = alpha * alpha + delta * delta + epsilon * epsilon;
  const double xi = x[i];
  const double xp = alpha * beta * xi;
  const double f = sqrt(epsilon * epsilon / denom);
  double h1 = sqrt(sqrt(alpha * alpha / denom)) * sqrt(beta) * exp(-delta * delta * xi * xi);
  out[i] = sigma * h1;
  if (M < 2) return;
  double h2 = f * sqrt(1.0 / 2.0) * 2.0 * xp * h1;
  out[i + ldo] = sigma * h2;
  for (int k = 3; k <= M; k++) {
    const double h3 = f * sqrt(1.0 / (2.0 * (k - 1))) * 2.0 * xp * h2 -
                      f * f * sqrt(1.0 / (4.0 * (k - 1) * (double)(k - 2))) * 2.0 * (k - 2) * h1;
    out[i + (long long)(k - 1) * ldo] = sigma * h3;
    h1 = h2;
    h2 = h3;
  }
}

int launch_approx_basis(Handle *h, int n, int M, double scale, const double *x, double sigma, double l, double *out,
                        long long ldo) {
  ProfScope ps__(h, PC_GRAM);
  approx_basis_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(n, M, scale, x, sigma, l, out, ldo);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// ---- launchers ---------------------------------------------------------------------------------
int launch_kernel_eval(Handle *h, int kind, long long len, const double *tj, const double *tk, double amp2,
                       double l, double *out) {
  if (len <= 0) return 0;
  const int blocks = (int)((len + 255) / 256 > 148 * 16 ? 148 * 16 : (len + 255) / 256);
  ProfScope ps__(h, PC_GRAM);
  kernel_eval_kernel<<<blocks, 256, 0, h->stream>>>(kind, len, tj, tk, amp2, l, out);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_outer(Handle *h, int kind, int n, int m, const double *x, const double *y, double amp2, double l,
                      double *K, long long ldk) {
  if (n <= 0 || m <= 0) return 0;
  dim3 grid((n + TILE - 1) / TILE, (m + TILE - 1) / TILE);
  ProfScope ps__(h, PC_GRAM);
  gram_outer_kernel<<<grid, 256, 0, h->stream>>>(kind, n, m, x, y, amp2, l, K, ldk);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_se_batched(Handle *h, int n, int np, const double *x, long long x_stride, const double *theta,
                           double jitter, int lower_only, double *K, long long stride, int batch, int *env,
                           const int *nvec) {
  const int nt = np / TILE;
  dim3 grid(nt * nt, batch);
  ProfScope ps__(h, PC_GRAM);
  if (nvec)
    gram_se_batched_kernel<true><<<grid, 256, 0, h->stream>>>(n, np, x, x_stride, theta, jitter, lower_only, K, stride, env, nvec);
  else
    gram_se_batched_kernel<false><<<grid, 256, 0, h->stream>>>(n, np, x, x_stride, theta, jitter, lower_only, K, stride, env,
                                                               nullptr);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_se_panel(Handle *h, int n, int np, const double *x, double alpha, double rho, double diag_add,
                         int col0, int ncols, double *P, long long ldp) {
  dim3 grid((np - col0) / TILE, ncols / TILE);
  ProfScope ps__(h, PC_GRAM);
  gram_se_panel_kernel<<<grid, 256, 0, h->stream>>>(n, np, x, alpha, rho, diag_add, col0, P, ldp);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_tangent(Handle *h, int n, int np, const double *x, double alpha, const double *ls, double dadd, int mode,
                        double *S, double *Sdot, long long stride, int batch) {
  dim3 grid(np / TILE, np / TILE, batch);
  ProfScope ps__(h, PC_GRAM);
  gram_tangent_kernel<<<grid, 256, 0, h->stream>>>(n, np, x, alpha, ls, dadd, mode, S, Sdot, stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_deriv(Handle *h, int n, int nblocks, const double *t, double alpha, double rho, const double *noise,
                      double jitter, int quirk, double *K, long long ldk) {
  const int N = n * nblocks;
  dim3 grid((N + TILE - 1) / TILE, (N + TILE - 1) / TILE);
  ProfScope ps__(h, PC_GRAM);
  gram_deriv_kernel<<<grid, 256, 0, h->stream>>>(n, nblocks, t, alpha, rho, noise[0], nblocks > 1 ? noise[1] : 0.0,
                                                nblocks > 2 ? noise[2] : 0.0, jitter, quirk, K, ldk);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_deriv_batched(Handle *h, int n, int order0, int nblocks, int np, const double *t, long long t_stride,
                              const double *theta, int theta_stride, double jitter, int lower_only, double *K,
                              long long stride, int batch) {
  const int nt = np / TILE;
  dim3 grid(nt * nt, batch);
  ProfScope ps__(h, PC_GRAM);
  gram_deriv_batched_kernel<<<grid, 256, 0, h->stream>>>(n, order0, nblocks, np, t, t_stride, theta, theta_stride, jitter,
                                                        lower_only, K, stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_cond_batched(Handle *h, int n, int m, int order, int np, const double *t, long long t_stride,
                             const double *s, long long s_stride, const double *theta, double jitter, double *K,
                             long long stride, int batch) {
  const int nt = np / TILE;
  dim3 grid(nt * nt, batch);
  ProfScope ps__(h, PC_GRAM);
  gram_cond_batched_kernel<<<grid, 256, 0, h->stream>>>(n, m, order, np, t, t_stride, s, s_stride, theta, jitter, K, stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_ard_batched(Handle *h, int n, int D, int np, const double *X, long long x_stride, const double *theta,
                            double jitter, double *K, long long stride, int batch) {
  const int nt = np / TILE;
  dim3 grid(nt * nt, batch);
  ProfScope ps__(h, PC_GRAM);
  gram_ard_batched_kernel<<<grid, 256, 0, h->stream>>>(n, D, np, X, x_stride, theta, jitter, K, stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_cond_ard_batched(Handle *h, int n, int m, int D, int np, const double *X, long long x_stride,
                                 const double *Xs, long long xs_stride, const double *theta, double jitter, double *K,
                                 long long stride, int batch) {
  const int nt = np / TILE;
  dim3 grid(nt * nt, batch);
  ProfScope ps__(h, PC_GRAM);
  gram_cond_ard_batched_kernel<<<grid, 256, 0, h->stream>>>(n, m, D, np, X, x_stride, Xs, xs_stride, theta, jitter, K,
                                                            stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gram_ard(Handle *h, int n, int m, int D, const double *X, long long ldx, const double *Y, long long ldy,
                    double alpha, const double *rho, int rho_len, double *K, long long ldk) {
  if (n <= 0 || m <= 0) return 0;
  dim3 grid((n + 127) / 128, (m + 63) / 64);
  ProfScope ps__(h, PC_GRAM);
  gram_ard_kernel<<<grid, 256, 0, h->stream>>>(n, m, D, X, ldx, Y, ldy, alpha, rho, rho_len, K, ldk);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

}  // namespace gpb
