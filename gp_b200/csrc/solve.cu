// HBM-bound pieces of the path (sm_100a): triangular mat-vecs and solves with warp-shuffle
// reductions, the deterministic LML/gradient finalisation, pack/unpack between caller matrices and
// the padded internal layout, Hermite interpolation of tabulated factors.
//
//   trmv_lower_n / trmv_lower_t   z = W y, a = W^T z   (and f = L z of exact_gp.stan:25)
//   trsv_blocked                  mdivide_left_tri_low inside multi_normal_cholesky
//                                 (models/fit_hyperparameters.stan:31) when no inverse is wanted
//   finalize                      lml = -n/2 log 2pi - sum log L_ii - 0.5 ||z||^2 and the three
//                                 gradient components from the fused trace partials
//   hermite                       covariance.cpp:63-66,85-88 / cubic_interpolated_gp.hpp:63-70
#include <algorithm>

#include "common.cuh"
#include "fastexp.cuh"
#include "gram.cuh"

namespace gpb {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// z[i] = sum_{k<=i} W[i,k] y[k] for one 128-row strip per CTA.  The strict upper triangle of the
// diagonal tile is zero by construction, so the strip is read as a dense 128 x (tile+1)*128 block.
__global__ void __launch_bounds__(256) trmv_lower_n_kernel(int np, const double *__restrict__ W, long long stride,
                                                          const double *__restrict__ y, long long y_stride,
                                                          int n_valid, double *__restrict__ z, long long z_stride) {
  __shared__ double part[TILE];
  __shared__ double ys[512];
  const int tile = blockIdx.x, tid = threadIdx.x;
  const long long b = blockIdx.y;
  const double *Wb = W + b * stride;
  const double *yb = y + b * y_stride;
  const int r = tid & 127, half = tid >> 7;
  const int kmax = (tile + 1) * TILE;
  const int i = tile * TILE + r;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int k0 = 0; k0 < kmax; k0 += 512) {
    __syncthreads();
    for (int q = tid; q < 512; q += 256) ys[q] = (k0 + q < n_valid) ? yb[k0 + q] : 0.0;
    __syncthreads();
    const int kend = min(512, kmax - k0);
    const double *wp = Wb + i + (long long)(k0 + half) * np;
#pragma unroll 4
    for (int k = half; k < kend; k += 8) {
      s0 = fma(wp[0], ys[k], s0);
      s1 = fma(wp[2LL * np], ys[k + 2], s1);
      s2 = fma(wp[4LL * np], ys[k + 4], s2);
      s3 = fma(wp[6LL * np], ys[k + 6], s3);
      wp += 8LL * np;
    }
  }
  const double s = (s0 + s1) + (s2 + s3);
  if (half == 1) part[r] = s;
  __syncthreads();
  if (half == 0) z[b * z_stride + i] = s + part[r];
}

// The same product for a SINGLE matrix (or a few): one 128-row strip per CTA leaves 140 of 148 SMs idle and the
// N^2/2 read of W crawls at a tenth of HBM speed.  Here blockIdx.y splits each strip's k-range into `ks` chunks of
// whole tiles; every CTA writes its partial sums to part[(item * ks + chunk) * np + i], and
// trmv_reduce_parts_kernel adds the chunks in a fixed order (deterministic, no atomics).
__global__ void __launch_bounds__(256) trmv_lower_n_split_kernel(int np, int ks, const double *__restrict__ W, long long stride,
                                                                const double *__restrict__ y, long long y_stride,
                                                                int n_valid, double *__restrict__ part) {
  __shared__ double psum[TILE];
  __shared__ double ys[TILE];
  const int tile = blockIdx.x, chunk = blockIdx.y, tid = threadIdx.x;
  const long long b = blockIdx.z;
  const int ktiles = tile + 1;
  const int kt0 = (int)((long long)chunk * ktiles / ks), kt1 = (int)((long long)(chunk + 1) * ktiles / ks);
  const double *Wb = W + b * stride;
  const double *yb = y + b * y_stride;
  const int r = tid & 127, half = tid >> 7;
  const int i = tile * TILE + r;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int kt = kt0; kt < kt1; kt++) {
    const int k0 = kt * TILE;
    __syncthreads();
    if (tid < TILE) ys[tid] = (k0 + tid < n_valid) ? yb[k0 + tid] : 0.0;
    __syncthreads();
    const double *wp = Wb + i + (long long)(k0 + half) * np;
#pragma unroll 4
    for (int k = half; k < TILE; k += 8) {
      s0 = fma(wp[0], ys[k], s0);
      s1 = fma(wp[2LL * np], ys[k + 2], s1);
      s2 = fma(wp[4LL * np], ys[k + 4], s2);
      s3 = fma(wp[6LL * np], ys[k + 6], s3);
      wp += 8LL * np;
    }
  }
  const double s = (s0 + s1) + (s2 + s3);
  if (half == 1) psum[r] = s;
  __syncthreads();
  if (half == 0) part[(b * ks + chunk) * np + i] = s + psum[r];
}

__global__ void trmv_reduce_parts_kernel(int np, int ks, const double *__restrict__ part, double *__restrict__ z, long long z_stride) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const long long b = blockIdx.y;
  if (i >= np) return;
  double s = 0.0;
  for (int c = 0; c < ks; c++) s += part[(b * ks + c) * np + i];
  z[b * z_stride + i] = s;
}

// a[k] = sum_{i>=k} W[i,k] z[i]; one warp per column, 16-byte loads, shuffle reduction.
__global__ void __launch_bounds__(256) trmv_lower_t_kernel(int np, const double *__restrict__ W, long long stride,
                                                          const double *__restrict__ z, long long z_stride,
                                                          double *__restrict__ a, long long a_stride) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k = blockIdx.x * 8 + warp;
  const long long b = blockIdx.y;
  const double *col = W + b * stride + (long long)k * np;
  const double *zb = z + b * z_stride;
  const int istart = (k / TILE) * TILE;
  double s0 = 0.0, s1 = 0.0;
  for (int i = istart + 2 * lane; i < np; i += 64) {
    const double2 w = *reinterpret_cast<const double2 *>(col + i);
    const double2 zz = *reinterpret_cast<const double2 *>(zb + i);
    s0 = fma(w.x, zz.x, s0);
    s1 = fma(w.y, zz.y, s1);
  }
  const double s = warp_sum(s0 + s1);
  if (lane == 0) a[b * a_stride + k] = s;
}

// Blocked forward substitution L z = (y - mu), one CTA per batch item.  Per 128-row block:
// s = rhs_j - L[j, 0:j] z[0:j] (two k-halves per row), then z_j = Wdiag_j s with the pre-inverted
// diagonal tile.  z lives in global memory (written and re-read by this CTA only, ordered by the
// block barriers), so any n fits.  With a tile envelope (env: F, the first nonzero tile column per tile row) the
// contraction of block j starts at tile F_j: L is exactly zero to its left, and since F_j * 128 is a multiple of the
// k stride every product still lands in the same partial sum, so z is bit-identical to the dense sweep.
constexpr int TRSV_KSPLIT = 8;  // k-groups per row: 1024 threads per item keep enough loads in flight to approach HBM speed
__global__ void __launch_bounds__(TILE * TRSV_KSPLIT) trsv_blocked_kernel(int np, const double *__restrict__ L,
                                                          const double *__restrict__ Wdiag, long long stride,
                                                          const double *__restrict__ y, long long y_stride,
                                                          const double *__restrict__ mu, int n_valid,
                                                          double *z, long long z_stride, const int *__restrict__ env) {
  constexpr int KS = TRSV_KSPLIT;
  __shared__ double part[KS][TILE];
  __shared__ double sv[TILE];
  const long long b = blockIdx.x;
  const double *Lb = L + b * stride, *Wb = Wdiag + b * stride;
  const double *yb = y + b * y_stride;
  double *zb = z + b * z_stride;
  const int tid = threadIdx.x, r = tid & 127, grp = tid >> 7;
  const int nt = np / TILE;
  for (int j = 0; j < nt; j++) {
    const int i = j * TILE + r;
    const int kmax = j * TILE;  // multiple of 128, so every group's strided range has the same length
    const int kmin = env ? env[b * 2 * nt + j] * TILE : 0;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const double *lp = Lb + i + (long long)(kmin + grp) * np;
    for (int k = kmin + grp; k < kmax; k += 4 * KS) {
      s0 = fma(lp[0], zb[k], s0);
      s1 = fma(lp[(long long)KS * np], zb[k + KS], s1);
      s2 = fma(lp[2LL * KS * np], zb[k + 2 * KS], s2);
      s3 = fma(lp[3LL * KS * np], zb[k + 3 * KS], s3);
      lp += 4LL * KS * np;
    }
    part[grp][r] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (grp == 0) {
      double acc = 0.0;
#pragma unroll
      for (int q = 0; q < KS; q++) acc += part[q][r];
      double rhs = 0.0;
      if (i < n_valid) rhs = yb[i] - (mu ? mu[i] : 0.0);
      sv[r] = rhs - acc;
    }
    __syncthreads();
    // z_j = Wdiag_j * sv  (lower-triangular 128x128, strict upper is zero)
    const double *wd = Wb + (long long)j * TILE * (np + 1);
    double t0 = 0.0, t1 = 0.0;
    for (int k = grp; k < TILE; k += 2 * KS) {
      t0 = fma(wd[r + (long long)k * np], sv[k], t0);
      t1 = fma(wd[r + (long long)(k + KS) * np], sv[k + KS], t1);
    }
    part[grp][r] = t0 + t1;
    __syncthreads();
    if (grp == 0) {
      double acc = 0.0;
#pragma unroll
      for (int q = 0; q < KS; q++) acc += part[q][r];
      zb[i] = acc;
    }
    __syncthreads();
  }
}

// Column-sweep forward substitution for small batches (one large matrix): per 128-column block j
//   trsv_diag:    z_j = Wdiag_j (rhs_j - acc_j)                       one CTA per item
//   trsv_update:  acc_i += L[i, j] z_j for every tile row i > j        (nt-1-j) CTAs per item
// so that the N^2/2 read of L is spread over the whole GPU instead of one CTA.
__global__ void __launch_bounds__(128) trsv_diag_kernel(long long ldw, long long w_off, int row0,
                                                       const double *__restrict__ Wdiag, long long stride,
                                                       const double *__restrict__ y, long long y_stride,
                                                       const double *__restrict__ mu, int n_valid,
                                                       const double *__restrict__ acc, double *__restrict__ z,
                                                       long long z_stride) {
  __shared__ double sv[TILE];
  const long long b = blockIdx.x;
  const int r = threadIdx.x, i = row0 + r;
  double rhs = 0.0;
  if (i < n_valid) rhs = y[b * y_stride + i] - (mu ? mu[i] : 0.0);
  sv[r] = rhs - acc[b * z_stride + i];
  __syncthreads();
  const double *wd = Wdiag + b * stride + w_off;
  double t0 = 0.0, t1 = 0.0;
  for (int k = 0; k < TILE; k += 2) {
    t0 = fma(wd[r + (long long)k * ldw], sv[k], t0);
    t1 = fma(wd[r + (long long)(k + 1) * ldw], sv[k + 1], t1);
  }
  z[b * z_stride + i] = t0 + t1;
}

// acc[acc_row0 + 128*blockIdx.x + r] += sum_k L[l_off + 128*blockIdx.x + r + k*ld] * z[z_row0 + k]
__global__ void __launch_bounds__(256) trsv_update_kernel(long long ld, long long l_off, int z_row0, int acc_row0,
                                                         const double *__restrict__ L, long long stride,
                                                         const double *__restrict__ z, double *__restrict__ acc,
                                                         long long z_stride) {
  __shared__ double zs[TILE];
  __shared__ double part[TILE];
  const long long b = blockIdx.y;
  const int tid = threadIdx.x, r = tid & 127, half = tid >> 7;
  if (tid < TILE) zs[tid] = z[b * z_stride + z_row0 + tid];
  __syncthreads();
  const double *lp = L + b * stride + l_off + (long long)blockIdx.x * TILE + r + (long long)half * ld;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll 4
  for (int k = half; k < TILE; k += 8) {
    s0 = fma(lp[0], zs[k], s0);
    s1 = fma(lp[2LL * ld], zs[k + 2], s1);
    s2 = fma(lp[4LL * ld], zs[k + 4], s2);
    s3 = fma(lp[6LL * ld], zs[k + 6], s3);
    lp += 8LL * ld;
  }
  const double ssum = (s0 + s1) + (s2 + s3);
  if (half == 1) part[r] = ssum;
  __syncthreads();
  if (half == 0) acc[b * z_stride + acc_row0 + blockIdx.x * TILE + r] += ssum + part[r];
}

// Deterministic finalisation, one CTA per batch item.
__global__ void __launch_bounds__(256) finalize_kernel(int n, int np, int want_grad, const double *__restrict__ dvec,
                                                      const double *__restrict__ z, const double *__restrict__ a,
                                                      const double *__restrict__ partial, int ntasks, int ntasks2,
                                                      const double *__restrict__ theta, double *__restrict__ lml,
                                                      double *__restrict__ grad) {
  __shared__ double red[8][6];
  const long long b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double ld = 0.0, qf = 0.0, aa = 0.0, p0 = 0.0, p1 = 0.0, p2 = 0.0;
  for (int i = tid; i < n; i += 256) {
    ld += log(dvec[b * np + i]);
    const double zi = z[b * np + i];
    qf = fma(zi, zi, qf);
    if (want_grad) {
      const double ai = a[b * np + i];
      aa = fma(ai, ai, aa);
    }
  }
  if (want_grad) {
    for (int q = tid; q < ntasks; q += 256) {
      const double *pp = partial + (b * ntasks + q) * 4;
      p0 += pp[0];
      p1 += pp[1];
      p2 += pp[2];
    }
    const double *part2 = partial + (long long)gridDim.x * ntasks * 4;   // second region (diagonal-split launch)
    for (int q = tid; q < ntasks2; q += 256) {
      const double *pp = part2 + (b * ntasks2 + q) * 4;
      p0 += pp[0];
      p1 += pp[1];
      p2 += pp[2];
    }
  }
  ld = warp_sum(ld); qf = warp_sum(qf); aa = warp_sum(aa);
  p0 = warp_sum(p0); p1 = warp_sum(p1); p2 = warp_sum(p2);
  if (lane == 0) {
    red[warp][0] = ld; red[warp][1] = qf; red[warp][2] = aa;
    red[warp][3] = p0; red[warp][4] = p1; red[warp][5] = p2;
  }
  __syncthreads();
  if (tid == 0) {
    double s[6] = {0, 0, 0, 0, 0, 0};
    for (int w = 0; w < 8; w++)
      for (int q = 0; q < 6; q++) s[q] += red[w][q];
    lml[b] = -0.5 * n * 1.8378770664093454835606594728112 - s[0] - 0.5 * s[1];
    if (want_grad) {
      const double alpha = theta[b * 3 + 0], rho = theta[b * 3 + 1], sigma = theta[b * 3 + 2];
      grad[b * 3 + 0] = alpha * s[3];                                   // 0.5 sum M * 2 alpha e
      grad[b * 3 + 1] = 0.5 * alpha * alpha * s[4] / (rho * rho * rho);  // 0.5 sum M * alpha^2 e d^2 / rho^3
      grad[b * 3 + 2] = sigma * (s[2] - s[5]);                          // 0.5 tr(M) 2 sigma
    }
  }
}

// out2[0] = sum z_i^2, out2[1] = sum log L_ii  (multi_normal_cholesky_lpdf pieces)
__global__ void __launch_bounds__(256) sumsq_logdiag_kernel(int n, const double *__restrict__ z,
                                                           const double *__restrict__ L, long long ldl,
                                                           double *__restrict__ out2) {
  __shared__ double red[8][2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double q = 0.0, ld = 0.0;
  for (int i = tid; i < n; i += 256) {
    q = fma(z[i], z[i], q);
    ld += log(L[i + (long long)i * ldl]);
  }
  q = warp_sum(q); ld = warp_sum(ld);
  if (lane == 0) { red[warp][0] = q; red[warp][1] = ld; }
  __syncthreads();
  if (tid == 0) {
    double s0 = 0, s1 = 0;
    for (int w = 0; w < 8; w++) { s0 += red[w][0]; s1 += red[w][1]; }
    out2[0] = s0; out2[1] = s1;
  }
}

// pack a caller matrix into the padded internal layout.
// mode 0: dense, zero padding.  mode 1: square, identity on the padded diagonal, + diag_add on the
// real diagonal.  mode 2: lower triangle only (strict upper zeroed), identity padding.
__global__ void pack_kernel(int rows, int cols, const double *__restrict__ src, long long lds, int rp, int cp,
                            double *__restrict__ dst, int mode, double diag_add) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y;
  if (i >= rp || j >= cp) return;
  double v = 0.0;
  if (i < rows && j < cols) {
    v = src[i + (long long)j * lds];
    if (mode == 1 && i == j) v += diag_add;
    if (mode == 2 && i < j) v = 0.0;
  } else if (mode != 0 && i == j) {
    v = 1.0;
  }
  dst[i + (long long)j * rp] = v;
}

// unpack.  mode 0: dense.  mode 1: lower (strict upper zero).  mode 2: symmetric, mirrored from the
// lower triangle.  diag_add is added on the diagonal.
__global__ void unpack_kernel(int rows, int cols, const double *__restrict__ src, long long lds_src,
                              double *__restrict__ dst, long long ldd, int mode, double diag_add) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y;
  if (i >= rows || j >= cols) return;
  double v;
  if (mode == 1) v = (i >= j) ? src[i + (long long)j * lds_src] : 0.0;
  else if (mode == 2) v = (i >= j) ? src[i + (long long)j * lds_src] : src[j + (long long)i * lds_src];
  else v = src[i + (long long)j * lds_src];
  if (i == j) v += diag_add;
  dst[i + (long long)j * ldd] = v;
}

// Phi for the forward-mode Cholesky tangent: keep the lower triangle, halve the diagonal, zero the
// strict upper part (only the diagonal tiles contain upper entries that are ever read).
__global__ void phi_lower_kernel(int np, double *__restrict__ A, long long stride) {
  A += (long long)blockIdx.z * stride;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y;
  if (i >= np) return;
  if ((i / TILE) != (j / TILE)) return;
  double *p = A + i + (long long)j * np;
  if (i == j) *p *= 0.5;
  else if (i < j) *p = 0.0;
}

// out[c] = add[c] + sum_r V[r,c] z[r]   (dense V^T z, warp per column)
__global__ void __launch_bounds__(256) gemv_t_kernel(int rows, int cols, const double *__restrict__ V, long long ldv,
                                                    const double *__restrict__ z, const double *__restrict__ add,
                                                    double *__restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * 8 + warp;
  if (c >= cols) return;
  double s = 0.0;
  for (int r = lane; r < rows; r += 32) s = fma(V[r + (long long)c * ldv], z[r], s);
  s = warp_sum(s);
  if (lane == 0) out[c] = s + (add ? add[c] : 0.0);
}

// Cubic-Hermite interpolation between two tabulated factors (lower triangle only; n x n dense
// column-major tables).  v -> interpolated L, dvdl -> its l-derivative (may be null).
__global__ void hermite_kernel(long long len, int n, const double *__restrict__ y1, const double *__restrict__ y2,
                               const double *__restrict__ k1, const double *__restrict__ k2, double x1, double x2,
                               double l, double *__restrict__ v, double *__restrict__ dvdl) {
  const double dx = x2 - x1, t = (l - x1) / dx, dtdl = 1.0 / dx;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < len; q += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(q % n), j = (int)(q / n);
    double vv = 0.0, dd = 0.0;
    if (j <= i) {
      const double a1 = y1[q], a2 = y2[q];
      const double a = k1[q] * dx - (a2 - a1);
      const double bb = -k2[q] * dx + (a2 - a1);
      vv = (1 - t) * a1 + t * a2 + t * (1 - t) * (a * (1 - t) + bb * t);
      dd = (bb * (2 - 3 * t) * t + a * (1 + t * (-4 + 3 * t)) - a1 + a2) * dtdl;
    }
    v[q] = vv;
    if (dvdl) dvdl[q] = dd;
  }
}

// approx_Lz fused (models/cubic_interpolated_gp.hpp:46-72): the four tables are read ONCE and the interpolated factor
// is never stored -- each thread owns a row i, walks a chunk of the columns j <= i, forms v_ij and dv_ij/dl from
// (y1, y2, k1, k2)_ij in registers and accumulates v_ij z_j and dv_ij z_j.  Consecutive threads read consecutive rows
// (coalesced); blockIdx.y splits the columns so that a 4096 x 4096 table still fills the GPU; the chunk sums are
// added in a fixed order by hermite_matvec_reduce_kernel.  HBM-bound: 4 * 8 * n^2 / 2 bytes.
__global__ void __launch_bounds__(128) hermite_matvec_kernel(int n, const double *__restrict__ y1, const double *__restrict__ y2,
                                                             const double *__restrict__ k1, const double *__restrict__ k2,
                                                             double x1, double x2, double l, const double *__restrict__ z,
                                                             double *__restrict__ part) {
  const int i = blockIdx.x * 128 + threadIdx.x;
  const int nchunk = gridDim.y;
  const int per = (n + nchunk - 1) / nchunk;
  const int j0 = blockIdx.y * per, j1 = min(n, j0 + per);
  const double dx = x2 - x1, t = (l - x1) / dx, dtdl = 1.0 / dx;
  const double omt = 1.0 - t, tomt = t * omt;
  double sv = 0.0, sd = 0.0;
  if (i < n) {
    const int jend = min(j1, i + 1);
    for (int j = j0; j < jend; j++) {
      const long long q = i + (long long)j * n;
      const double a1 = y1[q], a2 = y2[q];
      const double a = k1[q] * dx - (a2 - a1);
      const double bb = -k2[q] * dx + (a2 - a1);
      const double vv = omt * a1 + t * a2 + tomt * (a * omt + bb * t);
      const double dd = (bb * (2 - 3 * t) * t + a * (1 + t * (-4 + 3 * t)) - a1 + a2) * dtdl;
      const double zj = z[j];
      sv = fma(vv, zj, sv);
      sd = fma(dd, zj, sd);
    }
    part[((long long)blockIdx.y * n + i) * 2] = sv;
    part[((long long)blockIdx.y * n + i) * 2 + 1] = sd;
  }
}
__global__ void hermite_matvec_reduce_kernel(int n, int nchunk, const double *__restrict__ part, double *__restrict__ vz,
                                             double *__restrict__ dvz) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double a = 0.0, b = 0.0;
  for (int c = 0; c < nchunk; c++) {
    a += part[((long long)c * n + i) * 2];
    b += part[((long long)c * n + i) * 2 + 1];
  }
  vz[i] = a;
  if (dvz) dvz[i] = b;
}

// ---- launchers ---------------------------------------------------------------------------------
int launch_trmv_lower_n(Handle *h, int np, const double *W, long long stride, const double *y, long long y_stride,
                        int n_valid, double *z, long long z_stride, int batch) {
  dim3 grid(np / TILE, batch);
  ProfScope ps__(h, PC_SOLVE);
  trmv_lower_n_kernel<<<grid, 256, 0, h->stream>>>(np, W, stride, y, y_stride, n_valid, z, z_stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// number of k-chunks the split mat-vec uses for this shape (1 = the plain kernel is as good)
int trmv_split_chunks(int np, int batch) {
  const int nt = np / TILE;
  const long long ctas = (long long)nt * batch;
  if (ctas >= 2 * 148 || nt < 4) return 1;
  return (int)std::min<long long>(nt, (2 * 148 + ctas - 1) / ctas);
}

// z = W y with the k-range split over `ks` CTAs per strip; part holds batch * ks * np doubles
int launch_trmv_lower_n_split(Handle *h, int np, int ks, const double *W, long long stride, const double *y, long long y_stride,
                              int n_valid, double *part, double *z, long long z_stride, int batch) {
  {
    dim3 grid(np / TILE, ks, batch);
    ProfScope ps__(h, PC_SOLVE);
    trmv_lower_n_split_kernel<<<grid, 256, 0, h->stream>>>(np, ks, W, stride, y, y_stride, n_valid, part);
    GPB_LAUNCH_CHECK(h);
  }
  dim3 grid2((np + 255) / 256, batch);
  ProfScope ps__(h, PC_SOLVE);
  trmv_reduce_parts_kernel<<<grid2, 256, 0, h->stream>>>(np, ks, part, z, z_stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_trmv_lower_t(Handle *h, int np, const double *W, long long stride, const double *z, long long z_stride,
                        double *a, long long a_stride, int batch) {
  dim3 grid(np / 8, batch);
  ProfScope ps__(h, PC_SOLVE);
  trmv_lower_t_kernel<<<grid, 256, 0, h->stream>>>(np, W, stride, z, z_stride, a, a_stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_trsv_blocked(Handle *h, int np, const double *L, const double *Wdiag, long long stride, const double *y,
                        long long y_stride, const double *mu, int n_valid, double *z, long long z_stride, int batch,
                        const int *env) {
  ProfScope ps__(h, PC_SOLVE);
  trsv_blocked_kernel<<<batch, TILE * TRSV_KSPLIT, 0, h->stream>>>(np, L, Wdiag, stride, y, y_stride, mu, n_valid, z, z_stride, env);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_trsv_diag(Handle *h, long long ldw, long long w_off, int row0, const double *Wdiag, long long stride,
                     const double *y, long long y_stride, const double *mu, int n_valid, const double *acc, double *z,
                     long long z_stride, int batch) {
  ProfScope ps__(h, PC_SOLVE);
  trsv_diag_kernel<<<batch, 128, 0, h->stream>>>(ldw, w_off, row0, Wdiag, stride, y, y_stride, mu, n_valid, acc, z, z_stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_trsv_update(Handle *h, long long ld, long long l_off, int z_row0, int acc_row0, int ntiles, const double *L,
                       long long stride, const double *z, double *acc, long long z_stride, int batch) {
  if (ntiles <= 0) return 0;
  ProfScope ps__(h, PC_SOLVE);
  dim3 grid(ntiles, batch);
  trsv_update_kernel<<<grid, 256, 0, h->stream>>>(ld, l_off, z_row0, acc_row0, L, stride, z, acc, z_stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_trsv_sweep(Handle *h, int np, const double *L, const double *Wdiag, long long stride, const double *y,
                      long long y_stride, const double *mu, int n_valid, double *z, double *acc, long long z_stride,
                      int batch) {
  const int nt = np / TILE;
  cudaError_t e = cudaMemsetAsync(acc, 0, sizeof(double) * (size_t)z_stride * batch, h->stream);
  if (e != cudaSuccess) return -1000;
  for (int j = 0; j < nt; j++) {
    const long long doff = (long long)j * TILE * (np + 1);
    int rc = launch_trsv_diag(h, np, doff, j * TILE, Wdiag, stride, y, y_stride, mu, n_valid, acc, z, z_stride, batch);
    if (rc) return rc;
    rc = launch_trsv_update(h, np, doff + TILE, j * TILE, (j + 1) * TILE, nt - 1 - j, L, stride, z, acc, z_stride, batch);
    if (rc) return rc;
  }
  return 0;
}

// ---- tile envelope of the SE covariance ------------------------------------------------------------------------------
// env per item: F[0..nt) (first nonzero tile column of each tile row, filled by gram_se_batched; F_I <= I) and
// E[0..nt): E_J = the last tile row I with F_I <= J.  F need not be monotone (x unsorted).  For K > J, E_K >= E_J,
// which is what closes the selected-inverse recurrence over the contiguous range J+1..E_J.
__global__ void __launch_bounds__(256) envelope_profile_kernel(int nt, int *__restrict__ env) {
  extern __shared__ int sF[];
  int *F = env + (long long)blockIdx.x * 2 * nt, *E = F + nt;
  for (int i = threadIdx.x; i < nt; i += blockDim.x) sF[i] = min(F[i], i);
  __syncthreads();
  for (int j = threadIdx.x; j < nt; j += blockDim.x) {
    int e = j;
    for (int i = nt - 1; i > j; i--)
      if (sF[i] <= j) { e = i; break; }
    F[j] = sF[j];
    E[j] = e;
  }
}

int launch_envelope_profile(Handle *h, int nt, int *env, int batch) {
  ProfScope ps__(h, PC_OTHER);
  envelope_profile_kernel<<<batch, 256, nt * sizeof(int), h->stream>>>(nt, env);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// Trace partials of the gradient from the selected inverse Z = K^-1 (lower tiles and full diagonal tiles, valid on
// the envelope): one CTA per lower tile (I, J) of one item, the same sums as the EPI_TRACE epilogue of the dense route
//   [0] w sum (a_i a_j - Z_ij) e_ij,  [1] w sum (a_i a_j - Z_ij) e_ij d_ij^2,  [2] tr Z on diagonal tiles
// with w = 2 off the diagonal (the tile stands for its transpose too).  Outside the envelope e_ij is exactly zero:
// those CTAs only write zeros.
__global__ void __launch_bounds__(256) trace_sinv_kernel(int n, int np, const double *__restrict__ Z, long long stride,
                                                        const int *__restrict__ env, const double *__restrict__ x,
                                                        long long x_stride, const double *__restrict__ a,
                                                        const double *__restrict__ theta, double *__restrict__ partial) {
  __shared__ double xr[TILE], xc[TILE], ar[TILE], ac[TILE], red[8][3];
  const int nt = np / TILE, q = blockIdx.x, tid = threadIdx.x;
  const long long b = blockIdx.y;
  int I = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
  while (I * (I + 1) / 2 > q) I--;
  while ((I + 1) * (I + 2) / 2 <= q) I++;
  const int J = q - I * (I + 1) / 2;
  double *o = partial + (b * gridDim.x + q) * 4;
  if (J < env[b * 2 * nt + I]) {
    if (tid < 4) o[tid] = 0.0;
    return;
  }
  const double *xb = x + b * x_stride, *ab = a + b * np;
  if (tid < TILE) {
    const int i = I * TILE + tid;
    xr[tid] = i < n ? xb[i] : 0.0;
    ar[tid] = i < n ? ab[i] : 0.0;
  } else {
    const int j = J * TILE + tid - TILE;
    xc[tid - TILE] = j < n ? xb[j] : 0.0;
    ac[tid - TILE] = j < n ? ab[j] : 0.0;
  }
  __syncthreads();
  const double rho = theta[b * 3 + 1], nh = -0.5 / (rho * rho);
  const int r = tid & 127, cq = tid >> 7, i = I * TILE + r;
  const double *Zb = Z + b * stride + i + (long long)J * TILE * np;
  double s_se = 0.0, s_d2 = 0.0, s_tr = 0.0;
  if (i < n) {
    for (int c = cq; c < TILE; c += 2) {
      const int j = J * TILE + c;
      if (j >= n) break;
      const double G = Zb[(long long)c * np];
      const double d = xr[r] - xc[c], d2 = d * d, ek = exp_nonpos(d2 * nh);
      const double M = ar[r] * ac[c] - G;
      s_se += M * ek;
      s_d2 += M * ek * d2;
      if (i == j) s_tr += G;
    }
  }
  const double w = I == J ? 1.0 : 2.0;
  s_se = warp_sum(s_se * w);
  s_d2 = warp_sum(s_d2 * w);
  s_tr = warp_sum(s_tr);
  if ((tid & 31) == 0) { red[tid >> 5][0] = s_se; red[tid >> 5][1] = s_d2; red[tid >> 5][2] = s_tr; }
  __syncthreads();
  if (tid < 3) {
    double s = 0.0;
    for (int w8 = 0; w8 < 8; w8++) s += red[w8][tid];
    o[tid] = s;
  } else if (tid == 3) {
    o[3] = 0.0;
  }
}

int launch_trace_sinv(Handle *h, int n, int np, const double *Z, long long stride, const int *env, const double *x,
                      long long x_stride, const double *a, const double *theta, double *partial, int batch) {
  const int nt = np / TILE;
  dim3 grid(nt * (nt + 1) / 2, batch);
  ProfScope ps__(h, PC_OTHER);
  trace_sinv_kernel<<<grid, 256, 0, h->stream>>>(n, np, Z, stride, env, x, x_stride, a, theta, partial);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// Band-limited blocked back substitution a = L^-T z, one CTA of 32 warps per item, block rows from the last:
//   s = z_J - sum_{I=J+1..E_J} L[I,J]^T a_I,   a_J = Wdiag_J^T s
// Rows below E_J are exactly zero in block column J.  A warp owns four columns; its lanes run down a column
// (16-byte loads), so every read of L is coalesced.
__global__ void __launch_bounds__(1024) backsub_band_kernel(int np, const double *__restrict__ L, const double *__restrict__ Wdiag,
                                                           long long stride, const int *__restrict__ env,
                                                           const double *__restrict__ z, double *a) {
  __shared__ double sv[TILE];
  const long long b = blockIdx.x;
  const int nt = np / TILE, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double *Lb = L + b * stride, *Wb = Wdiag + b * stride, *zb = z + b * np;
  const int *E = env + b * 2 * nt + nt;
  double *ab = a + b * np;
  for (int J = nt - 1; J >= 0; J--) {
    const int i0 = (J + 1) * TILE, i1 = (E[J] + 1) * TILE;
    for (int c = warp; c < TILE; c += 32) {
      const int col = J * TILE + c;
      const double *lc = Lb + (long long)col * np;
      double s0 = 0.0, s1 = 0.0;
      for (int i = i0 + 2 * lane; i < i1; i += 64) {
        const double2 l2 = *reinterpret_cast<const double2 *>(lc + i);
        const double2 a2 = *reinterpret_cast<const double2 *>(ab + i);
        s0 = fma(l2.x, a2.x, s0);
        s1 = fma(l2.y, a2.y, s1);
      }
      const double s = warp_sum(s0 + s1);
      if (lane == 0) sv[c] = zb[col] - s;
    }
    __syncthreads();
    for (int c = warp; c < TILE; c += 32) {
      const double *wc = Wb + (long long)J * TILE * (np + 1) + (long long)c * np;  // column c of the diagonal tile inverse
      const double2 w2 = *reinterpret_cast<const double2 *>(wc + 2 * lane);
      const double2 w3 = *reinterpret_cast<const double2 *>(wc + 64 + 2 * lane);
      double s = fma(w2.x, sv[2 * lane], w2.y * sv[2 * lane + 1]);
      s = fma(w3.x, sv[64 + 2 * lane], fma(w3.y, sv[65 + 2 * lane], s));
      s = warp_sum(s);
      if (lane == 0) ab[J * TILE + c] = s;
    }
    __syncthreads();
  }
}

int launch_backsub_band(Handle *h, int np, const double *L, const double *Wdiag, long long stride, const int *env,
                        const double *z, double *a, int batch) {
  ProfScope ps__(h, PC_SOLVE);
  backsub_band_kernel<<<batch, 1024, 0, h->stream>>>(np, L, Wdiag, stride, env, z, a);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_finalize(Handle *h, int n, int np, int want_grad, const double *dvec, const double *z, const double *a,
                    const double *partial, int ntasks, int ntasks2, const double *theta, double *lml, double *grad, int batch) {
  ProfScope ps__(h, PC_OTHER);
  finalize_kernel<<<batch, 256, 0, h->stream>>>(n, np, want_grad, dvec, z, a, partial, ntasks, ntasks2, theta, lml, grad);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// The same for the derivative-observation LML (EPI_TRACE_DERIV partials: 8 doubles per tile = sum M k,
// sum M dk/dl, tr G over each of up to three blocks); theta = (alpha, rho, noise[nblocks]) per item,
// grad in the same layout.
__global__ void __launch_bounds__(256) finalize_deriv_kernel(int n_grid, int nblocks, int np, int want_grad,
                                                            const double *__restrict__ dvec, const double *__restrict__ z,
                                                            const double *__restrict__ a,
                                                            const double *__restrict__ partial, int ntasks, int ntasks2,
                                                            const double *__restrict__ theta, double *__restrict__ lml,
                                                            double *__restrict__ grad) {
  __shared__ double red[8][10];
  const long long b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = n_grid * nblocks, ts = 2 + nblocks;
  double v[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // logdet, quad, aa[3], sum_k, sum_dk, tr[3]
  for (int i = tid; i < n; i += 256) {
    v[0] += log(dvec[b * np + i]);
    const double zi = z[b * np + i];
    v[1] = fma(zi, zi, v[1]);
    if (want_grad) {
      const double ai = a[b * np + i];
      const int blk = (i >= n_grid) + (i >= 2 * n_grid);
      if (blk == 0) v[2] = fma(ai, ai, v[2]); else if (blk == 1) v[3] = fma(ai, ai, v[3]); else v[4] = fma(ai, ai, v[4]);
    }
  }
  if (want_grad) {
    for (int q = tid; q < ntasks; q += 256) {
      const double *pp = partial + (b * ntasks + q) * 8;
#pragma unroll
      for (int c = 0; c < 5; c++) v[5 + c] += pp[c];
    }
    const double *part2 = partial + (long long)gridDim.x * ntasks * 8;
    for (int q = tid; q < ntasks2; q += 256) {
      const double *pp = part2 + (b * ntasks2 + q) * 8;
#pragma unroll
      for (int c = 0; c < 5; c++) v[5 + c] += pp[c];
    }
  }
#pragma unroll
  for (int c = 0; c < 10; c++) v[c] = warp_sum(v[c]);
  if (lane == 0)
#pragma unroll
    for (int c = 0; c < 10; c++) red[warp][c] = v[c];
  __syncthreads();
  if (tid == 0) {
    double s[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int w = 0; w < 8; w++)
      for (int c = 0; c < 10; c++) s[c] += red[w][c];
    lml[b] = -0.5 * n * 1.8378770664093454835606594728112 - s[0] - 0.5 * s[1];
    if (want_grad) {
      const double *th = theta + b * ts;
      grad[b * ts + 0] = th[0] * s[5];                 // 0.5 sum M * 2 alpha k
      grad[b * ts + 1] = 0.5 * th[0] * th[0] * s[6];   // 0.5 sum M * alpha^2 dk/dl
      for (int q = 0; q < nblocks; q++) grad[b * ts + 2 + q] = th[2 + q] * (s[2 + q] - s[7 + q]);
    }
  }
}

int launch_finalize_deriv(Handle *h, int n_grid, int nblocks, int np, int want_grad, const double *dvec, const double *z,
                          const double *a, const double *partial, int ntasks, int ntasks2, const double *theta, double *lml,
                          double *grad, int batch) {
  ProfScope ps__(h, PC_OTHER);
  finalize_deriv_kernel<<<batch, 256, 0, h->stream>>>(n_grid, nblocks, np, want_grad, dvec, z, a, partial, ntasks, ntasks2, theta,
                                                     lml, grad);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_sumsq_logdiag(Handle *h, int n, const double *z, const double *L, long long ldl, double *out2) {
  ProfScope ps__(h, PC_OTHER);
  sumsq_logdiag_kernel<<<1, 256, 0, h->stream>>>(n, z, L, ldl, out2);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_pack(Handle *h, int rows, int cols, const double *src, long long lds, int rp, int cp, double *dst,
                int mode, double diag_add) {
  dim3 grid((rp + 255) / 256, cp);
  ProfScope ps__(h, PC_OTHER);
  pack_kernel<<<grid, 256, 0, h->stream>>>(rows, cols, src, lds, rp, cp, dst, mode, diag_add);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_unpack(Handle *h, int rows, int cols, const double *src, long long lds_src, double *dst, long long ldd,
                  int mode, double diag_add) {
  if (rows <= 0 || cols <= 0) return 0;
  dim3 grid((rows + 255) / 256, cols);
  ProfScope ps__(h, PC_OTHER);
  unpack_kernel<<<grid, 256, 0, h->stream>>>(rows, cols, src, lds_src, dst, ldd, mode, diag_add);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_phi_lower(Handle *h, int np, double *A, long long stride, int batch) {
  dim3 grid((np + 255) / 256, np, batch);
  ProfScope ps__(h, PC_OTHER);
  phi_lower_kernel<<<grid, 256, 0, h->stream>>>(np, A, stride);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_gemv_t(Handle *h, int rows, int cols, const double *V, long long ldv, const double *z, const double *add,
                  double *out) {
  ProfScope ps__(h, PC_SOLVE);
  gemv_t_kernel<<<(cols + 7) / 8, 256, 0, h->stream>>>(rows, cols, V, ldv, z, add, out);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_hermite(Handle *h, long long len, int n, const double *y1, const double *y2, const double *k1,
                   const double *k2, double x1, double x2, double l, double *v, double *dvdl) {
  const int blocks = (int)((len + 255) / 256 > 148 * 8 ? 148 * 8 : (len + 255) / 256);
  ProfScope ps__(h, PC_OTHER);
  hermite_kernel<<<blocks, 256, 0, h->stream>>>(len, n, y1, y2, k1, k2, x1, x2, l, v, dvdl);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

}  // namespace gpb

namespace gpb {
int hermite_matvec_chunks(int n) { return std::max(1, std::min(64, (2 * 148 * 128 + n - 1) / std::max(n, 1))); }

int launch_hermite_matvec(Handle *h, int n, const double *y1, const double *y2, const double *k1, const double *k2, double x1,
                          double x2, double l, const double *z, double *part, double *vz, double *dvz) {
  const int nchunk = hermite_matvec_chunks(n);
  ProfScope ps__(h, PC_SOLVE);
  dim3 grid((n + 127) / 128, nchunk);
  hermite_matvec_kernel<<<grid, 128, 0, h->stream>>>(n, y1, y2, k1, k2, x1, x2, l, z, part);
  GPB_LAUNCH_CHECK(h);
  hermite_matvec_reduce_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(n, nchunk, part, vz, dvz);
  GPB_LAUNCH_CHECK(h);
  return 0;
}
}  // namespace gpb
