// Whole-evaluation kernel for small problems (n <= 128): one CTA computes the LML and its gradient for one item with
// the matrix resident in shared memory from the Gram build to the trace contraction -- nothing O(n^2) touches HBM.
//
// This is config 1 of BASELINE.json (exact GP, N = 100: models/exact_gp.stan / test_interpolate.R:5-7 sizes) and the
// per-leapfrog call of the Stan seam at such sizes.  The tiled path pads n = 100 to a 128 tile and walks the general
// schedule (Gram, POTRF tile, tile inverse, two mat-vecs, LAUUM + trace, finalize: seven launches, 100 us); here it is
// one launch, two CTAs per SM (90 KB each at n = 100).
//
// Reference semantics (models/fit_hyperparameters.stan:18-31 and its reverse sweep):
//   K = cov_exp_quad(x, alpha, rho) + (sigma^2 + jitter) I ;  L = cholesky_decompose(K) ;  y ~ multi_normal_cholesky(0, L)
//   d lml / d theta = 0.5 tr((a a^T - K^-1) dK/dtheta),  a = K^-1 y
//
// Layout: n8 = n rounded up to 8, one column-major array T[n8][ld], ld = n8 + 4 (== 4 or 12 mod 16: mma fragment
// reads are bank-conflict free).  The lower triangle holds K, then L; X = L^-T (upper triangular) is written into the
// strict upper triangle, its diagonal into invd[]; K^-1 = X X^T is never stored: its 8x8 blocks go from the DMMA
// accumulators straight into the trace sums.
#include "common.cuh"
#include "fastexp.cuh"
#include "gram.cuh"
#include "panel_ll.cuh"

namespace gpb {

constexpr int SMALL_MAX_N = 128;

__device__ __forceinline__ void dmma884s(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c[0]), "+d"(c[1])
               : "d"(a), "d"(b));
}

__device__ __forceinline__ double warp_sum_s(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// RAGGED: item b has its own size nvec[b] <= n8 (gpb200_lml_grad_ragged); rows and columns from it to n8 are identity
template <bool RAGGED>
__global__ void __launch_bounds__(256, 2)
lml_small_kernel(int n_all, int n8, const double *__restrict__ x, long long x_stride, const double *__restrict__ y,
                 long long y_stride, const double *__restrict__ theta, double jitter, int want_grad,
                 double *__restrict__ lml, double *__restrict__ grad, int *__restrict__ info, const int *__restrict__ nvec) {
  const int n = RAGGED ? nvec[blockIdx.x] : n_all;
  extern __shared__ __align__(16) double sm[];
  const int ld = n8 + 4, nb = n8 >> 3;
  double *T = sm;                          // T[c * ld + r]
  double *xs = T + (size_t)n8 * ld;        // inputs
  double *ys = xs + SMALL_MAX_N;
  double *invd = ys + SMALL_MAX_N;         // 1 / L[i][i]  (= diagonal of X)
  double *zs = invd + SMALL_MAX_N;         // z = L^-1 y
  double *as = zs + SMALL_MAX_N;           // a = K^-1 y
  double *Dsm = as + SMALL_MAX_N;          // 64: the diagonal block being factored
  double *XD = Dsm + 64;                   // 8 warps x 2 row blocks x 64: full 8x8 diagonal blocks of X
  double *red = XD + 8 * 2 * 64;           // 8 warps x 8 reduction slots
  __shared__ int s_info;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const long long b = blockIdx.x;
  const double alpha = theta[b * 3 + 0], rho = theta[b * 3 + 1], sigma = theta[b * 3 + 2];
  const double a2 = alpha * alpha, nh = -0.5 / (rho * rho), dadd = sigma * sigma + jitter;

  if (tid == 0) s_info = 0;
  if (tid < SMALL_MAX_N) {
    xs[tid] = (tid < n) ? x[b * x_stride + tid] : 0.0;
    ys[tid] = (tid < n) ? y[b * y_stride + tid] : 0.0;
  }
  __syncthreads();

  // ---- 1. Gram, lower triangle + diagonal; identity in the padding ------------------------------------------
  for (int idx = tid; idx < n8 * n8; idx += 256) {
    const int j = idx / n8, i = idx - j * n8;
    if (i < j) continue;
    double v;
    if (i < n && j < n) {
      const double d = xs[i] - xs[j];
      v = (i == j) ? a2 + dadd : a2 * exp_nonpos(d * d * nh);
    } else {
      v = (i == j) ? 1.0 : 0.0;
    }
    T[j * ld + i] = v;
  }
  __syncthreads();

  // ---- 2. left-looking Cholesky over 8-column blocks; warp w owns row blocks w and w + 8 --------------------
#pragma unroll 1
  for (int cb = 0; cb < nb; cb++) {
    const int c0 = 8 * cb;
    if (cb > 0) {
      double s[2][2][2];
#pragma unroll
      for (int mt = 0; mt < 2; mt++)
#pragma unroll
        for (int ch = 0; ch < 2; ch++) s[mt][ch][0] = s[mt][ch][1] = 0.0;
      const bool m0 = warp >= cb && warp < nb, m1 = (warp + 8) >= cb && (warp + 8) < nb;
      if (m0 || m1) {
        const double *pa = T + t * ld + 8 * warp + g;
        const double *pb = T + t * ld + c0 + g;
        for (int kb = 0; kb < cb; kb++) {
#pragma unroll
          for (int ch = 0; ch < 2; ch++) {
            const int ko = (8 * kb + 4 * ch) * ld;
            const double bv = pb[ko];
            if (m0) dmma884s(s[0][ch], pa[ko], bv);
            if (m1) dmma884s(s[1][ch], pa[ko + 64], bv);
          }
        }
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
          if (!(mt ? m1 : m0)) continue;
#pragma unroll
          for (int e = 0; e < 2; e++) {
            double *p = T + (c0 + 2 * t + e) * ld + 8 * (warp + 8 * mt) + g;
            *p = (*p - s[mt][0][e]) - s[mt][1][e];
          }
        }
      }
    }
    if (warp == (cb & 7)) {  // owner of the diagonal block publishes it apart from the tile (see potrf_tile_ll_kernel)
      __syncwarp();
#pragma unroll
      for (int e = 0; e < 2; e++) Dsm[(2 * t + e) * 8 + g] = T[(c0 + 2 * t + e) * ld + c0 + g];
    }
    __syncthreads();
    {
      const int rb = warp + 8 * (lane >> 3);  // lanes 0-7: row block `warp`, lanes 8-15: row block `warp + 8`
      const bool any = (warp >= cb && warp < nb) || ((warp + 8) >= cb && (warp + 8) < nb);
      if (any) {
        double d[8][8], inv[8];
#pragma unroll
        for (int j = 0; j < 8; j++)
#pragma unroll
          for (int i = j; i < 8; i++) d[i][j] = Dsm[j * 8 + i];
        int bad;
        factor8_pairs(d, inv, bad);
        if (bad >= 0 && warp == (cb & 7) && lane == 0 && s_info == 0) s_info = c0 + bad + 1;
        if (lane < 16 && rb >= cb && rb < nb) {
          const int r = 8 * rb + (lane & 7);
          double xv[8];
#pragma unroll
          for (int c = 0; c < 8; c++) xv[c] = T[(c0 + c) * ld + r];
#pragma unroll
          for (int c = 0; c < 8; c++) {
            double sv = xv[c];
#pragma unroll
            for (int cp = 0; cp < c; cp++) sv = fma(-xv[cp], d[c][cp], sv);
            xv[c] = sv * inv[c];
          }
          const int i = r - c0;
#pragma unroll
          for (int c = 0; c < 8; c++)
            if (!(i < 8 && c > i)) T[(c0 + c) * ld + r] = xv[c];   // the strict upper part is not L's: leave it alone
        }
      }
    }
    __syncthreads();
  }
  if (tid < SMALL_MAX_N) invd[tid] = (tid < n8) ? 1.0 / T[tid * ld + tid] : 0.0;
  double logdet = 0.0;
  if (tid < n) logdet = log(T[tid * ld + tid]);
  __syncthreads();
  if (!want_grad) {
    // ---- LML only: forward substitution z = L^-1 y, one 8-row block at a time (warp 0) -----------------------
    if (warp == 0) {
      for (int rb = 0; rb < nb; rb++) {
        const int r0 = 8 * rb;
        // s[i] = y[r0 + i] - sum_{k < r0} L[r0 + i][k] z[k]: lane = (i, k-slice)
        const int i = lane & 7, ks = lane >> 3;
        double sv = 0.0;
        for (int k = ks; k < r0; k += 4) sv = fma(T[k * ld + r0 + i], zs[k], sv);
        sv += __shfl_xor_sync(0xffffffffu, sv, 8);
        sv += __shfl_xor_sync(0xffffffffu, sv, 16);
        double rhs = ys[r0 + i] - sv;
        // 8-step substitution inside the block; lane i < 8 ends up with z[r0 + i]
        double zi = 0.0;
#pragma unroll
        for (int c = 0; c < 8; c++) {
          const double zc = __shfl_sync(0xffffffffu, rhs, c) * invd[r0 + c];   // rhs of lane c is final at step c
          if (i == c) zi = zc;
          if (i > c) rhs = fma(-T[(r0 + c) * ld + r0 + i], zc, rhs);
        }
        if (lane < 8) zs[r0 + i] = zi;
        __syncwarp();
      }
    }
    __syncthreads();
  } else {
    // ---- 3. X = L^-T, rows independent: each warp takes row blocks rb = warp and nb - 1 - warp ------------------
#pragma unroll 1
    for (int slot = 0; slot < 2; slot++) {
      // slot 0: block `warp` (lower half and the middle), slot 1: its mirror nb - 1 - warp (upper half): long and
      // short rows of the triangle are paired, every block is taken exactly once
      const int rb = slot == 0 ? warp : nb - 1 - warp;
      if (slot == 0 ? (warp > nb - 1 - warp) : (nb - 1 - warp <= warp)) continue;
      const int r0 = 8 * rb;
      double *xd = XD + (warp * 2 + slot) * 64;       // xd[k * 8 + i] = X[r0 + i][r0 + k]
#pragma unroll 1
      for (int cb = rb; cb < nb; cb++) {
        const int c0 = 8 * cb;
        if (cb > rb) {
          double s[2][2];
          s[0][0] = s[0][1] = s[1][0] = s[1][1] = 0.0;
          const double *pb = T + t * ld + c0 + g;
          for (int kb = rb; kb < cb; kb++) {
#pragma unroll
            for (int ch = 0; ch < 2; ch++) {
              const double bv = pb[(8 * kb + 4 * ch) * ld];
              const double av = (kb == rb) ? xd[(4 * ch + t) * 8 + g] : T[(8 * kb + 4 * ch + t) * ld + r0 + g];
              dmma884s(s[ch], av, bv);
            }
          }
#pragma unroll
          for (int e = 0; e < 2; e++) T[(c0 + 2 * t + e) * ld + r0 + g] = -(s[0][e] + s[1][e]);   // P = 0 - sum
          __syncwarp();
        }
        if (lane < 8) {
          const int i = lane, r = r0 + i;
          double xv[8];
#pragma unroll
          for (int c = 0; c < 8; c++) xv[c] = (cb == rb) ? ((c == i) ? 1.0 : 0.0) : T[(c0 + c) * ld + r];
#pragma unroll
          for (int c = 0; c < 8; c++) {
            double sv = xv[c];
#pragma unroll
            for (int cp = 0; cp < c; cp++) sv = fma(-xv[cp], T[(c0 + cp) * ld + c0 + c], sv);
            xv[c] = sv * invd[c0 + c];
          }
          if (cb == rb) {
#pragma unroll
            for (int c = 0; c < 8; c++) {
              xd[c * 8 + i] = (c >= i) ? xv[c] : 0.0;
              if (c > i) T[(c0 + c) * ld + r] = xv[c];
            }
          } else {
#pragma unroll
            for (int c = 0; c < 8; c++) T[(c0 + c) * ld + r] = xv[c];
          }
        }
        __syncwarp();
      }
    }
    __syncthreads();
    // L is no longer needed: make the diagonal blocks of T hold X's (zeros below, 1/L_ii on the diagonal)
    for (int idx = tid; idx < nb * 64; idx += 256) {
      const int rb = idx >> 6, c = (idx >> 3) & 7, i = idx & 7;
      if (c < i) T[(8 * rb + c) * ld + 8 * rb + i] = 0.0;
      else if (c == i) T[(8 * rb + c) * ld + 8 * rb + i] = invd[8 * rb + i];
    }
    __syncthreads();
    // ---- 4. z = X^T y (= L^-1 y), a = X z (= K^-1 y) -------------------------------------------------------------
    for (int i = warp; i < n8; i += 8) {     // z[i] = sum_{k <= i} X[k][i] y[k]: column i of T, contiguous in k
      double sv = 0.0;
      for (int k = lane; k <= i; k += 32) sv = fma(T[i * ld + k], ys[k], sv);
      sv = warp_sum_s(sv);
      if (lane == 0) zs[i] = sv;
    }
    __syncthreads();
    if (tid < n8) {                          // a[r] = sum_{c >= r} X[r][c] z[c]: consecutive threads, consecutive rows
      double sv = 0.0;
      for (int c = tid; c < n8; c++) sv = fma(T[c * ld + tid], zs[c], sv);
      as[tid] = sv;
    }
    __syncthreads();
  }

  // ---- 5. K^-1 = X X^T block by block, fused with the trace contraction -----------------------------------------
  double s_se = 0.0, s_d2 = 0.0, s_tr = 0.0;
  if (want_grad) {
    const int ntask = nb * (nb + 1) / 2;
    for (int task = warp; task < ntask; task += 8) {
      // task -> (I, J), J <= I, enumerated row by row (small I = long contraction first)
      int I = 0, rem = task;
      while (rem > I) { rem -= I + 1; I++; }
      const int J = rem;
      double c2[2][2];
      c2[0][0] = c2[0][1] = c2[1][0] = c2[1][1] = 0.0;
      const double *pa = T + t * ld + 8 * I + g, *pb = T + t * ld + 8 * J + g;
      for (int kb = I; kb < nb; kb++) {
#pragma unroll
        for (int ch = 0; ch < 2; ch++) {
          const int ko = (8 * kb + 4 * ch) * ld;
          dmma884s(c2[ch], pa[ko], pb[ko]);
        }
      }
      const double wgt = (I == J) ? 1.0 : 2.0;
      const int i = 8 * I + g;
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int j = 8 * J + 2 * t + e;
        const double G = c2[0][e] + c2[1][e];
        if (i < n && j < n) {
          const double d = xs[i] - xs[j], d2 = d * d;
          const double ek = exp_nonpos(d2 * nh);
          const double M = as[i] * as[j] - G;
          s_se += wgt * M * ek;
          s_d2 += wgt * M * ek * d2;
          if (i == j) s_tr += G;
        }
      }
    }
  }
  // ---- 6. reductions and the result ---------------------------------------------------------------------------
  double qf = 0.0, aa = 0.0;
  if (tid < n) {
    qf = zs[tid] * zs[tid];
    if (want_grad) aa = as[tid] * as[tid];
  }
  logdet = warp_sum_s(logdet); qf = warp_sum_s(qf); aa = warp_sum_s(aa);
  s_se = warp_sum_s(s_se); s_d2 = warp_sum_s(s_d2); s_tr = warp_sum_s(s_tr);
  if (lane == 0) {
    red[warp * 8 + 0] = logdet; red[warp * 8 + 1] = qf; red[warp * 8 + 2] = aa;
    red[warp * 8 + 3] = s_se; red[warp * 8 + 4] = s_d2; red[warp * 8 + 5] = s_tr;
  }
  __syncthreads();
  if (tid == 0) {
    double r[6] = {0, 0, 0, 0, 0, 0};
    for (int w = 0; w < 8; w++)
      for (int q = 0; q < 6; q++) r[q] += red[w * 8 + q];
    lml[b] = -0.5 * n * 1.8378770664093454835606594728112 - r[0] - 0.5 * r[1];
    if (want_grad) {
      grad[b * 3 + 0] = alpha * r[3];
      grad[b * 3 + 1] = 0.5 * a2 * r[4] / (rho * rho * rho);
      grad[b * 3 + 2] = sigma * (r[2] - r[5]);
    }
    info[b] = (s_info != 0 && s_info <= n) ? s_info : 0;   // always written: the caller needs no memset
  }
}

static size_t small_smem_bytes(int n8) {
  return ((size_t)n8 * (n8 + 4) + 5 * SMALL_MAX_N + 64 + 8 * 2 * 64 + 64) * sizeof(double);
}

int small_smem_setup(Handle *h) {
  GPB_CUDA(h, cudaFuncSetAttribute(lml_small_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_smem_bytes(SMALL_MAX_N)));
  GPB_CUDA(h, cudaFuncSetAttribute(lml_small_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_smem_bytes(SMALL_MAX_N)));
  return 0;
}

bool lml_small_applies(const Handle *h, int n) { return h->small_kernel && n <= SMALL_MAX_N; }

int launch_lml_small(Handle *h, int n, const double *x, long long x_stride, const double *y, long long y_stride,
                     const double *theta, double jitter, int want_grad, double *lml, double *grad, int *info, int batch,
                     const int *nvec) {
  const int n8 = round_up(n, 8);
  ProfScope ps__(h, PC_OTHER);
  if (nvec)
    lml_small_kernel<true><<<batch, 256, small_smem_bytes(n8), h->stream>>>(n, n8, x, x_stride, y, y_stride, theta, jitter,
                                                                           want_grad, lml, grad, info, nvec);
  else
    lml_small_kernel<false><<<batch, 256, small_smem_bytes(n8), h->stream>>>(n, n8, x, x_stride, y, y_stride, theta, jitter,
                                                                            want_grad, lml, grad, info, nullptr);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

}  // namespace gpb
