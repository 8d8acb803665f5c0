// C-ABI entry points for the NON-CENTRED LATENT models (SURVEY CS-E, row f-2): models/exact_gp.stan:17-25,
// fit_full_gp.stan:18-26, westbrook_exact.stan:17-24 (one mat-vec f = L z) and heteroscedastic.stan:23-32 (two
// mat-vecs on one L).  Stan differentiates THROUGH cholesky_decompose; this is that reverse sweep as one pass:
//
//   forward   K = cov_exp_quad(x, alpha, rho) + diag_add I ;  L = chol(K) ;  f_m = L z_m
//   backward  given fbar_m:   zbar_m = u_m = L^T fbar_m
//             Lbar = sum_m tril(fbar_m z_m^T)                         (adjoint of the mat-vecs)
//             P    = Phi(L^T Lbar) = Phi(sum_m u_m z_m^T)             (Phi: lower triangle, diagonal halved)
//             Kbar = L^-T P L^-1 = W^T (P W),  W = L^-1               (adjoint of the Cholesky)
//             thetabar = sum_ij Kbar_ij dK_ij/dtheta                  (adjoint of cov_exp_quad)
// P W needs no GEMM: (P W)_ik = sum_m u_m,i * (sum_{k<=j<i} z_m,j W_jk + z_m,i W_ik / 2) is a running sum down each column
// of diag(z) W.  So the pass is one triangular inverse (N^3/3) and ONE tile GEMM W^T (P W) whose tiles go straight from
// the accumulators into the contraction with dK/dtheta (recomputed from x): N^3 in total for ALL parameters, where the
// forward-mode route (gpb200_se_chol_tangent) costs 5 N^3 / 3 per parameter.
#include "host.cuh"

using namespace gpb;

namespace {
enum { TK_LATENT_G = 60 };

unsigned long long hash_doubles(const double *x, int n) {   // FNV-1a over the bytes of a HOST array
  unsigned long long hsh = 1469598103934665603ULL;
  const unsigned char *b = reinterpret_cast<const unsigned char *>(x);
  for (size_t i = 0; i < (size_t)n * 8; i++) { hsh ^= b[i]; hsh *= 1099511628211ULL; }
  return hsh;
}

// T[i][k] (+)= u_i * (sum_{k <= j < i} z_j W[j][k] + z_i W[i][k] / 2) for i >= k; zero above the diagonal.
// One warp per column k; 32 rows at a time with a shuffle prefix sum: reads of W are contiguous along the column.
// blockIdx.y = item b: W and T at b * w_stride, u and z at b * v_stride.
__global__ void __launch_bounds__(256) latent_pw_kernel(int np, const double *__restrict__ W, long long w_stride,
                                                        const double *__restrict__ u, const double *__restrict__ z,
                                                        long long v_stride, int accumulate, double *__restrict__ T) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k = blockIdx.x * 8 + warp;
  if (k >= np) return;
  const long long b = blockIdx.y;
  u += b * v_stride;
  z += b * v_stride;
  const double *wc = W + b * w_stride + (long long)k * np;
  double *tc = T + b * w_stride + (long long)k * np;
  const int i0 = k & ~31;
  for (int i = lane; i < i0; i += 32)
    if (!accumulate) tc[i] = 0.0;
  double carry = 0.0;
  for (int base = i0; base < np; base += 32) {
    const int i = base + lane;
    const double v = (i >= k) ? z[i] * wc[i] : 0.0;
    double incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const double val = (i >= k) ? u[i] * (carry + (incl - v) + 0.5 * v) : 0.0;
    tc[i] = accumulate ? tc[i] + val : val;
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
}

// One CTA per item (blockIdx.x): the item's nrec partial records of the trace epilogue, summed in a fixed order.
// theta == nullptr: out2[2 b ..] = the two sums (the single-item call finishes on the host).  Otherwise out2[2 b ..] =
// theta_bar_b = (-2 alpha r0, -alpha^2 r1 / rho^3) from theta (B x 3), NaN when info[b] != 0.
__global__ void __launch_bounds__(256) latent_sum_kernel(long long nrec, const double *__restrict__ partial,
                                                         const double *__restrict__ theta, const int *__restrict__ info,
                                                         double *__restrict__ out2) {
  __shared__ double red[8][2];
  const long long item = blockIdx.x;
  partial += item * nrec * 4;
  double s0 = 0, s1 = 0;
  for (long long r = threadIdx.x; r < nrec; r += 256) { s0 += partial[r * 4]; s1 += partial[r * 4 + 1]; }
  for (int o = 16; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = s0; red[threadIdx.x >> 5][1] = s1; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int w = 0; w < 8; w++) { a += red[w][0]; b += red[w][1]; }
    if (!theta) {
      out2[2 * item] = a; out2[2 * item + 1] = b;
    } else if (info[item]) {
      out2[2 * item] = out2[2 * item + 1] = __longlong_as_double(0x7ff8000000000000LL);
    } else {
      // the epilogue accumulated M = 0 - G: Kbar contracted with e and e d^2 is minus those sums (the same expression
      // as the single-item call's host code, so that B = 1 gives the same bits)
      const double alpha = theta[3 * item], rho = theta[3 * item + 1];
      out2[2 * item] = -2.0 * alpha * a;
      out2[2 * item + 1] = -alpha * alpha * b / (rho * rho * rho);
    }
  }
}

// dst[v n + i] = src[v np + i] for the nv vectors v of length n (item v / nvec), NaN for every i of an item whose
// info != 0: the batched calls' f and zbar out of their padded buffers
__global__ void latent_rows_kernel(int n, int np, int nvec, long long nv, const double *__restrict__ src,
                                   const int *__restrict__ info, double *__restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (long long v = blockIdx.y; v < nv; v += gridDim.y)
    dst[v * n + i] = info[v / nvec] ? __longlong_as_double(0x7ff8000000000000LL) : src[v * np + i];
}

int launch_latent_rows(Handle *h, int n, int np, int nvec, long long nv, const double *src, const int *info, double *dst) {
  dim3 grid((n + 255) / 256, (unsigned)std::min<long long>(nv, 65535));
  ProfScope ps__(h, PC_OTHER);
  latent_rows_kernel<<<grid, 256, 0, h->stream>>>(n, np, nvec, nv, src, info, dst);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// TK_LATENT_G: every tile pair (I, J) of W^T T, the upper ones included, each contracted from max(I, J) down
int latent_tasks(Handle *h, int nt, TaskList *tl) {
  const long long key = tkey(TK_LATENT_G, nt);
  if (cached(h, key, tl)) return 0;
  std::vector<TileTask> t;
  for (int I = 0; I < nt; I++)
    for (int J = 0; J < nt; J++) {
      const int k0 = std::max(I, J);   // W[k][I] = 0 for k < I, (P W)[k][J] = 0 for k < J
      t.push_back({k0 * TILE, I * TILE, k0 * TILE, J * TILE, I * TILE, J * TILE, (nt - k0) * TILE,
                   TF_FULL_WEIGHT | (I >= J ? TF_A_TRI_FIRST : 0) | (J >= I ? TF_B_TRI_FIRST : 0)});
    }
  sort_desc(t, 0);
  std::vector<int> off = {0, (int)t.size()};
  return upload_tasks(h, key, t, off, tl);
}

// The record of gpb200_latent_forward_batched, carved from h->latent_rec: B padded factors, the z vectors zero-padded
// to np, x (one vector when shared), theta as B x 3 (alpha, rho, 0) and the per-item info.
struct LatentRecord {
  double *L, *z, *x, *theta;
  int *info;
};
size_t latent_record_bytes(int n, int B, int nvec, long long xs) {
  const size_t np = (size_t)round_up(n, TILE);
  return pad256((size_t)B * np * np * 8) + pad256((size_t)B * nvec * np * 8) + pad256((size_t)(xs ? B : 1) * n * 8) +
         pad256((size_t)B * 3 * 8) + pad256((size_t)B * 4);
}
LatentRecord latent_record(Handle *h, int n, int B, int nvec, long long xs) {
  const size_t np = (size_t)round_up(n, TILE);
  Arena r;
  r.base = reinterpret_cast<char *>(h->latent_rec);
  r.cap = h->latent_rec_bytes;
  LatentRecord rec;
  rec.L = r.take<double>((size_t)B * np * np);
  rec.z = r.take<double>((size_t)B * nvec * np);
  rec.x = r.take<double>((size_t)(xs ? B : 1) * n);
  rec.theta = r.take<double>((size_t)B * 3);
  rec.info = r.take<int>(B);
  return rec;
}

// builds (or finds cached) the padded factor of K = cov_exp_quad(x, alpha, rho) + diag_add I; returns LAPACK info
int latent_factor(Handle *h, int n, const double *x, double alpha, double rho, double diag_add, int *info_out) {
  const int np = round_up(n, TILE);
  const size_t bytes = (size_t)np * np * 8;
  const unsigned long long xh = h->device_ptrs ? (unsigned long long)(uintptr_t)x : hash_doubles(x, n);
  if (h->latent_L && h->latent_n == n && h->latent_key[0] == alpha && h->latent_key[1] == rho && h->latent_key[2] == diag_add &&
      h->latent_xhash == xh && !h->device_ptrs) {
    *info_out = 0;
    return 0;
  }
  if (h->latent_bytes < bytes) {
    if (h->latent_L) { GPB_CUDA(h, cudaStreamSynchronize(h->stream)); GPB_CUDA(h, cudaFree(h->latent_L)); h->latent_L = nullptr; }
    GPB_CUDA(h, cudaMalloc(&h->latent_L, bytes));
    h->latent_bytes = bytes;
  }
  h->latent_n = 0;
  Arena a;
  RC(ws_reserve(h, pad256(n * 8) + 1024, &a));
  double *dx = a.take<double>(n), *dth = a.take<double>(3);
  int *info = a.take<int>(1);
  RC(to_device(h, x, dx, n));
  const double th[3] = {alpha, rho, 0.0};
  GPB_CUDA(h, cudaMemcpyAsync(dth, th, sizeof(th), cudaMemcpyHostToDevice, h->stream));
  GPB_CUDA(h, cudaMemsetAsync(info, 0, sizeof(int), h->stream));
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  RC(launch_gram_se_batched(h, n, np, dx, 0, dth, diag_add, 1, h->latent_L, 0, 1));
  RC(chol_batched(h, h->latent_L, np, (long long)np * np, n, 1, info));
  RC(read_info(h, info, info_out));
  if (*info_out == 0) {
    h->latent_n = n;
    h->latent_key[0] = alpha; h->latent_key[1] = rho; h->latent_key[2] = diag_add;
    h->latent_xhash = xh;
  }
  return 0;
}
}  // namespace

// f_m = L z_m for m = 0..nvec-1 (z, f: nvec vectors of length n, consecutive).  L = chol(cov_exp_quad(x, alpha, rho) +
// diag_add I) is kept on the device for gpb200_latent_backward.
extern "C" int gpb200_latent_forward(gpb200_handle_t h, int n, const double *x, double alpha, double rho, double diag_add, int nvec,
                                     const double *z, double *f) {
  CHECK_H(h);
  if (n < 1 || nvec < 1) BAD_ARG(h, 2, "latent_forward: n and nvec must be >= 1");
  int info = 0;
  RC(latent_factor(h, n, x, alpha, rho, diag_add, &info));
  if (info) return info;
  const int np = round_up(n, TILE);
  Arena a;
  RC(ws_reserve(h, 2 * pad256((size_t)np * 8 * nvec) + 1024, &a));
  double *dz = a.take<double>((size_t)np * nvec), *df = a.take<double>((size_t)np * nvec);
  for (int m = 0; m < nvec; m++) {
    RC(to_device(h, z + (size_t)m * n, dz + (size_t)m * np, n));
    RC(launch_trmv_lower_n(h, np, h->latent_L, 0, dz + (size_t)m * np, 0, n, df + (size_t)m * np, 0, 1));
    RC(from_device(h, df + (size_t)m * np, f + (size_t)m * n, n * sizeof(double)));
  }
  return finish(h);
}

// Reverse sweep: given fbar_m = d lp / d f_m, returns zbar_m = L^T fbar_m (nvec x n) and
// theta_bar = (d lp / d alpha, d lp / d rho) THROUGH f_m = L z_m and the Cholesky.
extern "C" int gpb200_latent_backward(gpb200_handle_t h, int n, const double *x, double alpha, double rho, double diag_add, int nvec,
                                      const double *z, const double *fbar, double *theta_bar, double *zbar) {
  CHECK_H(h);
  if (n < 1 || nvec < 1) BAD_ARG(h, 2, "latent_backward: n and nvec must be >= 1");
  int info = 0;
  RC(latent_factor(h, n, x, alpha, rho, diag_add, &info));
  if (info) return info;
  const int np = round_up(n, TILE), nt = np / TILE;
  const size_t mat = (size_t)np * np;
  TaskList tl;
  RC(latent_tasks(h, nt, &tl));
  const int ntasks = tl.count(0);
  Arena a;
  RC(ws_reserve(h, 3 * pad256(mat * 8) + (3 * (size_t)nvec + 2) * pad256((size_t)np * 8) + pad256((size_t)ntasks * 4 * 4 * 8) + 4096, &a));
  double *W = a.take<double>(mat), *S = a.take<double>(mat), *T = a.take<double>(mat);
  double *dz = a.take<double>((size_t)np * nvec), *dfb = a.take<double>((size_t)np * nvec), *du = a.take<double>((size_t)np * nvec);
  double *dx = a.take<double>(np), *zero = a.take<double>(np), *dth = a.take<double>(3), *out2 = a.take<double>(2);
  double *partial = a.take<double>((size_t)ntasks * 4 * 4);
  if (!partial) BAD_ARG(h, 1002, "latent_backward: workspace exhausted");
  GPB_CUDA(h, cudaMemsetAsync(dz, 0, sizeof(double) * np * nvec, h->stream));
  GPB_CUDA(h, cudaMemsetAsync(dfb, 0, sizeof(double) * np * nvec, h->stream));
  GPB_CUDA(h, cudaMemsetAsync(zero, 0, sizeof(double) * np, h->stream));
  GPB_CUDA(h, cudaMemsetAsync(dx, 0, sizeof(double) * np, h->stream));
  RC(to_device(h, x, dx, n));
  const double th[3] = {alpha, rho, 0.0};
  GPB_CUDA(h, cudaMemcpyAsync(dth, th, sizeof(th), cudaMemcpyHostToDevice, h->stream));
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  GPB_CUDA(h, cudaMemcpyAsync(W, h->latent_L, mat * 8, cudaMemcpyDeviceToDevice, h->stream));
  RC(trtri_batched(h, W, S, np, (long long)mat, 1));
  for (int m = 0; m < nvec; m++) {
    RC(to_device(h, z + (size_t)m * n, dz + (size_t)m * np, n));
    RC(to_device(h, fbar + (size_t)m * n, dfb + (size_t)m * np, n));
    RC(launch_trmv_lower_t(h, np, h->latent_L, 0, dfb + (size_t)m * np, 0, du + (size_t)m * np, 0, 1));   // u = zbar = L^T fbar
    ProfScope ps__(h, PC_SOLVE);
    latent_pw_kernel<<<(np + 7) / 8, 256, 0, h->stream>>>(np, W, 0, du + (size_t)m * np, dz + (size_t)m * np, 0, m > 0, T);
    GPB_LAUNCH_CHECK(h);
    RC(from_device(h, du + (size_t)m * np, zbar + (size_t)m * n, n * sizeof(double)));
  }
  GemmParams p{};
  p.A = mref(W, np, 0);
  p.B = mref(T, np, 0);
  p.C = mref(nullptr, np, 0);
  p.tasks = tl.at(0);
  p.x = dx; p.x_stride = 0;
  p.avec = zero; p.a_stride = 0;
  p.theta = dth;
  p.partial = partial;
  p.n = n;
  p.ntasks = ntasks;
  RC(launch_gemm(h, LAYOUT_TN, EPI_TRACE, p, ntasks, 1));
  {
    ProfScope ps__(h, PC_OTHER);
    latent_sum_kernel<<<1, 256, 0, h->stream>>>((long long)ntasks * gemm_nsplit(h, ntasks, 1), partial, nullptr, nullptr, out2);
    GPB_LAUNCH_CHECK(h);
  }
  double r[2];
  GPB_CUDA(h, cudaMemcpyAsync(r, out2, sizeof(r), cudaMemcpyDeviceToHost, h->stream));
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  // the epilogue accumulated M = 0 - G: Kbar contracted with e and e d^2 is minus those sums
  const double tb[2] = {-2.0 * alpha * r[0], -alpha * alpha * r[1] / (rho * rho * rho)};
  if (h->device_ptrs) {
    GPB_CUDA(h, cudaMemcpyAsync(theta_bar, tb, sizeof(tb), cudaMemcpyHostToDevice, h->stream));
    GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  } else {
    theta_bar[0] = tb[0];
    theta_bar[1] = tb[1];
  }
  return 0;
}

// ---- B parameter states in one call ----------------------------------------------------------------------------------
// The forward call keeps a record on the handle (h->latent_rec, grow-only, outside the workspace): all B factors and
// copies of x, theta and z, so the caller may reuse its buffers before the backward call and nothing has to be keyed or
// hashed.  A call that fails for any reason leaves no record.  Nothing synchronises the host in device-pointer mode
// (except a first call that grows the record or the workspace).
extern "C" int gpb200_latent_forward_batched(gpb200_handle_t h, int n, int B, int nvec, const double *x, long long x_stride,
                                             const double *theta, double diag_add, const double *z, double *f, int *info) {
  CHECK_H(h);
  h->latent_rec_valid = 0;
  if (n < 1) BAD_ARG(h, 2, "latent_forward_batched: n must be >= 1");
  if (B < 1) BAD_ARG(h, 3, "latent_forward_batched: B must be >= 1");
  if (nvec < 1) BAD_ARG(h, 4, "latent_forward_batched: nvec must be >= 1");
  if ((long long)B * nvec > 2147483647LL) BAD_ARG(h, 4, "latent_forward_batched: B * nvec too large");
  if (!x) BAD_ARG(h, 5, "latent_forward_batched: x is NULL");
  if (x_stride != 0 && x_stride < n) BAD_ARG(h, 6, "latent_forward_batched: x_stride < n");
  if (!theta) BAD_ARG(h, 7, "latent_forward_batched: theta is NULL");
  if (!z) BAD_ARG(h, 9, "latent_forward_batched: z is NULL");
  if (!f) BAD_ARG(h, 10, "latent_forward_batched: f is NULL");
  if (!info) BAD_ARG(h, 11, "latent_forward_batched: info is NULL");
  const int np = round_up(n, TILE);
  const long long mat = (long long)np * np, xs = x_stride ? n : 0, nv = (long long)B * nvec;
  const bool host = !h->device_ptrs;

  // every factor stays resident until the backward call: the record is allocated whole, never chunked
  const size_t rec_bytes = latent_record_bytes(n, B, nvec, xs);
  if (h->latent_rec_bytes < rec_bytes) {
    if (h->latent_rec) {
      GPB_CUDA(h, cudaStreamSynchronize(h->stream));
      GPB_CUDA(h, cudaFree(h->latent_rec));
      h->latent_rec = nullptr;
      h->latent_rec_bytes = 0;
    }
    const cudaError_t e = cudaMalloc(&h->latent_rec, rec_bytes);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      h->latent_rec = nullptr;
      snprintf(h->err, sizeof(h->err),
               "latent_forward_batched: the record of %d factors of order %d (%zu bytes; all of them stay on the device until "
               "the backward call) could not be allocated: %s",
               B, np, rec_bytes, cudaGetErrorString(e));
      return -1002;
    }
    h->latent_rec_bytes = rec_bytes;
  }
  const LatentRecord rec = latent_record(h, n, B, nvec, xs);

  // padded f = L z (and, in host mode, f and info in the caller's layout before the copy out)
  const size_t need = pad256((size_t)nv * np * 8) + (host ? pad256((size_t)nv * n * 8) + pad256((size_t)B * 4) : 0) + 4096;
  if (h->ws_limit > 0 && need > (size_t)h->ws_limit)
    BAD_ARG(h, 1002, "latent_forward_batched: workspace limit too small for the mat-vec outputs");
  Arena a;
  RC(ws_reserve(h, need, &a));
  double *fpad = a.take<double>((size_t)nv * np);
  double *fout = host ? a.take<double>((size_t)nv * n) : f;
  if (!fout) BAD_ARG(h, 1002, "latent_forward_batched: workspace arithmetic error");

  if (x_stride) RC(to_device_2d(h, x, x_stride, rec.x, n, n, B)); else RC(to_device(h, x, rec.x, n));
  GPB_CUDA(h, cudaMemsetAsync(rec.theta, 0, (size_t)B * 3 * 8, h->stream));
  GPB_CUDA(h, cudaMemcpy2DAsync(rec.theta, 3 * sizeof(double), theta, 2 * sizeof(double), 2 * sizeof(double), B,
                                host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, h->stream));
  GPB_CUDA(h, cudaMemsetAsync(rec.z, 0, (size_t)nv * np * 8, h->stream));
  RC(to_device_2d(h, z, n, rec.z, np, n, (int)nv));
  GPB_CUDA(h, cudaMemsetAsync(rec.info, 0, (size_t)B * sizeof(int), h->stream));
  for (int b0 = 0; b0 < B; b0 += 65535) {  // gridDim.y of the batched launches
    const int bc = std::min(65535, B - b0);
    double *L = rec.L + (long long)b0 * mat;
    RC(launch_gram_se_batched(h, n, np, rec.x + (long long)b0 * xs, xs, rec.theta + 3LL * b0, diag_add, 1, L, mat, bc));
    RC(chol_batched(h, L, np, mat, n, bc, rec.info + b0));
    for (int m = 0; m < nvec; m++) {
      const long long off = ((long long)b0 * nvec + m) * np;
      RC(launch_trmv_lower_n(h, np, L, mat, rec.z + off, (long long)nvec * np, n, fpad + off, (long long)nvec * np, bc));
    }
  }
  RC(launch_latent_rows(h, n, np, nvec, nv, fpad, rec.info, fout));
  if (host) RC(from_device(h, fout, f, (size_t)nv * n * sizeof(double)));
  RC(from_device(h, rec.info, info, (size_t)B * sizeof(int)));
  RC(finish(h));
  h->latent_rec_n = n;
  h->latent_rec_B = B;
  h->latent_rec_nvec = nvec;
  h->latent_rec_xs = xs;
  h->latent_rec_valid = 1;
  return 0;
}

// Reverse sweep of the recorded batch, in chunks of items whose scratch (W = L^-1, T = sum_m P W in the trtri scratch,
// u = L^T fbar, fbar padded, the trace partials) fits the workspace limit.  Every kernel works per item, so the chunk
// size changes nothing but the GEMM configuration and Cholesky-inverse schedule the launches pick for their batch.
extern "C" int gpb200_latent_backward_batched(gpb200_handle_t h, int n, int B, int nvec, const double *fbar, double *theta_bar,
                                              double *zbar) {
  CHECK_H(h);
  if (n < 1) BAD_ARG(h, 2, "latent_backward_batched: n must be >= 1");
  if (B < 1) BAD_ARG(h, 3, "latent_backward_batched: B must be >= 1");
  if (nvec < 1) BAD_ARG(h, 4, "latent_backward_batched: nvec must be >= 1");
  if (!fbar) BAD_ARG(h, 5, "latent_backward_batched: fbar is NULL");
  if (!theta_bar) BAD_ARG(h, 6, "latent_backward_batched: theta_bar is NULL");
  if (!zbar) BAD_ARG(h, 7, "latent_backward_batched: zbar is NULL");
  if (!h->latent_rec_valid)
    BAD_ARG(h, 1, "latent_backward_batched: no recorded batch (call gpb200_latent_forward_batched first; a failed forward "
                  "call leaves none)");
  if (n != h->latent_rec_n || B != h->latent_rec_B || nvec != h->latent_rec_nvec) {
    snprintf(h->err, sizeof(h->err), "latent_backward_batched: (n, B, nvec) = (%d, %d, %d), the recorded batch has (%d, %d, %d)",
             n, B, nvec, h->latent_rec_n, h->latent_rec_B, h->latent_rec_nvec);
    return -2;
  }
  const int np = round_up(n, TILE), nt = np / TILE;
  const long long mat = (long long)np * np, xs = h->latent_rec_xs, vs = (long long)nvec * np;
  const bool host = !h->device_ptrs;
  const LatentRecord rec = latent_record(h, n, B, nvec, xs);
  TaskList tl;
  RC(latent_tasks(h, nt, &tl));
  const int ntasks = tl.count(0);
  const int nparts = ntasks * 4;  // trace partial records per item: one per CTA, at most four CTAs per tile

  const size_t per_item = 2 * pad256(mat * 8) + 2 * pad256((size_t)vs * 8) + pad256((size_t)nparts * 4 * 8) +
                          (host ? pad256((size_t)nvec * n * 8) : 0) + 64;
  const size_t fixed = pad256((size_t)np * 8) + (host ? pad256((size_t)B * 2 * 8) : 0) + 4096;
  int Bc = B;
  if (h->ws_limit > 0 || fixed + per_item * (size_t)B + 8192 > h->ws_bytes) {
    size_t limit = (size_t)h->ws_limit;
    if (h->ws_limit <= 0) {
      size_t freeb = 0, totalb = 0;
      GPB_CUDA(h, cudaMemGetInfo(&freeb, &totalb));
      limit = (size_t)((freeb + h->ws_bytes) * 0.85);
    }
    if (limit < fixed + per_item + 8192) BAD_ARG(h, 1002, "latent_backward_batched: workspace limit too small for one item");
    Bc = (int)std::min<size_t>((size_t)B, (limit - fixed - 8192) / per_item);
  }
  Bc = std::min(Bc, 65535);  // gridDim.y of the batched launches
  Arena a;
  RC(ws_reserve(h, fixed + per_item * (size_t)Bc + 8192, &a));
  double *W = a.take<double>((size_t)Bc * mat), *S = a.take<double>((size_t)Bc * mat);
  double *u = a.take<double>((size_t)Bc * vs), *fb = a.take<double>((size_t)Bc * vs);
  double *partial = a.take<double>((size_t)Bc * nparts * 4);
  double *zero = a.take<double>(np);
  double *zst = host ? a.take<double>((size_t)Bc * nvec * n) : nullptr;
  double *tb = host ? a.take<double>((size_t)B * 2) : theta_bar;
  if (!zero || !tb || (host && !zst)) BAD_ARG(h, 1002, "latent_backward_batched: workspace arithmetic error");
  GPB_CUDA(h, cudaMemsetAsync(zero, 0, (size_t)np * 8, h->stream));

  for (int b0 = 0; b0 < B; b0 += Bc) {
    const int bc = std::min(Bc, B - b0);
    const double *L = rec.L + (long long)b0 * mat;
    GPB_CUDA(h, cudaMemsetAsync(fb, 0, (size_t)bc * vs * 8, h->stream));
    RC(to_device_2d(h, fbar + (long long)b0 * nvec * n, n, fb, np, n, bc * nvec));
    for (int m = 0; m < nvec; m++)   // u = zbar = L^T fbar
      RC(launch_trmv_lower_t(h, np, L, mat, fb + (long long)m * np, vs, u + (long long)m * np, vs, bc));
    GPB_CUDA(h, cudaMemcpyAsync(W, L, (size_t)bc * mat * 8, cudaMemcpyDeviceToDevice, h->stream));
    RC(trtri_batched(h, W, S, np, mat, bc));
    for (int m = 0; m < nvec; m++) {  // T = sum_m P_m W, over the inverse's scratch
      ProfScope ps__(h, PC_SOLVE);
      latent_pw_kernel<<<dim3((np + 7) / 8, bc), 256, 0, h->stream>>>(np, W, mat, u + (long long)m * np,
                                                                      rec.z + ((long long)b0 * nvec + m) * np, vs, m > 0, S);
      GPB_LAUNCH_CHECK(h);
    }
    GemmParams p{};
    p.A = mref(W, np, mat);
    p.B = mref(S, np, mat);
    p.C = mref(nullptr, np, mat);
    p.tasks = tl.at(0);
    p.x = rec.x + (long long)b0 * xs; p.x_stride = xs;
    p.avec = zero; p.a_stride = 0;
    p.theta = rec.theta + 3LL * b0;
    p.partial = partial;
    p.n = n;
    p.ntasks = ntasks;
    RC(launch_gemm(h, LAYOUT_TN, EPI_TRACE, p, ntasks, bc));
    {
      ProfScope ps__(h, PC_OTHER);
      latent_sum_kernel<<<bc, 256, 0, h->stream>>>((long long)ntasks * gemm_nsplit(h, ntasks, bc), partial, rec.theta + 3LL * b0,
                                                   rec.info + b0, tb + 2LL * b0);
      GPB_LAUNCH_CHECK(h);
    }
    double *zout = host ? zst : zbar + (long long)b0 * nvec * n;
    RC(launch_latent_rows(h, n, np, nvec, (long long)bc * nvec, u, rec.info + b0, zout));
    if (host) RC(from_device(h, zst, zbar + (long long)b0 * nvec * n, (size_t)bc * nvec * n * sizeof(double)));
  }
  if (host) RC(from_device(h, tb, theta_bar, (size_t)B * 2 * sizeof(double)));
  return finish(h);
}
