// C-ABI entry points for posterior sampling (f-4): device normal numbers and mvrnorm.
#include "host.cuh"

using namespace gpb;

extern "C" int gpb200_normal_fill(gpb200_handle_t h, unsigned long long seed, unsigned long long offset, long long len,
                                  double *out) {
  CHECK_H(h);
  if (len < 0) BAD_ARG(h, 4, "normal_fill: negative length");
  if (offset & 1ULL) BAD_ARG(h, 3, "normal_fill: offset must be even (normals are generated in Box-Muller pairs)");
  if (len == 0) return 0;
  if (h->device_ptrs) {
    RC(launch_normal_fill(h, seed, offset, len, len, len, out));
    return 0;
  }
  Arena a;
  RC(ws_reserve(h, pad256((size_t)len * 8) + 256, &a));
  double *d = a.take<double>((size_t)len);
  RC(launch_normal_fill(h, seed, offset, len, len, len, d));
  RC(from_device(h, d, out, (size_t)len * sizeof(double)));
  return finish(h);
}

namespace {
int tasks_lz(Handle *h, int nt, int dt, TaskList *out) {
  const long long key = tkey(TK_MUL_LZ, nt, dt);
  if (cached(h, key, out)) return 0;
  std::vector<TileTask> v;
  for (int i = 0; i < nt; i++)
    for (int j = 0; j < dt; j++)  // X[i,j] = sum_{k<=i} L[i,k] Z[k,j]   (NN)
      v.push_back({i * TILE, 0, 0, j * TILE, i * TILE, j * TILE, (i + 1) * TILE, TF_A_TRI_LAST});
  sort_desc(v, 0);
  std::vector<int> off = {0, (int)v.size()};
  return upload_tasks(h, key, v, off, out);
}
}  // namespace

extern "C" int gpb200_mvrnorm(gpb200_handle_t h, int ndraws, int m, const double *mu, const double *Sigma, int lds,
                              double jitter, unsigned long long seed, double *out, int ldo) {
  CHECK_H(h);
  if (ndraws < 0) BAD_ARG(h, 2, "mvrnorm: negative number of draws");
  if (m < 1) BAD_ARG(h, 3, "mvrnorm: dimension must be >= 1");
  if (m > MAX_DENSE_N) BAD_ARG(h, 3, "mvrnorm: dimensions above 65407 are not supported");
  if (lds < m) BAD_ARG(h, 6, "mvrnorm: lds < m");
  if (ldo < std::max(1, ndraws)) BAD_ARG(h, 10, "mvrnorm: ldo < ndraws");
  if (ndraws == 0) return 0;
  const int mp = round_up(m, TILE), dp = round_up(ndraws, TILE);
  const size_t mat = (size_t)mp * mp, zsz = (size_t)mp * dp;
  Arena a;
  const size_t stage = h->device_ptrs ? 0 : pad256((size_t)m * m * 8) + pad256((size_t)m * 8) + pad256((size_t)ndraws * m * 8);
  RC(ws_reserve(h, pad256(mat * 8) + 2 * pad256(zsz * 8) + stage + 1024, &a));
  double *Lbuf = a.take<double>(mat), *Z = a.take<double>(zsz), *X = a.take<double>(zsz);
  int *info = a.take<int>(1);
  const double *dS = Sigma, *dmu = mu;
  long long ld = lds;
  double *dout = out;
  long long ldout = ldo;
  if (!h->device_ptrs) {
    double *s = a.take<double>((size_t)m * m), *mm = a.take<double>(m);
    dout = a.take<double>((size_t)ndraws * m);
    if (!dout) BAD_ARG(h, 1002, "mvrnorm: workspace exhausted");
    RC(to_device_2d(h, Sigma, lds, s, m, m, m));
    if (mu) RC(to_device(h, mu, mm, m));
    dS = s; ld = m; dmu = mu ? mm : nullptr; ldout = ndraws;
  }
  GPB_CUDA(h, cudaMemsetAsync(info, 0, sizeof(int), h->stream));
  RC(launch_pack(h, m, m, dS, ld, mp, mp, Lbuf, 1, jitter));
  RC(chol_batched(h, Lbuf, mp, (long long)mat, m, 1, info));
  int hinfo = 0;
  RC(read_info(h, info, &hinfo));
  if (hinfo) return hinfo;
  // Z: m x ndraws standard normals, element (i, d) = normal number i + d*m of the stream; zero padding
  GPB_CUDA(h, cudaMemsetAsync(Z, 0, zsz * sizeof(double), h->stream));
  RC(launch_normal_fill(h, seed, 0, (long long)m * ndraws, m, mp, Z));
  TaskList tl;
  RC(tasks_lz(h, mp / TILE, dp / TILE, &tl));
  GemmParams p{};
  p.A = mref(Lbuf, mp, 0); p.B = mref(Z, mp, 0); p.C = mref(X, mp, 0); p.alpha = 1.0; p.tasks = tl.at(0);
  RC(launch_gemm(h, LAYOUT_NN, EPI_AXPBY, p, tl.count(0), 1));
  RC(launch_add_mean_transpose(h, m, ndraws, X, mp, dmu, dout, ldout));
  if (!h->device_ptrs) RC(from_device_2d(h, dout, ndraws, out, ldo, ndraws, m));
  RC(finish(h));
  return 0;
}

namespace {
// Posterior draws for B hyper-parameter draws, one joint factorisation per item.  The Cholesky factor of
//   J = [[K, Ks^T], [Ks, Kss + jitter I]]  is  [[L11, 0], [L21, L22]]  with L21 = Ks L11^-T and L22 L22^T = cov,
// so with z1 = L11^-1 y the lower block of  L [z1; eps]  is  L21 z1 + L22 eps = mu + chol(cov) eps.
// The pivot index of the joint factorisation already is the item's info (1..n: K, n+1..n+m: cov).
//
// The chunked pipeline shared by the posterior-draw entry points, which keep their argument checks, the staging of
// their kernel inputs and the launch of their joint Gram.  `inputs` is the workspace (bytes, pad256-ed) of those
// inputs; stage(a) takes them from the arena a and enqueues their copies (nonzero on failure); gram(b0, bc, J, mat)
// builds the joint matrices of items [b0, b0 + bc) into J, np x np each, mat doubles apart.  The workspace is
//   fixed    = inputs + pad256((B yl + n) 8) + [z] pad256(B m 8) + (mu ? 2 : 1) pad256(B m 8) + pad256(4 B) + 6 * 256 + 4096
//   per_item = 2 np^2 8 + 2 np 8,   np = round_up(n + m, 128),   yl = y_stride ? n : 0
// and without a limit the batch runs in one chunk when fixed + B per_item + 8192 fits the current workspace.  Otherwise
// chunks of Bc = min(B, (limit - fixed - 8192) / per_item, 65535) items, the limit being the one set on the handle or
// 85 % of (free memory + current workspace).
template <class Stage, class Gram>
int posterior_draws_pipeline(Handle *h, const char *name, int n, int m, int B, size_t inputs, const double *y,
                             long long y_stride, const double *z, unsigned long long seed, double *draws, double *mu,
                             int *info, Stage stage, Gram gram) {
  const int N = n + m, np = round_up(N, TILE), nt = np / TILE;
  const long long mat = (long long)np * np;
  const long long yl = y_stride ? n : 0;
  const size_t per_item = 2 * (size_t)mat * 8 + 2 * (size_t)np * 8;
  const size_t fixed = inputs + pad256((size_t)(B * yl + n) * 8) + (z ? pad256((size_t)B * m * 8) : 0) +
                       (mu ? 2 : 1) * pad256((size_t)B * m * 8) + pad256((size_t)B * 4) + 6 * 256 + 4096;
  // chunk the batch under the workspace limit, sized like the fused LML path
  int Bc = B;
  if (h->ws_limit > 0 || fixed + per_item * (size_t)B + 8192 > h->ws_bytes) {
    size_t limit = (size_t)h->ws_limit;
    if (h->ws_limit <= 0) {
      size_t freeb = 0, totalb = 0;
      GPB_CUDA(h, cudaMemGetInfo(&freeb, &totalb));
      limit = (size_t)((freeb + h->ws_bytes) * 0.85);
    }
    if (limit < fixed + per_item + 8192) {
      snprintf(h->err, sizeof(h->err), "%s: workspace limit too small for one item", name);
      return -1002;
    }
    Bc = (int)std::min<size_t>((size_t)B, (limit - fixed - 8192) / per_item);
  }
  Bc = std::min(Bc, 65535);  // gridDim.y of the batched launches
  Arena a;
  RC(ws_reserve(h, fixed + per_item * (size_t)Bc + 8192, &a));
  RC(stage(a));
  double *dy = a.take<double>((size_t)B * yl + n), *dz = z ? a.take<double>((size_t)B * m) : nullptr;
  double *ddraw = a.take<double>((size_t)B * m), *dmu = mu ? a.take<double>((size_t)B * m) : nullptr;
  int *dinfo = a.take<int>(B);
  double *Lbuf = a.take<double>((size_t)Bc * mat), *Sbuf = a.take<double>((size_t)Bc * mat);
  double *zbuf = a.take<double>((size_t)Bc * np), *vbuf = a.take<double>((size_t)Bc * np);
  if (!vbuf) {
    snprintf(h->err, sizeof(h->err), "%s: workspace arithmetic error", name);
    return -1002;
  }

  if (y_stride) RC(to_device_2d(h, y, y_stride, dy, n, n, B)); else RC(to_device(h, y, dy, n));
  if (z) RC(to_device(h, z, dz, (size_t)B * m));
  GPB_CUDA(h, cudaMemsetAsync(dinfo, 0, (size_t)B * sizeof(int), h->stream));
  for (int b0 = 0; b0 < B; b0 += Bc) {
    const int bc = std::min(Bc, B - b0);
    const double *cy = dy + (long long)b0 * yl;
    int *cinfo = dinfo + b0;
    RC(gram(b0, bc, Lbuf, mat));
    RC(chol_batched(h, Lbuf, np, mat, N, bc, cinfo));
    // z[0, n) = L11^-1 y (the rhs is read as zero from row n on)
    RC(launch_tile_inverse(h, Lbuf, Sbuf, np, mat, nt, bc));
    if (bc >= 32) RC(launch_trsv_blocked(h, np, Lbuf, Sbuf, mat, cy, yl, nullptr, n, zbuf, np, bc));
    else RC(launch_trsv_sweep(h, np, Lbuf, Sbuf, mat, cy, yl, nullptr, n, zbuf, vbuf, np, bc));
    if (dmu) {  // rows [n, n+m) of L [z1; 0] = L21 z1 = mu
      RC(launch_trmv_lower_n(h, np, Lbuf, mat, zbuf, np, n, vbuf, np, bc));
      RC(launch_rows_or_nan(h, n, m, vbuf, np, cinfo, dmu + (long long)b0 * m, bc));
    }
    // z[n, n+m) = eps_b: the caller's normals, or normals [b*m, (b+1)*m) of the stream (independent of the chunking)
    if (dz) GPB_CUDA(h, cudaMemcpy2DAsync(zbuf + n, (size_t)np * 8, dz + (long long)b0 * m, (size_t)m * 8, (size_t)m * 8, bc,
                                          cudaMemcpyDeviceToDevice, h->stream));
    else RC(launch_normal_fill(h, seed, (unsigned long long)b0 * m, (long long)bc * m, m, np, zbuf + n));
    RC(launch_trmv_lower_n(h, np, Lbuf, mat, zbuf, np, N, vbuf, np, bc));
    RC(launch_rows_or_nan(h, n, m, vbuf, np, cinfo, ddraw + (long long)b0 * m, bc));
  }
  RC(from_device(h, ddraw, draws, (size_t)B * m * sizeof(double)));
  if (mu) RC(from_device(h, dmu, mu, (size_t)B * m * sizeof(double)));
  RC(from_device(h, dinfo, info, (size_t)B * sizeof(int)));
  return finish(h);
}
}  // namespace

extern "C" int gpb200_posterior_draws_batched(gpb200_handle_t h, int n, int m, int order, int B, const double *t,
                                              long long t_stride, const double *s, long long s_stride, const double *y,
                                              long long y_stride, const double *theta, double jitter, const double *z,
                                              unsigned long long seed, double *draws, double *mu, int *info) {
  CHECK_H(h);
  if (n < 1) BAD_ARG(h, 2, "posterior_draws_batched: n must be >= 1");
  if (m < 1) BAD_ARG(h, 3, "posterior_draws_batched: m must be >= 1");
  if (order < 0 || order > 2) BAD_ARG(h, 4, "posterior_draws_batched: derivative order must be 0, 1 or 2");
  if (B < 0) BAD_ARG(h, 5, "posterior_draws_batched: negative batch");
  if ((long long)n + m > MAX_DENSE_N) BAD_ARG(h, 3, "posterior_draws_batched: n + m above 65407 is not supported");
  if (t_stride != 0 && t_stride < n) BAD_ARG(h, 7, "posterior_draws_batched: t_stride < n");
  if (!s && m != n) BAD_ARG(h, 8, "posterior_draws_batched: s == NULL predicts on t and needs m == n");
  if (s && s_stride != 0 && s_stride < m) BAD_ARG(h, 9, "posterior_draws_batched: s_stride < m");
  if (y_stride != 0 && y_stride < n) BAD_ARG(h, 11, "posterior_draws_batched: y_stride < n");
  if (B == 0) return 0;
  if (!t || !y || !theta || !draws || !info) BAD_ARG(h, 6, "posterior_draws_batched: t, y, theta, draws and info are required");
  if (!s) { s = t; s_stride = t_stride; }

  const int np = round_up(n + m, TILE);
  const long long tl = t_stride ? n : 0, sl = s_stride ? m : 0;
  const size_t inputs = pad256((size_t)(B * tl + n) * 8) + pad256((size_t)(B * sl + m) * 8) + pad256((size_t)B * 3 * 8);
  double *dt = nullptr, *ds = nullptr, *dth = nullptr;
  auto stage = [&](Arena &a) -> int {
    dt = a.take<double>((size_t)B * tl + n); ds = a.take<double>((size_t)B * sl + m); dth = a.take<double>((size_t)B * 3);
    if (!dth) BAD_ARG(h, 1002, "posterior_draws_batched: workspace arithmetic error");
    if (t_stride) RC(to_device_2d(h, t, t_stride, dt, n, n, B)); else RC(to_device(h, t, dt, n));
    if (s_stride) RC(to_device_2d(h, s, s_stride, ds, m, m, B)); else RC(to_device(h, s, ds, m));
    return to_device(h, theta, dth, (size_t)B * 3);
  };
  auto gram = [&](int b0, int bc, double *J, long long mat) {
    return launch_gram_cond_batched(h, n, m, order, np, dt + (long long)b0 * tl, tl, ds + (long long)b0 * sl, sl,
                                    dth + (long long)b0 * 3, jitter, J, mat, bc);
  };
  return posterior_draws_pipeline(h, "posterior_draws_batched", n, m, B, inputs, y, y_stride, z, seed, draws, mu, info,
                                  stage, gram);
}

// The same for the ARD kernel on D-column inputs (gram_cond_ard_batched_kernel).  Its inputs add to the workspace of
// posterior_draws_pipeline
//   inputs = pad256((B xl + n D) 8) + pad256((B sl + m D) 8) + pad256(B (D + 2) 8),
//   xl = x_stride ? n D : 0,  sl = xs_stride ? m D : 0  (Xs == NULL stages a second copy of X with X's stride).
extern "C" int gpb200_posterior_draws_ard_batched(gpb200_handle_t h, int n, int m, int D, int B, const double *X,
                                                  long long x_stride, const double *Xs, long long xs_stride,
                                                  const double *y, long long y_stride, const double *theta, double jitter,
                                                  const double *z, unsigned long long seed, double *draws, double *mu,
                                                  int *info) {
  CHECK_H(h);
  if (n < 1) BAD_ARG(h, 2, "posterior_draws_ard_batched: n must be >= 1");
  if (m < 1) BAD_ARG(h, 3, "posterior_draws_ard_batched: m must be >= 1");
  if (D < 1 || D > ARD_MAX_D) BAD_ARG(h, 4, "posterior_draws_ard_batched: D must lie in 1..8");
  if (B < 0) BAD_ARG(h, 5, "posterior_draws_ard_batched: negative batch");
  if ((long long)n + m > MAX_DENSE_N) BAD_ARG(h, 3, "posterior_draws_ard_batched: n + m above 65407 is not supported");
  if ((long long)n * D > 2147483647LL / 2 || (long long)m * D > 2147483647LL / 2)
    BAD_ARG(h, 2, "posterior_draws_ard_batched: n * D or m * D too large");
  if (x_stride != 0 && x_stride < (long long)n * D) BAD_ARG(h, 7, "posterior_draws_ard_batched: x_stride < n * D");
  if (!Xs && m != n) BAD_ARG(h, 8, "posterior_draws_ard_batched: Xs == NULL predicts on X and needs m == n");
  if (Xs && xs_stride != 0 && xs_stride < (long long)m * D) BAD_ARG(h, 9, "posterior_draws_ard_batched: xs_stride < m * D");
  if (y_stride != 0 && y_stride < n) BAD_ARG(h, 11, "posterior_draws_ard_batched: y_stride < n");
  if (B == 0) return 0;
  if (!X || !y || !theta || !draws || !info) BAD_ARG(h, 6, "posterior_draws_ard_batched: X, y, theta, draws and info are required");
  if (!Xs) { Xs = X; xs_stride = x_stride; }

  const int np = round_up(n + m, TILE), ts = D + 2;
  const long long xl = x_stride ? (long long)n * D : 0, sl = xs_stride ? (long long)m * D : 0;
  const size_t inputs = pad256(((size_t)B * xl + (size_t)n * D) * 8) + pad256(((size_t)B * sl + (size_t)m * D) * 8) +
                        pad256((size_t)B * ts * 8);
  double *dX = nullptr, *dXs = nullptr, *dth = nullptr;
  auto stage = [&](Arena &a) -> int {
    dX = a.take<double>((size_t)B * xl + (size_t)n * D); dXs = a.take<double>((size_t)B * sl + (size_t)m * D);
    dth = a.take<double>((size_t)B * ts);
    if (!dth) BAD_ARG(h, 1002, "posterior_draws_ard_batched: workspace arithmetic error");
    if (x_stride) RC(to_device_2d(h, X, x_stride, dX, xl, (int)xl, B)); else RC(to_device(h, X, dX, (size_t)n * D));
    if (xs_stride) RC(to_device_2d(h, Xs, xs_stride, dXs, sl, (int)sl, B)); else RC(to_device(h, Xs, dXs, (size_t)m * D));
    return to_device(h, theta, dth, (size_t)B * ts);
  };
  auto gram = [&](int b0, int bc, double *J, long long mat) {
    return launch_gram_cond_ard_batched(h, n, m, D, np, dX + (long long)b0 * xl, xl, dXs + (long long)b0 * sl, sl,
                                        dth + (long long)b0 * ts, jitter, J, mat, bc);
  };
  return posterior_draws_pipeline(h, "posterior_draws_ard_batched", n, m, B, inputs, y, y_stride, z, seed, draws, mu,
                                  info, stage, gram);
}
