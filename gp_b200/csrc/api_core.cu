// C-ABI entry points: handle management, kernel/Gram functions (a9), factorisation and solves on
// caller matrices (a6-a8).  See include/gpb200.h.
#include "host.cuh"

using namespace gpb;

// =================================================================================================
// handle
// =================================================================================================
extern "C" int gpb200_version(void) { return 100; }

namespace {
void free_handle(gpb200_handle_s *h) {
  if (!h) return;
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (auto &kv : h->graphs) cudaGraphExecDestroy(kv.second.exec);
  if (h->gstream) { cudaStreamSynchronize(h->gstream); cudaStreamDestroy(h->gstream); }
  if (h->pstream) { cudaStreamSynchronize(h->pstream); cudaStreamDestroy(h->pstream); }
  if (h->cstream) { cudaStreamSynchronize(h->cstream); cudaStreamDestroy(h->cstream); }
  for (cudaEvent_t e : h->sync_events) cudaEventDestroy(e);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  for (cudaEvent_t e : h->mg_events) cudaEventDestroy(e);
  if (h->g_in) cudaEventDestroy(h->g_in);
  if (h->g_out) cudaEventDestroy(h->g_out);
  if (h->stream_switch) cudaEventDestroy(h->stream_switch);
  if (h->ws) cudaFree(h->ws);
  if (h->latent_L) cudaFree(h->latent_L);
  if (h->latent_rec) cudaFree(h->latent_rec);
  if (h->info_slot) cudaFree(h->info_slot);
  if (h->panel_flags) cudaFree(h->panel_flags);
  if (h->flops_dev) cudaFree(h->flops_dev);
  for (auto &kv : h->task_cache) cudaFree(kv.second.first);
  for (auto &kv : h->split_cache) if (kv.second.reg) cudaFree(kv.second.reg);
  delete h;
}
}  // namespace

extern "C" int gpb200_create(gpb200_handle_t *out, int device) {
  if (!out) return -1;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
    (void)cudaGetLastError();
    return -1000;  // no CUDA device: there is no CPU fallback
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -1000;
  if (prop.major < 10) return -1003;  // built for sm_100a only
  DeviceGuard guard(device);
  if (!guard.ok) return -1000;
  gpb200_handle_s *h = new (std::nothrow) gpb200_handle_s();
  if (!h) return -1002;
  h->device = device;
  if (panel_smem_setup(h) || gemm_smem_setup(h) || small_smem_setup(h)) { free_handle(h); return -1000; }
  if (cudaStreamCreateWithFlags(&h->gstream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->g_in, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->g_out, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->stream_switch, cudaEventDisableTiming) != cudaSuccess ||
      cudaMalloc(&h->info_slot, sizeof(int)) != cudaSuccess ||
      cudaMalloc(&h->panel_flags, 2 * PANEL_FUSED_MAX_BATCH * sizeof(int)) != cudaSuccess ||
      cudaMemset(h->panel_flags, 0, 2 * PANEL_FUSED_MAX_BATCH * sizeof(int)) != cudaSuccess) { free_handle(h); return -1000; }
  {
    int lo = 0, hi = 0;  // numerically lowest value = highest priority
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess ||
        cudaStreamCreateWithPriority(&h->pstream, cudaStreamNonBlocking, hi) != cudaSuccess) { free_handle(h); return -1000; }
  }
  const char *cp = getenv("GPB200_CHOL_PANEL");  // same meaning as gpb200_set_chol_panel_tiles
  if (cp && cp[0] >= '0' && cp[0] <= '9') h->chol_panel_override = atoi(cp);
  const char *sk = getenv("GPB200_SMALL_KERNEL");
  if (sk && sk[0] == '0') h->small_kernel = 0;
  const char *la = getenv("GPB200_LOOKAHEAD");
  if (la && la[0] == '0') h->lookahead = 0;
  const char *lb = getenv("GPB200_LOOKAHEAD_MAXB");
  if (lb && lb[0] >= '0' && lb[0] <= '9') h->lookahead_max_batch = atoi(lb);
  const char *qw = getenv("GPB200_QUARTER_WAVES");
  if (qw && qw[0] >= '0' && qw[0] <= '9') h->quarter_below_waves = atoi(qw);
  const char *gc = getenv("GPB200_GEMM_CFG");  // tuning knob, same meaning as gpb200_set_gemm_config
  if (gc && gc[0] >= '0' && gc[0] <= '3') h->gemm_cfg_override = gc[0] - '0';
  const char *tp = getenv("GPB200_TRSM_PIPELINED");
  if (tp && tp[0] == '0') h->trsm_pipelined = 0;
  const char *ds = getenv("GPB200_DIAG_SPLIT");
  if (ds && ds[0] == '0') h->diag_split = 0;
  const char *fc = getenv("GPB200_FINE_CFG");
  if (fc && fc[0] == '0') h->fine_cfg = 0;
  const char *pf = getenv("GPB200_PANEL_FUSED");
  if (pf && pf[0] == '0') h->panel_fused = 0;
  const char *ev = getenv("GPB200_ENVELOPE");  // 0: the dense SE route (reference for tests)
  if (ev && ev[0] == '0') h->envelope = 0;
  const char *sm = getenv("GPB200_SINV_MINB");
  if (sm && sm[0] >= '0' && sm[0] <= '9') h->sinv_min_batch = atoi(sm);
  const char *ng = getenv("GPB200_NO_GRAPH");
  if (ng && ng[0] == '1') h->graphs_enabled = 0;
  *out = h;
  return 0;
}

extern "C" int gpb200_destroy(gpb200_handle_t h) {
  if (!h) return 0;
  DeviceGuard guard(h->device);
  if (h->nccl_comm) gpb200_mg_comm_destroy(h);
  free_handle(h);
  return 0;
}

// Switching streams keeps stream order: whatever this handle enqueued on the old stream (it all works out of one
// workspace) completes before anything it enqueues on the new one starts -- an event, no host synchronisation.
extern "C" int gpb200_set_stream(gpb200_handle_t h, void *s) {
  CHECK_H(h);
  cudaStream_t ns = reinterpret_cast<cudaStream_t>(s);
  if (ns != h->stream) {
    GPB_CUDA(h, cudaEventRecord(h->stream_switch, h->stream));
    GPB_CUDA(h, cudaStreamWaitEvent(ns, h->stream_switch, 0));
    h->stream = ns;
  }
  return 0;
}
// The same without the ordering edge, for callers that run independent work of ONE handle on several streams and order
// it with their own events (the block-cyclic schedule: panel chain, side updates and trailing updates overlap).  Only the
// entry points that touch no handle-owned scratch may be used this way (gpb200_mg_panel_*, gpb200_mg_bcast / _wait).
extern "C" int gpb200_set_stream_unordered(gpb200_handle_t h, void *s) {
  CHECK_H(h);
  h->stream = reinterpret_cast<cudaStream_t>(s);
  return 0;
}
extern "C" int gpb200_set_pointer_mode(gpb200_handle_t h, int dev) {
  if (!h) return -1;
  h->device_ptrs = dev ? 1 : 0;
  return 0;
}
extern "C" int gpb200_synchronize(gpb200_handle_t h) {
  CHECK_H(h);
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  return 0;
}
extern "C" const char *gpb200_last_error(gpb200_handle_t h) { return h ? h->err : "null handle"; }
extern "C" long long gpb200_launch_count(gpb200_handle_t h) { return h ? h->launches : 0; }
extern "C" int gpb200_set_workspace_limit(gpb200_handle_t h, long long bytes) {
  if (!h) return -1;
  h->ws_limit = bytes;
  return 0;
}

// test/tuning knob: force the Cholesky panel width in 128-column tiles (0 = automatic)
extern "C" int gpb200_set_chol_panel_tiles(gpb200_handle_t h, int tiles) {
  if (!h || tiles < 0) return -1;
  h->chol_panel_override = tiles;
  return 0;
}

// test/tuning knob: 0 default, 1 one 128x128 CTA per SM, 2 two 128x64 half-tile CTAs per SM
extern "C" int gpb200_set_gemm_config(gpb200_handle_t h, int cfg) {
  if (!h || cfg < 0 || cfg > 3) return -1;
  h->gemm_cfg_override = cfg;
  return 0;
}

extern "C" int gpb200_set_profiling(gpb200_handle_t h, int on) {
  if (!h) return -1;
  h->profiling = on ? 1 : 0;
  h->prof.clear();
  h->ev_used = 0;
  if (on && h->ev_pool.size() < 1024) {
    // create the event pool up front: cudaEventCreate inside a timed region costs host time
    if (cudaSetDevice(h->device) != cudaSuccess) return -1000;
    while (h->ev_pool.size() < 1024) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) return -1000;
      h->ev_pool.push_back(e);
    }
  }
  return 0;
}

// Sums the event-bracketed launch durations per kernel class since profiling was switched on (or
// since the last call), then resets.  ms_out / count_out: arrays of 6 (gemm, potrf tile, trsm tile,
// gram, solves, other).  Synchronises the stream.
extern "C" int gpb200_get_profile(gpb200_handle_t h, double *ms_out, long long *count_out) {
  CHECK_H(h);
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  for (int c = 0; c < PC_COUNT; c++) { ms_out[c] = 0.0; count_out[c] = 0; }
  for (const auto &r : h->prof) {
    float ms = 0.f;
    GPB_CUDA(h, cudaEventElapsedTime(&ms, r.e0, r.e1));
    ms_out[r.cls] += ms;
    count_out[r.cls]++;
  }
  h->prof.clear();
  h->ev_used = 0;
  return 0;
}

// =================================================================================================
// a9 kernels
// =================================================================================================
extern "C" int gpb200_kernel_eval(gpb200_handle_t h, int kind, long long len, const double *tj, const double *tk,
                                  double amp2, double l, double *out) {
  CHECK_H(h);
  if (kind < 0 || kind > 9) BAD_ARG(h, 2, "kernel_eval: unknown kind");
  if (len < 0) BAD_ARG(h, 3, "kernel_eval: negative length");
  if (len == 0) return 0;
  if (h->device_ptrs) return launch_kernel_eval(h, kind, len, tj, tk, amp2, l, out);
  Arena a;
  RC(ws_reserve(h, 3 * pad256(len * sizeof(double)), &a));
  double *dj = a.take<double>(len), *dk = a.take<double>(len), *dout = a.take<double>(len);
  RC(to_device(h, tj, dj, len));
  RC(to_device(h, tk, dk, len));
  RC(launch_kernel_eval(h, kind, len, dj, dk, amp2, l, dout));
  RC(from_device(h, dout, out, len * sizeof(double)));
  return finish(h);
}

extern "C" int gpb200_gram_outer(gpb200_handle_t h, int kind, int n, int m, const double *x, const double *y,
                                 double amp2, double l, double *K, int ldk) {
  CHECK_H(h);
  if (kind < 0 || kind > 9) BAD_ARG(h, 2, "gram_outer: unknown kind");
  if (n < 0 || m < 0) BAD_ARG(h, 3, "gram_outer: negative size");
  if (ldk < std::max(1, n)) BAD_ARG(h, 10, "gram_outer: ldk < n");
  if (n == 0 || m == 0) return 0;
  if (h->device_ptrs) return launch_gram_outer(h, kind, n, m, x, y, amp2, l, K, ldk);
  Arena a;
  const int ldd = round_up(n, 2);
  RC(ws_reserve(h, pad256(n * 8) + pad256(m * 8) + pad256((size_t)ldd * m * 8), &a));
  double *dx = a.take<double>(n), *dy = a.take<double>(m), *dK = a.take<double>((size_t)ldd * m);
  RC(to_device(h, x, dx, n));
  RC(to_device(h, y, dy, m));
  RC(launch_gram_outer(h, kind, n, m, dx, dy, amp2, l, dK, ldd));
  RC(from_device_2d(h, dK, ldd, K, ldk, n, m));
  return finish(h);
}

extern "C" int gpb200_gram_ard(gpb200_handle_t h, int n, int m, int D, const double *X, int ldx, const double *Y,
                               int ldy, double alpha, const double *rho, double *K, int ldk) {
  CHECK_H(h);
  if (n < 0 || m < 0 || D < 1) BAD_ARG(h, 2, "gram_ard: bad sizes");
  if (ldx < std::max(1, n) || ldy < std::max(1, m) || ldk < std::max(1, n)) BAD_ARG(h, 6, "gram_ard: bad leading dimension");
  if (n == 0 || m == 0) return 0;
  if (h->device_ptrs) return launch_gram_ard(h, n, m, D, X, ldx, Y, ldy, alpha, rho, D, K, ldk);
  Arena a;
  RC(ws_reserve(h, pad256((size_t)n * D * 8) + pad256((size_t)m * D * 8) + pad256(D * 8) + pad256((size_t)n * m * 8), &a));
  double *dX = a.take<double>((size_t)n * D), *dY = a.take<double>((size_t)m * D), *dr = a.take<double>(D);
  double *dK = a.take<double>((size_t)n * m);
  RC(to_device_2d(h, X, ldx, dX, n, n, D));
  RC(to_device_2d(h, Y, ldy, dY, m, m, D));
  RC(to_device(h, rho, dr, D));
  RC(launch_gram_ard(h, n, m, D, dX, n, dY, m, alpha, dr, D, dK, n));
  RC(from_device_2d(h, dK, n, K, ldk, n, m));
  return finish(h);
}

extern "C" int gpb200_gram_se(gpb200_handle_t h, int n, const double *x, double alpha, double rho, double diag_add,
                              double *K, int ldk) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "gram_se: negative n");
  if (ldk < std::max(1, n)) BAD_ARG(h, 8, "gram_se: ldk < n");
  if (n == 0) return 0;
  const int np = round_up(n, TILE);
  Arena a;
  RC(ws_reserve(h, pad256((size_t)np * np * 8) + pad256(n * 8) + 256, &a));
  double *dK = a.take<double>((size_t)np * np), *dx = a.take<double>(n), *dth = a.take<double>(3);
  RC(to_device(h, x, dx, n));
  // sigma^2 + jitter = diag_add: pass sigma = 0 and jitter = diag_add
  const double th[3] = {alpha, rho, 0.0};
  GPB_CUDA(h, cudaMemcpyAsync(dth, th, sizeof(th), cudaMemcpyHostToDevice, h->stream));
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  RC(launch_gram_se_batched(h, n, np, dx, 0, dth, diag_add, 0, dK, 0, 1));
  RC(from_device_2d(h, dK, np, K, ldk, n, n));
  return finish(h);
}

extern "C" int gpb200_gram_deriv(gpb200_handle_t h, int n, const double *t, double alpha, double rho, int nblocks,
                                 const double *noise, double jitter, int quirk, double *K, int ldk) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "gram_deriv: negative n");
  if (nblocks < 1 || nblocks > 3) BAD_ARG(h, 6, "gram_deriv: nblocks must be 1..3");
  const int N = n * nblocks;
  if (ldk < std::max(1, N)) BAD_ARG(h, 11, "gram_deriv: ldk too small");
  if (n == 0) return 0;
  double nz[3] = {0, 0, 0};
  if (h->device_ptrs) {
    GPB_CUDA(h, cudaMemcpyAsync(nz, noise, nblocks * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    GPB_CUDA(h, cudaStreamSynchronize(h->stream));
    return launch_gram_deriv(h, n, nblocks, t, alpha, rho, nz, jitter, quirk, K, ldk);
  }
  for (int b = 0; b < nblocks; b++) nz[b] = noise[b];
  Arena a;
  RC(ws_reserve(h, pad256(n * 8) + pad256((size_t)N * N * 8), &a));
  double *dt = a.take<double>(n), *dK = a.take<double>((size_t)N * N);
  RC(to_device(h, t, dt, n));
  RC(launch_gram_deriv(h, n, nblocks, dt, alpha, rho, nz, jitter, quirk, dK, N));
  RC(from_device_2d(h, dK, N, K, ldk, N, N));
  return finish(h);
}

extern "C" int gpb200_approx_L_basis(gpb200_handle_t h, int n, int M, double scale, const double *x, double sigma,
                                     double l, double *out, int ldo) {
  CHECK_H(h);
  if (n < 0 || M < 1) BAD_ARG(h, 2, "approx_L_basis: bad sizes");
  if (ldo < std::max(1, n)) BAD_ARG(h, 9, "approx_L_basis: ldo < n");
  if (n == 0) return 0;
  if (h->device_ptrs) return launch_approx_basis(h, n, M, scale, x, sigma, l, out, ldo);
  Arena a;
  RC(ws_reserve(h, pad256(n * 8) + pad256((size_t)n * M * 8), &a));
  double *dx = a.take<double>(n), *dout = a.take<double>((size_t)n * M);
  RC(to_device(h, x, dx, n));
  RC(launch_approx_basis(h, n, M, scale, dx, sigma, l, dout, n));
  RC(from_device_2d(h, dout, n, out, ldo, n, M));
  return finish(h);
}

// =================================================================================================
// a6-a8 factorisation and solves on caller matrices
// =================================================================================================
extern "C" int gpb200_potrf(gpb200_handle_t h, int n, double *A, int lda) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "potrf: negative n");
  if (lda < std::max(1, n)) BAD_ARG(h, 4, "potrf: lda < n");
  if (n > MAX_DENSE_N) BAD_ARG(h, 2, "potrf: n above 65407 is not supported by the dense entry points (use the block-cyclic path)");
  if (n == 0) return 0;
  const int np = round_up(n, TILE);
  Arena a;
  const size_t mat = pad256((size_t)np * np * 8);
  RC(ws_reserve(h, mat + (h->device_ptrs ? 0 : mat) + 512, &a));
  double *Lbuf = a.take<double>((size_t)np * np);
  int *info = a.take<int>(1);
  GPB_CUDA(h, cudaMemsetAsync(info, 0, sizeof(int), h->stream));
  const double *src = A;
  long long lds = lda;
  if (!h->device_ptrs) {
    double *stage = a.take<double>((size_t)np * np);
    RC(to_device_2d(h, A, lda, stage, n, n, n));
    src = stage;
    lds = n;
  }
  RC(launch_pack(h, n, n, src, lds, np, np, Lbuf, 1, 0.0));
  RC(chol_batched(h, Lbuf, np, (long long)np * np, n, 1, info));
  int hinfo = 0;
  RC(read_info(h, info, &hinfo));
  if (h->device_ptrs) {
    RC(launch_unpack(h, n, n, Lbuf, np, A, lda, 1, 0.0));
  } else {
    double *stage = const_cast<double *>(src);
    RC(launch_unpack(h, n, n, Lbuf, np, stage, n, 1, 0.0));
    RC(from_device_2d(h, stage, n, A, lda, n, n));
  }
  RC(finish(h));
  return hinfo;
}

namespace {
// shared body of trsm_lower / potrs / trmv / mvn lpdf: bring L (n x n lower) into a padded buffer
int stage_lower(Handle *h, Arena &a, int n, int np, const double *L, int ldl, double **Lbuf_out) {
  double *Lbuf = a.take<double>((size_t)np * np);
  if (!Lbuf) BAD_ARG(h, 1002, "workspace exhausted");
  if (h->device_ptrs) {
    RC(launch_pack(h, n, n, L, ldl, np, np, Lbuf, 2, 0.0));
  } else {
    double *stage = a.take<double>((size_t)n * n);
    if (!stage) BAD_ARG(h, 1002, "workspace exhausted");
    RC(to_device_2d(h, L, ldl, stage, n, n, n));
    RC(launch_pack(h, n, n, stage, n, np, np, Lbuf, 2, 0.0));
  }
  *Lbuf_out = Lbuf;
  return 0;
}

// X = W * B (W lower-triangular inverse in Lbuf, B np x rp padded) and optionally X = W^T * X
int tasks_mul(Handle *h, int kind, int nt, int rt, TaskList *out) {
  const long long key = tkey(kind, nt, rt);
  if (cached(h, key, out)) return 0;
  std::vector<TileTask> t;
  for (int i = 0; i < nt; i++)
    for (int j = 0; j < rt; j++) {
      if (kind == TK_MUL_WB)  // X[i,j] = sum_{k<=i} W[i,k] B[k,j]   (NN)
        t.push_back({i * TILE, 0, 0, j * TILE, i * TILE, j * TILE, (i + 1) * TILE, 0});
      else                    // X[i,j] = sum_{k>=i} W[k,i] B[k,j]   (TN)
        t.push_back({i * TILE, i * TILE, i * TILE, j * TILE, i * TILE, j * TILE, (nt - i) * TILE, 0});
    }
  sort_desc(t, 0);
  std::vector<int> off = {0, (int)t.size()};
  return upload_tasks(h, key, t, off, out);
}

int solve_common(Handle *h, int n, int nrhs, const double *L, int ldl, double *B, int ldb, bool both) {
  const int np = round_up(n, TILE), rp = round_up(nrhs, TILE);
  const size_t mat = pad256((size_t)np * np * 8), rhs = pad256((size_t)np * rp * 8);
  Arena a;
  RC(ws_reserve(h, 3 * mat + 3 * rhs + 1024, &a));
  double *Lbuf = nullptr;
  RC(stage_lower(h, a, n, np, L, ldl, &Lbuf));
  double *Sbuf = a.take<double>((size_t)np * np);
  double *B0 = a.take<double>((size_t)np * rp), *B1 = a.take<double>((size_t)np * rp);
  const double *src = B;
  long long lds = ldb;
  if (!h->device_ptrs) {
    double *stage = a.take<double>((size_t)n * nrhs);
    RC(to_device_2d(h, B, ldb, stage, n, n, nrhs));
    src = stage;
    lds = n;
  }
  RC(launch_pack(h, n, nrhs, src, lds, np, rp, B0, 0, 0.0));
  RC(trtri_batched(h, Lbuf, Sbuf, np, (long long)np * np, 1));
  const int nt = np / TILE, rt = rp / TILE;
  TaskList t1;
  RC(tasks_mul(h, TK_MUL_WB, nt, rt, &t1));
  GemmParams p{};
  p.A = mref(Lbuf, np, 0);
  p.B = mref(B0, np, 0);
  p.C = mref(B1, np, 0);
  p.alpha = 1.0;
  p.tasks = t1.at(0);
  RC(launch_gemm(h, LAYOUT_NN, EPI_AXPBY, p, t1.count(0), 1));
  double *res = B1;
  if (both) {
    TaskList t2;
    RC(tasks_mul(h, TK_MUL_WTB, nt, rt, &t2));
    GemmParams q{};
    q.A = mref(Lbuf, np, 0);
    q.B = mref(B1, np, 0);
    q.C = mref(B0, np, 0);
    q.alpha = 1.0;
    q.tasks = t2.at(0);
    RC(launch_gemm(h, LAYOUT_TN, EPI_AXPBY, q, t2.count(0), 1));
    res = B0;
  }
  if (h->device_ptrs) {
    RC(launch_unpack(h, n, nrhs, res, np, B, ldb, 0, 0.0));
  } else {
    double *stage = const_cast<double *>(src);
    RC(launch_unpack(h, n, nrhs, res, np, stage, n, 0, 0.0));
    RC(from_device_2d(h, stage, n, B, ldb, n, nrhs));
  }
  return finish(h);
}
}  // namespace

extern "C" int gpb200_trsm_lower(gpb200_handle_t h, int n, int nrhs, const double *L, int ldl, double *B, int ldb) {
  CHECK_H(h);
  if (n < 0 || nrhs < 0) BAD_ARG(h, 2, "trsm_lower: negative size");
  if (ldl < std::max(1, n) || ldb < std::max(1, n)) BAD_ARG(h, 5, "trsm_lower: bad leading dimension");
  if (n == 0 || nrhs == 0) return 0;
  if (n > MAX_DENSE_N || nrhs > MAX_DENSE_N) BAD_ARG(h, 2, "trsm_lower: sizes above 65407 are not supported");
  return solve_common(h, n, nrhs, L, ldl, B, ldb, false);
}

extern "C" int gpb200_potrs(gpb200_handle_t h, int n, int nrhs, const double *L, int ldl, double *B, int ldb) {
  CHECK_H(h);
  if (n < 0 || nrhs < 0) BAD_ARG(h, 2, "potrs: negative size");
  if (ldl < std::max(1, n) || ldb < std::max(1, n)) BAD_ARG(h, 5, "potrs: bad leading dimension");
  if (n == 0 || nrhs == 0) return 0;
  if (n > MAX_DENSE_N || nrhs > MAX_DENSE_N) BAD_ARG(h, 2, "potrs: sizes above 65407 are not supported");
  return solve_common(h, n, nrhs, L, ldl, B, ldb, true);
}

extern "C" int gpb200_trmv_lower(gpb200_handle_t h, int n, const double *L, int ldl, const double *z, double *f) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "trmv_lower: negative n");
  if (ldl < std::max(1, n)) BAD_ARG(h, 4, "trmv_lower: ldl < n");
  if (n == 0) return 0;
  const int np = round_up(n, TILE);
  Arena a;
  RC(ws_reserve(h, 2 * pad256((size_t)np * np * 8) + 4 * pad256(np * 8), &a));
  double *Lbuf = nullptr;
  RC(stage_lower(h, a, n, np, L, ldl, &Lbuf));
  double *dz = a.take<double>(np), *df = a.take<double>(np);
  RC(to_device(h, z, dz, n));
  RC(launch_trmv_lower_n(h, np, Lbuf, 0, dz, 0, n, df, 0, 1));
  RC(from_device(h, df, f, n * sizeof(double)));
  return finish(h);
}

extern "C" int gpb200_trmv_lower_t(gpb200_handle_t h, int n, const double *L, int ldl, const double *z, double *f) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "trmv_lower_t: negative n");
  if (ldl < std::max(1, n)) BAD_ARG(h, 4, "trmv_lower_t: ldl < n");
  if (n == 0) return 0;
  const int np = round_up(n, TILE);
  Arena a;
  RC(ws_reserve(h, 2 * pad256((size_t)np * np * 8) + 4 * pad256(np * 8), &a));
  double *Lbuf = nullptr;
  RC(stage_lower(h, a, n, np, L, ldl, &Lbuf));
  double *dz = a.take<double>(np), *df = a.take<double>(np);
  GPB_CUDA(h, cudaMemsetAsync(dz, 0, sizeof(double) * np, h->stream));
  RC(to_device(h, z, dz, n));
  RC(launch_trmv_lower_t(h, np, Lbuf, 0, dz, 0, df, 0, 1));
  RC(from_device(h, df, f, n * sizeof(double)));
  return finish(h);
}

extern "C" int gpb200_mvn_chol_lpdf(gpb200_handle_t h, int n, const double *y, const double *mu, const double *L,
                                    int ldl, int drop_constants, double *lp) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "mvn_chol_lpdf: negative n");
  if (ldl < std::max(1, n)) BAD_ARG(h, 6, "mvn_chol_lpdf: ldl < n");
  const int np = round_up(std::max(n, 1), TILE);
  Arena a;
  RC(ws_reserve(h, 3 * pad256((size_t)np * np * 8) + 8 * pad256(np * 8), &a));
  double *Lbuf = nullptr;
  RC(stage_lower(h, a, n, np, L, ldl, &Lbuf));
  double *Wd = a.take<double>((size_t)np * np);
  double *dy = a.take<double>(np), *dmu = a.take<double>(np), *dz = a.take<double>(np), *out2 = a.take<double>(2);
  RC(to_device(h, y, dy, n));
  if (mu) RC(to_device(h, mu, dmu, n));
  RC(launch_tile_inverse(h, Lbuf, Wd, np, 0, np / TILE, 1));
  double *dacc = a.take<double>(np);
  RC(launch_trsv_sweep(h, np, Lbuf, Wd, 0, dy, 0, mu ? dmu : nullptr, n, dz, dacc, np, 1));
  RC(launch_sumsq_logdiag(h, n, dz, Lbuf, np, out2));
  double r[2];
  GPB_CUDA(h, cudaMemcpyAsync(r, out2, sizeof(r), cudaMemcpyDeviceToHost, h->stream));
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  double v = -r[1] - 0.5 * r[0];
  if (!drop_constants) v -= 0.5 * n * 1.8378770664093454835606594728112;
  if (h->device_ptrs) {
    GPB_CUDA(h, cudaMemcpyAsync(lp, &v, sizeof(double), cudaMemcpyHostToDevice, h->stream));
    GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  } else {
    *lp = v;
  }
  return 0;
}


// =================================================================================================
// tuning aid: times one panel kernel in isolation on `batch` synthetic SE Gram matrices of nt x nt tiles
// (CUDA events around each launch; the matrices are rebuilt before every repetition).
//   what = 0  POTRF of the first diagonal tile           (1 CTA per item)
//   what = 1  TRSM of the nt-1 tiles below it             (after the POTRF)
//   what = 2  inverse of the nt diagonal tiles            (after a full factorisation)
//   what = 3  POTRF + TRSM of the first block column      (one fused launch where that applies, else the two launches)
// ms_out[0] = mean kernel time in ms.  DEVICE work only; not part of the reference-facing surface.
// =================================================================================================
extern "C" int gpb200_debug_bench_panel(gpb200_handle_t h, int what, int nt, int batch, int reps, double *ms_out) {
  CHECK_H(h);
  if (nt < 1 || batch < 1 || reps < 1 || what < 0 || what > 3) BAD_ARG(h, 2, "debug_bench_panel: bad arguments");
  const int np = nt * TILE, n = np;
  const long long mat = (long long)np * np;
  Arena a;
  RC(ws_reserve(h, pad256(mat * 8) * batch * 2 + pad256(n * 8) + 4096, &a));
  double *Lbuf = a.take<double>((size_t)mat * batch), *Wbuf = a.take<double>((size_t)mat * batch);
  double *dx = a.take<double>(n), *dth = a.take<double>(3 * (size_t)batch);
  int *info = a.take<int>(batch);
  if (!info) BAD_ARG(h, 1002, "debug_bench_panel: workspace exhausted");
  std::vector<double> x(n), th(3 * (size_t)batch);
  for (int i = 0; i < n; i++) x[i] = 0.05 * i;
  for (int b = 0; b < batch; b++) { th[3 * b] = 1.0; th[3 * b + 1] = 1.0; th[3 * b + 2] = 0.3; }
  GPB_CUDA(h, cudaMemcpyAsync(dx, x.data(), n * 8, cudaMemcpyHostToDevice, h->stream));
  GPB_CUDA(h, cudaMemcpyAsync(dth, th.data(), th.size() * 8, cudaMemcpyHostToDevice, h->stream));
  GPB_CUDA(h, cudaMemsetAsync(info, 0, batch * sizeof(int), h->stream));
  cudaEvent_t e0, e1;
  GPB_CUDA(h, cudaEventCreate(&e0));
  GPB_CUDA(h, cudaEventCreate(&e1));
  double total = 0.0;
  int rc = 0;
  for (int r = 0; r < reps + 1 && !rc; r++) {  // repetition 0 is a warm-up
    rc = launch_gram_se_batched(h, n, np, dx, 0, dth, 0.0, 1, Lbuf, mat, batch);
    if (!rc && (what == 1 || what == 2)) rc = launch_potrf_tile(h, Lbuf, np, mat, 0, n, batch, info);
    if (!rc && what == 2) rc = chol_batched(h, Lbuf, np, mat, n, batch, info);
    if (rc) break;
    cudaEventRecord(e0, h->stream);
    if (what == 0) rc = launch_potrf_tile(h, Lbuf, np, mat, 0, n, batch, info);
    else if (what == 1) rc = launch_trsm_tiles(h, Lbuf, np, mat, 0, nt - 1, batch);
    else if (what == 3) rc = launch_potrf_trsm(h, Lbuf, np, mat, 0, nt - 1, n, batch, info);
    else rc = launch_tile_inverse(h, Lbuf, Wbuf, np, mat, nt, batch);
    cudaEventRecord(e1, h->stream);
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) rc = -1000;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (r > 0) total += ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (rc) return rc;
  ms_out[0] = total / reps;
  return 0;
}

// instrumented builds only (-DGPB_PANEL_TRACE): clock64 stamps the panel kernels left for CTA 0 (tuning aid)
extern "C" int gpb200_debug_panel_trace(gpb200_handle_t h, long long *out2048) {
  CHECK_H(h);
  GPB_CUDA(h, cudaDeviceSynchronize());
  return panel_trace_fetch(out2048);
}

// Accounting of the flops the DMMA GEMM launches really execute: 2 * tile area * k per CTA after the CTA-uniform skipping.
// Launches whose skipping is fixed by the task lists are counted on the host; launches that skip tiles outside an item's
// envelope count on the device, per CTA, into a counter the getter reads back (it waits for the handle's stream).
// on != 0 resets the counter and starts counting; the getter returns the running total.
extern "C" int gpb200_set_flop_counting(gpb200_handle_t h, int on) {
  CHECK_H(h);
  h->count_flops = on ? 1 : 0;
  h->executed_gemm_flops = 0.0;
  if (on) {
    if (!h->flops_dev) GPB_CUDA(h, cudaMalloc(&h->flops_dev, sizeof(unsigned long long)));
    GPB_CUDA(h, cudaMemsetAsync(h->flops_dev, 0, sizeof(unsigned long long), h->stream));
  }
  return 0;
}
extern "C" double gpb200_executed_gemm_flops(gpb200_handle_t h) {
  if (!h) return 0.0;
  DeviceGuard guard(h->device);
  unsigned long long dev = 0;
  if (h->flops_dev && (cudaMemcpyAsync(&dev, h->flops_dev, sizeof(dev), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
                       cudaStreamSynchronize(h->stream) != cudaSuccess))
    dev = 0;
  return h->executed_gemm_flops + (double)dev;
}
