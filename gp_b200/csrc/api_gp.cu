// C-ABI entry points: fused Gram -> Cholesky -> LML + gradient (CS-A), forward-mode Cholesky tangent
// (rbf_cov_chol and friends), Hermite interpolation of tabulated factors, conditioning (a10).
#include "host.cuh"

using namespace gpb;

// =================================================================================================
// =================================================================================================
// CS-A fused LML + gradient
// =================================================================================================
namespace {
// which covariance the fused path assembles: the SE kernel of fit_hyperparameters.stan (deriv = false,
// theta = (alpha, rho, sigma)), the joint derivative-observation covariance (deriv = true,
// theta = (alpha, rho, noise[nblocks])) on a grid of n_grid points, or the ARD kernel on n_grid points in
// ard_d > 0 dimensions (theta = (alpha, rho[ard_d], sigma); x per item n_grid x ard_d column-major)
struct LmlSpec { bool deriv; int n_grid, order0, nblocks; int ard_d; };

int lml_core(gpb200_handle_t h, const LmlSpec &sp, int B, const double *x, long long x_stride,
             const double *y, long long y_stride, const double *theta, double jitter,
             int want_grad, double *lml, double *grad, int *info) {
  const bool ard = sp.ard_d > 0;
  const int ng = sp.n_grid, n = sp.n_grid * sp.nblocks, ts = sp.deriv ? 2 + sp.nblocks : (ard ? 2 + sp.ard_d : 3);
  const int xl = ard ? ng * sp.ard_d : ng;  // doubles of x per item
  const GemmEpi epi = sp.deriv ? EPI_TRACE_DERIV : (ard ? EPI_TRACE_ARD : EPI_TRACE);
  const int pw = epi_partial_width(epi);  // doubles per tile partial
  if (B == 0) return 0;
  const int np = round_up(n, TILE), nt = np / TILE;
  const long long mat = (long long)np * np;
  TaskList tl;
  RC(tasks_lauum(h, nt, &tl));
  const int ntasks = tl.count(0);
  const int nparts = ntasks * 4;  // trace partial records per item: one per CTA, at most four CTAs per tile

  // chunk the batch so that the resident set fits the workspace limit.  cudaMemGetInfo costs
  // milliseconds with tens of GB allocated, so it is only consulted when the workspace must grow.
  // n <= 128: one CTA per item does the whole evaluation in shared memory (small.cu); no O(n^2) workspace at all
  const bool small = !sp.deriv && !ard && lml_small_applies(h, n);
  if (small && h->device_ptrs && info && lml && (grad || !want_grad)) {
    // device-pointer mode: the kernel reads the caller's arrays and writes the caller's results in place --
    // ONE launch per call, no staging copies, no memset (the kernel writes every info word)
    return launch_lml_small(h, n, x, x_stride, y, y_stride, theta, jitter, want_grad, lml, grad, info, B);
  }
  const int zks = trmv_split_chunks(np, B);  // k-chunks of the split z = W y (small batches only)
  // SE covariance: the envelope of every item (common.cuh, ENV_BLK) bounds the Cholesky, and larger batches compute the
  // gradient from the selected inverse instead of the explicit inverse + W^T W.  Measured on a B200 (1000 W), LML +
  // gradient per call on the bench.py family, dense / envelope + explicit inverse / envelope + selected inverse, ms:
  //   N = 1024: B = 1 0.452 / 0.458 / 0.85,  B = 32 2.10 / 1.98 / 2.12   (nt = 8: the band covers the matrix, the
  //             profile costs its launch; no envelope below 16 tile rows)
  //   N = 2048: B = 1 0.948 / 0.949 / 2.34,  B = 8 3.46 / 2.93 / 3.70,  B = 16 6.26 / 5.20 / 4.96,  B = 32 11.0 / 9.59 / 7.67
  //   N = 4096: B = 1 3.36 / 2.98 / 4.59,    B = 4 10.19 / 7.91 / 8.36,  B = 8 19.3 / 14.4 / 8.2,  B = 32 70.9 / 53.4 / 22.0
  // The selected inverse is a chain of 2 nt launches of a few tiles per item: it wins once B * nt >= 256.
  const bool use_env = !sp.deriv && !ard && h->envelope && !small && nt >= 16 && nt <= ENV_MAX_NT;
  const bool sinv = use_env && want_grad && (h->sinv_min_batch > 0 ? B >= h->sinv_min_batch : (long long)B * nt >= 256);
  const size_t per_item = small ? 0 : pad256(mat * 8) * 2 + 3 * pad256(np * 8) + pad256((size_t)nparts * pw * 8) + (zks > 1 ? pad256((size_t)zks * np * 8) : 0) + 64 +
                                      (use_env ? (size_t)(env_record_ints(nt) + 2) * sizeof(int) : 0);
  const size_t fixed = pad256((size_t)B * (x_stride ? xl : 0) * 8 + (size_t)xl * 8) + pad256((size_t)B * (y_stride ? n : 0) * 8 + n * 8) +
                       2 * pad256((size_t)B * ts * 8) + pad256((size_t)B * 8) + pad256((size_t)B * 4) + 4096 + (use_env ? 512 : 0);
  int Bc = B;
  if (!small && (h->ws_limit > 0 || fixed + per_item * (size_t)B + 8192 > h->ws_bytes)) {
    size_t limit = (size_t)h->ws_limit;
    if (h->ws_limit <= 0) {
      size_t freeb = 0, totalb = 0;
      GPB_CUDA(h, cudaMemGetInfo(&freeb, &totalb));
      limit = (size_t)((freeb + h->ws_bytes) * 0.85);
    }
    if (limit < fixed + per_item + 8192) BAD_ARG(h, 1002, "lml_grad_batched: workspace limit too small for one item");
    Bc = (int)std::min<size_t>((size_t)B, (limit - fixed - 8192) / per_item);
  }
  if (!small) Bc = std::min(Bc, 65535);  // gridDim.y of the batched launches
  Arena a;
  RC(ws_reserve(h, fixed + per_item * (size_t)Bc + 8192, &a));

  const long long xs = x_stride ? xl : 0, ys = y_stride ? n : 0;
  double *dx = a.take<double>(x_stride ? (size_t)B * xl : xl);
  double *dy = a.take<double>(y_stride ? (size_t)B * n : n);
  double *dth = a.take<double>((size_t)B * ts);
  double *dlml = a.take<double>(B), *dgrad = a.take<double>((size_t)B * ts);
  int *dinfo = a.take<int>(B);
  double *Lbuf = nullptr, *Sbuf = nullptr, *zbuf = nullptr, *abuf = nullptr, *dvec = nullptr, *partial = nullptr, *zpart = nullptr;
  int *env = nullptr, *order = nullptr;
  if (!small) {
    Lbuf = a.take<double>((size_t)Bc * mat); Sbuf = a.take<double>((size_t)Bc * mat);
    zbuf = a.take<double>((size_t)Bc * np); abuf = a.take<double>((size_t)Bc * np); dvec = a.take<double>((size_t)Bc * np);
    partial = a.take<double>((size_t)Bc * nparts * pw);
    zpart = zks > 1 ? a.take<double>((size_t)Bc * zks * np) : nullptr;
    if (use_env && (!(env = a.take<int>((size_t)Bc * env_record_ints(nt))) || !(order = a.take<int>((size_t)Bc * 2))))
      BAD_ARG(h, 1002, "lml_grad_batched: workspace arithmetic error");
    if (!partial) BAD_ARG(h, 1002, "lml_grad_batched: workspace arithmetic error");
  }
  if (!dinfo) BAD_ARG(h, 1002, "lml_grad_batched: workspace arithmetic error");

  // The kernel sequence (everything between staging the inputs and reading the outputs).
  auto run_sequence = [&]() -> int {
    GPB_CUDA(h, cudaMemsetAsync(dinfo, 0, (size_t)B * sizeof(int), h->stream));
    if (small) return launch_lml_small(h, n, dx, xs, dy, ys, dth, jitter, want_grad, dlml, dgrad, dinfo, B);
    for (int b0 = 0; b0 < B; b0 += Bc) {
      const int bc = std::min(Bc, B - b0);
      const double *cx = dx + (long long)b0 * xs, *cy = dy + (long long)b0 * ys, *cth = dth + (long long)b0 * ts;
      if (sp.deriv) RC(launch_gram_deriv_batched(h, ng, sp.order0, sp.nblocks, np, cx, xs, cth, ts, jitter, 1, Lbuf, mat, bc));
      else if (ard) RC(launch_gram_ard_batched(h, n, sp.ard_d, np, cx, xs, cth, jitter, Lbuf, mat, bc));
      else {
        if (env) GPB_CUDA(h, cudaMemsetAsync(env, 0xff, (size_t)bc * env_record_ints(nt) * sizeof(int), h->stream));  // fb UINT_MAX, er -1
        RC(launch_gram_se_batched(h, n, np, cx, xs, cth, jitter, 1, Lbuf, mat, bc, env));
        if (env) RC(launch_envelope_profile(h, nt, env, order, bc));
      }
      RC(chol_batched(h, Lbuf, np, mat, n, bc, dinfo + b0, env, order));
      RC(extract_diag(h, np, Lbuf, mat, dvec, bc));
      int n1 = 0, n2 = 0;
      if (sinv) {
        RC(launch_tile_inverse(h, Lbuf, Sbuf, np, mat, nt, bc));
        RC(launch_trsv_blocked(h, np, Lbuf, Sbuf, mat, cy, ys, nullptr, n, zbuf, np, bc, env));
        RC(launch_backsub_band(h, np, Lbuf, Sbuf, mat, env, zbuf, abuf, bc));
        RC(sinv_batched(h, Lbuf, Sbuf, np, mat, env, order, bc));
        RC(launch_trace_sinv(h, n, np, Lbuf, mat, env, cx, xs, abuf, cth, partial, bc));
        n1 = ntasks;
      } else if (want_grad) {
        RC(trtri_batched(h, Lbuf, Sbuf, np, mat, bc));
        if (zks > 1 && zpart) RC(launch_trmv_lower_n_split(h, np, zks, Lbuf, mat, cy, ys, n, zpart, zbuf, np, bc));
        else RC(launch_trmv_lower_n(h, np, Lbuf, mat, cy, ys, n, zbuf, np, bc));
        RC(launch_trmv_lower_t(h, np, Lbuf, mat, zbuf, np, abuf, np, bc));
        GemmParams p{};
        p.A = mref(Lbuf, np, mat);
        p.B = mref(Lbuf, np, mat);
        p.C = mref(nullptr, np, mat);
        p.tasks = tl.at(0);
        p.x = cx; p.x_stride = xs;
        p.avec = abuf; p.a_stride = np;
        p.theta = cth;
        p.partial = partial;
        p.n = n;
        p.ntasks = ntasks;
        p.n_grid = ng; p.order0 = sp.order0; p.theta_stride = ts;
        p.ard_d = sp.ard_d;
        RC(launch_gemm(h, LAYOUT_TN, epi, p, ntasks, bc));
      } else {
        RC(launch_tile_inverse(h, Lbuf, Sbuf, np, mat, nt, bc));
        if (bc >= 32) RC(launch_trsv_blocked(h, np, Lbuf, Sbuf, mat, cy, ys, nullptr, n, zbuf, np, bc, env));
        else RC(launch_trsv_sweep(h, np, Lbuf, Sbuf, mat, cy, ys, nullptr, n, zbuf, abuf, np, bc));
      }
      if (!sinv) RC(gemm_partial_layout(h, tl.at(0), ntasks, bc, &n1, &n2));
      if (ard)
        RC(launch_finalize_ard(h, n, sp.ard_d, np, want_grad, dvec, zbuf, abuf, partial, n1, n2, cth, dlml + b0,
                               dgrad + (long long)b0 * ts, bc));
      else if (sp.deriv)
        RC(launch_finalize_deriv(h, ng, sp.nblocks, np, want_grad, dvec, zbuf, abuf, partial, n1, n2, cth, dlml + b0,
                                 dgrad + (long long)b0 * ts, bc));
      else
        RC(launch_finalize(h, n, np, want_grad, dvec, zbuf, abuf, partial, n1, n2, cth, dlml + b0, dgrad + (long long)b0 * 3, bc));
    }
    return 0;
  };

  // Small problems are launch-latency bound (tens of launches of a few microseconds each): replay
  // them as one CUDA graph on the handle's own stream, ordered against the caller's stream by events.
  const bool use_graph = !small && h->graphs_enabled && !h->profiling && Bc == B && nt <= 64 && (long long)B * nt * nt <= 4096;
  cudaStream_t user_stream = h->stream;
  if (use_graph) {
    GPB_CUDA(h, cudaEventRecord(h->g_in, user_stream));
    GPB_CUDA(h, cudaStreamWaitEvent(h->gstream, h->g_in, 0));
    h->stream = h->gstream;
  }
  int rc = 0;
  do {
    if (x_stride) rc = to_device_2d(h, x, x_stride, dx, xl, xl, B); else rc = to_device(h, x, dx, xl);
    if (rc) break;
    if (y_stride) rc = to_device_2d(h, y, y_stride, dy, n, n, B); else rc = to_device(h, y, dy, n);
    if (rc) break;
    if ((rc = to_device(h, theta, dth, (size_t)B * ts))) break;
    if (!use_graph) {
      rc = run_sequence();
    } else {
      long long jbits;
      memcpy(&jbits, &jitter, sizeof(jbits));
      const std::vector<long long> key = {n, B, want_grad, xs, ys, jbits, (long long)(uintptr_t)h->ws, h->chol_panel_override,
                                          sp.deriv, sp.order0, sp.nblocks, h->gemm_cfg_override, h->lookahead, h->lookahead_max_batch,
                                          h->quarter_below_waves, h->trsm_pipelined, h->panel_fused, h->fine_cfg,
                                          h->envelope, h->sinv_min_batch, sp.ard_d};
      auto it = h->graphs.find(key);
      if (it == h->graphs.end()) {
        // task lists allocate and synchronise on first use, which a capture does not allow: a first uncaptured
        // pass builds every list the sequence needs (its results are simply overwritten by the replay)
        if ((rc = run_sequence())) break;
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(h->gstream, cudaStreamCaptureModeRelaxed) != cudaSuccess) { rc = -1000; break; }
        const long long before = h->launches;
        rc = run_sequence();
        const cudaError_t ce = cudaStreamEndCapture(h->gstream, &graph);
        if (rc || ce != cudaSuccess) { if (graph) cudaGraphDestroy(graph); if (!rc) rc = -1000; break; }
        cudaGraphExec_t exec = nullptr;
        if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) { cudaGraphDestroy(graph); rc = -1000; break; }
        cudaGraphDestroy(graph);
        it = h->graphs.emplace(key, Handle::GraphEntry{exec, h->launches - before}).first;
        h->launches = before;  // counted per replay below
      }
      if (cudaGraphLaunch(it->second.exec, h->gstream) != cudaSuccess) { rc = -1001; break; }
      h->launches += it->second.nodes;
      h->graph_replays++;
    }
    if (rc) break;
    if ((rc = from_device(h, dlml, lml, (size_t)B * sizeof(double)))) break;
    if (want_grad && grad && (rc = from_device(h, dgrad, grad, (size_t)B * ts * sizeof(double)))) break;
    if (info && (rc = from_device(h, dinfo, info, (size_t)B * sizeof(int)))) break;
    rc = finish(h);
  } while (0);
  if (use_graph) {
    h->stream = user_stream;
    cudaEventRecord(h->g_out, h->gstream);
    cudaStreamWaitEvent(user_stream, h->g_out, 0);
  }
  if (rc && !h->err[0]) snprintf(h->err, sizeof(h->err), "lml_grad: CUDA graph path failed (%d)", rc);
  return rc;
}
}  // namespace

extern "C" int gpb200_lml_grad_batched(gpb200_handle_t h, int n, int B, const double *x, long long x_stride,
                                       const double *y, long long y_stride, const double *theta, double jitter,
                                       int want_grad, double *lml, double *grad, int *info) {
  CHECK_H(h);
  if (n < 1) BAD_ARG(h, 2, "lml_grad_batched: n must be >= 1");
  if (B < 0) BAD_ARG(h, 3, "lml_grad_batched: negative batch");
  if (x_stride != 0 && x_stride < n) BAD_ARG(h, 5, "lml_grad_batched: x_stride < n");
  if (y_stride != 0 && y_stride < n) BAD_ARG(h, 7, "lml_grad_batched: y_stride < n");
  return lml_core(h, LmlSpec{false, n, 0, 1}, B, x, x_stride, y, y_stride, theta, jitter, want_grad, lml, grad, info);
}

extern "C" int gpb200_lml_grad_deriv_batched(gpb200_handle_t h, int n, int order0, int nblocks, int B, const double *t,
                                             long long t_stride, const double *y, long long y_stride,
                                             const double *theta, double jitter, int want_grad, double *lml,
                                             double *grad, int *info) {
  CHECK_H(h);
  if (n < 1) BAD_ARG(h, 2, "lml_grad_deriv_batched: n must be >= 1");
  if (order0 < 0 || nblocks < 1 || order0 + nblocks > 3)
    BAD_ARG(h, 3, "lml_grad_deriv_batched: derivative orders must lie in 0..2 (order0 >= 0, nblocks >= 1, order0 + nblocks <= 3)");
  if (B < 0) BAD_ARG(h, 5, "lml_grad_deriv_batched: negative batch");
  if ((long long)n * nblocks > 2147483647LL / 2) BAD_ARG(h, 2, "lml_grad_deriv_batched: n * nblocks too large");
  if (t_stride != 0 && t_stride < n) BAD_ARG(h, 7, "lml_grad_deriv_batched: t_stride < n");
  if (y_stride != 0 && y_stride < (long long)n * nblocks) BAD_ARG(h, 9, "lml_grad_deriv_batched: y_stride < n * nblocks");
  return lml_core(h, LmlSpec{true, n, order0, nblocks}, B, t, t_stride, y, y_stride, theta, jitter, want_grad, lml, grad, info);
}

extern "C" int gpb200_lml_grad_ard_batched(gpb200_handle_t h, int n, int D, int B, const double *X, long long x_stride,
                                           const double *y, long long y_stride, const double *theta, double jitter,
                                           int want_grad, double *lml, double *grad, int *info) {
  CHECK_H(h);
  if (n < 1) BAD_ARG(h, 2, "lml_grad_ard_batched: n must be >= 1");
  if (D < 1 || D > ARD_MAX_D) BAD_ARG(h, 3, "lml_grad_ard_batched: D must lie in 1..8");
  if (B < 0) BAD_ARG(h, 4, "lml_grad_ard_batched: negative batch");
  if ((long long)n * D > 2147483647LL / 2) BAD_ARG(h, 2, "lml_grad_ard_batched: n * D too large");
  if (x_stride != 0 && x_stride < (long long)n * D) BAD_ARG(h, 6, "lml_grad_ard_batched: x_stride < n * D");
  if (y_stride != 0 && y_stride < n) BAD_ARG(h, 8, "lml_grad_ard_batched: y_stride < n");
  return lml_core(h, LmlSpec{false, n, 0, 1, D}, B, X, x_stride, y, y_stride, theta, jitter, want_grad, lml, grad, info);
}

// ---- B GPs of different sizes in one call ---------------------------------------------------------------------------
// Items are bucketed by tile count nt = ceil(n_b / 128); each bucket is a uniform lock-step batch at np = 128 nt whose
// kernels read the per-item size nvec.  The padding is exact: y is zero there and K_b is [K_b 0; 0 I], so the
// Cholesky, the inverses, the solves and the selected inverse run unchanged, and only the Gram, the trace epilogues and
// finalize need n_b.  Every bucket takes the routes lml_core would take for a batch of its size at its np.
namespace {
struct RaggedBucket {
  int nt, slot0, count, max_n;
  long long dst0;  // first double of the bucket in the staged x / y
  double work;     // count * nt^3: the bucket with the most work is dispatched first
};

// per-item workspace of the tiled SE route at np (the same terms as lml_core)
size_t se_item_bytes(int np, int nparts, int zks, bool use_env) {
  const long long mat = (long long)np * np;
  return pad256(mat * 8) * 2 + 3 * pad256(np * 8) + pad256((size_t)nparts * 4 * 8) + (zks > 1 ? pad256((size_t)zks * np * 8) : 0) +
         64 + (use_env ? (size_t)(env_record_ints(np / TILE) + 2) * sizeof(int) : 0);
}
}  // namespace

extern "C" int gpb200_lml_grad_ragged(gpb200_handle_t h, int B, const long long *offsets, const double *x, const double *y,
                                      const double *theta, double jitter, int want_grad, double *lml, double *grad, int *info) {
  CHECK_H(h);
  if (B < 0) BAD_ARG(h, 2, "lml_grad_ragged: B must be >= 0 (negative batch)");
  if (B == 0) return 0;
  if (!offsets) BAD_ARG(h, 3, "lml_grad_ragged: offsets is NULL");
  if (offsets[0] != 0) BAD_ARG(h, 3, "lml_grad_ragged: offsets[0] must be 0");
  for (int b = 0; b < B; b++) {
    const long long nb = offsets[b + 1] - offsets[b];
    const char *why = nb < 0 ? "offsets must be non-decreasing" : nb == 0 ? "every group needs n_b >= 1 point"
                      : nb > MAX_DENSE_N ? "n_b above 65407" : nullptr;
    if (why) {
      snprintf(h->err, sizeof(h->err), "lml_grad_ragged: %s (offsets[%d] = %lld, offsets[%d] = %lld)", why, b, offsets[b], b + 1,
               offsets[b + 1]);
      return -3;
    }
  }
  const long long ntot = offsets[B];

  // ---- schedule: buckets by tile count, caller order inside a bucket, the most work first ----
  std::map<int, std::vector<int>> by_nt;
  for (int b = 0; b < B; b++) by_nt[(int)((offsets[b + 1] - offsets[b] + TILE - 1) / TILE)].push_back(b);
  std::vector<RaggedBucket> bk;
  for (const auto &kv : by_nt) bk.push_back({kv.first, 0, (int)kv.second.size(), 0, 0, (double)kv.second.size() * kv.first * kv.first * kv.first});
  std::stable_sort(bk.begin(), bk.end(), [](const RaggedBucket &a, const RaggedBucket &c) {
    return a.work != c.work ? a.work > c.work : a.nt > c.nt;
  });
  std::vector<RaggedSlot> meta(B);
  int slot = 0;
  long long dst = 0;
  for (auto &k : bk) {
    const int np = k.nt * TILE;
    k.slot0 = slot;
    k.dst0 = dst;
    for (int b : by_nt[k.nt]) {
      const int nb = (int)(offsets[b + 1] - offsets[b]);
      meta[slot++] = RaggedSlot{offsets[b], dst, nb, np, b, 0};
      k.max_n = std::max(k.max_n, nb);
      dst += np;
    }
  }
  const long long xtot = dst;

  // ---- routes and workspace: per bucket as lml_core decides them for a uniform batch of the bucket's size ----
  struct Route { bool small, use_env, sinv; int zks, ntasks, Bc; size_t per_item; };
  std::vector<Route> rt(bk.size());
  const bool host = !h->device_ptrs;
  // staged x, y, theta, slot-order results, sizes, slot table; in host mode also the caller's inputs and the results
  // in caller order
  const size_t fixed = 2 * pad256((size_t)xtot * 8) + 2 * pad256((size_t)B * 3 * 8) + pad256((size_t)B * 8) + 2 * pad256((size_t)B * 4) +
                       pad256((size_t)B * sizeof(RaggedSlot)) +
                       (host ? 2 * pad256((size_t)ntot * 8) + 2 * pad256((size_t)B * 3 * 8) + pad256((size_t)B * 8) + pad256((size_t)B * 4)
                             : 0) +
                       4096;
  size_t need = 0;
  for (size_t k = 0; k < bk.size(); k++) {
    Route &r = rt[k];
    const int nt = bk[k].nt, np = nt * TILE, Bk = bk[k].count;
    r.small = nt == 1 && lml_small_applies(h, bk[k].max_n);
    r.use_env = h->envelope && !r.small && nt >= 16 && nt <= ENV_MAX_NT;
    r.sinv = r.use_env && want_grad && (h->sinv_min_batch > 0 ? Bk >= h->sinv_min_batch : (long long)Bk * nt >= 256);
    r.zks = trmv_split_chunks(np, Bk);
    r.ntasks = 0;
    if (!r.small) {
      TaskList tl;
      RC(tasks_lauum(h, nt, &tl));
      r.ntasks = tl.count(0);
    }
    r.per_item = r.small ? 0 : se_item_bytes(np, r.ntasks * 4, r.zks, r.use_env);
    r.Bc = Bk;
    need = std::max(need, r.per_item * (size_t)Bk);
  }
  if (h->ws_limit > 0 || fixed + need + 8192 > h->ws_bytes) {
    size_t limit = (size_t)h->ws_limit;
    if (h->ws_limit <= 0) {
      size_t freeb = 0, totalb = 0;
      GPB_CUDA(h, cudaMemGetInfo(&freeb, &totalb));
      limit = (size_t)((freeb + h->ws_bytes) * 0.85);
    }
    need = 0;
    for (Route &r : rt) {
      if (r.small) continue;
      if (limit < fixed + r.per_item + 8192) BAD_ARG(h, 1002, "lml_grad_ragged: workspace limit too small for one item");
      r.Bc = (int)std::min<size_t>((size_t)r.Bc, (limit - fixed - 8192) / r.per_item);
      need = std::max(need, r.per_item * (size_t)r.Bc);
    }
  }
  for (Route &r : rt)
    if (!r.small) r.Bc = std::min(r.Bc, 65535);  // gridDim.y of the batched launches
  Arena a;
  RC(ws_reserve(h, fixed + need + 8192, &a));
  double *sx = a.take<double>((size_t)xtot), *sy = a.take<double>((size_t)xtot), *sth = a.take<double>((size_t)B * 3);
  double *slml = a.take<double>(B), *sgrad = a.take<double>((size_t)B * 3);
  int *sinfo = a.take<int>(B), *snv = a.take<int>(B);
  RaggedSlot *dmeta = a.take<RaggedSlot>(B);
  const double *cx = x, *cy = y, *cth = theta;
  double *olml = lml, *ograd = want_grad ? grad : nullptr;
  int *oinfo = info;
  if (host) {
    double *hx = a.take<double>((size_t)ntot), *hy = a.take<double>((size_t)ntot), *hth = a.take<double>((size_t)B * 3);
    olml = lml ? a.take<double>(B) : nullptr;
    ograd = want_grad && grad ? a.take<double>((size_t)B * 3) : nullptr;
    oinfo = info ? a.take<int>(B) : nullptr;
    if (!hth) BAD_ARG(h, 1002, "lml_grad_ragged: workspace arithmetic error");
    RC(to_device(h, x, hx, (size_t)ntot));
    RC(to_device(h, y, hy, (size_t)ntot));
    RC(to_device(h, theta, hth, (size_t)B * 3));
    cx = hx; cy = hy; cth = hth;
  }
  if (!dmeta) BAD_ARG(h, 1002, "lml_grad_ragged: workspace arithmetic error");
  // pageable source: the copy has taken the vector's contents when cudaMemcpyAsync returns
  GPB_CUDA(h, cudaMemcpyAsync(dmeta, meta.data(), (size_t)B * sizeof(RaggedSlot), cudaMemcpyHostToDevice, h->stream));
  RC(launch_ragged_stage(h, B, dmeta, cx, cy, cth, sx, sy, sth, snv));
  GPB_CUDA(h, cudaMemsetAsync(sinfo, 0, (size_t)B * sizeof(int), h->stream));

  for (size_t k = 0; k < bk.size(); k++) {
    const RaggedBucket &K = bk[k];
    const Route &r = rt[k];
    const int nt = K.nt, np = nt * TILE;
    const long long mat = (long long)np * np;
    const double *bx = sx + K.dst0, *by = sy + K.dst0, *bth = sth + 3LL * K.slot0;
    const int *bnv = snv + K.slot0;
    double *blml = slml + K.slot0, *bgrad = sgrad + 3LL * K.slot0;
    int *binfo = sinfo + K.slot0;
    if (r.small) {
      RC(launch_lml_small(h, K.max_n, bx, np, by, np, bth, jitter, want_grad, blml, bgrad, binfo, K.count, bnv));
      continue;
    }
    TaskList tl;
    RC(tasks_lauum(h, nt, &tl));
    Arena ab = a;  // the buckets run one after the other on one stream: each reuses the same scratch
    double *Lbuf = ab.take<double>((size_t)r.Bc * mat), *Sbuf = ab.take<double>((size_t)r.Bc * mat);
    double *zbuf = ab.take<double>((size_t)r.Bc * np), *abuf = ab.take<double>((size_t)r.Bc * np), *dvec = ab.take<double>((size_t)r.Bc * np);
    double *partial = ab.take<double>((size_t)r.Bc * r.ntasks * 4 * 4);
    double *zpart = r.zks > 1 ? ab.take<double>((size_t)r.Bc * r.zks * np) : nullptr;
    int *env = nullptr, *order = nullptr;
    if (r.use_env && (!(env = ab.take<int>((size_t)r.Bc * env_record_ints(nt))) || !(order = ab.take<int>((size_t)r.Bc * 2))))
      BAD_ARG(h, 1002, "lml_grad_ragged: workspace arithmetic error");
    if (!partial || (r.zks > 1 && !zpart)) BAD_ARG(h, 1002, "lml_grad_ragged: workspace arithmetic error");
    for (int b0 = 0; b0 < K.count; b0 += r.Bc) {
      const int bc = std::min(r.Bc, K.count - b0);
      const double *ccx = bx + (long long)b0 * np, *ccy = by + (long long)b0 * np, *cct = bth + 3LL * b0;
      const int *cnv = bnv + b0;
      if (env) GPB_CUDA(h, cudaMemsetAsync(env, 0xff, (size_t)bc * env_record_ints(nt) * sizeof(int), h->stream));  // fb UINT_MAX, er -1
      RC(launch_gram_se_batched(h, np, np, ccx, np, cct, jitter, 1, Lbuf, mat, bc, env, cnv));
      if (env) RC(launch_envelope_profile(h, nt, env, order, bc));
      RC(chol_batched(h, Lbuf, np, mat, np, bc, binfo + b0, env, order));  // padded pivots are 1: info stays within n_b
      RC(extract_diag(h, np, Lbuf, mat, dvec, bc));
      int n1 = 0, n2 = 0;
      if (r.sinv) {
        RC(launch_tile_inverse(h, Lbuf, Sbuf, np, mat, nt, bc));
        RC(launch_trsv_blocked(h, np, Lbuf, Sbuf, mat, ccy, np, nullptr, np, zbuf, np, bc, env));
        RC(launch_backsub_band(h, np, Lbuf, Sbuf, mat, env, zbuf, abuf, bc));
        RC(sinv_batched(h, Lbuf, Sbuf, np, mat, env, order, bc));
        RC(launch_trace_sinv(h, np, np, Lbuf, mat, env, ccx, np, abuf, cct, partial, bc, cnv));
        n1 = r.ntasks;
      } else if (want_grad) {
        RC(trtri_batched(h, Lbuf, Sbuf, np, mat, bc));
        if (r.zks > 1) RC(launch_trmv_lower_n_split(h, np, r.zks, Lbuf, mat, ccy, np, np, zpart, zbuf, np, bc));
        else RC(launch_trmv_lower_n(h, np, Lbuf, mat, ccy, np, np, zbuf, np, bc));
        RC(launch_trmv_lower_t(h, np, Lbuf, mat, zbuf, np, abuf, np, bc));
        GemmParams p{};
        p.A = mref(Lbuf, np, mat);
        p.B = mref(Lbuf, np, mat);
        p.C = mref(nullptr, np, mat);
        p.tasks = tl.at(0);
        p.x = ccx; p.x_stride = np;
        p.avec = abuf; p.a_stride = np;
        p.theta = cct;
        p.partial = partial;
        p.n = np;
        p.nvec = cnv;
        p.ntasks = r.ntasks;
        p.theta_stride = 3;
        RC(launch_gemm(h, LAYOUT_TN, EPI_TRACE_RAGGED, p, r.ntasks, bc));
      } else {
        RC(launch_tile_inverse(h, Lbuf, Sbuf, np, mat, nt, bc));
        if (bc >= 32) RC(launch_trsv_blocked(h, np, Lbuf, Sbuf, mat, ccy, np, nullptr, np, zbuf, np, bc, env));
        else RC(launch_trsv_sweep(h, np, Lbuf, Sbuf, mat, ccy, np, nullptr, np, zbuf, abuf, np, bc));
      }
      if (!r.sinv) RC(gemm_partial_layout(h, tl.at(0), r.ntasks, bc, &n1, &n2));
      RC(launch_finalize(h, np, np, want_grad, dvec, zbuf, abuf, partial, n1, n2, cct, blml + b0, bgrad + 3LL * b0, bc, cnv));
    }
  }
  if (olml || ograd || oinfo) RC(launch_ragged_scatter(h, B, dmeta, slml, sgrad, sinfo, olml, ograd, oinfo));
  if (host) {
    if (lml) RC(from_device(h, olml, lml, (size_t)B * sizeof(double)));
    if (ograd) RC(from_device(h, ograd, grad, (size_t)B * 3 * sizeof(double)));
    if (info) RC(from_device(h, oinfo, info, (size_t)B * sizeof(int)));
  }
  return finish(h);
}

// number of CUDA-graph replays so far (small evaluations are replayed as one graph)
extern "C" long long gpb200_graph_replays(gpb200_handle_t h) { return h ? h->graph_replays : 0; }

extern "C" int gpb200_lml_grad(gpb200_handle_t h, int n, const double *x, const double *y, const double *theta,
                               double jitter, double *lml, double *grad) {
  CHECK_H(h);
  if (h->device_ptrs) {
    // info must live on the device in device-pointer mode: the handle's persistent slot (no allocation, nothing
    // that synchronises the device); only the read of the status word waits for the handle's stream
    int rc = gpb200_lml_grad_batched(h, n, 1, x, 0, y, 0, theta, jitter, grad != nullptr, lml, grad, h->info_slot);
    int hinfo = 0;
    if (rc == 0) rc = read_info(h, h->info_slot, &hinfo);
    return rc ? rc : hinfo;
  }
  int info = 0;
  int rc = gpb200_lml_grad_batched(h, n, 1, x, 0, y, 0, theta, jitter, grad != nullptr, lml, grad, &info);
  return rc ? rc : info;
}

// =================================================================================================
// a1-a3 rbf_cov_chol and its consumers
// =================================================================================================
namespace {
int tasks_tangent(Handle *h, int nt, TaskList *t1, TaskList *ta, TaskList *tl) {
  const long long k1 = tkey(TK_TAN_T1, nt), k2 = tkey(TK_TAN_A, nt), k3 = tkey(TK_TAN_LDOT, nt);
  if (cached(h, k1, t1) && cached(h, k2, ta) && cached(h, k3, tl)) return 0;
  std::vector<TileTask> v1, v2, v3;
  for (int i = 0; i < nt; i++)
    for (int j = 0; j <= i; j++) {
      // T1[i,j] = sum_{k<=i} W[i,k] Kdot[k,j]                       (NN)
      v1.push_back({i * TILE, 0, 0, j * TILE, i * TILE, j * TILE, (i + 1) * TILE, TF_A_TRI_LAST});
      // A[i,j]  = sum_{k<=j} T1[i,k] W[j,k]                          (NT)
      v2.push_back({i * TILE, 0, j * TILE, 0, i * TILE, j * TILE, (j + 1) * TILE, TF_B_TRI_LAST});
      // Ldot[i,j] = sum_{k=j..i} L[i,k] Phi[k,j]                     (NN)
      v3.push_back({i * TILE, j * TILE, j * TILE, j * TILE, i * TILE, j * TILE, (i - j + 1) * TILE, TF_A_TRI_LAST | TF_B_TRI_FIRST});
    }
  sort_desc(v1, 0); sort_desc(v2, 0); sort_desc(v3, 0);
  std::vector<int> o1 = {0, (int)v1.size()}, o2 = {0, (int)v2.size()}, o3 = {0, (int)v3.size()};
  RC(upload_tasks(h, k1, v1, o1, t1));
  RC(upload_tasks(h, k2, v2, o2, ta));
  return upload_tasks(h, k3, v3, o3, tl);
}
}  // namespace

namespace {
// L = chol(S), dL = L Phi(L^-1 Sdot L^-T) for the Gram/tangent pair selected by `mode`
int chol_tangent_common(Handle *h, int n, const double *x1, double alpha, const double *ls_host, int P, double dadd,
                        int mode, double *L, double *dLdl, int *info_out_host) {
  const int np = round_up(n, TILE), nt = np / TILE;
  const size_t mat = (size_t)np * np;
  const long long st = (long long)mat;
  Arena a;
  RC(ws_reserve(h, 4 * P * pad256(mat * 8) + pad256(n * 8) + (h->device_ptrs ? 0 : pad256((size_t)2 * P * n * n * 8)) + pad256(P * 8) + pad256(P * 4) + 2048, &a));
  double *Lbuf = a.take<double>(mat * P), *Sbuf = a.take<double>(mat * P), *Dbuf = a.take<double>(mat * P),
         *Lkeep = a.take<double>(mat * P);
  double *dx = a.take<double>(n), *dls = a.take<double>(P);
  int *info = a.take<int>(P);
  double *stage = h->device_ptrs ? nullptr : a.take<double>((size_t)2 * P * n * n);
  if (!info || (!h->device_ptrs && !stage)) BAD_ARG(h, 1002, "chol_tangent: workspace exhausted");
  GPB_CUDA(h, cudaMemsetAsync(info, 0, sizeof(int) * P, h->stream));
  RC(to_device(h, x1, dx, n));
  GPB_CUDA(h, cudaMemcpyAsync(dls, ls_host, sizeof(double) * P, cudaMemcpyHostToDevice, h->stream));
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));  // ls_host may be a stack temporary
  RC(launch_gram_tangent(h, n, np, dx, alpha, dls, dadd, mode, Lbuf, Dbuf, st, P));
  RC(chol_batched(h, Lbuf, np, st, n, P, info));
  GPB_CUDA(h, cudaMemcpyAsync(info_out_host, info, sizeof(int) * P, cudaMemcpyDeviceToHost, h->stream));
  GPB_CUDA(h, cudaMemcpyAsync(Lkeep, Lbuf, mat * P * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  RC(trtri_batched(h, Lbuf, Sbuf, np, st, P));
  TaskList t1, ta, tl;
  RC(tasks_tangent(h, nt, &t1, &ta, &tl));
  {  // T1 = W Kdot  -> Sbuf (lower tiles)
    GemmParams p{};
    p.A = mref(Lbuf, np, st); p.B = mref(Dbuf, np, st); p.C = mref(Sbuf, np, st); p.alpha = 1.0; p.tasks = t1.at(0);
    RC(launch_gemm(h, LAYOUT_NN, EPI_AXPBY, p, t1.count(0), P));
  }
  {  // A = T1 W^T -> Dbuf (lower tiles)
    GemmParams p{};
    p.A = mref(Sbuf, np, st); p.B = mref(Lbuf, np, st); p.C = mref(Dbuf, np, st); p.alpha = 1.0; p.tasks = ta.at(0);
    RC(launch_gemm(h, LAYOUT_NT, EPI_AXPBY, p, ta.count(0), P));
  }
  RC(launch_phi_lower(h, np, Dbuf, st, P));
  {  // Ldot = L Phi(A) -> Sbuf (lower tiles)
    GemmParams p{};
    p.A = mref(Lkeep, np, st); p.B = mref(Dbuf, np, st); p.C = mref(Sbuf, np, st); p.alpha = 1.0; p.tasks = tl.at(0);
    RC(launch_gemm(h, LAYOUT_NN, EPI_AXPBY, p, tl.count(0), P));
  }
  const size_t nn = (size_t)n * n;
  for (int q = 0; q < P; q++) {
    if (h->device_ptrs) {
      RC(launch_unpack(h, n, n, Lkeep + q * mat, np, L + q * nn, n, 1, 0.0));
      RC(launch_unpack(h, n, n, Sbuf + q * mat, np, dLdl + q * nn, n, 1, 0.0));
    } else {
      // both matrices of a table are unpacked into one staging area and leave in back-to-back asynchronous copies;
      // the only synchronisation is the one at the end (round 1 did unpack -> copy -> sync per matrix)
      double *sl = stage + (size_t)q * 2 * nn, *sd = sl + nn;
      RC(launch_unpack(h, n, n, Lkeep + q * mat, np, sl, n, 1, 0.0));
      RC(launch_unpack(h, n, n, Sbuf + q * mat, np, sd, n, 1, 0.0));
      RC(from_device(h, sl, L + q * nn, nn * sizeof(double)));
      RC(from_device(h, sd, dLdl + q * nn, nn * sizeof(double)));
    }
  }
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));  // info_out_host is valid from here
  return 0;
}
}  // namespace

extern "C" int gpb200_rbf_cov_chol(gpb200_handle_t h, int n, const double *x1, double l, double *L, double *dLdl) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "rbf_cov_chol: negative n");
  if (n == 0) return 0;
  int info = 0;
  RC(chol_tangent_common(h, n, x1, 1.0, &l, 1, 1e-10, 0, L, dLdl, &info));
  return info;
}

// P length-scales in one call: the tables Ls[P], dLdls[P] that approx_L / approx_Lz interpolate
// (models/interpolated_gp.stan:15-21 builds them with P separate Choleskys; test_interpolate.R:9 uses
// P = 10).  ls and info are HOST arrays of length P; L, dLdl hold P consecutive n x n matrices.
extern "C" int gpb200_rbf_cov_chol_batched(gpb200_handle_t h, int n, const double *x1, int P, const double *ls,
                                           double *L, double *dLdl, int *info) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "rbf_cov_chol_batched: negative n");
  if (P < 0) BAD_ARG(h, 4, "rbf_cov_chol_batched: negative P");
  if (n == 0 || P == 0) return 0;
  if (P > 65535 || n > MAX_DENSE_N) BAD_ARG(h, 4, "rbf_cov_chol_batched: at most 65535 tables of n <= 65407");
  return chol_tangent_common(h, n, x1, 1.0, ls, P, 1e-10, 0, L, dLdl, info);
}

extern "C" int gpb200_se_chol_tangent(gpb200_handle_t h, int n, const double *x, double alpha, double rho,
                                      double diag_add, int wrt, double *L, double *dL) {
  CHECK_H(h);
  if (n < 0) BAD_ARG(h, 2, "se_chol_tangent: negative n");
  if (wrt != 0 && wrt != 1) BAD_ARG(h, 7, "se_chol_tangent: wrt must be 0 (alpha) or 1 (rho)");
  if (n == 0) return 0;
  int info = 0;
  RC(chol_tangent_common(h, n, x, alpha, &rho, 1, diag_add, wrt == 1 ? 1 : 2, L, dL, &info));
  return info;
}

namespace {
int bracket(double l, int P, const double *lp) {  // covariance.cpp:56-61
  int lidx = 0;
  for (; lidx < P - 1; lidx++)
    if (lp[lidx + 1] >= l) break;
  if (lidx > P - 2) lidx = P - 2;
  return lidx;
}
}  // namespace

extern "C" int gpb200_approx_Lz(gpb200_handle_t h, int n, double l, int P, const double *lp, const double *const *Ls,
                                const double *const *dLdls, const double *z, double *vz, double *dvdl_z) {
  CHECK_H(h);
  if (n < 1) BAD_ARG(h, 2, "approx_L: n must be >= 1");
  if (P < 2) BAD_ARG(h, 4, "approx_L: need at least two grid points");
  // lp and the pointer tables are always host arrays; the tables they point to follow the pointer mode
  const int lidx = bracket(l, P, lp);
  const size_t nn = (size_t)n * n;
  Arena a;
  const int nchunk = hermite_matvec_chunks(n);
  RC(ws_reserve(h, (h->device_ptrs ? 0 : 4) * pad256(nn * 8) + (z ? 0 : 1) * pad256(nn * 8) + pad256((size_t)nchunk * n * 16) +
                       4 * pad256((size_t)n * 8) + 1024, &a));
  const double *t[4] = {Ls[lidx], Ls[lidx + 1], dLdls[lidx], dLdls[lidx + 1]};
  const double *d[4];
  for (int q = 0; q < 4; q++) {
    if (h->device_ptrs) d[q] = t[q];
    else {
      double *s = a.take<double>(nn);
      if (!s) BAD_ARG(h, 1002, "approx_L: workspace exhausted");
      RC(to_device(h, t[q], s, nn));
      d[q] = s;
    }
  }
  if (!z) {  // approx_L proper: return the interpolated factor in vz
    double *v = a.take<double>(nn);
    if (!v) BAD_ARG(h, 1002, "approx_L: workspace exhausted");
    RC(launch_hermite(h, (long long)nn, n, d[0], d[1], d[2], d[3], lp[lidx], lp[lidx + 1], l, v, nullptr));
    RC(from_device(h, v, vz, nn * sizeof(double)));
    return finish(h);
  }
  // approx_Lz: one fused pass over the four tables, the interpolated factor is never materialised
  double *part = a.take<double>((size_t)nchunk * n * 2);
  double *dz = a.take<double>(n), *o1 = a.take<double>(n), *o2 = a.take<double>(n);
  if (!o2) BAD_ARG(h, 1002, "approx_Lz: workspace exhausted");
  RC(to_device(h, z, dz, n));
  RC(launch_hermite_matvec(h, n, d[0], d[1], d[2], d[3], lp[lidx], lp[lidx + 1], l, dz, part, o1, dvdl_z ? o2 : nullptr));
  RC(from_device(h, o1, vz, n * sizeof(double)));
  if (dvdl_z) RC(from_device(h, o2, dvdl_z, n * sizeof(double)));
  return finish(h);
}

extern "C" int gpb200_approx_L(gpb200_handle_t h, int n, double l, int P, const double *lp, const double *const *Ls,
                               const double *const *dLdls, double *out) {
  return gpb200_approx_Lz(h, n, l, P, lp, Ls, dLdls, nullptr, out, nullptr);
}

// =================================================================================================
// a10 conditioning
// =================================================================================================
namespace {
int tasks_cond(Handle *h, int nt, int mt, TaskList *tv, TaskList *tc) {
  const long long k1 = tkey(TK_COND_V, nt, mt), k2 = tkey(TK_COND_COV, nt, mt);
  if (cached(h, k1, tv) && cached(h, k2, tc)) return 0;
  std::vector<TileTask> v1, v2;
  for (int i = 0; i < nt; i++)
    for (int j = 0; j < mt; j++)  // V[i,j] = sum_{k<=i} W[i,k] Ks[j,k]   (NT), V is np x mp
      v1.push_back({i * TILE, 0, j * TILE, 0, i * TILE, j * TILE, (i + 1) * TILE, 0});
  for (int i = 0; i < mt; i++)
    for (int j = 0; j <= i; j++)  // C[i,j] = Kss[i,j] - sum_k V[k,i] V[k,j]   (TN), lower tiles
      v2.push_back({0, i * TILE, 0, j * TILE, i * TILE, j * TILE, nt * TILE, 0});
  sort_desc(v1, 0);
  std::vector<int> o1 = {0, (int)v1.size()}, o2 = {0, (int)v2.size()};
  RC(upload_tasks(h, k1, v1, o1, tv));
  return upload_tasks(h, k2, v2, o2, tc);
}

// all pointers here are DEVICE pointers; K (n x n, ldk), Ks (m x n), Kss (m x m); rhs length n;
// mean_add (length m) may be null.
int condition_device(Handle *h, Arena &a, int n, int m, const double *K, long long ldk, const double *Ks,
                     long long ldks, const double *Kss, long long ldkss, const double *rhs, const double *mean_add,
                     double noise_var, double jitter, double *mu, double *cov, long long ldcov, int *hinfo) {
  const int np = round_up(n, TILE), mp = round_up(m, TILE);
  const size_t mat = (size_t)np * np;
  double *Lbuf = a.take<double>(mat), *Sbuf = a.take<double>(mat);
  double *Ksp = a.take<double>((size_t)mp * np), *V = a.take<double>((size_t)np * mp), *Cp = a.take<double>((size_t)mp * mp);
  double *z = a.take<double>(np);
  int *info = a.take<int>(1);
  if (!info) BAD_ARG(h, 1002, "gp_condition: workspace exhausted");
  GPB_CUDA(h, cudaMemsetAsync(info, 0, sizeof(int), h->stream));
  RC(launch_pack(h, n, n, K, ldk, np, np, Lbuf, 1, noise_var));
  RC(launch_pack(h, m, n, Ks, ldks, mp, np, Ksp, 0, 0.0));
  RC(launch_pack(h, m, m, Kss, ldkss, mp, mp, Cp, 0, 0.0));
  RC(chol_batched(h, Lbuf, np, (long long)mat, n, 1, info));
  RC(read_info(h, info, hinfo));
  RC(trtri_batched(h, Lbuf, Sbuf, np, (long long)mat, 1));
  RC(launch_trmv_lower_n(h, np, Lbuf, 0, rhs, 0, n, z, 0, 1));
  TaskList tv, tc;
  RC(tasks_cond(h, np / TILE, mp / TILE, &tv, &tc));
  {
    GemmParams p{};
    p.A = mref(Lbuf, np, 0); p.B = mref(Ksp, mp, 0); p.C = mref(V, np, 0); p.alpha = 1.0; p.tasks = tv.at(0);
    RC(launch_gemm(h, LAYOUT_NT, EPI_AXPBY, p, tv.count(0), 1));
  }
  {
    GemmParams p{};
    p.A = mref(V, np, 0); p.B = mref(V, np, 0); p.C = mref(Cp, mp, 0); p.C0 = mref(Cp, mp, 0);
    p.alpha = -1.0; p.beta = 1.0; p.tasks = tc.at(0);
    RC(launch_gemm(h, LAYOUT_TN, EPI_AXPBY, p, tc.count(0), 1));
  }
  RC(launch_gemv_t(h, np, m, V, np, z, mean_add, mu));
  RC(launch_unpack(h, m, m, Cp, mp, cov, ldcov, 2, jitter));
  return 0;
}

size_t cond_ws(int n, int m) {
  const size_t np = round_up(n, TILE), mp = round_up(m, TILE);
  return 2 * pad256(np * np * 8) + 2 * pad256(np * mp * 8) + pad256(mp * mp * 8) + pad256(np * 8) + 1024;
}
}  // namespace

extern "C" int gpb200_gp_condition(gpb200_handle_t h, int n, int m, const double *K, int ldk, const double *Ks,
                                   int ldks, const double *Kss, int ldkss, const double *y, double noise_var,
                                   double jitter, double *mu, double *cov, int ldcov) {
  CHECK_H(h);
  if (n < 1 || m < 1) BAD_ARG(h, 2, "gp_condition: sizes must be >= 1");
  if (n > MAX_DENSE_N || m > MAX_DENSE_N) BAD_ARG(h, 2, "gp_condition: sizes above 65407 are not supported");
  if (ldk < n || ldks < m || ldkss < m || ldcov < m) BAD_ARG(h, 5, "gp_condition: bad leading dimension");
  Arena a;
  const size_t stage = h->device_ptrs ? 0 : pad256((size_t)n * n * 8) + pad256((size_t)m * n * 8) + 2 * pad256((size_t)m * m * 8) + pad256(n * 8) + pad256(m * 8);
  RC(ws_reserve(h, cond_ws(n, m) + stage + 1024, &a));
  int hinfo = 0;
  if (h->device_ptrs) {
    RC(condition_device(h, a, n, m, K, ldk, Ks, ldks, Kss, ldkss, y, nullptr, noise_var, jitter, mu, cov, ldcov, &hinfo));
    return hinfo;
  }
  double *dK = a.take<double>((size_t)n * n), *dKs = a.take<double>((size_t)m * n), *dKss = a.take<double>((size_t)m * m);
  double *dcov = a.take<double>((size_t)m * m), *dy = a.take<double>(n), *dmu = a.take<double>(m);
  RC(to_device_2d(h, K, ldk, dK, n, n, n));
  RC(to_device_2d(h, Ks, ldks, dKs, m, m, n));
  RC(to_device_2d(h, Kss, ldkss, dKss, m, m, m));
  RC(to_device(h, y, dy, n));
  RC(condition_device(h, a, n, m, dK, n, dKs, m, dKss, m, dy, nullptr, noise_var, jitter, dmu, dcov, m, &hinfo));
  RC(from_device(h, dmu, mu, m * sizeof(double)));
  RC(from_device_2d(h, dcov, m, cov, ldcov, m, m));
  RC(finish(h));
  return hinfo;
}

namespace {
__global__ void sub_kernel(int n, const double *a, const double *b, double *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] - (b ? b[i] : 0.0);
}
}  // namespace

extern "C" int gpb200_cond_mvn(gpb200_handle_t h, int ng, int nd, const double *mean, const double *sigma, int lds,
                               const double *x_given, double *cond_mean, double *cond_var, int ldv) {
  CHECK_H(h);
  if (ng < 1 || nd < 1) BAD_ARG(h, 2, "cond_mvn: sizes must be >= 1");
  if (ng > MAX_DENSE_N || nd > MAX_DENSE_N) BAD_ARG(h, 2, "cond_mvn: sizes above 65407 are not supported");
  const int N = ng + nd;
  if (lds < N || ldv < nd) BAD_ARG(h, 6, "cond_mvn: bad leading dimension");
  Arena a;
  const size_t stage = h->device_ptrs ? pad256(ng * 8) : pad256((size_t)N * N * 8) + 3 * pad256(N * 8) + pad256((size_t)nd * nd * 8) + pad256(nd * 8);
  RC(ws_reserve(h, cond_ws(ng, nd) + stage + 1024, &a));
  const double *dS = sigma, *dmean = mean, *dxg = x_given;
  long long ld = lds;
  double *dcm = cond_mean, *dcv = cond_var;
  long long ldo = ldv;
  if (!h->device_ptrs) {
    double *s = a.take<double>((size_t)N * N), *mm = a.take<double>(N), *xg = a.take<double>(ng);
    RC(to_device_2d(h, sigma, lds, s, N, N, N));
    if (mean) RC(to_device(h, mean, mm, N));
    RC(to_device(h, x_given, xg, ng));
    dS = s; dmean = mean ? mm : nullptr; dxg = xg; ld = N;
    dcm = a.take<double>(nd); dcv = a.take<double>((size_t)nd * nd); ldo = nd;
  }
  double *rhs = a.take<double>(ng);
  ProfScope ps__(h, PC_OTHER);
  sub_kernel<<<(ng + 255) / 256, 256, 0, h->stream>>>(ng, dxg, dmean, rhs);
  GPB_LAUNCH_CHECK(h);
  int hinfo = 0;
  // given block first: D = S[0:ng,0:ng], C = S[ng:,0:ng] (nd x ng), B = S[ng:,ng:]
  RC(condition_device(h, a, ng, nd, dS, ld, dS + ng, ld, dS + ng + (long long)ng * ld, ld, rhs,
                      dmean ? dmean + ng : nullptr, 0.0, 0.0, dcm, dcv, ldo, &hinfo));
  if (!h->device_ptrs) {
    RC(from_device(h, dcm, cond_mean, nd * sizeof(double)));
    RC(from_device_2d(h, dcv, nd, cond_var, ldv, nd, nd));
  }
  RC(finish(h));
  return hinfo;
}
