// Host-side engines of libgpb200: workspace arena, tile task lists and the tiled algorithms built
// from the DMMA GEMM and the panel kernels (left-looking batched Cholesky with an optional
// right-looking panel split, in-place recursive triangular inverse).  No C-ABI entry points here.
#include "host.cuh"

namespace gpb {

// ---------------------------------------------------------------------------------------------
// workspace arena
// ---------------------------------------------------------------------------------------------


int ws_reserve(Handle *h, size_t bytes, Arena *a) {
  if (bytes > h->ws_bytes) {
    if (h->ws) {
      GPB_CUDA(h, cudaStreamSynchronize(h->stream));
      if (h->gstream) GPB_CUDA(h, cudaStreamSynchronize(h->gstream));
      for (auto &kv : h->graphs) cudaGraphExecDestroy(kv.second.exec);  // they bake in workspace addresses
      h->graphs.clear();
      GPB_CUDA(h, cudaFree(h->ws));
      h->ws = nullptr;
      h->ws_bytes = 0;
    }
    cudaError_t e = cudaMalloc(&h->ws, bytes);
    if (e != cudaSuccess) {
      snprintf(h->err, sizeof(h->err), "workspace allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
      (void)cudaGetLastError();
      return -1002;
    }
    h->ws_bytes = bytes;
  }
  a->base = reinterpret_cast<char *>(h->ws);
  a->cap = h->ws_bytes;
  a->off = 0;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// task lists (host-built once per tile count, cached on the device)
// ---------------------------------------------------------------------------------------------


int upload_tasks(Handle *h, long long key, const std::vector<TileTask> &tasks, const std::vector<int> &offsets,
                 TaskList *out) {
  auto it = h->task_cache.find(key);
  if (it == h->task_cache.end()) {
    TileTask *dev = nullptr;
    const size_t bytes = std::max<size_t>(tasks.size(), 1) * sizeof(TileTask);
    GPB_CUDA(h, cudaMalloc(&dev, bytes));
    if (!tasks.empty())
      GPB_CUDA(h, cudaMemcpyAsync(dev, tasks.data(), tasks.size() * sizeof(TileTask), cudaMemcpyHostToDevice, h->stream));
    GPB_CUDA(h, cudaStreamSynchronize(h->stream));
    it = h->task_cache.emplace(key, std::make_pair(dev, offsets)).first;
    h->task_host[key] = tasks;
  }
  out->dev = it->second.first;
  out->offsets = &it->second.second;
  return 0;
}

bool cached(Handle *h, long long key, TaskList *out) {
  auto it = h->task_cache.find(key);
  if (it == h->task_cache.end()) return false;
  out->dev = it->second.first;
  out->offsets = &it->second.second;
  return true;
}


void sort_desc(std::vector<TileTask> &v, size_t from) {
  std::stable_sort(v.begin() + from, v.end(), [](const TileTask &x, const TileTask &y) { return x.k_len > y.k_len; });
}

// Cholesky task lists.  Panels of `pt` tile columns: inside a panel the factorisation is
// left-looking (step j updates block column j with the panel's columns to its left, K = (j-p0)*128);
// after a panel is complete one right-looking launch applies it to everything to its right
// (K = pt*128).  pt = nt is the pure left-looking algorithm used for large batches; a narrow panel
// gives a single large matrix enough tiles per launch to fill 148 SMs.
int tasks_chol(Handle *h, int nt, int pt, TaskList *upd, TaskList *trail) {
  const long long k1 = tkey(TK_CHOL, nt, pt), k2 = tkey(TK_CHOL_TRAIL, nt, pt);
  if (cached(h, k1, upd) && cached(h, k2, trail)) return 0;
  std::vector<TileTask> t, tt;
  std::vector<int> off(1, 0), offt(1, 0);
  for (int j = 0; j < nt; j++) {
    const int p0 = (j / pt) * pt;
    if (j > p0)
      for (int i = j; i < nt; i++)
        t.push_back({i * TILE, p0 * TILE, j * TILE, p0 * TILE, i * TILE, j * TILE, (j - p0) * TILE, i == j});
    off.push_back((int)t.size());
  }
  for (int p0 = 0; p0 < nt; p0 += pt) {
    const int p1 = std::min(nt, p0 + pt);
    for (int jj = p1; jj < nt; jj++)
      for (int i = jj; i < nt; i++)
        tt.push_back({i * TILE, p0 * TILE, jj * TILE, p0 * TILE, i * TILE, jj * TILE, (p1 - p0) * TILE, i == jj});
    offt.push_back((int)tt.size());
  }
  int rc = upload_tasks(h, k1, t, off, upd);
  if (rc) return rc;
  return upload_tasks(h, k2, tt, offt, trail);
}

struct Node { int lo, mid, hi, level; };
int build_nodes(int lo, int hi, std::vector<Node> &nodes) {
  if (hi - lo <= 1) return 0;
  const int mid = lo + (hi - lo + 1) / 2;
  const int l1 = build_nodes(lo, mid, nodes), l2 = build_nodes(mid, hi, nodes);
  const int lvl = std::max(l1, l2) + 1;
  nodes.push_back({lo, mid, hi, lvl});
  return lvl;
}

// in-place recursive inverse of the lower-triangular factor: per node (lo, mid, hi)
//   S^T = L21^T * W22^T      (scratch buffer, UPPER tiles)   S^T[j,i] = sum_{k=mid..i} L[k,j] W[i,k]
//   W21 = -S * W11           (over L21 in place)             W[i,j]  = -sum_{k=j..mid-1} S^T[k,i] W[k,j]
// S is kept transposed so that in BOTH products the triangular diagonal tile (W22[i,i], W11[j,j]) is the
// B operand of the tile GEMM, whose zero half the column-split configurations skip for a whole CTA.
int tasks_trtri(Handle *h, int nt, TaskList *s_out, TaskList *w_out) {
  const long long ks = tkey(TK_TRTRI_S, nt), kw = tkey(TK_TRTRI_W, nt);
  if (cached(h, ks, s_out) && cached(h, kw, w_out)) return 0;
  std::vector<Node> nodes;
  const int top = build_nodes(0, nt, nodes);
  std::vector<TileTask> ts, tw;
  std::vector<int> os(1, 0), ow(1, 0);
  for (int lvl = 1; lvl <= top; lvl++) {
    const size_t fs = ts.size(), fw = tw.size();
    for (const Node &nd : nodes) {
      if (nd.level != lvl) continue;
      for (int i = nd.mid; i < nd.hi; i++)
        for (int j = nd.lo; j < nd.mid; j++) {
          // LAYOUT_TT: A = L (k down the rows from mid, columns of tile j), B = W (rows of tile i, k along the columns)
          ts.push_back({nd.mid * TILE, j * TILE, i * TILE, nd.mid * TILE, j * TILE, i * TILE, (i - nd.mid + 1) * TILE, TF_B_TRI_LAST});
          // LAYOUT_TN: A = S^T (k down the rows from tile j, columns of tile i), B = W11 (k down the rows, columns of tile j)
          tw.push_back({j * TILE, i * TILE, j * TILE, j * TILE, i * TILE, j * TILE, (nd.mid - j) * TILE, TF_B_TRI_FIRST});
        }
    }
    sort_desc(ts, fs);
    sort_desc(tw, fw);
    os.push_back((int)ts.size());
    ow.push_back((int)tw.size());
  }
  int rc = upload_tasks(h, ks, ts, os, s_out);
  if (rc) return rc;
  return upload_tasks(h, kw, tw, ow, w_out);
}

// G = W^T W, one tile per unordered pair: G[j,i] = sum_{k>=i} W[k,j]^T W[k,i] for j <= i, i.e. the UPPER
// tiles (the transposes of the lower ones; the only consumer is the symmetric trace epilogue, nothing
// is stored).  Written this way the triangular operand tile W[i,i] is the B operand, whose zero half
// the column-split GEMM configurations skip for a whole CTA.
int tasks_lauum(Handle *h, int nt, TaskList *out) {
  const long long key = tkey(TK_LAUUM, nt);
  if (cached(h, key, out)) return 0;
  std::vector<TileTask> t;
  for (int i = 0; i < nt; i++)
    for (int j = 0; j <= i; j++)
      t.push_back({i * TILE, j * TILE, i * TILE, i * TILE, j * TILE, i * TILE, (nt - i) * TILE,
                   TF_B_TRI_FIRST | (i == j ? (TF_DIAG | TF_A_TRI_FIRST) : 0)});
  sort_desc(t, 0);
  std::vector<int> off = {0, (int)t.size()};
  return upload_tasks(h, key, t, off, out);
}

// ---------------------------------------------------------------------------------------------
// engines on padded device buffers
// ---------------------------------------------------------------------------------------------

static void set_env(GemmParams &p, const int *env, const int *order, int nt, int mode) {
  p.env = env;
  p.order = env ? order : nullptr;
  p.env_nt = nt;
  p.env_mode = env ? mode : ENV_NONE;
}

// Batched tiled Cholesky, in place on Lbuf (np x np per item, lower tiles valid on entry).  With an envelope (env, see
// ENV_CHOL_FINE) every update CTA starts its contraction at the first 16-column chunk where a row of both its operands
// can be nonzero and exits when nothing is left: L is bit-identical to the dense factorisation.  The look-ahead
// schedule keeps the tile rule (ENV_CHOL): its launches are bound by the panel chain, not by their flops.
// Panel width: pure left-looking when the batch alone fills the GPU, 8-tile (1024-column) panels
// with right-looking trailing updates otherwise.
int chol_panel_tiles(int nt, int batch) {
  if (batch >= 64 || nt <= 8) return nt;
  return 8;
}

// Trailing-update task lists of the look-ahead schedule: after panel [p0, p1) is factored, list 1 updates the block
// columns of the NEXT panel (the panel chain waits for it), list 2 everything to the right of that.
static int tasks_chol_lookahead(Handle *h, int nt, int pt, TaskList *la1, TaskList *la2) {
  const long long k1 = tkey(TK_CHOL_LA1, nt, pt), k2 = tkey(TK_CHOL_LA2, nt, pt);
  if (cached(h, k1, la1) && cached(h, k2, la2)) return 0;
  std::vector<TileTask> t1, t2;
  std::vector<int> o1(1, 0), o2(1, 0);
  for (int p0 = 0; p0 < nt; p0 += pt) {
    const int p1 = std::min(nt, p0 + pt), p2 = std::min(nt, p1 + pt);
    for (int jj = p1; jj < nt; jj++)
      for (int i = jj; i < nt; i++)
        (jj < p2 ? t1 : t2).push_back({i * TILE, p0 * TILE, jj * TILE, p0 * TILE, i * TILE, jj * TILE, (p1 - p0) * TILE, i == jj});
    o1.push_back((int)t1.size());
    o2.push_back((int)t2.size());
  }
  int rc = upload_tasks(h, k1, t1, o1, la1);
  if (rc) return rc;
  return upload_tasks(h, k2, t2, o2, la2);
}

bool chol_uses_lookahead(const Handle *h, int nt, int batch) {
  // few tiles in flight: the panel chain, not the DMMA work, bounds the factorisation (with more items the pure
  // left-looking schedule already fills the GPU and its deep-K updates are the more efficient GEMMs)
  return h->lookahead && h->pstream && batch <= h->lookahead_max_batch && (long long)batch * nt <= 256 && nt >= 3;
}
// panel width of the look-ahead schedule in tiles: one tile column per chain step for small matrices (the chain is all
// there is); wider panels halve the number of bulk launches and double their K as the matrix grows.  Measured, B = 1,
// LML + gradient: N = 2048 0.94 ms with 1 / 0.97 with 2; N = 4096 3.39 / 3.34 / 3.45 ms with 1 / 2 / 4; N = 8192 19.5 /
// 19.2 / 19.8 ms with 2 / 4 / 8; N = 16 384 135.1 / 132.1 / 132.5; N = 32 768 1040 / 1018 / 1008.
int chol_lookahead_panel(const Handle *h, int nt) {
  if (h->chol_panel_override > 0) return std::min(nt, h->chol_panel_override);
  return nt >= 192 ? 8 : (nt >= 48 ? 4 : (nt >= 24 ? 2 : 1));
}

// Look-ahead schedule (small batches; one matrix does not fill the GPU and the panel chain of one POTRF tile and
// one TRSM wave per block column is what bounds the factorisation):
//   side stream P :  [in-panel left-looking update] -> POTRF -> TRSM per block column, then the update of the NEXT
//                    panel's columns by this panel (list 1) -- the whole dependent chain is consecutive launches of
//                    ONE high-priority stream
//   main stream T :  wait(panel p factored) -> update of everything right of the next panel (list 2)
// so panel p+1 is factored while the bulk of panel p's trailing update still runs.  Every write to a block column
// is ordered: before P updates the next panel's columns it waits for T's previous trailing update, which was the
// last launch to write them; T's updates follow one another in stream order.
static int chol_lookahead(Handle *h, double *Lbuf, int np, long long stride, int n, int batch, int *info_dev, const int *env) {
  const int nt = np / TILE, pt = chol_lookahead_panel(h, nt);
  TaskList tl, tr, la1, la2;
  int rc = tasks_chol(h, nt, pt, &tl, &tr);
  if (rc) return rc;
  rc = tasks_chol_lookahead(h, nt, pt, &la1, &la2);
  if (rc) return rc;
  GemmParams p{};
  p.A = mref(Lbuf, np, stride);
  p.B = mref(Lbuf, np, stride);
  p.C = mref(Lbuf, np, stride);
  p.C0 = mref(Lbuf, np, stride);
  p.alpha = -1.0;
  p.beta = 1.0;
  set_env(p, env, nullptr, nt, ENV_CHOL);
  GemmParams pc = p;      // launches on the panel chain
  pc.latency_hint = 1;
  cudaStream_t T = h->stream, P = h->pstream;
  struct Restore { Handle *h; cudaStream_t s; ~Restore() { h->stream = s; } } restore{h, T};
  size_t ev = 0;
  GPB_CUDA(h, cudaEventRecord(h->sync_event(ev), T));
  GPB_CUDA(h, cudaStreamWaitEvent(P, h->sync_event(ev), 0));
  ev++;
  cudaEvent_t ev_trail = nullptr;  // T's most recent trailing update
  int panel = 0;
  for (int p0 = 0; p0 < nt; p0 += pt, panel++) {
    const int p1 = std::min(nt, p0 + pt);
    h->stream = P;
    for (int j = p0; j < p1; j++) {
      if (tl.count(j) > 0) {
        pc.tasks = tl.at(j);
        if ((rc = launch_gemm(h, LAYOUT_NT, EPI_AXPBY, pc, tl.count(j), batch))) return rc;
      }
      if ((rc = launch_potrf_trsm(h, Lbuf, np, stride, j, nt - 1 - j, n, batch, info_dev))) return rc;
    }
    cudaEvent_t ev_panel = h->sync_event(ev++);
    GPB_CUDA(h, cudaEventRecord(ev_panel, P));
    if (p1 < nt) {
      if (ev_trail) GPB_CUDA(h, cudaStreamWaitEvent(P, ev_trail, 0));
      pc.tasks = la1.at(panel);
      if ((rc = launch_gemm(h, LAYOUT_NT, EPI_AXPBY, pc, la1.count(panel), batch))) return rc;
    }
    h->stream = T;
    GPB_CUDA(h, cudaStreamWaitEvent(T, ev_panel, 0));
    if (p1 < nt && la2.count(panel) > 0) {
      p.tasks = la2.at(panel);
      if ((rc = launch_gemm(h, LAYOUT_NT, EPI_AXPBY, p, la2.count(panel), batch))) return rc;
      ev_trail = h->sync_event(ev++);
      GPB_CUDA(h, cudaEventRecord(ev_trail, T));
    }
  }
  return 0;  // T has waited for the last panel (which follows every launch on P): the side stream is joined
}

int chol_batched(Handle *h, double *Lbuf, int np, long long stride, int n, int batch, int *info_dev, const int *env,
                 const int *order) {
  const int nt = np / TILE;
  if (chol_uses_lookahead(h, nt, batch)) return chol_lookahead(h, Lbuf, np, stride, n, batch, info_dev, env);
  const int pt = h->chol_panel_override > 0 ? std::min(nt, h->chol_panel_override) : chol_panel_tiles(nt, batch);
  TaskList tl, tr;
  int rc = tasks_chol(h, nt, pt, &tl, &tr);
  if (rc) return rc;
  GemmParams p{};
  p.A = mref(Lbuf, np, stride);
  p.B = mref(Lbuf, np, stride);
  p.C = mref(Lbuf, np, stride);
  p.C0 = mref(Lbuf, np, stride);
  p.alpha = -1.0;
  p.beta = 1.0;
  set_env(p, env, order, nt, ENV_CHOL_FINE);
  for (int j = 0; j < nt; j++) {
    if (tl.count(j) > 0) {
      p.tasks = tl.at(j);
      rc = launch_gemm(h, LAYOUT_NT, EPI_AXPBY, p, tl.count(j), batch);
      if (rc) return rc;
    }
    rc = launch_potrf_trsm(h, Lbuf, np, stride, j, nt - 1 - j, n, batch, info_dev, env);
    if (rc) return rc;
    if ((j + 1) % pt == 0 && j + 1 < nt) {
      const int panel = j / pt;
      p.tasks = tr.at(panel);
      rc = launch_gemm(h, LAYOUT_NT, EPI_AXPBY, p, tr.count(panel), batch);
      if (rc) return rc;
    }
  }
  return 0;
}

// In-place inverse of the lower-triangular factor held in Lbuf; Sbuf is same-shaped scratch.
int trtri_batched(Handle *h, double *Lbuf, double *Sbuf, int np, long long stride, int batch) {
  const int nt = np / TILE;
  int rc = launch_tile_inverse(h, Lbuf, Lbuf, np, stride, nt, batch);
  if (rc) return rc;
  if (nt == 1) return 0;
  TaskList ts, tw;
  rc = tasks_trtri(h, nt, &ts, &tw);
  if (rc) return rc;
  const int chain = chol_uses_lookahead(h, nt, batch) ? 1 : 0;   // one or a few matrices: every launch is on the critical path
  for (int lvl = 0; lvl < ts.steps(); lvl++) {
    GemmParams p{};
    p.A = mref(Lbuf, np, stride);
    p.B = mref(Lbuf, np, stride);
    p.C = mref(Sbuf, np, stride);
    p.alpha = 1.0;
    p.beta = 0.0;
    p.latency_hint = chain;
    p.tasks = ts.at(lvl);
    rc = launch_gemm(h, LAYOUT_TT, EPI_AXPBY, p, ts.count(lvl), batch);
    if (rc) return rc;
    GemmParams q{};
    q.A = mref(Sbuf, np, stride);
    q.B = mref(Lbuf, np, stride);
    q.C = mref(Lbuf, np, stride);
    q.alpha = -1.0;
    q.beta = 0.0;
    q.latency_hint = chain;
    q.tasks = tw.at(lvl);
    rc = launch_gemm(h, LAYOUT_TN, EPI_AXPBY, q, tw.count(lvl), batch);
    if (rc) return rc;
  }
  return 0;
}

// Selected inverse (Takahashi recurrence) of a factor with a tile envelope: Z = K^-1 on the tiles (I, J) with
// J <= I <= E_J, which hold every tile where the SE covariance or its derivatives are nonzero.  With Y = L W
// (W_JJ = L_JJ^-1, the block column scaled by its diagonal inverse) and S = J+1..E_J:
//   Z[S,J] = -Z[S,S] Y[S,J],    Z[J,J] = W_JJ^T W_JJ - Y[S,J]^T Z[S,J]
// For K in S, E_K >= E_J, so every Z[S,S] tile the contraction reads was produced by an earlier step.  Rows of Y[S,J]
// past er_J are zero (ENV_BAND), so both contractions end there.
//   Y    all block columns in one launch (Sbuf, lower tiles)
//   D    W_JJ^T W_JJ over the diagonal tiles of Lbuf (full tiles)
//   per J from the last: Z[S,J] into Lbuf (lower tiles) and its transpose into the upper tiles, so that Z[S,S] is
//   read with one layout; then Z[J,J].
// On entry Lbuf holds L (lower tiles) and Sbuf W_JJ on its diagonal tiles; L is consumed.
static int tasks_sinv(Handle *h, int nt, TaskList *ty, TaskList *td, TaskList *tz, TaskList *tzd) {
  const long long k1 = tkey(TK_SINV_Y, nt), k2 = tkey(TK_SINV_D, nt), k3 = tkey(TK_SINV_Z, nt), k4 = tkey(TK_SINV_ZD, nt);
  if (cached(h, k1, ty) && cached(h, k2, td) && cached(h, k3, tz) && cached(h, k4, tzd)) return 0;
  std::vector<TileTask> y, d, z, zd;
  std::vector<int> oz(1, 0), ozd(1, 0);
  for (int j = 0; j < nt; j++) {
    // NN: Y[i,j] = L[i,j] W[j,j] (W lower: B zero where k < n)
    for (int i = j + 1; i < nt; i++) y.push_back({i * TILE, j * TILE, j * TILE, j * TILE, i * TILE, j * TILE, TILE, TF_B_TRI_FIRST});
    // TN: D[j,j] = W[j,j]^T W[j,j]
    d.push_back({j * TILE, j * TILE, j * TILE, j * TILE, j * TILE, j * TILE, TILE, TF_A_TRI_FIRST | TF_B_TRI_FIRST});
  }
  for (int j = 0; j < nt; j++) {  // step j of the lists: block column j
    const int k = (nt - 1 - j) * TILE;
    // NN: Z[i,j] = -sum_{k>j} Z[i,k] Y[k,j]
    for (int i = j + 1; i < nt; i++) z.push_back({i * TILE, (j + 1) * TILE, (j + 1) * TILE, j * TILE, i * TILE, j * TILE, k, 0});
    oz.push_back((int)z.size());
    // TN: Z[j,j] = D[j,j] - sum_{k>j} Y[k,j]^T Z[k,j]
    if (j + 1 < nt) zd.push_back({(j + 1) * TILE, j * TILE, (j + 1) * TILE, j * TILE, j * TILE, j * TILE, k, 0});
    ozd.push_back((int)zd.size());
  }
  std::vector<int> oy = {0, (int)y.size()}, od = {0, (int)d.size()};
  RC(upload_tasks(h, k1, y, oy, ty));
  RC(upload_tasks(h, k2, d, od, td));
  RC(upload_tasks(h, k3, z, oz, tz));
  return upload_tasks(h, k4, zd, ozd, tzd);
}

int sinv_batched(Handle *h, double *Lbuf, double *Sbuf, int np, long long stride, const int *env, const int *order, int batch) {
  const int nt = np / TILE;
  TaskList ty, td, tz, tzd;
  RC(tasks_sinv(h, nt, &ty, &td, &tz, &tzd));
  GemmParams p{};
  set_env(p, env, order, nt, ENV_BAND);
  p.alpha = 1.0;
  if (nt > 1) {
    p.A = mref(Lbuf, np, stride); p.B = mref(Sbuf, np, stride); p.C = mref(Sbuf, np, stride); p.tasks = ty.at(0);
    RC(launch_gemm(h, LAYOUT_NN, EPI_AXPBY, p, ty.count(0), batch));
  }
  GemmParams q{};
  q.A = mref(Sbuf, np, stride); q.B = mref(Sbuf, np, stride); q.C = mref(Lbuf, np, stride); q.alpha = 1.0; q.tasks = td.at(0);
  RC(launch_gemm(h, LAYOUT_TN, EPI_AXPBY, q, td.count(0), batch));
  for (int j = nt - 2; j >= 0; j--) {
    GemmParams pz = p;
    pz.alpha = -1.0;
    pz.A = mref(Lbuf, np, stride); pz.B = mref(Sbuf, np, stride); pz.C = mref(Lbuf, np, stride); pz.CT = mref(Lbuf, np, stride);
    pz.tasks = tz.at(j);
    RC(launch_gemm(h, LAYOUT_NN, EPI_AXPBY, pz, tz.count(j), batch));
    GemmParams pd = p;
    pd.alpha = -1.0;
    pd.beta = 1.0;
    pd.A = mref(Sbuf, np, stride); pd.B = mref(Lbuf, np, stride); pd.C = mref(Lbuf, np, stride); pd.C0 = mref(Lbuf, np, stride);
    pd.tasks = tzd.at(j);
    RC(launch_gemm(h, LAYOUT_TN, EPI_AXPBY, pd, tzd.count(j), batch));
  }
  return 0;
}

__global__ void extract_diag_kernel(int np, const double *__restrict__ L, long long stride, double *__restrict__ dvec) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < np) dvec[(long long)blockIdx.y * np + i] = L[(long long)blockIdx.y * stride + i + (long long)i * np];
}

int extract_diag(Handle *h, int np, const double *L, long long stride, double *dvec, int batch) {
  dim3 grid((np + 255) / 256, batch);
  ProfScope ps__(h, PC_OTHER);
  extract_diag_kernel<<<grid, 256, 0, h->stream>>>(np, L, stride, dvec);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// host<->device staging helpers -----------------------------------------------------------------
int to_device(Handle *h, const double *src, double *dev, size_t count) {
  GPB_CUDA(h, cudaMemcpyAsync(dev, src, count * sizeof(double), h->device_ptrs ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  return 0;
}
int from_device(Handle *h, const void *dev, void *dst, size_t bytes) {
  GPB_CUDA(h, cudaMemcpyAsync(dst, dev, bytes, h->device_ptrs ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
  return 0;
}
int to_device_2d(Handle *h, const double *src, long long lds, double *dev, long long ldd, int rows, int cols) {
  if (rows <= 0 || cols <= 0) return 0;
  GPB_CUDA(h, cudaMemcpy2DAsync(dev, ldd * sizeof(double), src, lds * sizeof(double), rows * sizeof(double), cols,
                               h->device_ptrs ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  return 0;
}
int from_device_2d(Handle *h, const double *dev, long long lds, double *dst, long long ldd, int rows, int cols) {
  if (rows <= 0 || cols <= 0) return 0;
  GPB_CUDA(h, cudaMemcpy2DAsync(dst, ldd * sizeof(double), dev, lds * sizeof(double), rows * sizeof(double), cols,
                               h->device_ptrs ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
  return 0;
}
int finish(Handle *h) {
  if (!h->device_ptrs) GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int read_info(Handle *h, const int *info_dev, int *out) {
  GPB_CUDA(h, cudaMemcpyAsync(out, info_dev, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  GPB_CUDA(h, cudaStreamSynchronize(h->stream));
  return 0;
}

}  // namespace gpb
