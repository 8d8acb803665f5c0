// Shared definitions for libgpb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <vector>

namespace gpb {

constexpr int PANEL_FUSED_MAX_BATCH = 148;  // matrices per panel_fused_kernel launch (flag slots in the handle)
constexpr int TILE = 128;  // tile edge of every tiled algorithm (internal matrices are padded to it)
constexpr int ENV_MAX_NT = 512;  // tile rows of a matrix with a tile envelope (the GEMM stages one part of it in shared memory)
// Envelope record of one item of the SE route, ints at these offsets (nt tile rows):
//   F  [0, nt)      first tile column of each tile row that holds a nonzero (F_I <= I)
//   E  [nt, 2nt)    per tile column J, the last tile row I with F_I <= J
//   fb [2nt, 4nt)   per 64-row block, the first column any of its rows has a nonzero in (the element profile)
//   er [4nt, 5nt)   per tile column J, the last row with a nonzero in column 128 J + 127 or left of it (E_J = er_J / 128)
// "Nonzero": exp(-d^2 / 2 rho^2) not exactly zero, NaN included, and every diagonal element.
constexpr int ENV_BLK = 64;  // rows per fb block: the smallest CTA extent of the tile GEMM
__host__ __device__ constexpr int env_record_ints(int nt) { return 5 * nt; }

inline int round_up(int n, int m) { return (n + m - 1) / m * m; }

// One tile task of the batched DMMA GEMM: C[c_r.., c_c..] = beta*C0 + alpha * sum_k A * B^T-like
// product over k_len elements of the contraction index.  Coordinates are element offsets inside
// the (padded) matrices; how k advances through A and B depends on the kernel's layout template.
struct TileTask {
  int a_r, a_c;  // start of the A operand (row, col) in its stored matrix
  int b_r, b_c;  // start of the B operand
  int c_r, c_c;  // output tile origin
  int k_len;     // contraction length (multiple of 16)
  int flags;     // TF_* bits
};
// task flags: bit0 = diagonal tile of a symmetric result (trace epilogue weight 1 instead of 2); the
// others mark a triangular operand tile at the first / last 128 of the k-range: a column-half CTA that
// only meets the zero half of a triangular B tile contracts over 64 fewer k (the A flags are descriptive)
enum { TF_DIAG = 1,
       TF_A_TRI_FIRST = 2,   // first k-tile of A is zero where k_local < m_local
       TF_A_TRI_LAST = 4,    // last  k-tile of A is zero where k_local > m_local
       TF_B_TRI_FIRST = 8,   // first k-tile of B is zero where k_local < n_local
       TF_B_TRI_LAST = 16,   // last  k-tile of B is zero where k_local > n_local
       TF_FULL_WEIGHT = 32 };// trace epilogue: the tile is NOT half of a symmetric pair (weight 1; reverse-mode adjoint)

// a task list cut in two for the diagonal-split launch: symmetric diagonal tiles (TF_DIAG) and everything else
struct SplitLists {
  TileTask *reg = nullptr, *diag = nullptr;
  int nreg = 0, ndiag = 0;
};

struct MatRef {
  double *p;
  long long ld;
  long long stride;  // batch stride in doubles
};

struct GemmParams {
  MatRef A, B, C, C0;  // C0.p == nullptr -> no addend
  double alpha, beta;
  const TileTask *tasks;
  // trace epilogue (EPI_TRACE)
  const double *x;  long long x_stride;      // inputs (per batch)
  const double *avec; long long a_stride;    // a = K^-1 y (padded length np)
  const double *theta;                       // B x 3 (alpha, rho, sigma)
  double *partial;                           // B x ntasks x 4
  int n;                                     // true matrix size (mask for the padding)
  int ntasks;
  // derivative-observation trace epilogue (EPI_TRACE_DERIV): the matrix is nblocks x nblocks blocks of
  // n_grid x n_grid; block b carries derivative order order0 + b; theta is B x theta_stride
  int n_grid, order0, theta_stride;
  int latency_hint;   // 1: this launch sits on a dependent chain (look-ahead Cholesky): small launches take the 16-warp fine tiles
  // envelope of a banded covariance (ENV_* below): the records of env_record_ints(env_nt) ints per item
  const int *env;
  int env_nt, env_mode;
  const int *order;             // envelope launches: item of blockIdx.y (envelope_order_kernel); nullptr: blockIdx.y itself
  MatRef CT;                    // EPI_AXPBY: when CT.p is set the transpose of the output tile is written there too
  unsigned long long *flops;    // when set: every CTA adds the flops it executes (after all skipping)
  int ard_d;                    // EPI_TRACE_ARD: input dimensions D (x is n x D column-major per item, theta_stride = D + 2)
  const int *nvec;              // EPI_TRACE_RAGGED: per-item sizes (the mask of item b is nvec[b] instead of n)
};
// envelope modes of the tile GEMM.  Only products with an exactly-zero operand are dropped, and the k order of the rest
// is kept, so a result is bit-identical to the dense launch (up to the sign of an all-zero tile).  The bounds move in
// 16-wide k-chunks (KC), so every DMMA that remains reads the same k as in the dense launch.
enum { ENV_NONE = 0,
       ENV_CHOL = 1,       // C(I,J) -= L(I,k) L(J,k)^T: exit when J < F_I (tile outside the profile), k starts at max(F_I, F_J)
       ENV_CHOL_FINE = 2,  // the same update, k starts at the first column where a row of this CTA's A and one of its B
                           // can both be nonzero (fb over the CTA's rows and over its columns, rounded down to 16)
       ENV_BAND = 3 };     // selected inverse: exit when I > E_J; row k of Y[S,J] = L[S,J] W_JJ is zero past er_J, so the
                           // contraction ends at er_J + 1 rounded up to 16

// Tile envelope of the batched TRSM below diagonal tile `col` (the throughput TRSM kernels of panel.cu): F points at the
// F entry of the first row tile of item 0, item stride `stride`.  Row tile r (counted from the first) is live when
// F[r] <= col.  Any other C tile is exactly zero -- the Gram wrote +0.0 there and no update touched it -- and so would
// its solution be, so it is left as it is.  F need not be monotone (unsorted inputs), so every tile is tested.
struct TrsmEnv {
  const int *F = nullptr;  // nullptr: every tile is live (dense route)
  int stride = 0, col = 0;
  __device__ bool live(int item, int r) const { return !F || F[(long long)item * stride + r] <= col; }
};

struct Handle {
  int device = 0;
  cudaStream_t stream = nullptr;
  int device_ptrs = 0;
  long long launches = 0;
  long long ws_limit = 0;
  int chol_panel_override = 0;
  int gemm_cfg_override = 0;  // 0 automatic, 1 one 128x128 CTA per SM, 2 two 128x64 half-tile CTAs per SM, 3 64x64 quarter-tile CTAs
  int quarter_below_waves = 2;  // automatic choice: quarter tiles while the half-tile grid is below this many waves of 2 x 148 CTAs
  int trsm_pipelined = 1;     // 0: one tile per CTA (the first TRSM tile kernel); env GPB200_TRSM_PIPELINED
  int fine_cfg = 1;           // 64x64 CTAs of sixteen 16x16 warps for small chain launches (env GPB200_FINE_CFG)
  int panel_fused = 1;        // POTRF tile and the TRSM below it in one launch when one wave holds both (panel_fused_kernel); env GPB200_PANEL_FUSED
  int *panel_flags = nullptr; // 2 ints per matrix for panel_fused_kernel (visible column blocks, finished TRSM CTAs), zero between launches
  char err[512] = {0};
  // grow-only device workspace
  void *ws = nullptr;
  size_t ws_bytes = 0;
  // cached device-side task lists keyed by (kind, nt)
  std::map<long long, std::pair<TileTask *, std::vector<int>>> task_cache;
  std::map<long long, std::vector<TileTask>> task_host;  // host copies (executed-flop accounting, gpb200_set_flop_counting)
  std::map<std::pair<const TileTask *, int>, SplitLists> split_cache;
  int diag_split = 1;           // large batches: symmetric diagonal tiles run as 64x64 quarter CTAs in their own launch (env GPB200_DIAG_SPLIT)
  int count_flops = 0;
  double executed_gemm_flops = 0.0;  // flops the DMMA GEMM launches actually executed (after CTA-level skipping)
  unsigned long long *flops_dev = nullptr;  // the same for launches whose skipping is decided on the device (envelope)
  int envelope = 1;             // SE path: envelope Cholesky and selected inverse (env GPB200_ENVELOPE=0: dense reference route)
  int sinv_min_batch = 0;       // 0: selected inverse for the gradient when B * nt >= 256 (api_gp.cu); > 0: from this batch size (env GPB200_SINV_MINB)
  // CUDA graphs of the launch sequence of small (launch-latency-bound) LML evaluations, keyed by the
  // problem signature; replayed on a handle-owned stream (the caller's stream may be the legacy
  // default stream, which cannot be captured).  Invalidated when the workspace moves.
  cudaStream_t gstream = nullptr;
  cudaEvent_t g_in = nullptr, g_out = nullptr;
  struct GraphEntry { cudaGraphExec_t exec; long long nodes; };
  std::map<std::vector<long long>, GraphEntry> graphs;
  int graphs_enabled = 1;
  long long graph_replays = 0;
  // look-ahead Cholesky for small batches: the panel chain (update of the next block column, POTRF, TRSM) runs on
  // a high-priority side stream while the rest of the trailing update runs on the handle's stream
  cudaStream_t pstream = nullptr;
  std::vector<cudaEvent_t> sync_events;
  // config 5: NCCL communicator owned by the handle (loaded at run time, api_mg.cu), its own stream and a ring of
  // events that order collectives against the compute stream
  void *nccl_comm = nullptr;
  int mg_rank = 0, mg_world = 1;
  cudaStream_t cstream = nullptr;
  std::vector<cudaEvent_t> mg_events;
  long long mg_tickets = 0;
  // factor kept between gpb200_latent_forward and gpb200_latent_backward (api_latent.cu)
  double *latent_L = nullptr;
  size_t latent_bytes = 0;
  double latent_key[4] = {0, 0, 0, 0};
  int latent_n = 0;
  unsigned long long latent_xhash = 0;
  // record of the last gpb200_latent_forward_batched, read by gpb200_latent_backward_batched (api_latent.cu): the B
  // padded factors, per-item info and device copies of x, theta and z (diag_add enters the backward sweep only
  // through L) in one grow-only allocation (not the workspace)
  void *latent_rec = nullptr;
  size_t latent_rec_bytes = 0;
  int latent_rec_valid = 0, latent_rec_n = 0, latent_rec_B = 0, latent_rec_nvec = 0;
  long long latent_rec_xs = 0;  // x stride in the record: 0 shared, n per item
  int *info_slot = nullptr;     // persistent device word for the single-evaluation entry point in device-pointer mode
  cudaEvent_t stream_switch = nullptr;
  int small_kernel = 1;         // one-CTA whole-evaluation kernel for n <= 128 (env GPB200_SMALL_KERNEL=0 disables)
  int lookahead = 1;            // env GPB200_LOOKAHEAD=0 disables
  int lookahead_max_batch = 64; // batches up to this size take the look-ahead schedule (measured: N = 1024 x 32 groups +7 %)
  cudaEvent_t sync_event(size_t i) {
    while (sync_events.size() <= i) {
      cudaEvent_t e;
      cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
      sync_events.push_back(e);
    }
    return sync_events[i];
  }
  // optional per-kernel-class timing with CUDA events on the handle's stream (bench.py roofline)
  int profiling = 0;
  struct ProfRec { int cls; cudaEvent_t e0, e1; };
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  cudaEvent_t prof_event() {
    if (ev_used == ev_pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ev_pool.push_back(e);
    }
    return ev_pool[ev_used++];
  }
};

enum ProfClass { PC_GEMM = 0, PC_POTRF = 1, PC_TRSM = 2, PC_GRAM = 3, PC_SOLVE = 4, PC_OTHER = 5, PC_COUNT = 6 };

// brackets one kernel launch with events when profiling is on
struct ProfScope {
  Handle *h;
  cudaEvent_t e0 = nullptr;
  int cls;
  ProfScope(Handle *h_, int cls_) : h(h_), cls(cls_) {
    if (h->profiling) {
      e0 = h->prof_event();
      cudaEventRecord(e0, h->stream);
    }
  }
  ~ProfScope() {
    if (h->profiling) {
      cudaEvent_t e1 = h->prof_event();
      cudaEventRecord(e1, h->stream);
      h->prof.push_back({cls, e0, e1});
    }
  }
};

#define GPB_CUDA(h, call)                                                                     \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess) {                                                                 \
      snprintf((h)->err, sizeof((h)->err), "%s failed: %s (%s:%d)", #call,                    \
               cudaGetErrorString(e__), __FILE__, __LINE__);                                  \
      return -1000;                                                                           \
    }                                                                                         \
  } while (0)

#define GPB_LAUNCH_CHECK(h)                                                                   \
  do {                                                                                        \
    (h)->launches++;                                                                          \
    cudaError_t e__ = cudaGetLastError();                                                     \
    if (e__ != cudaSuccess) {                                                                 \
      snprintf((h)->err, sizeof((h)->err), "kernel launch failed: %s (%s:%d)",                \
               cudaGetErrorString(e__), __FILE__, __LINE__);                                  \
      return -1001;                                                                           \
    }                                                                                         \
  } while (0)

// ---- launchers implemented in the .cu files --------------------------------------------------
enum GemmLayout { LAYOUT_NT = 0, LAYOUT_TN = 1, LAYOUT_NN = 2, LAYOUT_TT = 3 };  // TT: A k-contiguous, B n-contiguous
// EPI_TRACE_RAGGED: the EPI_TRACE epilogue with a per-item size (gpb200_lml_grad_ragged), its own instantiation so that
// the uniform one stays as it is
enum GemmEpi { EPI_AXPBY = 0, EPI_TRACE = 1, EPI_TRACE_DERIV = 2, EPI_TRACE_ARD = 3, EPI_TRACE_RAGGED = 4 };
constexpr int ARD_MAX_D = 8;  // input dimensions of the ARD covariance (gpb200_lml_grad_ard_batched)
// doubles per CTA partial record of a trace epilogue: (S_se, S_d2, tr G, 0); (S_k, S_dk, tr G per block, ...);
// (S_e, S_1 .. S_ARD_MAX_D, tr G)
__host__ __device__ constexpr int epi_partial_width(int epi) {
  return epi == EPI_TRACE_DERIV ? 8 : (epi == EPI_TRACE_ARD ? ARD_MAX_D + 2 : 4);
}

int launch_gemm(Handle *h, GemmLayout layout, GemmEpi epi, const GemmParams &p, int ntasks, int batch);
int gemm_smem_setup(Handle *h);
int gemm_nsplit(const Handle *h, int ntasks, int batch);
// trace-epilogue partial records per item: n1 in the first region (item stride n1), n2 in a second region that starts
// after all items' first-region records (the diagonal-split launch); n2 = 0 when the launch is not split
int gemm_partial_layout(Handle *h, const TileTask *tasks, int ntasks, int batch, int *n1, int *n2);

// panel kernels (panel.cu)
int launch_potrf_tile(Handle *h, double *L, long long ld, long long stride, int tile_idx, int n,
                      int batch, int *info);
int launch_trsm_tiles(Handle *h, double *L, long long ld, long long stride, int tile_col,
                      int ntiles_below, int batch);
int launch_tile_inverse(Handle *h, const double *L, double *W, long long ld, long long stride,
                        int ntiles, int batch);
int launch_potrf_tile_at(Handle *h, double *L, long long ld, long long stride, long long diag_off, int index_base,
                         int n, int batch, int *info);
int launch_trsm_tiles_at(Handle *h, double *L, long long ld, long long stride, long long diag_off, long long c_off,
                         int ntiles, int batch, TrsmEnv env = TrsmEnv{});
// POTRF of the diagonal tile at diag_off, then TRSM of the `ntiles` tiles from c_off down: one fused launch on the
// latency path, otherwise the two launches above (whose TRSM solves only the tiles live under `env`)
int launch_potrf_trsm_at(Handle *h, double *L, long long ld, long long stride, long long diag_off, int index_base, int n,
                         long long c_off, int ntiles, int batch, int *info, TrsmEnv env = TrsmEnv{});
// env: the envelope record of each item (env_record_ints(ld / TILE) ints, see ENV_BLK), or nullptr
int launch_potrf_trsm(Handle *h, double *L, long long ld, long long stride, int tile_col, int ntiles_below, int n, int batch,
                      int *info, const int *env = nullptr);
int launch_tile_inverse_at(Handle *h, const double *L, long long ld, long long l_off, long long l_step, double *W,
                           long long w_off, long long w_step, long long stride, int ntiles, int batch);
// tile envelope of the SE path (solve.cu): F, E and er from the element profile gram_se_batched records, the trace of the selected inverse
// and the band-limited back substitution.  launch_envelope_profile also writes the dispatch order of the envelope GEMM
// launches to order[0..batch) (order[batch..2 batch) is its scratch)
int launch_envelope_profile(Handle *h, int nt, int *env, int *order, int batch);
int launch_trace_sinv(Handle *h, int n, int np, const double *Z, long long stride, const int *env, const double *x,
                      long long x_stride, const double *a, const double *theta, double *partial, int batch,
                      const int *nvec = nullptr);  // nvec: per-item sizes (device), nullptr = n for every item
int launch_backsub_band(Handle *h, int np, const double *L, const double *Wdiag, long long stride, const int *env,
                        const double *z, double *a, int batch);
int panel_smem_setup(Handle *h);
int panel_trace_fetch(long long *out2048);  // instrumented builds (-DGPB_PANEL_TRACE) only

}  // namespace gpb
