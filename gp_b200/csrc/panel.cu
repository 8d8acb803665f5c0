// Panel kernels of the tiled FP64 Cholesky (sm_100a): the latency-critical 128x128 pieces that sit
// between the DMMA GEMM launches.  They replace the unblocked inner part of Eigen's LLT that runs
// under Stan Math's cholesky_decompose (models/fit_hyperparameters.stan:25, covariance.cpp:29).
//
//   trsm_tile_kernel             X = C L^-T for a 128x128 tile below the diagonal, tile in registers: true
//                                substitution on 8x8 diagonal blocks with quad shuffles, DMMA (mma.sync m8n8k4
//                                f64) for the rank-8 updates (batches)
//   trsm_tiles_pipelined_kernel  the same for several row tiles per CTA, next C tile prefetched (large batches)
//   potrf_tile_pw_kernel         left-looking Cholesky of one 128x128 diagonal tile per CTA in shared memory,
//                                a panel warp carrying the chain of 8x8 diagonal blocks (pivot check -> info)
//   trsm_ll_kernel<MT>           left-looking X = C L^-T, 32 MT rows per CTA (one or a few matrices)
//   tile_inverse_ll_kernel       L^-1 of a diagonal tile (seed of the recursive TRTRI)
//   panel_fused_kernel,          POTRF of the diagonal tile and the TRSM below it in one launch
//   panel_fused_tile_kernel
#include "common.cuh"
#include "panel_ll.cuh"

namespace gpb {

__device__ __forceinline__ void dmma884p(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c[0]), "+d"(c[1])
               : "d"(a), "d"(b));
}

// ------------------------------------------------------------------------------------------------
// TRSM tile: X L^T = C with L the 128x128 lower-triangular diagonal tile, C a 128x128 tile.
// 8 warps; warp w owns rows 16w..16w+15 as two m8 mma row tiles x sixteen n8 column tiles.
// C is read from and X written to the tile (in place); blockIdx.x = row tile, blockIdx.y = batch item.
// ------------------------------------------------------------------------------------------------
constexpr int LD_L = TILE + 4;
constexpr int TRSM_SMEM_BYTES = (TILE * LD_L + TILE) * (int)sizeof(double);

__global__ void __launch_bounds__(256, 1)
trsm_tile_kernel(const double *Ldiag_base, double *Cbase, long long ld, long long stride, long long diag_off,
                 long long c_off, TrsmEnv env) {
  extern __shared__ __align__(16) double sm[];
  double *Ls = sm;                     // Ls[k*LD_L + n] = L[n][k]
  double *invd = sm + TILE * LD_L;     // 1 / L[n][n]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int item = blockIdx.y;
  if (!env.live(item, blockIdx.x)) return;
  const double *Ld = Ldiag_base + (long long)item * stride + diag_off;
  double *Ct = Cbase + (long long)item * stride + c_off + (long long)blockIdx.x * TILE;

  // stage the diagonal tile with cp.async (column-major copy, 16B vectors): all 32 copies of a thread are
  // in flight at once, together with the C-tile loads below (both tiles are 128 KB and this kernel runs
  // one CTA per SM, so exposed load latency is what bounds it)
  for (int idx = tid; idx < TILE * TILE / 2; idx += 256) {
    const int k = idx >> 6, n2 = idx & 63;
    const unsigned dst = (unsigned)__cvta_generic_to_shared(Ls + k * LD_L + 2 * n2);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(Ld + 2 * n2 + (long long)k * ld) : "memory");
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");

  // the C tile goes straight to registers
  double acc[2][16][2];
  const int r0 = warp * 16;
#pragma unroll
  for (int mt = 0; mt < 2; mt++)
#pragma unroll
    for (int nt = 0; nt < 16; nt++)
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int r = r0 + mt * 8 + g, c = nt * 8 + 2 * t + e;
        acc[mt][nt][e] = Ct[r + (long long)c * ld];
      }

  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  __syncthreads();
  if (tid < TILE) invd[tid] = 1.0 / Ls[tid * LD_L + tid];
  __syncthreads();

  const unsigned FULL = 0xffffffffu;
  const int qbase = lane & ~3;
#pragma unroll
  for (int cb = 0; cb < 16; cb++) {
    // (i) substitution inside the 8x8 diagonal block; a row's 8 values live in one quad
#pragma unroll
    for (int c = 0; c < 8; c++) {
      const int owner = qbase + (c >> 1);
      const int n = cb * 8 + c;
      const double dinv = invd[n];
#pragma unroll
      for (int mt = 0; mt < 2; mt++) {
        double xv = acc[mt][cb][c & 1] * dinv;
        if (t == (c >> 1)) acc[mt][cb][c & 1] = xv;
        xv = __shfl_sync(FULL, xv, owner);
        // remaining columns c' > c of this block held by this lane: c' = 2t, 2t+1
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int cp = 2 * t + e;
          if (cp > c) acc[mt][cb][e] = fma(-xv, Ls[n * LD_L + cb * 8 + cp], acc[mt][cb][e]);
        }
      }
    }
    // (ii) re-layout the solved 8 columns from accumulator layout to mma A-operand layout
    double af[2][2];
#pragma unroll
    for (int mt = 0; mt < 2; mt++)
#pragma unroll
      for (int ks = 0; ks < 2; ks++) {
        const int src = qbase + 2 * ks + (t >> 1);
        const double v0 = __shfl_sync(FULL, acc[mt][cb][0], src);
        const double v1 = __shfl_sync(FULL, acc[mt][cb][1], src);
        af[mt][ks] = (t & 1) ? v1 : v0;
      }
    // (iii) rank-8 update of the columns to the right:  C[:, n] -= X[:, cb] * L[n, cb]^T
#pragma unroll
    for (int nt = 0; nt < 16; nt++) {
      if (nt > cb) {
#pragma unroll
        for (int ks = 0; ks < 2; ks++) {
          const double bfv = -Ls[(cb * 8 + ks * 4 + t) * LD_L + nt * 8 + g];
#pragma unroll
          for (int mt = 0; mt < 2; mt++) dmma884p(acc[mt][nt], af[mt][ks], bfv);
        }
      }
    }
  }

#pragma unroll
  for (int mt = 0; mt < 2; mt++)
#pragma unroll
    for (int nt = 0; nt < 16; nt++) {
      const int r = r0 + mt * 8 + g, c = nt * 8 + 2 * t;
      Ct[r + (long long)c * ld] = acc[mt][nt][0];
      Ct[r + (long long)(c + 1) * ld] = acc[mt][nt][1];
    }
}

// ------------------------------------------------------------------------------------------------
// Pipelined TRSM over several row tiles of one block column.  Timing the kernel above
// with its arithmetic removed showed 7.5 of its 18.1 ms per N=4096 step are exposed global-memory time
// (one CTA per SM: load 256 KB, compute, store 128 KB, nothing overlaps).  Here one CTA keeps the diagonal
// tile in shared memory for up to `tiles_per_cta` row tiles -- packed (only the lower triangle, in groups of
// 8 columns: 72 KB instead of 135 KB) so that a full 128x128 prefetch buffer fits next to it -- and the
// cp.async prefetch of the next C tile runs under the substitution + DMMA work of the current one.
// The arithmetic per element is that of trsm_tile_kernel.  What is left (14.4 of 17.3 ms with loads and stores
// removed) is the substitution chain itself: its DMUL/DFMA steps queue behind the other warps' DMMAs on the one
// FP64 pipe (ncu: 44.6 % DMMA-active, DFMA stalls 70 % short-scoreboard + 23 % math-pipe); 16 warps of 8 rows
// instead of 8 warps of 16 rows measured the same.
// ------------------------------------------------------------------------------------------------
__host__ __device__ constexpr int lpk_ld(int cb) { return TILE + 4 - 8 * cb; }   // rows 8cb..127 (+4 pad): == 4 or 12 mod 16
__host__ __device__ constexpr int lpk_off(int cb) { return 8 * (cb * (TILE + 4) - 4 * cb * (cb - 1)); }  // sum_{c<cb} 8*lpk_ld(c)
constexpr int LPK_DOUBLES = lpk_off(16);          // 9216
constexpr int LD_CB = TILE + 2;                   // prefetch buffer: column-major, 130 (conflict-free 8-byte reads)
constexpr int TRSM_PIPE_SMEM_BYTES = (LPK_DOUBLES + TILE + TILE * LD_CB) * (int)sizeof(double);

template <int MT>  // m8 row tiles per warp: 128 / (8 MT) warps per CTA
__global__ void __launch_bounds__(32 * (16 / MT), 1)
trsm_tiles_pipelined_kernel(const double *Ldiag_base, double *Cbase, long long ld, long long stride, long long diag_off,
                            long long c_off, int ntiles, int tiles_per_cta, TrsmEnv env) {
  extern __shared__ __align__(16) double sm[];
  double *Lp = sm;                      // packed: Lp[lpk_off(cb) + kk*lpk_ld(cb) + (n - 8cb)] = L[n][8cb + kk], n >= 8cb
  double *invd = sm + LPK_DOUBLES;      // 1 / L[n][n]
  double *Cb = invd + TILE;             // Cb[c*LD_CB + r] = C[r][c] of the tile being fetched
  constexpr int NTH = 32 * (16 / MT);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int item = blockIdx.y;
  const double *Ld = Ldiag_base + (long long)item * stride + diag_off;
  const int t1 = min(ntiles, (int)blockIdx.x * tiles_per_cta + tiles_per_cta);
  // only the live row tiles of this CTA's range are loaded, solved and stored; a CTA without one never stages L
  auto next_live = [&](int ti) {
    while (ti < t1 && !env.live(item, ti)) ti++;
    return ti;
  };
  int ti = next_live(blockIdx.x * tiles_per_cta);
  if (ti >= t1) return;
  double *Cc = Cbase + (long long)item * stride + c_off;

  auto cp16 = [](double *dst, const double *src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(src) : "memory");
  };
  auto prefetch_c = [&](const double *src) {
#pragma unroll 8
    for (int idx = tid; idx < TILE * TILE / 2; idx += NTH) {
      const int c = idx >> 6, r2 = idx & 63;
      cp16(Cb + c * LD_CB + 2 * r2, src + 2 * r2 + (long long)c * ld);
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  };

  // diagonal tile, packed by groups of 8 columns
#pragma unroll
  for (int cb = 0; cb < 16; cb++) {
    const int rows2 = (TILE - 8 * cb) / 2;          // 16-byte chunks per column of this group
    for (int idx = tid; idx < 8 * rows2; idx += NTH) {
      const int kk = idx / rows2, r2 = idx - kk * rows2;
      cp16(Lp + lpk_off(cb) + kk * lpk_ld(cb) + 2 * r2, Ld + (8 * cb + 2 * r2) + (long long)(8 * cb + kk) * ld);
    }
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  prefetch_c(Cc + (long long)ti * TILE);
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  __syncthreads();
  if (tid < TILE) invd[tid] = 1.0 / Lp[lpk_off(tid >> 3) + (tid & 7) * lpk_ld(tid >> 3) + (tid & 7)];
  __syncthreads();

  const unsigned FULL = 0xffffffffu;
  const int qbase = lane & ~3;
  const int r0 = warp * 8 * MT;
  while (ti < t1) {
    double acc[MT][16][2];
#pragma unroll
    for (int mt = 0; mt < MT; mt++)
#pragma unroll
      for (int nt = 0; nt < 16; nt++)
#pragma unroll
        for (int e = 0; e < 2; e++) acc[mt][nt][e] = Cb[(nt * 8 + 2 * t + e) * LD_CB + r0 + mt * 8 + g];
    __syncthreads();  // everybody has taken its rows out of the buffer
    const int tn = next_live(ti + 1);
    if (tn < t1) prefetch_c(Cc + (long long)tn * TILE);  // next live row tile, in flight during the arithmetic below

#pragma unroll
    for (int cb = 0; cb < 16; cb++) {
      const double *Lg = Lp + lpk_off(cb);  // group cb: Lg[kk*ld + (n - 8cb)]
      const int ldg = lpk_ld(cb);
      // (i) substitution inside the 8x8 diagonal block; a row's 8 values live in one quad
#pragma unroll
      for (int c = 0; c < 8; c++) {
        const int owner = qbase + (c >> 1);
        const double dinv = invd[cb * 8 + c];
#pragma unroll
        for (int mt = 0; mt < MT; mt++) {
          double xv = acc[mt][cb][c & 1] * dinv;
          if (t == (c >> 1)) acc[mt][cb][c & 1] = xv;
          xv = __shfl_sync(FULL, xv, owner);
#pragma unroll
          for (int e = 0; e < 2; e++) {
            const int cp = 2 * t + e;
            if (cp > c) acc[mt][cb][e] = fma(-xv, Lg[c * ldg + cp], acc[mt][cb][e]);
          }
        }
      }
      // (ii) re-layout the solved 8 columns from accumulator layout to mma A-operand layout
      double af[MT][2];
#pragma unroll
      for (int mt = 0; mt < MT; mt++)
#pragma unroll
        for (int ks = 0; ks < 2; ks++) {
          const int src = qbase + 2 * ks + (t >> 1);
          const double v0 = __shfl_sync(FULL, acc[mt][cb][0], src);
          const double v1 = __shfl_sync(FULL, acc[mt][cb][1], src);
          af[mt][ks] = (t & 1) ? v1 : v0;
        }
      // (iii) rank-8 update of the columns to the right:  C[:, n] -= X[:, cb] * L[n, cb]^T
      // (k-step outermost: the two DMMAs that accumulate into the same tile are a whole sweep apart)
#pragma unroll
      for (int ks = 0; ks < 2; ks++) {
#pragma unroll
        for (int nt = 0; nt < 16; nt++) {
          if (nt > cb) {
            const double bfv = -Lg[(ks * 4 + t) * ldg + (nt - cb) * 8 + g];
#pragma unroll
            for (int mt = 0; mt < MT; mt++) dmma884p(acc[mt][nt], af[mt][ks], bfv);
          }
        }
      }
    }

    double *Ct = Cc + (long long)ti * TILE;
#pragma unroll
    for (int mt = 0; mt < MT; mt++)
#pragma unroll
      for (int nt = 0; nt < 16; nt++) {
        const int r = r0 + mt * 8 + g, c = nt * 8 + 2 * t;
        Ct[r + (long long)c * ld] = acc[mt][nt][0];
        Ct[r + (long long)(c + 1) * ld] = acc[mt][nt][1];
      }
    ti = tn;
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncthreads();  // the next tile has landed for everybody
  }
}

// ------------------------------------------------------------------------------------------------
// Round-2 panel kernels: left-looking over 8-column blocks with the tile resident in SHARED memory.
//
// A 128x128 tile kept in registers in mma accumulator layout forces the sixteen block steps to be fully unrolled
// (register arrays need static indices): a register-resident POTRF in that form is 28 000 SASS instructions, each
// executed once -- it runs at instruction-fetch speed (46 us per tile).  With the tile in shared memory every
// index is dynamic, the block loop stays rolled, and the left-looking order needs no register-resident trailing matrix:
//
//   for cb = 0..15:   P  = T[:, 8cb:8cb+8] - T[:, 0:8cb] * T[8cb:8cb+8, 0:8cb]^T     DMMA, own rows
//                     D  = chol(P[8cb:8cb+8, :])                                     panel warp, in registers
//                     T[below, 8cb:8cb+8] = P[below] D^-T                            true substitution, one row per lane
//
// potrf_tile_pw_kernel  eight helper warps own the rows; a ninth PANEL WARP owns no rows and carries the serial chain
//                       of the sixteen 8x8 diagonal blocks beside the helpers' DMMA work instead of in front of it:
//                         phase 1  helpers substitute column block cb against D(cb)  | panel: partial sum of D(cb+1), k-blocks < cb
//                         phase 2  helpers update column block cb+1 for their rows   | panel: last k-block, factor D(cb+1), publish
// trsm_ll_kernel        the rows of X = C L^-T are independent: each warp runs its rows through all sixteen steps with
//                       no block barrier; a CTA takes 32 or 64 rows so that ONE matrix spreads a block column over the GPU
// tile_inverse_ll_kernel  X = L^-T row block by row block into the unused upper triangle of the staged tile
// panel_fused_kernel, panel_fused_tile_kernel   POTRF and TRSM of a block column in ONE launch: the TRSM CTAs follow
//                       the diagonal CTA's factorisation block by block through flags in global memory (64-row CTAs with
//                       the staged L resident, or 128-row CTAs with a double-buffered row block of L)
// Per-phase cycle counts (tools/panel_trace.py, instrumented build) are in profiles/panel_trace_r02.txt.
// ------------------------------------------------------------------------------------------------
constexpr int LD_T = TILE + 4;  // column-major tile in shared memory, 132: conflict-free mma fragment reads

#ifdef GPB_PANEL_TRACE
__device__ long long g_panel_trace[2048];
#define PTRACE(cond, idx) do { if ((cond) && blockIdx.x == 0 && lane == 0) g_panel_trace[(idx)] = clock64(); } while (0)
#define PTRACE_LAST(cond, idx) do { if ((cond) && blockIdx.x == gridDim.x - 1 && (threadIdx.x & 31) == 0) g_panel_trace[(idx)] = clock64(); } while (0)
#else
#define PTRACE(cond, idx) do { } while (0)
#define PTRACE_LAST(cond, idx) do { } while (0)
#endif
constexpr int POTRF_PW_THREADS = 288;
constexpr int POTRF_PW_SMEM_BYTES = (TILE * LD_T + 16 * 64 + 16 * 8 + 64) * (int)sizeof(double);

// FOLLOWED = true (the diagonal CTAs of panel_fused_kernel): every finished column block goes to its final place in
// global memory at once (instead of one write-back at the end) and *flag counts the column blocks that are visible
// device-wide, so that the TRSM CTAs of the same launch can trail the factorisation by one block.
template <bool FOLLOWED>
__device__ __forceinline__ void potrf_pw_body(double *sm, double *__restrict__ T, long long ld, int index_base, int n,
                                              int *info_slot, volatile int *pub_ready) {
  double *Ts = sm;                    // Ts[c * LD_T + r] = T[r][c]  (rows at / below the 8-block of c only)
  double *Dall = sm + TILE * LD_T;    // Dall[cb * 64 + c * 8 + cp] = L_D(cb)[c][cp], cp <= c (row-major), zero above
  double *Iall = Dall + 16 * 64;      // Iall[cb * 8 + c] = 1 / L_D(cb)[c][c]
  double *Dtmp = Iall + 16 * 8;       // the updated diagonal block on its way from mma layout to every lane
  __shared__ int s_info;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const bool panel = warp == 8;
  if (tid == 0) s_info = 0;
  // FOLLOWED: the CTA has a tenth warp (the publisher) that stays out of these barriers
  auto step_sync = [] {
    if (FOLLOWED) asm volatile("bar.sync 0, 288;\n" ::: "memory");
    else __syncthreads();
  };
  PTRACE(warp >= 7, (warp - 7) * 512 + 18 * 8 + 0);

  for (int idx = tid; idx < TILE * TILE / 2; idx += POTRF_PW_THREADS) {
    const int c = idx >> 6, r2 = idx & 63;
    if (2 * r2 + 1 >= (c & ~7)) {
      const unsigned dst = (unsigned)__cvta_generic_to_shared(Ts + c * LD_T + 2 * r2);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(T + 2 * r2 + (long long)c * ld) : "memory");
    }
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  for (int idx = tid; idx < 16 * 64; idx += POTRF_PW_THREADS) Dall[idx] = 0.0;
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  step_sync();

  // factor the 8x8 block whose updated values sit in Dtmp[c * 8 + r] (column-major) and publish it as block `blk`
  auto factor_publish = [&](int blk) {
    double d[8][8], inv[8];
#pragma unroll
    for (int j = 0; j < 8; j++)
#pragma unroll
      for (int i = j; i < 8; i++) d[i][j] = Dtmp[j * 8 + i];
    int bad;
    factor8_pairs(d, inv, bad);
    if (bad >= 0 && lane == 0 && s_info == 0) s_info = index_base + 8 * blk + bad + 1;
    if (lane == 0) {  // every lane holds the same values: one writes the 36 + 8 results (the upper part stays zero)
      double *o = Dall + blk * 64;
#pragma unroll
      for (int c = 0; c < 8; c++) {
#pragma unroll
        for (int cp = 0; cp <= c; cp++) o[c * 8 + cp] = d[c][cp];
        Iall[blk * 8 + c] = inv[c];
      }
    }
  };

  PTRACE(warp >= 7, (warp - 7) * 512 + 17 * 8 + 0);
  if (panel) {
#pragma unroll
    for (int e = 0; e < 2; e++) Dtmp[(2 * t + e) * 8 + g] = Ts[(2 * t + e) * LD_T + g];
    __syncwarp();
    factor_publish(0);
  }
  step_sync();

  const int r0 = warp * 16;
  double ps[2][2];  // panel warp: running sum of L[c1.., k] L[c1.., k]^T for the NEXT diagonal block
#pragma unroll 1
  for (int cb = 0; cb < 16; cb++) {
    const int c0 = 8 * cb, c1 = c0 + 8;
    PTRACE(warp >= 7, (warp - 7) * 512 + cb * 8 + 0);
    // ---- phase 1 ----------------------------------------------------------------------------------------------
    if (!panel) {
      const int r = r0 + lane;
      if (lane < 16 && (r >> 3) > cb) {
        double dl[8][8], inv[8], x[8];
        double *px = Ts + c0 * LD_T + r;
#pragma unroll
        for (int c = 0; c < 8; c++) x[c] = px[c * LD_T];
        load_block8(Dall + cb * 64, Iall + cb * 8, dl, inv);
        solve_row8(x, dl, inv);
#pragma unroll
        for (int c = 0; c < 8; c++) px[c * LD_T] = x[c];
      }
    } else if (cb < 15) {
      ps[0][0] = ps[0][1] = ps[1][0] = ps[1][1] = 0.0;
      if (cb > 0) {  // A and B fragments are the same registers: rows c1.. against themselves
        const double *pa = Ts + t * LD_T + c1 + g;
        double v0 = pa[0], v1 = pa[4 * LD_T];
        for (int kb = 0; kb < cb; kb++) {
          pa += 8 * LD_T;
          double n0 = 0.0, n1 = 0.0;
          if (kb + 1 < cb) { n0 = pa[0]; n1 = pa[4 * LD_T]; }
          dmma884v(ps[0], v0, v0);
          dmma884v(ps[1], v1, v1);
          v0 = n0; v1 = n1;
        }
      }
    }
    PTRACE(warp >= 7, (warp - 7) * 512 + cb * 8 + 1);
    step_sync();
    PTRACE(warp >= 7, (warp - 7) * 512 + cb * 8 + 2);
    if (FOLLOWED && tid == 0) *pub_ready = cb + 1;   // column block cb is final: the publisher warp takes it from here
    if (cb == 15) break;
    // ---- phase 2 ----------------------------------------------------------------------------------------------
    if (!panel) {
      // each helper updates the rows it owns.  (Dealing the remaining row blocks out evenly over all eight helpers was
      // measured SLOWER, 28.7 against 26.6 us per tile: the helpers are not the critical path, the panel warp is, and
      // every extra busy warp takes issue slots and FP64-pipe cycles from it.)
      const int rb0 = 2 * warp;
      const bool act[2] = {rb0 > cb + 1, rb0 + 1 > cb + 1};
      if (act[1]) {
        double s[2][2][2];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
          for (int ch = 0; ch < 2; ch++) s[mt][ch][0] = s[mt][ch][1] = 0.0;
        ll_accumulate<2>(s, Ts + t * LD_T + 8 * rb0 + g, Ts + t * LD_T + c1 + g, cb + 1, 8 * LD_T, 8 * LD_T, 4 * LD_T, 4 * LD_T, 8, act);
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
          if (!act[mt]) continue;
#pragma unroll
          for (int e = 0; e < 2; e++) {
            double *p = Ts + (c1 + 2 * t + e) * LD_T + 8 * (rb0 + mt) + g;
            *p = (*p - s[mt][0][e]) - s[mt][1][e];
          }
        }
      }
    } else {
      const double *pa = Ts + t * LD_T + c1 + g;
      const double v0 = pa[c0 * LD_T], v1 = pa[(c0 + 4) * LD_T];
      dmma884v(ps[0], v0, v0);
      dmma884v(ps[1], v1, v1);
#pragma unroll
      for (int e = 0; e < 2; e++)
        Dtmp[(2 * t + e) * 8 + g] = (Ts[(c1 + 2 * t + e) * LD_T + c1 + g] - ps[0][e]) - ps[1][e];
      __syncwarp();
      PTRACE(warp >= 7, (warp - 7) * 512 + cb * 8 + 3);
      factor_publish(cb + 1);
    }
    PTRACE(warp >= 7, (warp - 7) * 512 + cb * 8 + 4);
    step_sync();
    PTRACE(warp >= 7, (warp - 7) * 512 + cb * 8 + 5);
  }
  PTRACE(warp >= 7, (warp - 7) * 512 + 16 * 8 + 0);
  // write back: lower triangle = L (diagonal blocks from Dall), strict upper = 0 (Eigen matrixL() convention)
  for (int idx = tid; !FOLLOWED && idx < TILE * TILE / 2; idx += POTRF_PW_THREADS) {
    const int c = idx >> 6, r = 2 * (idx & 63);
    double2 v = make_double2(0.0, 0.0);
    if ((r >> 3) == (c >> 3)) {
      const double *o = Dall + (c >> 3) * 64;
      v.x = o[(r & 7) * 8 + (c & 7)];
      v.y = o[((r + 1) & 7) * 8 + (c & 7)];
    } else if (r > c) {
      v = *reinterpret_cast<const double2 *>(Ts + c * LD_T + r);
    }
    *reinterpret_cast<double2 *>(T + r + (long long)c * ld) = v;
  }
  PTRACE(warp >= 7, (warp - 7) * 512 + 16 * 8 + 1);
  if (tid == 0 && s_info != 0 && s_info <= n) {
    if (*info_slot == 0) *info_slot = s_info;
  }
}

// The tenth warp of a diagonal CTA of panel_fused_kernel.  When column block cb is final in shared memory (pub_ready,
// written after the barrier that ends its substitution) it stores the block to its final place in global memory
// (zeros above the diagonal block, the diagonal block from Dall, the substituted rows from Ts; lane -> column lane / 4,
// four consecutive rows out of every sixteen) and releases *flag = cb + 1.  The stores and above all the release
// (a device-scope fence: about a thousand cycles) are as long as a phase of the factorisation; on a warp of its own
// they are off the step barriers (done by an idle helper warp they added 300 to 600 cycles to every block step, traced).
__device__ __forceinline__ void potrf_publisher(const double *sm, double *__restrict__ T, long long ld, int *flag,
                                                volatile int *pub_ready) {
  const double *Ts = sm, *Dall = sm + TILE * LD_T;
  const int lane = threadIdx.x & 31;
#pragma unroll 1
  for (int cb = 0; cb < 16; cb++) {
    while (*pub_ready < cb + 1) __nanosleep(40);
    __syncwarp();
    __threadfence_block();
    const int c = 8 * cb + (lane >> 2);
    const double *o = Dall + cb * 64 + (c & 7);
    double *dst = T + (long long)c * ld;
#pragma unroll 2
    for (int k = 0; k < 8; k++) {
      const int rr = 16 * k + 4 * (lane & 3);
      double2 v0 = make_double2(0.0, 0.0), v1 = v0;
      if (rr >= 8 * cb + 8) {
        v0 = *reinterpret_cast<const double2 *>(Ts + c * LD_T + rr);
        v1 = *reinterpret_cast<const double2 *>(Ts + c * LD_T + rr + 2);
      } else if (rr >= 8 * cb) {
        v0 = make_double2(o[(rr & 7) * 8], o[((rr + 1) & 7) * 8]);
        v1 = make_double2(o[((rr + 2) & 7) * 8], o[((rr + 3) & 7) * 8]);
      }
      *reinterpret_cast<double2 *>(dst + rr) = v0;
      *reinterpret_cast<double2 *>(dst + rr + 2) = v1;
    }
    __syncwarp();
    if (lane == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(flag), "r"(cb + 1) : "memory");
  }
}

__global__ void __launch_bounds__(POTRF_PW_THREADS, 1)
potrf_tile_pw_kernel(double *__restrict__ Lbase, long long ld, long long stride, long long diag_off, int index_base,
                     int n, int *info) {
  extern __shared__ __align__(16) double sm[];
  potrf_pw_body<false>(sm, Lbase + (long long)blockIdx.x * stride + diag_off, ld, index_base, n, info + blockIdx.x, nullptr);
}

// X L^T = C for ROWS = 32 MT consecutive rows of a block column (in place, like trsm_tile_kernel), four warps
// of 8 MT rows each, no block barrier in the main loop.  blockIdx.x = row chunk, blockIdx.y = batch item.
// The diagonal tile sits in shared memory as a full square (constant strides: every fragment address is one base
// register plus an immediate), its sixteen 8x8 diagonal blocks once more row-major (Dall) for the substitution.
template <int MT>
struct TrsmLL {
  static constexpr int ROWS = 32 * MT;
  static constexpr int LD_C = ROWS + 4;
  static constexpr int SMEM_BYTES = (TILE * LD_T + 16 * 64 + TILE + TILE * LD_C) * (int)sizeof(double);
};

// FOLLOW = true (the TRSM CTAs of panel_fused_kernel): the diagonal tile is still being factored by another CTA of the
// same launch; column block cb of L is fetched from global memory when *flag says it is visible (>= cb + 1).  The 128
// working threads meet at named barrier 1 (the CTA has more threads than this role uses).
template <int MT, bool FOLLOW>
__device__ __forceinline__ void trsm_ll_body(double *sm, const double *Ld, double *Ct, long long ld, unsigned long long *ready) {
  constexpr int ROWS = TrsmLL<MT>::ROWS, LD_C = TrsmLL<MT>::LD_C;
  double *Ls = sm;                   // Ls[k * LD_T + n] = L[n][k]
  double *Dall = sm + TILE * LD_T;   // Dall[cb * 64 + c * 8 + cp] = L[8cb + c][8cb + cp]
  double *invd = Dall + 16 * 64;     // 1 / L[n][n]
  double *Cs = invd + TILE;          // Cs[c * LD_C + r] = C[r][c]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  auto role_sync = [] { asm volatile("bar.sync 1, 128;\n" ::: "memory"); };

  auto cp16 = [](double *dst, const double *src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(src) : "memory");
  };
  if (FOLLOW) PTRACE_LAST(warp == 0, 1024 + 18 * 8); else PTRACE(warp == 0, 1024 + 18 * 8);
  if (!FOLLOW) {
    for (int idx = tid; idx < TILE * TILE / 2; idx += 128) {
      const int k = idx >> 6, r2 = idx & 63;
      if (2 * r2 + 1 >= (k & ~7)) cp16(Ls + k * LD_T + 2 * r2, Ld + 2 * r2 + (long long)k * ld);  // rows at / below the block row of k
    }
  }
  for (int idx = tid; idx < TILE * ROWS / 2; idx += 128) {
    const int c = idx / (ROWS / 2), r2 = idx - c * (ROWS / 2);
    cp16(Cs + c * LD_C + 2 * r2, Ct + 2 * r2 + (long long)c * ld);
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  if (!FOLLOW) {
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    role_sync();
    if (tid < TILE) invd[tid] = 1.0 / Ls[tid * LD_T + tid];
    for (int idx = tid; idx < 16 * 64; idx += 128) {
      const int cb = idx >> 6, c = (idx >> 3) & 7, cp = idx & 7;
      Dall[idx] = Ls[(8 * cb + cp) * LD_T + 8 * cb + c];
    }
    role_sync();
  }

  const int r0 = warp * 8 * MT;
  bool act[MT];
#pragma unroll
  for (int mt = 0; mt < MT; mt++) act[mt] = true;
  if (FOLLOW) PTRACE_LAST(warp == 0, 1024 + 17 * 8); else PTRACE(warp == 0, 1024 + 17 * 8);
  if (FOLLOW) {
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    role_sync();   // the C chunk has landed for everybody
  }
#pragma unroll 1
  for (int cb = 0; cb < 16; cb++) {
    const int c0 = 8 * cb;
    if (FOLLOW) PTRACE_LAST(warp == 0, 1024 + cb * 8 + 0); else PTRACE(warp == 0, 1024 + cb * 8 + 0);
    double dl[8][8], inv[8];
    if (!FOLLOW) load_block8(Dall + cb * 64, invd + c0, dl, inv);   // fetched before the DMMA loop: landed long before the substitution
    if (cb > 0) {
      // S = X[rows, 0:c0] * L[c0:c0+8, 0:c0]^T, two independent accumulation chains per m-tile.  (FOLLOW: this part needs
      // only column blocks < cb, which arrived one step ago: it runs BEFORE the wait for block cb.)
      double s[MT][2][2];
#pragma unroll
      for (int mt = 0; mt < MT; mt++)
#pragma unroll
        for (int ch = 0; ch < 2; ch++) s[mt][ch][0] = s[mt][ch][1] = 0.0;
      ll_accumulate<MT>(s, Cs + t * LD_C + r0 + g, Ls + t * LD_T + c0 + g, cb, 8 * LD_C, 8 * LD_T, 4 * LD_C, 4 * LD_T, 8, act);
#pragma unroll
      for (int mt = 0; mt < MT; mt++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
          double *p = Cs + (c0 + 2 * t + e) * LD_C + r0 + mt * 8 + g;
          *p = (*p - s[mt][0][e]) - s[mt][1][e];
        }
      __syncwarp();
    }
    if (FOLLOW) {
      PTRACE_LAST(warp == 0, 1024 + cb * 8 + 3);
      // column block cb is staged by the loader warp (trsm_follow_loader) while these warps do the update above
      {
        const unsigned mb = (unsigned)__cvta_generic_to_shared(ready + cb);
        asm volatile(
            "{\n.reg .pred p;\nWAIT_BLOCK:\n"
            "mbarrier.try_wait.parity.shared.b64 p, [%0], 0;\n"
            "@!p bra WAIT_BLOCK;\n}\n" ::"r"(mb) : "memory");
      }
      // every lane reads the 8x8 diagonal block straight from the staged columns (lower part; the upper part is zero)
#pragma unroll
      for (int c = 0; c < 8; c++)
#pragma unroll
        for (int cp = 0; cp < 8; cp++) dl[c][cp] = cp < c ? Ls[(c0 + cp) * LD_T + c0 + c] : 0.0;
      const double my_inv = 1.0 / Ls[(c0 + (lane & 7)) * (LD_T + 1)];   // one reciprocal per lane, handed round
#pragma unroll
      for (int c = 0; c < 8; c++) inv[c] = __shfl_sync(0xffffffffu, my_inv, c);
    }
    if (FOLLOW) PTRACE_LAST(warp == 0, 1024 + cb * 8 + 1); else PTRACE(warp == 0, 1024 + cb * 8 + 1);
    // substitution against the 8x8 diagonal block, one row per lane
    if (lane < 8 * MT) {
      double *px = Cs + c0 * LD_C + r0 + lane;
      double x[8];
#pragma unroll
      for (int c = 0; c < 8; c++) x[c] = px[c * LD_C];
      solve_row8(x, dl, inv);
#pragma unroll
      for (int c = 0; c < 8; c++) px[c * LD_C] = x[c];
      if (FOLLOW) {   // finished columns go out at once: nothing is left to write when the last block has been solved
        double *out = Ct + r0 + lane + (long long)c0 * ld;
#pragma unroll
        for (int c = 0; c < 8; c++) out[(long long)c * ld] = x[c];
      }
    }
    __syncwarp();
    if (FOLLOW) PTRACE_LAST(warp == 0, 1024 + cb * 8 + 2); else PTRACE(warp == 0, 1024 + cb * 8 + 2);
  }
  if (FOLLOW) { PTRACE_LAST(warp == 0, 1024 + 16 * 8); return; }
  role_sync();
  PTRACE(warp == 0, 1024 + 16 * 8);
  for (int idx = tid; idx < TILE * ROWS / 2; idx += 128) {
    const int c = idx / (ROWS / 2), r2 = idx - c * (ROWS / 2);
    *reinterpret_cast<double2 *>(Ct + 2 * r2 + (long long)c * ld) = *reinterpret_cast<const double2 *>(Cs + c * LD_C + 2 * r2);
  }
}

// The fifth warp of a TRSM CTA of panel_fused_kernel: waits for each column block of the diagonal tile to become visible
// (*flag >= cb + 1, raised by the diagonal CTA) and copies its rows at and below the diagonal block into the CTA's staged L
// with cp.async; the copies of block cb complete on mbarrier ready[cb] (one arrival per lane, counted when that lane's
// copies have landed), which is what the four working warps wait on -- so the L2 round trips of the wait and of the copy
// run beside the working warps' DMMA updates, and this warp is already polling for block cb + 1 while block cb lands.
__device__ __forceinline__ void trsm_follow_loader(double *sm, const double *Ld, long long ld, const int *flag,
                                                   unsigned long long *ready) {
  double *Ls = sm;
  const int lane = threadIdx.x & 31;
#pragma unroll 1
  for (int cb = 0; cb < 16; cb++) {
    const int c0 = 8 * cb;
    PTRACE_LAST(true, 1536 + cb * 8 + 0);
    if (lane == 0) {
      int seen;
      do {   // relaxed polls (an acquire load invalidates the L1 on every iteration), one acquire fence at the end
        asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];\n" : "=r"(seen) : "l"(flag) : "memory");
      } while (seen < cb + 1);
      asm volatile("fence.acq_rel.gpu;\n" ::: "memory");
    }
    __syncwarp();
    PTRACE_LAST(true, 1536 + cb * 8 + 1);
    // all 128 rows of the eight columns (the rows above the diagonal block are zeros nobody reads): a fixed pattern of
    // sixteen 16-byte copies per lane keeps this loop a few dozen instructions long
    {
      const double *src = Ld + (long long)c0 * ld + 2 * lane;
      const unsigned dst = (unsigned)__cvta_generic_to_shared(Ls + c0 * LD_T + 2 * lane);
#pragma unroll
      for (int c = 0; c < 8; c++) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst + (unsigned)(c * LD_T * 8)), "l"(src + (long long)c * ld) : "memory");
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst + (unsigned)(c * LD_T * 8 + 512)), "l"(src + (long long)c * ld + 64) : "memory");
      }
    }
    const unsigned mb = (unsigned)__cvta_generic_to_shared(ready + cb);
    asm volatile("cp.async.mbarrier.arrive.noinc.shared.b64 [%0];\n" ::"r"(mb) : "memory");
    PTRACE_LAST(true, 1536 + cb * 8 + 2);
  }
  asm volatile("cp.async.wait_all;\n" ::: "memory");   // nothing of this warp is in flight when it exits
}

template <int MT>
__global__ void __launch_bounds__(128)
trsm_ll_kernel(const double *Ldiag_base, double *Cbase, long long ld, long long stride, long long diag_off, long long c_off) {
  extern __shared__ __align__(16) double sm[];
  trsm_ll_body<MT, false>(sm, Ldiag_base + (long long)blockIdx.y * stride + diag_off,
                          Cbase + (long long)blockIdx.y * stride + c_off + (long long)blockIdx.x * TrsmLL<MT>::ROWS, ld, nullptr);
}

// POTRF of the diagonal tile and the TRSM of the tiles below it in ONE launch (the latency path: one or a few matrices).
// CTAs [0, batch) factor the diagonal tiles and publish them column block by column block; CTAs [batch, ...) take
// 64 rows each of the block column below and trail the factorisation by about one 8-column block instead of
// starting when it has finished (16.5 us later and a launch gap).  The diagonal CTAs wait for nobody and have the
// lowest block indices, so every waiting CTA waits for a CTA that is already resident.  flags[2 m] counts matrix m's
// visible column blocks, flags[2 m + 1] its finished TRSM CTAs; the last one to finish clears both for the next launch.
constexpr int PANEL_FUSED_SMEM_BYTES = TrsmLL<2>::SMEM_BYTES > POTRF_PW_SMEM_BYTES ? TrsmLL<2>::SMEM_BYTES : POTRF_PW_SMEM_BYTES;
constexpr int PANEL_FUSED_THREADS = POTRF_PW_THREADS + 32;

__global__ void __launch_bounds__(PANEL_FUSED_THREADS, 1)
panel_fused_kernel(double *__restrict__ Lbase, long long ld, long long stride, long long diag_off, long long c_off,
                   int chunks, int batch, int index_base, int n, int *info, int *flags) {
  extern __shared__ __align__(16) double sm[];
  if ((int)blockIdx.x < batch) {
    __shared__ int s_pub;
    const int m = blockIdx.x;
    double *T = Lbase + (long long)m * stride + diag_off;
    if (threadIdx.x == POTRF_PW_THREADS) s_pub = 0;
    __syncthreads();
    if (threadIdx.x >= POTRF_PW_THREADS) potrf_publisher(sm, T, ld, flags + 2 * m, &s_pub);
    else potrf_pw_body<true>(sm, T, ld, index_base, n, info + m, &s_pub);
    return;
  }
  __shared__ __align__(8) unsigned long long s_ready[16];   // one mbarrier per column block, each used for one phase
  if (threadIdx.x >= 160) return;
  const int idx = (int)blockIdx.x - batch, m = idx / chunks, chunk = idx - m * chunks;
  double *base = Lbase + (long long)m * stride;
  if (threadIdx.x >= 128 && threadIdx.x < 144) {
    const unsigned mb = (unsigned)__cvta_generic_to_shared(s_ready + (threadIdx.x - 128));
    asm volatile("mbarrier.init.shared.b64 [%0], 32;\n" ::"r"(mb) : "memory");
  }
  asm volatile("bar.sync 2, 160;\n" ::: "memory");
  if (threadIdx.x >= 128) {
    trsm_follow_loader(sm, base + diag_off, ld, flags + 2 * m, s_ready);
    return;
  }
  trsm_ll_body<2, true>(sm, base + diag_off, base + c_off + (long long)chunk * TrsmLL<2>::ROWS, ld, s_ready);
  if (threadIdx.x == 0) {
    if (atomicAdd(flags + 2 * m + 1, 1) == chunks - 1) {
      flags[2 * m + 1] = 0;
      *reinterpret_cast<volatile int *>(flags + 2 * m) = 0;
    }
  }
}

// ---- the TRSM CTAs of panel_fused_tile_kernel (more row tiles than 64-row CTAs fit in one wave) -------------------
// One CTA per 128-row tile below the diagonal tile: eight working warps of sixteen rows each, one loader warp.  The
// diagonal tile is still being factored by another CTA of the same launch, which publishes it column block by
// column block (*flag = number of visible blocks).  Step cb of the substitution needs row block cb of L:
//   part A  L[8cb .. 8cb+7][0 .. 8cb-1]   lies in column blocks < cb: visible one step EARLIER (flag >= cb)
//   part D  the 8x8 diagonal block         visible when flag >= cb + 1
// so the loader stages part A of row block i and part D of block i - 1 when the flag reaches i; the working warps do
// the DMMA update of step cb (part A) while block cb is still on its way and wait only for its 64 diagonal-block
// numbers.  Part A lives in two alternating buffers (full / empty mbarriers), part D in sixteen one-shot slots.
// Only the C tile is resident (135 KB): a row tile per CTA, so one launch covers up to 147 row tiles.
constexpr int LD_R = 20;   // row-block buffer RB[k * LD_R + i] = L[8cb + i][k]; 20 = 4 (mod 16): conflict-free B fragments
template <int NW>   // working warps per CTA: 4 (64 rows) or 8 (128 rows)
struct Follow {
  static constexpr int ROWS = 16 * NW, LD_C = ROWS + 4;
  static constexpr int C_DOUBLES = TILE * LD_C;
  static constexpr int SMEM_BYTES = (C_DOUBLES + 2 * TILE * LD_R + 16 * 64) * (int)sizeof(double);
};

struct FollowBars {
  unsigned long long fullD[16], fullR[2], emptyR[2];
};

__device__ __forceinline__ void mbar_wait(const unsigned long long *bar, unsigned parity) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  unsigned ok;
  do {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(a), "r"(parity) : "memory");
  } while (!ok);
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared.b64 st, [%0];\n}\n" ::"r"(a) : "memory");
}
__device__ __forceinline__ void mbar_arrive_on_copies(unsigned long long *bar) {   // counted when this thread's cp.asyncs have landed
  const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("cp.async.mbarrier.arrive.noinc.shared.b64 [%0];\n" ::"r"(a) : "memory");
}

__device__ __forceinline__ void trsm_tile_follow_loader(double *RB, const double *Ld, long long ld, const int *flag, FollowBars *bars) {
  double *Dbuf = RB + 2 * TILE * LD_R;
  const int lane = threadIdx.x & 31;
  const int part = lane & 3, colq = lane >> 2;
#pragma unroll 1
  for (int i = 1; i <= 16; i++) {
    PTRACE_LAST(true, 1536 + (i - 1) * 8 + 0);
    if (lane == 0) {
      int seen;
      do {   // relaxed polls (an acquire load invalidates the L1 on every iteration), one acquire fence at the end
        asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];\n" : "=r"(seen) : "l"(flag) : "memory");
      } while (seen < i);
      asm volatile("fence.acq_rel.gpu;\n" ::: "memory");
    }
    __syncwarp();
    PTRACE_LAST(true, 1536 + (i - 1) * 8 + 1);
    {  // part D of block i - 1: 8 columns x 8 rows, one 16-byte piece per lane
      const int d0 = 8 * (i - 1);
      const unsigned dst = (unsigned)__cvta_generic_to_shared(Dbuf + (i - 1) * 64 + colq * 8 + 2 * part);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(Ld + d0 + 2 * part + (long long)(d0 + colq) * ld) : "memory");
      mbar_arrive_on_copies(&bars->fullD[i - 1]);
    }
    if (i <= 15) {  // part A of row block i: rows 8i .. 8i+7 of columns 0 .. 8i-1
      const int b = i & 1, use = (i - 1) >> 1;
      if (use >= 1) mbar_wait(&bars->emptyR[b], (use - 1) & 1);
      const double *src = Ld + 8 * i + 2 * part + (long long)colq * ld;
      unsigned dst = (unsigned)__cvta_generic_to_shared(RB + b * TILE * LD_R + colq * LD_R + 2 * part);
#pragma unroll 1
      for (int col = colq; col < 8 * i; col += 8) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(src) : "memory");
        src += 8 * ld;
        dst += 8 * LD_R * 8;
      }
      mbar_arrive_on_copies(&bars->fullR[b]);
    }
    PTRACE_LAST(true, 1536 + (i - 1) * 8 + 2);
  }
  asm volatile("cp.async.wait_all;\n" ::: "memory");   // nothing of this warp is in flight when it exits
}

template <int NW>
__device__ __forceinline__ void trsm_tile_follow_compute(double *sm, double *Ct, long long ld, FollowBars *bars) {
  constexpr int ROWS = Follow<NW>::ROWS, LD_C = Follow<NW>::LD_C;
  double *Cs = sm;   // Cs[c * LD_C + r] = C[r][c], ROWS rows of the block column
  const double *RB = sm + Follow<NW>::C_DOUBLES, *Dbuf = RB + 2 * TILE * LD_R;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  PTRACE_LAST(warp == 0, 1024 + 18 * 8);
  for (int idx = tid; idx < TILE * ROWS / 2; idx += 32 * NW) {
    const int c = idx / (ROWS / 2), r2 = idx - c * (ROWS / 2);
    const unsigned d = (unsigned)__cvta_generic_to_shared(Cs + c * LD_C + 2 * r2);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(Ct + 2 * r2 + (long long)c * ld) : "memory");
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  asm volatile("bar.sync 1, %0;\n" ::"n"(32 * NW) : "memory");   // the C rows have landed for all working warps
  const int r0 = warp * 16;
  const bool act[2] = {true, true};
  PTRACE_LAST(warp == 0, 1024 + 17 * 8);
#pragma unroll 1
  for (int cb = 0; cb < 16; cb++) {
    const int c0 = 8 * cb;
    PTRACE_LAST(warp == 0, 1024 + cb * 8 + 0);
    if (cb > 0) {
      const int b = cb & 1;
      mbar_wait(&bars->fullR[b], ((cb - 1) >> 1) & 1);
      // S = X[rows, 0:c0] * L[c0:c0+8, 0:c0]^T, two independent accumulation chains per m-tile
      double s[2][2][2];
#pragma unroll
      for (int mt = 0; mt < 2; mt++)
#pragma unroll
        for (int ch = 0; ch < 2; ch++) s[mt][ch][0] = s[mt][ch][1] = 0.0;
      ll_accumulate<2>(s, Cs + t * LD_C + r0 + g, RB + b * TILE * LD_R + t * LD_R + g, cb, 8 * LD_C, 8 * LD_R, 4 * LD_C, 4 * LD_R, 8, act);
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->emptyR[b]);   // this warp is done with the row-block buffer
#pragma unroll
      for (int mt = 0; mt < 2; mt++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
          double *p = Cs + (c0 + 2 * t + e) * LD_C + r0 + mt * 8 + g;
          *p = (*p - s[mt][0][e]) - s[mt][1][e];
        }
      __syncwarp();
    }
    PTRACE_LAST(warp == 0, 1024 + cb * 8 + 3);
    mbar_wait(&bars->fullD[cb], 0);
    double dl[8][8], inv[8];
    const double *D = Dbuf + cb * 64;   // D[c * 8 + r] = L[c0 + r][c0 + c]
#pragma unroll
    for (int c = 0; c < 8; c++)
#pragma unroll
      for (int cp = 0; cp < 8; cp++) dl[c][cp] = cp < c ? D[cp * 8 + c] : 0.0;
    const double my_inv = 1.0 / D[(lane & 7) * 9];   // one reciprocal per lane, handed round
#pragma unroll
    for (int c = 0; c < 8; c++) inv[c] = __shfl_sync(0xffffffffu, my_inv, c);
    PTRACE_LAST(warp == 0, 1024 + cb * 8 + 1);
    // substitution against the 8x8 diagonal block, one row per lane; finished columns go out at once, so nothing is left
    // to write when the last block has been solved
    if (lane < 16) {
      double *px = Cs + c0 * LD_C + r0 + lane;
      double x[8];
#pragma unroll
      for (int c = 0; c < 8; c++) x[c] = px[c * LD_C];
      solve_row8(x, dl, inv);
      double *out = Ct + r0 + lane + (long long)c0 * ld;
#pragma unroll
      for (int c = 0; c < 8; c++) {
        px[c * LD_C] = x[c];
        out[(long long)c * ld] = x[c];
      }
    }
    __syncwarp();
    PTRACE_LAST(warp == 0, 1024 + cb * 8 + 2);
  }
  PTRACE_LAST(warp == 0, 1024 + 16 * 8);
}

constexpr int PANEL_FUSED_TILE_SMEM_BYTES = Follow<8>::SMEM_BYTES > POTRF_PW_SMEM_BYTES ? Follow<8>::SMEM_BYTES : POTRF_PW_SMEM_BYTES;

// The same fused launch with one TRSM CTA per 128-row tile (eight working warps; only the C tile and a row block of L
// are resident): covers up to 147 row tiles, at steps about 7 % slower than the 64-row form above.
__global__ void __launch_bounds__(POTRF_PW_THREADS + 32, 1)
panel_fused_tile_kernel(double *__restrict__ Lbase, long long ld, long long stride, long long diag_off, long long c_off,
                        int tiles, int batch, int index_base, int n, int *info, int *flags) {
  extern __shared__ __align__(16) double sm[];
  if ((int)blockIdx.x < batch) {
    __shared__ int s_pub;
    const int m = blockIdx.x;
    double *T = Lbase + (long long)m * stride + diag_off;
    if (threadIdx.x == POTRF_PW_THREADS) s_pub = 0;
    __syncthreads();
    if (threadIdx.x >= POTRF_PW_THREADS) potrf_publisher(sm, T, ld, flags + 2 * m, &s_pub);
    else potrf_pw_body<true>(sm, T, ld, index_base, n, info + m, &s_pub);
    return;
  }
  constexpr int NW = 8, WORK = 32 * NW, ALL = WORK + 32;   // working threads, plus the loader warp
  __shared__ __align__(8) FollowBars bars;
  if (threadIdx.x >= ALL) return;
  const int idx = (int)blockIdx.x - batch, m = idx / tiles, tile = idx - m * tiles;
  double *base = Lbase + (long long)m * stride;
  if (threadIdx.x >= WORK && threadIdx.x < WORK + 20) {
    const int k = threadIdx.x - WORK;   // fullD[0..15], fullR[0..1]: 32 loader lanes each; emptyR[0..1]: one arrival per working warp
    unsigned long long *bar = k < 16 ? &bars.fullD[k] : (k < 18 ? &bars.fullR[k - 16] : &bars.emptyR[k - 18]);
    const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.init.shared.b64 [%0], %1;\n" ::"r"(a), "r"(k < 18 ? 32 : NW) : "memory");
  }
  asm volatile("bar.sync 2, %0;\n" ::"n"(ALL) : "memory");
  if (threadIdx.x >= WORK) {
    trsm_tile_follow_loader(sm + Follow<NW>::C_DOUBLES, base + diag_off, ld, flags + 2 * m, &bars);
    return;
  }
  trsm_tile_follow_compute<NW>(sm, base + c_off + (long long)tile * TILE, ld, &bars);
  asm volatile("bar.sync 1, %0;\n" ::"n"(WORK) : "memory");
  if (threadIdx.x == 0) {
    if (atomicAdd(flags + 2 * m + 1, 1) == tiles - 1) {
      flags[2 * m + 1] = 0;
      *reinterpret_cast<volatile int *>(flags + 2 * m) = 0;
    }
  }
}

// W = L^-1 of one 128x128 lower-triangular tile per CTA (W lower triangular, strict upper zero; in place allowed).  X = L^-T is computed row block by row block -- its rows are independent, so
// the eight warps never meet at a barrier -- left-looking over the column blocks at and right of the row block
// (everything left of it is zero and is skipped).  X is upper triangular and lives in the UNUSED upper triangle of
// the staged L tile; its 8x8 diagonal blocks, which would collide with L's, go to a side buffer.  Warp w takes row
// blocks w and 15 - w (a long and a short one).
constexpr int TINV_SMEM_BYTES = (TILE * LD_T + 16 * 64 + TILE + 16 * 64) * (int)sizeof(double);

__global__ void __launch_bounds__(256, 1)
tile_inverse_ll_kernel(const double *Lbase, double *Wbase, long long ld, long long stride, long long l_off, long long l_step,
                       long long w_off, long long w_step) {
  extern __shared__ __align__(16) double sm[];
  double *Ls = sm;                   // lower: Ls[k * LD_T + n] = L[n][k]; strict upper (outside diagonal blocks): X[r][c] at Ls[c * LD_T + r]
  double *Dall = sm + TILE * LD_T;   // Dall[cb * 64 + c * 8 + cp] = L[8cb + c][8cb + cp]
  double *invd = Dall + 16 * 64;     // 1 / L[n][n] = X[n][n]
  double *XD = invd + TILE;          // XD[rb * 64 + k * 8 + i] = X[8rb + i][8rb + k]  (upper triangular incl. diagonal)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const double *Ld = Lbase + (long long)blockIdx.y * stride + l_off + (long long)blockIdx.x * l_step;
  double *Wt = Wbase + (long long)blockIdx.y * stride + w_off + (long long)blockIdx.x * w_step;

  for (int idx = tid; idx < TILE * TILE / 2; idx += 256) {
    const int k = idx >> 6, r2 = idx & 63;
    if (2 * r2 + 1 >= (k & ~7)) {
      const unsigned dst = (unsigned)__cvta_generic_to_shared(Ls + k * LD_T + 2 * r2);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(Ld + 2 * r2 + (long long)k * ld) : "memory");
    }
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
  __syncthreads();
  if (tid < TILE) invd[tid] = 1.0 / Ls[tid * LD_T + tid];
  for (int idx = tid; idx < 16 * 64; idx += 256) {
    const int cb = idx >> 6, c = (idx >> 3) & 7, cp = idx & 7;
    Dall[idx] = Ls[(8 * cb + cp) * LD_T + 8 * cb + c];
  }
  __syncthreads();

  const bool act[1] = {true};
#pragma unroll 1
  for (int slot = 0; slot < 2; slot++) {
    const int rb = slot == 0 ? warp : 15 - warp;
    const int r0 = 8 * rb;
    double *xd = XD + rb * 64;
#pragma unroll 1
    for (int cb = rb; cb < 16; cb++) {
      const int c0 = 8 * cb;
      double dl[8][8], inv[8];
      load_block8(Dall + cb * 64, invd + c0, dl, inv);
      if (cb > rb) {
        double s[1][2][2];
        s[0][0][0] = s[0][0][1] = s[0][1][0] = s[0][1][1] = 0.0;
        const double *pb = Ls + t * LD_T + c0 + g;
#pragma unroll
        for (int ch = 0; ch < 2; ch++) dmma884v(s[0][ch], xd[(4 * ch + t) * 8 + g], pb[(r0 + 4 * ch) * LD_T]);   // k-block rb: the diagonal block of X
        ll_accumulate<1>(s, Ls + t * LD_T + r0 + g + (r0 + 8) * LD_T, pb + (r0 + 8) * LD_T, cb - rb - 1, 8 * LD_T, 8 * LD_T, 4 * LD_T,
                         4 * LD_T, 0, act);
#pragma unroll
        for (int e = 0; e < 2; e++) Ls[(c0 + 2 * t + e) * LD_T + r0 + g] = -(s[0][0][e] + s[0][1][e]);
        __syncwarp();
      }
      if (lane < 8) {
        const int i = lane, r = r0 + i;
        double x[8];
#pragma unroll
        for (int c = 0; c < 8; c++) x[c] = (cb == rb) ? ((c == i) ? 1.0 : 0.0) : Ls[(c0 + c) * LD_T + r];
        solve_row8(x, dl, inv);
        if (cb == rb) {
#pragma unroll
          for (int c = 0; c < 8; c++) xd[c * 8 + i] = (c >= i) ? x[c] : 0.0;
        } else {
#pragma unroll
          for (int c = 0; c < 8; c++) Ls[(c0 + c) * LD_T + r] = x[c];
        }
      }
      __syncwarp();
    }
  }
  __syncthreads();
  // W[c][r] = X[r][c] for c >= r, zero above: column r of W is row r of X
  for (int idx = tid; idx < TILE * TILE / 2; idx += 256) {
    const int r = idx >> 6, c = 2 * (idx & 63);
    double v[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int cc = c + e;
      v[e] = (cc < r) ? 0.0 : (((cc >> 3) == (r >> 3)) ? XD[(r >> 3) * 64 + (cc & 7) * 8 + (r & 7)] : Ls[cc * LD_T + r]);
    }
    *reinterpret_cast<double2 *>(Wt + c + (long long)r * ld) = make_double2(v[0], v[1]);
  }
}

int panel_trace_fetch(long long *out2048) {
#ifdef GPB_PANEL_TRACE
  return cudaMemcpyFromSymbol(out2048, g_panel_trace, sizeof(long long) * 2048) == cudaSuccess ? 0 : -1000;
#else
  (void)out2048;
  return -1;
#endif
}

int panel_smem_setup(Handle *h) {
  GPB_CUDA(h, cudaFuncSetAttribute(trsm_tiles_pipelined_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TRSM_PIPE_SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(trsm_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TRSM_SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(tile_inverse_ll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TINV_SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(potrf_tile_pw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF_PW_SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(trsm_ll_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, TrsmLL<1>::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(trsm_ll_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TrsmLL<2>::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(panel_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PANEL_FUSED_SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(panel_fused_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PANEL_FUSED_TILE_SMEM_BYTES));
  return 0;
}

int launch_potrf_tile_at(Handle *h, double *L, long long ld, long long stride, long long diag_off, int index_base,
                         int n, int batch, int *info) {
  ProfScope ps__(h, PC_POTRF);
  potrf_tile_pw_kernel<<<batch, POTRF_PW_THREADS, POTRF_PW_SMEM_BYTES, h->stream>>>(L, ld, stride, diag_off, index_base, n, info);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_potrf_tile(Handle *h, double *L, long long ld, long long stride, int tile_idx, int n, int batch, int *info) {
  return launch_potrf_tile_at(h, L, ld, stride, (long long)tile_idx * TILE * (ld + 1), tile_idx * TILE, n, batch, info);
}

// X = C L^-T for `ntiles` consecutive 128-row tiles starting at element offset c_off (tile step = 128
// rows), against the diagonal tile at element offset diag_off.
int launch_trsm_tiles_at(Handle *h, double *L, long long ld, long long stride, long long diag_off, long long c_off,
                         int ntiles, int batch, TrsmEnv env) {
  if (ntiles <= 0) return 0;
  const long long total = (long long)ntiles * batch;
  ProfScope ps__(h, PC_TRSM);
  // Few tiles (one large matrix, batch 1..2: the latency path): the row-split left-looking kernel, 32 or 64 rows per
  // CTA, so that one block column covers the GPU in a single wave.  Otherwise the register-tile DMMA-throughput
  // kernels: one tile per CTA, or several row tiles per CTA pipelined when there are many.
  if (total * 4 <= 148) {
    dim3 grid(ntiles * 4, batch);
    trsm_ll_kernel<1><<<grid, 128, TrsmLL<1>::SMEM_BYTES, h->stream>>>(L, L, ld, stride, diag_off, c_off);
  } else if (total * 2 <= 148) {
    dim3 grid(ntiles * 2, batch);
    trsm_ll_kernel<2><<<grid, 128, TrsmLL<2>::SMEM_BYTES, h->stream>>>(L, L, ld, stride, diag_off, c_off);
  } else {
    // (an eight-warp, whole-tile form of the left-looking kernel was measured for this regime too: 611 us against 503 for
    // 128 x 31 tiles -- with the C tile in shared memory the DMMA operands cost two shared-memory loads each, where the
    // register-tile kernels feed A from registers; those stay for batches)
    // With an envelope a block column has a few live row tiles per item (N = 4096, bench.py's draws: 176 of 496 per
    // item), and two rows per CTA measured best there (B200, 1000 W, TRSM class per call: 7.52 ms with 2, 7.72 with
    // 4 -- what the dense count picks -- 7.57 with 1).
    const int tpc = env.F ? 2 : (total >= 148 * 16 ? 4 : (total >= 148 * 6 ? 2 : 1));
    if (tpc == 1 || h->trsm_pipelined == 0) {
      dim3 grid(ntiles, batch);
      trsm_tile_kernel<<<grid, 256, TRSM_SMEM_BYTES, h->stream>>>(L, L, ld, stride, diag_off, c_off, env);
    } else {
      dim3 grid((ntiles + tpc - 1) / tpc, batch);
      trsm_tiles_pipelined_kernel<2><<<grid, 256, TRSM_PIPE_SMEM_BYTES, h->stream>>>(L, L, ld, stride, diag_off, c_off, ntiles, tpc, env);
    }
  }
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_trsm_tiles(Handle *h, double *L, long long ld, long long stride, int tile_col, int ntiles_below, int batch) {
  return launch_trsm_tiles_at(h, L, ld, stride, (long long)tile_col * TILE * (ld + 1),
                              (long long)(tile_col + 1) * TILE + (long long)tile_col * TILE * ld, ntiles_below, batch);
}

int launch_potrf_trsm_at(Handle *h, double *L, long long ld, long long stride, long long diag_off, int index_base, int n,
                         long long c_off, int ntiles, int batch, int *info, TrsmEnv env) {
  // one launch when the diagonal CTAs and the 64-row (or 128-row) TRSM CTAs of all matrices fit one wave at one CTA per SM
  const bool fused = h->panel_fused && ntiles > 0 && batch <= PANEL_FUSED_MAX_BATCH;
  if (fused && (long long)batch * (1 + 2 * ntiles) <= 148) {
    ProfScope ps__(h, PC_POTRF);
    const int chunks = ntiles * 2;
    panel_fused_kernel<<<batch * (1 + chunks), PANEL_FUSED_THREADS, PANEL_FUSED_SMEM_BYTES, h->stream>>>(
        L, ld, stride, diag_off, c_off, chunks, batch, index_base, n, info, h->panel_flags);
    GPB_LAUNCH_CHECK(h);
    return 0;
  }
  if (fused && (long long)batch * (1 + ntiles) <= 148) {
    ProfScope ps__(h, PC_POTRF);
    panel_fused_tile_kernel<<<batch * (1 + ntiles), POTRF_PW_THREADS + 32, PANEL_FUSED_TILE_SMEM_BYTES, h->stream>>>(
        L, ld, stride, diag_off, c_off, ntiles, batch, index_base, n, info, h->panel_flags);
    GPB_LAUNCH_CHECK(h);
    return 0;
  }
  int rc = launch_potrf_tile_at(h, L, ld, stride, diag_off, index_base, n, batch, info);
  if (rc) return rc;
  return launch_trsm_tiles_at(h, L, ld, stride, diag_off, c_off, ntiles, batch, env);
}

int launch_potrf_trsm(Handle *h, double *L, long long ld, long long stride, int tile_col, int ntiles_below, int n, int batch,
                      int *info, const int *env) {
  TrsmEnv te;
  if (env) te = TrsmEnv{env + tile_col + 1, env_record_ints((int)(ld / TILE)), tile_col};
  return launch_potrf_trsm_at(h, L, ld, stride, (long long)tile_col * TILE * (ld + 1), tile_col * TILE, n,
                              (long long)(tile_col + 1) * TILE + (long long)tile_col * TILE * ld, ntiles_below, batch, info, te);
}

// inverse of `ntiles` diagonal tiles: L tiles at l_off + t*l_step, W tiles at w_off + t*w_step
int launch_tile_inverse_at(Handle *h, const double *L, long long ld, long long l_off, long long l_step, double *W,
                           long long w_off, long long w_step, long long stride, int ntiles, int batch) {
  dim3 grid(ntiles, batch);
  ProfScope ps__(h, PC_TRSM);
  tile_inverse_ll_kernel<<<grid, 256, TINV_SMEM_BYTES, h->stream>>>(L, W, ld, stride, l_off, l_step, w_off, w_step);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

int launch_tile_inverse(Handle *h, const double *L, double *W, long long ld, long long stride, int ntiles, int batch) {
  const long long step = (long long)TILE * (ld + 1);
  return launch_tile_inverse_at(h, L, ld, 0, step, W, 0, step, stride, ntiles, batch);
}

}  // namespace gpb
