// Batched FP64 tensor-core (DMMA) tile GEMM for sm_100a.
//
// One CTA (or a pair of column-half CTAs) computes one 128x128 output tile of one matrix of the batch
// from a task list (blockIdx.x = task * NSPLIT + half, blockIdx.y = batch item).  The contraction
// streams 16-wide k-chunks of both operands through a cp.async (LDGSTS) pipeline into padded shared
// memory; fragments are read conflict-free (leading dimensions == 4 mod 16 doubles) and fed to
// mma.sync.aligned.m8n8k4.f64 (SASS DMMA.8x8x4 -- tcgen05 has no FP64 kind, so this IS the FP64
// tensor path on B200; measured peak 37.0 TFLOP/s, profiles/fp64_peak_r01.json).
//
// The mma is used "transposed" (mma rows <-> n, mma cols <-> m) so that each thread's two
// accumulator values are adjacent in the column-major output: 16-byte global accesses.
//
// This kernel carries every O(N^3) stage of the path:
//   NT  C = C0 - A B^T          left-looking Cholesky block-column update (replaces the inside of
//                               Eigen LLT under cholesky_decompose, fit_hyperparameters.stan:25)
//   TT  S^T = L21^T W22^T  and  TN  W21 = -S W11     recursive triangular inverse (K^-1 for the gradient)
//   TN  G = W^T W  + fused trace epilogue  0.5 tr((a a^T - K^-1) dK/dtheta)  (the reverse sweep
//                               of multi_normal_cholesky -> cholesky_decompose -> cov_exp_quad), for the
//                               SE kernel and for the joint derivative-observation kernels
//   NN                          products of the forward-mode tangent and of mvrnorm
#include <algorithm>
#include <utility>

#include "common.cuh"
#include "fastexp.cuh"

namespace gpb {

#ifndef GPB_DEFAULT_CFG
#define GPB_DEFAULT_CFG 2
#endif
constexpr int KC = 16;
// Two configurations of the same kernel are built (gpb200_set_gemm_config; 2 is the default):
//   1 Big    128x128 CTA tile, 2x4 warps of 64x32, 4 stages, 1 CTA/SM (the first design, kept as the baseline)
//   2 Half8  128x64 CTA tile, 4x2 warps of 32x32, 3 stages, 2 CTAs/SM
// With one CTA per SM every per-chunk barrier, prologue and epilogue is a bubble in the DMMA pipe
// (91.5 % active, profiles/ncu_summary_r01b.md).  Two independent half-tile CTAs per SM cover each
// other's bubbles (95 %), and with 32x32 warp tiles each sub-partition still has two warps of the other
// CTA to draw DMMAs from while one CTA sits in a barrier or in its epilogue (a 2x2-warp half tile of 64x32
// warp tiles reached 96 % on the Cholesky update but only 91 % on LAUUM + trace).  Splitting the tile along n
// also makes the zero half of a triangular B operand tile skippable for a whole CTA; per-warp skipping inside
// a CTA (a 16-warp 128x128 configuration, round-1 history) cost more than it saved and is gone.
template <int WARPS_M_, int WARPS_N_, int TN_ = TILE, int STAGES_ = 4, int MINB_ = 1, int TM_ = TILE>
struct GemmCfg {
  static constexpr int WARPS_M = WARPS_M_, WARPS_N = WARPS_N_;  // warp grid over the TM x TN CTA tile
  static constexpr int TM = TM_, TN = TN_;                      // CTA tile extents in m and n
  static constexpr int NSPLIT_M = TILE / TM_, NSPLIT_N = TILE / TN_;
  static constexpr int NSPLIT = NSPLIT_M * NSPLIT_N;            // CTAs per 128x128 task
  static constexpr int WM = TM_ / WARPS_M_, WN = TN_ / WARPS_N_;  // warp tile
  static constexpr int MI = WM / 8, NI = WN / 8;                // 8x8 mma tiles per warp
  static constexpr int NTHREADS = 32 * WARPS_M_ * WARPS_N_;
  static constexpr int NCOPY_A = KC * TM_ / 2 / NTHREADS;       // 16-byte copies per thread per stage
  static constexpr int NCOPY_B = KC * TN_ / 2 / NTHREADS;
  static constexpr int STAGES = STAGES_, MINB = MINB_;
  static constexpr int LD_MC_A = TM_ + 4;                       // A stage with m contiguous: [KC][TM+4]
  static constexpr int LD_MC_B = TN_ + 4;                       // B stage with n contiguous: [KC][TN+4]
  static constexpr int STAGE_A = TM_ * (KC + 4);                // >= KC * (TM + 4)
  static constexpr int STAGE_B = TN_ * (KC + 4);                // >= KC * (TN + 4)
  static constexpr int SMEM_BYTES = STAGES_ * (STAGE_A + STAGE_B) * (int)sizeof(double);
};
using CfgBig = GemmCfg<2, 4>;
using CfgHalf8 = GemmCfg<4, 2, 64, 3, 2>;
// 3 Quarter: 64x64 CTA tile, 2x2 warps of 32x32, 3 stages, 3 CTAs/SM.  Four CTAs per 128x128 task: a launch
// with few tasks (one large matrix, batch 1: the latency path) still covers the GPU, the zero half of a triangular
// operand tile is skipped for A as well as for B, and the redundant upper-right quadrant of a symmetric diagonal
// tile is not computed at all (its CTA exits).
using CfgQuarter = GemmCfg<2, 2, 64, 3, 3, 64>;
// 4 Fine: the quarter tile on sixteen warps of 16x16 (one CTA per SM).  A 32x32 warp tile issues 64 DMMAs per 16-wide
// k-chunk, about 1 050 cycles on its scheduler: a K = 128 update on the Cholesky's dependent chain is bound by that issue
// rate, not by the SM's FP64 pipe.  Four times the warps, a quarter of the DMMAs each.  AXPBY epilogue, NT / TN / TT layouts (Cholesky chain, recursive inverse).
using CfgFine = GemmCfg<4, 4, 64, 3, 1, 64>;
constexpr int LD_KC = KC + 4;    // operand with k contiguous:             stage[128][20]
constexpr int EPI_SCRATCH_DOUBLES = 4 * TILE + 5 * 16 + 8;
static_assert(EPI_SCRATCH_DOUBLES * 8 <= CfgHalf8::SMEM_BYTES, "epilogue scratch must fit the pipeline buffers");
static_assert(EPI_SCRATCH_DOUBLES * 8 <= CfgQuarter::SMEM_BYTES, "epilogue scratch must fit the pipeline buffers");
static_assert((CfgHalf8::LD_MC_B % 16) == 4 && (CfgBig::LD_MC_A % 16) == 4 && (CfgQuarter::LD_MC_A % 16) == 4 && (LD_KC % 16) == 4, "conflict-free fragment loads");

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(c[0]), "+d"(c[1])
      : "d"(a), "d"(b));
}

template <class Cfg, bool A_KC, bool B_KC, int EPI>
__global__ void __launch_bounds__(Cfg::NTHREADS, Cfg::MINB) gemm_tile_kernel(const GemmParams p) {
  constexpr int WARPS_N = Cfg::WARPS_N, WM = Cfg::WM, WN = Cfg::WN, MI = Cfg::MI, NI = Cfg::NI;
  constexpr int NTHREADS = Cfg::NTHREADS, NCOPY_A = Cfg::NCOPY_A, NCOPY_B = Cfg::NCOPY_B;
  constexpr int STAGES = Cfg::STAGES, TN = Cfg::TN, LD_MC_B = Cfg::LD_MC_B;
  constexpr int STAGE_DOUBLES = Cfg::STAGE_A, STAGE_PAIR = Cfg::STAGE_A + Cfg::STAGE_B;
  extern __shared__ __align__(16) double smem[];
  constexpr int TM = Cfg::TM, LD_MC = Cfg::LD_MC_A;
  TileTask task = p.tasks[blockIdx.x / Cfg::NSPLIT];
  // the half of the item's envelope this launch uses (F for ENV_CHOL, E for ENV_BAND), read beside the task rather
  // than after it: on the dependent chain of the look-ahead Cholesky a second dependent load is a visible latency
  __shared__ int s_env[ENV_MAX_NT];
  if (p.env_mode != ENV_NONE) {
    const int *src = p.env + (long long)blockIdx.y * 2 * p.env_nt + (p.env_mode == ENV_CHOL ? 0 : p.env_nt);
    for (int q = threadIdx.x; q < p.env_nt; q += Cfg::NTHREADS) s_env[q] = src[q];
    __syncthreads();
  }
  const int split = (Cfg::NSPLIT > 1) ? (int)(blockIdx.x % Cfg::NSPLIT) : 0;
  const int m0 = (Cfg::NSPLIT_M > 1) ? (split / Cfg::NSPLIT_N) * TM : 0;
  const int n0 = (Cfg::NSPLIT_N > 1) ? (split % Cfg::NSPLIT_N) * TN : 0;
  // symmetric diagonal tile: the upper-right quadrant mirrors the lower-left one and no consumer reads it
  const bool sym_skip = Cfg::NSPLIT_M > 1 && (task.flags & TF_DIAG) && m0 < n0;
  if (Cfg::NSPLIT > 1) {  // this CTA owns rows [m0, m0 + TM) x columns [n0, n0 + TN) of the task's 128x128 tile
    if (A_KC) task.a_c += m0; else task.a_r += m0;
    if (B_KC) task.b_c += n0; else task.b_r += n0;
    task.c_r += m0;
    task.c_c += n0;
    // A triangular operand tile is all zero over half of its k-range for one of the two halves: that CTA
    // simply contracts over 64 fewer k (uniform for the whole CTA).
    const bool skip_first = (Cfg::NSPLIT_N > 1 && (task.flags & TF_B_TRI_FIRST) && n0 >= TILE / 2) ||  // zero where k_local < n_local
                            (Cfg::NSPLIT_M > 1 && (task.flags & TF_A_TRI_FIRST) && m0 >= TILE / 2);    // zero where k_local < m_local
    const bool skip_last = (Cfg::NSPLIT_N > 1 && (task.flags & TF_B_TRI_LAST) && n0 < TILE / 2) ||     // zero where k_local > n_local
                           (Cfg::NSPLIT_M > 1 && (task.flags & TF_A_TRI_LAST) && m0 < TILE / 2);       // zero where k_local > m_local
    if (skip_first) {
      if (A_KC) task.a_r += TILE / 2; else task.a_c += TILE / 2;
      if (B_KC) task.b_r += TILE / 2; else task.b_c += TILE / 2;
      task.k_len -= TILE / 2;
    }
    if (skip_last) task.k_len -= TILE / 2;
    if (sym_skip) task.k_len = 0;
  }
  const long long b = blockIdx.y;
  if (p.env_mode != ENV_NONE) {  // the item's tile envelope: leave out the contraction over exactly-zero operand tiles
    const int *F = s_env, *E = s_env;
    const int ti = task.c_r / TILE, tj = task.c_c / TILE;
    int k0 = A_KC ? task.a_r : task.a_c, k1 = k0 + task.k_len;
    bool out;
    if (p.env_mode == ENV_CHOL) {
      out = tj < F[ti];
      k0 = max(k0, max(F[ti], F[tj]) * TILE);
    } else {
      out = ti > E[tj];
      k1 = min(k1, (E[tj] + 1) * TILE);
    }
    const int shift = k0 - (A_KC ? task.a_r : task.a_c);
    if (A_KC) task.a_r += shift; else task.a_c += shift;
    if (B_KC) task.b_r += shift; else task.b_c += shift;
    task.k_len = max(k1 - k0, 0);
    // an update of the factor in place with nothing left to add leaves C as it is
    if (out || (p.env_mode == ENV_CHOL && task.k_len == 0)) {
      if (EPI != EPI_AXPBY && threadIdx.x < (EPI == EPI_TRACE_DERIV ? 8 : 4))
        p.partial[((long long)b * gridDim.x + blockIdx.x) * (EPI == EPI_TRACE_DERIV ? 8 : 4) + threadIdx.x] = 0.0;
      return;
    }
  }
  if (p.flops && threadIdx.x == 0 && task.k_len > 0) atomicAdd(p.flops, 2ull * TM * TN * (unsigned long long)task.k_len);
  const double *__restrict__ A = p.A.p + b * p.A.stride;
  const double *__restrict__ Bm = p.B.p + b * p.B.stride;
  const long long lda = p.A.ld, ldb = p.B.ld;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  // Warp -> sub-tile map: a Latin square over (warp % WARPS_N, warp / WARPS_N), so that the two warps a
  // sub-partition (warp % 4) holds of this CTA sit in different column bands (measured 0.5 % faster than the
  // plain row-major map on the N=4096 step).
  const int wm = (warp / WARPS_N) * WM, wn = (((warp % WARPS_N) + (warp / WARPS_N)) % WARPS_N) * WN;

  double acc[NI][MI][2];
#pragma unroll
  for (int ni = 0; ni < NI; ni++)
#pragma unroll
    for (int mi = 0; mi < MI; mi++) acc[ni][mi][0] = acc[ni][mi][1] = 0.0;

  const int nk = task.k_len / KC;

  // per-thread copy descriptors: NCOPY_A x 16B for A and NCOPY_B x 16B for B per stage
  const double *srcA[NCOPY_A], *srcB[NCOPY_B];
  int dstA[NCOPY_A], dstB[NCOPY_B];
#pragma unroll
  for (int r = 0; r < NCOPY_A; r++) {
    const int idx = tid + NTHREADS * r;
    if (!A_KC) {
      const int k = idx / (TM / 2), m2 = idx % (TM / 2);
      srcA[r] = A + (task.a_r + 2 * m2) + (long long)(task.a_c + k) * lda;
      dstA[r] = k * LD_MC + 2 * m2;
    } else {
      const int m = idx >> 3, k2 = idx & 7;
      srcA[r] = A + (task.a_r + 2 * k2) + (long long)(task.a_c + m) * lda;
      dstA[r] = m * LD_KC + 2 * k2;
    }
  }
#pragma unroll
  for (int r = 0; r < NCOPY_B; r++) {
    const int idx = tid + NTHREADS * r;
    if (!B_KC) {
      const int k = idx / (TN / 2), n2 = idx % (TN / 2);
      srcB[r] = Bm + (task.b_r + 2 * n2) + (long long)(task.b_c + k) * ldb;
      dstB[r] = k * LD_MC_B + 2 * n2;
    } else {
      const int n = idx >> 3, k2 = idx & 7;
      srcB[r] = Bm + (task.b_r + 2 * k2) + (long long)(task.b_c + n) * ldb;
      dstB[r] = n * LD_KC + 2 * k2;
    }
  }
  const long long stepA = A_KC ? (long long)KC : (long long)KC * lda;
  const long long stepB = B_KC ? (long long)KC : (long long)KC * ldb;

  // The source addresses are recomputed from constant bases for every chunk: incrementing the
  // registers an in-flight LDGSTS still reads costs a long-scoreboard (WAR) stall per chunk.
  auto load_stage = [&](int stage, int chunk) {
    double *sA = smem + stage * STAGE_PAIR;
    double *sB = sA + STAGE_DOUBLES;
    const long long offA = (long long)chunk * stepA, offB = (long long)chunk * stepB;
#pragma unroll
    for (int r = 0; r < NCOPY_A; r++) cp_async16(sA + dstA[r], srcA[r] + offA);
#pragma unroll
    for (int r = 0; r < NCOPY_B; r++) cp_async16(sB + dstB[r], srcB[r] + offB);
  };
  auto load_frags = [&](const double *sA, const double *sB, int kk, double (&af)[MI], double (&bf)[NI]) {
#pragma unroll
    for (int mi = 0; mi < MI; mi++)
      af[mi] = A_KC ? sA[(wm + mi * 8 + g) * LD_KC + kk * 4 + t] : sA[(kk * 4 + t) * LD_MC + wm + mi * 8 + g];
#pragma unroll
    for (int ni = 0; ni < NI; ni++)
      bf[ni] = B_KC ? sB[(wn + ni * 8 + g) * LD_KC + kk * 4 + t] : sB[(kk * 4 + t) * LD_MC_B + wn + ni * 8 + g];
  };

  // prologue: all STAGES stages in flight, wait for chunk 0, first fragments in registers
#pragma unroll
  for (int s = 0; s < STAGES; s++) {
    if (s < nk) load_stage(s, s);
    cp_async_commit();
  }
  cp_async_wait<STAGES - 1>();
  __syncthreads();
  double af[2][MI], bf[2][NI];
  load_frags(smem, smem + STAGE_DOUBLES, 0, af[0], bf[0]);

  for (int kc = 0; kc < nk; kc++) {
    const double *sA = smem + (kc % STAGES) * STAGE_PAIR;
    const double *sB = sA + STAGE_DOUBLES;
#pragma unroll
    for (int kk = 0; kk < KC / 4; kk++) {
      const int cur = kk & 1, nxt = cur ^ 1;
      if (kk < KC / 4 - 1) {
        load_frags(sA, sB, kk + 1, af[nxt], bf[nxt]);
      } else {
        // Chunk transition, hidden behind the DMMAs of this last k-step: everybody has finished
        // reading stage kc (its last fragments are in registers), chunk kc+1 has landed.
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        if (kc + STAGES < nk) load_stage(kc % STAGES, kc + STAGES);
        cp_async_commit();
        if (kc + 1 < nk) {
          const double *nA = smem + ((kc + 1) % STAGES) * STAGE_PAIR;
          load_frags(nA, nA + STAGE_DOUBLES, 0, af[nxt], bf[nxt]);
        }
      }
#pragma unroll
      for (int ni = 0; ni < NI; ni++)
#pragma unroll
        for (int mi = 0; mi < MI; mi++) dmma884(acc[ni][mi], bf[cur][ni], af[cur][mi]);
    }
  }
  cp_async_wait<0>();

  if (sym_skip) {  // uniform for the CTA
    if (EPI != EPI_AXPBY && tid < (EPI == EPI_TRACE_DERIV ? 8 : 4))
      p.partial[((long long)b * gridDim.x + blockIdx.x) * (EPI == EPI_TRACE_DERIV ? 8 : 4) + tid] = 0.0;
    return;
  }
  if (EPI == EPI_AXPBY) {
    double *__restrict__ C = p.C.p + b * p.C.stride;
    const double *__restrict__ C0 = p.C0.p ? p.C0.p + b * p.C0.stride : nullptr;
    const double alpha = p.alpha, beta = p.beta;
#pragma unroll
    for (int ni = 0; ni < NI; ni++) {
      const int n = task.c_c + wn + ni * 8 + g;
#pragma unroll
      for (int mi = 0; mi < MI; mi++) {
        const int m = task.c_r + wm + mi * 8 + 2 * t;
        double2 v = make_double2(alpha * acc[ni][mi][0], alpha * acc[ni][mi][1]);
        if (C0) {
          const double2 c0 = *reinterpret_cast<const double2 *>(C0 + m + (long long)n * p.C0.ld);
          v.x = fma(beta, c0.x, v.x);
          v.y = fma(beta, c0.y, v.y);
        }
        *reinterpret_cast<double2 *>(C + m + (long long)n * p.C.ld) = v;
        if (p.CT.p) {
          double *CT = p.CT.p + b * p.CT.stride + n;
          CT[(long long)m * p.CT.ld] = v.x;
          CT[(long long)(m + 1) * p.CT.ld] = v.y;
        }
      }
    }
  } else if (EPI == EPI_TRACE_DERIV) {
    // ---- fused trace epilogue for the joint derivative-observation covariance -------------------
    // K[I,J] = alpha^2 k_pq(t_i - t_j) (+ diagonal), p / q the derivative orders of row / column block:
    //   k_pq(d)      = (-1)^p He_m(u) l^-m e,  m = p + q, u = d / l, e = exp(-u^2 / 2)
    //   d k_pq / d l = (-1)^p l^-(m+1) e (He_{m+2}(u) + He_m(u))
    // (He = probabilists' Hermite polynomials; restates derivative_kernels.R:39-73 -- checked against
    // those nine closed forms in tests/).  Partials per tile: sum M k, sum M dk/dl, tr G per block.
    __syncthreads();
    double *xr = smem, *xc = smem + TILE, *ar = smem + 2 * TILE, *ac = smem + 3 * TILE;
    double *red = smem + 4 * TILE;
    const int ng = p.n_grid;
    const double *x = p.x + b * p.x_stride;
    const double *av = p.avec + b * p.a_stride;
    for (int q = tid; q < TM + TN; q += NTHREADS) {
      const bool row = q < TM;
      const int ql = row ? q : q - TM;
      const int i = (row ? task.c_r : task.c_c) + ql;
      const int gi = i - (i >= ng ? ng : 0) - (i >= 2 * ng ? ng : 0);
      (row ? xr : xc)[ql] = (i < p.n) ? x[gi] : 0.0;
      (row ? ar : ac)[ql] = (i < p.n) ? av[i] : 0.0;
    }
    __syncthreads();
    const double l = p.theta[b * p.theta_stride + 1];
    const double il = 1.0 / l;
    const bool diag_tile = (task.flags & 1) != 0;
    double s_k = 0.0, s_dk = 0.0, s_tr[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int ni = 0; ni < NI; ni++) {
      const int nl = wn + ni * 8 + g;
      const int j = task.c_c + nl;
      const int bj = (j >= ng) + (j >= 2 * ng);
#pragma unroll
      for (int mi = 0; mi < MI; mi++) {
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int ml = wm + mi * 8 + 2 * t + e;
          const int i = task.c_r + ml;
          const double G = acc[ni][mi][e];
          if (i < p.n && j < p.n) {
            const int bi = (i >= ng) + (i >= 2 * ng);
            const int pi = p.order0 + bi, m = pi + p.order0 + bj;
            const double u = (xr[ml] - xc[nl]) * il;
            const double ek = exp_nonpos(-0.5 * u * u);
            double hp = 0.0, hc = 1.0, lp = 1.0, hm = 1.0, lm = 1.0, hm2 = 0.0;
#pragma unroll
            for (int k = 1; k <= 6; k++) {
              const double hn = u * hc - (double)(k - 1) * hp;
              hp = hc; hc = hn; lp *= il;
              if (k == m) { hm = hc; lm = lp; }
              if (k == m + 2) hm2 = hc;
            }
            const double sg = (pi & 1) ? -ek : ek;
            const double M = ar[ml] * ac[nl] - G;
            s_k += M * (sg * hm * lm);
            s_dk += M * (sg * lm * il * (hm2 + hm));
            if (diag_tile && i == j) {
              if (bi == 0) s_tr[0] += G; else if (bi == 1) s_tr[1] += G; else s_tr[2] += G;
            }
          }
        }
      }
    }
    const double w = ((task.flags & TF_FULL_WEIGHT) || (diag_tile && (Cfg::NSPLIT_M == 1 || m0 == n0))) ? 1.0 : 2.0;  // a diagonal quadrant / full diagonal tile holds both (i,j) and (j,i)
    s_k *= w;
    s_dk *= w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s_k += __shfl_xor_sync(0xffffffffu, s_k, o);
      s_dk += __shfl_xor_sync(0xffffffffu, s_dk, o);
#pragma unroll
      for (int q = 0; q < 3; q++) s_tr[q] += __shfl_xor_sync(0xffffffffu, s_tr[q], o);
    }
    if (lane == 0) {
      red[warp * 5 + 0] = s_k;
      red[warp * 5 + 1] = s_dk;
      red[warp * 5 + 2] = s_tr[0];
      red[warp * 5 + 3] = s_tr[1];
      red[warp * 5 + 4] = s_tr[2];
    }
    __syncthreads();
    if (tid < 5) {
      double r = 0.0;
      for (int w8 = 0; w8 < NTHREADS / 32; w8++) r += red[w8 * 5 + tid];
      p.partial[((long long)b * gridDim.x + blockIdx.x) * 8 + tid] = r;
    }
  } else {
    // ---- fused trace epilogue: this tile of G = K^-1 never has to reach HBM -----------------
    __syncthreads();  // everyone is done with the pipeline buffers
    double *xr = smem, *xc = smem + TILE, *ar = smem + 2 * TILE, *ac = smem + 3 * TILE;
    double *red = smem + 4 * TILE;
    const double *x = p.x + b * p.x_stride;
    const double *av = p.avec + b * p.a_stride;
    for (int q = tid; q < TM + TN; q += NTHREADS) {
      const bool row = q < TM;
      const int ql = row ? q : q - TM;
      const int i = (row ? task.c_r : task.c_c) + ql;
      (row ? xr : xc)[ql] = (i < p.n) ? x[i] : 0.0;
      (row ? ar : ac)[ql] = (i < p.n) ? av[i] : 0.0;
    }
    __syncthreads();
    const double rho = p.theta[b * 3 + 1];
    const double nh = -0.5 / (rho * rho);
    const bool diag_tile = (task.flags & 1) != 0;
    double s_se = 0.0, s_d2 = 0.0, s_tr = 0.0;
    double *__restrict__ C = p.C.p ? p.C.p + b * p.C.stride : nullptr;
#pragma unroll
    for (int ni = 0; ni < NI; ni++) {
      const int nl = wn + ni * 8 + g;
      const int j = task.c_c + nl;
#pragma unroll
      for (int mi = 0; mi < MI; mi++) {
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int ml = wm + mi * 8 + 2 * t + e;
          const int i = task.c_r + ml;
          const double G = acc[ni][mi][e];
          if (i < p.n && j < p.n) {
            const double d = xr[ml] - xc[nl];
            const double d2 = d * d;
            const double ek = exp_nonpos(d2 * nh);
            const double M = ar[ml] * ac[nl] - G;
            s_se += M * ek;
            s_d2 += M * ek * d2;
            if (diag_tile && i == j) s_tr += G;
          }
        }
        if (C) {
          const int m = task.c_r + wm + mi * 8 + 2 * t;
          *reinterpret_cast<double2 *>(C + m + (long long)j * p.C.ld) =
              make_double2(acc[ni][mi][0], acc[ni][mi][1]);
        }
      }
    }
    const double w = ((task.flags & TF_FULL_WEIGHT) || (diag_tile && (Cfg::NSPLIT_M == 1 || m0 == n0))) ? 1.0 : 2.0;  // a diagonal quadrant / full diagonal tile holds both (i,j) and (j,i)
    s_se *= w;
    s_d2 *= w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s_se += __shfl_xor_sync(0xffffffffu, s_se, o);
      s_d2 += __shfl_xor_sync(0xffffffffu, s_d2, o);
      s_tr += __shfl_xor_sync(0xffffffffu, s_tr, o);
    }
    if (lane == 0) {
      red[warp * 3 + 0] = s_se;
      red[warp * 3 + 1] = s_d2;
      red[warp * 3 + 2] = s_tr;
    }
    __syncthreads();
    if (tid == 0) {
      double r0 = 0, r1 = 0, r2 = 0;
      for (int w8 = 0; w8 < NTHREADS / 32; w8++) {
        r0 += red[w8 * 3 + 0];
        r1 += red[w8 * 3 + 1];
        r2 += red[w8 * 3 + 2];
      }
      double *o = p.partial + ((long long)b * gridDim.x + blockIdx.x) * 4;
      o[0] = r0;
      o[1] = r1;
      o[2] = r2;
      o[3] = 0.0;
    }
  }
}

template <class Cfg, bool A_KC, bool B_KC, int EPI>
static int launch_one(Handle *h, const GemmParams &p, int ntasks, int batch) {
  auto kern = gemm_tile_kernel<Cfg, A_KC, B_KC, EPI>;
  dim3 grid(ntasks * Cfg::NSPLIT, batch);
  ProfScope ps__(h, PC_GEMM);
  kern<<<grid, Cfg::NTHREADS, Cfg::SMEM_BYTES, h->stream>>>(p);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

template <class Cfg>
static int smem_setup_cfg(Handle *h) {
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<Cfg, false, false, EPI_AXPBY>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<Cfg, true, true, EPI_AXPBY>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<Cfg, false, true, EPI_AXPBY>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<Cfg, true, false, EPI_AXPBY>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<Cfg, true, true, EPI_TRACE>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<Cfg, false, false, EPI_TRACE>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<Cfg, true, true, EPI_TRACE_DERIV>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  return 0;
}

// The opt-in to > 48 KB of dynamic shared memory is a per-device function attribute: it is set when a
// handle is created (gpb200_create), once per handle, so one process may hold handles on several GPUs.
int gemm_smem_setup(Handle *h) {
  int rc = smem_setup_cfg<CfgBig>(h);
  if (!rc) rc = smem_setup_cfg<CfgHalf8>(h);
  if (!rc) rc = smem_setup_cfg<CfgQuarter>(h);
  if (rc) return rc;
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<CfgFine, false, false, EPI_AXPBY>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgFine::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<CfgFine, true, true, EPI_AXPBY>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgFine::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_tile_kernel<CfgFine, true, false, EPI_AXPBY>, cudaFuncAttributeMaxDynamicSharedMemorySize, CfgFine::SMEM_BYTES));
  return 0;
}

template <class Cfg>
static int launch_cfg(Handle *h, GemmLayout layout, GemmEpi epi, const GemmParams &p, int ntasks, int batch) {
  if (epi == EPI_AXPBY) {
    switch (layout) {
      case LAYOUT_NT: return launch_one<Cfg, false, false, EPI_AXPBY>(h, p, ntasks, batch);
      case LAYOUT_TN: return launch_one<Cfg, true, true, EPI_AXPBY>(h, p, ntasks, batch);
      case LAYOUT_NN: return launch_one<Cfg, false, true, EPI_AXPBY>(h, p, ntasks, batch);
      case LAYOUT_TT: return launch_one<Cfg, true, false, EPI_AXPBY>(h, p, ntasks, batch);
    }
  } else if (layout == LAYOUT_TN) {
    if (epi == EPI_TRACE_DERIV) return launch_one<Cfg, true, true, EPI_TRACE_DERIV>(h, p, ntasks, batch);
    return launch_one<Cfg, true, true, EPI_TRACE>(h, p, ntasks, batch);
  } else if (layout == LAYOUT_NT && epi == EPI_TRACE) {
    return launch_one<Cfg, false, false, EPI_TRACE>(h, p, ntasks, batch);  // G = X X^T of the distributed gradient (api_mg.cu)
  }
  snprintf(h->err, sizeof(h->err), "launch_gemm: unsupported layout/epilogue %d/%d", (int)layout, (int)epi);
  return -2;
}

// configuration choice: 1 Big, 2 Half8 (two CTAs per SM; wins or ties at every batched size from N=512 to N=4096,
// profiles/bench_configs_r01.json), 3 Quarter (64x64 CTAs).  Automatic: Quarter while the launch is too small to
// give every SM its two Half8 CTAs (the single-matrix latency path), Half8 otherwise.
int gemm_pick_cfg(const Handle *h, int ntasks, int batch) {
  if (h->gemm_cfg_override) return h->gemm_cfg_override;
  if (GPB_DEFAULT_CFG != 2) return GPB_DEFAULT_CFG;
  return ((long long)ntasks * batch * CfgHalf8::NSPLIT < 2LL * 148 * h->quarter_below_waves) ? 3 : 2;
}

// CTAs per 128x128 task of the configuration launch_gemm will pick for this launch (the trace epilogues write
// one partial record per CTA)
int gemm_nsplit(const Handle *h, int ntasks, int batch) {
  const int c = gemm_pick_cfg(h, ntasks, batch);
  return c == 3 ? CfgQuarter::NSPLIT : (c == 2 ? CfgHalf8::NSPLIT : 1);
}

// Flops a launch really executes: per CTA 2 * TM * TN * k, with k shortened by the CTA-uniform skipping of triangular
// operand tiles and zero for the skipped quadrant of symmetric diagonal tiles -- the same rules as in the kernel.
static double executed_flops_host(const Handle *h, const TileTask *dev_tasks, int ntasks, int batch, int cfg_regular, int cfg_diag) {
  const TileTask *host = nullptr;
  for (const auto &kv : h->task_cache) {
    const TileTask *base = kv.second.first;
    const auto it = h->task_host.find(kv.first);
    if (it == h->task_host.end()) continue;
    if (dev_tasks >= base && dev_tasks < base + it->second.size()) { host = it->second.data() + (dev_tasks - base); break; }
  }
  if (!host) return 0.0;
  double total = 0.0;
  for (int q = 0; q < ntasks; q++) {
    const TileTask &t = host[q];
    const int cfg = (t.flags & TF_DIAG) ? cfg_diag : cfg_regular;
    const int sm = cfg == 3 ? 2 : 1, sn = cfg == 1 ? 1 : 2;   // CTAs per task along m and n
    const int tm = TILE / sm, tn = TILE / sn;
    for (int mh = 0; mh < sm; mh++)
      for (int nh = 0; nh < sn; nh++) {
        if (sm > 1 && (t.flags & TF_DIAG) && mh < nh) continue;
        int k = t.k_len;
        const bool first = (sn > 1 && (t.flags & TF_B_TRI_FIRST) && nh == 1) || (sm > 1 && (t.flags & TF_A_TRI_FIRST) && mh == 1);
        const bool last = (sn > 1 && (t.flags & TF_B_TRI_LAST) && nh == 0) || (sm > 1 && (t.flags & TF_A_TRI_LAST) && mh == 0);
        if (first) k -= TILE / 2;
        if (last) k -= TILE / 2;
        total += 2.0 * tm * tn * (double)std::max(k, 0);
      }
  }
  return total * batch;
}

// Diagonal split (large batches): the symmetric diagonal tiles of a launch -- one per block column of the Cholesky
// update, nt of nt (nt + 1) / 2 in LAUUM -- go to a second launch of 64x64 quarter CTAs, which drop the redundant
// upper-right quadrant and skip the zero half of BOTH triangular operand tiles; everything else stays on the 128x64
// half-tile CTAs (2 % more efficient per executed flop, profiles/bench_r02*.json).  Same stream, back to back.
static bool diag_split_applies(const Handle *h, int ntasks, int batch, int cfg) {
  return h->diag_split && cfg == 2 && batch >= 16 && (long long)ntasks * batch >= 2048;
}

static int get_split(Handle *h, const TileTask *tasks, int ntasks, SplitLists *out) {
  const auto key = std::make_pair(tasks, ntasks);
  auto it = h->split_cache.find(key);
  if (it == h->split_cache.end()) {
    const TileTask *host = nullptr;
    for (const auto &kv : h->task_cache) {
      const TileTask *base = kv.second.first;
      const auto ht = h->task_host.find(kv.first);
      if (ht == h->task_host.end()) continue;
      if (tasks >= base && tasks < base + ht->second.size()) { host = ht->second.data() + (tasks - base); break; }
    }
    SplitLists sl;
    if (host) {
      std::vector<TileTask> reg, diag;
      for (int q = 0; q < ntasks; q++) ((host[q].flags & TF_DIAG) ? diag : reg).push_back(host[q]);
      if (!reg.empty() && !diag.empty()) {
        TileTask *dev = nullptr;
        GPB_CUDA(h, cudaMalloc(&dev, (reg.size() + diag.size()) * sizeof(TileTask)));
        GPB_CUDA(h, cudaMemcpy(dev, reg.data(), reg.size() * sizeof(TileTask), cudaMemcpyHostToDevice));
        GPB_CUDA(h, cudaMemcpy(dev + reg.size(), diag.data(), diag.size() * sizeof(TileTask), cudaMemcpyHostToDevice));
        sl.reg = dev;
        sl.diag = dev + reg.size();
        sl.nreg = (int)reg.size();
        sl.ndiag = (int)diag.size();
      }
    }
    it = h->split_cache.emplace(key, sl).first;
  }
  *out = it->second;
  return 0;
}

int gemm_partial_layout(Handle *h, const TileTask *tasks, int ntasks, int batch, int *n1, int *n2) {
  const int c = gemm_pick_cfg(h, ntasks, batch);
  *n1 = ntasks * (c == 3 ? CfgQuarter::NSPLIT : (c == 2 ? CfgHalf8::NSPLIT : 1));
  *n2 = 0;
  if (diag_split_applies(h, ntasks, batch, c)) {
    SplitLists sl;
    int rc = get_split(h, tasks, ntasks, &sl);
    if (rc) return rc;
    if (sl.ndiag > 0) {
      *n1 = sl.nreg * CfgHalf8::NSPLIT;
      *n2 = sl.ndiag * CfgQuarter::NSPLIT;
    }
  }
  return 0;
}

int launch_gemm(Handle *h, GemmLayout layout, GemmEpi epi, const GemmParams &p_in, int ntasks, int batch) {
  if (ntasks <= 0 || batch <= 0) return 0;
  // which tiles an envelope launch skips is only known on the device: there the CTAs count what they execute
  GemmParams p = p_in;
  const bool count_here = h->count_flops && p.env_mode == ENV_NONE;
  if (h->count_flops && p.env_mode != ENV_NONE) p.flops = h->flops_dev;
  const int c = gemm_pick_cfg(h, ntasks, batch);
  if (diag_split_applies(h, ntasks, batch, c)) {
    SplitLists sl;
    int rc = get_split(h, p.tasks, ntasks, &sl);
    if (rc) return rc;
    if (sl.ndiag > 0) {
      GemmParams pr = p, pd = p;
      pr.tasks = sl.reg;
      pr.ntasks = sl.nreg;
      pd.tasks = sl.diag;
      pd.ntasks = sl.ndiag;
      if (epi != EPI_AXPBY && p.partial) pd.partial = p.partial + (long long)batch * sl.nreg * CfgHalf8::NSPLIT * (epi == EPI_TRACE_DERIV ? 8 : 4);
      if (count_here) h->executed_gemm_flops += executed_flops_host(h, p.tasks, ntasks, batch, 2, 3);
      rc = launch_cfg<CfgHalf8>(h, layout, epi, pr, sl.nreg, batch);
      if (rc) return rc;
      return launch_cfg<CfgQuarter>(h, layout, epi, pd, sl.ndiag, batch);
    }
  }
  if (count_here) h->executed_gemm_flops += executed_flops_host(h, p.tasks, ntasks, batch, c, c);
  if (c == 3 && p.latency_hint && h->fine_cfg && epi == EPI_AXPBY && layout != LAYOUT_NN &&
      (long long)ntasks * batch * CfgFine::NSPLIT <= 148) {
    if (layout == LAYOUT_NT) return launch_one<CfgFine, false, false, EPI_AXPBY>(h, p, ntasks, batch);
    if (layout == LAYOUT_TN) return launch_one<CfgFine, true, true, EPI_AXPBY>(h, p, ntasks, batch);
    return launch_one<CfgFine, true, false, EPI_AXPBY>(h, p, ntasks, batch);
  }
  if (c == 1) return launch_cfg<CfgBig>(h, layout, epi, p, ntasks, batch);
  if (c == 3) return launch_cfg<CfgQuarter>(h, layout, epi, p, ntasks, batch);
  return launch_cfg<CfgHalf8>(h, layout, epi, p, ntasks, batch);
}

}  // namespace gpb
