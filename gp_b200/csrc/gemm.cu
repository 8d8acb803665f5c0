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
//                               SE kernel, for the joint derivative-observation kernels and for the ARD
//                               kernel (gemm_trace_ard_kernel)
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

__device__ __forceinline__ double warp_sum_(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(c[0]), "+d"(c[1])
      : "d"(a), "d"(b));
}

template <class Cfg, bool A_KC, bool B_KC, int EPI>
__global__ void __launch_bounds__(Cfg::NTHREADS, Cfg::MINB) gemm_tile_kernel(const GemmParams p) {
#include "gemm_tile_body.cuh"
}

// TN layout + the ARD trace epilogue (G = W^T W of the LML gradient of gpb200_lml_grad_ard_batched): the main loop
// of gemm_tile_kernel under its own name, so that profiles and SASS reports tell it apart from the tile GEMM proper
template <class Cfg, bool A_KC, bool B_KC, int EPI>
__global__ void __launch_bounds__(Cfg::NTHREADS, Cfg::MINB) gemm_trace_ard_kernel(const GemmParams p) {
  static_assert(A_KC && B_KC && EPI == EPI_TRACE_ARD, "gemm_trace_ard_kernel is the TN layout with the ARD epilogue");
#include "gemm_tile_body.cuh"
}

// TN layout + the SE trace epilogue masked by a per-item size (gpb200_lml_grad_ragged), under its own name as well
template <class Cfg, bool A_KC, bool B_KC, int EPI>
__global__ void __launch_bounds__(Cfg::NTHREADS, Cfg::MINB) gemm_trace_ragged_kernel(const GemmParams p) {
  static_assert(A_KC && B_KC && EPI == EPI_TRACE_RAGGED, "gemm_trace_ragged_kernel is the TN layout with the ragged SE epilogue");
#include "gemm_tile_body.cuh"
}

template <class Cfg, bool A_KC, bool B_KC, int EPI>
static int launch_one(Handle *h, const GemmParams &p, int ntasks, int batch) {
  void (*kern)(const GemmParams);
  if constexpr (EPI == EPI_TRACE_ARD) kern = gemm_trace_ard_kernel<Cfg, A_KC, B_KC, EPI>;
  else if constexpr (EPI == EPI_TRACE_RAGGED) kern = gemm_trace_ragged_kernel<Cfg, A_KC, B_KC, EPI>;
  else kern = gemm_tile_kernel<Cfg, A_KC, B_KC, EPI>;
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
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_trace_ragged_kernel<Cfg, true, true, EPI_TRACE_RAGGED>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  GPB_CUDA(h, cudaFuncSetAttribute(gemm_trace_ard_kernel<Cfg, true, true, EPI_TRACE_ARD>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
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
    if (epi == EPI_TRACE_ARD) return launch_one<Cfg, true, true, EPI_TRACE_ARD>(h, p, ntasks, batch);
    if (epi == EPI_TRACE_RAGGED) return launch_one<Cfg, true, true, EPI_TRACE_RAGGED>(h, p, ntasks, batch);
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
      if (epi != EPI_AXPBY && p.partial) pd.partial = p.partial + (long long)batch * sl.nreg * CfgHalf8::NSPLIT * epi_partial_width(epi);
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
