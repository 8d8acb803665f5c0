// Body of the tile GEMM kernels of gemm.cu (no include guard: it is included once inside each kernel definition,
// where Cfg, A_KC, B_KC, EPI and the parameter block p are in scope).  The kernels share it textually: moving it
// into a __forceinline__ device function called by all of them changes the register allocation of the existing
// gemm_tile_kernel instantiations, and the ARD and ragged epilogues run under their own kernel names.
  constexpr int WARPS_N = Cfg::WARPS_N, WM = Cfg::WM, WN = Cfg::WN, MI = Cfg::MI, NI = Cfg::NI;
  constexpr int NTHREADS = Cfg::NTHREADS, NCOPY_A = Cfg::NCOPY_A, NCOPY_B = Cfg::NCOPY_B;
  constexpr int STAGES = Cfg::STAGES, TN = Cfg::TN, LD_MC_B = Cfg::LD_MC_B;
  constexpr int STAGE_DOUBLES = Cfg::STAGE_A, STAGE_PAIR = Cfg::STAGE_A + Cfg::STAGE_B;
  extern __shared__ __align__(16) double smem[];
  constexpr int TM = Cfg::TM, LD_MC = Cfg::LD_MC_A;
  TileTask task = p.tasks[blockIdx.x / Cfg::NSPLIT];
  // the part of the item's envelope record this launch uses (F for ENV_CHOL, fb for ENV_CHOL_FINE, er for ENV_BAND),
  // read beside the task rather than after it: on the dependent chain of the look-ahead Cholesky a second dependent
  // load is a visible latency
  __shared__ int s_env[2 * ENV_MAX_NT];
  const long long b = p.order ? p.order[blockIdx.y] : blockIdx.y;  // the batch item
  if (p.env_mode != ENV_NONE) {
    const int nt = p.env_nt;
    const int *src = p.env + b * env_record_ints(nt) + (p.env_mode == ENV_CHOL ? 0 : (p.env_mode == ENV_CHOL_FINE ? 2 * nt : 4 * nt));
    const int cnt = p.env_mode == ENV_CHOL_FINE ? 2 * nt : nt;
    for (int q = threadIdx.x; q < cnt; q += Cfg::NTHREADS) s_env[q] = src[q];
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
  if (p.env_mode != ENV_NONE) {  // the item's envelope: leave out the contraction over exactly-zero operand rows
    const int ti = task.c_r / TILE, tj = task.c_c / TILE;
    int k0 = A_KC ? task.a_r : task.a_c, k1 = k0 + task.k_len;
    bool out = false;
    if (p.env_mode == ENV_CHOL) {
      const int *F = s_env;
      out = tj < F[ti];
      k0 = max(k0, max(F[ti], F[tj]) * TILE);
    } else if (p.env_mode == ENV_CHOL_FINE) {
      // A is L(rows of C, :) and B is L(columns of C, :): a CTA whose C block lies left of the profile ends with k_len 0
      const int *fb = s_env;
      int ka = fb[task.c_r / ENV_BLK], kb = fb[task.c_c / ENV_BLK];
      if (TM > ENV_BLK) ka = min(ka, fb[task.c_r / ENV_BLK + 1]);
      if (TN > ENV_BLK) kb = min(kb, fb[task.c_c / ENV_BLK + 1]);
      k0 = max(k0, max(ka, kb) & ~(KC - 1));
    } else {
      const int er = s_env[tj];
      out = ti > er / TILE;
      k1 = min(k1, (er + KC) & ~(KC - 1));
    }
    const int shift = k0 - (A_KC ? task.a_r : task.a_c);
    if (A_KC) task.a_r += shift; else task.a_c += shift;
    if (B_KC) task.b_r += shift; else task.b_c += shift;
    task.k_len = max(k1 - k0, 0);
    // an update of the factor in place with nothing left to add leaves C as it is
    if (out || (p.env_mode != ENV_BAND && task.k_len == 0)) {
      if (EPI != EPI_AXPBY && threadIdx.x < epi_partial_width(EPI))
        p.partial[((long long)b * gridDim.x + blockIdx.x) * epi_partial_width(EPI) + threadIdx.x] = 0.0;
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
    if (EPI != EPI_AXPBY && tid < epi_partial_width(EPI))
      p.partial[((long long)b * gridDim.x + blockIdx.x) * epi_partial_width(EPI) + tid] = 0.0;
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
  } else if (EPI == EPI_TRACE_ARD) {
    // ---- fused trace epilogue for the ARD covariance K = alpha^2 e + c I, e = exp(-0.5 sum_d q_d^2),
    // q_d = (X_id - X_jd) / rho_d.  Partials per CTA: S_e = sum M e, S_d = sum M e q_d^2 (d < D), tr G.
    // The coordinates are staged already divided by rho_d, exactly as gram_ard_batched_kernel divides them.
    __syncthreads();
    constexpr int PW = epi_partial_width(EPI_TRACE_ARD);
    double *qr = smem, *qc = smem + ARD_MAX_D * TILE, *ar = smem + 2 * ARD_MAX_D * TILE, *ac = ar + TILE;
    double *red = ac + TILE;
    const int D = p.ard_d;
    // the task's output origin, flags and the batch item are read again rather than kept live across the main loop
    const TileTask tk = p.tasks[blockIdx.x / Cfg::NSPLIT];
    const int c_r = tk.c_r + m0, c_c = tk.c_c + n0;
    const long long bi = blockIdx.y;
    const double *x = p.x + bi * p.x_stride;
    const double *av = p.avec + bi * p.a_stride;
    const double *th = p.theta + bi * p.theta_stride;
    for (int q = tid; q < TM + TN; q += NTHREADS) {
      const bool row = q < TM;
      const int ql = row ? q : q - TM;
      const int i = (row ? c_r : c_c) + ql;
      for (int d = 0; d < D; d++) (row ? qr : qc)[d * TILE + ql] = (i < p.n) ? x[i + (long long)d * p.n] / th[1 + d] : 0.0;
      (row ? ar : ac)[ql] = (i < p.n) ? av[i] : 0.0;
    }
    __syncthreads();
    const bool diag_tile = (tk.flags & 1) != 0;
    const double w = ((tk.flags & TF_FULL_WEIGHT) || (diag_tile && (Cfg::NSPLIT_M == 1 || m0 == n0))) ? 1.0 : 2.0;  // a diagonal quadrant / full diagonal tile holds both (i,j) and (j,i)
    // Pass 1: S_e and tr G, and M e of every element of the thread parked in shared memory (0 outside the matrix).
    // Pass 2 takes S_d one dimension at a time from there: the tile's accumulators and D + 2 sums together do not fit
    // the 128 registers of the two-CTA half-tile configuration without spilling.
    static_assert(EPI != EPI_TRACE_ARD || (2 * ARD_MAX_D * TILE + 2 * TILE + 8 * PW + TM * TN) * 8 <= Cfg::SMEM_BYTES,
                  "ARD epilogue scratch must fit the pipeline buffers");
    double *me = red + 8 * PW;  // [NI * MI * 2][NTHREADS]
    double s_e = 0.0, s_tr = 0.0;
#pragma unroll
    for (int ni = 0; ni < NI; ni++) {
      const int nl = wn + ni * 8 + g;
      const int j = c_c + nl;
#pragma unroll
      for (int mi = 0; mi < MI; mi++) {
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int ml = wm + mi * 8 + 2 * t + e;
          const int i = c_r + ml;
          const double G = acc[ni][mi][e];
          double Me = 0.0;
          if (i < p.n && j < p.n) {
            double r2 = 0.0;
#pragma unroll
            for (int d = 0; d < ARD_MAX_D; d++)
              if (d < D) {
                const double dq = qr[d * TILE + ml] - qc[d * TILE + nl];
                r2 = fma(dq, dq, r2);
              }
            Me = (ar[ml] * ac[nl] - G) * exp_nonpos(-0.5 * r2);
            if (diag_tile && i == j) s_tr += G;
          }
          s_e += Me;
          me[((ni * MI + mi) * 2 + e) * NTHREADS + tid] = Me;
        }
      }
    }
    s_e = warp_sum_(s_e * w);
    s_tr = warp_sum_(s_tr);
    if (lane == 0) {
      red[warp * PW + 0] = s_e;
      red[warp * PW + PW - 1] = s_tr;
    }
#pragma unroll 1
    for (int d = 0; d < ARD_MAX_D; d++) {
      double s_d = 0.0;
      if (d < D) {  // uniform
        const double *qrd = qr + d * TILE, *qcd = qc + d * TILE;
#pragma unroll
        for (int ni = 0; ni < NI; ni++) {
          const double qn = qcd[wn + ni * 8 + g];
#pragma unroll
          for (int mi = 0; mi < MI; mi++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
              const double dq = qrd[wm + mi * 8 + 2 * t + e] - qn;
              s_d = fma(me[((ni * MI + mi) * 2 + e) * NTHREADS + tid], dq * dq, s_d);
            }
        }
        s_d = warp_sum_(s_d * w);
      }
      if (lane == 0) red[warp * PW + 1 + d] = s_d;
    }
    __syncthreads();
    if (tid < PW) {
      double r = 0.0;
      for (int w8 = 0; w8 < NTHREADS / 32; w8++) r += red[w8 * PW + tid];
      p.partial[(bi * gridDim.x + blockIdx.x) * PW + tid] = r;
    }
  } else {
    // ---- fused trace epilogue: this tile of G = K^-1 never has to reach HBM -----------------
    __syncthreads();  // everyone is done with the pipeline buffers
    double *xr = smem, *xc = smem + TILE, *ar = smem + 2 * TILE, *ac = smem + 3 * TILE;
    double *red = smem + 4 * TILE;
    const double *x = p.x + b * p.x_stride;
    const double *av = p.avec + b * p.a_stride;
    // the item's true size, the mask of its padding (spelled out at each use: a local copy changes the SASS of the
    // uniform EPI_TRACE instantiations)
#define GPB_TRACE_N ((EPI == EPI_TRACE_RAGGED) ? p.nvec[b] : p.n)
    for (int q = tid; q < TM + TN; q += NTHREADS) {
      const bool row = q < TM;
      const int ql = row ? q : q - TM;
      const int i = (row ? task.c_r : task.c_c) + ql;
      (row ? xr : xc)[ql] = (i < GPB_TRACE_N) ? x[i] : 0.0;
      (row ? ar : ac)[ql] = (i < GPB_TRACE_N) ? av[i] : 0.0;
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
          if (i < GPB_TRACE_N && j < GPB_TRACE_N) {
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
#undef GPB_TRACE_N
  }
