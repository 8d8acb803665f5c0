// Device random numbers for posterior sampling (f-4): counter-based Philox4x32-10 -> 53-bit uniforms ->
// Box-Muller standard normals.  Stateless: element e of a stream is a pure function of (seed, e), so a
// draw is reproducible across launches, grid shapes and GPUs, and a CPU restatement in the test
// suite can check it bit for bit on the integer part.  Replaces the host RNG behind MASS::mvrnorm
// (pendulum_fit.R:253, lorenz.Rmd:105) and numpy.random.randn (ch2.py:43-45).
#include <algorithm>

#include "common.cuh"
#include "gram.cuh"

namespace gpb {

__device__ __forceinline__ void philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0,
                                              unsigned k1, unsigned (&out)[4]) {
  constexpr unsigned M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const unsigned hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    const unsigned hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    const unsigned n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// two 32-bit words -> uniform in (0, 1) with 53 random bits, never 0 or 1
__device__ __forceinline__ double u53(unsigned a, unsigned b) {
  const unsigned long long m = ((unsigned long long)(a >> 5) << 26) | (unsigned long long)(b >> 6);
  return ((double)m + 0.5) * (1.0 / 9007199254740992.0);
}

// out[e] for e in [0, len): normal number offset + e of stream `seed`.  Counter q = (offset + e) / 2
// yields the Box-Muller pair (offset + e even: cos branch, odd: sin branch).  ld / rows lay the stream out as
// a column-major matrix with padding rows left untouched (rows == ld for a flat vector).  An odd offset
// (a chunk of draws of odd length starting mid-pair) regenerates the pair it starts in and keeps its sin half.
__global__ void normal_fill_kernel(unsigned long long seed, unsigned long long offset, long long len, long long rows,
                                   long long ld, double *__restrict__ out) {
  const long long first = (long long)(offset & 1ULL);
  const long long npairs = (len + first + 1) / 2;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < npairs; q += (long long)gridDim.x * blockDim.x) {
    const unsigned long long ctr = (offset >> 1) + (unsigned long long)q;
    unsigned r[4];
    philox4x32_10((unsigned)ctr, (unsigned)(ctr >> 32), 0u, 0u, (unsigned)seed, (unsigned)(seed >> 32), r);
    const double u1 = u53(r[0], r[1]), u2 = u53(r[2], r[3]);
    const double rad = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    const long long e0 = 2 * q - first, e1 = e0 + 1;
    if (e0 >= 0) out[(e0 / rows) * ld + (e0 % rows)] = rad * c;
    if (e1 < len) out[(e1 / rows) * ld + (e1 % rows)] = rad * s;
  }
}

int launch_normal_fill(Handle *h, unsigned long long seed, unsigned long long offset, long long len, long long rows,
                       long long ld, double *out) {
  if (len <= 0) return 0;
  const long long npairs = (len + (long long)(offset & 1ULL) + 1) / 2;
  const int blocks = (int)std::min<long long>((npairs + 255) / 256, 148 * 8);
  ProfScope ps__(h, PC_OTHER);
  normal_fill_kernel<<<blocks, 256, 0, h->stream>>>(seed, offset, len, rows, ld, out);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// out[d + i*ldo] = mu[i] + X[i + d*ldx]  (transpose of the padded m x ndraws product into R's
// ndraws x m mvrnorm layout)
__global__ void add_mean_transpose_kernel(int m, int ndraws, const double *__restrict__ X, long long ldx,
                                          const double *__restrict__ mu, double *__restrict__ out, long long ldo) {
  __shared__ double tile[32][33];
  const int i0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int i = i0 + threadIdx.x, d = d0 + r;
    tile[r][threadIdx.x] = (i < m && d < ndraws) ? X[i + (long long)d * ldx] + (mu ? mu[i] : 0.0) : 0.0;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int d = d0 + threadIdx.x, i = i0 + r;
    if (i < m && d < ndraws) out[d + (long long)i * ldo] = tile[threadIdx.x][r];
  }
}

int launch_add_mean_transpose(Handle *h, int m, int ndraws, const double *X, long long ldx, const double *mu,
                              double *out, long long ldo) {
  dim3 grid((m + 31) / 32, (ndraws + 31) / 32), block(32, 8);
  ProfScope ps__(h, PC_OTHER);
  add_mean_transpose_kernel<<<grid, block, 0, h->stream>>>(m, ndraws, X, ldx, mu, out, ldo);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

// dst[b*rows + i] = src[b*src_stride + row0 + i], or NaN for every i when info[b] != 0 (a failed item)
__global__ void rows_or_nan_kernel(int row0, int rows, const double *__restrict__ src, long long src_stride,
                                   const int *__restrict__ info, double *__restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const long long b = blockIdx.y;
  if (i >= rows) return;
  dst[b * rows + i] = info[b] ? __longlong_as_double(0x7ff8000000000000LL) : src[b * src_stride + row0 + i];
}

int launch_rows_or_nan(Handle *h, int row0, int rows, const double *src, long long src_stride, const int *info,
                       double *dst, int batch) {
  dim3 grid((rows + 255) / 256, batch);
  ProfScope ps__(h, PC_OTHER);
  rows_or_nan_kernel<<<grid, 256, 0, h->stream>>>(row0, rows, src, src_stride, info, dst);
  GPB_LAUNCH_CHECK(h);
  return 0;
}

}  // namespace gpb
