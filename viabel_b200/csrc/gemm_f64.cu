// General float64 GEMM on the FP64 tensor pipe (mma.sync m8n8k4, DMMA) with the fused pro-/epilogues the
// full-rank MultivariateT path needs (mvt.cu; reference approximations.py:342-357, _distributions.py:7-38 and the
// autograd VJPs of sqrtm / eigh the reference leans on):
//
//     C[m,n] = epilogue( alpha * sum_k  A'(m,k) * kscale[k] * B'(k,n) )
//     A'(m,k) = TA ? A[k*lda + m] : A[m*lda + k]          B'(k,n) = TB ? B[n*ldb + k] : B[k*ldb + n]
//     epilogue(v) = v * rowscale[m]  /  (divm[m] + divn[n])  +  bias[n]          (each optional)
//
// 64 x 64 output tiles, K slabs of 32 through shared memory, 8 warps of 16 x 32 accumulators each (the same tiling
// as the SYRK in moments.cu).  Deterministic: no split-K.  The tiles are numbered row-major on a 1-D grid (gridDim.x
// allows 2^31 - 1 blocks, gridDim.y only 65535), so M and N are both limited only by their int type: the GLM plugins
// put the sample count on N in one GEMM and on M in the next.
#include "gemm_internal.cuh"

namespace vb {

constexpr int kGT = 64, kGK = 32, kGP = 68;

__device__ __forceinline__ void dmma_g(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

template <bool TA, bool TB>
__global__ void __launch_bounds__(256) gemm_f64_kernel(GemmArgs g) {
  __shared__ double sa[kGK][kGP], sb[kGK][kGP];
  const unsigned tiles_n = (unsigned)ceil_div(g.N, kGT);
  const int m0 = (int)(blockIdx.x / tiles_n) * kGT, n0 = (int)(blockIdx.x % tiles_n) * kGT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wm = warp >> 1, wn = warp & 1;
  const int gq = lane >> 2, t = lane & 3;
  double acc[2][4][2];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;

  for (int k0 = 0; k0 < g.K; k0 += kGK) {
    __syncthreads();
    // ---- A slab -> sa[k][m] ----
    if (TA) {       // A stored [K][M]: contiguous along m
      const int c = threadIdx.x & 63, r = threadIdx.x >> 6;
#pragma unroll
      for (int p = 0; p < kGK / 4; ++p) {
        const int k = p * 4 + r;
        double v = 0.0;
        if (k0 + k < g.K && m0 + c < g.M) v = g.A[(size_t)(k0 + k) * g.lda + m0 + c];
        if (g.kscale && k0 + k < g.K) v *= g.kscale[k0 + k];
        sa[k][c] = v;
      }
    } else {        // A stored [M][K]: contiguous along k
      const int k = threadIdx.x & 31, r = threadIdx.x >> 5;
#pragma unroll
      for (int p = 0; p < kGT / 8; ++p) {
        const int c = p * 8 + r;
        double v = 0.0;
        if (k0 + k < g.K && m0 + c < g.M) v = g.A[(size_t)(m0 + c) * g.lda + k0 + k];
        if (g.kscale && k0 + k < g.K) v *= g.kscale[k0 + k];
        sa[k][c] = v;
      }
    }
    // ---- B slab -> sb[k][n] ----
    if (!TB) {      // B stored [K][N]
      const int c = threadIdx.x & 63, r = threadIdx.x >> 6;
#pragma unroll
      for (int p = 0; p < kGK / 4; ++p) {
        const int k = p * 4 + r;
        double v = 0.0;
        if (k0 + k < g.K && n0 + c < g.N) v = g.B[(size_t)(k0 + k) * g.ldb + n0 + c];
        sb[k][c] = v;
      }
    } else {        // B stored [N][K]
      const int k = threadIdx.x & 31, r = threadIdx.x >> 5;
#pragma unroll
      for (int p = 0; p < kGT / 8; ++p) {
        const int c = p * 8 + r;
        double v = 0.0;
        if (k0 + k < g.K && n0 + c < g.N) v = g.B[(size_t)(n0 + c) * g.ldb + k0 + k];
        sb[k][c] = v;
      }
    }
    __syncthreads();
#pragma unroll
    for (int k4 = 0; k4 < kGK; k4 += 4) {
      double af[2], bf[4];
#pragma unroll
      for (int a = 0; a < 2; ++a) af[a] = sa[k4 + t][wm * 16 + a * 8 + gq];
#pragma unroll
      for (int b = 0; b < 4; ++b) bf[b] = sb[k4 + t][wn * 32 + b * 8 + gq];
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) dmma_g(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
    }
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int m = m0 + wm * 16 + a * 8 + gq;
      if (m >= g.M) continue;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int n = n0 + wn * 32 + b * 8 + 2 * t + u;
        if (n >= g.N) continue;
        double v = g.alpha * acc[a][b][u];
        if (g.rowscale) v *= g.rowscale[m];
        if (g.divm) v /= (g.divm[m] + g.divn[n]);
        if (g.bias) v += g.bias[n];
        g.C[(size_t)m * g.ldc + n] = v;
      }
    }
}

int gemm_f64(const GemmArgs& g, bool ta, bool tb, cudaStream_t stream) {
  if (g.M <= 0 || g.N <= 0 || g.K < 0 || !g.A || !g.B || !g.C) return set_error(VB_ERR_INVALID_ARG, "gemm_f64: bad arguments");
  const int64_t tiles = ceil_div(g.M, kGT) * ceil_div(g.N, kGT);
  if (tiles > INT32_MAX) return set_error(VB_ERR_UNSUPPORTED, "gemm_f64: more than 2^31 - 1 output tiles");
  const dim3 grid((unsigned)tiles);
  if (ta && tb) gemm_f64_kernel<true, true><<<grid, 256, 0, stream>>>(g);
  else if (ta) gemm_f64_kernel<true, false><<<grid, 256, 0, stream>>>(g);
  else if (tb) gemm_f64_kernel<false, true><<<grid, 256, 0, stream>>>(g);
  else gemm_f64_kernel<false, false><<<grid, 256, 0, stream>>>(g);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

}  // namespace vb
using namespace vb;

extern "C" int vb_gemm_f64(int trans_a, int trans_b, int M, int N, int K, double alpha, const double* A, int64_t lda,
                           const double* B, int64_t ldb, double* C, int64_t ldc, const double* kscale, const double* rowscale,
                           const double* bias, const double* divm, const double* divn, cudaStream_t stream) {
  if ((divm == nullptr) != (divn == nullptr)) return set_error(VB_ERR_INVALID_ARG, "gemm_f64: divm and divn come together");
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.alpha = alpha;
  g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc;
  g.kscale = kscale; g.rowscale = rowscale; g.bias = bias; g.divm = divm; g.divn = divn;
  return gemm_f64(g, trans_a != 0, trans_b != 0, stream);
}
