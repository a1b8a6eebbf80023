// DISInclusiveKL score of the low-rank LRGaussian family (Sigma = B B^T + D^2, D = diag(sigma), sigma = exp(ls),
// var_param = [mu, ls, B (d x k, row-major)]):  value = -sum_r c_r log q(x_r),  x_r = x[idx[r]],  and its gradient.
// With P = [C^-1 | P_B] (k x (k + d)), P_B = -C^-1 B^T D^-1, C C^T = M = I + B^T D^-2 B (the projection that
// lr_stream.cu also takes; see there for why |u|^2 - |a|^2 is the Mahalanobis term):
//
//     u_r = D^-1 (x_r - mu),   a_r = P_B u_r,   s_r = D^-1 (u_r - P_B^T a_r) = Sigma^-1 (x_r - mu)
//     log q_r = -1/2 (d log 2 pi + 2 sum ls + |u_r|^2 - |a_r|^2) + sum_l log P_ll
//     gbar_mu = -sum_r c_r s_r
//     lsbar_j = -sigma_j^2 sum_r c_r s_rj^2 + C_tot (1 - |P_B[:, j]|^2)            (sigma_j^2 Sigma^-1_jj = 1 - |P_B[:, j]|^2)
//     Bbar    = -S^T diag(c) (S B) + C_tot D^-2 B M^-1,   D^-2 B M^-1 = -D^-1 P_B^T C^-1,   C_tot = sum_r c_r
//
// The four n x d x k products (A = U P_B^T, S = D^-1 (U - A P_B), S B and S^T diag(c) (S B): about 8 n d k flops) run
// on the FP64 tensor pipe through gemm_f64; the rest are row and column passes over n x d with fixed summation orders.
// Nothing of size d x d is formed, nothing is atomic, and the host is never synchronised.
#include "gemm_internal.cuh"

namespace vb {

// U[r][j] = (x[i_r][j] - mu_j) / sigma_j,  i_r = idx ? idx[r] : r   (grid-stride over n x d)
__global__ void lr_score_u_kernel(const double* __restrict__ vp, const double* __restrict__ x, const long long* __restrict__ idx,
                                  int64_t n, int d, double* __restrict__ U) {
  const int64_t total = n * d;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / d;
    const int j = (int)(e - r * d);
    const int64_t src = idx ? idx[r] : r;
    U[e] = (x[src * d + j] - vp[j]) / exp(vp[d + j]);
  }
}

// per row (one warp, grid-stride): rowt[r] = |u_r|^2 - |a_r|^2, cr[r] = scale w[r], and S_r = (U_r + T_r) / sigma in
// place of T_r = -P_B^T a_r, which S holds on entry when k > 0 (with k = 0, S_r = U_r / sigma)
__global__ void __launch_bounds__(256) lr_score_rows_kernel(const double* __restrict__ vp, const double* __restrict__ U,
                                                            const double* __restrict__ A, const double* __restrict__ w,
                                                            double scale, int64_t n, int d, int k, double* __restrict__ S,
                                                            double* __restrict__ rowt, double* __restrict__ cr) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; r < n; r += nwarps) {
    double uu = 0.0, aa = 0.0;
    for (int j = lane; j < d; j += 32) {
      const double u = U[r * d + j];
      uu += u * u;
      S[r * d + j] = (k > 0 ? u + S[r * d + j] : u) / exp(vp[d + j]);
    }
    for (int l = lane; l < k; l += 32) {
      const double a = A[r * k + l];
      aa += a * a;
    }
    uu = warp_sum(uu);
    aa = warp_sum(aa);
    if (lane == 0) {
      rowt[r] = uu - aa;
      cr[r] = scale * (w ? w[r] : 1.0);
    }
  }
}

// scal = {value, C_tot}, value[0] = scal[0]   (single block, fixed summation order)
__global__ void __launch_bounds__(1024) lr_score_value_kernel(const double* __restrict__ vp, const double* __restrict__ P,
                                                              const double* __restrict__ rowt, const double* __restrict__ cr,
                                                              int64_t n, int d, int k, double* __restrict__ scal,
                                                              double* __restrict__ value) {
  __shared__ double red[32];
  double a = 0.0, b = 0.0;
  for (int j = threadIdx.x; j < d; j += blockDim.x) a += vp[d + j];
  for (int l = threadIdx.x; l < k; l += blockDim.x) b += log(P[(size_t)l * (k + d) + l]);
  a = block_sum(a, red);
  b = block_sum(b, red);
  const double lqc = -0.5 * kLog2Pi * d - a + b;
  double v = 0.0, c = 0.0;
  for (int64_t r = threadIdx.x; r < n; r += blockDim.x) {
    v += cr[r] * (lqc - 0.5 * rowt[r]);
    c += cr[r];
  }
  v = block_sum(v, red);
  c = block_sum(c, red);
  if (threadIdx.x == 0) {
    scal[0] = value[0] = -v;
    scal[1] = c;
  }
}

// grad[j] = -sum_r c_r S[r][j],  grad[d + j] = -sigma_j^2 sum_r c_r S[r][j]^2 + C_tot (1 - |P_B[:, j]|^2)
// (block = 32 columns x 32 row groups; the groups are summed in order)
__global__ void __launch_bounds__(1024) lr_score_cols_kernel(const double* __restrict__ vp, const double* __restrict__ P,
                                                             const double* __restrict__ S, const double* __restrict__ cr,
                                                             const double* __restrict__ scal, int64_t n, int d, int k,
                                                             double* __restrict__ grad) {
  __shared__ double sm[2][32][33];
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + x;
  double a = 0.0, b = 0.0;
  if (j < d)
    for (int64_t r = y; r < n; r += 32) {
      const double s = S[r * d + j], c = cr[r];
      a += c * s;
      b += c * s * s;
    }
  sm[0][y][x] = a;
  sm[1][y][x] = b;
  __syncthreads();
  if (y == 0 && j < d) {
    double ta = 0.0, tb = 0.0;
#pragma unroll
    for (int q = 0; q < 32; ++q) { ta += sm[0][q][x]; tb += sm[1][q][x]; }
    double pb = 0.0;
    for (int m = 0; m < k; ++m) {
      const double p = P[(size_t)m * (k + d) + k + j];
      pb += p * p;
    }
    const double sig = exp(vp[d + j]);
    grad[j] = -ta;
    grad[d + j] = -sig * sig * tb + scal[1] * (1.0 - pb);
  }
}

// Bbar[j][l] += C_tot (D^-2 B M^-1)[j][l] = -C_tot / sigma_j sum_m P_B[m][j] C^-1[m][l]   (grid-stride over d x k)
__global__ void lr_score_bfix_kernel(const double* __restrict__ vp, const double* __restrict__ P, const double* __restrict__ scal,
                                     int d, int k, double* __restrict__ Bbar) {
  const int64_t total = (int64_t)d * k;
  const double ctot = scal[1];
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(e / k), l = (int)(e - (int64_t)j * k);
    double a = 0.0;
    for (int m = 0; m < k; ++m) a += P[(size_t)m * (k + d) + k + j] * P[(size_t)m * (k + d) + l];
    Bbar[e] -= ctot / exp(vp[d + j]) * a;
  }
}

static inline int lr_ew_grid(int64_t n) {
  const int64_t b = (n + 255) / 256, cap = 16LL * sm_count();
  return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}

struct LrScoreLayout {
  size_t off_U, off_A, off_S, off_SB, off_rowt, off_cr, off_scal, total;
};
static void lr_score_layout(int64_t n, int d, int k, LrScoreLayout& l) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  l.off_U = take(sizeof(double) * (size_t)n * d);
  l.off_A = take(sizeof(double) * (size_t)n * k);
  l.off_S = take(sizeof(double) * (size_t)n * d);
  l.off_SB = take(sizeof(double) * (size_t)n * k);
  l.off_rowt = take(sizeof(double) * (size_t)n);
  l.off_cr = take(sizeof(double) * (size_t)n);
  l.off_scal = take(sizeof(double) * 4);
  l.total = off;
}

static int gemm(bool ta, bool tb, int M, int N, int K, double alpha, const double* A, int64_t lda, const double* B,
                int64_t ldb, double* C, int64_t ldc, const double* kscale, cudaStream_t stream) {
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc;
  g.kscale = kscale; g.rowscale = nullptr; g.bias = nullptr; g.divm = nullptr; g.divn = nullptr;
  return gemm_f64(g, ta, tb, stream);
}

}  // namespace vb
using namespace vb;

/* workspace of vb_lr_score_f64: 2 n d + 2 n k + 2 n + 4 doubles (256-byte aligned pieces) */
extern "C" size_t vb_lr_score_workspace_bytes(int64_t n, int d, int k) {
  if (n <= 0 || d <= 0 || k < 0) return 0;
  LrScoreLayout l;
  lr_score_layout(n, d, k, l);
  return l.total;
}

/* value[1] = -sum_r c_r log q(x_{i_r}; var_param) and grad[2d + d k] for LRGaussian (see the top of this file),
 * c_r = scale * w[r] (w NULL: 1), i_r = idx[r] (idx NULL: r), P = [C^-1 | -C^-1 B^T D^-1] (k x (k + d), NULL when
 * k = 0). */
extern "C" int vb_lr_score_f64(const double* var_param, const double* P, const double* x, const int64_t* idx, const double* w,
                               double scale, int64_t n, int d, int k, double* value, double* grad, void* workspace,
                               size_t workspace_bytes, cudaStream_t stream) {
  if (!var_param || !x || n <= 0 || d <= 0 || k < 0 || (k > 0 && !P) || !value || !grad)
    return set_error(VB_ERR_INVALID_ARG, "lr_score: bad arguments");
  LrScoreLayout l;
  lr_score_layout(n, d, k, l);
  if (!workspace || workspace_bytes < l.total) return set_error(VB_ERR_WORKSPACE, "lr_score: workspace too small");
  if (n > INT32_MAX || ceil_div(n, 64) * ceil_div(d, 64) > INT32_MAX)
    return set_error(VB_ERR_UNSUPPORTED, "lr_score: more than 2^31 - 1 tiles");
  char* ws = static_cast<char*>(workspace);
  double* U = reinterpret_cast<double*>(ws + l.off_U);
  double* A = reinterpret_cast<double*>(ws + l.off_A);
  double* S = reinterpret_cast<double*>(ws + l.off_S);
  double* SB = reinterpret_cast<double*>(ws + l.off_SB);
  double* rowt = reinterpret_cast<double*>(ws + l.off_rowt);
  double* cr = reinterpret_cast<double*>(ws + l.off_cr);
  double* scal = reinterpret_cast<double*>(ws + l.off_scal);
  const int nr = (int)n, K1 = k + d;
  const double* PB = P ? P + k : nullptr;
  lr_score_u_kernel<<<lr_ew_grid(n * d), 256, 0, stream>>>(var_param, x, reinterpret_cast<const long long*>(idx), n, d, U);
  VB_CHECK_LAUNCH();
  int rc;
  if (k > 0) {
    rc = gemm(false, true, nr, k, d, 1.0, U, d, PB, K1, A, k, nullptr, stream);       // A = U P_B^T
    if (rc) return rc;
    rc = gemm(false, false, nr, d, k, -1.0, A, k, PB, K1, S, d, nullptr, stream);     // -A P_B
    if (rc) return rc;
  }
  const int64_t blocks = ceil_div(n, 256 / 32), cap = 64LL * sm_count();
  lr_score_rows_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, stream>>>(var_param, U, A, w, scale, n, d, k, S, rowt, cr);
  VB_CHECK_LAUNCH();
  lr_score_value_kernel<<<1, 1024, 0, stream>>>(var_param, P, rowt, cr, n, d, k, scal, value);
  VB_CHECK_LAUNCH();
  lr_score_cols_kernel<<<(d + 31) / 32, 1024, 0, stream>>>(var_param, P, S, cr, scal, n, d, k, grad);
  VB_CHECK_LAUNCH();
  if (k > 0) {
    const double* Bm = var_param + 2 * (size_t)d;
    double* Bbar = grad + 2 * (size_t)d;
    rc = gemm(false, false, nr, k, d, 1.0, S, d, Bm, k, SB, k, nullptr, stream);      // S B
    if (rc) return rc;
    rc = gemm(true, false, d, k, nr, -1.0, S, d, SB, k, Bbar, k, cr, stream);         // -S^T diag(c) (S B)
    if (rc) return rc;
    lr_score_bfix_kernel<<<lr_ew_grid((int64_t)d * k), 256, 0, stream>>>(var_param, P, scal, d, k, Bbar);
    VB_CHECK_LAUNCH();
  }
  return VB_OK;
}
