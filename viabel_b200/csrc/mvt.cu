// Full-rank MultivariateT family (reference approximations.py:322-382, _distributions.py:7-38) and its
// ExclusiveKL / AlphaDivergence objectives (objectives.py:154-164, :443-460) on the device.
//
//   var_param = [mu(d), row-major lower triangle of F],  L = tril(F,-1) + diag(exp(diag F)),  Sigma = L L^T
//   (paragami PSDSymmetricMatrixPattern, approximations.py:315-319).  Samples use the SYMMETRIC square root
//   A = V sqrt(W) V^T of Sigma (sqrtm, :348); the eigen-decomposition Sigma = V W V^T is the caller's (cuSOLVER).
//
// A is never formed: with P = (Z / u) V,
//     theta = mu + (P . sqrt(w)) V^T                                  two S x d x d GEMMs
//     Abar  = c (Z/u)^T (sv . G)    =>   V^T Abar V = c P^T Q,  Q = (sv . G) V        (rank <= S: S x d x d GEMMs)
//     Sbar  = V [ (V^T Abar V) ./ (sqrt(w_a) + sqrt(w_b)) ] V^T       (the Sylvester solve of the sqrtm VJP)
//     Lbar  = (Sbar + Sbar^T) L,   Fbar = tril(Lbar,-1) + diag(diag(Lbar) . diag(L) + diag_add)
// All GEMMs are the float64 DMMA kernel of gemm_f64.cu with the row / column / division scalings fused into its
// pro- and epilogues.  SURVEY.md App. A.3 has the derivation.
#include "gemm_internal.cuh"
#include "mvt_internal.cuh"

namespace vb {

__global__ void mvt_unpack_kernel(const double* __restrict__ vp, int d, double* __restrict__ L) {
  const int64_t total = (int64_t)d * d;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / d), j = (int)(idx - (int64_t)i * d);
    double v = 0.0;
    if (j <= i) {
      const double f = vp[d + (int64_t)i * (i + 1) / 2 + j];
      v = i == j ? exp(f) : f;
    }
    L[idx] = v;
  }
}

// out[0] = sum_i F_ii (= 0.5 log det Sigma)
__global__ void __launch_bounds__(256) mvt_logdiag_kernel(const double* __restrict__ vp, int d, double* __restrict__ out) {
  __shared__ double red[32];
  double a = 0.0;
  for (int i = threadIdx.x; i < d; i += blockDim.x) a += vp[d + (int64_t)i * (i + 1) / 2 + i];
  a = block_sum(a, red);
  if (threadIdx.x == 0) out[0] = a;
}

// inv_u[s] = 1 / sqrt(chi2_s / df);  zu2[s] = |z_s / u_s|^2   (one warp per sample, grid-stride over samples)
__global__ void __launch_bounds__(256) mvt_rows_kernel(const double* __restrict__ z, const double* __restrict__ chi2, double df,
                                                       int S, int d, double* __restrict__ inv_u, double* __restrict__ zu2) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t s = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; s < S; s += nwarps) {
    const double iu = 1.0 / sqrt(chi2[s] / df);
    double a = 0.0;
    for (int j = lane; j < d; j += 32) {
      const double v = z[s * d + j] * iu;
      a += v * v;
    }
    a = warp_sum(a);
    if (lane == 0) {
      inv_u[s] = iu;
      zu2[s] = a;
    }
  }
}

// sqrtw[k] = sqrt(max(w_k, 0));  winv[k] = |w_k| <= 1e-10 ? 0 : 1 / w_k   (_distributions.py:26-28);
// rinv[k] = winv_k sqrtw_k = w_k > 1e-10 ? 1 / sqrt(w_k) : 0   (Sigma^+ A = V diag(rinv) V^T)
__global__ void mvt_eig_kernel(const double* __restrict__ w, int d, double* __restrict__ sqrtw, double* __restrict__ winv,
                               double* __restrict__ rinv) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= d) return;
  const double v = w[k];
  if (sqrtw) sqrtw[k] = sqrt(fmax(v, 0.0));
  if (winv) winv[k] = fabs(v) <= 1e-10 ? 0.0 : 1.0 / v;
  if (rinv) rinv[k] = v > 1e-10 ? 1.0 / sqrt(v) : 0.0;
}

// Sample weights and objective value (single block).  scal: [0] value, [1] diag_add.
__global__ void __launch_bounds__(1024) mvt_weights_kernel(const double* __restrict__ f, const double* __restrict__ zu2, int S, int d,
                                                           double df, double logq_const, const double* __restrict__ sld,
                                                           int objective, double alpha, double* __restrict__ sv,
                                                           double* __restrict__ scal) {
  __shared__ double red[32];
  const double half_logdet = sld[0];
  if (objective == VB_OBJ_EXCLUSIVE_KL_PATH) {
    // -mean(f - log q) at var_param held fixed (objectives.py:156-159); no entropy term in the gradient
    double a = 0.0;
    for (int s = threadIdx.x; s < S; s += blockDim.x) {
      a += f[s] - (logq_const - half_logdet - 0.5 * (df + d) * log1p(zu2[s] / df));
      sv[s] = 1.0;
    }
    a = block_sum(a, red);
    if (threadIdx.x == 0) {
      scal[0] = -a / (double)S;
      scal[1] = 0.0;
    }
    return;
  }
  if (objective == VB_OBJ_EXCLUSIVE_KL) {
    double a = 0.0;
    for (int s = threadIdx.x; s < S; s += blockDim.x) {
      a += f[s];
      sv[s] = 1.0;
    }
    a = block_sum(a, red);
    if (threadIdx.x == 0) {
      scal[0] = -(a / (double)S + half_logdet);          // entropy (up to df-only constants) = 0.5 log det Sigma (:351-354)
      scal[1] = -1.0;
    }
    return;
  }
  // lw = f - log q, log q = const - 0.5 log det - 0.5 (df + d) log1p(|z/u|^2 / df): the Mahalanobis term at a
  // reparameterised sample is |z/u|^2 exactly (theta - mu = (z/u) A, A Sigma^-1 A = I)
  double m = -INFINITY;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    const double lq = logq_const - half_logdet - 0.5 * (df + d) * log1p(zu2[s] / df);
    const double lw = f[s] - lq;
    sv[s] = lw;
    m = fmax(m, lw);
  }
  m = block_max(m, red);
  double a = 0.0;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    const double v = pow(exp(sv[s] - m), alpha);
    sv[s] = v;
    a += v;
  }
  a = block_sum(a, red);
  if (threadIdx.x == 0) {
    scal[0] = log(a / (double)S) / alpha + m;
    scal[1] = alpha / (double)S * a;
  }
}

// gmu[j] = c * sum_s sv_s G[s][j]   (block = 32 columns x 32 sample groups)
__global__ void __launch_bounds__(1024) mvt_gmu_kernel(const double* __restrict__ G, const double* __restrict__ sv, int S, int d,
                                                       double c, double* __restrict__ gmu) {
  __shared__ double sm[32][33];
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + x;
  double a = 0.0;
  if (j < d)
    for (int s = y; s < S; s += 32) a += sv[s] * G[(size_t)s * d + j];
  sm[y][x] = a;
  __syncthreads();
  if (y == 0 && j < d) {
    double t = 0.0;
#pragma unroll
    for (int r = 0; r < 32; ++r) t += sm[r][x];
    gmu[j] = c * t;
  }
}

// Path-derivative ExclusiveKL, sqrtm mode: y_s = Sigma^+ (theta_s - mu) = V diag(rinv) P_s^T with the reference's
// eigenvalue floor, so delta_s = (theta_s - mu)^T Sigma^+ (theta_s - mu) = sum over unfloored k of P[s][k]^2 and
// kappa_s = (df + d) / (df + delta_s)   (one warp per sample)
__global__ void __launch_bounds__(256) mvt_path_delta_kernel(const double* __restrict__ P, const double* __restrict__ rinv, int S,
                                                             int d, double df, double* __restrict__ delta,
                                                             double* __restrict__ kappa) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t s = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; s < S; s += nwarps) {
    double a = 0.0;
    for (int k = lane; k < d; k += 32) {
      const double p = P[s * d + k];
      if (rinv[k] > 0.0) a += p * p;
    }
    a = warp_sum(a);
    if (lane == 0) {
      delta[s] = a;
      kappa[s] = (df + d) / (df + a);
    }
  }
}

// (G + diag(kappa) Y) V = Q + diag(kappa) P diag(rinv):  Q[s][k] += kappa_s rinv_k P[s][k]
__global__ void mvt_path_q_kernel(const double* __restrict__ P, const double* __restrict__ kappa, const double* __restrict__ rinv,
                                  int S, int d, double* __restrict__ Q) {
  const int64_t total = (int64_t)S * d;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = idx / d, k = idx - s * d;
    Q[idx] += kappa[s] * (rinv[k] * P[idx]);
  }
}

// out = in + in^T
__global__ void mvt_symmetrise_kernel(const double* __restrict__ in, int d, double* __restrict__ out) {
  __shared__ double tile[32][33];
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;        // 32 x 8
  for (int r = ty; r < 32; r += 8)
    tile[r][tx] = (bx + r < d && by + tx < d) ? in[(size_t)(bx + r) * d + by + tx] : 0.0;       // block (bx, by) of `in`
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int i = by + r, j = bx + tx;                           // writes block (by, bx): out[i][j] = in[i][j] + in[j][i]
    if (i < d && j < d) out[(size_t)i * d + j] = in[(size_t)i * d + j] + tile[tx][r];
  }
}

// grad[d + i(i+1)/2 + j] = i > j ? Lbar[i][j] : Lbar[i][i] * L[i][i] + diag_add
__global__ void mvt_pack_kernel(const double* __restrict__ Lbar, const double* __restrict__ L, int d,
                                const double* __restrict__ scal, double* __restrict__ grad) {
  const int64_t total = (int64_t)d * d;
  const double diag_add = scal[1];
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / d), j = (int)(idx - (int64_t)i * d);
    if (j > i) continue;
    const double v = i == j ? Lbar[idx] * L[idx] + diag_add : Lbar[idx];
    grad[d + (int64_t)i * (i + 1) / 2 + j] = v;
  }
}

// out[i] = const - 0.5 sum log w - 0.5 (df + d) log(1 + sum_k R[i][k]^2 winv_k / df)   (one warp per row)
__global__ void __launch_bounds__(256) mvt_logpdf_kernel(const double* __restrict__ R, const double* __restrict__ winv,
                                                         const double* __restrict__ logpdet, int64_t n, int d, double df,
                                                         double logq_const, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  double a = 0.0;
  for (int k = lane; k < d; k += 32) {
    const double r = R[i * d + k];
    a += r * r * winv[k];
  }
  a = warp_sum(a);
  if (lane == 0) out[i] = logq_const - 0.5 * logpdet[0] - 0.5 * (df + d) * log(1.0 + a / df);
}

__global__ void __launch_bounds__(256) mvt_sumlog_kernel(const double* __restrict__ w, int d, double* __restrict__ out) {
  __shared__ double red[32];
  double a = 0.0;
  for (int i = threadIdx.x; i < d; i += blockDim.x) a += log(w[i]);
  a = block_sum(a, red);
  if (threadIdx.x == 0) out[0] = a;
}

int mvt_rows(const double* z, const double* chi2, double df, int S, int d, double* inv_u, double* zu2, cudaStream_t stream) {
  const int64_t blocks = ceil_div(S, 256 / 32), cap = 64LL * sm_count();
  mvt_rows_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, stream>>>(z, chi2, df, S, d, inv_u, zu2);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

int mvt_logdiag(const double* var_param, int d, double* out, cudaStream_t stream) {
  mvt_logdiag_kernel<<<1, 256, 0, stream>>>(var_param, d, out);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

int mvt_weights_gmu(const double* f, const double* G, const double* zu2, const double* half_logdet, int S, int d, double df,
                    int objective, double alpha, double* sv, double* scal, double* value, double* gmu, cudaStream_t stream) {
  const double c = objective == VB_OBJ_ALPHA ? alpha / S : -1.0 / S;
  mvt_weights_kernel<<<1, 1024, 0, stream>>>(f, zu2, S, d, df, mvt_const(df, d), half_logdet, objective, alpha, sv, scal);
  VB_CHECK_LAUNCH();
  VB_CUDA(cudaMemcpyAsync(value, scal, sizeof(double), cudaMemcpyDeviceToDevice, stream));
  return mvt_gmu(G, sv, S, d, c, gmu, stream);
}

int mvt_gmu(const double* G, const double* sv, int S, int d, double c, double* gmu, cudaStream_t stream) {
  mvt_gmu_kernel<<<(d + 31) / 32, 1024, 0, stream>>>(G, sv, S, d, c, gmu);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

static inline int ew_grid(int64_t n) {
  int64_t b = (n + 255) / 256;
  const int64_t cap = 16LL * sm_count();
  return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}

static int gemm(bool ta, bool tb, int M, int N, int K, double alpha, const double* A, int64_t lda, const double* B, int64_t ldb,
                double* C, int64_t ldc, const double* kscale, const double* rowscale, const double* bias, const double* divm,
                const double* divn, cudaStream_t stream) {
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc;
  g.kscale = kscale; g.rowscale = rowscale; g.bias = bias; g.divm = divm; g.divn = divn;
  return gemm_f64(g, ta, tb, stream);
}

}  // namespace vb
using namespace vb;

/* L[d,d] (dense lower triangular) and half_logdet[1] = sum_i F_ii from var_param */
extern "C" int vb_mvt_unpack_f64(const double* var_param, int d, double* L, double* half_logdet, cudaStream_t stream) {
  if (!var_param || d <= 0 || !L) return set_error(VB_ERR_INVALID_ARG, "mvt_unpack: bad arguments");
  mvt_unpack_kernel<<<ew_grid((int64_t)d * d), 256, 0, stream>>>(var_param, d, L);
  VB_CHECK_LAUNCH();
  return half_logdet ? mvt_logdiag(var_param, d, half_logdet, stream) : VB_OK;
}

/* Sigma = L L^T */
extern "C" int vb_mvt_sigma_f64(const double* L, int d, double scale, double* Sigma, cudaStream_t stream) {
  if (!L || d <= 0 || !Sigma) return set_error(VB_ERR_INVALID_ARG, "mvt_sigma: bad arguments");
  return gemm(false, true, d, d, d, scale, L, d, L, d, Sigma, d, nullptr, nullptr, nullptr, nullptr, nullptr, stream);
}

/* workspace: S + d doubles (256-byte aligned pieces) */
extern "C" size_t vb_mvt_transform_workspace_bytes(int S, int d) {
  if (S <= 0 || d <= 0) return 0;
  return align_up(sizeof(double) * S, 256) + align_up(sizeof(double) * d, 256);
}

/* P[S,d] = (z / u) V,  theta[S,d] = mu + (P . sqrt(w)) V^T,  zu2[S] = |z_s / u_s|^2;  u_s = sqrt(chi2_s / df)
 * (chi2 == NULL: u = 1, a Gaussian).  mu = var_param[:d]. */
extern "C" int vb_mvt_transform_f64(const double* var_param, const double* z, const double* chi2, double df, int S, int d,
                                    const double* w, const double* V, double* P, double* theta, double* zu2, void* workspace,
                                    size_t workspace_bytes, cudaStream_t stream) {
  if (!var_param || !z || !chi2 || S <= 0 || d <= 0 || !w || !V || !P || !theta || !zu2)
    return set_error(VB_ERR_INVALID_ARG, "mvt_transform: bad arguments");
  if (!(df > 2.0)) return set_error(VB_ERR_INVALID_ARG, "df must be greater than 2");
  if (!workspace || workspace_bytes < vb_mvt_transform_workspace_bytes(S, d)) return set_error(VB_ERR_WORKSPACE, "mvt_transform: workspace too small");
  char* ws = static_cast<char*>(workspace);
  double* inv_u = reinterpret_cast<double*>(ws);
  double* sqrtw = reinterpret_cast<double*>(ws + align_up(sizeof(double) * S, 256));
  int rc = mvt_rows(z, chi2, df, S, d, inv_u, zu2, stream);
  if (rc) return rc;
  mvt_eig_kernel<<<(d + 255) / 256, 256, 0, stream>>>(w, d, sqrtw, nullptr, nullptr);
  VB_CHECK_LAUNCH();
  rc = gemm(false, false, S, d, d, 1.0, z, d, V, d, P, d, nullptr, inv_u, nullptr, nullptr, nullptr, stream);
  if (rc) return rc;
  return gemm(false, true, S, d, d, 1.0, P, d, V, d, theta, d, sqrtw, nullptr, var_param, nullptr, nullptr, stream);
}

struct MvtObjLayout {
  size_t off_sv, off_scal, off_sqrtw, off_Q, off_M, off_M2, off_T, off_Lbar, total;
  size_t off_delta, off_kappa, off_rinv, off_gmu, off_ksum, total_path;     // path-derivative ExclusiveKL only
};
static void mvt_obj_layout(int S, int d, MvtObjLayout& l) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  l.off_sv = take(sizeof(double) * S);
  l.off_scal = take(sizeof(double) * 4);
  l.off_sqrtw = take(sizeof(double) * d);
  l.off_Q = take(sizeof(double) * (size_t)S * d);
  l.off_M = take(sizeof(double) * (size_t)d * d);
  l.off_M2 = take(sizeof(double) * (size_t)d * d);
  l.off_T = take(sizeof(double) * (size_t)d * d);
  l.off_Lbar = take(sizeof(double) * (size_t)d * d);
  l.total = off;
  l.off_delta = take(sizeof(double) * S);
  l.off_kappa = take(sizeof(double) * S);
  l.off_rinv = take(sizeof(double) * d);
  l.off_gmu = take(sizeof(double) * d);
  l.off_ksum = take(sizeof(double) * d);
  l.total_path = off;
}

extern "C" size_t vb_mvt_objective_workspace_bytes(int S, int d) {
  if (S <= 0 || d <= 0) return 0;
  MvtObjLayout l;
  mvt_obj_layout(S, d, l);
  return l.total;
}

/* workspace of vb_mvt_objective_f64 with VB_OBJ_EXCLUSIVE_KL_PATH: the above plus 2 S + 3 d doubles */
extern "C" size_t vb_mvt_path_workspace_bytes(int S, int d) {
  if (S <= 0 || d <= 0) return 0;
  MvtObjLayout l;
  mvt_obj_layout(S, d, l);
  return l.total_path;
}

/* value[1] and grad[d + d(d+1)/2] of ExclusiveKL (entropy or path-derivative form) / AlphaDivergence from the model's
 * per-sample log density f[S] and gradient G[S,d] at theta (vb_mvt_transform_f64), L and half_logdet
 * (vb_mvt_unpack_f64), w / V (eigh of Sigma), P and zu2 (vb_mvt_transform_f64).  The path-derivative form runs the
 * entropy form's VJP on G + diag(kappa) Y, Y = (theta - mu) Sigma^+ (floored pseudo-inverse), without the entropy
 * term: (G + diag(kappa) Y) V = Q + diag(kappa) P diag(rinv), and the mean part gains c V (rinv . sum_s kappa_s P_s). */
extern "C" int vb_mvt_objective_f64(const double* L, const double* half_logdet, const double* w, const double* V,
                                    const double* P, const double* zu2, const double* f, const double* G, int S, int d,
                                    double df, int objective, double alpha, double* value, double* grad, void* workspace,
                                    size_t workspace_bytes, cudaStream_t stream) {
  if (!L || !half_logdet || !w || !V || !P || !zu2 || !f || !G || S <= 0 || d <= 0 || !value || !grad)
    return set_error(VB_ERR_INVALID_ARG, "mvt_objective: bad arguments");
  if (objective != VB_OBJ_EXCLUSIVE_KL && objective != VB_OBJ_EXCLUSIVE_KL_PATH && objective != VB_OBJ_ALPHA)
    return set_error(VB_ERR_UNSUPPORTED, "mvt_objective: unknown objective");
  const bool path = objective == VB_OBJ_EXCLUSIVE_KL_PATH;
  MvtObjLayout l;
  mvt_obj_layout(S, d, l);
  if (!workspace || workspace_bytes < (path ? l.total_path : l.total))
    return set_error(VB_ERR_WORKSPACE, "mvt_objective: workspace too small");
  char* ws = static_cast<char*>(workspace);
  double* sv = reinterpret_cast<double*>(ws + l.off_sv);
  double* scal = reinterpret_cast<double*>(ws + l.off_scal);
  double* sqrtw = reinterpret_cast<double*>(ws + l.off_sqrtw);
  double* Q = reinterpret_cast<double*>(ws + l.off_Q);
  double* M = reinterpret_cast<double*>(ws + l.off_M);
  double* M2 = reinterpret_cast<double*>(ws + l.off_M2);
  double* T = reinterpret_cast<double*>(ws + l.off_T);
  double* Lbar = reinterpret_cast<double*>(ws + l.off_Lbar);
  const double c = objective == VB_OBJ_ALPHA ? alpha / S : -1.0 / S;
  int rc;
  if (path) {
    double* delta = reinterpret_cast<double*>(ws + l.off_delta);
    double* kappa = reinterpret_cast<double*>(ws + l.off_kappa);
    double* rinv = reinterpret_cast<double*>(ws + l.off_rinv);
    double* gmu = reinterpret_cast<double*>(ws + l.off_gmu);
    double* ksum = reinterpret_cast<double*>(ws + l.off_ksum);
    mvt_eig_kernel<<<(d + 255) / 256, 256, 0, stream>>>(w, d, sqrtw, nullptr, rinv);
    VB_CHECK_LAUNCH();
    const int64_t blocks = ceil_div(S, 256 / 32), cap = 64LL * sm_count();
    mvt_path_delta_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, stream>>>(P, rinv, S, d, df, delta, kappa);
    VB_CHECK_LAUNCH();
    rc = mvt_weights_gmu(f, G, delta, half_logdet, S, d, df, objective, alpha, sv, scal, value, gmu, stream);
    if (rc) return rc;
    rc = gemm(false, false, S, d, d, 1.0, G, d, V, d, Q, d, nullptr, sv, nullptr, nullptr, nullptr, stream);   // Q = G V
    if (rc) return rc;
    mvt_path_q_kernel<<<ew_grid((int64_t)S * d), 256, 0, stream>>>(P, kappa, rinv, S, d, Q);
    VB_CHECK_LAUNCH();
    mvt_gmu_kernel<<<(d + 31) / 32, 1024, 0, stream>>>(P, kappa, S, d, 1.0, ksum);                         // sum_s kappa_s P_s
    VB_CHECK_LAUNCH();
    rc = gemm(false, true, 1, d, d, c, ksum, d, V, d, grad, d, rinv, nullptr, gmu, nullptr, nullptr, stream);   // + c V (rinv . ksum)
    if (rc) return rc;
  } else {
    rc = mvt_weights_gmu(f, G, zu2, half_logdet, S, d, df, objective, alpha, sv, scal, value, grad, stream);
    if (rc) return rc;
    mvt_eig_kernel<<<(d + 255) / 256, 256, 0, stream>>>(w, d, sqrtw, nullptr, nullptr);
    VB_CHECK_LAUNCH();
    rc = gemm(false, false, S, d, d, 1.0, G, d, V, d, Q, d, nullptr, sv, nullptr, nullptr, nullptr, stream);   // Q = (sv . G) V
    if (rc) return rc;
  }
  rc = gemm(true, false, d, d, S, c, P, d, Q, d, M, d, nullptr, nullptr, nullptr, sqrtw, sqrtw, stream);           // c P^T Q ./ (rw + rw')
  if (rc) return rc;
  mvt_symmetrise_kernel<<<dim3((d + 31) / 32, (d + 31) / 32), 256, 0, stream>>>(M, d, M2);
  VB_CHECK_LAUNCH();
  rc = gemm(false, false, d, d, d, 1.0, V, d, M2, d, T, d, nullptr, nullptr, nullptr, nullptr, nullptr, stream);   // V M''
  if (rc) return rc;
  rc = gemm(false, true, d, d, d, 1.0, T, d, V, d, M, d, nullptr, nullptr, nullptr, nullptr, nullptr, stream);     // (V M'') V^T
  if (rc) return rc;
  rc = gemm(false, false, d, d, d, 1.0, M, d, L, d, Lbar, d, nullptr, nullptr, nullptr, nullptr, nullptr, stream); // (Sbar + Sbar^T) L
  if (rc) return rc;
  mvt_pack_kernel<<<ew_grid((int64_t)d * d), 256, 0, stream>>>(Lbar, L, d, scal, grad);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

/* workspace: n*d + 2d + 8 doubles */
extern "C" size_t vb_mvt_log_density_workspace_bytes(int64_t n, int d) {
  if (n <= 0 || d <= 0) return 0;
  return align_up(sizeof(double) * (size_t)n * d, 256) + 2 * align_up(sizeof(double) * d, 256) + 256;
}

/* out[i] = multivariate_t_logpdf(x_i; mu, Sigma = V diag(w) V^T, df)   (_distributions.py:7-38) */
extern "C" int vb_mvt_log_density_f64(const double* var_param, const double* w, const double* V, const double* x, int64_t n, int d,
                                      double df, double* out, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!var_param || !w || !V || !x || n <= 0 || d <= 0 || !out) return set_error(VB_ERR_INVALID_ARG, "mvt_log_density: bad arguments");
  if (!workspace || workspace_bytes < vb_mvt_log_density_workspace_bytes(n, d)) return set_error(VB_ERR_WORKSPACE, "mvt_log_density: workspace too small");
  if (n > 2000000000LL) return set_error(VB_ERR_UNSUPPORTED, "mvt_log_density: at most 2e9 rows per call");
  char* ws = static_cast<char*>(workspace);
  double* R = reinterpret_cast<double*>(ws);
  double* nmv = reinterpret_cast<double*>(ws + align_up(sizeof(double) * (size_t)n * d, 256));
  double* winv = nmv + align_up(sizeof(double) * d, 256) / sizeof(double);
  double* lpd = winv + align_up(sizeof(double) * d, 256) / sizeof(double);
  mvt_eig_kernel<<<(d + 255) / 256, 256, 0, stream>>>(w, d, nullptr, winv, nullptr);
  VB_CHECK_LAUNCH();
  mvt_sumlog_kernel<<<1, 256, 0, stream>>>(w, d, lpd);
  VB_CHECK_LAUNCH();
  int rc = gemm(false, false, 1, d, d, -1.0, var_param, d, V, d, nmv, d, nullptr, nullptr, nullptr, nullptr, nullptr, stream);   // -mu V
  if (rc) return rc;
  rc = gemm(false, false, (int)n, d, d, 1.0, x, d, V, d, R, d, nullptr, nullptr, nmv, nullptr, nullptr, stream);                 // (x - mu) V
  if (rc) return rc;
  mvt_logpdf_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, stream>>>(R, winv, lpd, n, d, df, mvt_const(df, d), out);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
