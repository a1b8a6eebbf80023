// Derivatives of the GLM log-likelihood at ONE point (the variational mean), float64: gradient, Hessian-vector
// products and the full Hessian.  They feed the control-variate ExclusiveKL estimators (reference
// objectives.py:170-273: `grad_f(m_mean)` :203/:221, `make_hvp(f_model)(m_mean)` :220/:238/:256,
// `hessian(f_model)(m_mean)` :200-204, all obtained there from autograd).
//
//   a_n = y_n x_n.theta,  r_n = dloglik/da,  c_n = -d^2 loglik/da^2 >= 0     (y in {-1,+1}: y^2 = 1)
//   grad    = sum_n y_n r_n x_n
//   hvp_k   = -sum_n c_n (x_n.v_k) x_n                        K <= 8 vectors per call
//   hessian = -sum_n c_n x_n x_n^T                             (weighted SYRK on the DMMA pipe, moments.cu)
// One pass over X for gradient + HVPs (HBM bound: N d 8 bytes); the caller adds the prior's part.
#include "moments_internal.cuh"

namespace vb {

constexpr int kPointRows = 32;      // rows per tile: 8 warps x 4 rows
constexpr int kPointMaxK = 8;
constexpr int kPointMaxCols = 8;    // columns per thread: d <= 2048

template <int K>
__global__ void __launch_bounds__(256) glm_point_kernel(const double* __restrict__ X, int64_t ldx,
                                                        const double* __restrict__ y, int64_t N, int d, int link,
                                                        const double* __restrict__ theta, const double* __restrict__ V,
                                                        double* __restrict__ curv, double* __restrict__ ll_part,
                                                        double* __restrict__ grad_part, double* __restrict__ hvp_part) {
  __shared__ double rs[kPointRows];
  __shared__ double ts[kPointRows][K > 0 ? K : 1];
  __shared__ double red[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double accg[kPointMaxCols], acch[kPointMaxCols][K > 0 ? K : 1];
#pragma unroll
  for (int m = 0; m < kPointMaxCols; ++m) {
    accg[m] = 0.0;
#pragma unroll
    for (int k = 0; k < (K > 0 ? K : 1); ++k) acch[m][k] = 0.0;
  }
  double ll_acc = 0.0;
  const int64_t tiles = (N + kPointRows - 1) / kPointRows;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t n0 = tile * kPointRows;
    // phase A: one warp per 4 rows -- dot products with theta and the K vectors
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int row = warp * 4 + rr;
      const int64_t n = n0 + row;
      double dot = 0.0, dv[K > 0 ? K : 1];
#pragma unroll
      for (int k = 0; k < (K > 0 ? K : 1); ++k) dv[k] = 0.0;
      if (n < N) {
        const double* xr = X + n * ldx;
        for (int j = lane; j < d; j += 32) {
          const double xv = xr[j];
          dot += xv * theta[j];
#pragma unroll
          for (int k = 0; k < K; ++k) dv[k] += xv * V[(size_t)k * d + j];
        }
      }
      dot = warp_sum(dot);
#pragma unroll
      for (int k = 0; k < K; ++k) dv[k] = warp_sum(dv[k]);
      if (lane == 0) {
        double r = 0.0, c = 0.0;
        if (n < N) {
          const double yv = y[n], a = yv * dot;
          double ll, dl;
          if (link == VB_LINK_LOGISTIC) {
            link_logistic(a, ll, dl);
            c = logistic_curvature(a);                 // sigmoid(a) sigmoid(-a)
          } else {
            link_probit(a, ll, dl);
            c = probit_curvature(a, dl);               // -(log Phi)'' = r (a + r)
          }
          ll_acc += ll;
          r = yv * dl;
          if (curv) curv[n] = c;
        }
        rs[row] = r;
#pragma unroll
        for (int k = 0; k < K; ++k) ts[row][k] = c * dv[k];
      }
    }
    __syncthreads();
    // phase B: thread owns columns tid + 256 m; the tile's rows were just read (L1 / L2 hits)
    const int rows = (int)((N - n0) < kPointRows ? (N - n0) : kPointRows);
#pragma unroll
    for (int m = 0; m < kPointMaxCols; ++m) {
      const int j = threadIdx.x + 256 * m;
      if (j < d) {
        for (int row = 0; row < rows; ++row) {
          const double xv = X[(n0 + row) * ldx + j];
          accg[m] += xv * rs[row];
#pragma unroll
          for (int k = 0; k < K; ++k) acch[m][k] += xv * ts[row][k];
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int m = 0; m < kPointMaxCols; ++m) {
    const int j = threadIdx.x + 256 * m;
    if (j < d) {
      grad_part[(size_t)blockIdx.x * d + j] = accg[m];
#pragma unroll
      for (int k = 0; k < K; ++k) hvp_part[((size_t)blockIdx.x * K + k) * d + j] = -acch[m][k];
    }
  }
  ll_acc = block_sum(ll_acc, red);
  if (threadIdx.x == 0) ll_part[blockIdx.x] = ll_acc;
}

// out[i] = sum_b part[b][i], i < n (fixed order)
__global__ void point_reduce_kernel(const double* __restrict__ part, int nblk, int64_t n, double* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  double t = 0.0;
  for (int b = 0; b < nblk; ++b) t += part[(size_t)b * n + i];
  out[i] = t;
}

struct PointPlan {
  int grid;
  size_t off_ll, off_grad, off_hvp, off_curv, off_syrk, total;
};

static void point_plan(int64_t N, int d, int K, int want_hessian, PointPlan& p) {
  const int64_t tiles = (N + kPointRows - 1) / kPointRows;
  int grid = 2 * sm_count();
  if (tiles < grid) grid = (int)(tiles < 1 ? 1 : tiles);
  p.grid = grid;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  p.off_ll = take(sizeof(double) * grid);
  p.off_grad = take(sizeof(double) * (size_t)grid * d);
  p.off_hvp = take(sizeof(double) * (size_t)grid * (K > 0 ? K : 1) * d);
  p.off_curv = take(want_hessian ? sizeof(double) * (size_t)(N > 0 ? N : 1) : 8);
  p.off_syrk = off;
  if (want_hessian) {
    SyrkPlan s;
    syrk_plan(N, d, s);
    off += s.bytes;
  }
  p.total = off;
}

template <int K>
static int launch_point(const PointPlan& p, const double* X, int64_t ldx, const double* y, int64_t N, int d, int link,
                        const double* theta, const double* V, double* curv, double* llp, double* gp, double* hp,
                        cudaStream_t stream) {
  glm_point_kernel<K><<<p.grid, 256, 0, stream>>>(X, ldx, y, N, d, link, theta, V, curv, llp, gp, hp);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

}  // namespace vb
using namespace vb;

extern "C" size_t vb_glm_point_workspace_bytes(int64_t N, int d, int K, int want_hessian) {
  if (N < 0 || d <= 0 || K < 0 || K > kPointMaxK) return 0;
  PointPlan p;
  point_plan(N, d, K, want_hessian, p);
  return p.total;
}

extern "C" int vb_glm_point_f64(const double* X, int64_t ldx, const double* y, int64_t N, int d, int link,
                                const double* theta, const double* V, int K, double* out_ll, double* out_grad,
                                double* out_hvp, double* out_hessian, void* workspace, size_t workspace_bytes,
                                cudaStream_t stream) {
  if (!X || !y || !theta || N < 0 || d <= 0 || ldx < d || !out_grad)
    return set_error(VB_ERR_INVALID_ARG, "glm_point: bad arguments");
  if (link != VB_LINK_LOGISTIC && link != VB_LINK_PROBIT) return set_error(VB_ERR_UNSUPPORTED, "glm_point: logistic / probit links only");
  if (K < 0 || K > kPointMaxK || (K > 0 && (!V || !out_hvp))) return set_error(VB_ERR_INVALID_ARG, "glm_point: 0 <= K <= 8 vectors");
  if (K > 4 && K < 8) return set_error(VB_ERR_UNSUPPORTED, "glm_point: K must be 0..4 or 8");
  if (d > 256 * kPointMaxCols) return set_error(VB_ERR_UNSUPPORTED, "glm_point: d > 2048 not supported");
  PointPlan p;
  point_plan(N, d, K, out_hessian != nullptr, p);
  if (!workspace || workspace_bytes < p.total) return set_error(VB_ERR_WORKSPACE, "glm_point: workspace too small");
  char* ws = static_cast<char*>(workspace);
  double* llp = reinterpret_cast<double*>(ws + p.off_ll);
  double* gp = reinterpret_cast<double*>(ws + p.off_grad);
  double* hp = reinterpret_cast<double*>(ws + p.off_hvp);
  double* curv = out_hessian ? reinterpret_cast<double*>(ws + p.off_curv) : nullptr;
  int rc;
  switch (K) {
    case 0: rc = launch_point<0>(p, X, ldx, y, N, d, link, theta, V, curv, llp, gp, hp, stream); break;
    case 1: rc = launch_point<1>(p, X, ldx, y, N, d, link, theta, V, curv, llp, gp, hp, stream); break;
    case 2: rc = launch_point<2>(p, X, ldx, y, N, d, link, theta, V, curv, llp, gp, hp, stream); break;
    case 3: rc = launch_point<3>(p, X, ldx, y, N, d, link, theta, V, curv, llp, gp, hp, stream); break;
    case 4: rc = launch_point<4>(p, X, ldx, y, N, d, link, theta, V, curv, llp, gp, hp, stream); break;
    default: rc = launch_point<8>(p, X, ldx, y, N, d, link, theta, V, curv, llp, gp, hp, stream); break;
  }
  if (rc) return rc;
  point_reduce_kernel<<<(d + 255) / 256, 256, 0, stream>>>(gp, p.grid, d, out_grad);
  VB_CHECK_LAUNCH();
  if (K > 0) {
    point_reduce_kernel<<<(unsigned)(((int64_t)K * d + 255) / 256), 256, 0, stream>>>(hp, p.grid, (int64_t)K * d, out_hvp);
    VB_CHECK_LAUNCH();
  }
  if (out_ll) {
    point_reduce_kernel<<<1, 32, 0, stream>>>(llp, p.grid, 1, out_ll);
    VB_CHECK_LAUNCH();
  }
  if (out_hessian) {
    if (N == 0) {
      VB_CUDA(cudaMemsetAsync(out_hessian, 0, sizeof(double) * (size_t)d * d, stream));
    } else {
      rc = syrk_f64(X, N, d, ldx, curv, nullptr, -1.0, 0.0, out_hessian, ws + p.off_syrk, workspace_bytes - p.off_syrk, stream);
      if (rc) return rc;
    }
  }
  return VB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Per-sample GLM gradients (full-rank / low-rank / flow families need grad f(theta_s) for EVERY sample: their
// cotangents are not sums over s).  G[S,d] = sum_n y_n r[n,s] x_n is a GEMM with K = N, so the path is
//   A[Nc,S] = y . (X_c Theta^T)      vb_gemm_f64 (row scaling fused)
//   link     (this kernel)           ll[s] += sum_n loglik(A[n,s]);  A[n,s] <- y_n dloglik/da
//   G       += A^T X_c               vb_gemm_f64 (transposed A)
// over row chunks (the reference runs the user's numpy log density under autograd: models.py:27-39).  The link kernel
// is elementwise over the chunk with deterministic column sums: block = 32 columns x 8 row groups, per-block partials,
// a finishing kernel adds them in block order.  The (column block, row block) CTAs are numbered column-fastest on a
// 1-D grid, so Nc is not capped by gridDim.y's 65535 row blocks.
// ---------------------------------------------------------------------------------------------------------------
namespace vb {

constexpr int kLinkRowsPerBlock = 512;

__global__ void __launch_bounds__(256) glm_link_kernel(double* __restrict__ A, const double* __restrict__ y, int64_t Nc, int S,
                                                       int link, double* __restrict__ part) {
  __shared__ double red[8][33];
  const int cx = threadIdx.x & 31, rg = threadIdx.x >> 5;
  const unsigned ncb = (unsigned)ceil_div(S, 32);
  const unsigned rb = blockIdx.x / ncb;
  const int s = (int)(blockIdx.x % ncb) * 32 + cx;
  const int64_t r0 = (int64_t)rb * kLinkRowsPerBlock;
  const int64_t r1 = r0 + kLinkRowsPerBlock < Nc ? r0 + kLinkRowsPerBlock : Nc;
  double acc = 0.0;
  if (s < S) {
    for (int64_t r = r0 + rg; r < r1; r += 8) {
      const double a = A[r * S + s];
      double ll, dl;
      if (link == VB_LINK_LOGISTIC) link_logistic(a, ll, dl);
      else link_probit(a, ll, dl);
      acc += ll;
      A[r * S + s] = y[r] * dl;
    }
  }
  red[rg][cx] = acc;
  __syncthreads();
  if (rg == 0 && s < S) {
    double t = 0.0;
#pragma unroll
    for (int g = 0; g < 8; ++g) t += red[g][cx];
    part[(size_t)rb * S + s] = t;
  }
}

__global__ void glm_link_finish_kernel(const double* __restrict__ part, int nblk, int S, double* __restrict__ ll) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  double t = 0.0;
  for (int b = 0; b < nblk; ++b) t += part[(size_t)b * S + s];
  ll[s] += t;
}

}  // namespace vb

extern "C" size_t vb_glm_link_workspace_bytes(int64_t Nc, int S) {
  if (Nc <= 0 || S <= 0) return 0;
  return (size_t)((Nc + vb::kLinkRowsPerBlock - 1) / vb::kLinkRowsPerBlock) * S * sizeof(double);
}

extern "C" int vb_glm_link_f64(double* A, const double* y, int64_t Nc, int S, int link, double* ll_accum, void* workspace,
                               size_t workspace_bytes, cudaStream_t stream) {
  using namespace vb;
  if (!A || !y || !ll_accum || Nc <= 0 || S <= 0) return set_error(VB_ERR_INVALID_ARG, "glm_link: bad arguments");
  if (link != VB_LINK_LOGISTIC && link != VB_LINK_PROBIT) return set_error(VB_ERR_UNSUPPORTED, "glm_link: logistic or probit");
  if (!workspace || workspace_bytes < vb_glm_link_workspace_bytes(Nc, S)) return set_error(VB_ERR_WORKSPACE, "glm_link: workspace too small");
  const int64_t nblk = ceil_div(Nc, kLinkRowsPerBlock);
  const int64_t ctas = ceil_div(S, 32) * nblk;
  if (ctas > INT32_MAX) return set_error(VB_ERR_UNSUPPORTED, "glm_link: more than 2^31 - 1 (column, row) blocks");
  double* part = static_cast<double*>(workspace);
  glm_link_kernel<<<(unsigned)ctas, 256, 0, stream>>>(A, y, Nc, S, link, part);
  VB_CHECK_LAUNCH();
  glm_link_finish_kernel<<<(S + 127) / 128, 128, 0, stream>>>(part, (int)nblk, S, ll_accum);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
