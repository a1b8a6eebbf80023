// Hierarchical linear regression plugin (BASELINE.json configs[3]; SURVEY.md 8(d) C4) with PER-SAMPLE gradients,
// which the full-rank families need (the d x d cotangent uses every sample's gradient):
//
//   y_i ~ N(x_i . beta_{g(i)}, sigma),  beta_g ~ N(m, tau I),  m ~ N(0, 10 I),  log tau ~ N(0,1),  log sigma ~ N(0,1)
//   theta = [beta (G*p, group-major), m (p), log tau, log sigma],   D = G p + p + 2
//
// The reference evaluates user Python under autograd (models.py:27-39).  Here the observations are stored sorted by
// group (rows goff[g] .. goff[g+1]-1 belong to group g) and the likelihood is a GROUPED contraction: one CTA per
// (group, 128 samples) stages the group's rows in shared memory, each thread owns one sample and keeps its p
// coefficients and p gradient accumulators in registers -- 4 N p S flops instead of the 4 N (G p) S of a
// block-expanded dense design matrix.  p <= 32.  The (group, sample tile) CTAs are numbered group-fastest on a 1-D
// grid, so S is not capped by gridDim.y's 65535.
#include "common.cuh"

namespace vb {

constexpr int kHierP = 32, kHierRows = 64, kHierThreads = 128;

__global__ void __launch_bounds__(kHierThreads) hier_lik_kernel(const double* __restrict__ X, const double* __restrict__ y,
                                                                const long long* __restrict__ goff, int p, int G, int D,
                                                                const double* __restrict__ theta, int S, int want_grad,
                                                                double* __restrict__ ssr_part, double* __restrict__ grad) {
  __shared__ double xs[kHierRows][kHierP + 1];
  __shared__ double ys[kHierRows];
  const int g = (int)(blockIdx.x % (unsigned)G);
  const int s = (int)(blockIdx.x / (unsigned)G) * kHierThreads + threadIdx.x;
  const bool active = s < S;
  double beta[kHierP], acc[kHierP];
#pragma unroll
  for (int j = 0; j < kHierP; ++j) {
    beta[j] = (active && j < p) ? theta[(size_t)s * D + (size_t)g * p + j] : 0.0;
    acc[j] = 0.0;
  }
  double ssr = 0.0;
  const long long r0 = goff[g], r1 = goff[g + 1];
  for (long long rb = r0; rb < r1; rb += kHierRows) {
    const int rows = (int)((r1 - rb) < kHierRows ? (r1 - rb) : kHierRows);
    __syncthreads();
    for (int idx = threadIdx.x; idx < rows * p; idx += kHierThreads) {
      const int r = idx / p, j = idx - r * p;
      xs[r][j] = X[(size_t)(rb + r) * p + j];
    }
    for (int r = threadIdx.x; r < rows; r += kHierThreads) ys[r] = y[rb + r];
    __syncthreads();
    if (active) {
      for (int r = 0; r < rows; ++r) {
        double e = ys[r];
#pragma unroll
        for (int j = 0; j < kHierP; ++j)
          if (j < p) e -= xs[r][j] * beta[j];
        ssr += e * e;
        if (want_grad) {
#pragma unroll
          for (int j = 0; j < kHierP; ++j)
            if (j < p) acc[j] += xs[r][j] * e;
        }
      }
    }
  }
  if (!active) return;
  ssr_part[(size_t)g * S + s] = ssr;
  if (want_grad) {
#pragma unroll
    for (int j = 0; j < kHierP; ++j)
      if (j < p) grad[(size_t)s * D + (size_t)g * p + j] = acc[j];        // raw sum_i x_ij (y_i - x_i . beta); scaled below
  }
}

// one block per sample: priors, log density, and the remaining gradient entries
__global__ void __launch_bounds__(256) hier_finish_kernel(const double* __restrict__ theta, int S, int p, int G, int D, long long N,
                                                          const double* __restrict__ ssr_part, int want_grad,
                                                          double* __restrict__ lp, double* __restrict__ grad) {
  __shared__ double red[32];
  __shared__ double msum[kHierP];
  const int s = blockIdx.x;
  const double* th = theta + (size_t)s * D;
  const double c = 0.5 * kLog2Pi;
  const double ltau = th[G * p + p], lsig = th[G * p + p + 1];
  const double inv_sig = exp(-lsig), inv_tau = exp(-ltau);
  if (threadIdx.x < kHierP) msum[threadIdx.x] = 0.0;
  __syncthreads();
  double ssr = 0.0;
  for (int g = threadIdx.x; g < G; g += blockDim.x) ssr += ssr_part[(size_t)g * S + s];
  ssr = block_sum(ssr, red) * inv_sig * inv_sig;
  double ssb = 0.0, sm2 = 0.0;
  for (int idx = threadIdx.x; idx < G * p; idx += blockDim.x) {
    const int j = idx % p;
    const double db = (th[idx] - th[G * p + j]) * inv_tau;
    ssb += db * db;
    if (want_grad) grad[(size_t)s * D + idx] = grad[(size_t)s * D + idx] * inv_sig * inv_sig - db * inv_tau;
  }
  ssb = block_sum(ssb, red);
  if (want_grad) {
    // d/dm_j: sum_g db_gj / tau - m_j / 100 (fixed order over the groups)
    for (int j = threadIdx.x; j < p; j += blockDim.x) {
      double t = 0.0;
      for (int g = 0; g < G; ++g) t += (th[(size_t)g * p + j] - th[G * p + j]) * inv_tau;
      grad[(size_t)s * D + G * p + j] = t * inv_tau - th[G * p + j] / 100.0;
    }
  }
  for (int j = threadIdx.x; j < p; j += blockDim.x) {
    const double mj = th[G * p + j] / 10.0;
    sm2 += mj * mj;
  }
  sm2 = block_sum(sm2, red);
  if (threadIdx.x == 0) {
    lp[s] = -0.5 * ssr - (double)N * (lsig + c) - 0.5 * ssb - (double)(G * p) * (ltau + c) - 0.5 * sm2 -
            (double)p * (log(10.0) + c) - 0.5 * ltau * ltau - c - 0.5 * lsig * lsig - c;
    if (want_grad) {
      grad[(size_t)s * D + G * p + p] = ssb - (double)(G * p) - ltau;
      grad[(size_t)s * D + G * p + p + 1] = ssr - (double)N - lsig;
    }
  }
}

}  // namespace vb
using namespace vb;

extern "C" size_t vb_hier_workspace_bytes(int G, int S) { return G > 0 && S > 0 ? sizeof(double) * (size_t)G * S : 0; }

/* X[N,p], y[N] sorted by group, goff[G+1] (device int64) row offsets; theta[S,D], D = G p + p + 2;
 * out_lp[S], out_grad[S,D] (optional). */
extern "C" int vb_hier_logp_grad_f64(const double* X, const double* y, const int64_t* goff, int64_t N, int p, int G,
                                     const double* theta, int S, double* out_lp, double* out_grad, void* workspace,
                                     size_t workspace_bytes, cudaStream_t stream) {
  if (!X || !y || !goff || N < 0 || p <= 0 || G <= 0 || !theta || S <= 0 || !out_lp)
    return set_error(VB_ERR_INVALID_ARG, "hier_logp_grad: bad arguments");
  if (p > kHierP) return set_error(VB_ERR_UNSUPPORTED, "hier_logp_grad: at most 32 coefficients per group");
  if (!workspace || workspace_bytes < vb_hier_workspace_bytes(G, S)) return set_error(VB_ERR_WORKSPACE, "hier_logp_grad: workspace too small");
  const int D = G * p + p + 2;
  double* ssr_part = static_cast<double*>(workspace);
  const int64_t ctas = (int64_t)G * ceil_div(S, kHierThreads);
  if (ctas > INT32_MAX) return set_error(VB_ERR_UNSUPPORTED, "hier_logp_grad: more than 2^31 - 1 (group, sample tile) pairs");
  hier_lik_kernel<<<(unsigned)ctas, kHierThreads, 0, stream>>>(
      X, y, reinterpret_cast<const long long*>(goff), p, G, D, theta, S, out_grad != nullptr, ssr_part, out_grad);
  VB_CHECK_LAUNCH();
  hier_finish_kernel<<<S, 256, 0, stream>>>(theta, S, p, G, D, (long long)N, ssr_part, out_grad != nullptr, out_lp, out_grad);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
