// Mean-field families (MFGaussian / MFStudentT) and the objective assembly around the GLM sweep.
// var_param = [mu(d), log_sigma(d)]  (reference approximations.py:185-189).
#include "common.cuh"

namespace vb {

// theta = mu + exp(log_sigma) * base   (approximations.py:212-216, :270-274)
__global__ void mf_sample_kernel(const double* __restrict__ vp, const double* __restrict__ base,
                                 double* __restrict__ theta, int64_t S, int d) {
  PDL_SYNC();
  const int64_t total = S * d;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(i % d);
    theta[i] = vp[j] + exp(vp[d + j]) * base[i];
  }
}

// one warp per row: sum_j logpdf((x-mu)/sigma) - log_sigma   (approximations.py:231-236, :281-286)
__global__ void mf_log_density_kernel(const double* __restrict__ vp, const double* __restrict__ x,
                                      int64_t n, int d, int family, double df, double tconst,
                                      double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < n; i += nwarps) {
    double acc = 0.0;
    for (int j = lane; j < d; j += 32) {
      const double ls = vp[d + j];
      const double z = (x[i * d + j] - vp[j]) / exp(ls);   // same op order as scipy: (x-loc)/scale
      if (family == VB_FAMILY_MF_GAUSSIAN)
        acc += -0.5 * z * z - ls - 0.5 * kLog2Pi;
      else
        acc += tconst - 0.5 * (df + 1.0) * log1p(z * z / df) - ls;
    }
    acc = warp_sum(acc);
    if (lane == 0) out[i] = acc;
  }
}

// per-sample pieces: prior_s = log N(theta_s; 0, prior_sd^2 I); logq_s = log q(theta_s) with z = base
// (theta = mu + sigma*base, so the standardised variate IS the base draw)
__device__ __forceinline__ void sample_terms(const double* __restrict__ vp, const double* __restrict__ theta,
                                             const double* __restrict__ base, int64_t s, int d, int family,
                                             double df, double tconst, double inv_tau2, double prior_const,
                                             bool want_logq, int lane, double& prior, double& logq) {
  double sq = 0.0, lq = 0.0;
  for (int j = lane; j < d; j += 32) {
    const double th = theta[s * d + j];
    sq += th * th;
    if (want_logq) {
      const double e = base[s * d + j], ls = vp[d + j];
      if (family == VB_FAMILY_MF_GAUSSIAN)
        lq += -0.5 * e * e - ls - 0.5 * kLog2Pi;
      else
        lq += tconst - 0.5 * (df + 1.0) * log1p(e * e / df) - ls;
    }
  }
  sq = warp_sum(sq);
  lq = warp_sum(lq);
  prior = -0.5 * sq * inv_tau2 + prior_const;
  logq = lq;
}

// lw[s] = ll[s] + prior_s - logq_s   (objectives.py:443-446), one warp per sample
__global__ void mf_log_weights_kernel(const double* __restrict__ vp, const double* __restrict__ theta,
                                      const double* __restrict__ base, const double* __restrict__ ll,
                                      int64_t S, int d, int family, double df, double tconst,
                                      double inv_tau2, double prior_const, double* __restrict__ lw) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t s = warp; s < S; s += nwarps) {
    double prior, logq;
    sample_terms(vp, theta, base, s, d, family, df, tconst, inv_tau2, prior_const, true, lane, prior, logq);
    if (lane == 0) lw[s] = ll[s] + prior - logq;
  }
}

// m = max lw; w = exp(alpha (lw - m)); value = log(mean w)/alpha + m   (objectives.py:457-459)
__global__ void alpha_weights_kernel(const double* __restrict__ lw, int64_t S, double alpha,
                                     double* __restrict__ w, double* __restrict__ value) {
  __shared__ double red[32];
  double m = -INFINITY;
  for (int64_t s = threadIdx.x; s < S; s += blockDim.x) m = fmax(m, lw[s]);
  m = block_max(m, red);
  double acc = 0.0;
  for (int64_t s = threadIdx.x; s < S; s += blockDim.x) {
    const double v = pow(exp(lw[s] - m), alpha);     // np.exp(lw - m) ** alpha
    w[s] = v;
    acc += v;
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) value[0] = log(acc / (double)S) / alpha + m;
}

// value for ExclusiveKL (entropy or path-derivative form) + per-sample model log density
__global__ void __launch_bounds__(256) mf_value_kernel(const double* __restrict__ vp, const double* __restrict__ theta,
                                                       const double* __restrict__ base, const double* __restrict__ ll,
                                                       int64_t S, int d, int family, double df, double tconst,
                                                       double inv_tau2, double prior_const, int objective,
                                                       double* __restrict__ part, double* __restrict__ logp) {
  PDL_SYNC();
  // one warp per sample, 8 samples per block; part[blockIdx.x] receives the block's share of the value
  __shared__ double red[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool path = objective == VB_OBJ_EXCLUSIVE_KL_PATH;
  double acc = 0.0;
  const int64_t s = (int64_t)blockIdx.x * 8 + warp;
  if (s < S) {
    double prior, logq;
    sample_terms(vp, theta, base, s, d, family, df, tconst, inv_tau2, prior_const, path, lane, prior, logq);
    const double f = ll[s] + prior;
    if (lane == 0) {
      if (logp) logp[s] = f;
      acc = path ? (f - logq) : f;
    }
  }
  if (objective == VB_OBJ_ALPHA) return;    // value comes from alpha_weights_kernel
  acc = block_sum(acc, red);
  double H = 0.0;
  if (blockIdx.x == 0 && !path) {
    for (int j = threadIdx.x; j < d; j += blockDim.x) H += vp[d + j];
    H = block_sum(H, red);
    if (family == VB_FAMILY_MF_GAUSSIAN) H += 0.5 * d * (1.0 + kLog2Pi);   // approximations.py:218-220
  }
  if (threadIdx.x == 0) part[blockIdx.x] = -(acc / (double)S + H);
}

// value[0] = sum of the n block shares of mf_value_kernel, in a fixed order (one block): deterministic
__global__ void __launch_bounds__(256) mf_value_sum_kernel(const double* __restrict__ part, int64_t n,
                                                           double* __restrict__ value) {
  PDL_SYNC();
  __shared__ double red[32];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += part[i];
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) value[0] = acc;
}

// gradient wrt [mu, log_sigma]  (SURVEY.md App. A.1): block = 32 coordinates x 8 sample groups
__global__ void __launch_bounds__(256) mf_grad_kernel(const double* __restrict__ vp, const double* __restrict__ theta,
                                                      const double* __restrict__ base, const double* __restrict__ gmu,
                                                      const double* __restrict__ ge, const double* __restrict__ w,
                                                      int64_t S, int d, int family, double df, double inv_tau2,
                                                      int objective, double alpha, double* __restrict__ grad) {
  PDL_SYNC();
  __shared__ double sm[5][8][33];
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + x;
  double p1 = 0.0, p2 = 0.0, pa = 0.0, pb = 0.0, sw = 0.0;
  if (j < d) {
    for (int64_t s = y; s < S; s += 8) {
      const double ws = w ? w[s] : 1.0;
      const double th = theta[s * d + j], e = base[s * d + j];
      p1 += ws * th;
      p2 += ws * th * e;
      sw += ws;
      if (objective == VB_OBJ_EXCLUSIVE_KL_PATH) {
        if (family == VB_FAMILY_MF_GAUSSIAN) {
          pa += e;
          pb += e * e;
        } else {
          const double q = (df + 1.0) / (df + e * e);
          pa += q * e;
          pb += q * e * e;
        }
      }
    }
  }
  sm[0][y][x] = p1; sm[1][y][x] = p2; sm[2][y][x] = pa; sm[3][y][x] = pb; sm[4][y][x] = sw;
  __syncthreads();
  if (y != 0 || j >= d) return;
  p1 = p2 = pa = pb = sw = 0.0;
#pragma unroll
  for (int r = 0; r < 8; ++r) {            // fixed order: deterministic
    p1 += sm[0][r][x]; p2 += sm[1][r][x]; pa += sm[2][r][x]; pb += sm[3][r][x]; sw += sm[4][r][x];
  }
  const double sig = exp(vp[d + j]);
  const double a = gmu[j] - p1 * inv_tau2;          // sum_s w_s g_s[j]
  const double b = ge[j] - p2 * inv_tau2;           // sum_s w_s g_s[j] e_s[j]
  const double invS = 1.0 / (double)S;
  if (objective == VB_OBJ_EXCLUSIVE_KL) {
    grad[j] = -invS * a;
    grad[d + j] = -invS * b * sig - 1.0;
  } else if (objective == VB_OBJ_EXCLUSIVE_KL_PATH) {
    grad[j] = -invS * (a + pa / sig);
    grad[d + j] = -invS * (b * sig + pb);
  } else {
    grad[j] = alpha * invS * a;
    grad[d + j] = alpha * invS * (b * sig + sw);
  }
}

static inline void prior_consts(double prior_sd, int d, double& inv_tau2, double& prior_const) {
  if (prior_sd > 0.0 && isfinite(prior_sd)) {
    inv_tau2 = 1.0 / (prior_sd * prior_sd);
    prior_const = -(double)d * log(prior_sd * sqrt(2.0 * 3.14159265358979323846));
  } else {      // flat prior
    inv_tau2 = 0.0;
    prior_const = 0.0;
  }
}

static inline int grid_for(int64_t n, int threads) {
  int64_t b = (n + threads - 1) / threads;
  int64_t cap = (int64_t)sm_count() * 16;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace vb
using namespace vb;

static int check_family(int family, double df) {
  if (family != VB_FAMILY_MF_GAUSSIAN && family != VB_FAMILY_MF_STUDENT)
    return set_error(VB_ERR_INVALID_ARG, "unknown mean-field family");
  if (family == VB_FAMILY_MF_STUDENT && !(df > 2.0))
    return set_error(VB_ERR_INVALID_ARG, "df must be greater than 2");   // approximations.py:258-259
  return VB_OK;
}

extern "C" int vb_mf_sample_f64(const double* var_param, const double* base, double* theta, int64_t S, int d,
                                cudaStream_t stream) {
  if (S < 0 || d <= 0 || !var_param || (S > 0 && (!base || !theta)))
    return set_error(VB_ERR_INVALID_ARG, "mf_sample: bad arguments");
  if (S == 0) return VB_OK;
  VB_CUDA(launch_pdl(mf_sample_kernel, dim3(grid_for(S * d, 256)), dim3(256), stream, var_param, base, theta, S, d));
  return VB_OK;
}

extern "C" int vb_mf_log_density_f64(const double* var_param, const double* x, int64_t n, int d, int family,
                                     double df, double* out, cudaStream_t stream) {
  if (n < 0 || d <= 0 || !var_param || (n > 0 && (!x || !out)))
    return set_error(VB_ERR_INVALID_ARG, "mf_log_density: bad arguments");
  int rc = check_family(family, df);
  if (rc) return rc;
  if (n == 0) return VB_OK;
  const double tc = family == VB_FAMILY_MF_STUDENT ? student_t_log_const(df) : 0.0;
  mf_log_density_kernel<<<grid_for(n * 32, 256), 256, 0, stream>>>(var_param, x, n, d, family, df, tc, out);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

extern "C" int vb_mf_alpha_weights_f64(const double* var_param, const double* theta, const double* base,
                                       const double* ll, int64_t S, int d, int family, double df,
                                       double prior_sd, double alpha, double* lw, double* w, double* value,
                                       cudaStream_t stream) {
  if (S <= 0 || d <= 0 || !var_param || !theta || !base || !ll || !lw || !w || !value)
    return set_error(VB_ERR_INVALID_ARG, "mf_alpha_weights: bad arguments");
  int rc = check_family(family, df);
  if (rc) return rc;
  double inv_tau2, pc;
  prior_consts(prior_sd, d, inv_tau2, pc);
  const double tc = family == VB_FAMILY_MF_STUDENT ? student_t_log_const(df) : 0.0;
  mf_log_weights_kernel<<<grid_for(S * 32, 256), 256, 0, stream>>>(var_param, theta, base, ll, S, d, family, df,
                                                                   tc, inv_tau2, pc, lw);
  VB_CHECK_LAUNCH();
  alpha_weights_kernel<<<1, 1024, 0, stream>>>(lw, S, alpha, w, value);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

extern "C" size_t vb_mf_objective_finish_workspace_bytes(int64_t S) {
  return S > 0 ? sizeof(double) * (size_t)((S + 7) / 8) : 0;
}

extern "C" int vb_mf_objective_finish_f64(const double* var_param, const double* theta, const double* base,
                                          const double* ll, const double* gmu, const double* ge,
                                          const double* w, int64_t S, int d, int family, double df,
                                          double prior_sd, int objective, double alpha, double* value,
                                          double* grad, double* logp, void* workspace, size_t workspace_bytes,
                                          cudaStream_t stream) {
  if (S <= 0 || d <= 0 || !var_param || !theta || !base || !ll)
    return set_error(VB_ERR_INVALID_ARG, "mf_objective_finish: bad arguments");
  if (objective < VB_OBJ_EXCLUSIVE_KL || objective > VB_OBJ_ALPHA)
    return set_error(VB_ERR_INVALID_ARG, "mf_objective_finish: unknown objective");
  if (objective == VB_OBJ_ALPHA && !w)
    return set_error(VB_ERR_INVALID_ARG, "mf_objective_finish: alpha objective needs the sweep weights");
  if (grad && (!gmu || !ge)) return set_error(VB_ERR_INVALID_ARG, "mf_objective_finish: grad needs gmu, ge");
  int rc = check_family(family, df);
  if (rc) return rc;
  double inv_tau2, pc;
  prior_consts(prior_sd, d, inv_tau2, pc);
  const double tc = family == VB_FAMILY_MF_STUDENT ? student_t_log_const(df) : 0.0;
  const bool want_value = objective != VB_OBJ_ALPHA && (value || logp);
  if (want_value) {
    if (!value) return set_error(VB_ERR_INVALID_ARG, "mf_objective_finish: value is required");
    if (!workspace || workspace_bytes < vb_mf_objective_finish_workspace_bytes(S))
      return set_error(VB_ERR_WORKSPACE, "mf_objective_finish: workspace too small");
  }
  if (value || logp) {
    const int64_t nb = (S + 7) / 8;
    double* part = want_value ? static_cast<double*>(workspace) : nullptr;
    VB_CUDA(launch_pdl(mf_value_kernel, dim3((unsigned)nb), dim3(256), stream, var_param, theta, base, ll, S, d, family,
                       df, tc, inv_tau2, pc, objective, part, logp));
    if (want_value) VB_CUDA(launch_pdl(mf_value_sum_kernel, dim3(1), dim3(256), stream, (const double*)part, nb, value));
  }
  if (grad) {
    VB_CUDA(launch_pdl(mf_grad_kernel, dim3((d + 31) / 32), dim3(256), stream, var_param, theta, base, gmu, ge,
                                                         objective == VB_OBJ_ALPHA ? w : nullptr, S, d, family,
                                                         df, inv_tau2, objective, alpha, grad));
  }
  return VB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Reduction of PER-SAMPLE model gradients G[S,d] (a plugin without a fused sweep: targets, hierarchical regression,
// user models) to the two vectors the mean-field gradient assembly needs (SURVEY.md App. A.1):
//   gmu[j] = sum_s w_s G[s,j],   ge[j] = sum_s w_s G[s,j] e[s,j]          (w = 1 when NULL)
// -- the reverse sweep autograd performs through `mu + sigma * eps` in the reference (approximations.py:212-216 under
// objectives.py:161-167).  One block per 32 columns walks all S rows (8 row groups, fixed-order combination):
// deterministic, coalesced 256-byte row segments.
// ---------------------------------------------------------------------------------------------------------------
namespace vb {
__global__ void __launch_bounds__(256) mf_reduce_grads_kernel(const double* __restrict__ G, const double* __restrict__ w,
                                                              const double* __restrict__ e, int64_t S, int d,
                                                              double* __restrict__ gmu, double* __restrict__ ge) {
  __shared__ double r0[8][33], r1[8][33];
  const int cx = threadIdx.x & 31, rg = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + cx;
  double a = 0.0, b = 0.0;
  if (j < d) {
    for (int64_t s = rg; s < S; s += 8) {
      const double g = (w ? w[s] : 1.0) * G[s * d + j];
      a += g;
      b = fma(g, e[s * d + j], b);
    }
  }
  r0[rg][cx] = a;
  r1[rg][cx] = b;
  __syncthreads();
  if (rg == 0 && j < d) {
    double ta = 0.0, tb = 0.0;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      ta += r0[g][cx];
      tb += r1[g][cx];
    }
    gmu[j] = ta;
    ge[j] = tb;
  }
}
}  // namespace vb

extern "C" int vb_mf_reduce_grads_f64(const double* G, const double* w, const double* base, int64_t S, int d, double* gmu,
                                      double* ge, cudaStream_t stream) {
  if (!G || !base || !gmu || !ge || S <= 0 || d <= 0) return set_error(VB_ERR_INVALID_ARG, "mf_reduce_grads: bad arguments");
  mf_reduce_grads_kernel<<<(d + 31) / 32, 256, 0, stream>>>(G, w, base, S, d, gmu, ge);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
