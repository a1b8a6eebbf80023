// Distilled importance sampling objective (DISInclusiveKL, reference objectives.py:283-416) -- forward-only in the
// model; the device work is on S-vectors of weights and on the score terms of log q at FIXED samples:
//   vb_dis_bisection_f64  the 50-round bisection on the tempering epsilon so that the effective sample size of
//                         w = exp(eps * log_prior + (1 - eps) * log_p - log_q) meets ess_target (:317-366, weights NOT
//                         max-shifted, as the reference), in ONE launch (the reference does 51 numpy passes)
//   vb_mf_score_f64       value = -sum_r c_r log q(x_r; lambda) and its gradient wrt [mu, log sigma] (:405-416; autograd
//                         differentiates approx.log_density there), c_r = scale * w[r], rows optionally gathered by idx
#include "common.cuh"

namespace vb {

__global__ void __launch_bounds__(1024) dis_bisection_kernel(const double* __restrict__ log_prior, const double* __restrict__ log_p,
                                                             const double* __restrict__ log_q, int64_t S, double eps_guess,
                                                             double max_eps, double ess_target, int max_its,
                                                             double* __restrict__ w, double* __restrict__ out) {
  __shared__ double red[32];
  double lower = 0.0, upper = eps_guess, eps = (lower + upper) / 2.0;
  double ess = 0.0, sw = 0.0;
  bool all_zero = false;
  for (int it = 0; it <= max_its; ++it) {
    double a = 0.0, b = 0.0, mx = -INFINITY;
    for (int64_t s = threadIdx.x; s < S; s += blockDim.x) {
      const double lw = eps * log_prior[s] + (1.0 - eps) * log_p[s] - log_q[s];
      const double v = exp(lw);
      mx = fmax(mx, lw);
      a += v;
      b += v * v;
      if (it == max_its) w[s] = v;
    }
    a = block_sum(a, red);
    b = block_sum(b, red);
    mx = block_max(mx, red);
    if (mx == -INFINITY) all_zero = true;          // 'All weights zero!' (:323-325)
    ess = (a * a) / b;
    sw = a;
    if (it == max_its) break;
    if (ess > ess_target) upper = eps;
    else lower = eps;
    eps = (lower + upper) / 2.0;
  }
  // extreme values if they are still end points (:362-366); the weights stay those of the last midpoint
  if (lower == 0.0) eps = 0.0;
  if (upper == max_eps) eps = max_eps;
  if (threadIdx.x == 0) {
    out[0] = eps;
    out[1] = ess;
    out[2] = all_zero ? 1.0 : 0.0;
    out[3] = sw;
  }
}

constexpr int kScoreGroups = 32;

// block = 32 columns x 32 row groups; out: grad[j], grad[d + j] and one partial of the value per block
__global__ void __launch_bounds__(32 * kScoreGroups) mf_score_kernel(const double* __restrict__ vp, const double* __restrict__ x,
                                                                     const long long* __restrict__ idx, const double* __restrict__ w,
                                                                     double scale, int64_t n, int d, int family, double df,
                                                                     double tconst, double* __restrict__ grad,
                                                                     double* __restrict__ val_part) {
  __shared__ double sm[3][kScoreGroups][33];
  __shared__ double red[32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  double gm = 0.0, gl = 0.0, val = 0.0;
  if (j < d) {
    const double mu = vp[j], ls = vp[d + j], sig = exp(ls);
    for (int64_t r = ty; r < n; r += kScoreGroups) {
      const int64_t s = idx ? idx[r] : r;
      const double c = scale * (w ? w[r] : 1.0);
      const double z = (x[s * d + j] - mu) / sig;
      double lq, dmu, dls;
      if (family == VB_FAMILY_MF_GAUSSIAN) {
        lq = -0.5 * z * z - ls - 0.5 * kLog2Pi;
        dmu = z / sig;
        dls = z * z - 1.0;
      } else {
        const double q = (df + 1.0) / (df + z * z);
        lq = tconst - 0.5 * (df + 1.0) * log1p(z * z / df) - ls;
        dmu = q * z / sig;
        dls = q * z * z - 1.0;
      }
      val -= c * lq;
      gm -= c * dmu;
      gl -= c * dls;
    }
  }
  sm[0][ty][tx] = gm; sm[1][ty][tx] = gl; sm[2][ty][tx] = val;
  __syncthreads();
  double v = 0.0;
  if (ty == 0) {
    double a = 0.0, b = 0.0;
#pragma unroll
    for (int r = 0; r < kScoreGroups; ++r) { a += sm[0][r][tx]; b += sm[1][r][tx]; v += sm[2][r][tx]; }
    if (j < d) {
      grad[j] = a;
      grad[d + j] = b;
    }
  }
  v = block_sum(v, red);
  if (threadIdx.x == 0) val_part[blockIdx.x] = v;
}

__global__ void sum_small_kernel(const double* __restrict__ part, int n, double* __restrict__ out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < n; ++i) t += part[i];
    out[0] = t;
  }
}

}  // namespace vb
using namespace vb;

extern "C" int vb_dis_bisection_f64(const double* log_prior, const double* log_p, const double* log_q, int64_t S,
                                    double eps_guess, double max_eps, double ess_target, int max_its, double* w,
                                    double* out4, cudaStream_t stream) {
  if (!log_prior || !log_p || !log_q || S <= 0 || max_its < 0 || !w || !out4)
    return set_error(VB_ERR_INVALID_ARG, "dis_bisection: bad arguments");
  dis_bisection_kernel<<<1, 1024, 0, stream>>>(log_prior, log_p, log_q, S, eps_guess, max_eps, ess_target, max_its, w, out4);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

extern "C" size_t vb_mf_score_workspace_bytes(int d) { return d > 0 ? sizeof(double) * (size_t)((d + 31) / 32) : 0; }

extern "C" int vb_mf_score_f64(const double* var_param, const double* x, const int64_t* idx, const double* w, double scale,
                               int64_t n, int d, int family, double df, double* value, double* grad, void* workspace,
                               size_t workspace_bytes, cudaStream_t stream) {
  if (!var_param || !x || n <= 0 || d <= 0 || !value || !grad) return set_error(VB_ERR_INVALID_ARG, "mf_score: bad arguments");
  if (family != VB_FAMILY_MF_GAUSSIAN && family != VB_FAMILY_MF_STUDENT) return set_error(VB_ERR_INVALID_ARG, "unknown mean-field family");
  if (family == VB_FAMILY_MF_STUDENT && !(df > 2.0)) return set_error(VB_ERR_INVALID_ARG, "df must be greater than 2");
  const int nb = (d + 31) / 32;
  if (!workspace || workspace_bytes < vb_mf_score_workspace_bytes(d)) return set_error(VB_ERR_WORKSPACE, "mf_score: workspace too small");
  const double tc = family == VB_FAMILY_MF_STUDENT ? student_t_log_const(df) : 0.0;
  double* part = static_cast<double*>(workspace);
  mf_score_kernel<<<nb, 32 * kScoreGroups, 0, stream>>>(var_param, x, reinterpret_cast<const long long*>(idx), w, scale, n, d,
                                                        family, df, tc, grad, part);
  VB_CHECK_LAUNCH();
  sum_small_kernel<<<1, 32, 0, stream>>>(part, nb, value);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
