// Product-target model plugins: log density and PER-SAMPLE gradient of
//   kind 0:  sum_j N(theta_j; loc_j, scale_j)            (the reference tests' Gaussian target, tests/test_objectives.py:18-19)
//   kind 1:  sum_j t_df(theta_j; loc_j, scale_j)         (SURVEY.md 8(d) C5: product Student-t target)
// at S sample points theta[S,d] in one launch (north_star: "Gaussian/Student-t targets" as GPU-resident model plugins).
// In the reference these are user Python under autograd (models.py:27-39, objectives.py:161-167).  One warp per sample
// row: coalesced reads of theta, coalesced writes of the gradient row, a warp reduction for log p.  HBM bound
// (16 S d bytes), O(S d) flops; the streamed form used by vi_diagnostics at scale is stream_lw.cu.
#include "stream_internal.cuh"

namespace vb {

__global__ void __launch_bounds__(256) target_logp_grad_kernel(const double* __restrict__ theta, int64_t S, int d, int kind,
                                                               const double* __restrict__ loc,
                                                               const double* __restrict__ scale, double df, double cst,
                                                               double* __restrict__ logp, double* __restrict__ grad) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t s = warp; s < S; s += nwarps) {
    double lp = 0.0;
    for (int j = lane; j < d; j += 32) {
      const double sc = scale[j];
      const double z = (theta[s * d + j] - loc[j]) / sc;
      if (kind == 0) {
        lp += product_target_term(0, z, df);
        if (grad) grad[s * d + j] = -z / sc;
      } else {
        lp += product_target_term(1, z, df);
        if (grad) grad[s * d + j] = -(df + 1.0) * z / ((df + z * z) * sc);
      }
    }
    lp = warp_sum(lp);
    if (lane == 0) logp[s] = lp + cst;
  }
}

}  // namespace vb

using namespace vb;

extern "C" int vb_target_logp_grad_f64(const double* theta, int64_t S, int d, int kind, const double* loc,
                                       const double* scale, double df, double log_norm_const, double* logp, double* grad,
                                       cudaStream_t stream) {
  if (!theta || !logp || S <= 0 || d <= 0) return set_error(VB_ERR_INVALID_ARG, "target_logp_grad: bad arguments");
  const int rc = check_product_target("target_logp_grad", kind, false, loc, scale, df);
  if (rc) return rc;
  int64_t blocks = (S + 7) / 8;                     // 8 warps per CTA, one sample row per warp
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  target_logp_grad_kernel<<<(unsigned)blocks, 256, 0, stream>>>(theta, S, d, kind, loc, scale, df, log_norm_const, logp, grad);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
