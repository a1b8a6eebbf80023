// Streaming log-weights for vi_diagnostics at scale (reference convenience.py:136-179: samples_and_log_weights
// draws samples[n,d], evaluates log p - log q and hands both to PSIS; at BASELINE configs[4], n = 1e8 and d = 256,
// samples[n,d] alone would be 204.8 GB).  For a mean-field family and a product target (the built-in Gaussian /
// Student-t target plugins) ONE kernel regenerates the family's Philox draws by offset, reparameterises, and
// accumulates log p(theta_i) - log q(theta_i) per draw: nothing but lw[n] (8 bytes per draw) ever reaches HBM.
//   draw i, coordinate j  =  element offset + i*d + j of the family's stream (vb_philox_normal_f64 /
//   vb_philox_student_t_f64), exactly what approx.sample(var_param, n) would have drawn.
// ALU bound (Box-Muller / Marsaglia-Tsang per element), not an HBM kernel.
#include "philox_draws.cuh"
#include "stream_internal.cuh"

namespace vb {

constexpr int kLwMaxDim = 4096;

// one warp per draw; the per-coordinate parameters sit in shared memory
__global__ void __launch_bounds__(256) mf_target_lw_kernel(const double* __restrict__ vp, int64_t n, int d, int family, double df,
                                                           double tconst_q, unsigned long long seed, unsigned long long offset,
                                                           int quantize, int target_kind, const double* __restrict__ loc,
                                                           const double* __restrict__ scale, double target_df, double tconst_p,
                                                           double* __restrict__ lw, double* __restrict__ theta_out) {
  extern __shared__ double sh[];
  double* mu = sh;
  double* sig = sh + d;
  double* tl = sh + 2 * d;
  double* ts = sh + 3 * d;
  double qconst = 0.0, pconst = 0.0;                        // sum_j log sigma_j, sum_j log scale_j
  for (int j = threadIdx.x; j < d; j += blockDim.x) {
    mu[j] = vp[j];
    sig[j] = exp(vp[d + j]);
    tl[j] = loc[j];
    ts[j] = scale[j];
  }
  __syncthreads();
  for (int j = 0; j < d; ++j) {                             // every thread: the same fixed-order sums
    qconst += log(sig[j]);
    pconst += log(ts[j]);
  }
  const Philox ph(seed);
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < n; i += nwarps) {
    double lq = 0.0, lp = 0.0;
    for (int j = lane; j < d; j += 32) {
      const unsigned long long e_idx = offset + (unsigned long long)i * d + j;
      const double e = family == VB_FAMILY_MF_GAUSSIAN ? normal_element(ph, e_idx, quantize)
                                                       : student_element(ph, e_idx, df, quantize);
      const double th = mu[j] + sig[j] * e;
      if (theta_out) theta_out[i * d + j] = th;
      lq += family == VB_FAMILY_MF_GAUSSIAN ? -0.5 * e * e - 0.5 * kLog2Pi
                                            : tconst_q - 0.5 * (df + 1.0) * log1p(e * e / df);
      const double z = (th - tl[j]) / ts[j];
      lp += target_kind == 0 ? product_target_term(0, z, target_df) - 0.5 * kLog2Pi
                             : tconst_p + product_target_term(1, z, target_df);
    }
    lq = warp_sum(lq);
    lp = warp_sum(lp);
    if (lane == 0) lw[i] = (lp - pconst) - (lq - qconst);
  }
}

}  // namespace vb
using namespace vb;

extern "C" int vb_mf_target_log_weights_f64(const double* var_param, int64_t n, int d, int family, double df, uint64_t seed,
                                            uint64_t offset, int quantize, int target_kind, const double* target_loc,
                                            const double* target_scale, double target_df, double* lw, double* theta_out,
                                            cudaStream_t stream) {
  if (!var_param || n < 0 || d <= 0 || (n > 0 && !lw))
    return set_error(VB_ERR_INVALID_ARG, "mf_target_log_weights: bad arguments");
  const int rc = check_product_target("mf_target_log_weights", target_kind, false, target_loc, target_scale, target_df);
  if (rc) return rc;
  if (d > kLwMaxDim) return set_error(VB_ERR_UNSUPPORTED, "mf_target_log_weights: d > 4096 not supported");
  if (family != VB_FAMILY_MF_GAUSSIAN && family != VB_FAMILY_MF_STUDENT) return set_error(VB_ERR_INVALID_ARG, "unknown mean-field family");
  if (family == VB_FAMILY_MF_STUDENT && !(df > 2.0)) return set_error(VB_ERR_INVALID_ARG, "df must be greater than 2");
  if (n == 0) return VB_OK;
  const size_t smem = sizeof(double) * 4 * (size_t)d;
  if (smem > 48 * 1024) VB_CUDA(cudaFuncSetAttribute(mf_target_lw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int64_t blocks = (n * 32 + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  mf_target_lw_kernel<<<(unsigned)blocks, 256, smem, stream>>>(
      var_param, n, d, family, df, family == VB_FAMILY_MF_STUDENT ? student_t_log_const(df) : 0.0, seed, offset, quantize,
      target_kind, target_loc, target_scale, target_df, target_kind == 1 ? student_t_log_const(target_df) : 0.0, lw, theta_out);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
