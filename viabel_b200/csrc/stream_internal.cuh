// Shared by the streamed log-weight kernels (stream_lw.cu, mvt_stream.cu, lr_stream.cu) and the product-target plugin
// (targets.cu): the product target and its argument checks, the tensor-core tile epilogue, the persistent-grid size.
#pragma once
#include <stdio.h>

#include "common.cuh"

namespace vb {

// Product target sum_j log t(theta_j; loc_j, scale_j), kind 0 Gaussian, kind 1 Student-t with df: the term of one
// coordinate at z = (theta_j - loc_j) / scale_j, without the constants.
__device__ __forceinline__ double product_target_term(int kind, double z, double df) {
  return kind == 0 ? -0.5 * z * z : -0.5 * (df + 1.0) * log1p(z * z / df);
}

// d x the per-coordinate constant (0 for kind -1, no target)
inline double product_target_const(int kind, int d, double df) {
  return kind == 0 ? -0.5 * kLog2Pi * d : kind == 1 ? d * student_t_log_const(df) : 0.0;
}

// target_const - sum_j log scale_j, one fixed-order block sum; valid in every thread, contains __syncthreads
__device__ __forceinline__ double product_target_log_const(double target_const, const double* scale, int d, double* red) {
  double a = 0.0;
  for (int j = threadIdx.x; j < d; j += blockDim.x) a += log(scale[j]);
  return target_const - block_sum(a, red);
}

// kind 0 or 1, or -1 (no target) where allow_none; a target needs loc and scale, a Student-t one df > 0
inline int check_product_target(const char* who, int kind, bool allow_none, const double* loc, const double* scale,
                                double df) {
  if (kind >= (allow_none ? -1 : 0) && kind <= 1 && (kind < 0 || (loc && scale)) && (kind != 1 || df > 0.0))
    return VB_OK;
  char msg[200];
  snprintf(msg, sizeof(msg), "%s: the target is kind %s0 (Gaussian, loc, scale) or 1 (Student-t, loc, scale, df > 0)",
           who, allow_none ? "-1 (none), " : "");
  return set_error(VB_ERR_INVALID_ARG, msg);
}

constexpr int kTileM = 32;                   // draws per tile of the full-rank and low-rank kernels
constexpr int kTileN = 128;                  // their theta column block

// Epilogue of a kTileM x kTileN block of theta in mma.sync m8n8k4 accumulators, 8 warps of 16 x 32.  theta_row(r)
// returns the map (n, acc) -> theta of tile row r (draw i0 + r), coordinate n; theta goes to theta_out if asked and the
// target terms are summed over the fragment, over t by two shuffles, then over the four warp columns through s_red
// ([4][kTileM]) into s_lp in a fixed order.  p: the kernel's argument struct.  One __syncthreads, between the s_red
// writes and the s_lp update; the caller orders s_red and s_lp against their next use.
template <class Args, class ThetaRow>
__device__ __forceinline__ void target_tile_epilogue(const Args& p, const double (&acc)[2][4][2], int64_t i0, int rows,
                                                     int n0, double* s_red, double* s_lp, ThetaRow theta_row) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3, gq = lane >> 2, t = lane & 3, d = p.d;
#pragma unroll
  for (int a = 0; a < 2; ++a) {
    const int r = wm * 16 + a * 8 + gq;
    const bool live = r < rows;
    const auto theta = theta_row(r);
    double part = 0.0;
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int n = n0 + wn * 32 + b * 8 + 2 * t + u;
        if (!live || n >= d) continue;
        const double th = theta(n, acc[a][b][u]);
        if (p.theta_out) p.theta_out[(size_t)(i0 - p.first + r) * d + n] = th;
        if (p.target_kind >= 0) part += product_target_term(p.target_kind, (th - p.loc[n]) / p.scale[n], p.target_df);
      }
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    if (t == 0) s_red[wn * kTileM + r] = part;
  }
  __syncthreads();
  if (tid < kTileM) s_lp[tid] += ((s_red[tid] + s_red[kTileM + tid]) + s_red[2 * kTileM + tid]) + s_red[3 * kTileM + tid];
}

// CTAs per launch of a persistent grid, as many as can be resident (per SM x SMs: far inside a launch's 2^31 - 1)
template <class... A>
inline int persistent_ctas(void (*kern)(A...), int block, size_t smem, int64_t* ctas) {
  VB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  VB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, block, smem));
  *ctas = (int64_t)per_sm * sm_count();
  return per_sm >= 1 ? VB_OK : set_error(VB_ERR_UNSUPPORTED, "streamed log-weights: the kernel does not fit on an SM");
}

}  // namespace vb
