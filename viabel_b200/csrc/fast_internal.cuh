// Internal (non-ABI) interface of the tensor-core GLM sweep, shared by glm_fast.cu and engine.cu: the fused
// step engine packs the operands itself (draw + reparameterise + pack in one kernel) and consumes the sweep's
// per-CTA partial sums directly (reduce + exchange + finish + optimiser in one kernel).
#pragma once
#include <cuda_fp16.h>
#include <cuda_fp8.h>

#include "common.cuh"

namespace vb {
namespace fast {

constexpr int kPadS = 256;      // padded sample count of a sweep (= kSP in glm_fast.cu)

struct FastOperands {
  __half* Th;    // Theta^T hi  [4][d_pad][64]
  __half* E;     // base draws  [d_pad/64][256][64]
  float* wf;     // sample weights [256]
  // fp8 correction operands: e5m2 copies [2: Theta_h * 2^-ax | Theta_l * 2^bx][2 groups][d_pad][128 s]
  uint8_t* T8;
  int ax, bx;    // static power-of-two scales of the model (X_l8 = X_l * 2^ax, X_h8 = X_h * 2^-bx): each pass's operand scales multiply to 1
};

// e5m2 (1-5-2) of a float, round to nearest, saturating
__device__ __forceinline__ uint8_t to_e5m2(float x) {
  return (uint8_t)__nv_cvt_float_to_fp8(x, __NV_SATFINITE, __NV_E5M2);
}

struct FastPartials {
  const double* ll_part;    // [nblk_ll][stride_ll]  sums of softplus (negate)
  const double* gmu_part;   // [nblk_g][stride_g]
  const double* ge_part;    // [nblk_g][stride_g]
  int nblk_ll, nblk_g;
  int64_t stride_ll, stride_g;
};

int fast_dims(void* handle, int64_t* N, int* d, int* d_pad);
int fast_operands(void* handle, void* workspace, size_t workspace_bytes, FastOperands* ops);
int fast_launch(void* handle, void* workspace, size_t workspace_bytes, int S, int want_grad, int ll_total_only,
                int uniform_w, float* debug, cudaStream_t stream, FastPartials* parts);

}  // namespace fast
}  // namespace vb
