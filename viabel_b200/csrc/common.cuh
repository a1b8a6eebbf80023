// Shared device/host helpers for libviabel_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/viabel_b200.h"

namespace vb {

#define VB_CHECK_LAUNCH()                                     \
  do {                                                        \
    cudaError_t e__ = cudaGetLastError();                     \
    if (e__ != cudaSuccess) return vb::set_cuda_error(e__);   \
  } while (0)

#define VB_CUDA(call)                                         \
  do {                                                        \
    cudaError_t e__ = (call);                                 \
    if (e__ != cudaSuccess) return vb::set_cuda_error(e__);   \
  } while (0)

int set_cuda_error(cudaError_t e);
int set_error(int code, const char* msg);
int sm_count();

constexpr double kLog2Pi = 1.8378770664093454835606594728112;
constexpr double kInvSqrt2 = 0.70710678118654752440084436210485;

// log of the Student-t density's normaliser, lgamma((df+1)/2) - lgamma(df/2) - log(pi df)/2 (host)
inline double student_t_log_const(double df) {
  return lgamma(0.5 * (df + 1.0)) - lgamma(0.5 * df) - 0.5 * log(df * 3.14159265358979323846);
}

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- warp / block reductions ------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum; `red` is >= 32 doubles of shared memory.  Result valid in every thread.
__device__ __forceinline__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double r = (lane < nw) ? red[lane] : 0.0;
  r = warp_sum(r);
  return r;
}
__device__ __forceinline__ double block_max(double v, double* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double r = (lane < nw) ? red[lane] : -INFINITY;
  r = warp_max(r);
  return r;
}

// ---- Philox4x32-10 counter RNG ------------------------------------------------------------
struct Philox {
  uint32_t key[2];
  __host__ __device__ Philox(uint64_t seed) {
    key[0] = (uint32_t)seed;
    key[1] = (uint32_t)(seed >> 32);
  }
  __host__ __device__ static inline void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
    uint64_t p = (uint64_t)a * b;
    hi = (uint32_t)(p >> 32);
    lo = (uint32_t)p;
  }
  // counter = (c0..c3); returns 4 x 32 random bits
  __host__ __device__ inline void operator()(uint64_t ctr_lo, uint64_t ctr_hi, uint32_t out[4]) const {
    uint32_t c0 = (uint32_t)ctr_lo, c1 = (uint32_t)(ctr_lo >> 32);
    uint32_t c2 = (uint32_t)ctr_hi, c3 = (uint32_t)(ctr_hi >> 32);
    uint32_t k0 = key[0], k1 = key[1];
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      uint32_t hi0, lo0, hi1, lo1;
      mulhilo(0xD2511F53u, c0, hi0, lo0);
      mulhilo(0xCD9E8D57u, c2, hi1, lo1);
      uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
      c0 = n0; c1 = n1; c2 = n2; c3 = n3;
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
  }
};

// 2 x 32 bits -> uniform double in (0,1] with 53 bits: from v = 2^52 up, v + 0.5 rounds to even, so the top value
// (2^53 - 1) gives exactly 1.0 (harmless: Box-Muller's radius is then 0 and the gamma boost 1)
__host__ __device__ inline double u01_53(uint32_t a, uint32_t b) {
  uint64_t v = (((uint64_t)a << 32) | b) >> 11;                 // 53 bits
  return ((double)v + 0.5) * (1.0 / 9007199254740992.0);
}

// ---- link functions (double) ---------------------------------------------------------------
// a = y*z ; returns log-likelihood term and d/da of it
__device__ __forceinline__ void link_logistic(double a, double& ll, double& dl) {
  double e = exp(-fabs(a));
  double l1p = log1p(e);
  ll = -(fmax(-a, 0.0) + l1p);                                  // -softplus(-a)
  double inv = 1.0 / (1.0 + e);
  dl = (a >= 0.0) ? e * inv : inv;                              // sigmoid(-a)
}
__device__ __forceinline__ void link_probit(double a, double& ll, double& dl) {
  // log Phi(a) and phi(a)/Phi(a); erfcx keeps the left tail finite
  double u = -a * kInvSqrt2;
  if (u > 0.0) {
    double ex = erfcx(u);                                       // Phi(a) = 0.5*erfcx(u)*exp(-u^2)
    ll = log(0.5 * ex) - u * u;
    dl = 0.79788456080286535587989211986876 / ex;               // sqrt(2/pi)/erfcx(u)
  } else {
    // a >= 0: Phi(a) = 1 - q with q = Phi(-a) <= 1/2; log1p keeps ll accurate relative to itself as Phi -> 1
    double q = 0.5 * erfc(-u);
    ll = log1p(-q);
    // phi(a) with a^2 = h + l split exactly: exp(-h/2) then the first-order factor of l, so that the exponent's
    // rounding (u a^2 / 2 absolute) does not reach dl
    const double h = a * a, l = fma(a, a, -h);
    dl = exp(-0.5 * h) * (1.0 - 0.5 * l) * 0.39894228040143267793994605993438 / (1.0 - q);
  }
}
// -(log Phi)''(a) = r (a + r), r = phi(a) / Phi(a).  For a < -6, r ~ -a and a + r cancels (relative error ~ u a^2); there
// a + r = 1 / (x + 2 / (x + 3 / (x + ...))), x = -a, the continued fraction of the Mills ratio, whose 24 terms reach
// full double precision for every x > 6.
__device__ __forceinline__ double probit_curvature(double a, double r) {
  if (a >= -6.0) return r * (a + r);
  const double x = -a;
  double t = 0.0;
#pragma unroll
  for (int k = 24; k >= 2; --k) t = k / (x + t);
  return r / (x + t);
}
// sigmoid(a) sigmoid(-a) = e / (1 + e)^2, e = exp(-|a|): no 1 - sigmoid cancellation for either sign
__device__ __forceinline__ double logistic_curvature(double a) {
  const double e = exp(-fabs(a)), inv = 1.0 / (1.0 + e);
  return e * inv * inv;
}

}  // namespace vb

// Programmatic dependent launch: a kernel launched with launch_pdl() starts with PDL_SYNC() (wait until the kernels before it in the stream have completed and flushed) followed by a trigger
// that lets the NEXT kernel's blocks be scheduled while this one runs, so the launch ramps overlap.
#define PDL_SYNC()                                               \
  do {                                                           \
    asm volatile("griddepcontrol.wait;" ::: "memory");           \
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); \
  } while (0)

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

