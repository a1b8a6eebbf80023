// Fused ELBO-gradient step for mean-field families on the GLM plugins, and the peer-memory communicator.
//
// The reference loop (optimization.py:95-98) makes three calls per iteration:
//     value, grad = objective(var_param)            objectives.py:154-168 (sample -> model -> reduce, autograd)
//     direction   = sgo.descent_direction(grad)     optimization.py:188-197 / :308-326
//     var_param   = objective.update(var_param, lr * direction)   objectives.py:57-59
// Here one step is THREE kernels, all enqueued without a host round trip (so the step can be captured in a
// CUDA graph and replayed):
//   1. mf_pre_kernel   Philox base draws at a device-resident stream position + reparameterisation
//                      (approximations.py:212-216, :270-274) + the tensor-core operand pack (Theta^T hi/lo, E) +
//                      per-sample |theta|^2 / log q partial sums for the prior / path-derivative terms
//   2. the GLM sweep   glm_fast.cu (tcgen05) or glm_f64.cu (DMMA): per-CTA partial sums of ll, gmu, ge
//   3. mf_post_kernel  reduction of the per-CTA partials, ONE-SHOT all-reduce of the S + 2d sums across ranks
//                      through peer memory (NVLink stores + flags; no NCCL call), objective value, gradient
//                      wrt [mu, log sigma] (SURVEY.md App. A.1), RMSProp / Adam state and parameter update,
//                      value / iterate histories, and the step counters.
//
// Peer-memory communicator (SURVEY.md 8(b)#7 `vb_comm_*`): every rank cudaMalloc's one buffer
// [flags | 2 parities x world slots], exports it with cudaIpcGetMemHandle, and maps the others'.  A collective
// of epoch e: each rank stores its vector into slot [e & 1][rank] of EVERY peer, fences, raises flag[rank] = e
// on every peer, waits until all its own flags reach e, and sums the slots in rank order -- every rank computes
// bit-identical sums, which keeps the replicated optimiser state identical.  Double buffering by parity is
// enough because a rank can only be one collective ahead of the slowest one.
#include <cuda_fp16.h>

#include <cstring>

#include "fast_internal.cuh"
#include "philox_draws.cuh"

namespace vb {

constexpr int kMaxWorld = 16;
constexpr size_t kCommHeader = 1024;       // flags (world x 8 bytes) live in the first KB of the shared buffer

struct CommView {
  int rank, world;
  int64_t slot_doubles;
  unsigned long long* epoch;               // local (not shared): number of collectives completed
  int* err;                                // local: set to 1 when a wait timed out
  unsigned long long* flags_local;         // [world]: flags_local[r] = last epoch rank r has delivered here
  double* data_local;                      // [2][world][slot_doubles]
  unsigned long long* flags_peer[kMaxWorld];
  double* data_peer[kMaxWorld];
};

struct Comm {
  int rank, world;
  size_t slot_bytes, total_bytes;
  char* local;                 // shared buffer (cudaMalloc)
  char* priv;                  // epoch + err (cudaMalloc, not shared)
  void* peers[kMaxWorld];      // mapped peer buffers (peers[rank] == local)
  bool opened[kMaxWorld];
  bool connected;
  CommView view;
};

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// Called by ONE block after every block of the grid has stored its part into the peers' slots (and fenced):
// raise this rank's flag on every peer, wait for every peer's flag here.  Bounded wait: a peer that never
// arrives (a crashed rank) sets *err instead of hanging the GPU.
__device__ __forceinline__ void comm_signal_and_wait(const CommView& c, unsigned long long e) {
  __threadfence_system();
  __syncthreads();
  if ((int)threadIdx.x < c.world) {
    st_release_sys(c.flags_peer[threadIdx.x] + c.rank, e);
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys(c.flags_local + threadIdx.x) < e) {
      if (global_timer_ns() - t0 > 4000000000ull) {       // 4 s
        *c.err = 1;
        break;
      }
      __nanosleep(64);
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// generic small in-place all-reduce (sum, float64) over the communicator
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) comm_allreduce_kernel(CommView c, double* __restrict__ buf, int64_t n,
                                                             unsigned int* ticket) {
  PDL_SYNC();
  const unsigned long long e = *c.epoch + 1;
  const int64_t par_off = (int64_t)(e & 1) * c.world * c.slot_doubles;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = buf[i];
    for (int r = 0; r < c.world; ++r) c.data_peer[r][par_off + (int64_t)c.rank * c.slot_doubles + i] = v;
  }
  __threadfence_system();
  __shared__ unsigned int last;
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
  __syncthreads();
  if (!last) return;
  comm_signal_and_wait(c, e);
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    double t = 0.0;
    for (int r = 0; r < c.world; ++r) t += __ldcg(c.data_local + par_off + (int64_t)r * c.slot_doubles + i);
    buf[i] = t;
  }
  if (threadIdx.x == 0) {
    *ticket = 0;
    *c.epoch = e;
  }
}

// ---------------------------------------------------------------------------------------------
// step kernels
// ---------------------------------------------------------------------------------------------
struct StepCfg {
  int family, objective, S, d, optimizer, quantize, inject, fast;
  int d_pad, chunks, rowsA;          // pre-kernel geometry: rowsA sample rows, `chunks` column tiles of 64
  double df, tconst, inv_tau2, prior_const;
  double lr, beta1, beta2, jitter;
  unsigned long long seed, stride;
};

struct StepPtrs {
  double* vp;
  double* opt_m;
  double* opt_nu;
  unsigned long long* counters;      // [0] step (history index), [1] optimiser steps taken, [2] draw-stream offset of step 0
  double* base;
  double* theta;
  double* value;
  double* grad;
  double* logp;
  double* direction;
  double* value_hist;
  double* param_hist;
  double* grad_hist;
  double* dir_hist;
  long long hist_len, ring;
  // engine workspace
  double* sq_part;                   // [S][chunks]
  double* lq_part;                   // [S][chunks]
  double* vec;                       // [S + 2d] reduced (and all-reduced) sweep sums
  double* aux;                       // [4][d]: p1, p2, pa, pb
  unsigned int* ticket;
};

__device__ __forceinline__ double draw_element(const StepCfg& c, const Philox& ph, unsigned long long offset,
                                               int64_t i) {
  const unsigned long long e = offset + (unsigned long long)i;
  if (c.family == VB_FAMILY_MF_GAUSSIAN) return normal_element(ph, e, c.quantize);
  return student_element(ph, e, c.df, c.quantize);
}

// One block = a tile of 16 samples x 64 columns (grid: column tiles x sample tiles).  Each thread owns one column
// pair and two rows, so a Box-Muller pair is evaluated once when the element index is even (the common case),
// base / theta / E rows are written as contiguous runs, Theta^T hi/lo go through a shared-memory transpose into
// 32-byte runs, and the per-sample partial sums are warp reductions (one warp = one row of the tile).
constexpr int kPreRows = 16, kPreCols = 64;

__global__ void __launch_bounds__(256) mf_pre_kernel(StepCfg c, StepPtrs p, fast::FastOperands ops) {
  PDL_SYNC();
  __shared__ float tt[kPreCols][kPreRows + 1];
  const Philox ph(c.seed);
  const unsigned long long offset = p.counters[2] + p.counters[0] * c.stride;
  const int d = c.d;
  const int s0 = blockIdx.y * kPreRows, j0 = blockIdx.x * kPreCols;
  const int cp = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int j = j0 + 2 * cp;
  const bool path = c.objective == VB_OBJ_EXCLUSIVE_KL_PATH;
  double mu[2] = {0.0, 0.0}, ls[2] = {0.0, 0.0}, sig[2] = {0.0, 0.0};
#pragma unroll
  for (int u = 0; u < 2; ++u)
    if (j + u < d) {
      mu[u] = p.vp[j + u];
      ls[u] = p.vp[d + j + u];
      sig[u] = exp(ls[u]);
    }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int row = w + 8 * r, s = s0 + row;
    double e[2] = {0.0, 0.0}, th[2] = {0.0, 0.0};
    if (s < c.S) {
      const int64_t i = (int64_t)s * d + j;
      if (c.inject) {
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if (j + u < d) e[u] = p.base[i + u];
      } else {
        const unsigned long long e0 = offset + (unsigned long long)i;
        if (c.family == VB_FAMILY_MF_GAUSSIAN && !(e0 & 1) && j + 1 < d) {
          normal_pair(ph, e0 >> 1, 0, e[0], e[1]);          // both elements of one Philox counter
          if (c.quantize) {
            e[0] = quantize_draw(e[0], c.quantize);
            e[1] = quantize_draw(e[1], c.quantize);
          }
        } else {
#pragma unroll
          for (int u = 0; u < 2; ++u)
            if (j + u < d) e[u] = draw_element(c, ph, offset, i + u);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if (j + u < d) p.base[i + u] = e[u];
      }
#pragma unroll
      for (int u = 0; u < 2; ++u)
        if (j + u < d) {
          th[u] = mu[u] + sig[u] * e[u];
          p.theta[i + u] = th[u];
        }
    }
    if (c.fast) {
      if (j < c.d_pad) {
        const __half2 h2 = __floats2half2_rn((float)e[0], (float)e[1]);
        *reinterpret_cast<__half2*>(ops.E + ((size_t)blockIdx.x * fast::kPadS + s) * 64 + 2 * cp) = h2;
      }
      tt[2 * cp][row] = (float)th[0];
      tt[2 * cp + 1][row] = (float)th[1];
    }
    // per-sample partial sums over this tile's 64 columns: the 32 lanes of this warp hold row `row`
    double sq = th[0] * th[0] + th[1] * th[1];
    sq = warp_sum(sq);
    if (cp == 0 && s < c.S) p.sq_part[(size_t)s * c.chunks + blockIdx.x] = sq;
    if (path) {
      double lq = 0.0;
      if (s < c.S) {
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if (j + u < d)
            lq += c.family == VB_FAMILY_MF_GAUSSIAN ? -0.5 * e[u] * e[u] - ls[u] - 0.5 * kLog2Pi
                                                    : c.tconst - 0.5 * (c.df + 1.0) * log1p(e[u] * e[u] / c.df) - ls[u];
      }
      lq = warp_sum(lq);
      if (cp == 0 && s < c.S) p.lq_part[(size_t)s * c.chunks + blockIdx.x] = lq;
    }
  }
  if (!c.fast) return;
  __syncthreads();
  {   // Theta^T hi: column jj of the tile, 4 consecutive samples per thread -> 8-byte stores, 32-byte runs
    const int jj = threadIdx.x >> 2, q4 = (threadIdx.x & 3) * 4;
    __align__(8) __half hi[4];
    float lof[4];                      // residual in fp32: the e5m2 copy must not inherit an fp16 underflow
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float t = tt[jj][q4 + u];
      hi[u] = __float2half_rn(t);
      lof[u] = t - __half2float(hi[u]);
    }
    const int sg = s0 + q4;                                     // 16 | 64: the 4 samples stay inside one 64-group
    const size_t o = ((size_t)(sg >> 6) * c.d_pad + (j0 + jj)) * 64 + (sg & 63);
    *reinterpret_cast<uint2*>(ops.Th + o) = *reinterpret_cast<const uint2*>(hi);
    // e5m2 copies for the fp8 correction passes: Theta_h * 2^-ax and Theta_l * 2^bx, 128-sample groups
    const float sh = exp2f((float)-ops.ax), sl = exp2f((float)ops.bx);
    uint32_t h8 = 0, l8 = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      h8 |= (uint32_t)fast::to_e5m2(__half2float(hi[u]) * sh) << (8 * u);
      l8 |= (uint32_t)fast::to_e5m2(lof[u] * sl) << (8 * u);
    }
    const size_t o8 = ((size_t)(sg >> 7) * c.d_pad + (j0 + jj)) * 128 + (sg & 127);
    *reinterpret_cast<uint32_t*>(ops.T8 + o8) = h8;
    *reinterpret_cast<uint32_t*>(ops.T8 + (size_t)2 * c.d_pad * 128 + o8) = l8;
  }
  if (blockIdx.x == 0 && blockIdx.y == 0) ops.wf[threadIdx.x] = (int)threadIdx.x < c.S ? 1.0f : 0.0f;
}

struct PartDesc {
  const double* ll_part;
  const double* gmu_part;
  const double* ge_part;
  int nblk_ll, nblk_g;
  long long stride_ll, stride_g;
  double sign_ll;
};

constexpr int kPostGroups = 32;      // row groups of the post kernel's reduction: block = 32 columns x 32 groups

__global__ void __launch_bounds__(32 * kPostGroups) mf_post_kernel(StepCfg c, StepPtrs p, PartDesc q, CommView cm) {
  PDL_SYNC();
  __shared__ double sm[3][kPostGroups][33];
  __shared__ double red[32];
  __shared__ unsigned int last;
  const int S = c.S, d = c.d, nvec = S + 2 * d;
  const bool path = c.objective == VB_OBJ_EXCLUSIVE_KL_PATH;
  const bool multi = cm.world > 1;
  const unsigned long long e = multi ? *cm.epoch + 1 : 0;
  const int64_t par_off = multi ? (int64_t)(e & 1) * cm.world * cm.slot_doubles : 0;

  // ---- phase 1: every block reduces 32 entries of [ll | gmu | ge] over the sweep's per-CTA partials, and the
  //      per-column sums over the samples that the prior / path terms of the gradient need ----
  {
    const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + x;
    double acc = 0.0, pp = 0.0, pq = 0.0;
    int kind = -1, col = 0;               // 0: ll, 1: gmu, 2: ge
    if (i < nvec) {
      const double* part;
      int nblk;
      long long stride;
      if (i < S) { kind = 0; col = i; part = q.ll_part; nblk = q.nblk_ll; stride = q.stride_ll; }
      else if (i < S + d) { kind = 1; col = i - S; part = q.gmu_part; nblk = q.nblk_g; stride = q.stride_g; }
      else { kind = 2; col = i - S - d; part = q.ge_part; nblk = q.nblk_g; stride = q.stride_g; }
#pragma unroll 4
      for (int b = y; b < nblk; b += kPostGroups) acc += part[(size_t)b * stride + col];
      if (kind == 1) {
#pragma unroll 4
        for (int s = y; s < S; s += kPostGroups) {
          const double th = p.theta[(size_t)s * d + col];
          pp += th;                                            // sum_s theta_sj
          if (path) {
            const double ee = p.base[(size_t)s * d + col];
            pq += c.family == VB_FAMILY_MF_GAUSSIAN ? ee : (c.df + 1.0) / (c.df + ee * ee) * ee;
          }
        }
      } else if (kind == 2) {
#pragma unroll 4
        for (int s = y; s < S; s += kPostGroups) {
          const double th = p.theta[(size_t)s * d + col], ee = p.base[(size_t)s * d + col];
          pp += th * ee;                                       // sum_s theta_sj e_sj
          if (path) pq += c.family == VB_FAMILY_MF_GAUSSIAN ? ee * ee : (c.df + 1.0) / (c.df + ee * ee) * ee * ee;
        }
      }
    }
    sm[0][y][x] = acc; sm[1][y][x] = pp; sm[2][y][x] = pq;
    __syncthreads();
    if (y == 0 && i < nvec) {
      double t = 0.0, tp = 0.0, tq = 0.0;
#pragma unroll
      for (int r = 0; r < kPostGroups; ++r) { t += sm[0][r][x]; tp += sm[1][r][x]; tq += sm[2][r][x]; }     // fixed order
      t *= kind == 0 ? q.sign_ll : 1.0;
      if (multi) {
        for (int r = 0; r < cm.world; ++r) cm.data_peer[r][par_off + (int64_t)cm.rank * cm.slot_doubles + i] = t;
      } else {
        p.vec[i] = t;
      }
      if (kind == 1) { p.aux[col] = tp; p.aux[2 * d + col] = tq; }
      if (kind == 2) { p.aux[d + col] = tp; p.aux[3 * d + col] = tq; }
    }
  }
  if (multi) __threadfence_system(); else __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(p.ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
  __syncthreads();
  if (!last) return;
  __threadfence();

  // ---- phase 2 (the last block): exchange, value, gradient, optimiser, histories ----
  if (multi) {
    comm_signal_and_wait(cm, e);
    for (int i = threadIdx.x; i < nvec; i += blockDim.x) {
      double t = 0.0;
      for (int r = 0; r < cm.world; ++r) t += __ldcg(cm.data_local + par_off + (int64_t)r * cm.slot_doubles + i);
      p.vec[i] = t;
    }
    __syncthreads();
  }
  const unsigned long long step = p.counters[0];
  const double invS = 1.0 / (double)S;
  const int first = p.counters[1] == 0;
  // One pass, no barriers inside: thread j owns BOTH entries of coordinate j (mu_j and log sigma_j), so it reads the
  // old parameter values before it writes the new ones and no other thread touches them; the threads beyond d (and
  // all threads again, strided) accumulate the per-sample terms of the value.  All loads of a thread are independent.
  double va = 0.0, vb_ = 0.0, vh = 0.0;
  for (int j = threadIdx.x; j < d; j += blockDim.x) {
    const double mu_old = p.vp[j], ls_old = p.vp[d + j];
    const double sig = exp(ls_old);
    const double a = __ldcg(p.vec + S + j) - __ldcg(p.aux + j) * c.inv_tau2;              // sum_s g_s[j]
    const double b = __ldcg(p.vec + S + d + j) - __ldcg(p.aux + d + j) * c.inv_tau2;      // sum_s g_s[j] e_s[j]
    double g[2];
    if (path) {
      g[0] = -invS * (a + __ldcg(p.aux + 2 * d + j) / sig);
      g[1] = -invS * (b * sig + __ldcg(p.aux + 3 * d + j));
    } else {
      g[0] = -invS * a;
      g[1] = -invS * b * sig - 1.0;
      vh += ls_old;                                                                        // entropy: sum_j log sigma_j
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = u * d + j;
      const double gi = g[u];
      p.grad[i] = gi;
      if (p.grad_hist && p.ring > 0) p.grad_hist[(size_t)(step % (unsigned long long)p.ring) * (2 * d) + i] = gi;
      if (c.optimizer == 0) continue;
      double dd;
      if (c.optimizer == 1) {                    // RMSProp: nu starts at grad**2 (optimization.py:189-190)
        const double g2 = gi * gi;
        double v = first ? g2 : p.opt_nu[i];
        v = v * c.beta1;
        v += (1.0 - c.beta1) * g2;
        p.opt_nu[i] = v;
        dd = gi / sqrt(c.jitter + v);
      } else {                                   // Adam, incl. the first-step aliasing of `momentum = grad` (:314-320)
        double mi, vi;
        if (first) {
          const double gs = gi * c.beta1;
          mi = gs + (1.0 - c.beta1) * gs;
          vi = (gi * gi) * c.beta2;
          vi += (1.0 - c.beta2) * (mi * mi);
        } else {
          mi = p.opt_m[i] * c.beta1;
          mi += (1.0 - c.beta1) * gi;
          vi = p.opt_nu[i] * c.beta2;
          vi += (1.0 - c.beta2) * (gi * gi);
        }
        p.opt_m[i] = mi;
        p.opt_nu[i] = vi;
        dd = mi / sqrt(c.jitter + vi);
      }
      if (p.direction) p.direction[i] = dd;
      if (p.dir_hist && p.ring > 0) p.dir_hist[(size_t)(step % (unsigned long long)p.ring) * (2 * d) + i] = dd;
      const double nv = (u == 0 ? mu_old : ls_old) - c.lr * dd;     // objectives.py:57-59
      p.vp[i] = nv;
      if (p.param_hist && p.ring > 0) p.param_hist[(size_t)(step % (unsigned long long)p.ring) * (2 * d) + i] = nv;
    }
  }
  // value (objectives.py:161-164): -(mean_s f(theta_s) + H), or -(mean_s (f - log q)) for the path-derivative form;
  // samples are taken from the top of the block so that they overlap the coordinate work above
  for (int s = (int)blockDim.x - 1 - (int)threadIdx.x; s < S; s += blockDim.x) {
    double sq = 0.0, lq = 0.0;
    for (int k = 0; k < c.chunks; ++k) {
      sq += __ldcg(p.sq_part + s * c.chunks + k);
      if (path) lq += __ldcg(p.lq_part + s * c.chunks + k);
    }
    const double f = __ldcg(p.vec + s) + (-0.5 * sq * c.inv_tau2 + c.prior_const);
    if (p.logp) p.logp[s] = f;
    va += f;
    vb_ += lq;
  }
  va = block_sum(va, red);
  vb_ = block_sum(vb_, red);
  vh = block_sum(vh, red);
  if (threadIdx.x == 0) {
    if (!path && c.family == VB_FAMILY_MF_GAUSSIAN) vh += 0.5 * d * (1.0 + kLog2Pi);     // approximations.py:218-220
    const double v = path ? -((va - vb_) * invS) : -(va * invS + vh);
    p.value[0] = v;
    if (p.value_hist && (long long)step < p.hist_len) p.value_hist[step] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    p.counters[0] = step + 1;
    if (c.optimizer) p.counters[1] += 1;
    *p.ticket = 0;
    if (multi) *cm.epoch = e;
  }
}

static inline double student_const_h(double df) {
  return lgamma(0.5 * (df + 1.0)) - lgamma(0.5 * df) - 0.5 * log(df * 3.14159265358979323846);
}

}  // namespace vb

using namespace vb;

// =================================================================================================
// communicator
// =================================================================================================
extern "C" int vb_comm_create(void** comm, int rank, int world, size_t slot_bytes, unsigned char* handle_out) {
  if (!comm || world < 1 || world > kMaxWorld || rank < 0 || rank >= world || slot_bytes == 0)
    return set_error(VB_ERR_INVALID_ARG, "comm_create: bad arguments (world <= 16)");
  Comm* c = new Comm();
  memset(c, 0, sizeof(Comm));
  c->rank = rank;
  c->world = world;
  c->slot_bytes = align_up(slot_bytes, 256);
  c->total_bytes = kCommHeader + 2 * (size_t)world * c->slot_bytes;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&c->local), c->total_bytes);
  if (e == cudaSuccess) e = cudaMemset(c->local, 0, c->total_bytes);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->priv), 256);
  if (e == cudaSuccess) e = cudaMemset(c->priv, 0, 256);
  if (e == cudaSuccess && handle_out) {
    cudaIpcMemHandle_t h;
    e = cudaIpcGetMemHandle(&h, c->local);
    if (e == cudaSuccess) memcpy(handle_out, &h, sizeof(h));
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    if (c->local) cudaFree(c->local);
    if (c->priv) cudaFree(c->priv);
    delete c;
    return set_cuda_error(e);
  }
  *comm = c;
  return VB_OK;
}

static void comm_build_view(Comm* c) {
  CommView& v = c->view;
  v.rank = c->rank;
  v.world = c->world;
  v.slot_doubles = (int64_t)(c->slot_bytes / sizeof(double));
  v.epoch = reinterpret_cast<unsigned long long*>(c->priv);
  v.err = reinterpret_cast<int*>(c->priv + 64);
  v.flags_local = reinterpret_cast<unsigned long long*>(c->local);
  v.data_local = reinterpret_cast<double*>(c->local + kCommHeader);
  for (int r = 0; r < c->world; ++r) {
    v.flags_peer[r] = reinterpret_cast<unsigned long long*>(c->peers[r]);
    v.data_peer[r] = reinterpret_cast<double*>(static_cast<char*>(c->peers[r]) + kCommHeader);
  }
  c->connected = true;
}

/* all_handles: world x 64 bytes (host), rank order, as returned by vb_comm_create on every rank */
extern "C" int vb_comm_connect(void* comm, const unsigned char* all_handles) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c || !all_handles) return set_error(VB_ERR_INVALID_ARG, "comm_connect: bad arguments");
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank) {
      c->peers[r] = c->local;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, all_handles + (size_t)r * sizeof(h), sizeof(h));
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return set_cuda_error(e);
    c->peers[r] = ptr;
    c->opened[r] = true;
  }
  comm_build_view(c);
  return VB_OK;
}

/* in-process variant (several ranks driven by one process, e.g. tests): peer_ptrs[r] = vb_comm_buffer of rank r */
extern "C" int vb_comm_connect_ptrs(void* comm, void* const* peer_ptrs) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c || !peer_ptrs) return set_error(VB_ERR_INVALID_ARG, "comm_connect_ptrs: bad arguments");
  for (int r = 0; r < c->world; ++r) c->peers[r] = r == c->rank ? c->local : peer_ptrs[r];
  comm_build_view(c);
  return VB_OK;
}

extern "C" void* vb_comm_buffer(void* comm) { return comm ? static_cast<Comm*>(comm)->local : nullptr; }

/* 1 when a collective timed out waiting for a peer (host-synchronising read) */
extern "C" int vb_comm_error(void* comm) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c) return 0;
  int err = 0;
  if (cudaMemcpy(&err, c->priv + 64, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  return err;
}

extern "C" int vb_comm_destroy(void* comm) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c) return VB_OK;
  for (int r = 0; r < c->world; ++r)
    if (c->opened[r]) cudaIpcCloseMemHandle(c->peers[r]);
  cudaFree(c->local);
  cudaFree(c->priv);
  delete c;
  return VB_OK;
}

/* in place: buf[i] <- sum over ranks, summed in rank order on every rank (bit-identical results).  n doubles must
 * fit the slot size given to vb_comm_create.  Latency-bound one-shot algorithm for small vectors. */
extern "C" int vb_comm_allreduce_sum_f64(void* comm, double* buf, int64_t n, cudaStream_t stream) {
  Comm* c = static_cast<Comm*>(comm);
  if (!c || !buf || n < 0) return set_error(VB_ERR_INVALID_ARG, "comm_allreduce: bad arguments");
  if (!c->connected) return set_error(VB_ERR_INVALID_ARG, "comm_allreduce: communicator is not connected");
  if ((size_t)n * sizeof(double) > c->slot_bytes) return set_error(VB_ERR_WORKSPACE, "comm_allreduce: vector exceeds the slot size");
  if (n == 0 || c->world == 1) return VB_OK;
  int blocks = (int)((n + 255) / 256);
  if (blocks > 32) blocks = 32;
  unsigned int* ticket = reinterpret_cast<unsigned int*>(c->priv + 128);
  VB_CUDA(launch_pdl(comm_allreduce_kernel, dim3(blocks), dim3(256), stream, c->view, buf, n, ticket));
  return VB_OK;
}

// =================================================================================================
// fused step
// =================================================================================================
struct StepLayout {
  size_t off_sq, off_lq, off_vec, off_aux, off_ticket, total;
  int chunks, rowsA, d_pad;
};

static void step_layout(int S, int d, int fast, StepLayout& L) {
  L.d_pad = fast ? (int)(ceil_div(d, 256) * 256) : d;
  L.chunks = (int)ceil_div(L.d_pad, kPreCols);          // column tiles of the pre kernel
  L.rowsA = fast ? fast::kPadS : S;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  L.off_sq = take(sizeof(double) * (size_t)S * L.chunks);
  L.off_lq = take(sizeof(double) * (size_t)S * L.chunks);
  L.off_vec = take(sizeof(double) * ((size_t)S + 2 * (size_t)d));
  L.off_aux = take(sizeof(double) * 4 * (size_t)d);
  L.off_ticket = take(256);
  L.total = off;
}

extern "C" size_t vb_mf_step_workspace_bytes(int S, int d) {
  if (S <= 0 || d <= 0) return 0;
  StepLayout L;
  step_layout(S, d, 1, L);         // the fast layout is the larger one
  return L.total;
}

extern "C" int vb_mf_step_glm(const vb_step_config* cfg, const vb_step_buffers* buf, const vb_step_model* model,
                              void* comm, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!cfg || !buf || !model || !workspace) return set_error(VB_ERR_INVALID_ARG, "mf_step: null argument");
  const int S = cfg->S, d = cfg->d;
  if (S <= 0 || d <= 0) return set_error(VB_ERR_INVALID_ARG, "mf_step: bad shape");
  if (cfg->family != VB_FAMILY_MF_GAUSSIAN && cfg->family != VB_FAMILY_MF_STUDENT)
    return set_error(VB_ERR_INVALID_ARG, "unknown mean-field family");
  if (cfg->family == VB_FAMILY_MF_STUDENT && !(cfg->df > 2.0)) return set_error(VB_ERR_INVALID_ARG, "df must be greater than 2");
  if (cfg->objective != VB_OBJ_EXCLUSIVE_KL && cfg->objective != VB_OBJ_EXCLUSIVE_KL_PATH)
    return set_error(VB_ERR_UNSUPPORTED, "mf_step: only the ExclusiveKL objectives have a fused step");
  if (cfg->optimizer < 0 || cfg->optimizer > 2) return set_error(VB_ERR_INVALID_ARG, "mf_step: unknown optimiser");
  if (!buf->var_param || !buf->counters || !buf->base || !buf->theta || !buf->value || !buf->grad)
    return set_error(VB_ERR_INVALID_ARG, "mf_step: missing buffer");
  if (cfg->optimizer && !buf->opt_nu) return set_error(VB_ERR_INVALID_ARG, "mf_step: optimiser state missing");
  if (cfg->optimizer == 2 && !buf->opt_m) return set_error(VB_ERR_INVALID_ARG, "mf_step: Adam needs opt_m");
  const int fast = model->fast_handle != nullptr;
  if (fast && S > fast::kPadS) return set_error(VB_ERR_UNSUPPORTED, "mf_step: the tensor-core sweep takes at most 256 samples");
  // the pre kernel's row tiles sit on gridDim.y (at most 65535)
  if (ceil_div(S, kPreRows) > 65535) return set_error(VB_ERR_UNSUPPORTED, "mf_step: at most 1048560 samples per step");
  StepLayout L;
  step_layout(S, d, fast, L);
  if (workspace_bytes < L.total) return set_error(VB_ERR_WORKSPACE, "mf_step: workspace too small");
  Comm* cm = static_cast<Comm*>(comm);
  CommView view;
  memset(&view, 0, sizeof(view));
  view.world = 1;
  if (cm && cm->world > 1) {
    if (!cm->connected) return set_error(VB_ERR_INVALID_ARG, "mf_step: communicator is not connected");
    if (((size_t)S + 2 * (size_t)d) * sizeof(double) > cm->slot_bytes)
      return set_error(VB_ERR_WORKSPACE, "mf_step: communicator slots are too small for S + 2d doubles");
    view = cm->view;
  }

  StepCfg c;
  c.family = cfg->family; c.objective = cfg->objective; c.S = S; c.d = d; c.optimizer = cfg->optimizer;
  c.quantize = cfg->quantize; c.inject = cfg->inject_base; c.fast = fast;
  c.d_pad = L.d_pad; c.chunks = L.chunks; c.rowsA = L.rowsA;
  c.df = cfg->df;
  c.tconst = cfg->family == VB_FAMILY_MF_STUDENT ? student_const_h(cfg->df) : 0.0;
  if (cfg->prior_sd > 0.0 && isfinite(cfg->prior_sd)) {
    c.inv_tau2 = 1.0 / (cfg->prior_sd * cfg->prior_sd);
    c.prior_const = -(double)d * log(cfg->prior_sd * sqrt(2.0 * 3.14159265358979323846));
  } else {
    c.inv_tau2 = 0.0;
    c.prior_const = 0.0;
  }
  c.lr = cfg->lr; c.beta1 = cfg->beta1; c.beta2 = cfg->beta2; c.jitter = cfg->jitter;
  c.seed = cfg->seed;
  const unsigned long long n = (unsigned long long)S * (unsigned long long)d;
  c.stride = n + (n & 1);

  char* ws = static_cast<char*>(workspace);
  StepPtrs p;
  p.vp = buf->var_param; p.opt_m = buf->opt_m; p.opt_nu = buf->opt_nu;
  p.counters = reinterpret_cast<unsigned long long*>(buf->counters);
  p.base = buf->base; p.theta = buf->theta; p.value = buf->value; p.grad = buf->grad; p.logp = buf->logp;
  p.direction = buf->direction;
  p.value_hist = buf->value_hist; p.param_hist = buf->param_hist; p.grad_hist = buf->grad_hist; p.dir_hist = buf->dir_hist;
  p.hist_len = buf->hist_len; p.ring = buf->ring;
  p.sq_part = reinterpret_cast<double*>(ws + L.off_sq);
  p.lq_part = reinterpret_cast<double*>(ws + L.off_lq);
  p.vec = reinterpret_cast<double*>(ws + L.off_vec);
  p.aux = reinterpret_cast<double*>(ws + L.off_aux);
  p.ticket = reinterpret_cast<unsigned int*>(ws + L.off_ticket);

  fast::FastOperands ops = {};
  memset(&ops, 0, sizeof(ops));
  if (fast) {
    int md = 0, mdp = 0;
    int rc = fast::fast_dims(model->fast_handle, nullptr, &md, &mdp);
    if (rc) return rc;
    if (md != d || mdp != L.d_pad) return set_error(VB_ERR_INVALID_ARG, "mf_step: model dimension does not match d");
    rc = fast::fast_operands(model->fast_handle, model->fast_workspace, model->fast_workspace_bytes, &ops);
    if (rc) return rc;
  }
  // 1. draws + reparameterisation + operand pack
  VB_CUDA(launch_pdl(mf_pre_kernel, dim3(L.chunks, (unsigned)ceil_div(L.rowsA, kPreRows)), dim3(256), stream, c, p, ops));

  // 2. the sweep over this rank's observations
  PartDesc q;
  const int total_only = (cfg->objective == VB_OBJ_EXCLUSIVE_KL && !buf->logp) ? 1 : 0;
  if (fast) {
    fast::FastPartials parts;
    int rc = fast::fast_launch(model->fast_handle, model->fast_workspace, model->fast_workspace_bytes, S, 1, total_only, 1,
                               nullptr, stream, &parts);
    if (rc) return rc;
    q.ll_part = parts.ll_part; q.gmu_part = parts.gmu_part; q.ge_part = parts.ge_part;
    q.nblk_ll = parts.nblk_ll; q.nblk_g = parts.nblk_g;
    q.stride_ll = parts.stride_ll; q.stride_g = parts.stride_g;
    q.sign_ll = -1.0;
  } else {
    if (!model->X || !model->y || !model->sweep_workspace) return set_error(VB_ERR_INVALID_ARG, "mf_step: float64 model data missing");
    // the float64 sweep reduces its own partials: its outputs are one-row "partials" placed in its workspace tail
    const size_t need = vb_glm_sweep_workspace_bytes(model->N, d, S);
    if (need == 0) return set_error(VB_ERR_UNSUPPORTED, "model dimension too large for the fused sweep");
    const size_t tail = align_up(need, 256);
    if (model->sweep_workspace_bytes < tail + sizeof(double) * ((size_t)S + 2 * (size_t)d))
      return set_error(VB_ERR_WORKSPACE, "mf_step: float64 sweep workspace too small (needs S + 2d extra doubles)");
    double* out = reinterpret_cast<double*>(static_cast<char*>(model->sweep_workspace) + tail);
    int rc = vb_glm_sweep_f64(model->X, model->ldx, model->y, model->N, d, model->link, buf->theta, buf->base, nullptr,
                              nullptr, S, 1, out, out + S, out + S + d, model->sweep_workspace, need, stream);
    if (rc) return rc;
    q.ll_part = out; q.gmu_part = out + S; q.ge_part = out + S + d;
    q.nblk_ll = 1; q.nblk_g = 1; q.stride_ll = S; q.stride_g = d; q.sign_ll = 1.0;
  }

  // 3. reduce + exchange + finish + optimiser
  const int nblocks_post = (S + 2 * d + 31) / 32;
  VB_CUDA(launch_pdl(mf_post_kernel, dim3(nblocks_post), dim3(32 * kPostGroups), stream, c, p, q, view));
  return VB_OK;
}
