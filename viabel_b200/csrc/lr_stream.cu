// Streaming log-weights of the low-rank LRGaussian family (Sigma = B B^T + D^2, D = diag(sigma)) for vi_diagnostics
// at scale; the mean-field version is stream_lw.cu and the full-rank MultivariateT version mvt_stream.cu.  Draw i of
// n_total is regenerated from the family's Philox stream by offset -- z_i[l] is element offset + i k + l and eps_i[j]
// element offset + n_total k + ((n_total k) & 1) + i d + j of the normal stream, exactly what
// LRGaussian.base_draws(n_total) draws -- and, with u_i = [z_i, eps_i] in R^(k+d),
//
//     theta_i = mu + B z_i + sigma * eps_i
//     w_i     = P u_i,   P = [C^-1 | -C^-1 B^T D^-1]  (k x (k+d)),   C C^T = M = I + B^T D^-2 B
//     log q_i = -1/2 (d log 2 pi + |u_i|^2 - |w_i|^2) - sum_j log sigma_j + sum_l log P_ll
//     lw_i    = log p(theta_i) - log q_i            (product Gaussian / Student-t target, or -log q_i with no target)
//
// theta_i - mu = [B, D] u_i, so the Mahalanobis term is the squared norm of the projection of u_i onto the row space
// of [B, D]; the rows of P are an orthonormal basis of its null space, hence |u|^2 - |P u|^2.  No solve per draw.
//
// Persistent grid; a CTA takes 32 draws at a time and owns every column block of them.  The tile's u rows (z and eps
// parts, row strides = 4 mod 8 doubles so that the MMA fragment loads hit distinct banks) are generated once into
// shared memory (k + d <= 512) or into the CTA's slice of the workspace (L2 resident).  Both products run on the FP64
// tensor pipe (mma.sync m8n8k4 f64):
//   w = U P^T   N = k is small, so the K = k + d sweep is split over the 8 warps (each 32 rows x 32 columns of P, k4
//               steps warp, warp + 8, ...); the 8 partial tiles are summed in warp order before squaring.
//   theta       Z B^T over 128-wide column blocks, 8 warps of 16 x 32; the epilogue adds mu and sigma * eps, writes
//               theta_out if asked and sums the target terms over lanes and warps in a fixed order.
// No atomics and nothing depends on where a draw sits in its tile, so repeated calls give identical bits and a slice
// computed alone equals the same draws of a longer call.
#include "mvt_internal.cuh"
#include "philox_draws.cuh"

namespace vb {

constexpr int kLrM = 32;                     // draws per tile
constexpr int kLrN = 128;                    // theta column block
constexpr int kLrWN = 32;                    // w column block (rows of P)
constexpr int kLrUSharedMax = 512;           // u tile in shared memory while k + d <= this
constexpr int kLrMaxWidth = 1 << 26;         // k + d: tile offsets stay in 32 bits

struct LrStreamArgs {
  const double* vp;
  const double* P;
  const double* consts;                      // [0]: -d/2 log 2 pi - sum log sigma + sum log P_ll; [1]: target constant
  const double* sig;                         // sigma = exp(log_sigma)
  const double* loc;
  const double* scale;
  double* lw;
  double* theta_out;
  double* uws;                               // per-CTA u tiles when they do not fit in shared memory
  int64_t first, count;
  uint64_t seed, z_off, e_off;
  int d, k, ldz, lde, kq, target_kind;
  double target_df;
};

// row stride = 4 (mod 8) doubles: the 8 rows x 4 columns of an MMA fragment fall on distinct shared-memory banks
__host__ __device__ inline int lr_ld(int w) { return w + ((4 - w) & 7); }

// rows x w consecutive elements of the normal stream from element e0 into t (row stride ld), one Box-Muller pair per
// counter; a run that starts or ends on an odd element uses one value of the boundary pair
__device__ __forceinline__ void lr_fill(const Philox& ph, uint64_t e0, int rows, int w, double* t, int ld) {
  const int ne = rows * w;
  if (ne == 0) return;
  const uint64_t c0 = e0 >> 1, c1 = (e0 + ne - 1) >> 1;
  for (uint64_t c = c0 + threadIdx.x; c <= c1; c += blockDim.x) {
    double z0, z1;
    normal_pair(ph, c, 0, z0, z1);
    const int l = (int)(2 * c - e0);         // -1 for the unused half of a leading odd pair
    if (l >= 0) {
      const int r = l / w;
      t[(size_t)r * ld + (l - r * w)] = z0;
    }
    if (l + 1 < ne) {
      const int r = (l + 1) / w;
      t[(size_t)r * ld + (l + 1 - r * w)] = z1;
    }
  }
}

template <bool kUShared>
__global__ void __launch_bounds__(256, 2) lr_stream_lw_kernel(const LrStreamArgs p) {
  extern __shared__ double sh[];
  double* s_red = sh;                        // [4][kLrM]: per-warp-column partial sums of the target terms
  double* s_lp = s_red + 4 * kLrM;
  double* s_uu = s_lp + kLrM;                // |u|^2
  double* s_ww = s_uu + kLrM;                // |w|^2
  double* wbuf = s_ww + kLrM;                // [8][kLrM][kq]: per-warp partial w tiles
  const int d = p.d, k = p.k, ldz = p.ldz, lde = p.lde, kq = p.kq, K1 = k + d;
  double* zt = kUShared ? wbuf + 8 * kLrM * kq : p.uws + (size_t)blockIdx.x * kLrM * (ldz + lde);
  double* et = zt + (size_t)kLrM * ldz;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3;
  const int gq = lane >> 2, t = lane & 3;
  const int nb = (d + kLrN - 1) / kLrN;
  const bool want_theta = p.theta_out != nullptr || p.target_kind >= 0;
  const double lqc = p.consts[0], pconst = p.consts[1];
  const double* Bm = p.vp + 2 * (size_t)d;   // B[n][l] = Bm[n k + l]
  const Philox ph(p.seed);
  const int64_t ntiles = (p.count + kLrM - 1) / kLrM;

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t i0 = p.first + tile * kLrM;
    const int rows = (int)min((int64_t)kLrM, p.first + p.count - i0);
    __syncthreads();                         // the previous tile is done with the u tile and the per-draw arrays
    lr_fill(ph, p.z_off + (uint64_t)i0 * k, rows, k, zt, ldz);
    lr_fill(ph, p.e_off + (uint64_t)i0 * d, rows, d, et, lde);
    if (tid < kLrM) s_lp[tid] = s_ww[tid] = 0.0;
    __syncthreads();
    for (int r = warp; r < rows; r += 8) {
      double a = 0.0;
      for (int j = lane; j < k; j += 32) a += zt[r * ldz + j] * zt[r * ldz + j];
      for (int j = lane; j < d; j += 32) a += et[r * lde + j] * et[r * lde + j];
      a = warp_sum(a);
      if (lane == 0) s_uu[r] = a;
    }

    // w = U P^T, 32 columns of it at a time; rows past `rows` hold stale values and only reach their own outputs
    const int nsteps = (K1 + 3) >> 2;
    for (int m0 = 0; m0 < k; m0 += kLrWN) {
      double acc[4][4][2];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
      for (int s = warp; s < nsteps; s += 8) {
        const int c = 4 * s + t;
        double af[4], bf[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const int r = a * 8 + gq;
          af[a] = c < k ? zt[r * ldz + c] : c < K1 ? et[r * lde + c - k] : 0.0;
        }
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int m = m0 + b * 8 + gq;
          bf[b] = (m < k && c < K1) ? __ldg(p.P + (size_t)m * K1 + c) : 0.0;
        }
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          if (b * 8 >= kq) break;
#pragma unroll
          for (int a = 0; a < 4; ++a) dmma(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
        }
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int cl = b * 8 + 2 * t + u;
            if (cl < kq) wbuf[(warp * kLrM + a * 8 + gq) * kq + cl] = acc[a][b][u];
          }
      __syncthreads();
      for (int e = tid; e < kLrM * kq; e += blockDim.x) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) v += wbuf[w * kLrM * kq + e];
        wbuf[e] = v * v;
      }
      __syncthreads();
      if (tid < kLrM) {
        double a = 0.0;
        for (int cl = 0; cl < kq; ++cl) a += wbuf[tid * kq + cl];
        s_ww[tid] += a;
      }
      __syncthreads();                       // wbuf is rewritten by the next column block
    }

    // theta = mu + Z B^T + sigma * eps over 128-wide column blocks, target terms summed per draw
    for (int cb = 0; want_theta && cb < nb; ++cb) {
      const int n0 = cb * kLrN;
      double acc[2][4][2];
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
      for (int k0 = 0; k0 < k; k0 += 4) {
        const int l = k0 + t;
        double af[2], bf[4];
#pragma unroll
        for (int a = 0; a < 2; ++a) af[a] = l < k ? zt[(wm * 16 + a * 8 + gq) * ldz + l] : 0.0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int n = n0 + wn * 32 + b * 8 + gq;
          bf[b] = (l < k && n < d) ? __ldg(Bm + (size_t)n * k + l) : 0.0;
        }
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) dmma(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
      }
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        const int r = wm * 16 + a * 8 + gq;
        const bool live = r < rows;
        double part = 0.0;
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int n = n0 + wn * 32 + b * 8 + 2 * t + u;
            if (!live || n >= d) continue;
            const double th = p.vp[n] + acc[a][b][u] + p.sig[n] * et[r * lde + n];
            if (p.theta_out) p.theta_out[(size_t)(i0 - p.first + r) * d + n] = th;
            if (p.target_kind >= 0) {
              const double zz = (th - p.loc[n]) / p.scale[n];
              part += p.target_kind == 0 ? -0.5 * zz * zz : -0.5 * (p.target_df + 1.0) * log1p(zz * zz / p.target_df);
            }
          }
        part += __shfl_xor_sync(0xffffffffu, part, 1);
        part += __shfl_xor_sync(0xffffffffu, part, 2);
        if (t == 0) s_red[wn * kLrM + r] = part;
      }
      __syncthreads();
      if (tid < kLrM) s_lp[tid] += ((s_red[tid] + s_red[kLrM + tid]) + s_red[2 * kLrM + tid]) + s_red[3 * kLrM + tid];
      __syncthreads();                       // s_red is rewritten by the next column block
    }
    __syncthreads();
    if (tid < rows) {
      const double lq = lqc - 0.5 * (s_uu[tid] - s_ww[tid]);
      p.lw[i0 - p.first + tid] = (p.target_kind >= 0 ? s_lp[tid] + pconst : 0.0) - lq;
    }
  }
}

// once per call: sigma = exp(log_sigma) and the two per-call constants, each a fixed-order block sum
__global__ void __launch_bounds__(256) lr_stream_prep_kernel(const double* vp, const double* P, int d, int k,
                                                              int target_kind, const double* scale, double target_const,
                                                              double* consts, double* sig) {
  __shared__ double red[32];
  double a = 0.0, b = 0.0, c = 0.0;
  for (int j = threadIdx.x; j < d; j += blockDim.x) {
    const double ls = vp[d + j];
    sig[j] = exp(ls);
    a += ls;
    if (target_kind >= 0) c += log(scale[j]);
  }
  for (int l = threadIdx.x; l < k; l += blockDim.x) b += log(P[(size_t)l * (k + d) + l]);
  a = block_sum(a, red);
  b = block_sum(b, red);
  c = block_sum(c, red);
  if (threadIdx.x == 0) {
    consts[0] = -0.5 * kLog2Pi * d - a + b;
    consts[1] = target_const - c;
  }
}

static inline int lr_kq(int k) { return k >= kLrWN ? kLrWN : (k + 7) / 8 * 8; }

static inline size_t lr_smem(bool ushared, int d, int k) {
  return sizeof(double) * ((size_t)7 * kLrM + (size_t)8 * kLrM * lr_kq(k) +
                           (ushared ? (size_t)kLrM * (lr_ld(k) + lr_ld(d)) : 0));
}

// CTAs per launch (persistent grid: as many as can be resident)
static int lr_ctas(int d, int k, int64_t* ctas) {
  const bool ushared = k + d <= kLrUSharedMax;
  auto kern = ushared ? lr_stream_lw_kernel<true> : lr_stream_lw_kernel<false>;
  const size_t smem = lr_smem(ushared, d, k);
  VB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  VB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem));
  if (per_sm < 1) return set_error(VB_ERR_UNSUPPORTED, "lr_target_log_weights: kernel does not fit on an SM");
  *ctas = (int64_t)per_sm * sm_count();
  return VB_OK;
}

// 256 bytes of constants, sigma[d], then one 32-row u tile per resident CTA when k + d > 512
static size_t lr_ws_layout(int d, int k, int64_t ctas, size_t* off_sig, size_t* off_u) {
  *off_sig = 256;
  *off_u = 256 + align_up(sizeof(double) * (size_t)d, 256);
  return *off_u + (k + d > kLrUSharedMax ? sizeof(double) * (size_t)ctas * kLrM * (lr_ld(k) + lr_ld(d)) : 0);
}

static inline double lr_t_coord_const(double df) {
  return lgamma(0.5 * (df + 1.0)) - lgamma(0.5 * df) - 0.5 * log(df * 3.14159265358979323846);
}

}  // namespace vb
using namespace vb;

/* workspace: 256 bytes + sigma[d], plus one 32 x (k + d) float64 u tile per resident CTA when k + d > 512; independent
 * of n */
extern "C" size_t vb_lr_target_log_weights_workspace_bytes(int d, int k) {
  if (d <= 0 || k < 0 || (int64_t)k + d >= kLrMaxWidth) return 0;
  int64_t ctas = 0;
  if (lr_ctas(d, k, &ctas)) return 0;
  size_t off_sig, off_u;
  return lr_ws_layout(d, k, ctas, &off_sig, &off_u);
}

/* lw[count] = log p(theta_i) - log q(theta_i) for draws i = first .. first + count - 1 of n_total (see the top of
 * this file); theta_out[count, d] optional. */
extern "C" int vb_lr_target_log_weights_f64(const double* var_param, const double* P, int64_t n_total, int64_t first,
                                            int64_t count, int d, int k, uint64_t seed, uint64_t offset,
                                            int target_kind, const double* target_loc, const double* target_scale,
                                            double target_df, double* lw, double* theta_out, void* workspace,
                                            size_t workspace_bytes, cudaStream_t stream) {
  if (!var_param || d <= 0 || k < 0 || (k > 0 && !P) || n_total < 0 || first < 0 || count < 0 ||
      count > n_total - first || (count > 0 && !lw))
    return set_error(VB_ERR_INVALID_ARG, "lr_target_log_weights: bad arguments");
  if (n_total > (INT64_MAX / 2) / ((int64_t)d + k))
    return set_error(VB_ERR_INVALID_ARG, "lr_target_log_weights: n_total * (d + k) too large");
  if (target_kind < -1 || target_kind > 1)
    return set_error(VB_ERR_INVALID_ARG, "lr_target_log_weights: target_kind is -1 (none), 0 (Gaussian) or 1 (Student-t)");
  if (target_kind >= 0 && (!target_loc || !target_scale))
    return set_error(VB_ERR_INVALID_ARG, "lr_target_log_weights: bad arguments");
  if (target_kind == 1 && !(target_df > 0.0))
    return set_error(VB_ERR_INVALID_ARG, "lr_target_log_weights: target_df must be positive");
  if ((int64_t)k + d >= kLrMaxWidth) return set_error(VB_ERR_UNSUPPORTED, "lr_target_log_weights: k + d too large");
  int64_t ctas = 0;
  int rc = lr_ctas(d, k, &ctas);
  if (rc) return rc;
  size_t off_sig, off_u;
  if (!workspace || workspace_bytes < lr_ws_layout(d, k, ctas, &off_sig, &off_u))
    return set_error(VB_ERR_WORKSPACE, "lr_target_log_weights: workspace too small");
  if (count == 0) return VB_OK;
  const int64_t tiles = ceil_div(count, kLrM);
  const int64_t grid = tiles < ctas ? tiles : ctas;
  if (grid > INT32_MAX) return set_error(VB_ERR_UNSUPPORTED, "lr_target_log_weights: more than 2^31 - 1 CTAs");
  char* ws = static_cast<char*>(workspace);
  double* consts = reinterpret_cast<double*>(ws);
  double* sig = reinterpret_cast<double*>(ws + off_sig);
  const double target_const =
      target_kind == 0 ? -0.5 * kLog2Pi * d : target_kind == 1 ? d * lr_t_coord_const(target_df) : 0.0;
  lr_stream_prep_kernel<<<1, 256, 0, stream>>>(var_param, P, d, k, target_kind, target_scale, target_const, consts, sig);
  VB_CHECK_LAUNCH();
  LrStreamArgs p;
  p.vp = var_param;
  p.P = P;
  p.consts = consts;
  p.sig = sig;
  p.loc = target_loc;
  p.scale = target_scale;
  p.lw = lw;
  p.theta_out = theta_out;
  p.uws = reinterpret_cast<double*>(ws + off_u);
  p.first = first;
  p.count = count;
  p.seed = seed;
  const uint64_t nk = (uint64_t)n_total * k;
  p.z_off = offset;
  p.e_off = offset + nk + (nk & 1);
  p.d = d;
  p.k = k;
  p.ldz = lr_ld(k);
  p.lde = lr_ld(d);
  p.kq = lr_kq(k);
  p.target_kind = target_kind;
  p.target_df = target_df;
  const bool ushared = k + d <= kLrUSharedMax;
  if (ushared)
    lr_stream_lw_kernel<true><<<(unsigned)grid, 256, lr_smem(true, d, k), stream>>>(p);
  else
    lr_stream_lw_kernel<false><<<(unsigned)grid, 256, lr_smem(false, d, k), stream>>>(p);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
