// Streaming log-weights of the full-rank MultivariateT family for vi_diagnostics at scale (the mean-field version is
// stream_lw.cu).  Draw i of n_total is regenerated from the family's Philox stream by offset -- chi2_i is element
// offset + i of the chi-square stream, z_i[j] element offset + n_total + (n_total & 1) + i d + j of the normal stream,
// exactly what MultivariateT.base_draws(n_total) draws -- and
//
//     zhat_i = z_i / u_i,   u_i = sqrt(chi2_i / df),   theta_i = mu + M zhat_i
//     log q_i = lgamma((df + d)/2) - lgamma(df/2) - d/2 log(pi df) - sum_j F_jj - (df + d)/2 log1p(|zhat_i|^2 / df)
//     lw_i = log p(theta_i) - log q_i            (product Gaussian / Student-t target, or -log q_i with no target)
//
// with M = L read from the packed triangle of var_param (Cholesky mode, triangular product) or a dense d x d map
// A = V diag(sqrt w) V^T formed by the caller (sqrtm mode).  log q at a reparameterised draw is a closed form in
// |zhat|^2 (the identity mvt_weights_kernel uses), so no solve and no eigensolver runs per draw.
//
// Persistent grid; a CTA takes 32 draws at a time and owns every column block of them, so every tile does the same
// work and the per-draw sum of target terms stays in the CTA.  The tile's z rows are generated once into shared memory
// (d <= 512) or into the CTA's slice of the workspace (L2 resident), then theta = mu + diag(1/u) Z M^T runs on the
// FP64 tensor pipe (mma.sync m8n8k4 f64) over 128-wide column blocks: 8 warps of 16 x 32, 8 independent accumulators
// per warp, register-prefetched 32-deep K slabs; the triangular case skips the slabs above the diagonal.  The
// epilogue adds mu, scales by 1/u and sums the target terms over lanes and warps into a per-draw accumulator in a
// fixed order.  No atomics and nothing depends on where a draw sits in its tile, so repeated calls give identical
// bits and a slice computed alone equals the same draws of a longer call.  Nothing of size n d is stored unless the
// caller asks for theta_out.
#include "mvt_internal.cuh"
#include "philox_draws.cuh"
#include "stream_internal.cuh"

namespace vb {

constexpr int kSM = kTileM;                  // draws per tile
constexpr int kSN = kTileN;                  // column block width
constexpr int kSK = 32;                      // K slab
constexpr int kSPadM = kSM + 4, kSPadN = kSN + 4;
constexpr int kZSharedMaxDim = 512;          // z tile in shared memory up to here (128 KB)

struct MvtStreamArgs {
  const double* vp;
  const double* A;                           // NULL: Cholesky mode
  const double* half_logdet;                 // sum_j F_jj
  const double* loc;
  const double* scale;
  double* lw;
  double* theta_out;
  double* zws;                               // per-CTA z tiles when they do not fit in shared memory
  int64_t first, count;
  uint64_t seed, chi_off, z_off;
  int d, target_kind;
  double df, logq_const, target_df, target_const;   // target_const: d x the per-coordinate constant
};

struct StreamStage {
  double a[kSK * kSM / 256];                 // zhat tile rows (unscaled z)
  double b[kSK * kSN / 256];                 // rows of M
};

__device__ __forceinline__ void stream_load(StreamStage& st, const MvtStreamArgs& p, const double* zt, int rows, int n0,
                                            int k0) {
  const int k = threadIdx.x & 31, r = threadIdx.x >> 5;
  const int d = p.d, kk = k0 + k;
#pragma unroll
  for (int q = 0; q < kSM / 8; ++q) {
    const int m = q * 8 + r;
    st.a[q] = (m < rows && kk < d) ? zt[(size_t)m * d + kk] : 0.0;
  }
#pragma unroll
  for (int q = 0; q < kSN / 8; ++q) {
    const int n = n0 + q * 8 + r;
    double v = 0.0;
    if (p.A) {
      if (n < d && kk < d) v = p.A[(size_t)n * d + kk];
    } else if (n < d && kk <= n) {
      v = p.vp[d + tri(n) + kk];             // row n of L is contiguous in k
      if (kk == n) v = exp(v);
    }
    st.b[q] = v;
  }
}

template <bool kZShared>
__global__ void __launch_bounds__(256, 2) mvt_stream_lw_kernel(const MvtStreamArgs p) {
  extern __shared__ double sh[];
  double(*sa)[kSPadM] = reinterpret_cast<double(*)[kSPadM]>(sh);
  double(*sb)[kSPadN] = reinterpret_cast<double(*)[kSPadN]>(sh + kSK * kSPadM);
  double* s_iu = sh + kSK * (kSPadM + kSPadN);
  double* s_zu2 = s_iu + kSM;
  double* s_lp = s_zu2 + kSM;
  double* s_red = s_lp + kSM;                // [4][kSM]: per-warp-column partial sums
  double* s_misc = s_red + 4 * kSM;          // [32] block_sum scratch
  double* zt = kZShared ? s_misc + 32 : p.zws + (size_t)blockIdx.x * kSM * p.d;

  const int d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3;
  const int gq = lane >> 2, t = lane & 3;
  const bool dense = p.A != nullptr;
  const int nb = (d + kSN - 1) / kSN;
  const int dslabs = (d + kSK - 1) / kSK;

  // target_const - sum_j log scale_j: the same fixed-order sum in every CTA
  double pconst = 0.0;
  if (p.target_kind >= 0) pconst = product_target_log_const(p.target_const, p.scale, d, s_misc);
  const double hl = p.half_logdet[0];
  const Philox ph(p.seed);
  const int64_t ntiles = (p.count + kSM - 1) / kSM;

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t i0 = p.first + tile * kSM;
    const int rows = (int)min((int64_t)kSM, p.first + p.count - i0);
    __syncthreads();                         // the previous tile is done with zt and the per-draw arrays
    // z rows of the tile: elements e0 .. e0 + rows d - 1 of the normal stream, one Box-Muller pair per counter
    {
      const uint64_t e0 = p.z_off + (uint64_t)i0 * d;
      const int64_t ne = (int64_t)rows * d;
      const uint64_t c0 = e0 >> 1, c1 = (e0 + ne - 1) >> 1;
      for (uint64_t c = c0 + tid; c <= c1; c += blockDim.x) {
        double z0, z1;
        normal_pair(ph, c, 0, z0, z1);
        const int64_t l = (int64_t)(2 * c - e0);
        if (l >= 0) zt[l] = z0;
        if (l + 1 < ne) zt[l + 1] = z1;
      }
    }
    if (tid < rows) s_iu[tid] = 1.0 / sqrt(2.0 * gamma_draw(ph, p.chi_off + (uint64_t)(i0 + tid), 1, 0.5 * p.df) / p.df);
    if (tid < kSM) s_lp[tid] = 0.0;
    __syncthreads();
    // |zhat|^2 per draw, in mvt_rows_kernel's order
    for (int r = warp; r < rows; r += 8) {
      const double iu = s_iu[r];
      double a = 0.0;
      for (int j = lane; j < d; j += 32) {
        const double v = zt[(size_t)r * d + j] * iu;
        a += v * v;
      }
      a = warp_sum(a);
      if (lane == 0) s_zu2[r] = a;
    }

    // flattened (column block, K slab) sequence; column block c takes all d / 32 slabs (dense) or those up to its
    // diagonal (triangular)
    auto nslabs = [&](int cb) { return dense ? dslabs : (min(d, (cb + 1) * kSN) + kSK - 1) / kSK; };
    int cb = 0, sl = 0, ns = nslabs(0);
    double acc[2][4][2];
    StreamStage st;
    stream_load(st, p, zt, rows, 0, 0);
    while (true) {
      if (sl == 0) {
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
      }
      __syncthreads();
      {
        const int k = tid & 31, r = tid >> 5;
#pragma unroll
        for (int q = 0; q < kSM / 8; ++q) sa[k][q * 8 + r] = st.a[q];
#pragma unroll
        for (int q = 0; q < kSN / 8; ++q) sb[k][q * 8 + r] = st.b[q];
      }
      __syncthreads();
      int ncb = cb, nsl = sl + 1;
      if (nsl == ns) {
        ++ncb;
        nsl = 0;
      }
      if (ncb < nb) stream_load(st, p, zt, rows, ncb * kSN, nsl * kSK);
#pragma unroll
      for (int k4 = 0; k4 < kSK; k4 += 4) {
        double af[2], bf[4];
#pragma unroll
        for (int a = 0; a < 2; ++a) af[a] = sa[k4 + t][wm * 16 + a * 8 + gq];
#pragma unroll
        for (int b = 0; b < 4; ++b) bf[b] = sb[k4 + t][wn * 32 + b * 8 + gq];
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) dmma(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
      }
      if (sl + 1 == ns)                      // last slab of column block cb: epilogue
        target_tile_epilogue(p, acc, i0, rows, cb * kSN, s_red, s_lp, [&](int r) {
          const double iu = s_iu[r];
          return [&p, iu](int n, double v) { return p.vp[n] + iu * v; };
        });
      if (ncb >= nb) break;
      if (ncb != cb) ns = nslabs(ncb);
      cb = ncb;
      sl = nsl;
    }
    __syncthreads();
    if (tid < rows) {
      const double lq = p.logq_const - hl - 0.5 * (p.df + d) * log1p(s_zu2[tid] / p.df);
      p.lw[i0 - p.first + tid] = (p.target_kind >= 0 ? s_lp[tid] + pconst : 0.0) - lq;
    }
  }
}

static inline size_t stream_smem(bool zshared, int d) {
  return sizeof(double) * ((size_t)kSK * (kSPadM + kSPadN) + 7 * kSM + 32 + (zshared ? (size_t)kSM * d : 0));
}

// CTAs per launch; the workspace holds one z tile per CTA for d > 512
static int stream_ctas(int d, int64_t* ctas) {
  const bool zshared = d <= kZSharedMaxDim;
  return persistent_ctas(zshared ? mvt_stream_lw_kernel<true> : mvt_stream_lw_kernel<false>, 256, stream_smem(zshared, d),
                         ctas);
}

static size_t stream_ws_layout(int d, int64_t ctas, size_t* off_z) {
  *off_z = 256;
  return 256 + (d > kZSharedMaxDim ? sizeof(double) * (size_t)ctas * kSM * d : 0);
}

}  // namespace vb
using namespace vb;

/* workspace: 256 bytes, plus one 32 x d float64 z tile per resident CTA when d > 512; independent of n */
extern "C" size_t vb_mvt_target_log_weights_workspace_bytes(int d) {
  if (d <= 0) return 0;
  int64_t ctas = 0;
  if (stream_ctas(d, &ctas)) return 0;
  size_t off_z;
  return stream_ws_layout(d, ctas, &off_z);
}

/* lw[count] = log p(theta_i) - log q(theta_i) for draws i = first .. first + count - 1 of n_total (see the top of
 * this file); theta_out[count, d] optional. */
extern "C" int vb_mvt_target_log_weights_f64(const double* var_param, const double* A, int64_t n_total, int64_t first,
                                             int64_t count, int d, double df, uint64_t seed, uint64_t offset,
                                             int target_kind, const double* target_loc, const double* target_scale,
                                             double target_df, double* lw, double* theta_out, void* workspace,
                                             size_t workspace_bytes, cudaStream_t stream) {
  if (!var_param || d <= 0 || n_total < 0 || first < 0 || count < 0 || count > n_total - first || (count > 0 && !lw))
    return set_error(VB_ERR_INVALID_ARG, "mvt_target_log_weights: bad arguments");
  if (n_total > (INT64_MAX / 2) / d) return set_error(VB_ERR_INVALID_ARG, "mvt_target_log_weights: n_total * d too large");
  if (!(df > 2.0)) return set_error(VB_ERR_INVALID_ARG, "df must be greater than 2");
  int rc = check_product_target("mvt_target_log_weights", target_kind, true, target_loc, target_scale, target_df);
  if (rc) return rc;
  int64_t ctas = 0;
  rc = stream_ctas(d, &ctas);
  if (rc) return rc;
  size_t off_z;
  if (!workspace || workspace_bytes < stream_ws_layout(d, ctas, &off_z))
    return set_error(VB_ERR_WORKSPACE, "mvt_target_log_weights: workspace too small");
  if (count == 0) return VB_OK;
  const int64_t tiles = ceil_div(count, kSM), grid = tiles < ctas ? tiles : ctas;
  char* ws = static_cast<char*>(workspace);
  MvtStreamArgs p;
  p.vp = var_param;
  p.A = A;
  p.half_logdet = reinterpret_cast<double*>(ws);
  p.loc = target_loc;
  p.scale = target_scale;
  p.lw = lw;
  p.theta_out = theta_out;
  p.zws = reinterpret_cast<double*>(ws + off_z);
  p.first = first;
  p.count = count;
  p.seed = seed;
  p.chi_off = offset;
  p.z_off = offset + (uint64_t)n_total + ((uint64_t)n_total & 1);
  p.d = d;
  p.target_kind = target_kind;
  p.df = df;
  p.logq_const = mvt_const(df, d);
  p.target_df = target_df;
  p.target_const = product_target_const(target_kind, d, target_df);
  rc = mvt_logdiag(var_param, d, reinterpret_cast<double*>(ws), stream);
  if (rc) return rc;
  const bool zshared = d <= kZSharedMaxDim;
  if (zshared)
    mvt_stream_lw_kernel<true><<<(unsigned)grid, 256, stream_smem(true, d), stream>>>(p);
  else
    mvt_stream_lw_kernel<false><<<(unsigned)grid, 256, stream_smem(false, d), stream>>>(p);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
