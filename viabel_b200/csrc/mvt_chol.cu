// Cholesky reparameterisation of the full-rank MultivariateT family (MultivariateT(..., reparam='cholesky')):
//
//     theta_s = mu + L zhat_s,   zhat_s = z_s / u_s,   L = tril(F,-1) + diag(exp(diag F)),   var_param = [mu, tril(F)]
//
// LL^T = Sigma, so the draws have the distribution of the reference's sqrtm map (approximations.py:342-349) and the
// ExclusiveKL / AlphaDivergence objectives are the same functions of var_param; only the per-draw mapping differs.
// Nothing here needs an eigensolver or a d x d temporary:
//
//     transform   theta = mu + diag(1/u) Z L^T                       (B operand: rows of L read from the packed triangle)
//     cotangent   Fbar[i,j] = c sum_s sv_s G[s,i] zhat_s[j]   (j < i)
//                 Fbar[i,i] = (c sum_s sv_s G[s,i] zhat_s[i]) L_ii + diag_add
//
// with c = -1/S (ExclusiveKL, sv = 1) or alpha/S (AlphaDivergence); the value, the weights sv and diag_add come from
// the kernels the sqrtm path uses (mvt_internal.cuh), because log q at a reparameterised draw is the same closed form.
//
// Both products run on the FP64 tensor pipe (mma.sync m8n8k4 f64, DMMA) with one warp owning each output fragment and
// a fixed k order: no split-K, no atomics, so repeated calls give identical bits.  Workspace is O(S).
#include "mvt_internal.cuh"

namespace vb {

constexpr int kSlab = 32;                    // K slab through shared memory
constexpr int kTN = 64;                      // output tile width (columns of theta / of Fbar)
constexpr int kTM = 32;                      // transform: rows (samples) per tile
constexpr int kPadM = kTM + 4, kPadN = kTN + 4;   // row pitches; conflict-free fragment reads

// ---- triangular transform ------------------------------------------------------------------------------------------
// Column block b of theta needs the K range [0, 64 (b + 1)): its work grows with b.  CTA (p, r) computes rows
// [32 r, 32 r + 32) of column blocks p and nb - 1 - p, so every CTA does nb + 1 slabs of 64 -- at S = 256, d = 2048 that
// is 8 x 16 = 128 equal CTAs, one wave on 148 SMs.  8 warps, each a 16 x 16 fragment of the 32 x 64 tile; the next
// slab is loaded into registers while the current one is multiplied.  The CTAs are numbered p-fastest on a 1-D grid
// (gridDim.y would cap S at 65535 row tiles).
struct TrmmStage {
  double a[kSlab * kTM / 256];               // Z[s, k]
  double b[kSlab * kTN / 256];               // L[n, k]
};

__device__ __forceinline__ void trmm_load(TrmmStage& st, const double* __restrict__ vp, const double* __restrict__ z, int S,
                                          int d, int m0, int n0, int k0) {
  const int k = threadIdx.x & 31, r = threadIdx.x >> 5;
  const int kk = k0 + k;
#pragma unroll
  for (int p = 0; p < kTM / 8; ++p) {
    const int s = m0 + p * 8 + r;
    st.a[p] = (s < S && kk < d) ? z[(size_t)s * d + kk] : 0.0;
  }
#pragma unroll
  for (int p = 0; p < kTN / 8; ++p) {
    const int n = n0 + p * 8 + r;
    double v = 0.0;
    if (n < d && kk <= n) {
      v = vp[d + tri(n) + kk];               // row n of L is contiguous in k
      if (kk == n) v = exp(v);
    }
    st.b[p] = v;
  }
}

__device__ __forceinline__ void trmm_store(const TrmmStage& st, double (*sa)[kPadM], double (*sb)[kPadN]) {
  const int k = threadIdx.x & 31, r = threadIdx.x >> 5;
#pragma unroll
  for (int p = 0; p < kTM / 8; ++p) sa[k][p * 8 + r] = st.a[p];
#pragma unroll
  for (int p = 0; p < kTN / 8; ++p) sb[k][p * 8 + r] = st.b[p];
}

__global__ void __launch_bounds__(256) mvt_chol_trmm_kernel(const double* __restrict__ vp, const double* __restrict__ z,
                                                            const double* __restrict__ inv_u, int S, int d,
                                                            double* __restrict__ theta) {
  __shared__ double sa[kSlab][kPadM], sb[kSlab][kPadN];
  const int nb = (d + kTN - 1) / kTN;
  const unsigned npairs = (unsigned)(nb + 1) / 2;
  const int pair = (int)(blockIdx.x % npairs);
  const int m0 = (int)(blockIdx.x / npairs) * kTM;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wm = warp >> 2, wn = warp & 3;
  const int gq = lane >> 2, t = lane & 3;
  const int cb0 = pair, cb1 = nb - 1 - pair;
  // flattened (column block, slab) sequence; column block c takes ceil(min(d, 64 (c+1)) / 32) slabs
  const int ns0 = (min(d, (cb0 + 1) * kTN) + kSlab - 1) / kSlab;
  const int total = ns0 + (cb1 == cb0 ? 0 : (min(d, (cb1 + 1) * kTN) + kSlab - 1) / kSlab);

  double acc[2][2][2];
  TrmmStage st;
  trmm_load(st, vp, z, S, d, m0, cb0 * kTN, 0);
  for (int it = 0; it < total; ++it) {
    const bool second = it >= ns0;
    const int sl = second ? it - ns0 : it;
    const int n0 = (second ? cb1 : cb0) * kTN;
    const int nsl = second ? total - ns0 : ns0;
    if (sl == 0) {
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
    }
    __syncthreads();
    trmm_store(st, sa, sb);
    __syncthreads();
    if (it + 1 < total) {
      const bool second1 = it + 1 >= ns0;
      trmm_load(st, vp, z, S, d, m0, (second1 ? cb1 : cb0) * kTN, (second1 ? it + 1 - ns0 : it + 1) * kSlab);
    }
#pragma unroll
    for (int k4 = 0; k4 < kSlab; k4 += 4) {
      double af[2], bf[2];
#pragma unroll
      for (int a = 0; a < 2; ++a) af[a] = sa[k4 + t][wm * 16 + a * 8 + gq];
#pragma unroll
      for (int b = 0; b < 2; ++b) bf[b] = sb[k4 + t][wn * 16 + b * 8 + gq];
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) dmma(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
    }
    if (sl + 1 == nsl) {                   // last slab of this column block: epilogue
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        const int s = m0 + wm * 16 + a * 8 + gq;
        if (s >= S) continue;
        const double iu = inv_u[s];
#pragma unroll
        for (int b = 0; b < 2; ++b)
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int n = n0 + wn * 16 + b * 8 + 2 * t + u;
            if (n < d) theta[(size_t)s * d + n] = vp[n] + iu * acc[a][b][u];
          }
      }
    }
  }
}

// ---- cotangent ---------------------------------------------------------------------------------------------------
// Fbar = G^T diag(c sv / u) Z on the lower-triangular 64 x 64 tiles only (one CTA per tile, K = S), written straight
// into the packed gradient.  8 warps of 16 x 32 fragments; register-prefetched slabs as above.
struct CotStage {
  double a[kSlab * kTN / 256];               // w_s G[s, i]
  double b[kSlab * kTN / 256];               // Z[s, j]
};

__device__ __forceinline__ void cot_load(CotStage& st, const double* __restrict__ G, const double* __restrict__ z,
                                         const double* __restrict__ sv, const double* __restrict__ inv_u, double c, int S,
                                         int d, int i0, int j0, int k0) {
  const int col = threadIdx.x & 63, r = threadIdx.x >> 6;
#pragma unroll
  for (int p = 0; p < kSlab / 4; ++p) {
    const int s = k0 + p * 4 + r;
    double va = 0.0, vb = 0.0;
    if (s < S) {
      if (i0 + col < d) va = G[(size_t)s * d + i0 + col] * (c * sv[s] * inv_u[s]);
      if (j0 + col < d) vb = z[(size_t)s * d + j0 + col];
    }
    st.a[p] = va;
    st.b[p] = vb;
  }
}

__global__ void __launch_bounds__(256) mvt_chol_cotangent_kernel(const double* __restrict__ vp, const double* __restrict__ z,
                                                                 const double* __restrict__ inv_u, const double* __restrict__ G,
                                                                 const double* __restrict__ sv, const double* __restrict__ scal,
                                                                 double c, int S, int d, double* __restrict__ grad) {
  __shared__ double sa[kSlab][kPadN], sb[kSlab][kPadN];
  // lower-triangular tile index -> (bi, bj), bj <= bi
  const int64_t tix = blockIdx.x;
  int bi = (int)((sqrt(8.0 * (double)tix + 1.0) - 1.0) * 0.5);
  while (tri(bi) > tix) --bi;
  while (tri(bi + 1) <= tix) ++bi;
  const int bj = (int)(tix - tri(bi));
  const int i0 = bi * kTN, j0 = bj * kTN;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wm = warp >> 1, wn = warp & 1;
  const int gq = lane >> 2, t = lane & 3;
  double acc[2][4][2];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;

  const int col = threadIdx.x & 63, r = threadIdx.x >> 6;
  CotStage st;
  cot_load(st, G, z, sv, inv_u, c, S, d, i0, j0, 0);
  for (int k0 = 0; k0 < S; k0 += kSlab) {
    __syncthreads();
#pragma unroll
    for (int p = 0; p < kSlab / 4; ++p) {
      sa[p * 4 + r][col] = st.a[p];
      sb[p * 4 + r][col] = st.b[p];
    }
    __syncthreads();
    if (k0 + kSlab < S) cot_load(st, G, z, sv, inv_u, c, S, d, i0, j0, k0 + kSlab);
#pragma unroll
    for (int k4 = 0; k4 < kSlab; k4 += 4) {
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
  }
  const double diag_add = scal[1];
#pragma unroll
  for (int a = 0; a < 2; ++a) {
    const int i = i0 + wm * 16 + a * 8 + gq;
    if (i >= d) continue;
    double* row = grad + d + tri(i);
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int j = j0 + wn * 32 + b * 8 + 2 * t + u;
        if (j > i) continue;
        const double v = acc[a][b][u];
        row[j] = j == i ? v * exp(vp[d + tri(i) + i]) + diag_add : v;
      }
  }
}

struct CholObjLayout {
  size_t off_sv, off_scal, off_hl, total;
};
static void chol_obj_layout(int S, CholObjLayout& l) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  l.off_sv = take(sizeof(double) * S);
  l.off_scal = take(sizeof(double) * 4);
  l.off_hl = take(sizeof(double));
  l.total = off;
}

}  // namespace vb
using namespace vb;

/* theta[S,d] = mu + diag(1/u) z L^T (MultivariateT.sample with reparam='cholesky'; the reference's sample is
 * approximations.py:342-349), inv_u[S] = 1/u, zu2[S] = |z_s / u_s|^2, u_s = sqrt(chi2_s / df). */
extern "C" int vb_mvt_chol_transform_f64(const double* var_param, const double* z, const double* chi2, double df, int S, int d,
                                         double* theta, double* inv_u, double* zu2, cudaStream_t stream) {
  if (!var_param || !z || !chi2 || S <= 0 || d <= 0 || !theta || !inv_u || !zu2)
    return set_error(VB_ERR_INVALID_ARG, "mvt_chol_transform: bad arguments");
  if (!(df > 2.0)) return set_error(VB_ERR_INVALID_ARG, "df must be greater than 2");
  int rc = mvt_rows(z, chi2, df, S, d, inv_u, zu2, stream);
  if (rc) return rc;
  const int64_t nb = ceil_div(d, kTN);
  const int64_t ctas = (nb + 1) / 2 * ceil_div(S, kTM);
  if (ctas > INT32_MAX) return set_error(VB_ERR_UNSUPPORTED, "mvt_chol_transform: more than 2^31 - 1 tiles");
  mvt_chol_trmm_kernel<<<(unsigned)ctas, 256, 0, stream>>>(var_param, z, inv_u, S, d, theta);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

/* workspace: S + 5 doubles (256-byte aligned pieces) */
extern "C" size_t vb_mvt_chol_objective_workspace_bytes(int S, int d) {
  if (S <= 0 || d <= 0) return 0;
  CholObjLayout l;
  chol_obj_layout(S, l);
  return l.total;
}

/* value[1] and grad[d + d(d+1)/2] of ExclusiveKL (entropy form) / AlphaDivergence (objectives.py:154-164, :443-460)
 * in the Cholesky reparameterisation, from the model's f[S] and G[S,d] at theta and inv_u / zu2 of
 * vb_mvt_chol_transform_f64. */
extern "C" int vb_mvt_chol_objective_f64(const double* var_param, const double* z, const double* inv_u, const double* zu2,
                                         const double* f, const double* G, int S, int d, double df, int objective, double alpha,
                                         double* value, double* grad, void* workspace, size_t workspace_bytes,
                                         cudaStream_t stream) {
  if (!var_param || !z || !inv_u || !zu2 || !f || !G || S <= 0 || d <= 0 || !value || !grad)
    return set_error(VB_ERR_INVALID_ARG, "mvt_chol_objective: bad arguments");
  if (objective != VB_OBJ_EXCLUSIVE_KL && objective != VB_OBJ_ALPHA)
    return set_error(VB_ERR_UNSUPPORTED, "path-derivative estimator is not available for MultivariateT");
  CholObjLayout l;
  chol_obj_layout(S, l);
  if (!workspace || workspace_bytes < l.total) return set_error(VB_ERR_WORKSPACE, "mvt_chol_objective: workspace too small");
  char* ws = static_cast<char*>(workspace);
  double* sv = reinterpret_cast<double*>(ws + l.off_sv);
  double* scal = reinterpret_cast<double*>(ws + l.off_scal);
  double* hl = reinterpret_cast<double*>(ws + l.off_hl);
  int rc = mvt_logdiag(var_param, d, hl, stream);
  if (rc) return rc;
  rc = mvt_weights_gmu(f, G, zu2, hl, S, d, df, objective, alpha, sv, scal, value, grad, stream);
  if (rc) return rc;
  const double c = objective == VB_OBJ_EXCLUSIVE_KL ? -1.0 / S : alpha / S;
  const int nb = (d + kTN - 1) / kTN;
  mvt_chol_cotangent_kernel<<<(unsigned)(nb * (nb + 1) / 2), 256, 0, stream>>>(var_param, z, inv_u, G, sv, scal, c, S, d, grad);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
