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
// The path-derivative ExclusiveKL feeds the cotangent G + diag(kappa) Zhat L^-1 instead of G (below) and needs a
// d x d inverse: its workspace is O(d^2 + S d).
//
// Both products run on the FP64 tensor pipe (mma.sync m8n8k4 f64, DMMA) with one warp owning each output fragment and
// a fixed k order: no split-K, no atomics, so repeated calls give identical bits.  Workspace is O(S) (entropy form,
// AlphaDivergence).
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

template <bool kScore>
__device__ __forceinline__ void trmm_load(TrmmStage& st, const double* __restrict__ vp, const double* __restrict__ z,
                                          const long long* __restrict__ idx, const double* __restrict__ X, int S, int d,
                                          int m0, int n0, int k0) {
  const int k = threadIdx.x & 31, r = threadIdx.x >> 5;
  const int kk = k0 + k;
#pragma unroll
  for (int p = 0; p < kTM / 8; ++p) {
    const int s = m0 + p * 8 + r;
    double v = 0.0;
    if (s < S && kk < d) {
      if (kScore) v = z[(size_t)(idx ? idx[s] : s) * d + kk] - vp[kk];     // x - mu before the product
      else v = z[(size_t)s * d + kk];
    }
    st.a[p] = v;
  }
#pragma unroll
  for (int p = 0; p < kTN / 8; ++p) {
    const int n = n0 + p * 8 + r;
    double v = 0.0;
    if (n < d && kk <= n) {
      if (kScore) {
        v = X[(size_t)n * d + kk];           // row n of L^-1
      } else {
        v = vp[d + tri(n) + kk];             // row n of L is contiguous in k
        if (kk == n) v = exp(v);
      }
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

// kScore: Y = (x[idx] - mu) L^-T for the DIS score (below), with B read from the dense L^-1 X and no epilogue scaling.
template <bool kScore>
__global__ void __launch_bounds__(256) mvt_chol_trmm_kernel(const double* __restrict__ vp, const double* __restrict__ z,
                                                            const long long* __restrict__ idx, const double* __restrict__ X,
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
  trmm_load<kScore>(st, vp, z, idx, X, S, d, m0, cb0 * kTN, 0);
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
      trmm_load<kScore>(st, vp, z, idx, X, S, d, m0, (second1 ? cb1 : cb0) * kTN, (second1 ? it + 1 - ns0 : it + 1) * kSlab);
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
        const double iu = kScore ? 1.0 : inv_u[s];
#pragma unroll
        for (int b = 0; b < 2; ++b)
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int n = n0 + wn * 16 + b * 8 + 2 * t + u;
            if (n < d) theta[(size_t)s * d + n] = kScore ? acc[a][b][u] : vp[n] + iu * acc[a][b][u];
          }
      }
    }
  }
}

// ---- cotangent ---------------------------------------------------------------------------------------------------
// Fbar = G^T diag(c sv / u) Z on the lower-triangular 64 x 64 tiles only (one CTA per tile, K = S), written straight
// into the packed gradient; inv_u NULL means u = 1 (the DIS score).  8 warps of 16 x 32 fragments; register-prefetched slabs as above.
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
      if (i0 + col < d) va = G[(size_t)s * d + i0 + col] * (inv_u ? c * sv[s] * inv_u[s] : c * sv[s]);
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

// ---- path-derivative ExclusiveKL: G + diag(kappa) Y,  Y = Zhat L^-1 ------------------------------------------------
// The path gradient is the cotangent above with G_s replaced by G_s + kappa_s y_s (minus the score of log q at a
// var_param held fixed), y_s = Sigma^-1 (theta_s - mu) = L^-T zhat_s, kappa_s = (df + d) / (df + |zhat_s|^2), and no
// entropy term.  As rows Y = Zhat X with X = L^-1, which is formed on the device in three steps:
//   1. the ceil(d/64) diagonal 64 x 64 blocks of X by substitution in shared memory, one CTA each;
//   2. log2 doubling levels: at half-size h, blocks [r0, r0 + h) and [r0 + h, r0 + 2h) (r0 = 2 h p) combine through
//      X21 = -X22 (L21 X11), two batched products whose tiles all run at once;
//   3. Gt = G + diag(kappa / u) Z X, where column n of the product has the K range [n, d).
// All on the FP64 tensor pipe with a fixed k order.  X is lower triangular; the upper half of every diagonal 64 x 64
// block is written as zeros, and no reader touches a block above those.
// L's block sits in the lower triangle of sm (sm[i][k], k <= i), its inverse transposed above it (X[i][j] at
// sm[j][i + 1], i >= j): one 33 KB array.  Thread j forms column j of the inverse by forward substitution.
__global__ void __launch_bounds__(kTN) mvt_chol_diaginv_kernel(const double* __restrict__ vp, int d, double* __restrict__ X) {
  __shared__ double sm[kTN][kTN + 1];
  const int r0 = blockIdx.x * kTN, n = min(kTN, d - r0);
  const int j = threadIdx.x;
  for (int i = 0; i < n; ++i)
    if (j <= i) {
      const double v = vp[d + tri(r0 + i) + r0 + j];
      sm[i][j] = i == j ? exp(v) : v;
    }
  __syncthreads();
  if (j < n) {
    double* x = sm[j] + 1;                   // x[i] = X[i][j]
    x[j] = 1.0 / sm[j][j];
    for (int i = j + 1; i < n; ++i) {
      double a = 0.0;
      for (int k = j; k < i; ++k) a += sm[i][k] * x[k];
      x[i] = -a / sm[i][i];
    }
    for (int i = 0; i < n; ++i) X[(size_t)(r0 + i) * d + r0 + j] = j <= i ? x[i] : 0.0;
  }
}

// One doubling level at half-size h (a multiple of 64), one CTA per 64 x 64 output tile of every pair:
//   kSecond = false:  T21 = L21 X11,  tile (i0, j0) with K range [j0, r0 + h)        (X11 lower triangular)
//   kSecond = true:   X21 = -X22 T21, tile (i0, j0) with K range [r0 + h, i0 + 64)   (X22 lower triangular)
// 8 warps of 16 x 32 fragments, register-prefetched slabs as in the cotangent kernel.
template <bool kSecond>
__global__ void __launch_bounds__(256) mvt_chol_invlevel_kernel(const double* __restrict__ vp, int d, int h,
                                                                double* __restrict__ X, double* __restrict__ T) {
  __shared__ double sa[kSlab][kPadN], sb[kSlab][kPadN];
  const int tpb = h / kTN;
  const int64_t per = (int64_t)tpb * tpb;
  const int pair = (int)(blockIdx.x / per), tix = (int)(blockIdx.x % per);
  const int r0 = 2 * h * pair, r2 = r0 + h;
  const int i0 = r2 + (tix / tpb) * kTN, j0 = r0 + (tix % tpb) * kTN;
  if (i0 >= d) return;                       // past the end of a short last block: the whole CTA leaves
  const int kb = kSecond ? r2 : j0, ke = kSecond ? min(i0 + kTN, d) : r2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wm = warp >> 1, wn = warp & 1;
  const int gq = lane >> 2, t = lane & 3;
  double acc[2][4][2];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;

  // A[i][k] (L21 from the packed triangle, or X22) is read along k, B[k][j] (X11 or T21) along j
  double ra[kSlab * kTN / 256], rb[kSlab * kTN / 256];
  auto load = [&](int k0) {
#pragma unroll
    for (int p = 0; p < kSlab * kTN / 256; ++p) {
      const int i = i0 + p * 8 + warp, k = k0 + lane;
      double v = 0.0;
      if (i < d && k < d) v = kSecond ? X[(size_t)i * d + k] : vp[d + tri(i) + k];     // k < r2 <= i: strictly lower
      ra[p] = v;
      const int kr = k0 + p * 4 + (threadIdx.x >> 6), j = j0 + (threadIdx.x & 63);
      rb[p] = kr < d ? (kSecond ? T : X)[(size_t)kr * d + j] : 0.0;
    }
  };
  load(kb);
  for (int k0 = kb; k0 < ke; k0 += kSlab) {
    __syncthreads();
#pragma unroll
    for (int p = 0; p < kSlab * kTN / 256; ++p) {
      sa[lane][p * 8 + warp] = ra[p];
      sb[p * 4 + (threadIdx.x >> 6)][threadIdx.x & 63] = rb[p];
    }
    __syncthreads();
    if (k0 + kSlab < ke) load(k0 + kSlab);
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
  double* out = kSecond ? X : T;
#pragma unroll
  for (int a = 0; a < 2; ++a) {
    const int i = i0 + wm * 16 + a * 8 + gq;
    if (i >= d) continue;
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int j = j0 + wn * 32 + b * 8 + 2 * t + u;
        out[(size_t)i * d + j] = kSecond ? -acc[a][b][u] : acc[a][b][u];
      }
  }
}

// Gt[s][n] = G[s][n] + kappa_s / u_s sum_{k >= n} Z[s][k] X[k][n]  (G NULL: 0, inv_u NULL: u = 1, as the DIS score uses).  Column block c has the K range [64 c, d), so CTA
// (p, r) takes column blocks p and nb - 1 - p of row tile r to even out the work, as the triangular transform does.
__global__ void __launch_bounds__(256) mvt_chol_solve_kernel(const double* __restrict__ z, const double* __restrict__ X,
                                                             const double* __restrict__ G, const double* __restrict__ inv_u,
                                                             const double* __restrict__ zu2, double df, int S, int d,
                                                             double* __restrict__ Gt) {
  __shared__ double sa[kSlab][kPadM], sb[kSlab][kPadN];
  const int nb = (d + kTN - 1) / kTN;
  const unsigned npairs = (unsigned)(nb + 1) / 2;
  const int pair = (int)(blockIdx.x % npairs);
  const int m0 = (int)(blockIdx.x / npairs) * kTM;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wm = warp >> 2, wn = warp & 3;
  const int gq = lane >> 2, t = lane & 3;
  const int cb0 = pair, cb1 = nb - 1 - pair;
  const int ns0 = (d - cb0 * kTN + kSlab - 1) / kSlab;
  const int total = ns0 + (cb1 == cb0 ? 0 : (d - cb1 * kTN + kSlab - 1) / kSlab);

  double ra[kSlab * kTM / 256], rb[kSlab * kTN / 256];
  auto load = [&](int n0, int k0) {
#pragma unroll
    for (int p = 0; p < kSlab * kTM / 256; ++p) {
      const int s = m0 + p * 8 + warp, k = k0 + lane;
      ra[p] = (s < S && k < d) ? z[(size_t)s * d + k] : 0.0;
    }
#pragma unroll
    for (int p = 0; p < kSlab * kTN / 256; ++p) {
      const int k = k0 + p * 4 + (threadIdx.x >> 6), n = n0 + (threadIdx.x & 63);
      rb[p] = (k < d && n < d) ? X[(size_t)k * d + n] : 0.0;
    }
  };
  double acc[2][2][2];
  load(cb0 * kTN, cb0 * kTN);
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
#pragma unroll
    for (int p = 0; p < kSlab * kTM / 256; ++p) sa[lane][p * 8 + warp] = ra[p];
#pragma unroll
    for (int p = 0; p < kSlab * kTN / 256; ++p) sb[p * 4 + (threadIdx.x >> 6)][threadIdx.x & 63] = rb[p];
    __syncthreads();
    if (it + 1 < total) {
      const bool second1 = it + 1 >= ns0;
      const int c1 = second1 ? cb1 : cb0;
      load(c1 * kTN, c1 * kTN + (second1 ? it + 1 - ns0 : it + 1) * kSlab);
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
    if (sl + 1 == nsl) {
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        const int s = m0 + wm * 16 + a * 8 + gq;
        if (s >= S) continue;
        const double kappa = (df + d) / (df + zu2[s]), kiu = inv_u ? kappa * inv_u[s] : kappa;
#pragma unroll
        for (int b = 0; b < 2; ++b)
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int n = n0 + wn * 16 + b * 8 + 2 * t + u;
            if (n < d) Gt[(size_t)s * d + n] = G ? G[(size_t)s * d + n] + kiu * acc[a][b][u] : kiu * acc[a][b][u];
          }
      }
    }
  }
}

struct CholObjLayout {
  size_t off_sv, off_scal, off_hl, total;
  size_t off_X, off_T, off_Gt, total_path;     // path-derivative ExclusiveKL only
};
static void chol_obj_layout(int S, int d, CholObjLayout& l) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  l.off_sv = take(sizeof(double) * S);
  l.off_scal = take(sizeof(double) * 4);
  l.off_hl = take(sizeof(double));
  l.total = off;
  l.off_X = take(sizeof(double) * (size_t)d * d);
  l.off_T = take(sizeof(double) * (size_t)d * d);
  l.off_Gt = take(sizeof(double) * (size_t)S * d);
  l.total_path = off;
}

// X = L^-1 (dense, lower triangular; see above): the diagonal blocks, then the doubling levels; T is d x d scratch
static int chol_inverse(const double* vp, int d, double* X, double* T, cudaStream_t stream) {
  const int nb = (d + kTN - 1) / kTN;
  mvt_chol_diaginv_kernel<<<nb, kTN, 0, stream>>>(vp, d, X);
  VB_CHECK_LAUNCH();
  for (int h = kTN; h < d; h *= 2) {
    const int64_t ctas = ceil_div(d - h, 2 * h) * (int64_t)(h / kTN) * (h / kTN);
    mvt_chol_invlevel_kernel<false><<<(unsigned)ctas, 256, 0, stream>>>(vp, d, h, X, T);
    VB_CHECK_LAUNCH();
    mvt_chol_invlevel_kernel<true><<<(unsigned)ctas, 256, 0, stream>>>(vp, d, h, X, T);
    VB_CHECK_LAUNCH();
    if (h > INT32_MAX / 2) break;
  }
  return VB_OK;
}

// Gt = G + diag(kappa) Zhat L^-1 (see above); X and T are d x d scratch
static int chol_path_gradient(const double* vp, const double* z, const double* inv_u, const double* zu2, const double* G,
                              int S, int d, double df, double* X, double* T, double* Gt, cudaStream_t stream) {
  const int nb = (d + kTN - 1) / kTN;
  int rc = chol_inverse(vp, d, X, T, stream);
  if (rc) return rc;
  const int64_t ctas = (nb + 1) / 2 * ceil_div(S, kTM);
  mvt_chol_solve_kernel<<<(unsigned)ctas, 256, 0, stream>>>(z, X, G, inv_u, zu2, df, S, d, Gt);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

// ---- DISInclusiveKL score: value = -sum_r c_r log q(x_r), gradient at the fixed rows x_r = x[idx[r]] ----------------
// With y_r = L^-1 (x_r - mu), delta_r = |y_r|^2, kappa_r = (df + d) / (df + delta_r) and v_r = L^-T y_r (rows of
// V = Y L^-1):
//     log q_r  = const - sum_i F_ii - (df + d)/2 log1p(delta_r / df)
//     gbar_mu  = -sum_r c_r kappa_r v_r
//     Fbar_ij  = -sum_r c_r kappa_r v_ri y_rj  (j < i),   Fbar_ii = -L_ii sum_r c_r kappa_r v_ri y_ri + sum_r c_r
// i.e. the cotangent above with G -> diag(kappa) V, Z -> Y, u = 1, sv = c, c = -1 and diag_add = sum_r c_r.  Pipeline:
// L^-1 (chol_inverse), Y (triangular transform, x - mu formed on load), delta and c (one warp per row), the value
// (one block, fixed order), diag(kappa) V (the solve kernel), gbar_mu (mvt_gmu) and Fbar (cotangent kernel).

// delta[r] = |Y_r|^2,  cr[r] = scale * w[r]   (one warp per row, grid-stride)
__global__ void __launch_bounds__(256) mvt_score_rows_kernel(const double* __restrict__ Y, const double* __restrict__ w,
                                                             double scale, int n, int d, double* __restrict__ delta,
                                                             double* __restrict__ cr) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; r < n; r += nwarps) {
    double a = 0.0;
    for (int j = lane; j < d; j += 32) {
      const double v = Y[r * d + j];
      a += v * v;
    }
    a = warp_sum(a);
    if (lane == 0) {
      delta[r] = a;
      cr[r] = scale * (w ? w[r] : 1.0);
    }
  }
}

// scal = {value, sum_r c_r}, value[0] = scal[0]   (single block, fixed summation order)
__global__ void __launch_bounds__(1024) mvt_score_value_kernel(const double* __restrict__ delta, const double* __restrict__ cr,
                                                               int n, int d, double df, double logq_const,
                                                               const double* __restrict__ hl, double* __restrict__ scal,
                                                               double* __restrict__ value) {
  __shared__ double red[32];
  const double c0 = logq_const - hl[0];
  double a = 0.0, b = 0.0;
  for (int r = threadIdx.x; r < n; r += blockDim.x) {
    a += cr[r] * (c0 - 0.5 * (df + d) * log1p(delta[r] / df));
    b += cr[r];
  }
  a = block_sum(a, red);
  b = block_sum(b, red);
  if (threadIdx.x == 0) {
    scal[0] = value[0] = -a;
    scal[1] = b;
  }
}

struct ScoreLayout {
  size_t off_X, off_T, off_Y, off_KV, off_delta, off_cr, off_scal, off_hl, total;
};
static void score_layout(int64_t n, int d, ScoreLayout& l) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  l.off_X = take(sizeof(double) * (size_t)d * d);
  l.off_T = take(sizeof(double) * (size_t)d * d);
  l.off_Y = take(sizeof(double) * (size_t)n * d);
  l.off_KV = take(sizeof(double) * (size_t)n * d);
  l.off_delta = take(sizeof(double) * (size_t)n);
  l.off_cr = take(sizeof(double) * (size_t)n);
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
  mvt_chol_trmm_kernel<false><<<(unsigned)ctas, 256, 0, stream>>>(var_param, z, nullptr, nullptr, inv_u, S, d, theta);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

/* workspace: S + 5 doubles (256-byte aligned pieces) */
extern "C" size_t vb_mvt_chol_objective_workspace_bytes(int S, int d) {
  if (S <= 0 || d <= 0) return 0;
  CholObjLayout l;
  chol_obj_layout(S, d, l);
  return l.total;
}

/* workspace of vb_mvt_chol_objective_f64 with VB_OBJ_EXCLUSIVE_KL_PATH: the above plus 2 d^2 + S d doubles */
extern "C" size_t vb_mvt_chol_path_workspace_bytes(int S, int d) {
  if (S <= 0 || d <= 0) return 0;
  CholObjLayout l;
  chol_obj_layout(S, d, l);
  return l.total_path;
}

/* value[1] and grad[d + d(d+1)/2] of ExclusiveKL (entropy or path-derivative form) / AlphaDivergence
 * (objectives.py:154-164, :443-460) in the Cholesky reparameterisation, from the model's f[S] and G[S,d] at theta and
 * inv_u / zu2 of vb_mvt_chol_transform_f64. */
extern "C" int vb_mvt_chol_objective_f64(const double* var_param, const double* z, const double* inv_u, const double* zu2,
                                         const double* f, const double* G, int S, int d, double df, int objective, double alpha,
                                         double* value, double* grad, void* workspace, size_t workspace_bytes,
                                         cudaStream_t stream) {
  if (!var_param || !z || !inv_u || !zu2 || !f || !G || S <= 0 || d <= 0 || !value || !grad)
    return set_error(VB_ERR_INVALID_ARG, "mvt_chol_objective: bad arguments");
  if (objective != VB_OBJ_EXCLUSIVE_KL && objective != VB_OBJ_EXCLUSIVE_KL_PATH && objective != VB_OBJ_ALPHA)
    return set_error(VB_ERR_UNSUPPORTED, "mvt_chol_objective: unknown objective");
  const bool path = objective == VB_OBJ_EXCLUSIVE_KL_PATH;
  CholObjLayout l;
  chol_obj_layout(S, d, l);
  if (!workspace || workspace_bytes < (path ? l.total_path : l.total))
    return set_error(VB_ERR_WORKSPACE, "mvt_chol_objective: workspace too small");
  const int nb = (d + kTN - 1) / kTN;
  if (path && ((nb + 1) / 2 * ceil_div(S, kTM) > INT32_MAX || (int64_t)nb * nb > INT32_MAX))
    return set_error(VB_ERR_UNSUPPORTED, "mvt_chol_objective: more than 2^31 - 1 tiles");
  char* ws = static_cast<char*>(workspace);
  double* sv = reinterpret_cast<double*>(ws + l.off_sv);
  double* scal = reinterpret_cast<double*>(ws + l.off_scal);
  double* hl = reinterpret_cast<double*>(ws + l.off_hl);
  int rc = mvt_logdiag(var_param, d, hl, stream);
  if (rc) return rc;
  const double* Gc = G;
  if (path) {
    double* Gt = reinterpret_cast<double*>(ws + l.off_Gt);
    rc = chol_path_gradient(var_param, z, inv_u, zu2, G, S, d, df, reinterpret_cast<double*>(ws + l.off_X),
                            reinterpret_cast<double*>(ws + l.off_T), Gt, stream);
    if (rc) return rc;
    Gc = Gt;
  }
  rc = mvt_weights_gmu(f, Gc, zu2, hl, S, d, df, objective, alpha, sv, scal, value, grad, stream);
  if (rc) return rc;
  const double c = objective == VB_OBJ_ALPHA ? alpha / S : -1.0 / S;
  mvt_chol_cotangent_kernel<<<(unsigned)(nb * (nb + 1) / 2), 256, 0, stream>>>(var_param, z, inv_u, Gc, sv, scal, c, S, d, grad);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

/* workspace of vb_mvt_score_f64: 2 d^2 + 2 n d + 2 n + 5 doubles (256-byte aligned pieces) */
extern "C" size_t vb_mvt_score_workspace_bytes(int64_t n, int d) {
  if (n <= 0 || d <= 0) return 0;
  ScoreLayout l;
  score_layout(n, d, l);
  return l.total;
}

/* value[1] = -sum_r c_r log q(x_{i_r}; var_param) and grad[d + d(d+1)/2] (DISInclusiveKL's score, see above),
 * c_r = scale * w[r] (w NULL: 1), i_r = idx[r] (idx NULL: r).  Both reparameterisations: the score depends on
 * var_param and the fixed rows only. */
extern "C" int vb_mvt_score_f64(const double* var_param, const double* x, const int64_t* idx, const double* w, double scale,
                                int64_t n, int d, double df, double* value, double* grad, void* workspace,
                                size_t workspace_bytes, cudaStream_t stream) {
  if (!var_param || !x || n <= 0 || d <= 0 || !value || !grad) return set_error(VB_ERR_INVALID_ARG, "mvt_score: bad arguments");
  if (!(df > 2.0)) return set_error(VB_ERR_INVALID_ARG, "df must be greater than 2");
  ScoreLayout l;
  score_layout(n, d, l);
  if (!workspace || workspace_bytes < l.total) return set_error(VB_ERR_WORKSPACE, "mvt_score: workspace too small");
  const int64_t nb = ceil_div(d, kTN);
  const int64_t row_ctas = (nb + 1) / 2 * ceil_div(n, kTM);
  if (n > INT32_MAX || row_ctas > INT32_MAX || nb * nb > INT32_MAX)
    return set_error(VB_ERR_UNSUPPORTED, "mvt_score: more than 2^31 - 1 tiles");
  char* ws = static_cast<char*>(workspace);
  double* X = reinterpret_cast<double*>(ws + l.off_X);
  double* Y = reinterpret_cast<double*>(ws + l.off_Y);
  double* KV = reinterpret_cast<double*>(ws + l.off_KV);
  double* delta = reinterpret_cast<double*>(ws + l.off_delta);
  double* cr = reinterpret_cast<double*>(ws + l.off_cr);
  double* scal = reinterpret_cast<double*>(ws + l.off_scal);
  double* hl = reinterpret_cast<double*>(ws + l.off_hl);
  const int nr = (int)n;
  int rc = chol_inverse(var_param, d, X, reinterpret_cast<double*>(ws + l.off_T), stream);
  if (rc) return rc;
  mvt_chol_trmm_kernel<true><<<(unsigned)row_ctas, 256, 0, stream>>>(var_param, x, reinterpret_cast<const long long*>(idx), X,
                                                                       nullptr, nr, d, Y);
  VB_CHECK_LAUNCH();
  const int64_t blocks = ceil_div(n, 256 / 32), cap = 64LL * sm_count();
  mvt_score_rows_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, stream>>>(Y, w, scale, nr, d, delta, cr);
  VB_CHECK_LAUNCH();
  rc = mvt_logdiag(var_param, d, hl, stream);
  if (rc) return rc;
  mvt_score_value_kernel<<<1, 1024, 0, stream>>>(delta, cr, nr, d, df, mvt_const(df, d), hl, scal, value);
  VB_CHECK_LAUNCH();
  mvt_chol_solve_kernel<<<(unsigned)row_ctas, 256, 0, stream>>>(Y, X, nullptr, nullptr, delta, df, nr, d, KV);
  VB_CHECK_LAUNCH();
  rc = mvt_gmu(KV, cr, nr, d, -1.0, grad, stream);
  if (rc) return rc;
  mvt_chol_cotangent_kernel<<<(unsigned)(nb * (nb + 1) / 2), 256, 0, stream>>>(var_param, Y, nullptr, KV, cr, scal, -1.0, nr, d,
                                                                                grad);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
