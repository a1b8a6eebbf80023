// Device helpers shared by the one-column PSIS pipeline (psis.cu) and the batched one-CTA-per-column kernel
// (psis_batch.cu): order-preserving keys, the single-CTA radix select, the generalised Pareto weights, log-products
// and inverse, the control block and the 16-slot result layout.
#pragma once
#include <float.h>

#include "common.cuh"

namespace vb {

constexpr int kSelThreads = 1024;
constexpr int kDigitBits = 11;
constexpr int kBins = 1 << kDigitBits;

// result[] slots (doubles, device memory)
enum { R_KHAT = 0, R_SIGMA, R_N2, R_CUTOFF, R_LSE, R_MAX, R_STATUS, R_SUMV, R_SUMEXP2V, R_M, R_NCAND, R_SMOOTHED,
       R_COUNT = 16 };

struct PsisScalars {           // device-resident control block
  unsigned long long maxkey;   // order-preserving key of the global max
  unsigned long long t0key;    // candidate threshold (key)
  unsigned long long cutkey;   // key of the (M+1)-th largest raw value
  unsigned int ncand;          // candidates found by pass A
  unsigned int ntail;          // n2
  unsigned int status;         // 0 ok, 1 fast path failed (rerun exact), 2 internal overflow
  unsigned int strict;         // exact mode: candidates are strictly above t0
  double t0;                   // threshold as a double
  double maxv, cutoff, expcut; // max, shifted cutoff, exp(shifted cutoff)
  double body_below;           // sum exp(x - t0) over x below the threshold
  double body_cand;            // sum exp(x - max) over candidates that are not tail
  double tail_sum;             // sum exp(v) over (smoothed) tail values
  double k, sigma, lse, bhat;
  double sumv, sumexp2v;       // moments of v = out + lse over the tail
  double vscale;               // bins per unit of (v - cutoff)
  int smoothed;
  int M;
  int shift;                   // digit position of the candidate histogram
  unsigned int bstar;          // boundary bin of the candidate histogram
  unsigned int need;           // rank (from the top) of the cutoff inside the boundary bin
  unsigned int members;        // population of the boundary bin
  unsigned int gcount;         // keys gathered from it
  unsigned long long prefix;   // exact-mode radix state
  unsigned long long kth;
  double hist_hi;              // upper end of the candidate histogram's linear bins (sample maximum / merged maximum)
  double tbase;                // base of pass A's exponentials: t0, or the next double above it in exact mode
  double below_sv, below_se2;  // one-pass moments: sum (x - tbase), sum exp(2 (x - tbase)) over x below the threshold
  double cand_sv, cand_se2;    // one-pass moments: sum v, sum exp(2 v) over candidates that are not tail
  long long n_local;           // draws this control block's pass A covered
  int onepass;                 // moments-only mode: no pass B, the bound moments come out of pass A
  unsigned int gpd_done;       // blocks of the GPD grid kernel that have finished
  unsigned int gather_done, count_done, values_done, select_done;      // same for the kernels whose last block runs the next (single-CTA) step
};

__device__ __forceinline__ unsigned long long dkey(double x) {
  unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double dkey_inv(unsigned long long k) {
  unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

// ---------------------------------------------------------------------------------------------
// single-CTA radix select over keys in GLOBAL/SHARED memory: key of the K-th largest (K >= 1)
// ---------------------------------------------------------------------------------------------
// all threads of a 1024-thread CTA: find the bin (scanning from the TOP bin down) that holds rank K;
// sh[0] = bin, sh[1] = rank inside that bin.  nb <= 2048.  Ends with a __syncthreads().
static __device__ void cta_find_bin(const unsigned int* hist, unsigned int nb, unsigned long long K, unsigned long long* sh,
                             unsigned int* wtot /*[32]*/) {
  const unsigned int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int b0 = (int)nb - 1 - 2 * (int)t, b1 = b0 - 1;          // this thread's two bins, higher first
  const unsigned int c0 = b0 >= 0 ? hist[b0] : 0u, c1 = b1 >= 0 ? hist[b1] : 0u;
  unsigned int incl = c0 + c1;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= (unsigned)o) incl += v;
  }
  if (lane == 31) wtot[w] = incl;
  __syncthreads();
  if (w == 0) {
    const unsigned int v = wtot[lane];
    unsigned int in = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int u = __shfl_up_sync(0xffffffffu, in, o);
      if (lane >= (unsigned)o) in += u;
    }
    wtot[lane] = in - v;                                          // exclusive warp offsets
  }
  __syncthreads();
  const unsigned long long ex = (unsigned long long)wtot[w] + incl - (c0 + c1);   // entries in higher bins
  if (ex < K && K <= ex + c0) {
    sh[0] = (unsigned long long)b0;
    sh[1] = K - ex;
  } else if (ex + c0 < K && K <= ex + c0 + c1) {
    sh[0] = (unsigned long long)b1;
    sh[1] = K - ex - c0;
  }
  __syncthreads();
}

static __device__ unsigned long long cta_select_kth_largest(const unsigned long long* keys, unsigned int cnt, unsigned long long K,
                                                     unsigned int* hist /*[kBins]*/, unsigned long long* sh /*[2]*/,
                                                     unsigned int* wtot /*[32]*/) {
  unsigned long long prefix = 0, mask = 0;
  int shift = 64;
  while (shift > 0) {
    const int bits = shift >= kDigitBits ? kDigitBits : shift;
    shift -= bits;
    const unsigned int nb = 1u << bits;
    for (unsigned int b = threadIdx.x; b < nb; b += blockDim.x) hist[b] = 0;
    __syncthreads();
    for (unsigned int i0 = 0; i0 < cnt; i0 += blockDim.x) {
      const unsigned int i = i0 + threadIdx.x;
      const unsigned long long key = i < cnt ? keys[i] : 0ull;
      const bool ok = i < cnt && ((key & mask) == prefix);
      const unsigned int dig = ok ? (unsigned int)((key >> shift) & (nb - 1)) : 0xffffffffu;
      const unsigned int peers = __match_any_sync(0xffffffffu, dig);
      if (ok && (threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&hist[dig], __popc(peers));
    }
    __syncthreads();
    cta_find_bin(hist, nb, K, sh, wtot);
    prefix |= sh[0] << shift;
    mask |= (unsigned long long)(nb - 1) << shift;
    K = sh[1];
    __syncthreads();
  }
  return prefix;
}

// profile likelihood weights -> posterior mean of b (:288-312)
__device__ __forceinline__ void gpd_weights(PsisScalars* sc, const double* bs, const double* part, int nparts, double* Ls,
                                            int N, int m, double* red) {
  for (int j = threadIdx.x; j < m; j += blockDim.x) {
    double ksum = 0.0;
    for (int u0 = 0; u0 < nparts; u0 += 8) {                   // loads of a batch are independent: one L2 latency per 8
      double pv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) pv[u] = u0 + u < nparts ? __ldcg(part + j * nparts + u0 + u) : 0.0;     // written by other blocks
#pragma unroll
      for (int u = 0; u < 8; ++u) ksum += pv[u];
    }
    const double kj = ksum / (double)N;
    double L = __ldcg(bs + j) / kj;
    L = log(-L);
    L -= kj;
    L -= 1.0;
    Ls[j] = L * (double)N;
  }
  __syncthreads();
  // w_j = 1 / sum_i exp(L_i - L_j)  (:295-298)  ==  exp(L_j - Lmax) / sum_i exp(L_i - Lmax): O(m) instead of
  // O(m^2), identical up to rounding, and the reference's "benign overflow -> weight 0" becomes an underflow
  double lmax = -INFINITY;
  for (int j = threadIdx.x; j < m; j += blockDim.x) lmax = fmax(lmax, Ls[j]);
  lmax = block_max(lmax, red);
  double den = 0.0;
  for (int j = threadIdx.x; j < m; j += blockDim.x) den += exp(Ls[j] - lmax);
  den = block_sum(den, red);
  double wsum = 0.0, bsum = 0.0;
  for (int j = threadIdx.x; j < m; j += blockDim.x) {
    const double w = exp(Ls[j] - lmax) / den;
    if (w >= 10.0 * DBL_EPSILON) {
      wsum += w;
      bsum += __ldcg(bs + j) * w;
    }
  }
  wsum = block_sum(wsum, red);
  bsum = block_sum(bsum, red);
  if (threadIdx.x == 0) sc->bhat = bsum / wsum;
}

// sum_i log1p(nb * x_i) as the log of running products: 8 terms per log instead of one log1p per term (the fit
// evaluates 6.1 M of them at n2 = 30 000, _psis.py:283-286).  1 + nb x_i is formed with one rounding (fma); every
// term lies in (~1e-4, ~1e5) for the Zhang-Stephens grid (b < 1/x_max), so a product of 8 stays far inside the
// double range, and the relative rounding error of a product (8 x 1.1e-16) is an ABSOLUTE error of the same size
// in its log -- the same order as the rounding of the eight separate log1p results it replaces.
struct LogProd {
  double prod = 1.0, acc = 0.0;
  int cnt = 0;
  __device__ __forceinline__ void add(double nb, double x) {
    prod *= fma(nb, x, 1.0);
    if (++cnt == 8) {
      acc += log(prod);
      prod = 1.0;
      cnt = 0;
    }
  }
  __device__ __forceinline__ double result() const { return cnt ? acc + log(prod) : acc; }
};

__device__ __forceinline__ double gpinv1(double p, double k, double sigma) {
  // _psis.py:335-377 for 0 < p < 1
  double q;
  if (fabs(k) < DBL_EPSILON)
    q = -log1p(-p);
  else
    q = expm1(-k * log1p(-p)) / k;
  return q * sigma;
}

}  // namespace vb
