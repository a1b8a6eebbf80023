// Pareto-smoothed importance sampling on the device (reference viabel/_psis.py:113-209,
// gpdfitnew :212-332, gpinv :335-377, sumlogs :380-396) plus the 2-divergence moments that
// diagnostics.divergence_bound (:148-186) needs, without ever sorting the n log-weights.
//
// The reference does a full argsort of n values to find one order statistic.  Here:
//   pass A (1 read of lw)   : global max, compaction of "candidates" >= t0 (a threshold estimated
//                             from a strided sample so that #candidates is a few times the tail
//                             length M), and sum exp(x - t0) over everything below t0;
//   small kernels           : histogram select of the (M+1)-th largest among the candidates (the
//                             cutoff is an order-statistic VALUE, so this is exact), bucketed
//                             counting rank of the <= M tail entries, Zhang-Stephens GPD fit,
//                             smoothed quantiles, log-sum-exp;
//   pass B (1 read, 1 write): out = x - max - lse, tail entries replaced by their smoothed values,
//                             and sum(out), sum exp(2 out) for the CUBO / ELBO bounds.
// Algorithmic traffic: 24 bytes per draw.  If the sample-based threshold fails (candidate buffer
// overflow or fewer than M+1 candidates) status=1 is reported and the caller re-runs in exact mode,
// which finds the cutoff with full radix passes.  Ordinary inputs do reach it: on draws sorted either
// way the 16-CTA select's group maxima (16 consecutive sample entries) are correlated, so n = 1e6
// sorted overflows (118 733 candidates, capacity 95 321) and n = 3e4 sorted descending finds too few;
// so do inputs periodic with the sample stride (tests/_psis_ref.py predicts each case).
#include <mutex>

#include "psis_internal.cuh"

namespace vb {

constexpr int kSampleMax = 16384;        // 1024 threads x 16 keys held in registers
constexpr int kGather = 8192;            // boundary-bucket members selected in shared memory
constexpr int kVBins = 8192;             // linear bins on the shifted tail values
constexpr int kGpdJ = 8;                 // quadrature points per CTA of the GPD grid kernel
constexpr int kGpdChunk = 2048;          // tail values per CTA of the GPD grid kernel (256 threads x 8, held in registers)

// exp(x) for x <= 0: x = (1024 k + j) ln2/1024 + r, exp = 2^k * 2^(j/1024) * e^r, |r| <= ln2/2048, so a degree-3
// polynomial is enough (r^4/24 < 5.5e-16 relative, far inside the 1e-10 budget of the log-sum-exp).  The two
// streaming passes are bound by the FP64 pipe, not by HBM, at ~14 double-precision operations per draw with the
// textbook 32-entry table: the larger table removes three of them.
constexpr int kExpTab = 256;
__device__ double g_exp2_tab[kExpTab];
// polynomial / reduction constants live in the constant bank so every DFMA takes them as a direct
// operand (no per-call re-materialisation of 64-bit immediates)
__constant__ double c_expk[8] = {369.3299304675746322841407 /* 256/ln2 */, 6755399441055744.0 /* 1.5 * 2^52 */,
                                 -2.7076061733168899081640625e-03 /* -ln2_hi/256 */,
                                 -7.453964567463233203203125e-13 /* -ln2_lo/256 */,
                                 4.1666666666666664e-02, 1.6666666666666666e-01, 0.5,
                                 -2.7076061740622863e-03 /* -ln2/256, correctly rounded (exp_stream) */};
// `tab` is the 32-bit shared-memory address of a per-CTA copy of the table (per-lane indices would serialise on the
// constant cache; shared memory serves them at full rate)
__device__ __forceinline__ uint32_t load_exp_table(double* tab) {
  for (int i = threadIdx.x; i < kExpTab; i += blockDim.x) tab[i] = g_exp2_tab[i];
  __syncthreads();
  return (uint32_t)__cvta_generic_to_shared(tab);
}
__device__ __forceinline__ double exp_nonpos(double x, uint32_t tab) {
  const double t = fma(x, c_expk[0], c_expk[1]);
  const int n = __double2loint(t);
  const double kf = t - c_expk[1];
  double r = fma(kf, c_expk[2], x);
  r = fma(kf, c_expk[3], r);
  double p = c_expk[4];
  p = fma(p, r, c_expk[5]);
  p = fma(p, r, c_expk[6]);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  const int k = n >> 8;
  double tj;
  asm("ld.shared.f64 %0, [%1];" : "=d"(tj) : "r"(tab + ((uint32_t)(n & (kExpTab - 1)) << 3)));
  const double v = p * tj;                           // in [1, 2.001)
  const double res = __hiloint2double(__double2hiint(v) + (k << 20), __double2loint(v));
  // x <= -707.75 (incl. -inf): the result would be subnormal (< 2^-1021).  Every sum these terms enter is
  // >= 1 (it contains exp(0) for the maximum), so they are below half an ulp of it: flushed to zero.
  return ((unsigned int)__double2hiint(x) >= 0xC0861E00u) ? 0.0 : res;
}

// exp(x), x <= 0, for the moments-only pass (sum exp(2 v) of the CUBO term, 16 B/draw mode), 7 double-precision
// operations instead of 9: one-step range reduction with the correctly rounded ln2/256 (the error of the constant
// times |k| <= 745 * 256 is below 3e-14 in r) and a degree-3 polynomial (r^4/24 <= 1.4e-13, |r| <= ln2/512); the sum
// enters a result whose budget is 1e-10.  Measured: diagnostics-only PSIS 0.44 -> 0.40 ms at n = 1e8.  Pass B keeps the
// 9-operation form: it already runs at the HBM peak, and with fewer registers its occupancy rises from 4 to 6 CTAs
// per SM, which made the read+write stream SLOWER (245 -> 300 us).
__device__ __forceinline__ double exp_stream(double x, uint32_t tab) {
  const double t = fma(x, c_expk[0], c_expk[1]);
  const int n = __double2loint(t);
  const double kf = t - c_expk[1];
  const double r = fma(kf, c_expk[7], x);
  double p = c_expk[5];
  p = fma(p, r, c_expk[6]);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  const int k = n >> 8;
  double tj;
  asm("ld.shared.f64 %0, [%1];" : "=d"(tj) : "r"(tab + ((uint32_t)(n & (kExpTab - 1)) << 3)));
  const double v = p * tj;                           // in [1, 2.001)
  const double res = __hiloint2double(__double2hiint(v) + (k << 20), __double2loint(v));
  return ((unsigned int)__double2hiint(x) >= 0xC0861E00u) ? 0.0 : res;
}

// ---------------------------------------------------------------------------------------------
__global__ void psis_init_kernel(PsisScalars* sc, int M, unsigned int* hist, unsigned int* vhist, int onepass,
                                 long long n_local) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    sc->hist_hi = -INFINITY; sc->tbase = -INFINITY; sc->below_sv = 0; sc->below_se2 = 0; sc->cand_sv = 0; sc->cand_se2 = 0;
    sc->onepass = onepass; sc->n_local = n_local;
    sc->maxkey = 0; sc->t0key = 0; sc->cutkey = 0; sc->ncand = 0; sc->ntail = 0; sc->status = 0; sc->strict = 0;
    sc->gpd_done = 0; sc->gather_done = 0; sc->count_done = 0; sc->values_done = 0; sc->select_done = 0;
    sc->t0 = -INFINITY; sc->maxv = 0; sc->cutoff = 0; sc->expcut = 0; sc->body_below = 0; sc->body_cand = 0;
    sc->tail_sum = 0; sc->k = INFINITY; sc->sigma = 0; sc->lse = 0; sc->bhat = 0; sc->sumv = 0; sc->sumexp2v = 0;
    sc->vscale = 0; sc->smoothed = 0; sc->M = M; sc->shift = 0; sc->bstar = 0; sc->need = 0; sc->members = 0; sc->gcount = 0; sc->prefix = 0; sc->kth = 0;
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kBins; i += gridDim.x * blockDim.x) hist[i] = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * kVBins; i += gridDim.x * blockDim.x) vhist[i] = 0;
}

// register-resident radix select: K-th largest of NK keys per thread (invalid keys are 0 = below everything)
// stop_shift > 0: stop once the digits above bit `stop_shift` are fixed and return the LOWER BOUND of that bucket
// (remaining bits zero) -- a valid, marginally looser threshold for half the passes.
template <int NK>
__device__ unsigned long long reg_select_kth_largest(const unsigned long long (&kreg)[NK], unsigned long long K,
                                                     unsigned int* hist, unsigned long long* sh, unsigned int* wtot,
                                                     int stop_shift = 0) {
  unsigned long long prefix = 0, mask = 0;
  int shift = 64;
  while (shift > stop_shift) {
    const int bits = shift >= kDigitBits ? kDigitBits : shift;
    shift -= bits;
    const unsigned int nb = 1u << bits;
    for (unsigned int b = threadIdx.x; b < nb; b += blockDim.x) hist[b] = 0;
    __syncthreads();
#pragma unroll
    for (int u = 0; u < NK; ++u) {
      const bool ok = kreg[u] != 0ull && ((kreg[u] & mask) == prefix);
      const unsigned int dig = ok ? (unsigned int)((kreg[u] >> shift) & (nb - 1)) : 0xffffffffu;
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

// maximum of the sample (all threads of one CTA call this): the upper end of the candidate histogram's bins
__device__ __forceinline__ void sample_max(PsisScalars* sc, unsigned long long km, unsigned long long* smaxk /*[32]*/) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long v = __shfl_xor_sync(0xffffffffu, km, o);
    km = v > km ? v : km;
  }
  if ((threadIdx.x & 31) == 0) smaxk[threadIdx.x >> 5] = km;
  __syncthreads();
  if (threadIdx.x < 32) {
    km = threadIdx.x < (blockDim.x >> 5) ? smaxk[threadIdx.x] : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long v = __shfl_xor_sync(0xffffffffu, km, o);
      km = v > km ? v : km;
    }
    if (threadIdx.x == 0) sc->hist_hi = dkey_inv(km);
  }
}

// candidate threshold t0 from a strided sample of m <= 16384 keys (16 per thread, in registers).
// R <= 256: the R-th largest of the 1024 per-thread maxima, which is <= the R-th largest of the whole
// sample (a subset's order statistic), i.e. errs on the side of a few more candidates and needs one key
// per thread; larger R (only for n of a few 1e5 or less): the exact R-th largest of the sample.
__global__ void __launch_bounds__(kSelThreads) psis_sample_select_kernel(const double* __restrict__ lw, int64_t stride,
                                                                          int m, unsigned int R, PsisScalars* sc,
                                                                          unsigned long long* gmax) {
  __shared__ unsigned int hist[kBins];
  __shared__ unsigned long long sh[2];
  __shared__ unsigned int wtot[32];
  __shared__ unsigned int last;
  __shared__ unsigned long long smaxk[32];
  if (R >= (unsigned)m) {
    if (blockIdx.x == 0 && threadIdx.x == 0) { sc->t0key = 0; sc->t0 = -INFINITY; }
    return;
  }
  unsigned long long key;
  if (gridDim.x > 1) {
    // R <= 256 and a full sample: 16 CTAs load one key per thread (a single SM cannot keep 16384 scattered DRAM
    // reads in flight), groups of 16 threads keep their maximum, the last CTA to finish selects among the 1024 maxima
    const unsigned int g = blockIdx.x * kSelThreads + threadIdx.x;
    unsigned long long k = dkey(lw[(int64_t)g * stride]);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      const unsigned long long v = __shfl_xor_sync(0xffffffffu, k, o);
      k = v > k ? v : k;
    }
    if ((threadIdx.x & 15) == 0) gmax[g >> 4] = k;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(&sc->select_done, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    unsigned long long kmax[1] = {__ldcg(gmax + threadIdx.x)};
    // sign + exponent + 21 mantissa bits (3 digit passes) decide the threshold: relative resolution 5e-7
    key = reg_select_kth_largest<1>(kmax, R, hist, sh, wtot, 31);
    sample_max(sc, kmax[0], smaxk);
  } else {
    unsigned long long kreg[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int i = u * kSelThreads + threadIdx.x;
      kreg[u] = i < m ? dkey(lw[(int64_t)i * stride]) : 0ull;          // key 0 = below everything
    }
    unsigned long long kmax[1] = {0ull};
#pragma unroll
    for (int u = 0; u < 16; ++u) kmax[0] = kreg[u] > kmax[0] ? kreg[u] : kmax[0];
    sample_max(sc, kmax[0], smaxk);
    if (R <= 256) {
      key = reg_select_kth_largest<1>(kmax, R, hist, sh, wtot);
    } else {
      key = reg_select_kth_largest<16>(kreg, R, hist, sh, wtot);
    }
  }
  if (threadIdx.x == 0) { sc->t0key = key; sc->t0 = dkey_inv(key); }
}

// pass A: candidate compaction (everything >= the threshold; the global max is among them) and
// sum exp(x - t0) over everything below the threshold.  Candidates are staged per warp in shared
// memory and flushed with ONE global atomic per CTA (same-address atomics with a return value
// serialise at ~2 ns each in L2: one per candidate-bearing warp iteration cost more than the HBM pass).
constexpr int kStage = 64;      // per-warp staging entries (>= 2 * 32: every push of up to 32 candidates checks for room)

// linear value bins of the candidate histogram over [t0, hist_hi] (monotone in x)
__device__ __forceinline__ unsigned int cbin(double x, double lo, double scale) {
  const double f = (x - lo) * scale;
  const int b = (int)f;
  return b < 0 ? 0u : (b >= kBins ? (unsigned)(kBins - 1) : (unsigned)b);
}
__device__ __forceinline__ double cand_scale(const PsisScalars* sc, double& lo) {
  const double hi = sc->hist_hi;               // values above it (the sample maximum) share the top bin
  lo = sc->t0;
  return (lo > -INFINITY && hi > lo) ? (double)kBins / (hi - lo) : 0.0;      // 0: everything in bin 0
}

// exp(d) for -707.75 < d <= ~0 WITHOUT the underflow select (the caller screens the sign/exponent word of d):
// the 7-operation form of exp_stream.  Its relative error (<= 1.4e-13 truncation, <= 1e-14 from the one-step
// reduction for every term that matters) enters a sum whose budget is 1e-10.
__device__ __forceinline__ double exp_core(double d, uint32_t tab) {
  const double t = fma(d, c_expk[0], c_expk[1]);
  const int n = __double2loint(t);
  const double kf = t - c_expk[1];
  const double r = fma(kf, c_expk[7], d);
  double p = c_expk[5];
  p = fma(p, r, c_expk[6]);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  double tj;
  asm("ld.shared.f64 %0, [%1];" : "=d"(tj) : "r"(tab + ((uint32_t)(n & (kExpTab - 1)) << 3)));
  const double v = p * tj;                           // in [1, 2.001)
  return __hiloint2double(__double2hiint(v) + ((n & ~(kExpTab - 1)) << 12), __double2loint(v));
}

// pass A, lean form.  A plain loop over predicated quads profiled at 150 instructions per 4 draws of which only 52
// are double-precision arithmetic -- the rest were the two selects per draw (candidate, underflow), the -inf
// initialisation of predicated loads, register copies of the software pipeline and 64-bit index arithmetic.  Here
// the main loop covers only iterations in which every thread has a full quad (no predication), is unrolled by two so
// that the prefetched quads alternate between two register sets, and accumulates all four exponentials
// unconditionally; ONE integer test per draw on the high word of d = x - tbase (d >= 0: candidate, d < -707.75:
// underflow; as a signed integer both are "hi >= 0xC0861E00") and one warp vote send the rare iterations that hold a
// candidate or an underflowing term to a slow path that zeroes those terms and stages the candidates.
// kMom: also sum d and exp(2 d) (moments-only PSIS: the CUBO / ELBO sums without a second pass over the draws).
constexpr int kHiSpecial = (int)0xC0861E00;
template <bool kMom>
__global__ void __launch_bounds__(256, 4) psis_pass_a_lean_kernel(const double* __restrict__ lw, int64_t n, int64_t idx_off,
                                                               PsisScalars* sc, double* __restrict__ cand_x,
                                                               int64_t* __restrict__ cand_i, unsigned int cap,
                                                               double* __restrict__ blk_sum, double* __restrict__ blk_mom,
                                                               unsigned int* __restrict__ ghist) {
  __shared__ double red[32];
  __shared__ unsigned long long redk[32];
  __shared__ double etab_s[kExpTab];
  __shared__ double sx[8][kStage];
  __shared__ long long si[8][kStage];
  __shared__ unsigned int wcnt[8], cta_base;
  const uint32_t etab = load_exp_table(etab_s);
  const double t0 = sc->t0;
  const bool all = !(t0 > -INFINITY);       // threshold -inf: everything is a candidate
  // candidates are x >= tb; in exact mode (candidates STRICTLY above t0) tb is the next double above t0
  const double tb = all ? -INFINITY : (sc->strict ? nextafter(t0, INFINITY) : t0);
  if (blockIdx.x == 0 && threadIdx.x == 0) sc->tbase = tb;
  // the candidate histogram (linear bins over [t0, sample maximum]) is filled here, from the slow path: one global
  // atomic per candidate spread over 2048 bins and the whole pass (the separate histogram kernel cost 7 us)
  __shared__ double hpar[2];                // read on the slow path only: keeps two doubles out of the hot loop's registers
  if (threadIdx.x == 0) {
    double lo;
    hpar[1] = cand_scale(sc, lo);
    hpar[0] = lo;
  }
  __syncthreads();
  double mx = -INFINITY, acc0 = 0.0, acc1 = 0.0, s1 = 0.0, s3 = 0.0;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  unsigned int staged = 0;                  // warp-uniform number of staged candidates
  auto flush_warp = [&]() {
    unsigned int base = 0;
    if (lane == 0) base = atomicAdd(&sc->ncand, staged);
    base = __shfl_sync(0xffffffffu, base, 0);
    for (unsigned int i = lane; i < staged; i += 32)
      if (base + i < cap) {
        cand_x[base + i] = sx[w][i];
        cand_i[base + i] = si[w][i];
      }
    __syncwarp();
    staged = 0;
  };
  auto push = [&](double x, int64_t i, bool is_cand) {
    const unsigned int ball = __ballot_sync(0xffffffffu, is_cand);
    if (ball) {
      if (staged + 32 > kStage) flush_warp();
      if (is_cand) {
        mx = fmax(mx, x);
        const double hscale = hpar[1];
        if (hscale > 0.0) atomicAdd(&ghist[cbin(x, hpar[0], hscale)], 1u);
        else if (lane == __ffs(ball) - 1) atomicAdd(&ghist[0], (unsigned int)__popc(ball));    // degenerate range: one bin
        const unsigned int slot = staged + __popc(ball & ((1u << lane) - 1));
        sx[w][slot] = x;
        si[w][slot] = i + idx_off;      // global draw index (idx_off = this rank's first draw)
      }
      staged += __popc(ball);
    }
  };
  // one quad of draws; q = index of the quad
  auto quad = [&](const double2 a, const double2 b, const int64_t q) {
    double d0 = a.x - tb, d1 = a.y - tb, d2 = b.x - tb, d3 = b.y - tb;
    double e0 = exp_core(d0, etab), e1 = exp_core(d1, etab), e2 = exp_core(d2, etab), e3 = exp_core(d3, etab);
    const int h0 = __double2hiint(d0), h1 = __double2hiint(d1), h2 = __double2hiint(d2), h3 = __double2hiint(d3);
    const bool special = (h0 >= kHiSpecial) | (h1 >= kHiSpecial) | (h2 >= kHiSpecial) | (h3 >= kHiSpecial);
    if (__any_sync(0xffffffffu, special)) {
      const bool c0 = a.x >= tb, c1 = a.y >= tb, c2 = b.x >= tb, c3 = b.y >= tb;
      // (a NaN draw is no candidate and must poison the sums, as it poisons the reference's max and logsumexp)
      e0 = h0 >= kHiSpecial ? (d0 != d0 ? d0 : 0.0) : e0;
      e1 = h1 >= kHiSpecial ? (d1 != d1 ? d1 : 0.0) : e1;
      e2 = h2 >= kHiSpecial ? (d2 != d2 ? d2 : 0.0) : e2;
      e3 = h3 >= kHiSpecial ? (d3 != d3 ? d3 : 0.0) : e3;
      if (kMom) {
        d0 = c0 ? 0.0 : d0;
        d1 = c1 ? 0.0 : d1;
        d2 = c2 ? 0.0 : d2;
        d3 = c3 ? 0.0 : d3;
      }
      push(a.x, 4 * q, c0);
      push(a.y, 4 * q + 1, c1);
      push(b.x, 4 * q + 2, c2);
      push(b.y, 4 * q + 3, c3);
    }
    acc0 += e0 + e2;
    acc1 += e1 + e3;
    if (kMom) {
      s1 += (d0 + d1) + (d2 + d3);
      s3 = fma(e0, e0, s3);
      s3 = fma(e1, e1, s3);
      s3 = fma(e2, e2, s3);
      s3 = fma(e3, e3, s3);
    }
  };
  int64_t done = 0;
  if ((reinterpret_cast<uintptr_t>(lw) & 31) == 0 && !all) {
    const int64_t full = (n / 4) / nthreads;          // iterations in which EVERY thread owns a quad
    if (full > 0) {
      const double2* p = reinterpret_cast<const double2*>(lw) + 2 * tid;
      const int64_t st = 2 * nthreads;
      double2 a = __ldcs(p), b = __ldcs(p + 1);
      int64_t q = tid, it = 0;
      for (; it + 2 <= full; it += 2) {
        const double2 c = __ldcs(p + st), d = __ldcs(p + st + 1);
        quad(a, b, q);
        p += 2 * st;
        if (it + 2 < full) {
          a = __ldcs(p);
          b = __ldcs(p + 1);
        }
        quad(c, d, q + nthreads);
        q += 2 * nthreads;
      }
      if (it < full) quad(a, b, q);
    }
    done = full * nthreads * 4;
  }
  {   // the rest (< 4 draws per thread), or the whole array when unaligned / when everything is a candidate
    const int64_t rest = n - done;
    const int64_t iters = (rest + nthreads - 1) / nthreads;
    for (int64_t it = 0; it < iters; ++it) {
      const int64_t i = done + it * nthreads + tid;
      const bool v = i < n;
      const double x = v ? lw[i] : -INFINITY;
      const bool c = v && (all || x >= tb);
      if (v && !c) {
        const double d = x - tb;
        const double e = d != d ? d : ((unsigned int)__double2hiint(d) >= 0xC0861E00u ? 0.0 : exp_core(d, etab));
        acc0 += e;
        if (kMom) {
          s1 += d;
          s3 = fma(e, e, s3);
        }
      }
      push(x, i, c);
    }
  }
  // block reductions and the single per-CTA flush of the staged candidates
  double acc = warp_sum(acc0 + acc1);
  if (kMom) {
    s1 = warp_sum(s1);
    s3 = warp_sum(s3);
  }
  unsigned long long mk = dkey(mx);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long t = __shfl_xor_sync(0xffffffffu, mk, o);
    mk = t > mk ? t : mk;
  }
  if (lane == 0) {
    red[w] = acc;
    redk[w] = mk;
    wcnt[w] = staged;
    if (kMom) {
      red[8 + w] = s1;
      red[16 + w] = s3;
    }
  }
  __syncthreads();
  if (w == 0) {
    double a = lane < 8 ? red[lane] : 0.0;
    unsigned long long k = lane < 8 ? redk[lane] : 0ull;
    unsigned int c = lane < 8 ? wcnt[lane] : 0u;
    a = warp_sum(a);
    double m1 = 0.0, m3 = 0.0;
    if (kMom) {
      m1 = warp_sum(lane < 8 ? red[8 + lane] : 0.0);
      m3 = warp_sum(lane < 8 ? red[16 + lane] : 0.0);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      unsigned long long t = __shfl_xor_sync(0xffffffffu, k, o);
      k = t > k ? t : k;
      c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    if (lane == 0) {
      blk_sum[blockIdx.x] = a;
      if (kMom) {
        blk_mom[2 * blockIdx.x] = m1;
        blk_mom[2 * blockIdx.x + 1] = m3;
      }
      if (k > dkey(-INFINITY)) atomicMax(&sc->maxkey, k);
      cta_base = c ? atomicAdd(&sc->ncand, c) : 0u;
    }
  }
  __syncthreads();
  unsigned int base = cta_base;
  for (int u = 0; u < w; ++u) base += wcnt[u];
  for (unsigned int i = lane; i < staged; i += 32)
    if (base + i < cap) {
      cand_x[base + i] = sx[w][i];
      cand_i[base + i] = si[w][i];
    }
}

// ---- cutoff among the candidates: one histogram pass on LINEAR value bins over [t0, max] (monotone in x,
// so every entry of a higher bin is larger than every entry of a lower one), then an exact key select
// of the boundary bin in shared memory
__global__ void __launch_bounds__(256) psis_cand_hist_kernel(PsisScalars* sc, const double* __restrict__ cand_x,
                                                             unsigned int cap, unsigned int* __restrict__ ghist) {
  PDL_SYNC();
  __shared__ unsigned int hist[kBins];
  const unsigned int C = sc->ncand;
  if (sc->strict || C > cap || C < (unsigned)(sc->M + 1)) return;
  double lo;
  const double scale = cand_scale(sc, lo);
  for (unsigned int b = threadIdx.x; b < kBins; b += blockDim.x) hist[b] = 0;
  __syncthreads();
  for (unsigned int i0 = blockIdx.x * blockDim.x; i0 < C; i0 += gridDim.x * blockDim.x) {
    const unsigned int i = i0 + threadIdx.x;
    const bool ok = i < C;
    const unsigned int dig = ok ? (scale > 0.0 ? cbin(cand_x[i], lo, scale) : 0u) : 0xffffffffu;
    const unsigned int peers = __match_any_sync(0xffffffffu, dig);
    if (ok && (threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&hist[dig], __popc(peers));
  }
  __syncthreads();
  for (unsigned int b = threadIdx.x; b < kBins; b += blockDim.x)
    if (hist[b]) atomicAdd(&ghist[b], hist[b]);
}

// every CTA locates the boundary bin from the global histogram, then gathers the keys of its slice of
// that bin into a small global buffer
// cutoff = (M+1)-th largest candidate (one CTA of kSelThreads threads; run by the last block of the gather kernel)
__device__ __forceinline__ void cutoff_block(PsisScalars* sc, const double* cand_x, unsigned int cap,
                                             const unsigned long long* gbuf, const double* blk_sum,
                                             const double* blk_mom, int nblk,
                                             unsigned int* hist, unsigned long long* sh, unsigned int* wtot, double* red) {
  const unsigned int C = sc->ncand;
  const int M = sc->M;
  double s = 0.0;
  for (int b = threadIdx.x; b < nblk; b += blockDim.x) s += blk_sum[b];
  s = block_sum(s, red);
  double m1 = 0.0, m3 = 0.0;
  if (sc->onepass) {            // one-pass moments: pass A's per-CTA sums of d and exp(2 d)
    for (int b = threadIdx.x; b < nblk; b += blockDim.x) {
      m1 += blk_mom[2 * b];
      m3 += blk_mom[2 * b + 1];
    }
    m1 = block_sum(m1, red);
    m3 = block_sum(m3, red);
  }
  // exact mode collects only values strictly above t0: when there are none the maximum is t0 itself
  const unsigned long long maxkey = (sc->strict && sc->maxkey < sc->t0key) ? sc->t0key : sc->maxkey;
  const double maxv = dkey_inv(maxkey);
  unsigned long long cutkey;
  if (sc->strict) {
    cutkey = sc->t0key;                        // exact mode: t0 IS the (M+1)-th largest value
    if (C > cap) { if (threadIdx.x == 0) sc->status = 2; return; }
  } else {
    if (C > cap || C < (unsigned)(M + 1)) {
      if (threadIdx.x == 0) sc->status = 1;
      return;
    }
    const unsigned int bstar = sc->bstar, members = sc->members;
    const unsigned long long need = sc->need;
    if (members <= kSelThreads) {
      // the usual case (a boundary bin of 1 / 2048 of the candidate range holds a few hundred keys): one key per
      // thread, rank by counting against the others in shared memory -- one step instead of six radix passes
      unsigned long long* sk = reinterpret_cast<unsigned long long*>(hist);      // kBins x 4 bytes = 1024 keys
      const unsigned long long key = threadIdx.x < members ? gbuf[threadIdx.x] : 0ull;
      sk[threadIdx.x] = key;
      __syncthreads();
      unsigned int gt = 0, ge = 0;
      for (unsigned int j = 0; j < members; ++j) {
        const unsigned long long o = sk[j];
        gt += o > key;
        ge += o >= key;
      }
      if (threadIdx.x < members && gt < need && need <= ge) sh[0] = key;         // ties write the same key
      __syncthreads();
      cutkey = sh[0];
    } else if (members <= kGather) {
      // exact 64-bit radix select over the gathered boundary bin (<= 8192 keys, L2 resident)
      cutkey = cta_select_kth_largest(gbuf, members, need, hist, sh, wtot);
    } else {
      // huge boundary bin (massive ties): radix passes over the candidates in global memory
      double lo;
      const double scale = cand_scale(sc, lo);
      unsigned long long pfx = 0, msk = 0, K = need;
      int sft = 64;
      while (sft > 0) {
        const int bits = sft >= kDigitBits ? kDigitBits : sft;
        sft -= bits;
        const unsigned int nb = 1u << bits;
        for (unsigned int b = threadIdx.x; b < nb; b += blockDim.x) hist[b] = 0;
        __syncthreads();
        for (unsigned int i0 = 0; i0 < C; i0 += blockDim.x) {
          const unsigned int i = i0 + threadIdx.x;
          const double x = i < C ? cand_x[i] : 0.0;
          const unsigned long long key = dkey(x);
          const bool ok = i < C && (scale > 0.0 ? cbin(x, lo, scale) : 0u) == bstar && ((key & msk) == pfx);
          const unsigned int dig = ok ? (unsigned int)((key >> sft) & (nb - 1)) : 0xffffffffu;
          const unsigned int peers = __match_any_sync(0xffffffffu, dig);
          if (ok && (threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&hist[dig], __popc(peers));
        }
        __syncthreads();
        cta_find_bin(hist, nb, K, sh, wtot);
        pfx |= sh[0] << sft;
        msk |= (unsigned long long)(nb - 1) << sft;
        K = sh[1];
        __syncthreads();
      }
      cutkey = pfx;
    }
  }
  if (threadIdx.x == 0) {
    const double cutraw = dkey_inv(cutkey);
    const double cutoff = fmax(cutraw - maxv, log(DBL_MIN));       // _psis.py:159, :170-173
    sc->cutkey = cutkey;
    sc->maxkey = maxkey;
    sc->maxv = maxv;
    sc->cutoff = cutoff;
    sc->expcut = exp(cutoff);
    sc->body_below = s;
    sc->below_sv = m1;
    sc->below_se2 = m3;
    sc->vscale = (cutoff < 0.0) ? (double)kVBins / (-cutoff) : 0.0;
  }
}

__global__ void __launch_bounds__(kSelThreads) psis_cand_gather_kernel(PsisScalars* sc, const double* __restrict__ cand_x,
                                                                        unsigned int cap, const unsigned int* __restrict__ ghist,
                                                                        unsigned long long* gbuf, const double* blk_sum,
                                                                        const double* blk_mom, int nblk) {
  PDL_SYNC();
  __shared__ __align__(8) unsigned int hist[kBins];      // cutoff_block reuses it as 1024 64-bit keys
  static_assert(kBins * sizeof(unsigned int) >= kSelThreads * sizeof(unsigned long long), "key buffer");
  __shared__ unsigned long long sh[2];
  __shared__ unsigned int wtot[32];
  __shared__ double red[32];
  __shared__ unsigned int last;
  const unsigned int C = sc->ncand;
  if (!(sc->strict || C > cap || C < (unsigned)(sc->M + 1))) {
    for (unsigned int b = threadIdx.x; b < kBins; b += blockDim.x) hist[b] = ghist[b];
    __syncthreads();
    cta_find_bin(hist, kBins, (unsigned long long)(sc->M + 1), sh, wtot);
    const unsigned int bstar = (unsigned int)sh[0];
    const unsigned int members = hist[bstar];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      sc->bstar = bstar;
      sc->need = (unsigned int)sh[1];
      sc->members = members;
    }
    if (members <= kGather) {                  // else the cutoff step falls back to radix passes
      double lo;
      const double scale = cand_scale(sc, lo);
      for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < C; i += gridDim.x * blockDim.x) {
        const double x = cand_x[i];
        if ((scale > 0.0 ? cbin(x, lo, scale) : 0u) == bstar) {
          const unsigned int slot = atomicAdd(&sc->gcount, 1u);
          if (slot < kGather) gbuf[slot] = dkey(x);
        }
      }
    }
  }
  // the last block to finish selects the cutoff among the gathered keys (saves a single-CTA launch)
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&sc->gather_done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) {
    __threadfence();
    cutoff_block(sc, cand_x, cap, gbuf, blk_sum, blk_mom, nblk, hist, sh, wtot, red);
  }
}

__device__ __forceinline__ int vbin(double v, double cutoff, double vscale) {
  const double f = (v - cutoff) * vscale;
  int b = (int)f;
  return b < 0 ? 0 : (b >= kVBins ? kVBins - 1 : b);
}

// tail membership (shifted value > cutoff), per-bin tail counts, LSE contribution of the other candidates
// exclusive scan of the tail bins (ascending value) -> bin offsets; n2
__device__ __forceinline__ void tail_scan_block(PsisScalars* sc, const unsigned int* vhist, unsigned int* voff,
                                                unsigned int* wsum) {
  constexpr int per = kVBins / kSelThreads;       // 8 bins per thread
  unsigned int loc[per], tot = 0;
#pragma unroll
  for (int u = 0; u < per; ++u) {
    loc[u] = vhist[threadIdx.x * per + u];
    tot += loc[u];
  }
  unsigned int incl = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
    if ((threadIdx.x & 31) >= o) incl += t;
  }
  if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
  __syncthreads();
  if (threadIdx.x < 32) {
    unsigned int v = wsum[threadIdx.x], in = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int t = __shfl_up_sync(0xffffffffu, in, o);
      if (threadIdx.x >= o) in += t;
    }
    wsum[threadIdx.x] = in - v;
    if (threadIdx.x == 31) sc->ntail = in;
  }
  __syncthreads();
  unsigned int base = wsum[threadIdx.x >> 5] + incl - tot;
#pragma unroll
  for (int u = 0; u < per; ++u) {
    voff[threadIdx.x * per + u] = base;
    base += loc[u];
  }
}

__global__ void __launch_bounds__(kSelThreads) psis_tail_count_kernel(PsisScalars* sc, const double* __restrict__ cand_x,
                                                                       unsigned int* vhist, unsigned int* __restrict__ voff) {
  PDL_SYNC();
  __shared__ double red[32];
  __shared__ unsigned int wsum[32];
  __shared__ unsigned int last;
  if (sc->status) return;
  const unsigned int C = sc->ncand;
  const double maxv = sc->maxv, cutoff = sc->cutoff, vscale = sc->vscale;
  const bool onepass = sc->onepass != 0;
  double acc = 0.0, accv = 0.0, acc2 = 0.0;
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < C; i += gridDim.x * blockDim.x) {
    const double v = cand_x[i] - maxv;
    if (v > cutoff) {
      atomicAdd(&vhist[vbin(v, cutoff, vscale)], 1u);
    } else {
      const double e = exp(v);
      acc += e;
      accv += v;
      acc2 = fma(e, e, acc2);
    }
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0 && acc != 0.0) atomicAdd(&sc->body_cand, acc);
  if (onepass) {
    accv = block_sum(accv, red);
    acc2 = block_sum(acc2, red);
    if (threadIdx.x == 0) {
      atomicAdd(&sc->cand_sv, accv);
      atomicAdd(&sc->cand_se2, acc2);
    }
  }
  // the last block to finish scans the bin counts into offsets (saves a single-CTA launch)
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&sc->count_done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) {
    __threadfence();
    tail_scan_block(sc, vhist, voff, wsum);
  }
}

// bin-ordered placement of the tail entries (order inside a bin is arbitrary here)
__global__ void __launch_bounds__(256) psis_tail_place_kernel(PsisScalars* sc, const double* __restrict__ cand_x,
                                                              const int64_t* __restrict__ cand_i,
                                                              const unsigned int* __restrict__ voff,
                                                              unsigned int* __restrict__ vcur, double* __restrict__ tmp_v,
                                                              int64_t* __restrict__ tmp_i, int* __restrict__ tmp_b,
                                                              unsigned int tail_cap, int raw) {
  PDL_SYNC();
  if (sc->status) return;
  const unsigned int C = sc->ncand;
  const double maxv = sc->maxv, cutoff = sc->cutoff, vscale = sc->vscale;
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < C; i += gridDim.x * blockDim.x) {
    const double v = cand_x[i] - maxv;
    if (v > cutoff) {
      const int b = vbin(v, cutoff, vscale);
      const unsigned int pos = voff[b] + atomicAdd(&vcur[b], 1u);
      if (pos < tail_cap) {
        tmp_v[pos] = raw ? cand_x[i] : v;          // raw: a sharded rank ships unshifted values
        tmp_i[pos] = cand_i[i];
        tmp_b[pos] = b;
      }
    }
  }
}

// exact rank by counting inside the (small) bin; output arrays are in ascending (value, index) order
__global__ void __launch_bounds__(256) psis_tail_rank_kernel(PsisScalars* sc, const double* __restrict__ tmp_v,
                                                             const int64_t* __restrict__ tmp_i, const int* __restrict__ tmp_b,
                                                             const unsigned int* __restrict__ voff,
                                                             const unsigned int* __restrict__ vhist,
                                                             double* __restrict__ tail_v, int64_t* __restrict__ tail_i,
                                                             double* __restrict__ sorted_x) {
  PDL_SYNC();
  if (sc->status) return;
  const unsigned int n2 = sc->ntail;
  const double expcut = sc->expcut;
  for (unsigned int p = blockIdx.x * blockDim.x + threadIdx.x; p < n2; p += gridDim.x * blockDim.x) {
    const double v = tmp_v[p];
    const int64_t ii = tmp_i[p];
    const int b = tmp_b[p];
    const unsigned int lo = voff[b], cnt = vhist[b];
    unsigned int r = lo;
    for (unsigned int q = lo; q < lo + cnt; ++q) {
      const double vq = tmp_v[q];
      r += (vq < v) || (vq == v && tmp_i[q] < ii);
    }
    tail_v[r] = v;
    tail_i[r] = ii;
    sorted_x[r] = exp(v) - expcut;                  // _psis.py:185-186
  }
}

// optional: tail indices in ascending index order with their value ranks (O(n2^2), API nicety / tests)
__global__ void __launch_bounds__(256) psis_tail_index_order_kernel(PsisScalars* sc, const int64_t* __restrict__ tail_i,
                                                                    int64_t* __restrict__ idx_sorted, int* __restrict__ order_rank) {
  PDL_SYNC();
  __shared__ int64_t si[256];
  if (sc->status) return;
  const unsigned int n2 = sc->ntail;
  for (unsigned int i0 = blockIdx.x * blockDim.x; i0 < n2; i0 += gridDim.x * blockDim.x) {
    const unsigned int i = i0 + threadIdx.x;
    const bool valid = i < n2;
    const int64_t ii = valid ? tail_i[i] : 0;
    int p = 0;
    for (unsigned int j0 = 0; j0 < n2; j0 += 256) {
      __syncthreads();
      const unsigned int j = j0 + threadIdx.x;
      si[threadIdx.x] = j < n2 ? tail_i[j] : INT64_MAX;
      __syncthreads();
      const int lim = (n2 - j0) < 256 ? (int)(n2 - j0) : 256;
      for (int q = 0; q < lim; ++q) p += si[q] < ii;
    }
    if (valid) {
      idx_sorted[p] = ii;
      order_rank[p] = (int)i;
    }
  }
}

// ---- generalised Pareto fit (_psis.py:212-332), split so that no stage is a long serial loop --------
// partial sums of log1p(-b_j x_i).  grid = (ceil(mgrid / kGpdJ), ceil(tail_cap / kGpdChunk)): a CTA keeps 2048 tail
// values in registers (8 per thread, one batch of independent loads) and evaluates kGpdJ quadrature points on them, so
// the tail array crosses L2 -> SM m / 8 times instead of m times (the first version -- one CTA per (j, eighth of the
// tail) -- moved 49 MB through L2 and ran in two waves: 25 us; this form 6 MB, one wave).  Each thread's 8 terms of
// one quadrature point become ONE log of their product (see LogProd).
__global__ void __launch_bounds__(256) psis_gpd_grid_kernel(PsisScalars* sc, const double* __restrict__ sorted_x,
                                                            double* __restrict__ bs, double* __restrict__ part,
                                                            double* __restrict__ Ls) {
  PDL_SYNC();
  __shared__ double red[32];
  __shared__ double wpart[8][kGpdJ];
  __shared__ unsigned int last;
  if (sc->status) return;
  const int N = (int)sc->ntail;
  if (N <= 4) return;
  const int m = 30 + (int)sqrt((double)N);
  const int nparts = gridDim.y;
  const int j0 = blockIdx.x * kGpdJ;
  if (j0 >= m) return;                                   // (mgrid is sized for the largest possible tail)
  const int jgroups = (m + kGpdJ - 1) / kGpdJ;
  const double xq = sorted_x[(int)(N / 4.0 + 0.5) - 1];
  const double xmax = sorted_x[N - 1];
  const int base = blockIdx.y * kGpdChunk;
  double x[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int i = base + u * 256 + (int)threadIdx.x;
    x[u] = i < N ? sorted_x[i] : 0.0;                    // a term 1 + nb * 0 = 1 leaves the product alone
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __shared__ double nbs[kGpdJ];
  if (threadIdx.x < kGpdJ) {          // the grid point's sqrt and two divisions once per CTA, not once per thread
    const int j = j0 + (int)threadIdx.x;
    double b = 1.0 - sqrt((double)m / ((double)(j + 1) - 0.5));
    b /= 3.0 * xq;
    b += 1.0 / xmax;
    if (blockIdx.y == 0 && j < m) bs[j] = b;
    nbs[threadIdx.x] = j < m ? -b : 0.0;
  }
  __syncthreads();
#pragma unroll
  for (int jj = 0; jj < kGpdJ; ++jj) {
    const double nb = nbs[jj];
    double prod = fma(nb, x[0], 1.0);
#pragma unroll
    for (int u = 1; u < 8; ++u) prod *= fma(nb, x[u], 1.0);
    const double v = warp_sum(log(prod));
    if (lane == 0) wpart[w][jj] = v;
  }
  __syncthreads();
  if (threadIdx.x < kGpdJ && j0 + (int)threadIdx.x < m) {
    double a = 0.0;
#pragma unroll
    for (int u = 0; u < 8; ++u) a += wpart[u][threadIdx.x];
    part[(j0 + threadIdx.x) * nparts + blockIdx.y] = a;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&sc->gpd_done, 1u) == (unsigned)(jgroups * nparts) - 1u;
  __syncthreads();
  if (last) {              // every partial sum is visible: the last block turns them into the posterior mean of b
    __threadfence();
    gpd_weights(sc, bs, part, nparts, Ls, N, m, red);
  }
}

// partial sums of log1p(-bhat x_i)
__global__ void __launch_bounds__(256) psis_gpd_k_kernel(PsisScalars* sc, const double* __restrict__ sorted_x,
                                                         double* __restrict__ part) {
  PDL_SYNC();
  __shared__ double red[32];
  if (sc->status) return;
  const int N = (int)sc->ntail;
  double acc = 0.0;
  if (N > 4) {
    const double nb = -sc->bhat;
    LogProd lp;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) lp.add(nb, sorted_x[i]);
    acc = lp.result();
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = acc;
}

// log-sum-exp of everything and the result vector (first warp of the last block of the tail-values kernel)
__device__ __forceinline__ void lse_warp(PsisScalars* sc, const double* part3, int nparts, double* result) {
  if (sc->status) {
    if (threadIdx.x == 0) result[R_STATUS] = (double)sc->status;
    return;
  }
  double ts = 0.0, sv = 0.0, se = 0.0;
  for (int i = threadIdx.x; i < nparts; i += 32) {
    ts += part3[3 * i];
    sv += part3[3 * i + 1];
    se += part3[3 * i + 2];
  }
  ts = warp_sum(ts);
  sv = warp_sum(sv);
  se = warp_sum(se);
  if (threadIdx.x != 0) return;
  const double below = sc->body_below == 0.0 ? 0.0 : sc->body_below * exp(sc->tbase - sc->maxv)   /* NaN passes */;
  const double total = below + sc->body_cand + ts;
  if (sc->onepass) {
    // moments of v = x - max over ALL draws from pass A's sums (relative to tbase), the candidate list and the tail
    const double nbelow = (double)(sc->n_local - (long long)sc->ncand);
    const double shift = sc->tbase - sc->maxv;
    result[R_SUMV] = (nbelow > 0.0 ? sc->below_sv + nbelow * shift : 0.0) + sc->cand_sv + sv;
    result[R_SUMEXP2V] = (sc->below_se2 == 0.0 ? 0.0 : sc->below_se2 * exp(2.0 * shift)) + sc->cand_se2 + se;
  }
  sc->tail_sum = ts;
  sc->sumv = sv;
  sc->sumexp2v = se;
  sc->lse = log(total);
  // a NaN among the draws: the reference's max is NaN, every output is NaN, the tail {x > cutoff} is empty and
  // k-hat is therefore +inf (_psis.py:154-180)
  result[R_KHAT] = total != total ? INFINITY : sc->k;
  result[R_SIGMA] = sc->sigma;
  result[R_N2] = (double)sc->ntail;
  result[R_CUTOFF] = sc->cutoff;
  result[R_LSE] = sc->lse;
  result[R_MAX] = sc->maxv;
  result[R_STATUS] = 0.0;
  result[R_M] = (double)sc->M;
  result[R_NCAND] = (double)sc->ncand;
  result[R_SMOOTHED] = (double)sc->smoothed;
}

// k-hat, sigma (:313-324) and the smoothing decision (:188); then the per-rank tail values
__global__ void __launch_bounds__(256) psis_tail_values_kernel(PsisScalars* sc, const double* __restrict__ kpart, int nkpart,
                                                               const double* __restrict__ tail_v, double* __restrict__ tail_out,
                                                               double* part3, double* __restrict__ result) {
  PDL_SYNC();
  __shared__ double red[32];
  __shared__ unsigned int last;
  if (sc->status) {
    if (blockIdx.x == 0 && threadIdx.x == 0) result[R_STATUS] = (double)sc->status;
    return;
  }
  const int N = (int)sc->ntail;
  double k = INFINITY, sigma = 0.0;
  if (N > 4) {
    // same reduction tree in every CTA (a serial loop of dependent loads cost ~300 cycles per entry)
    double s = 0.0;
    for (int i = threadIdx.x & 31; i < nkpart; i += 32) s += kpart[i];
    s = warp_sum(s);
    k = s / (double)N;
    sigma = -k / sc->bhat;
    k = k * (double)N / ((double)N + 10.0) + 5.0 / ((double)N + 10.0);
  }
  const bool smooth = (k >= 1.0 / 3.0) && !isinf(k);
  const bool onepass = sc->onepass != 0;
  const double expcut = sc->expcut;
  double ts = 0.0, sv = 0.0, se = 0.0;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < N; r += gridDim.x * blockDim.x) {
    double v;
    if (smooth) {
      v = log(gpinv1(((double)r + 0.5) / (double)N, k, sigma) + expcut);      // :190-197
      v = v > 0.0 ? 0.0 : v;                                                   // :199
    } else {
      v = tail_v[r];
    }
    tail_out[r] = v;
    ts += exp(v);
    if (smooth || onepass) {          // moments of the tail (pass B covers everything it writes itself)
      sv += v;
      se += exp(2.0 * v);
    }
  }
  ts = block_sum(ts, red);
  sv = block_sum(sv, red);
  se = block_sum(se, red);
  if (threadIdx.x == 0) {
    part3[3 * blockIdx.x] = ts;
    part3[3 * blockIdx.x + 1] = sv;
    part3[3 * blockIdx.x + 2] = se;
    if (blockIdx.x == 0) {
      sc->k = k;
      sc->sigma = sigma;
      sc->smoothed = smooth ? 1 : 0;
    }
  }
  // the last block to finish folds the partial sums into the log-sum-exp (saves a one-warp launch)
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(&sc->values_done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last && threadIdx.x < 32) {
    __threadfence();
    lse_warp(sc, part3, gridDim.x, result);
  }
}

// pass B: out = (x - max) - lse for the body (tail entries are written by the scatter kernel when
// smoothing is on); moments of v = out + lse for the divergence bounds
__global__ void __launch_bounds__(256) psis_pass_b_kernel(const double* __restrict__ lw, double* __restrict__ out, int64_t n,
                                                          PsisScalars* sc, double* __restrict__ blk_mom) {
  PDL_SYNC();
  __shared__ double red[32];
  __shared__ double etab_s[kExpTab];
  const uint32_t etab = load_exp_table(etab_s);
  if (sc->status) return;
  const double maxv = sc->maxv, lse = sc->lse, cutoff = sc->cutoff;
  const bool smoothed = sc->smoothed != 0;
  double sv0 = 0.0, sv1 = 0.0, se0 = 0.0, se1 = 0.0;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const bool aligned = ((reinterpret_cast<uintptr_t>(lw) | reinterpret_cast<uintptr_t>(out)) & 31) == 0;
  if (aligned) {
    const int64_t n4 = n / 4;
    double2 na = make_double2(0.0, 0.0), nb = na;     // software pipeline: next iteration's loads in flight
    if (tid < n4) {
      na = __ldcs(reinterpret_cast<const double2*>(lw) + 2 * tid);
      nb = __ldcs(reinterpret_cast<const double2*>(lw) + 2 * tid + 1);
    }
    for (int64_t q = tid; q < n4; q += nthreads) {
      const double2 a = na, b = nb;
      const int64_t qn = q + nthreads;
      if (qn < n4) {
        na = __ldcs(reinterpret_cast<const double2*>(lw) + 2 * qn);
        nb = __ldcs(reinterpret_cast<const double2*>(lw) + 2 * qn + 1);
      }
      const double v0 = a.x - maxv, v1 = a.y - maxv, v2 = b.x - maxv, v3 = b.y - maxv;
      const bool t0 = smoothed && v0 > cutoff, t1 = smoothed && v1 > cutoff, t2 = smoothed && v2 > cutoff,
                 t3 = smoothed && v3 > cutoff;
      sv0 += (t0 ? 0.0 : v0) + (t2 ? 0.0 : v2);
      sv1 += (t1 ? 0.0 : v1) + (t3 ? 0.0 : v3);
      se0 += (t0 ? 0.0 : exp_nonpos(2.0 * v0, etab)) + (t2 ? 0.0 : exp_nonpos(2.0 * v2, etab));
      se1 += (t1 ? 0.0 : exp_nonpos(2.0 * v1, etab)) + (t3 ? 0.0 : exp_nonpos(2.0 * v3, etab));
      if (!(t0 | t1 | t2 | t3)) {
        __stcs(reinterpret_cast<double2*>(out) + 2 * q, make_double2(v0 - lse, v1 - lse));
        __stcs(reinterpret_cast<double2*>(out) + 2 * q + 1, make_double2(v2 - lse, v3 - lse));
      } else {
        if (!t0) out[4 * q] = v0 - lse;
        if (!t1) out[4 * q + 1] = v1 - lse;
        if (!t2) out[4 * q + 2] = v2 - lse;
        if (!t3) out[4 * q + 3] = v3 - lse;
      }
    }
    for (int64_t i = n4 * 4 + tid; i < n; i += nthreads) {
      const double v = lw[i] - maxv;
      if (!(smoothed && v > cutoff)) {
        sv0 += v;
        se0 += exp_nonpos(2.0 * v, etab);
        out[i] = v - lse;
      }
    }
  } else {
    for (int64_t i = tid; i < n; i += nthreads) {
      const double v = lw[i] - maxv;
      if (!(smoothed && v > cutoff)) {
        sv0 += v;
        se0 += exp_nonpos(2.0 * v, etab);
        out[i] = v - lse;
      }
    }
  }
  const double sv = block_sum(sv0 + sv1, red);
  const double se = block_sum(se0 + se1, red);
  if (threadIdx.x == 0) {
    blk_mom[2 * blockIdx.x] = sv;
    blk_mom[2 * blockIdx.x + 1] = se;
  }
}

// moments without writing an output array (k-hat / bounds only): 16 bytes per draw in total
__global__ void __launch_bounds__(256) psis_pass_b_moments_kernel(const double* __restrict__ lw, int64_t n, PsisScalars* sc,
                                                                  double* __restrict__ blk_mom) {
  PDL_SYNC();
  __shared__ double red[32];
  __shared__ double etab_s[kExpTab];
  const uint32_t etab = load_exp_table(etab_s);
  if (sc->status) return;
  const double maxv = sc->maxv, cutoff = sc->cutoff;
  const bool smoothed = sc->smoothed != 0;
  double sv = 0.0, se = 0.0;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t done = 0;
  if ((reinterpret_cast<uintptr_t>(lw) & 31) == 0) {
    // same streaming structure as pass B: 2 x LDG.128 per thread with the next iteration's loads in flight,
    // two independent accumulation chains
    const int64_t n4 = n / 4;
    double sv1 = 0.0, se1 = 0.0;
    double2 na = make_double2(0.0, 0.0), nb = na;
    if (tid < n4) {
      na = __ldcs(reinterpret_cast<const double2*>(lw) + 2 * tid);
      nb = __ldcs(reinterpret_cast<const double2*>(lw) + 2 * tid + 1);
    }
    for (int64_t q = tid; q < n4; q += nthreads) {
      const double2 a = na, b = nb;
      const int64_t qn = q + nthreads;
      if (qn < n4) {
        na = __ldcs(reinterpret_cast<const double2*>(lw) + 2 * qn);
        nb = __ldcs(reinterpret_cast<const double2*>(lw) + 2 * qn + 1);
      }
      const double v0 = a.x - maxv, v1 = a.y - maxv, v2 = b.x - maxv, v3 = b.y - maxv;
      const bool t0 = smoothed && v0 > cutoff, t1 = smoothed && v1 > cutoff, t2 = smoothed && v2 > cutoff,
                 t3 = smoothed && v3 > cutoff;
      sv += (t0 ? 0.0 : v0) + (t2 ? 0.0 : v2);
      sv1 += (t1 ? 0.0 : v1) + (t3 ? 0.0 : v3);
      se += (t0 ? 0.0 : exp_stream(2.0 * v0, etab)) + (t2 ? 0.0 : exp_stream(2.0 * v2, etab));
      se1 += (t1 ? 0.0 : exp_stream(2.0 * v1, etab)) + (t3 ? 0.0 : exp_stream(2.0 * v3, etab));
    }
    sv += sv1;
    se += se1;
    done = n4 * 4;
  }
  for (int64_t i = done + tid; i < n; i += nthreads) {
    const double v = lw[i] - maxv;
    if (!(smoothed && v > cutoff)) {
      sv += v;
      se += exp_stream(2.0 * v, etab);
    }
  }
  sv = block_sum(sv, red);
  se = block_sum(se, red);
  if (threadIdx.x == 0) {
    blk_mom[2 * blockIdx.x] = sv;
    blk_mom[2 * blockIdx.x + 1] = se;
  }
}

// smoothed tail values into place (_psis.py:190-199) and final moment reduction
__global__ void __launch_bounds__(256) psis_tail_scatter_kernel(double* __restrict__ out, int64_t n, int64_t idx_off,
                                                                PsisScalars* sc, const int64_t* __restrict__ tail_i,
                                                                const double* __restrict__ tail_out,
                                                                const double* __restrict__ blk_mom, int nblk,
                                                                int add_tail, double* __restrict__ result) {
  PDL_SYNC();
  __shared__ double red[32];
  if (sc->status) return;
  const int N = (int)sc->ntail;
  const double lse = sc->lse;
  if (out && sc->smoothed) {
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < N; r += gridDim.x * blockDim.x) {
      const int64_t li = tail_i[r] - idx_off;             // draws of other ranks are theirs to write
      if (li >= 0 && li < n) out[li] = tail_out[r] - lse;
    }
  }
  if (blockIdx.x == 0) {
    double sv = 0.0, se = 0.0;
    for (int b = threadIdx.x; b < nblk; b += blockDim.x) {
      sv += blk_mom[2 * b];
      se += blk_mom[2 * b + 1];
    }
    sv = block_sum(sv, red);
    se = block_sum(se, red);
    if (threadIdx.x == 0) {
      sv += add_tail ? sc->sumv : 0.0;                             // sharded: rank 0 alone carries the tail's share
      result[R_SUMV] = sv;
      // v <= 0 or NaN, so sum v is NaN exactly when some v is; exp_nonpos flushes a NaN with the sign bit set (the
      // v = inf - inf of a +inf draw) to 0, and the reference's sum exp(2 v) is NaN then
      result[R_SUMEXP2V] = sv != sv ? sv : se + (add_tail ? sc->sumexp2v : 0.0);
    }
  }
}

// ---- exact mode: full-data radix select of the (M+1)-th largest key ----------------------------
__global__ void __launch_bounds__(256) psis_exact_hist_kernel(const double* __restrict__ lw, int64_t n, PsisScalars* sc,
                                                              int shift, int bits, unsigned long long mask,
                                                              unsigned int* __restrict__ ghist) {
  __shared__ unsigned int hist[kBins];
  const unsigned int nb = 1u << bits;
  for (unsigned int b = threadIdx.x; b < nb; b += blockDim.x) hist[b] = 0;
  __syncthreads();
  const unsigned long long prefix = sc->prefix;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const int64_t iters = (n + nthreads - 1) / nthreads;
  for (int64_t it = 0; it < iters; ++it) {
    const int64_t i = it * nthreads + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    unsigned long long key = 0;
    bool ok = false;
    if (i < n) {
      key = dkey(lw[i]);
      ok = (key & mask) == prefix;
    }
    const unsigned int dig = ok ? (unsigned int)((key >> shift) & (nb - 1)) : 0xffffffffu;
    const unsigned int peers = __match_any_sync(0xffffffffu, dig);
    if (ok && (threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&hist[dig], __popc(peers));
  }
  __syncthreads();
  for (unsigned int b = threadIdx.x; b < nb; b += blockDim.x)
    if (hist[b]) atomicAdd(&ghist[b], hist[b]);
}

__global__ void psis_exact_scan_kernel(PsisScalars* sc, int shift, int bits, unsigned int* __restrict__ ghist, int last) {
  if (threadIdx.x != 0) return;
  const unsigned int nb = 1u << bits;
  unsigned long long K = sc->kth, cum = 0;
  for (int b = (int)nb - 1; b >= 0; --b) {
    const unsigned long long c = ghist[b];
    if (cum + c >= K) {
      sc->prefix |= (unsigned long long)b << shift;
      sc->kth = K - cum;
      break;
    }
    cum += c;
  }
  for (unsigned int b = 0; b < nb; ++b) ghist[b] = 0;
  if (last) {
    sc->t0key = sc->prefix;
    sc->t0 = dkey_inv(sc->prefix);
    sc->strict = 1;
  }
}

__global__ void psis_exact_begin_kernel(PsisScalars* sc) { sc->kth = (unsigned long long)sc->M + 1; sc->prefix = 0; }

// ---- stand-alone divergence-bound moments (diagnostics.py:148-186) --------------------------------
// pass 1: max; pass 2: sums.  out[0]=max, out[1]=sum r, out[2]=sum x, out[4]=sum (x-max)^2, out[5]=sum r^2,
// r = exp(x - max)^alpha (the second moments feed mean_and_check_mc_error, diagnostics.py:189-198)
__global__ void __launch_bounds__(256) dbound_max_kernel(const double* __restrict__ x, int64_t n, unsigned long long* mk) {
  double mx = -INFINITY;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    mx = fmax(mx, x[i]);
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) atomicMax(mk, dkey(mx));
}
__global__ void __launch_bounds__(256) dbound_sum_kernel(const double* __restrict__ x, int64_t n, double alpha,
                                                         const unsigned long long* mk, double* __restrict__ out) {
  __shared__ double red[32];
  const double mx = dkey_inv(*mk);
  double se = 0.0, sx = 0.0, sc = 0.0, se2 = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = x[i];
    const double r = pow(exp(v - mx), alpha);        // np.exp(lw - max) ** alpha
    se += r;
    se2 += r * r;
    sx += v;
    const double c = v - mx;
    sc += c * c;
  }
  se = block_sum(se, red);
  sx = block_sum(sx, red);
  sc = block_sum(sc, red);
  se2 = block_sum(se2, red);
  if (threadIdx.x == 0) {
    atomicAdd(&out[1], se);
    atomicAdd(&out[2], sx);
    atomicAdd(&out[4], sc);
    atomicAdd(&out[5], se2);
    if (blockIdx.x == 0) out[0] = mx;
  }
}

// ---------------------------------------------------------------------------------------------
struct PsisPlan {
  int M, m_sample, grid, tail_cap, mgrid, gchunks, kparts, vparts;
  unsigned int cap, cap_local, R;
  int64_t stride;
  size_t off_sc, off_candx, off_candi, off_blk, off_tmpv, off_tmpi, off_tmpb, off_tailv, off_taili, off_tailout,
      off_sorted, off_idxsorted, off_orderrank, off_bs, off_part, off_Ls, off_kpart, off_part3, off_mom, off_ghist,
      off_vhist, off_voff, off_gbuf, total;
};

static void psis_plan(int64_t n, double reff, PsisPlan& p, int64_t n_global = 0, int world = 1) {
  if (n_global <= 0) n_global = n;
  // tail length from the GLOBAL number of draws (_psis.py:158); a rank may own all of the tail
  p.M = (int)ceil(fmin(0.2 * (double)n_global, 3.0 * sqrt((double)n_global / reff)));
  if (p.M < 0) p.M = 0;
  p.m_sample = (int)(n < kSampleMax ? n : kSampleMax);
  p.stride = n / p.m_sample;
  const double f = (double)(p.M + 1) * (double)p.m_sample / (double)n;      // expected sample hits above the cutoff
  double R = ceil(f + 8.0 * sqrt(f) + 16.0);
  if (p.m_sample == n) R = p.M + 1;                                          // sample is everything: exact
  if (R > (double)n) R = (double)n;
  p.R = (unsigned int)fmin(R, 4.0e9);
  double expect = (double)p.R * (double)n / (double)p.m_sample;
  double cap = 4.0 * expect + 65536.0;
  if (cap > (double)n) cap = (double)n;
  if (cap < (double)(p.M + 1) && (double)(p.M + 1) <= (double)n) cap = (double)(p.M + 1);
  p.cap_local = (unsigned int)cap;
  // sharded: the same buffer later holds every rank's top (M+1) (see vb_psis_dist_global)
  p.cap = (unsigned int)fmin(fmax(cap, world > 1 ? (double)world * (p.M + 1) : 0.0), 4.0e9);
  p.tail_cap = p.M + 1;
  p.grid = sm_count() * 8;
  const int64_t need = (n / 4 + 255) / 256;
  if (need < p.grid) p.grid = (int)(need < 1 ? 1 : need);
  p.mgrid = 30 + (int)sqrt((double)p.tail_cap) + 2;
  p.kparts = 64;
  p.vparts = 64;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  p.off_sc = take(sizeof(PsisScalars));
  p.off_candx = take(sizeof(double) * p.cap);
  p.off_candi = take(sizeof(int64_t) * p.cap);
  p.off_blk = take(sizeof(double) * p.grid);
  p.off_tmpv = take(sizeof(double) * p.tail_cap);
  p.off_tmpi = take(sizeof(int64_t) * p.tail_cap);
  p.off_tmpb = take(sizeof(int) * p.tail_cap);
  p.off_tailv = take(sizeof(double) * p.tail_cap);
  p.off_taili = take(sizeof(int64_t) * p.tail_cap);
  p.off_tailout = take(sizeof(double) * p.tail_cap);
  p.off_sorted = take(sizeof(double) * p.tail_cap);
  p.off_idxsorted = take(sizeof(int64_t) * p.tail_cap);
  p.off_orderrank = take(sizeof(int) * p.tail_cap);
  p.off_bs = take(sizeof(double) * p.mgrid);
  p.gchunks = (p.tail_cap + kGpdChunk - 1) / kGpdChunk;
  p.off_part = take(sizeof(double) * (p.mgrid + kGpdJ) * p.gchunks);
  p.off_Ls = take(sizeof(double) * p.mgrid);
  p.off_kpart = take(sizeof(double) * p.kparts);
  p.off_part3 = take(sizeof(double) * 3 * p.vparts);
  p.off_mom = take(sizeof(double) * 2 * p.grid);
  p.off_ghist = take(sizeof(unsigned int) * kBins);
  p.off_vhist = take(sizeof(unsigned int) * 2 * kVBins);       // tail-bin counts, then cursors
  p.off_voff = take(sizeof(unsigned int) * kVBins);
  p.off_gbuf = take(sizeof(unsigned long long) * kGather);
  p.total = off;
}

// The table is a per-device __device__ symbol: track its upload per device (a process may drive several GPUs)
// and serialise the first upload (several host threads may enter together).
static std::mutex g_tab_mutex;
static bool g_tab_ready[64] = {false};
static int ensure_exp_table() {
  int dev = 0;
  VB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return set_error(VB_ERR_UNSUPPORTED, "psis: device ordinal out of range");
  std::lock_guard<std::mutex> lock(g_tab_mutex);
  if (g_tab_ready[dev]) return VB_OK;
  double tab[kExpTab];
  for (int j = 0; j < kExpTab; ++j) tab[j] = exp2((double)j / (double)kExpTab);
  VB_CUDA(cudaMemcpyToSymbol(g_exp2_tab, tab, sizeof(tab)));
  g_tab_ready[dev] = true;
  return VB_OK;
}

}  // namespace vb
using namespace vb;

extern "C" size_t vb_psis_workspace_bytes(int64_t n, double reff) {
  if (n <= 1 || !(reff > 0)) return 0;
  PsisPlan p;
  psis_plan(n, reff, p);
  return p.total;
}

extern "C" int64_t vb_psis_tail_capacity(int64_t n, double reff) {
  if (n <= 1 || !(reff > 0)) return 0;
  PsisPlan p;
  psis_plan(n, reff, p);
  return p.tail_cap;
}

namespace vb {
struct PsisPtrs {
  PsisScalars* sc;
  double *candx, *blk, *tmpv, *tailv, *tailout, *sorted, *bs, *part, *Ls, *kpart, *part3, *mom;
  int64_t *candi, *tmpi, *taili, *idxsorted;
  int *tmpb, *orderrank;
  unsigned int *ghist, *vhist, *vcur, *voff;
  unsigned long long* gbuf;
};
static void psis_ptrs(char* ws, const PsisPlan& p, PsisPtrs& q) {
  q.sc = reinterpret_cast<PsisScalars*>(ws + p.off_sc);
  q.candx = reinterpret_cast<double*>(ws + p.off_candx);
  q.candi = reinterpret_cast<int64_t*>(ws + p.off_candi);
  q.blk = reinterpret_cast<double*>(ws + p.off_blk);
  q.tmpv = reinterpret_cast<double*>(ws + p.off_tmpv);
  q.tmpi = reinterpret_cast<int64_t*>(ws + p.off_tmpi);
  q.tmpb = reinterpret_cast<int*>(ws + p.off_tmpb);
  q.tailv = reinterpret_cast<double*>(ws + p.off_tailv);
  q.taili = reinterpret_cast<int64_t*>(ws + p.off_taili);
  q.tailout = reinterpret_cast<double*>(ws + p.off_tailout);
  q.sorted = reinterpret_cast<double*>(ws + p.off_sorted);
  q.idxsorted = reinterpret_cast<int64_t*>(ws + p.off_idxsorted);
  q.orderrank = reinterpret_cast<int*>(ws + p.off_orderrank);
  q.bs = reinterpret_cast<double*>(ws + p.off_bs);
  q.part = reinterpret_cast<double*>(ws + p.off_part);
  q.Ls = reinterpret_cast<double*>(ws + p.off_Ls);
  q.kpart = reinterpret_cast<double*>(ws + p.off_kpart);
  q.part3 = reinterpret_cast<double*>(ws + p.off_part3);
  q.mom = reinterpret_cast<double*>(ws + p.off_mom);
  q.ghist = reinterpret_cast<unsigned int*>(ws + p.off_ghist);
  q.vhist = reinterpret_cast<unsigned int*>(ws + p.off_vhist);
  q.vcur = q.vhist + kVBins;
  q.voff = reinterpret_cast<unsigned int*>(ws + p.off_voff);
  q.gbuf = reinterpret_cast<unsigned long long*>(ws + p.off_gbuf);
}

// stage 1 (per rank): threshold, pass A over this rank's draws
static int psis_stage_local(const double* lw, int64_t n, int64_t idx_off, int exact, const PsisPlan& p, PsisPtrs& q,
                            cudaStream_t stream, int onepass = 0) {
  psis_init_kernel<<<8, 1024, 0, stream>>>(q.sc, p.M, q.ghist, q.vhist, onepass, (long long)n);
  VB_CHECK_LAUNCH();
  if (!exact) {
    psis_sample_select_kernel<<<(p.R <= 256 && p.m_sample == kSampleMax) ? kSampleMax / kSelThreads : 1, kSelThreads, 0, stream>>>(
        lw, p.stride, p.m_sample, p.R, q.sc, q.gbuf);
    VB_CHECK_LAUNCH();
  } else {
    psis_exact_begin_kernel<<<1, 1, 0, stream>>>(q.sc);
    VB_CHECK_LAUNCH();
    int shift = 64;
    unsigned long long mask = 0;
    while (shift > 0) {
      const int bits = shift >= kDigitBits ? kDigitBits : shift;
      shift -= bits;
      psis_exact_hist_kernel<<<p.grid, 256, 0, stream>>>(lw, n, q.sc, shift, bits, mask, q.ghist);
      VB_CHECK_LAUNCH();
      psis_exact_scan_kernel<<<1, 32, 0, stream>>>(q.sc, shift, bits, q.ghist, shift == 0);
      VB_CHECK_LAUNCH();
      mask |= (unsigned long long)((1u << bits) - 1) << shift;
    }
  }
  if (onepass)
    psis_pass_a_lean_kernel<true><<<p.grid, 256, 0, stream>>>(lw, n, idx_off, q.sc, q.candx, q.candi, p.cap, q.blk, q.mom, q.ghist);
  else
    psis_pass_a_lean_kernel<false><<<p.grid, 256, 0, stream>>>(lw, n, idx_off, q.sc, q.candx, q.candi, p.cap, q.blk, q.mom, q.ghist);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

// stage 2 (replicated): cutoff, tail ranking, GPD fit, smoothed values, log-sum-exp from the candidate list
static int psis_stage_select(const PsisPlan& p, PsisPtrs& q, int nblk, int raw, cudaStream_t stream, bool need_hist) {
  const int cgrid = sm_count() * 2;
  if (need_hist)      // pass A fills the histogram itself; candidates imported from records need it built here
    VB_CUDA(launch_pdl(psis_cand_hist_kernel, dim3(cgrid), dim3(256), stream, q.sc, q.candx, p.cap, q.ghist));
  VB_CUDA(launch_pdl(psis_cand_gather_kernel, dim3(cgrid / 4 > 0 ? cgrid / 4 : 1), dim3(kSelThreads), stream, q.sc, q.candx, p.cap, q.ghist, q.gbuf,
                     q.blk, q.mom, nblk));
  VB_CUDA(launch_pdl(psis_tail_count_kernel, dim3(cgrid / 4 > 0 ? cgrid / 4 : 1), dim3(kSelThreads), stream, q.sc, q.candx, q.vhist, q.voff));
  VB_CUDA(launch_pdl(psis_tail_place_kernel, dim3(cgrid), dim3(256), stream, q.sc, q.candx, q.candi, q.voff, q.vcur, q.tmpv, q.tmpi, q.tmpb,
                                                    (unsigned)p.tail_cap, raw));
  return VB_OK;
}

static int psis_stage_global(const PsisPlan& p, PsisPtrs& q, int nblk, double* result, int64_t* tail_idx,
                             int32_t* tail_rank, cudaStream_t stream, bool need_hist) {
  int rc = psis_stage_select(p, q, nblk, 0, stream, need_hist);
  if (rc) return rc;
  int blocks = (p.tail_cap + 255) / 256;
  if (blocks > sm_count() * 4) blocks = sm_count() * 4;
  VB_CUDA(launch_pdl(psis_tail_rank_kernel, dim3(blocks), dim3(256), stream, q.sc, q.tmpv, q.tmpi, q.tmpb, q.voff, q.vhist, q.tailv, q.taili, q.sorted));
  if (tail_idx && tail_rank) {
    VB_CUDA(launch_pdl(psis_tail_index_order_kernel, dim3(blocks), dim3(256), stream, q.sc, q.taili, tail_idx, tail_rank));
  }
  VB_CUDA(launch_pdl(psis_gpd_grid_kernel, dim3((p.mgrid + kGpdJ - 1) / kGpdJ, p.gchunks), dim3(256), stream, q.sc, q.sorted, q.bs, q.part, q.Ls));
  VB_CUDA(launch_pdl(psis_gpd_k_kernel, dim3(p.kparts), dim3(256), stream, q.sc, q.sorted, q.kpart));
  VB_CUDA(launch_pdl(psis_tail_values_kernel, dim3(p.vparts), dim3(256), stream, q.sc, q.kpart, p.kparts, q.tailv, q.tailout, q.part3, result));
  return VB_OK;
}

// stage 3 (per rank): pass B over this rank's draws and the scatter of its own smoothed tail entries
static int psis_stage_apply(const double* lw, double* out, int64_t n, int64_t idx_off, int add_tail, const PsisPlan& p,
                            PsisPtrs& q, double* result, cudaStream_t stream) {
  if (out) {
    VB_CUDA(launch_pdl(psis_pass_b_kernel, dim3(p.grid), dim3(256), stream, lw, out, n, q.sc, q.mom));
  } else {
    VB_CUDA(launch_pdl(psis_pass_b_moments_kernel, dim3(p.grid), dim3(256), stream, lw, n, q.sc, q.mom));
  }
  int blocks = (p.tail_cap + 255) / 256;
  if (blocks > sm_count()) blocks = sm_count();
  VB_CUDA(launch_pdl(psis_tail_scatter_kernel, dim3(blocks), dim3(256), stream, out, n, idx_off, q.sc, q.taili, q.tailout, q.mom, p.grid, add_tail,
                                                       result));
  return VB_OK;
}

// ---- draw-sharded PSIS: the record a rank ships = its top (M+1) values with their global indices ------------
// record (doubles): [0] local max, [1] c_r = local (M+1)-th largest (raw; -inf if the rank has < M+1 draws),
// [2] log sum exp(x - max_r) over the local draws NOT represented in the record, [3] count (-status on failure),
// then vals[M+1], then idx[M+1] (int64 bit patterns).  The local tail (values > c_r, at most M) is padded
// with copies of c_r (index -1): a rank's top (M+1) with ties cut.  The global (M+1)-th largest is the
// (M+1)-th largest of the union of the records, and every member of the global tail is in its rank's local tail.
__global__ void __launch_bounds__(256) psis_export_kernel(const PsisScalars* sc, const double* __restrict__ tmp_v,
                                                          const int64_t* __restrict__ tmp_i,
                                                          const double* __restrict__ cand_x,
                                                          const int64_t* __restrict__ cand_i, int small,
                                                          double* __restrict__ rec) {
  const int K = sc->M + 1;
  double* vals = rec + 4;
  int64_t* idx = reinterpret_cast<int64_t*>(rec + 4 + K);
  const double maxv = dkey_inv(sc->maxkey);
  if (small) {            // fewer than M+1 local draws: all of them are candidates (t0 = local minimum)
    const int C = (int)sc->ncand;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < K; j += gridDim.x * blockDim.x) {
      vals[j] = j < C ? cand_x[j] : -INFINITY;
      idx[j] = j < C ? cand_i[j] : -1;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      rec[0] = maxv; rec[1] = -INFINITY; rec[2] = -INFINITY; rec[3] = (double)C;
    }
    return;
  }
  if (sc->status) {
    if (blockIdx.x == 0 && threadIdx.x == 0) { rec[0] = maxv; rec[1] = -INFINITY; rec[2] = -INFINITY; rec[3] = -(double)sc->status; }
    return;
  }
  const int nt = (int)sc->ntail;
  const double c = dkey_inv(sc->cutkey);
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < K; j += gridDim.x * blockDim.x) {
    vals[j] = j < nt ? tmp_v[j] : c;
    idx[j] = j < nt ? tmp_i[j] : -1;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const double below = sc->body_below == 0.0 ? 0.0 : sc->body_below * exp(sc->tbase - maxv);
    double body = below + sc->body_cand - (double)(K - nt) * exp(c - maxv);     // the copies of c_r travel in the record
    if (!(body > 0.0) && body == body) body = 0.0;          // (a NaN stays: it must reach every rank's log-sum-exp)
    rec[0] = maxv; rec[1] = c; rec[2] = log(body); rec[3] = (double)K;
  }
}

// merged candidate list + global scalars into the control block (replicated on every rank)
__global__ void __launch_bounds__(256) psis_import_kernel(PsisScalars* sc, const double* __restrict__ recs, int world,
                                                          int reclen, double* __restrict__ cand_x,
                                                          int64_t* __restrict__ cand_i, double* __restrict__ blk, int nblk) {
  const int K = sc->M + 1;
  int bad = 0;
  for (int r = 0; r < world; ++r) bad |= recs[(size_t)r * reclen + 3] < 0.0;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double mx = -INFINITY, t0 = -INFINITY, below = 0.0;
    unsigned int total = 0;
    for (int r = 0; r < world; ++r) {
      const double* h = recs + (size_t)r * reclen;
      mx = fmax(mx, h[0]);
      t0 = fmax(t0, h[1]);
      if (h[3] > 0.0) total += (unsigned int)h[3];
    }
    for (int r = 0; r < world; ++r) {
      const double* h = recs + (size_t)r * reclen;
      if (h[2] > -INFINITY || h[2] != h[2]) below += exp(h[2] + h[0] - t0);          // every term is <= exp(c_r - t0) * count <= count
    }
    sc->maxkey = dkey(mx);
    sc->t0 = t0;
    sc->hist_hi = mx;
    sc->tbase = t0;
    sc->t0key = dkey(t0);
    sc->ncand = bad ? 0u : total;
    sc->strict = 0;
    if (bad) sc->status = 1;              // some rank's sampled threshold missed: every rank reruns exact
    blk[0] = below;
  }
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < nblk; b += gridDim.x * blockDim.x)
    if (b > 0) blk[b] = 0.0;
  if (bad) return;
  for (int r = blockIdx.y; r < world; r += gridDim.y) {
    unsigned int off = 0;
    for (int q = 0; q < r; ++q) off += (unsigned int)recs[(size_t)q * reclen + 3];
    const double* h = recs + (size_t)r * reclen;
    const int cnt = (int)h[3];
    const double* vals = h + 4;
    const int64_t* idx = reinterpret_cast<const int64_t*>(h + 4 + K);
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < cnt; j += gridDim.x * blockDim.x) {
      cand_x[off + j] = vals[j];
      cand_i[off + j] = idx[j];
    }
  }
}
}  // namespace vb

extern "C" int vb_psislw_f64(const double* lw, double* out, int64_t n, double reff, int exact, double* result,
                             int64_t* tail_idx, int32_t* tail_rank, void* workspace, size_t workspace_bytes,
                             cudaStream_t stream) {
  if (n <= 1) return set_error(VB_ERR_INVALID_ARG, "More than one log-weight needed.");       // _psis.py:144-145
  if (!(reff > 0)) return set_error(VB_ERR_INVALID_ARG, "psislw: Reff must be positive");
  if (!lw || !result) return set_error(VB_ERR_INVALID_ARG, "psislw: null pointer");
  PsisPlan p;
  psis_plan(n, reff, p);
  if (!workspace || workspace_bytes < p.total) return set_error(VB_ERR_WORKSPACE, "psislw: workspace too small");
  int rc = ensure_exp_table();
  if (rc) return rc;
  PsisPtrs q;
  psis_ptrs(static_cast<char*>(workspace), p, q);
  VB_CUDA(cudaMemsetAsync(result, 0, sizeof(double) * R_COUNT, stream));
  // no output array: k-hat and the bound moments from ONE pass over the draws
  const int onepass = !out ? 1 : 0;
  if ((rc = psis_stage_local(lw, n, 0, exact, p, q, stream, onepass))) return rc;
  if ((rc = psis_stage_global(p, q, p.grid, result, tail_idx, tail_rank, stream, false))) return rc;
  if (onepass) return VB_OK;
  return psis_stage_apply(lw, out, n, 0, 1, p, q, result, stream);
}

// ---- draw-sharded PSIS (SURVEY.md 8(e)): stage 1 on each rank, one fixed-size all-gather of the records on the
// host side (NCCL), stage 2 replicated on the merged records, stage 3 on each rank.  No host sync in between. ----
extern "C" size_t vb_psis_dist_workspace_bytes(int64_t n_local, int64_t n_global, double reff, int world) {
  if (n_local <= 1 || n_global < n_local || !(reff > 0) || world < 1) return 0;
  PsisPlan p;
  psis_plan(n_local, reff, p, n_global, world);
  return p.total;
}

extern "C" int64_t vb_psis_dist_record_doubles(int64_t n_global, double reff) {
  if (n_global <= 1 || !(reff > 0)) return 0;
  PsisPlan p;
  psis_plan(n_global, reff, p);
  return 4 + 2 * (int64_t)(p.M + 1);
}

extern "C" int vb_psis_dist_local(const double* lw, int64_t n_local, int64_t idx_off, int64_t n_global, double reff,
                                  int world, int exact, double* record, void* workspace, size_t workspace_bytes,
                                  cudaStream_t stream) {
  if (n_local <= 1 || n_global < n_local || !(reff > 0) || world < 1 || !lw || !record)
    return set_error(VB_ERR_INVALID_ARG, "psis_dist_local: bad arguments");
  PsisPlan p;
  psis_plan(n_local, reff, p, n_global, world);
  if (!workspace || workspace_bytes < p.total) return set_error(VB_ERR_WORKSPACE, "psis_dist_local: workspace too small");
  int rc = ensure_exp_table();
  if (rc) return rc;
  PsisPtrs q;
  psis_ptrs(static_cast<char*>(workspace), p, q);
  const bool small = n_local < (int64_t)p.M + 1;         // the sample is the whole shard and everything is a candidate
  if ((rc = psis_stage_local(lw, n_local, idx_off, small ? 0 : exact, p, q, stream))) return rc;
  if (!small && (rc = psis_stage_select(p, q, p.grid, 1, stream, false))) return rc;
  int blocks = (p.M + 1 + 255) / 256;
  if (blocks > sm_count()) blocks = sm_count();
  psis_export_kernel<<<blocks, 256, 0, stream>>>(q.sc, q.tmpv, q.tmpi, q.candx, q.candi, small ? 1 : 0, record);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

extern "C" int vb_psis_dist_global(const double* records, int64_t n_local, int64_t n_global, double reff, int world,
                                   double* result, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!records || !result || world < 1) return set_error(VB_ERR_INVALID_ARG, "psis_dist_global: bad arguments");
  PsisPlan p;
  psis_plan(n_local, reff, p, n_global, world);
  if (!workspace || workspace_bytes < p.total) return set_error(VB_ERR_WORKSPACE, "psis_dist_global: workspace too small");
  PsisPtrs q;
  psis_ptrs(static_cast<char*>(workspace), p, q);
  VB_CUDA(cudaMemsetAsync(result, 0, sizeof(double) * R_COUNT, stream));
  psis_init_kernel<<<8, 1024, 0, stream>>>(q.sc, p.M, q.ghist, q.vhist, 0, (long long)n_local);
  VB_CHECK_LAUNCH();
  const int reclen = 4 + 2 * (p.M + 1);
  int bx = (p.M + 1 + 255) / 256;
  if (bx > 64) bx = 64;
  psis_import_kernel<<<dim3(bx, world > 64 ? 64 : world), 256, 0, stream>>>(q.sc, records, world, reclen, q.candx, q.candi,
                                                                          q.blk, p.grid);
  VB_CHECK_LAUNCH();
  return psis_stage_global(p, q, p.grid, result, nullptr, nullptr, stream, true);
}

extern "C" int vb_psis_dist_apply(const double* lw, double* out, int64_t n_local, int64_t idx_off, int64_t n_global,
                                  double reff, int world, int rank, double* result, void* workspace,
                                  size_t workspace_bytes, cudaStream_t stream) {
  if (!lw || !result || n_local <= 1) return set_error(VB_ERR_INVALID_ARG, "psis_dist_apply: bad arguments");
  PsisPlan p;
  psis_plan(n_local, reff, p, n_global, world);
  if (!workspace || workspace_bytes < p.total) return set_error(VB_ERR_WORKSPACE, "psis_dist_apply: workspace too small");
  PsisPtrs q;
  psis_ptrs(static_cast<char*>(workspace), p, q);
  return psis_stage_apply(lw, out, n_local, idx_off, rank == 0, p, q, result, stream);
}

extern "C" int vb_divergence_moments_f64(const double* lw, int64_t n, double alpha, double* out3, cudaStream_t stream) {
  if (n <= 0 || !lw || !out3) return set_error(VB_ERR_INVALID_ARG, "divergence_moments: bad arguments");
  if (!(alpha > 1.0)) return set_error(VB_ERR_INVALID_ARG, "alpha must be greater than 1");      // diagnostics.py:172-173
  // out[3] doubles as scratch for the max key
  VB_CUDA(cudaMemsetAsync(out3, 0, sizeof(double) * 8, stream));
  int grid = sm_count() * 8;
  const int64_t need = (n + 255) / 256;
  if (need < grid) grid = (int)need;
  dbound_max_kernel<<<grid, 256, 0, stream>>>(lw, n, reinterpret_cast<unsigned long long*>(out3 + 3));
  VB_CHECK_LAUNCH();
  dbound_sum_kernel<<<grid, 256, 0, stream>>>(lw, n, alpha, reinterpret_cast<unsigned long long*>(out3 + 3), out3);
  VB_CHECK_LAUNCH();
  return VB_OK;
}
