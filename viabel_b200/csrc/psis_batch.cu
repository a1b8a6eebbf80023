// Batched PSIS: every column of a column-major n x m matrix of log-weights smoothed in ONE launch
// (reference viabel/_psis.py:113-209 for 2-D input, and the psislw + sumlogs of psisloo :69-110).
//
// One CTA of 1024 threads owns one column at a time (a persistent grid walks the columns), keeps the whole column in
// shared memory as order-preserving keys and runs the reference's one-column PSIS on it (tail ties ranked by index):
//   load     : one read of the column, maximum key, NaN test;
//   select   : (M+1)-th largest key by the 64-bit radix select of the one-column pipeline (cta_select_kth_largest),
//              cutoff = max(that value - max, log(DBL_MIN));
//   tail     : compaction of {x - max > cutoff} (n2 <= M entries), rank by counting on (value, index) -- the stable
//              argsort of psislw_1d -- into exp(v) - exp(cutoff) in ascending order;
//   fit      : Zhang-Stephens grid (one warp per grid point, LogProd), gpd_weights, k-hat, sigma, prior;
//   smooth   : tail entries replaced by log(gpinv((r + 0.5) / n2) + exp(cutoff)) clipped at 0 -- their keys in shared
//              memory become markers (NaN keys, which a column that reaches this point cannot hold) naming rank r;
//   finish   : log-sum-exp over the column, out = v - lse written once, and optionally the psisloo term
//              log-sum-exp_i(out_i - lw_i), so that psisloo can run without an output array (8 bytes per entry).
// Traffic: one read (and with `out` one write) of each entry.  All sums run in a fixed order and the only atomics
// are integer ones, so repeated calls are bitwise equal.
#include <mutex>

#include "psis_internal.cuh"

namespace vb {

constexpr int kBatchThreads = kSelThreads;           // the select's bin scan covers 2048 bins with two per thread
constexpr size_t kBatchSmemMax = 232448;             // 227 KB: the per-block shared-memory opt-in of sm_100
constexpr unsigned long long kInfKey = 0xFFF0000000000000ull;   // dkey(+inf); keys above it are NaN bit patterns
constexpr unsigned long long kMark = kInfKey + 1;                // kMark + r: tail entry of rank r, smoothed

// Shared-memory plan of one CTA: the column's keys (8 n bytes), then a region used first as the select's histogram
// and then as the tail arrays (24 bytes per possible tail entry), the GPD grid's profile likelihoods, and a small
// fixed part (reduction scratch, the control block gpd_weights writes b-hat into).
struct BatchLayout {
  int M, mg;
  size_t off_red, off_kred, off_wtot, off_sh, off_sc, off_cnt, off_keys, off_u, off_ci, off_sx, off_sidx,
      off_Ls, total;
};

static void batch_layout(int64_t n, double reff, BatchLayout& L) {
  L.M = (int)ceil(fmin(0.2 * (double)n, 3.0 * sqrt((double)n / reff)));     // _psis.py:158, as psis_plan
  L.mg = 30 + (int)sqrt((double)L.M);                                        // grid points of the longest tail
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 16); return o; };
  L.off_red = take(sizeof(double) * 32);
  L.off_kred = take(sizeof(unsigned long long) * 32);
  L.off_wtot = take(sizeof(unsigned int) * 32);
  L.off_sh = take(sizeof(unsigned long long) * 2);
  L.off_sc = take(sizeof(PsisScalars));
  L.off_cnt = take(sizeof(unsigned int) * 4);
  L.off_keys = take(sizeof(unsigned long long) * (size_t)n);
  // union: the select's histogram, then cv/tx[M] (value at compaction, later the raw draw by rank), ci[M], sx[M], sidx[M]
  const size_t K = (size_t)L.M;
  const size_t tail = align_up(8 * K, 16) + align_up(4 * K, 16) + align_up(8 * K, 16) + 4 * K;
  L.off_u = take(tail > sizeof(unsigned int) * kBins ? tail : sizeof(unsigned int) * kBins);
  L.off_ci = L.off_u + align_up(8 * K, 16);
  L.off_sx = L.off_ci + align_up(4 * K, 16);
  L.off_sidx = L.off_sx + align_up(8 * K, 16);
  L.off_Ls = take(sizeof(double) * L.mg);
  L.total = off;
}

struct BatchArgs {
  const double* lw;
  int64_t ld;
  int n;
  int64_t m;
  double* out;
  int64_t ldo;
  double* khat;
  double* result;
  double* loo;
  double* scratch;       // [gridDim.x][2 mg]: the grid points b_j and the sums of log1p(-b_j x) gpd_weights reads
};

__global__ void __launch_bounds__(kBatchThreads, 1) psis_batch_kernel(BatchArgs a, BatchLayout L) {
  extern __shared__ __align__(16) unsigned char smem[];
  double* red = reinterpret_cast<double*>(smem + L.off_red);
  unsigned long long* kred = reinterpret_cast<unsigned long long*>(smem + L.off_kred);
  unsigned int* wtot = reinterpret_cast<unsigned int*>(smem + L.off_wtot);
  unsigned long long* sh = reinterpret_cast<unsigned long long*>(smem + L.off_sh);
  PsisScalars* scs = reinterpret_cast<PsisScalars*>(smem + L.off_sc);
  unsigned int* cnt = reinterpret_cast<unsigned int*>(smem + L.off_cnt);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem + L.off_keys);
  unsigned int* hist = reinterpret_cast<unsigned int*>(smem + L.off_u);
  double* cv = reinterpret_cast<double*>(smem + L.off_u);        // tail values at compaction; tx by rank later
  double* tx = cv;
  int* ci = reinterpret_cast<int*>(smem + L.off_ci);
  double* sx = reinterpret_cast<double*>(smem + L.off_sx);
  int* sidx = reinterpret_cast<int*>(smem + L.off_sidx);
  double* Ls = reinterpret_cast<double*>(smem + L.off_Ls);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int n = a.n, M = L.M;
  double* bs = a.scratch + (size_t)blockIdx.x * 2 * L.mg;
  double* part = bs + L.mg;

  for (int64_t j = blockIdx.x; j < a.m; j += gridDim.x) {
    // ---- load: keys, maximum, NaN test
    const double* col = a.lw + j * a.ld;
    unsigned long long kmax = 0;
    bool nan = false;
#pragma unroll 4
    for (int i = tid; i < n; i += kBatchThreads) {
      const double x = col[i];
      nan |= x != x;
      const unsigned long long k = dkey(x);
      keys[i] = k;
      kmax = k > kmax ? k : kmax;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long v = __shfl_xor_sync(0xffffffffu, kmax, o);
      kmax = v > kmax ? v : kmax;
    }
    if (lane == 0) kred[w] = kmax;
    if (tid == 0) cnt[0] = 0;
    double* ocol = a.out ? a.out + j * a.ldo : nullptr;
    if (__syncthreads_or(nan)) {
      // a NaN makes the reference's maximum NaN: every output is NaN and the tail {x > cutoff} is empty (k-hat +inf)
      if (ocol)
        for (int i = tid; i < n; i += kBatchThreads) ocol[i] = NAN;
      if (tid < R_COUNT && a.result) {
        const double v = tid == R_KHAT ? INFINITY : (tid == R_CUTOFF || tid == R_LSE || tid == R_MAX) ? NAN
                         : tid == R_M ? (double)M : tid == R_NCAND ? (double)n : 0.0;
        a.result[j * R_COUNT + tid] = v;
      }
      if (tid == 0) {
        a.khat[j] = INFINITY;
        if (a.loo) a.loo[j] = NAN;
      }
      __syncthreads();
      continue;
    }
    kmax = 0;
#pragma unroll 8
    for (int u = 0; u < 32; ++u) kmax = kred[u] > kmax ? kred[u] : kmax;
    const double maxv = dkey_inv(kmax);

    // ---- cutoff: the (M+1)-th largest value, exactly
    const unsigned long long cutkey = cta_select_kth_largest(keys, (unsigned int)n, (unsigned long long)M + 1, hist, sh, wtot);
    const double cutoff = fmax(dkey_inv(cutkey) - maxv, log(DBL_MIN));       // _psis.py:159, :170-173
    const double expcut = exp(cutoff);

    // ---- tail compaction (order arbitrary here; ranked below)
    for (int i0 = 0; i0 < n; i0 += kBatchThreads) {
      const int i = i0 + tid;
      const double v = i < n ? dkey_inv(keys[i]) - maxv : -INFINITY;
      const bool t = v > cutoff;
      const unsigned int ball = __ballot_sync(0xffffffffu, t);
      if (ball) {
        unsigned int base = 0;
        if (lane == __ffs(ball) - 1) base = atomicAdd(cnt, (unsigned int)__popc(ball));
        base = __shfl_sync(0xffffffffu, base, __ffs(ball) - 1);
        if (t) {
          const unsigned int slot = base + __popc(ball & ((1u << lane) - 1));
          cv[slot] = v;
          ci[slot] = i;
        }
      }
    }
    __syncthreads();
    const int n2 = (int)cnt[0];
    // ---- rank by (value, index): psislw_1d's stable argsort of the tail
    for (int c = tid; c < n2; c += kBatchThreads) {
      const double v = cv[c];
      const int id = ci[c];
      int r = 0;
      for (int d = 0; d < n2; ++d) {
        const double vd = cv[d];
        r += (vd < v) || (vd == v && ci[d] < id);
      }
      sx[r] = exp(v) - expcut;                       // _psis.py:185-186
      sidx[r] = id;
    }
    __syncthreads();

    // ---- generalised Pareto fit (_psis.py:212-332)
    double k = INFINITY, sigma = 0.0;
    if (n2 > 4) {
      const int mg = 30 + (int)sqrt((double)n2);
      const double xq = sx[(int)(n2 / 4.0 + 0.5) - 1];
      const double xmax = sx[n2 - 1];
      for (int jj = w; jj < mg; jj += kBatchThreads / 32) {
        double b = 1.0 - sqrt((double)mg / ((double)(jj + 1) - 0.5));
        b /= 3.0 * xq;
        b += 1.0 / xmax;
        LogProd lp;
        for (int i = lane; i < n2; i += 32) lp.add(-b, sx[i]);
        const double s = warp_sum(lp.result());
        if (lane == 0) {
          bs[jj] = b;
          part[jj] = s;
        }
      }
      __threadfence();
      __syncthreads();
      gpd_weights(scs, bs, part, 1, Ls, n2, mg, red);
      __syncthreads();
      const double bhat = scs->bhat;
      LogProd lp;
      for (int i = tid; i < n2; i += kBatchThreads) lp.add(-bhat, sx[i]);
      const double s = block_sum(lp.result(), red);
      k = s / (double)n2;
      sigma = -k / bhat;
      k = k * (double)n2 / ((double)n2 + 10.0) + 5.0 / ((double)n2 + 10.0);
    }
    const bool smooth = (k >= 1.0 / 3.0) && !isinf(k);
    if (smooth) {
      for (int r = tid; r < n2; r += kBatchThreads) {
        double v = log(gpinv1(((double)r + 0.5) / (double)n2, k, sigma) + expcut);     // :190-197
        v = v > 0.0 ? 0.0 : v;                                                           // :199
        const int id = sidx[r];
        tx[r] = dkey_inv(keys[id]);
        sx[r] = v;
        keys[id] = kMark + (unsigned long long)r;
      }
      __syncthreads();
    }

    // ---- log-sum-exp, outputs, psisloo term
    double acc = 0.0;
    for (int i = tid; i < n; i += kBatchThreads) {
      const unsigned long long key = keys[i];
      acc += exp(key > kInfKey ? sx[key - kMark] : dkey_inv(key) - maxv);    // (a NaN from a +inf draw reaches the sum)
    }
    const double total = block_sum(acc, red);
    const double lse = log(total);
    double tmax = -INFINITY;
    bool tnan = false;
    for (int i = tid; i < n; i += kBatchThreads) {
      const unsigned long long key = keys[i];
      double v, x;
      if (key > kInfKey) {
        v = sx[key - kMark];
        x = tx[key - kMark];
      } else {
        x = dkey_inv(key);
        v = x - maxv;
      }
      const double o = v - lse;
      if (ocol) ocol[i] = o;
      const double t = o + (-x);
      tnan |= t != t;
      tmax = fmax(tmax, t);
    }
    double loo = 0.0;
    if (a.loo) {        // sumlogs (_psis.py:380-396) of lw_smoothed + log_lik, log_lik = -lw
      tmax = block_max(tmax, red);
      const bool anynan = __syncthreads_or(tnan);
      double s = 0.0;
      for (int i = tid; i < n; i += kBatchThreads) {
        const unsigned long long key = keys[i];
        double v, x;
        if (key > kInfKey) {
          v = sx[key - kMark];
          x = tx[key - kMark];
        } else {
          x = dkey_inv(key);
          v = x - maxv;
        }
        const double d = ((v - lse) + (-x)) - tmax;
        s += exp(d);
      }
      s = block_sum(s, red);
      loo = anynan ? NAN : log(s) + tmax;
    }
    const double kh = total != total ? INFINITY : k;
    if (tid < R_COUNT && a.result) {
      double v = 0.0;
      switch (tid) {
        case R_KHAT: v = kh; break;
        case R_SIGMA: v = sigma; break;
        case R_N2: v = (double)n2; break;
        case R_CUTOFF: v = cutoff; break;
        case R_LSE: v = lse; break;
        case R_MAX: v = maxv; break;
        case R_M: v = (double)M; break;
        case R_NCAND: v = (double)n; break;
        case R_SMOOTHED: v = smooth ? 1.0 : 0.0; break;
        default: break;
      }
      a.result[j * R_COUNT + tid] = v;
    }
    if (tid == 0) {
      a.khat[j] = kh;
      if (a.loo) a.loo[j] = loo;
    }
    __syncthreads();        // the next column overwrites the keys and the tail arrays
  }
}

// Scratch for gpd_weights (it reads the grid points and their sums through L2), from a per-device stream-ordered
// pool that keeps its memory between calls: no host synchronisation, and concurrent calls on different streams get
// different blocks.
static std::mutex g_pool_mutex;
static cudaMemPool_t g_pool[64];
static bool g_kernel_ready[64] = {false};
static int batch_prepare(int dev, cudaMemPool_t* pool) {
  std::lock_guard<std::mutex> lock(g_pool_mutex);
  if (!g_kernel_ready[dev]) {
    VB_CUDA(cudaFuncSetAttribute(psis_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBatchSmemMax));
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    VB_CUDA(cudaMemPoolCreate(&g_pool[dev], &props));
    uint64_t keep = 64ull << 20;
    VB_CUDA(cudaMemPoolSetAttribute(g_pool[dev], cudaMemPoolAttrReleaseThreshold, &keep));
    g_kernel_ready[dev] = true;
  }
  *pool = g_pool[dev];
  return VB_OK;
}

}  // namespace vb
using namespace vb;

extern "C" int64_t vb_psis_batch_max_n(double reff) {
  if (!(reff > 0)) return 0;
  BatchLayout L;
  int64_t lo = 1, hi = (int64_t)(kBatchSmemMax / sizeof(unsigned long long)) + 1;     // layout(lo) fits, layout(hi) not
  batch_layout(2, reff, L);
  if (L.total > kBatchSmemMax) return 0;
  while (hi - lo > 1) {
    const int64_t mid = lo + (hi - lo) / 2;
    batch_layout(mid, reff, L);
    if (L.total <= kBatchSmemMax) lo = mid; else hi = mid;
  }
  return lo;
}

extern "C" int vb_psislw_batch_f64(const double* lw, int64_t ld, int64_t n, int64_t m, double reff, double* out,
                                   int64_t ldo, double* khat, double* result, double* loo, cudaStream_t stream) {
  if (n <= 1) return set_error(VB_ERR_INVALID_ARG, "More than one log-weight needed.");       // _psis.py:144-145
  if (m < 0 || ld < n || (out && ldo < n)) return set_error(VB_ERR_INVALID_ARG, "psislw_batch: bad shape or leading dimension");
  if (!(reff > 0)) return set_error(VB_ERR_INVALID_ARG, "psislw: Reff must be positive");
  if (!lw || !khat) return set_error(VB_ERR_INVALID_ARG, "psislw_batch: null pointer");
  if (n > vb_psis_batch_max_n(reff))
    return set_error(VB_ERR_UNSUPPORTED, "psislw_batch: column longer than vb_psis_batch_max_n(reff)");
  if (m == 0) return VB_OK;
  BatchLayout L;
  batch_layout(n, reff, L);
  int rc, dev = 0;
  VB_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return set_error(VB_ERR_UNSUPPORTED, "psis: device ordinal out of range");
  cudaMemPool_t pool;
  if ((rc = batch_prepare(dev, &pool))) return rc;
  int per_sm = 0;
  VB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, psis_batch_kernel, kBatchThreads, L.total));
  if (per_sm < 1) return set_error(VB_ERR_UNSUPPORTED, "psislw_batch: the kernel does not fit on an SM");
  const int64_t resident = (int64_t)per_sm * sm_count();
  const int grid = (int)(m < resident ? m : resident);
  BatchArgs a{lw, ld, (int)n, m, out, ldo, khat, result, loo, nullptr};
  VB_CUDA(cudaMallocFromPoolAsync(reinterpret_cast<void**>(&a.scratch), sizeof(double) * 2 * L.mg * (size_t)grid, pool, stream));
  psis_batch_kernel<<<grid, kBatchThreads, L.total, stream>>>(a, L);
  const cudaError_t e = cudaGetLastError();
  VB_CUDA(cudaFreeAsync(a.scratch, stream));
  if (e != cudaSuccess) return set_cuda_error(e);
  return VB_OK;
}
