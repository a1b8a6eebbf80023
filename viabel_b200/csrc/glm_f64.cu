// Float64 "exact path" of the GLM model plugin: one fused sweep over the observations.
//
//   z[n,s] = sum_j X[n,j] theta[s,j]          (DMMA m8n8k4, X tile resident in shared memory)
//   ll[s]  = sum_n loglik(y_n, z[n,s])        (link epilogue on the accumulators, in registers)
//   gmu[j] = sum_n X[n,j] sum_s w_s r[n,s]    r = dloglik/dz
//   ge[j]  = sum_n X[n,j] (r.w E)[n,j]        second DMMA whose A operand IS the epilogue's
//                                             register fragment (no N x S intermediate anywhere)
//
// Replaces the user's numpy log_density + autograd reverse sweep (reference models.py:27-39,
// objectives.py:161-167): X.Theta^T, logaddexp, sum, and the transposed GEMM of the VJP.
//
// Data layout: X row-major [N,ldx] fp64 in HBM, read once per sweep.  theta / base draws are
// re-packed once per sweep into mma-fragment order (glm_pack_f64_kernel) so every operand load
// in the hot loop is a fully coalesced 512-byte LDG.128 that hits L2.
#include "common.cuh"

namespace vb {


__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile(
      "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(c0), "+d"(c1)
      : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------------------
// Packing: thetaP[((sb*KG + kg)*32 + lane)] = (theta[8sb+g][8kg+2t], theta[8sb+g][8kg+2t+1])
//          baseP [((sb*KG + jb)*32 + lane)] = (w? no: base[8sb+2t][8jb+g], base[8sb+2t+1][8jb+g])
// with g = lane>>2, t = lane&3; out-of-range entries are zero.  wP/auxP are padded copies.
// ---------------------------------------------------------------------------------------------
__global__ void glm_pack_f64_kernel(const double* __restrict__ theta, const double* __restrict__ base,
                                    const double* __restrict__ w, const double* __restrict__ aux,
                                    int64_t S, int d, int KG, int SB, double2* __restrict__ thetaP,
                                    double2* __restrict__ baseP, double* __restrict__ wP,
                                    double* __restrict__ auxP) {
  const int64_t total = (int64_t)SB * KG * 32;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int lane = (int)(i & 31);
    const int64_t blk = i >> 5;
    const int kg = (int)(blk % KG);
    const int64_t sb = blk / KG;
    const int g = lane >> 2, t = lane & 3;
    {
      const int64_t s = sb * 8 + g;
      const int j = kg * 8 + 2 * t;
      double2 v = make_double2(0.0, 0.0);
      if (s < S) {
        if (j < d) v.x = theta[s * d + j];
        if (j + 1 < d) v.y = theta[s * d + j + 1];
      }
      thetaP[i] = v;
    }
    if (base != nullptr) {
      const int64_t s = sb * 8 + 2 * t;
      const int j = kg * 8 + g;
      double2 v = make_double2(0.0, 0.0);
      if (j < d) {
        if (s < S) v.x = base[s * d + j];
        if (s + 1 < S) v.y = base[(s + 1) * d + j];
      }
      baseP[i] = v;
    }
  }
  const int64_t Sp = (int64_t)SB * 8;
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < Sp;
       s += (int64_t)gridDim.x * blockDim.x) {
    wP[s] = (s < S) ? (w ? w[s] : 1.0) : 0.0;
    auxP[s] = (s < S && aux) ? aux[s] : 1.0;
  }
}

struct SweepArgs {
  const double* X;
  int64_t ldx;
  const double* y;
  int64_t N;
  int d;
  const double2* thetaP;
  const double2* baseP;
  const double* wP;
  const double* auxP;
  int WC;   // number of warp-chunks of 8 * kJN samples (S padded to that)
  int KG;   // ceil(d/8)
  int P;    // shared-memory row pitch of the X tile, in doubles
  int want_grad;
  int64_t numTiles;
  double* ll_part;   // [grid][WC*32]
  double* gmu_part;  // [grid][KG*8]
  double* ge_part;   // [grid][KG*8]
  double* ge_rows;   // [grid][warps][KG*8], per-warp ge rows in global memory when they do not fit on chip (!PRIV)
};

template <int LINK>
__device__ __forceinline__ void link_eval(double z, double yv, double auxv, double& ll, double& r) {
  if (LINK == VB_LINK_LOGISTIC) {
    double dl;
    link_logistic(yv * z, ll, dl);
    r = yv * dl;
  } else if (LINK == VB_LINK_PROBIT) {
    double dl;
    link_probit(yv * z, ll, dl);
    r = yv * dl;
  } else {  // gaussian, aux = 1/sigma_s
    double e = (yv - z) * auxv;
    ll = -0.5 * e * e + log(auxv) - 0.5 * kLog2Pi;
    r = e * auxv;
  }
}

// kJN = 8-sample blocks per warp: 16 warps of 16 samples.  Against 8 warps of 32 samples this is the same operand
// traffic from L2 (every warp still loads only its own slice of theta / E), twice the shared-memory reads of the X tile
// (far from a bound), and FOUR warps per scheduler instead of two: with two, a warp's link epilogue, its shuffles and
// the fixed issue distance between dependent DMMAs left the FP64 tensor pipe idle 39 % of the time
// (profiles/f64_ncu_full_r02.csv: `wait` was the top stall reason).
// PRIV: every warp accumulates ge into its own shared-memory row (plain read-modify-write) instead of atomicAdd on
// one shared row -- a double-precision shared atomic is a compare-and-swap loop, and 16 warps spinning on the same
// 8 addresses per step were ~10 % of the sweep's samples.  Used whenever the rows fit beside the X tile.  Otherwise each
// warp adds into its own row of a global-memory slice (a fire-and-forget RED that stays in L2; one thread per address, so
// the adds land in program order).  Either way the rows are summed in warp order at the end, and the row sums of R
// (rbar) also go through per-warp rows summed in warp order: no sum depends on the order in which warps arrive, so the
// outputs are bitwise reproducible.
constexpr int kJN = 2;
template <int BM, int LINK, bool PRIV>
__global__ void __launch_bounds__(32 * (32 / kJN), 1) glm_sweep_f64_kernel(SweepArgs a) {
  constexpr int MT = BM / 8;
  constexpr int kSweepWarps = 32 / kJN;
  constexpr int kSweepThreads = 32 * kSweepWarps;
  extern __shared__ __align__(16) double smem[];
  const int Dp = a.KG * 8;
  double* Xs = smem;                        // [BM][P]
  double* ys = Xs + (size_t)BM * a.P;       // [BM]
  double* rbar = ys + BM;                   // [BM]
  double* gmu_s = rbar + BM;                // [Dp]
  double* ge_s = gmu_s + Dp;                // [warps][Dp] with PRIV; without, the slot holds rbar_w
  double* rbar_w = PRIV ? ge_s + (size_t)kSweepWarps * Dp : ge_s;   // [warps][BM] per-warp row sums of R
  double* ge_g = PRIV ? nullptr : a.ge_rows + (size_t)blockIdx.x * kSweepWarps * Dp;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;

  for (int j = tid; j < (PRIV ? 1 + kSweepWarps : 1) * Dp; j += kSweepThreads) gmu_s[j] = 0.0;   // gmu_s and ge_s are adjacent
  if (!PRIV && a.want_grad) {
    // ordered before the first RED by the __syncthreads at the top of the first tile
    for (int j = tid; j < kSweepWarps * Dp; j += kSweepThreads) ge_g[j] = 0.0;
  }

  const int numSuper = (a.WC + kSweepWarps - 1) / kSweepWarps;
  const bool vec_ok = ((a.ldx & 1) == 0) && ((reinterpret_cast<uintptr_t>(a.X) & 15) == 0);

  for (int sc = 0; sc < numSuper; ++sc) {
    const int wc = sc * kSweepWarps + warp;
    const bool active = wc < a.WC;
    double llacc[kJN][2];
#pragma unroll
    for (int jn = 0; jn < kJN; ++jn)
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        llacc[jn][c] = 0.0;
      }

    for (int64_t tile = blockIdx.x; tile < a.numTiles; tile += gridDim.x) {
      const int64_t n0 = tile * BM;
      __syncthreads();   // previous tile's readers of Xs / rbar are done
      // ---- stage the X tile (zero padded) ----------------------------------------------
      if (vec_ok) {
        // asynchronous 16-byte copies, zero filled beyond N / d: every copy of the tile is in flight at once, so the
        // HBM latency is paid once per tile (a load -> store loop paid it once per iteration: 11 % of the sweep)
        const int half = a.P >> 1;
        for (int idx = tid; idx < BM * half; idx += kSweepThreads) {
          const int r = idx / half, c2 = idx - r * half;
          const int64_t n = n0 + r;
          const int j = 2 * c2;
          const bool row_ok = n < a.N;
          const uint32_t bytes = (row_ok && j + 1 < a.d) ? 16u : ((row_ok && j < a.d) ? 8u : 0u);
          const double* src = bytes ? a.X + n * a.ldx + j : a.X;
          const uint32_t dst = (uint32_t)__cvta_generic_to_shared(Xs + (size_t)r * a.P + 2 * c2);
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      } else {
        for (int idx = tid; idx < BM * a.P; idx += kSweepThreads) {
          const int r = idx / a.P, c = idx - r * a.P;
          const int64_t n = n0 + r;
          Xs[(size_t)r * a.P + c] = (n < a.N && c < a.d) ? a.X[n * a.ldx + c] : 0.0;
        }
      }
      if (tid < BM) ys[tid] = (n0 + tid < a.N) ? a.y[n0 + tid] : 0.0;
      __syncthreads();

      double acc[MT][kJN][2];
      if (active) {
        // ---- phase A: z = X_tile . theta^T for this warp's 8 * kJN samples -------------
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
          for (int jn = 0; jn < kJN; ++jn) acc[i][jn][0] = acc[i][jn][1] = 0.0;

        const double2* tp = a.thetaP + ((size_t)wc * kJN * a.KG) * 32 + lane;
        const size_t sbStride = (size_t)a.KG * 32;
        double2 bcur[kJN], bnxt[kJN];
#pragma unroll
        for (int jn = 0; jn < kJN; ++jn) bcur[jn] = tp[jn * sbStride];
        for (int kg = 0; kg < a.KG; ++kg) {
          if (kg + 1 < a.KG) {
#pragma unroll
            for (int jn = 0; jn < kJN; ++jn) bnxt[jn] = tp[jn * sbStride + (size_t)(kg + 1) * 32];
          }
          double2 af[MT];
#pragma unroll
          for (int i = 0; i < MT; ++i)
            af[i] = *reinterpret_cast<const double2*>(Xs + (size_t)(8 * i + g) * a.P + 8 * kg + 2 * t);
          // the two k-halves of a tile update the same accumulators: issue all 4 MT tiles of the first half
          // before the second, so that a DMMA never waits for the one issued just before it
#pragma unroll
          for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int jn = 0; jn < kJN; ++jn) dmma884(acc[i][jn][0], acc[i][jn][1], af[i].x, bcur[jn].x);
#pragma unroll
          for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int jn = 0; jn < kJN; ++jn) dmma884(acc[i][jn][0], acc[i][jn][1], af[i].y, bcur[jn].y);
#pragma unroll
          for (int jn = 0; jn < kJN; ++jn) bcur[jn] = bnxt[jn];
        }

        // ---- phase B: link epilogue in registers -----------------------------------------
        // (the per-sample weights are re-read here, L1 hits, rather than held in registers across the tile: phase C
        // needs those registers to keep its DMMA chains interleaved)
        double wv[kJN][2], av[kJN][2];
#pragma unroll
        for (int jn = 0; jn < kJN; ++jn)
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const int s = wc * (8 * kJN) + jn * 8 + 2 * t + c;
            wv[jn][c] = __ldg(a.wP + s);
            av[jn][c] = (LINK == VB_LINK_GAUSSIAN) ? __ldg(a.auxP + s) : 1.0;
          }
        double rsum[MT];
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          const int r = 8 * i + g;
          const double yv = ys[r];
          const double rv = (n0 + r < a.N) ? 1.0 : 0.0;
          double rs = 0.0;
#pragma unroll
          for (int jn = 0; jn < kJN; ++jn)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              double ll, rr;
              link_eval<LINK>(acc[i][jn][c], yv, av[jn][c], ll, rr);
              llacc[jn][c] += ll * rv;
              rr *= wv[jn][c] * rv;
              acc[i][jn][c] = rr;
              rs += rr;
            }
          rsum[i] = rs;
        }
        if (a.want_grad) {
#pragma unroll
          for (int i = 0; i < MT; ++i) {
            double rs = rsum[i];
            rs += __shfl_xor_sync(0xffffffffu, rs, 1);
            rs += __shfl_xor_sync(0xffffffffu, rs, 2);
            if (t == 0) rbar_w[warp * BM + 8 * i + g] = rs;
          }
        }
      }
      if (a.want_grad) {
        __syncthreads();   // rbar_w complete
        if (tid < BM) {
          const int nact = min(kSweepWarps, a.WC - sc * kSweepWarps);
          double v = 0.0;
          for (int w2 = 0; w2 < nact; ++w2) v += rbar_w[w2 * BM + tid];   // fixed order: deterministic
          rbar[tid] = v;
        }
        __syncthreads();   // rbar complete
        // ---- gmu[j] += sum_n X[n,j] rbar[n] -------------------------------------------------
        for (int j = tid; j < Dp; j += kSweepThreads) {
          double s = 0.0;
#pragma unroll 8
          for (int r = 0; r < BM; ++r) s += Xs[(size_t)r * a.P + j] * rbar[r];
          gmu_s[j] += s;
        }
        if (active) {
          // ---- phase C: T = (r.w) E for this warp's samples; ge += colsum(X .* T) -------
          // Software pipelined: the DMMAs of column block jb + 1 are issued BEFORE the reduction of block jb (its
          // dependent X products, three shuffle levels and the shared-memory update), so that chain of latencies
          // runs under tensor work of the same warp instead of in front of it.
          const double2* bp = a.baseP + ((size_t)wc * kJN * a.KG) * 32 + lane;
          const size_t sbStride = (size_t)a.KG * 32;
          double* ge_w = PRIV ? ge_s + (size_t)warp * Dp : ge_s;
          double2 e1[kJN];
          double tc0[MT], tc1[MT], tn0[MT], tn1[MT];
          auto issue = [&](double (&u0)[MT], double (&u1)[MT], const double2 (&e)[kJN]) {
#pragma unroll
            for (int i = 0; i < MT; ++i) u0[i] = u1[i] = 0.0;
            // MT independent accumulation chains, interleaved (a chain's next DMMA is MT instructions away)
#pragma unroll
            for (int jn = 0; jn < kJN; ++jn) {
#pragma unroll
              for (int i = 0; i < MT; ++i) dmma884(u0[i], u1[i], acc[i][jn][0], e[jn].x);
#pragma unroll
              for (int i = 0; i < MT; ++i) dmma884(u0[i], u1[i], acc[i][jn][1], e[jn].y);
            }
          };
#pragma unroll
          for (int jn = 0; jn < kJN; ++jn) e1[jn] = bp[jn * sbStride];
          issue(tc0, tc1, e1);
          if (a.KG > 1) {
#pragma unroll
            for (int jn = 0; jn < kJN; ++jn) e1[jn] = bp[jn * sbStride + 32];
          }
#pragma unroll 2
          for (int jb = 0; jb < a.KG; ++jb) {
            if (jb + 1 < a.KG) issue(tn0, tn1, e1);
            if (jb + 2 < a.KG) {      // the E fragments of block jb + 2 arrive under this block's reduction
#pragma unroll
              for (int jn = 0; jn < kJN; ++jn) e1[jn] = bp[jn * sbStride + (size_t)(jb + 2) * 32];
            }
            double p0 = 0.0, p1 = 0.0;
#pragma unroll
            for (int i = 0; i < MT; ++i) {
              const double2 xv =
                  *reinterpret_cast<const double2*>(Xs + (size_t)(8 * i + g) * a.P + 8 * jb + 2 * t);
              p0 += xv.x * tc0[i];
              p1 += xv.y * tc1[i];
            }
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
              p0 += __shfl_xor_sync(0xffffffffu, p0, o);
              p1 += __shfl_xor_sync(0xffffffffu, p1, o);
            }
            if (g == 0) {
              if (PRIV) {
                double2* q = reinterpret_cast<double2*>(ge_w + 8 * jb) + t;
                double2 v = *q;
                v.x += p0;
                v.y += p1;
                *q = v;
              } else {
                atomicAdd(&ge_g[(size_t)warp * Dp + 8 * jb + 2 * t], p0);
                atomicAdd(&ge_g[(size_t)warp * Dp + 8 * jb + 2 * t + 1], p1);
              }
            }
#pragma unroll
            for (int i = 0; i < MT; ++i) {
              tc0[i] = tn0[i];
              tc1[i] = tn1[i];
            }
          }
        }
      }
    }  // tiles

    // ---- per-CTA log-likelihood partials for this super-chunk ------------------------------
    if (active) {
#pragma unroll
      for (int jn = 0; jn < kJN; ++jn)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          double v = llacc[jn][c];
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
          if (g == 0) a.ll_part[(size_t)blockIdx.x * a.WC * (8 * kJN) + wc * (8 * kJN) + jn * 8 + 2 * t + c] = v;
        }
    }
  }  // super-chunks
  __syncthreads();
  if (a.want_grad) {
    for (int j = tid; j < Dp; j += kSweepThreads) {
      a.gmu_part[(size_t)blockIdx.x * Dp + j] = gmu_s[j];
      double v;
      if (PRIV) {
        v = ge_s[j];
        for (int w2 = 1; w2 < kSweepWarps; ++w2) v += ge_s[(size_t)w2 * Dp + j];      // fixed order: deterministic
      } else {
        v = __ldcg(ge_g + j);                                                          // L2: where the REDs landed
        for (int w2 = 1; w2 < kSweepWarps; ++w2) v += __ldcg(ge_g + (size_t)w2 * Dp + j);
      }
      a.ge_part[(size_t)blockIdx.x * Dp + j] = v;
    }
  }
}

// out[i] = sum_b part[b][i]  (fixed order -> deterministic)
__global__ void reduce_partials_f64_kernel(const double* __restrict__ part, int nblk, int64_t stride,
                                           int64_t n, double* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int b = 0; b < nblk; ++b) s += part[(size_t)b * stride + i];
    out[i] = s;
  }
}

struct SweepPlan {
  int BM, KG, P, WC, SB, priv, grid;
  int64_t numTiles;
  size_t smem;
  size_t off_thetaP, off_baseP, off_wP, off_auxP, off_ll, off_gmu, off_ge, off_ge_rows, total;
};

static bool make_plan(int64_t N, int d, int64_t S, SweepPlan& p) {
  p.KG = (int)ceil_div(d, 8);
  const int Dp = p.KG * 8;
  p.P = (Dp % 16 == 0) ? Dp + 8 : Dp + 16;
  p.WC = (int)ceil_div(S, 8 * kJN);
  p.SB = p.WC * kJN;
  p.BM = 0;
  for (int bm : {32, 16, 8}) {
    size_t bytes = sizeof(double) * ((size_t)bm * p.P + 2 * bm + 2 * (size_t)Dp);
    if (bytes <= 227 * 1024) {
      p.BM = bm;
      p.smem = bytes;
      break;
    }
  }
  if (p.BM == 0) return false;
  {   // per-warp ge rows when they fit beside the tile; the per-warp rbar rows after them, or in the unused ge slot
    const int warps = 32 / kJN;
    const size_t extra = sizeof(double) * ((size_t)(warps - 1) * Dp + (size_t)warps * p.BM);
    p.priv = (p.smem + extra <= 227 * 1024) ? 1 : 0;
    if (p.priv) {
      p.smem += extra;
    } else if (warps * p.BM > Dp) {
      p.smem += sizeof(double) * (size_t)(warps * p.BM - Dp);
      if (p.smem > 227 * 1024) return false;
    }
  }
  p.numTiles = ceil_div(N, p.BM);
  int sms = sm_count();
  p.grid = (int)((p.numTiles < sms) ? (p.numTiles > 0 ? p.numTiles : 1) : sms);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  const size_t packed = (size_t)p.SB * p.KG * 32 * sizeof(double2);
  p.off_thetaP = take(packed);
  p.off_baseP = take(packed);
  p.off_wP = take((size_t)p.SB * 8 * sizeof(double));
  p.off_auxP = take((size_t)p.SB * 8 * sizeof(double));
  p.off_ll = take((size_t)p.grid * p.SB * 8 * sizeof(double));
  p.off_gmu = take((size_t)p.grid * Dp * sizeof(double));
  p.off_ge = take((size_t)p.grid * Dp * sizeof(double));
  p.off_ge_rows = take(p.priv ? 0 : (size_t)p.grid * (32 / kJN) * Dp * sizeof(double));
  p.total = off;
  return true;
}

template <int BM, int LINK, bool PRIV>
static int launch_sweep_priv(const SweepArgs& a, const SweepPlan& p, cudaStream_t stream) {
  auto kern = glm_sweep_f64_kernel<BM, LINK, PRIV>;
  VB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  kern<<<p.grid, 32 * (32 / kJN), p.smem, stream>>>(a);
  VB_CHECK_LAUNCH();
  return VB_OK;
}

template <int BM, int LINK>
static int launch_sweep(const SweepArgs& a, const SweepPlan& p, cudaStream_t stream) {
  return p.priv ? launch_sweep_priv<BM, LINK, true>(a, p, stream) : launch_sweep_priv<BM, LINK, false>(a, p, stream);
}

template <int LINK>
static int launch_sweep_bm(const SweepArgs& a, const SweepPlan& p, cudaStream_t stream) {
  switch (p.BM) {
    case 32: return launch_sweep<32, LINK>(a, p, stream);
    case 16: return launch_sweep<16, LINK>(a, p, stream);
    default: return launch_sweep<8, LINK>(a, p, stream);
  }
}

}  // namespace vb

using namespace vb;

extern "C" size_t vb_glm_sweep_workspace_bytes(int64_t N, int d, int64_t S) {
  SweepPlan p;
  if (N < 0 || d <= 0 || S <= 0 || !make_plan(N, d, S, p)) return 0;
  return p.total;
}

extern "C" int vb_glm_sweep_f64(const double* X, int64_t ldx, const double* y, int64_t N, int d,
                                int link, const double* theta, const double* base, const double* w,
                                const double* aux, int64_t S, int want_grad, double* out_ll,
                                double* out_gmu, double* out_ge, void* workspace,
                                size_t workspace_bytes, cudaStream_t stream) {
  if (N < 0 || d <= 0 || S <= 0 || ldx < d) return set_error(VB_ERR_INVALID_ARG, "glm_sweep: bad shape");
  if (!X || !y || !theta || !out_ll) return set_error(VB_ERR_INVALID_ARG, "glm_sweep: null pointer");
  if (want_grad && (!base || !out_gmu || !out_ge))
    return set_error(VB_ERR_INVALID_ARG, "glm_sweep: want_grad needs base, out_gmu, out_ge");
  if (link == VB_LINK_GAUSSIAN && !aux)
    return set_error(VB_ERR_INVALID_ARG, "glm_sweep: gaussian link needs aux = 1/sigma_s");
  if (link < 0 || link > VB_LINK_GAUSSIAN) return set_error(VB_ERR_INVALID_ARG, "glm_sweep: unknown link");
  SweepPlan p;
  if (!make_plan(N, d, S, p)) return set_error(VB_ERR_UNSUPPORTED, "glm_sweep: d too large for one tile");
  if (!workspace || workspace_bytes < p.total) return set_error(VB_ERR_WORKSPACE, "glm_sweep: workspace too small");
  char* ws = static_cast<char*>(workspace);
  const int Dp = p.KG * 8;

  SweepArgs a;
  a.X = X; a.ldx = ldx; a.y = y; a.N = N; a.d = d;
  a.thetaP = reinterpret_cast<double2*>(ws + p.off_thetaP);
  a.baseP = reinterpret_cast<double2*>(ws + p.off_baseP);
  a.wP = reinterpret_cast<double*>(ws + p.off_wP);
  a.auxP = reinterpret_cast<double*>(ws + p.off_auxP);
  a.WC = p.WC; a.KG = p.KG; a.P = p.P; a.want_grad = want_grad; a.numTiles = p.numTiles;
  a.ll_part = reinterpret_cast<double*>(ws + p.off_ll);
  a.gmu_part = reinterpret_cast<double*>(ws + p.off_gmu);
  a.ge_part = reinterpret_cast<double*>(ws + p.off_ge);
  a.ge_rows = reinterpret_cast<double*>(ws + p.off_ge_rows);

  {
    const int64_t total = (int64_t)p.SB * p.KG * 32;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 4 * sm_count()) blocks = 4 * sm_count();
    glm_pack_f64_kernel<<<blocks, 256, 0, stream>>>(theta, want_grad ? base : nullptr, w, aux, S, d, p.KG,
                                                    p.SB, const_cast<double2*>(a.thetaP),
                                                    const_cast<double2*>(a.baseP),
                                                    const_cast<double*>(a.wP), const_cast<double*>(a.auxP));
    VB_CHECK_LAUNCH();
  }
  if (N == 0) {
    VB_CUDA(cudaMemsetAsync(out_ll, 0, sizeof(double) * S, stream));
    if (want_grad) {
      VB_CUDA(cudaMemsetAsync(out_gmu, 0, sizeof(double) * d, stream));
      VB_CUDA(cudaMemsetAsync(out_ge, 0, sizeof(double) * d, stream));
    }
    return VB_OK;
  }
  int rc;
  switch (link) {
    case VB_LINK_LOGISTIC: rc = launch_sweep_bm<VB_LINK_LOGISTIC>(a, p, stream); break;
    case VB_LINK_PROBIT: rc = launch_sweep_bm<VB_LINK_PROBIT>(a, p, stream); break;
    default: rc = launch_sweep_bm<VB_LINK_GAUSSIAN>(a, p, stream); break;
  }
  if (rc != VB_OK) return rc;
  reduce_partials_f64_kernel<<<(int)ceil_div(S, 256), 256, 0, stream>>>(a.ll_part, p.grid, (int64_t)p.SB * 8, S, out_ll);
  VB_CHECK_LAUNCH();
  if (want_grad) {
    reduce_partials_f64_kernel<<<(int)ceil_div(d, 256), 256, 0, stream>>>(a.gmu_part, p.grid, Dp, d, out_gmu);
    VB_CHECK_LAUNCH();
    reduce_partials_f64_kernel<<<(int)ceil_div(d, 256), 256, 0, stream>>>(a.ge_part, p.grid, Dp, d, out_ge);
    VB_CHECK_LAUNCH();
  }
  return VB_OK;
}
