// Tensor-core "fast path" of the GLM model plugin (logistic link), sm_100a only:
// TMA -> shared memory -> tcgen05.mma (fp16 / e5m2 operands, fp32 accumulators in TMEM).
//
// One kernel, glm_fast_pair_kernel: persistent clusters of two CTAs (cta_group::2), each pair working on a 256-row
// super-tile (two 128-observation tiles) at a time:
//   GEMM1  Z[n,s]  = sum_j Xy[n,j] Theta[s,j]        M=256 (n), N=256 (s), K=d
//          Xy = y*X and Theta are split hi + lo (22-bit operands): one fp16 pass Xh.Th plus the two correction
//          products Xl.Th and Xh.Tl on e5m2 copies with reciprocal power-of-two scales, as kind::f8f6f4 MMAs
//   E1     link epilogue out of TMEM: ll[s] += -softplus(-z), R[n,s] = w_s*sigmoid(-z) -> fp16 tile in
//          shared memory (the N x S logits / residuals never touch HBM), rbar[n] = sum_s R[n,s]
//   GEMM2  Tt[j,n] = sum_s E[s,j] R[n,s]             M=256 (j), N=128 (n), K=256 (s); A = E (MN-major)
//   E2     thread owns j: ge[j] += sum_n Xy[n,j] Tt[j,n],  gmu[j] += sum_n Xy[n,j] rbar[n]
//          (Xy = X_h + X_l8 2^-ax read straight from global memory, an L2 hit)
// Replaces the same reference code as glm_f64.cu (user log_density under autograd:
// models.py:27-39, objectives.py:161-167).  Tolerance of this path: 1e-4 relative (BASELINE.json).
//
// Shared memory per CTA: 10 x 16 KB operand ring, 64 KB R tile, barriers.  TMEM: Z 256 cols, Tt 2 x 128 cols.
//
// HBM layout (chosen for the kernel; X produced once by vb_glm_fast_create, Theta and E rebuilt every sweep):
//   X_h, X_l : fp16 [numTiles][2][d_pad][64]   "tile-transposed": for each 128-row tile and each 64-row half the
//              d_pad x 64 block (column j = one 128-byte row) is contiguous, so GEMM1 reads it as an MN-major
//              A operand (64-element groups, 128-byte swizzle) and E2's column-owning threads read 128-byte runs.
//              X_l only feeds fast_prepare_x8_kernel.
//   X8       : e5m2 [X_l 2^ax | X_h 2^-bx][numTiles][d_pad][128]   one 128-byte row = a tile's 128 rows of column j
//   Th       : fp16 [4][d_pad][64]  Theta_h^T in 64-sample groups (MN-major B operand)
//   T8       : e5m2 [Theta_h 2^-ax | Theta_l 2^bx][2][d_pad][128]  Theta^T in 128-sample groups
//   E        : fp16 [d_pad/64][256][64]  base draws in 64-column groups (MN-major A operand of GEMM2)
// Every operand group is a dense array of 128-byte rows, so ONE multi-dimensional TMA box per pipeline stage and
// operand writes all its groups (the TMA unit is op-rate bound at 4 KB boxes).
// All operands are MN-major with the 128-byte swizzle, so the K extent of a pipeline stage is free:
// GEMM1 streams K = 32 per stage (16 KB for X, 16 KB for Theta).
#include <cuda.h>
#include <cuda_fp16.h>

#include <cstring>
#include <mutex>

#include "common.cuh"
#include "fast_internal.cuh"

namespace vb {
namespace fast {

constexpr int kBM = 128;
constexpr int kSP = 256;                 // padded sample count (UMMA N of GEMM1, K of GEMM2)
constexpr int kSlotBytes = 16384;
constexpr int kNumSlots = 10;
constexpr int kRingBytes = kSlotBytes * kNumSlots;      // 163840
constexpr int kRBytes = kBM * kSP * 2;                  // 65536
constexpr int kMiscBytes = 3072;
constexpr int kSmemBytes = kRingBytes + kRBytes + kMiscBytes;   // 232448 = 227 KB
constexpr uint32_t kTmemCols = 512;

// ---- PTX wrappers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar_cluster) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(bar_cluster)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                                 uint32_t bar_cluster) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar_cluster)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// ---- cluster / CTA-pair helpers (cta_group::2) ---------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same variable in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cl(uint32_t bar, uint32_t parity) {      // acquire at cluster scope
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
// long waits (thousands of cycles): back off so that the spinning warp leaves the issue slots to the epilogue warps
__device__ __forceinline__ void mbar_wait_cl_sleep(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t done;
  for (;;) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(ns);
  }
}
__device__ __forceinline__ void st_cluster_f32(uint32_t cluster_addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(cluster_addr), "f"(v) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 8-bit float operands (e4m3 / e5m2 per the instruction descriptor), K = 32 per instruction, fp32 accumulate
__device__ __forceinline__ void umma_f8_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at the same shared-memory offset in both CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(mask)
               : "memory");
}

// 32 lanes x 32 columns of 32-bit accumulators -> 32 registers per thread
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- descriptors -------------------------------------------------------------------------------
// shared-memory matrix descriptor, 128-byte swizzle (layout_type = 2), descriptor version 1
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;     // version
  d |= (uint64_t)2 << 61;     // SWIZZLE_128B
  return d;
}
// instruction descriptor: f16 x f16 -> f32
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) /*c=f32*/ | (0u << 7) /*a=f16*/ | (0u << 10) /*b=f16*/ | ((uint32_t)a_mn_major << 15) |
         ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// instruction descriptor: e5m2 x e5m2 -> f32 (kind::f8f6f4; a_format / b_format: 0 = e4m3, 1 = e5m2)
__host__ __device__ constexpr uint32_t make_idesc8(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) /*c=f32*/ | (1u << 7) /*a=e5m2*/ | (1u << 10) /*b=e5m2*/ | ((uint32_t)a_mn_major << 15) |
         ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

struct Params {
  int64_t N;
  int d_pad;       // multiple of 128
  int S;           // valid samples (<= 256)
  int numTiles;
  int want_grad;
  int ll_total_only;  // 1: only sum_s ll[s] is needed (plain ExclusiveKL value): skip the per-sample column sums
  const float* w;  // [256] sample weights, 0 beyond S
  double* ll_part;   // [grid][256]
  double* gmu_part;  // [grid][d_pad]
  double* ge_part;   // [grid][d_pad]
  long long* tim;    // optional: clock64 timestamps of CTA 0
  int uniform_w;     // 1: every valid sample has weight 1 (w == NULL on the host side)
  const __half* Xh;  // E2 reads its X rows from global memory
  float xl_scale;      // 2^-ax
  const uint8_t* Xl8;  // e5m2 of X_l * 2^ax, [tile][d_pad][128 n]
};

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// =================================================================================================
// The sweep kernel (cta_group::2): two CTAs of a cluster work on a 256-row super-tile.
//   GEMM1  M = 256 (rank r owns rows 128r..128r+127), N = 256: each CTA stages only HALF of Theta^T per K stage
//   GEMM2  M = 256 j (rank r owns j-block r of the 256-j pair block), N = 128 tile rows (64 from each CTA's R tile),
//          two such units (tile-row halves) per group; each CTA stages only its half of E, one 16 KB slot per
//          64 samples, released as soon as both units have consumed it
//   E2     reads its X values straight from global memory / L2 (256-bit evict-first loads; a thread owns column j,
//          whose 64 rows of a tile half are one contiguous 128-byte run in the tile-transposed layout), so the
//          operand ring only carries tensor-core operands
// Pairing the CTAs takes the operand fills per 128 rows from 1280 KB (one CTA per tile, bound by the per-SM fill rate)
// to 896 KB at d = 512, 640 KB of them through TMA.  GEMM2 of super-tile i-1 is interleaved with GEMM1 of super-tile i (the
// R tile of i-1 stays valid until E1 of i starts, which is after every MMA issued before Z(i) was committed), so
// the tensor pipe only idles during E1; one pool of 16 epilogue warps runs E2 of i-1 and then E1 of i.
// Warps: 0 producer, 1 MMA (rank 0 issues for the pair), 2..17 epilogue (E2 of super-tile i-1, then E1 of i).
constexpr int kThreadsP = 64 + 32 * 8 + 32 * 8;      // 576
constexpr int kFullRing = 8;

struct MiscP {
  uint64_t empty[kNumSlots];
  uint64_t g1_full[kFullRing];        // leader: bytes of both CTAs' halves of a GEMM1 stage
  uint64_t e_full[16];                // leader: both CTAs' halves of one 64-sample slice of E (ring > slices in flight)
  uint64_t z_full;                    // local, multicast commit
  uint64_t r_full;                    // leader, count 2: both R tiles written, both Z read
  uint64_t rb_full;                   // local, count 2: rb[] written by both CTAs
  uint64_t t_full;                    // local, multicast commit: both units of a group
  uint64_t t_empty;                   // leader, count 2
  uint32_t tmem_base;
  uint32_t pad;
  alignas(16) float rbar[kBM];        // E1: row sums of R over sample quarter 1 (fixed-order sum, see E1)
  alignas(16) float rb[2][2 * kBM];   // [iteration parity][row of the super-tile]: sum_s R[n,s]
};
static_assert(sizeof(MiscP) <= kMiscBytes, "misc smem overflow");

__device__ __forceinline__ void epi1_barrier() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
__device__ __forceinline__ void ldg256(const void* ptr, uint32_t* r) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "l"(ptr));
}


__device__ __forceinline__ float fast_lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Link epilogue of 32 accumulator columns held by one thread (one tile row), staged so that the 16 independent
// MUFU chains of a half-chunk are in flight together (the compiler keeps the order of these loops).
//   in : v[i] = z (margin y * x.theta)
//   out: packed = fp16 pairs of r = w * sigmoid(-z) (rows beyond N give 0), v[i] = softplus(-z) when KEEP_SP,
//        spsum += sum_i softplus(-z_i), rsum += sum_i r_i
// PLAIN: all rows valid and all weights 1 -> no masking.
template <bool PLAIN, bool KEEP_SP>
__device__ __forceinline__ void link_chunk(float (&v)[32], uint32_t (&packed)[16], float& spsum, float& rsum, float wl,
                                           float rowvalid) {
  float lgsum = 0.0f, mxsum = 0.0f, rs = 0.0f;
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    float t[16], lg[16], ri[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) t[i] = fast_exp2(-fabsf(v[16 * hh + i]) * 1.4426950408889634f);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float den = 1.0f + t[i];
      lg[i] = fast_lg2(den);
      ri[i] = fast_rcp(den);
    }
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
      float r2[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float a = v[16 * hh + i + u];
        const float mx = fmaxf(-a, 0.0f);
        float r = (a >= 0.0f ? t[i + u] : 1.0f) * ri[i + u];              // sigmoid(-a)
        if (!PLAIN) r *= __shfl_sync(0xffffffffu, wl, 16 * hh + i + u) * rowvalid;
        if (KEEP_SP) v[16 * hh + i + u] = PLAIN ? fmaf(lg[i + u], 0.6931471805599453f, mx)
                                                : fmaf(lg[i + u], 0.6931471805599453f, mx) * rowvalid;
        lgsum += lg[i + u];
        mxsum += mx;
        rs += r;
        r2[u] = r;
      }
      const __half2 h2 = __floats2half2_rn(r2[0], r2[1]);
      packed[(16 * hh + i) >> 1] = *reinterpret_cast<const uint32_t*>(&h2);
    }
  }
  const float sp = fmaf(lgsum, 0.6931471805599453f, mxsum);
  spsum += PLAIN ? sp : sp * rowvalid;
  rsum += rs;
}

// PLAIN link epilogue when only sum softplus is needed (plain ExclusiveKL): the 32 logs become two -- log2 of the running
// product of 1 + t over 16 elements (each factor in [1, 2], so the product stays below 2^16) -- which takes the MUFU
// work of E1 from 3 to 2 operations per element (E1 is MUFU bound: 16 per clock per SM).
__device__ __forceinline__ void link_chunk_total(float (&v)[32], uint32_t (&packed)[16], float& spsum, float& rsum) {
  float lgsum = 0.0f, mxsum = 0.0f, rs = 0.0f;
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    float t[16], ri[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) t[i] = fast_exp2(-fabsf(v[16 * hh + i]) * 1.4426950408889634f);
    float prod0 = 1.0f, prod1 = 1.0f;
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
      const float d0 = 1.0f + t[i], d1 = 1.0f + t[i + 1];
      ri[i] = fast_rcp(d0);
      ri[i + 1] = fast_rcp(d1);
      prod0 *= d0;
      prod1 *= d1;
    }
    lgsum += fast_lg2(prod0 * prod1);
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
      float r2[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float a = v[16 * hh + i + u];
        mxsum += fmaxf(-a, 0.0f);
        const float r = (a >= 0.0f ? t[i + u] : 1.0f) * ri[i + u];        // sigmoid(-a)
        rs += r;
        r2[u] = r;
      }
      const __half2 h2 = __floats2half2_rn(r2[0], r2[1]);
      packed[(16 * hh + i) >> 1] = *reinterpret_cast<const uint32_t*>(&h2);
    }
  }
  spsum += fmaf(lgsum, 0.6931471805599453f, mxsum);
  rsum += rs;
}

// Fill sequence of iteration i (identical in every role and in both CTAs; `fill` counts 16 KB slots):
//   for kc in 0..KC-1:  slot A = X_h (2 halves, 8 KB) | X_l8 | X_h8 (4 KB each: 32 j-rows x 128 n bytes),
//                       slot B = Theta_h (2 groups, 8 KB) | Theta_h8 | Theta_l8 (this CTA's 128 samples)
//       after the stages with (kc & 7) == 1 (and i > 0): the 4 E slots of GEMM2 group jbp = kc >> 3 of super-tile i-1,
//       consumed after stage (kc & 7) == 3
//   a last iteration i = nIter only carries the GEMM2 groups of the final super-tile.
// The two CORRECTION passes of GEMM1 run on e5m2 copies with reciprocal power-of-two scales
// (tools/emulate_fp8_scheme.py), (X_l 2^ax)(Theta_h 2^-ax) and (X_h 2^-bx)(Theta_l 2^bx), as kind::f8f6f4 (K = 32 per
// instruction, twice the fp16 rate): their terms are 2^-11 of the product, so 3 significant bits per operand leave
// 2^-13 overall -- GEMM1 costs 1 + 1/2 + 1/2 fp16 pass units instead of 3.  E2 takes its X as X_h + X_l8 2^-ax
// (3 bytes per element from L2 instead of 4).
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsP, 1)
glm_fast_pair_kernel(const __grid_constant__ CUtensorMap tmX,      // 4-D [tile][half][j][64 n] (X_h)
                     const __grid_constant__ CUtensorMap tmT,      // 3-D [group][j][64 s] (Theta_h)
                     const __grid_constant__ CUtensorMap tmE,      // 3-D: [j group][s][64 j]
                     const __grid_constant__ CUtensorMap tmX8,     // 4-D [X_l8|X_h8][tile][j][128 n] bytes
                     const __grid_constant__ CUtensorMap tmT8,     // 4-D [Theta_h8|Theta_l8][group][j][128 s] bytes
                     Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;
  uint8_t* rtile = smem + kRingBytes;
  MiscP* misc = reinterpret_cast<MiscP*>(smem + kRingBytes + kRBytes);
  const uint32_t ring_u = smem_u32(ring), rtile_u = smem_u32(rtile);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int numSuper = (p.numTiles + 1) >> 1;
  const int nIter = cluster_id < numSuper ? (numSuper - cluster_id + num_clusters - 1) / num_clusters : 0;
  const int KC = p.d_pad / 32, JBP = p.d_pad / 256;      // KC = 8 JBP
  const bool grad = p.want_grad != 0;
  double ll_acc[2] = {0.0, 0.0};                // epilogue warps: column sums of softplus
  double ge_acc[8], gmu_acc[8];                 // epilogue warps: gradient partials of column j per 256-column block
#pragma unroll
  for (int i = 0; i < 8; ++i) ge_acc[i] = gmu_acc[i] = 0.0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kNumSlots; ++i) mbar_init(smem_u32(&misc->empty[i]), 1);
    for (int i = 0; i < kFullRing; ++i) mbar_init(smem_u32(&misc->g1_full[i]), 1);
    for (int i = 0; i < 16; ++i) mbar_init(smem_u32(&misc->e_full[i]), 1);
    mbar_init(smem_u32(&misc->z_full), 1);
    mbar_init(smem_u32(&misc->r_full), 2);
    mbar_init(smem_u32(&misc->rb_full), 2);
    mbar_init(smem_u32(&misc->t_full), 1);
    mbar_init(smem_u32(&misc->t_empty), 2);
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&misc->tmem_base)),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                      // barriers of both CTAs initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem = misc->tmem_base;
  PDL_SYNC();                              // everything above overlapped the previous kernel; global memory from here on

  if (warp == 0) {
    // ================================ TMA producer (both CTAs) ================================
    if (lane == 0) {
      prefetch_tmap(&tmX); prefetch_tmap(&tmT); prefetch_tmap(&tmE);
      prefetch_tmap(&tmX8); prefetch_tmap(&tmT8);
      uint32_t fill = 0, sc = 0, ec = 0;
      auto acquire = [&]() -> uint32_t {
        const uint32_t slot = fill % kNumSlots, par = (fill / kNumSlots) & 1;
        mbar_wait_cl_sleep(smem_u32(&misc->empty[slot]), par ^ 1, 32);
        ++fill;
        return ring_u + slot * kSlotBytes;
      };
      auto g2_fills = [&](int jbp) {
        const int j0 = jbp * 256 + (int)rank * 128;                 // this CTA's 128 columns of the pair block
        for (int g = 0; g < 4; ++g, ++ec) {
          const uint32_t ebar_l = smem_u32(&misc->e_full[ec & 15]);
          if (leader) mbar_expect_tx(ebar_l, 2 * kSlotBytes);
          const uint32_t ebar = mapa_u32(ebar_l, 0);
          const uint32_t dst = acquire();
          tma_load_3d_pair(dst, &tmE, 0, 64 * g, j0 >> 6, ebar);           // 64 samples x (2 x 64 columns): 16 KB
        }
      };
      for (int it = 0; it <= nIter; ++it) {
        const int sup = cluster_id + it * num_clusters;
        if (it < nIter) {
          const int tile = 2 * sup + (int)rank;                     // this CTA's 128 rows
          for (int kc = 0; kc < KC; ++kc, ++sc) {
            const int j0 = kc * 32;
            const uint32_t bar_l = smem_u32(&misc->g1_full[sc % kFullRing]);
            if (leader) mbar_expect_tx(bar_l, 4 * kSlotBytes);
            const uint32_t bar = mapa_u32(bar_l, 0);
            uint32_t dst = acquire();
            tma_load_4d_pair(dst, &tmX, 0, j0, 0, tile, bar);            // X_h n0 | n1: 8 KB
            tma_load_4d_pair(dst + 8192, &tmX8, 0, j0, tile, 0, bar);    // X_l8 | X_h8: 2 x 4 KB
            dst = acquire();
            tma_load_3d_pair(dst, &tmT, 0, j0, 2 * (int)rank, bar);      // Theta_h g0 | g1 (this CTA's half): 8 KB
            tma_load_4d_pair(dst + 8192, &tmT8, 0, j0, (int)rank, 0, bar);   // Theta_h8 | Theta_l8 of its 128 samples
            if (grad && it > 0 && (kc & 7) == 1) g2_fills(kc >> 3);     // two stages ahead of the group that consumes them
          }
        } else if (grad && it > 0) {
          for (int jbp = 0; jbp < JBP; ++jbp) g2_fills(jbp);
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer: rank 0 only ================================
    if (leader) {
      constexpr uint32_t idesc1 = make_idesc(256, 256, 1, 1);
      constexpr uint32_t idesc2 = make_idesc(256, 128, 1, 0);
      uint32_t fill = 0, sc = 0, ec = 0, gc = 0;
      long long w_g1 = 0, w_e = 0, w_t = 0;
      const bool timing = p.tim && blockIdx.x == 0;
      uint32_t e_base = 0;                  // first of the 4 ring slots holding the E slices of the pending group
      auto g2_group = [&]() {
        long long c0 = timing ? clock64() : 0;
        mbar_wait_cl(smem_u32(&misc->t_empty), (gc & 1) ^ 1);      // both CTAs' E2 have drained the previous group
        if (timing) w_t += clock64() - c0;
        ++gc;
        for (int g = 0; g < 4; ++g, ++ec) {
          const uint32_t slot = (e_base + g) % kNumSlots;
          c0 = timing ? clock64() : 0;
          mbar_wait_cl(smem_u32(&misc->e_full[ec & 15]), (ec >> 4) & 1);
          if (timing) w_e += clock64() - c0;
          tc_fence_after();
          if (elect_one()) {
            const uint32_t es = ring_u + slot * kSlotBytes;
#pragma unroll
            for (int nh = 0; nh < 2; ++nh) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_f16_pair(tmem + 256 + 128 * nh, make_desc(es + k * 2048, 8192, 1024),
                              make_desc(rtile_u + g * 16384 + nh * 8192 + k * 32, 16, 1024), idesc2, (g | k) ? 1u : 0u);
            }
            umma_commit_pair(smem_u32(&misc->empty[slot]));
            if (g == 3) umma_commit_pair(smem_u32(&misc->t_full));
          }
          __syncwarp();
        }
      };
      for (int it = 0; it <= nIter; ++it) {
        if (timing && it < 8 && lane == 0) p.tim[it * 16 + 0] = clock64();
        if (it > 0) {                    // Z(it-1) read and R(it-1) written by both CTAs
          mbar_wait_cl_sleep(smem_u32(&misc->r_full), (it - 1) & 1, 64);
          tc_fence_after();
        }
        if (timing && it < 8 && lane == 0) p.tim[it * 16 + 1] = clock64();
        if (it < nIter) {
          for (int kc = 0; kc < KC; ++kc, ++sc) {
            const uint32_t sa = fill % kNumSlots, sb = (fill + 1) % kNumSlots;
            fill += 2;
            const uint32_t ax = ring_u + sa * kSlotBytes, bh = ring_u + sb * kSlotBytes;
            const long long c0 = timing ? clock64() : 0;
            mbar_wait_cl(smem_u32(&misc->g1_full[sc % kFullRing]), (sc / kFullRing) & 1);
            if (timing) w_g1 += clock64() - c0;
            tc_fence_after();
            if (elect_one()) {
              constexpr uint32_t idesc8 = make_idesc8(256, 256, 1, 1);
#pragma unroll
              for (int k = 0; k < 2; ++k)                 // X_h . Theta_h, fp16, K = 16 each
                umma_f16_pair(tmem, make_desc(ax + k * 2048, 4096, 1024), make_desc(bh + k * 2048, 4096, 1024), idesc1,
                              (kc | k) ? 1u : 0u);
              // corrections, e5m2, K = 32: one 128-byte row holds all 128 rows / samples of this CTA (a single MN group)
              umma_f8_pair(tmem, make_desc(ax + 8192, 4096, 1024), make_desc(bh + 8192, 4096, 1024), idesc8, 1u);     // X_l8 . Theta_h8
              umma_f8_pair(tmem, make_desc(ax + 12288, 4096, 1024), make_desc(bh + 12288, 4096, 1024), idesc8, 1u);   // X_h8 . Theta_l8
              umma_commit_pair(smem_u32(&misc->empty[sa]));
              umma_commit_pair(smem_u32(&misc->empty[sb]));
              if (kc == KC - 1) umma_commit_pair(smem_u32(&misc->z_full));
            }
            __syncwarp();
            if (grad && it > 0 && (kc & 7) == 1) {      // the E slices were filled here, two stages ahead
              e_base = fill;
              fill += 4;
            }
            if (grad && it > 0 && (kc & 7) == 3) g2_group();
          }
        } else if (grad && it > 0) {
          for (int jbp = 0; jbp < JBP; ++jbp) {
            e_base = fill;
            fill += 4;
            g2_group();
          }
        }
        if (timing && it < 8 && lane == 0) {
          p.tim[it * 16 + 2] = clock64();
          p.tim[it * 16 + 3] = w_g1;
          p.tim[it * 16 + 4] = w_e;
          p.tim[it * 16 + 5] = w_t;
        }
        w_g1 = w_e = w_t = 0;
      }
    }
  } else {
    // ================================ epilogue warps (16): E2 of super-tile it-1, then E1 of super-tile it ==========
    // The two jobs never overlap in time for long (E2 groups arrive while GEMM1 streams, E1 starts when Z is
    // complete and the tensor pipe idles until E1 is done), so one pool of warps does both at full width.
    const int ew = warp - 2;
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int k = ew >> 2;             // E1: sample-column quarter;  E2: (tile t, tile-row half nh)
    const int row = 32 * q + lane;     // TMEM lane = row of this CTA's tile (E1) / column j of its block (E2)
    const uint32_t lane_addr = tmem + ((uint32_t)(32 * q) << 16);
    const uint32_t r_full_leader = mapa_u32(smem_u32(&misc->r_full), 0);
    const uint32_t t_empty_leader = mapa_u32(smem_u32(&misc->t_empty), 0);
    const uint32_t rbf_own = mapa_u32(smem_u32(&misc->rb_full), rank), rbf_peer = mapa_u32(smem_u32(&misc->rb_full), rank ^ 1);
    const bool tthread = p.tim && blockIdx.x == 0 && threadIdx.x == 64;
    const int t2 = k & 1, nh2 = k >> 1;
    const size_t tstride = (size_t)p.d_pad * kBM;
    uint32_t gc = 0;
    long long w_tf = 0, busy = 0;

    auto e2_group = [&](int itp, int jbp) {      // GEMM2 group jbp of iteration itp: this warp's 64 tile rows
      const int sup = cluster_id + itp * num_clusters;
      const int j = jbp * 256 + 128 * (int)rank + row;
      // this thread's X values: column j, the 64 rows of half nh2 of tile t2 (128 contiguous bytes of X_h, 64 of X_l8)
      const __half* xhp = p.Xh + ((size_t)((2 * sup + t2) * 2 + nh2) * p.d_pad + j) * 64;
      uint32_t xa[32], xb[32];                   // [0,16): hi, [16,24): 32 e5m2 bytes of lo, of a 32-row step
      ldg256(xhp, xa);                           // X does not depend on the MMA: in flight while waiting
      ldg256(xhp + 16, xa + 8);
      ldg256(xhp + 32, xb);
      ldg256(xhp + 48, xb + 8);
      const uint8_t* xl8 = p.Xl8 + ((size_t)(2 * sup + t2) * p.d_pad + j) * 128 + 64 * nh2;
      ldg256(xl8, xa + 16);
      ldg256(xl8 + 32, xb + 16);
      float ge = 0.0f, gm = 0.0f;
      auto compute = [&](const uint32_t* x, int part) {
        const float* rbp = &misc->rb[itp & 1][128 * t2 + 64 * nh2 + 32 * part];
        float tv[32];
        tmem_ld32(lane_addr + 256 + 128 * nh2 + 64 * t2 + 32 * part, tv);
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          const float2 fh2 = __half22float2(*reinterpret_cast<const __half2*>(&x[e]));
          // an e5m2 byte is the high byte of the fp16 with the same value: spread two bytes into an fp16 pair
          const uint32_t h2 = __byte_perm(x[16 + (e >> 1)], 0u, (e & 1) ? 0x3424u : 0x1404u);
          const float2 fl2 = __half22float2(*reinterpret_cast<const __half2*>(&h2));
          const float x0 = fmaf(fl2.x, p.xl_scale, fh2.x);
          const float x1 = fmaf(fl2.y, p.xl_scale, fh2.y);
          const float2 rb2 = *reinterpret_cast<const float2*>(rbp + 2 * e);
          ge = fmaf(x0, tv[2 * e], ge);
          ge = fmaf(x1, tv[2 * e + 1], ge);
          gm = fmaf(x0, rb2.x, gm);
          gm = fmaf(x1, rb2.y, gm);
        }
      };
      const long long c1 = tthread ? clock64() : 0;
      mbar_wait_cl_sleep(smem_u32(&misc->t_full), gc & 1, 64);
      ++gc;
      const long long c2 = tthread ? clock64() : 0;
      w_tf += c2 - c1;
      tc_fence_after();
      if (tthread && itp < 8 && jbp == 0) p.tim[itp * 16 + 10] = c2;
      compute(xa, 0);
      compute(xb, 1);
      tc_fence_before();
      epi1_barrier();
      if (tthread) busy += clock64() - c2;
      if (threadIdx.x == 64) mbar_arrive_cluster(t_empty_leader);
      ge_acc[jbp & 7] += (double)ge;
      gmu_acc[jbp & 7] += (double)gm;
    };

    for (int it = 0; it <= nIter; ++it) {
      // ---------------- E2 of the previous super-tile ----------------
      if (grad && it > 0) {
        mbar_wait_cl_sleep(smem_u32(&misc->rb_full), (it - 1) & 1, 64);      // rb[(it-1)&1] complete (both CTAs)
        for (int jbp = 0; jbp < JBP; ++jbp) e2_group(it - 1, jbp);
        if (tthread && it < 8) {
          p.tim[it * 16 + 12] = w_tf;
          p.tim[it * 16 + 13] = busy;
        }
        w_tf = busy = 0;
      }
      if (it == nIter) break;
      // ---------------- E1: link epilogue on Z ----------------
      const int sup = cluster_id + it * num_clusters;
      const int64_t n = ((int64_t)2 * sup + rank) * kBM + row;
      const float rowvalid = n < p.N ? 1.0f : 0.0f;
      mbar_wait_cl_sleep(smem_u32(&misc->z_full), it & 1, 32);
      tc_fence_after();
      if (tthread && it < 8) p.tim[it * 16 + 8] = clock64();
      float rsum = 0.0f, lls0 = 0.0f, lls1 = 0.0f;
      // plain: every row of the tile is a real observation and every sample of this column quarter has weight 1
      // (the common case: ExclusiveKL away from the last tile) -> no per-element masking / weighting
      const bool plain = p.uniform_w && (64 * k + 64 <= p.S) && (((int64_t)2 * sup + rank) * kBM + kBM <= p.N);
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        const int col0 = 64 * k + 32 * c;
        float v[32];
        tmem_ld32(lane_addr + col0, v);
        uint32_t packed[16];
        float spsum = 0.0f;
        if (plain) {
          if (p.ll_total_only) link_chunk_total(v, packed, spsum, rsum);
          else link_chunk<true, true>(v, packed, spsum, rsum, 1.0f, 1.0f);
        } else {
          const float wl = __ldg(p.w + col0 + lane);                       // lane i holds the weight of column col0 + i
          if (p.ll_total_only) link_chunk<false, false>(v, packed, spsum, rsum, wl, rowvalid);
          else link_chunk<false, true>(v, packed, spsum, rsum, wl, rowvalid);
        }
        {   // R tile: K-group k (64 samples, 16 KB), row-major 128-byte rows, 128-byte swizzle
          uint8_t* rowp = rtile + k * 16384 + row * 128;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int chunk = (4 * c + u) ^ (row & 7);
            *reinterpret_cast<uint4*>(rowp + chunk * 16) =
                make_uint4(packed[4 * u], packed[4 * u + 1], packed[4 * u + 2], packed[4 * u + 3]);
          }
        }
        if (p.ll_total_only) {
          lls0 += spsum;
        } else {
          // column sums of softplus over this warp's 32 rows (transpose-reduce): lane l ends with column l
#pragma unroll
          for (int o = 16, cnt = 16; o >= 1; o >>= 1, cnt >>= 1) {
            const bool up = (lane & o) != 0;
#pragma unroll
            for (int i = 0; i < cnt; ++i) {
              const float send = up ? v[i] : v[i + cnt];
              const float keep = up ? v[i + cnt] : v[i];
              v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
          }
          lls0 += c == 0 ? v[0] : 0.0f;            // static registers: a dynamically indexed array would live in local memory
          lls1 += c == 1 ? v[0] : 0.0f;
        }
      }
      ll_acc[0] += (double)lls0;
      ll_acc[1] += (double)lls1;
      if (tthread && it < 8) p.tim[it * 16 + 6] = clock64();
      float* rbl = &misc->rb[it & 1][128 * rank + row];
      fence_proxy_async();       // R tile writes -> visible to the tensor core (async proxy)
      tc_fence_before();
      epi1_barrier();
      // Z has been read and R written by this CTA: the leader may start the next GEMM1 (critical path) ...
      if (threadIdx.x == 64) mbar_arrive_cluster(r_full_leader);
      if (tthread && it < 8) p.tim[it * 16 + 7] = clock64();
      // ... while the row sums go into BOTH CTAs' rb (E2 of either CTA sweeps all 256 rows; needed later).
      // Row sums of R over the four sample quarters in a fixed order, so that a sweep is reproducible bit for bit.
      // Scratch for the partials of quarters 1..3: rbar and the other parity of rb.  Nothing reads that parity before
      // E2 of super-tile it + 1, and the peer writes it only after its E2 of super-tile it, which waits for rb_full below.
      if (grad) {
        float* other = misc->rb[(it + 1) & 1];
        if (k != 0) (k == 1 ? misc->rbar : other + 128 * (k - 2))[row] = rsum;
        epi1_barrier();
        if (k == 0) {
          const float s = ((rsum + misc->rbar[row]) + other[row]) + other[128 + row];
          *rbl = s;
          st_cluster_f32(mapa_u32(smem_u32(rbl), rank ^ 1), s);
        }
        epi1_barrier();          // CTA-scope ordering of the stores before the (cumulative) cluster-scope release below
        if (threadIdx.x == 64) {
          mbar_arrive_cluster(rbf_own);
          mbar_arrive_cluster(rbf_peer);
        }
      }
      if (tthread && it < 8) p.tim[it * 16 + 9] = clock64();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp >= 2) {
    // -------- per-CTA partials (every MMA has completed: the R tile is free scratch) --------
    const int ew = warp - 2, q = warp & 3, k = ew >> 2;
    const int row = 32 * q + lane;
    double (*red)[kBM] = reinterpret_cast<double (*)[kBM]>(rtile);       // [4][128] doubles
    if (p.ll_total_only) {
      double tot = ll_acc[0];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
      if (lane == 0) red[0][ew] = tot;
      epi1_barrier();
      double sum = 0.0;
      for (int i = 0; i < 16; ++i) sum += red[0][i];
      // padded sample columns (theta = 0) each contributed softplus(0) = ln2 (as computed in fp32) per valid row
      int64_t rows = 0;
      for (int it = 0; it < nIter; ++it) {
        const int64_t left = p.N - ((int64_t)2 * (cluster_id + it * num_clusters) + rank) * kBM;
        rows += left <= 0 ? 0 : (left < kBM ? left : kBM);
      }
      sum -= (double)(kSP - p.S) * (double)rows * (double)(1.0f * 0.6931471805599453f);
      if (threadIdx.x - 64 < kSP) p.ll_part[(size_t)blockIdx.x * kSP + (threadIdx.x - 64)] = sum / (double)p.S;
    } else {
      // lane l of (q,k) holds column 64k + 32c + l summed over the rows of quarter q -> sum the 4 quarters
      for (int c = 0; c < 2; ++c) {
        epi1_barrier();
        if (q != 0) red[k][(q - 1) * 32 + lane] = ll_acc[c];
        epi1_barrier();
        if (q == 0) {
          const double sum = ll_acc[c] + red[k][lane] + red[k][32 + lane] + red[k][64 + lane];
          p.ll_part[(size_t)blockIdx.x * kSP + 64 * k + 32 * c + lane] = sum;
        }
      }
    }
    if (grad) {
      // the four warps that share a lane quarter swept different tile rows of the same columns j
      for (int jbp = 0; jbp < JBP; ++jbp) {
        for (int which = 0; which < 2; ++which) {
          epi1_barrier();
          if (k != 0) red[k][row] = which ? gmu_acc[jbp & 7] : ge_acc[jbp & 7];
          epi1_barrier();
          if (k == 0) {
            const double sum = (which ? gmu_acc[jbp & 7] : ge_acc[jbp & 7]) + red[1][row] + red[2][row] + red[3][row];
            const size_t o = (size_t)cluster_id * p.d_pad + jbp * 256 + 128 * rank + row;
            (which ? p.gmu_part : p.ge_part)[o] = sum;
          }
        }
      }
    }
  }
  cluster_sync_all();                      // no CTA leaves while its pair may still touch its shared memory / TMEM
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
  }
}

// ---- operand preparation ------------------------------------------------------------------------
// Xy = y*X split into fp16 hi + lo, written tile-transposed: Xt[((tile*2 + half)*d_pad + j)*64 + (n % 64)]
__global__ void fast_prepare_x_kernel(const double* __restrict__ X, int64_t ldx, const double* __restrict__ y, int64_t N,
                                      int d, int64_t numTiles, int d_pad, __half* __restrict__ Xh, __half* __restrict__ Xl,
                                      float* __restrict__ absmax) {
  __shared__ float tile[32][33];
  float mx = 0.0f;
  double sq = 0.0;                         // sum of squares: the typical magnitude sets the fp8 operand scales
  // 32 x 32 transposes: coalesced reads along j, coalesced writes along n
  const int64_t blocksPerTile = (int64_t)(d_pad / 32) * 4;
  const int64_t total = numTiles * blocksPerTile;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;        // 32 x 8 threads
  for (int64_t b = blockIdx.x; b < total; b += gridDim.x) {
    const int64_t t = b / blocksPerTile;
    const int rem = (int)(b - t * blocksPerTile);
    const int jblk = rem >> 2, nblk = rem & 3;
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
      const int64_t n = t * 128 + nblk * 32 + r;
      const int j = jblk * 32 + tx;
      float v = 0.0f;
      if (n < N && j < d) v = (float)(X[n * ldx + j] * y[n]);
      tile[r][tx] = v;
      mx = fmaxf(mx, v == v ? fabsf(v) : INFINITY);      // NaN counts as out of range (fmaxf would drop it)
      sq += (double)v * (double)v;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
      const int j = jblk * 32 + r;
      const float v = tile[tx][r];
      const __half hi = __float2half_rn(v);
      const size_t o = (((size_t)t * 2 + (nblk >> 1)) * d_pad + j) * 64 + (nblk & 1) * 32 + tx;
      Xh[o] = hi;
      Xl[o] = __float2half_rn(v - __half2float(hi));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(absmax), __float_as_int(mx));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(reinterpret_cast<double*>(absmax + 2), sq);
}

// e5m2 copies of the split X for the fp8 correction passes, [X_l * 2^ax | X_h * 2^-bx][tile][d_pad][128 n] (one 128-byte row =
// the 128 rows of a tile for one column j: a single MN group of the 8-bit MN-major operand)
__global__ void fast_prepare_x8_kernel(const __half* __restrict__ Xh, const __half* __restrict__ Xl, int64_t numTiles, int d_pad,
                                       float sl, float sh, uint8_t* __restrict__ X8) {
  const int64_t total = numTiles * (int64_t)d_pad * 128;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(i & 127);
    const int64_t tj = i >> 7;                       // tile * d_pad + j
    const int64_t t = tj / d_pad;
    const int j = (int)(tj - t * d_pad);
    const size_t o = (((size_t)t * 2 + (n >> 6)) * d_pad + j) * 64 + (n & 63);
    X8[i] = to_e5m2(__half2float(Xl[o]) * sl);
    X8[total + i] = to_e5m2(__half2float(Xh[o]) * sh);
  }
}

// Theta^T hi [4][d_pad][64], E [d_pad/64][256][64] (fp16), the e5m2 Theta copies and weights, zero padded
__global__ void fast_prepare_theta_kernel(const double* __restrict__ theta, const double* __restrict__ base,
                                          const double* __restrict__ w, int64_t S, int d, int d_pad,
                                          __half* __restrict__ Th, __half* __restrict__ E,
                                          float* __restrict__ wf, uint8_t* __restrict__ T8, int ax, int bx) {
  PDL_SYNC();
  const int64_t total = (int64_t)kSP * d_pad;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    {   // E: [s][j]
      const int64_t s = i / d_pad;
      const int j = (int)(i - s * d_pad);
      float e = 0.0f;
      if (base && s < S && j < d) e = (float)base[s * d + j];
      E[((size_t)(j >> 6) * kSP + s) * 64 + (j & 63)] = __float2half_rn(e);
    }
    {   // Theta^T: [j][s]
      const int j = (int)(i / kSP);
      const int64_t s = i - (int64_t)j * kSP;
      float t = 0.0f;
      if (s < S && j < d) t = (float)theta[s * d + j];
      const __half hi = __float2half_rn(t);
      const size_t o = ((size_t)(s >> 6) * d_pad + j) * 64 + (s & 63);
      Th[o] = hi;
      const float lof = t - __half2float(hi);       // fp32 residual: the e5m2 copy must not inherit an fp16 underflow
      const size_t o8 = ((size_t)(s >> 7) * d_pad + j) * 128 + (s & 127);
      T8[o8] = to_e5m2(__half2float(hi) * exp2f((float)-ax));
      T8[(size_t)2 * d_pad * 128 + o8] = to_e5m2(lof * exp2f((float)bx));
    }
  }
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < kSP; s += (int64_t)gridDim.x * blockDim.x)
    wf[s] = s < S ? (w ? (float)w[s] : 1.0f) : 0.0f;
}

// out[i] = sign * sum_b part[b][i] for up to three arrays in one launch (blockIdx.y selects the array):
// 32 columns x 8 row groups per block, coalesced 256-byte row reads, shared-memory reduction over the groups
struct Reduce3 {
  const double* part[3];
  double* out[3];
  int nblk[3];
  int64_t stride[3], n[3];
  double sign[3];
};
__global__ void __launch_bounds__(256) reduce_partials3_kernel(Reduce3 a) {
  PDL_SYNC();
  __shared__ double sm[8][33];
  const int which = blockIdx.y;
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * 32 + x;
  const int64_t n = a.n[which];
  if ((int64_t)blockIdx.x * 32 >= n) return;
  double acc = 0.0;
  if (i < n) {
    const double* p = a.part[which] + i;
    const int64_t stride = a.stride[which];
    for (int b = y; b < a.nblk[which]; b += 8) acc += p[(size_t)b * stride];
  }
  sm[y][x] = acc;
  __syncthreads();
  if (y == 0 && i < n) {
    double t = 0.0;
#pragma unroll
    for (int r = 0; r < 8; ++r) t += sm[r][x];
    a.out[which][i] = a.sign[which] * t;
  }
}

// ---- host side -----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// fp16 tensor of 128-byte rows (innermost dimension 64), 128-byte swizzle.  dims/box are innermost first;
// strides (bytes) are those of dims[1..rank-1].
static bool encode_nd(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides,
                      const uint32_t* box, CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_FLOAT16) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t gd[5], gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i + 1 < rank) gs[i] = strides[i];
  }
  CUresult r = enc(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

struct FastModel {
  int64_t N, numTiles;
  int d, d_pad;
  const __half* Xh;
  const uint8_t* X8;                         // e5m2 [X_l 2^ax | X_h 2^-bx][tile][d_pad][128]
  int ax, bx;
  CUtensorMap tmXP16, tmXP8;                 // 4-D [tile][half][j][64] over X_h; 4-D [which][tile][j][128] bytes
};

struct FastLayout {
  size_t off_Th, off_E, off_w, off_ll, off_gmu, off_ge, off_T8, total;
  int grid;
};

static void fast_layout(int64_t N, int d_pad, FastLayout& L) {
  const int64_t tiles = ceil_div(N, kBM);
  int sms = sm_count();
  const int64_t ctas = ceil_div(tiles, 2) * 2;                  // the pair kernel runs two CTAs per 256-row super-tile
  L.grid = (int)(ctas < sms ? (ctas > 1 ? ctas : 2) : sms);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 1024); return o; };
  L.off_Th = take((size_t)kSP * d_pad * 2);
  L.off_E = take((size_t)kSP * d_pad * 2);
  L.off_w = take(kSP * sizeof(float));
  L.off_ll = take((size_t)L.grid * kSP * sizeof(double));
  L.off_gmu = take((size_t)L.grid * d_pad * sizeof(double));
  L.off_ge = take((size_t)L.grid * d_pad * sizeof(double));
  L.off_T8 = take((size_t)2 * kSP * d_pad);                    // e5m2 Theta_h8 | Theta_l8
  L.total = off;
}

}  // namespace fast
}  // namespace vb

using namespace vb;
using namespace vb::fast;

extern "C" size_t vb_glm_fast_model_bytes(int64_t N, int d) {
  if (N <= 0 || d <= 0) return 0;
  const int64_t N_pad = ceil_div(N, 2 * kBM) * 2 * kBM;        // whole 256-row super-tiles (CTA pairs)
  const int64_t d_pad = ceil_div(d, 256) * 256;
  return (size_t)(2 * N_pad * d_pad * 2) + 1024 + (size_t)(2 * N_pad * d_pad);       // fp16 hi | lo, absmax, e5m2 X_l8 | X_h8
}

extern "C" size_t vb_glm_fast_workspace_bytes(int64_t N, int d, int64_t S) {
  if (N <= 0 || d <= 0 || S <= 0 || S > kSP) return 0;
  FastLayout L;
  fast_layout(N, (int)(ceil_div(d, 256) * 256), L);
  return L.total;
}

extern "C" int vb_glm_fast_create(void** handle, const double* X, int64_t ldx, const double* y, int64_t N, int d,
                                  int link, void* model_mem, size_t model_bytes, float* absmax_host,
                                  cudaStream_t stream) {
  if (!handle || !X || !y || N <= 0 || d <= 0 || ldx < d || !model_mem)
    return set_error(VB_ERR_INVALID_ARG, "glm_fast_create: bad arguments");
  if (link != VB_LINK_LOGISTIC) return set_error(VB_ERR_UNSUPPORTED, "glm_fast: only the logistic link has a tensor-core path");
  if (d > 2048) return set_error(VB_ERR_UNSUPPORTED, "glm_fast: d > 2048 not supported");
  if (model_bytes < vb_glm_fast_model_bytes(N, d)) return set_error(VB_ERR_WORKSPACE, "glm_fast_create: model buffer too small");
  if ((reinterpret_cast<uintptr_t>(model_mem) & 1023) != 0)
    return set_error(VB_ERR_INVALID_ARG, "glm_fast_create: model buffer must be 1024-byte aligned");
  FastModel* m = new FastModel();
  m->N = N;
  m->d = d;
  m->numTiles = ceil_div(N, 2 * kBM) * 2;                       // even: the pair kernel works on super-tiles
  m->d_pad = (int)(ceil_div(d, 256) * 256);
  const size_t elems = (size_t)m->numTiles * kBM * m->d_pad;
  __half* Xh = static_cast<__half*>(model_mem);
  __half* Xl = Xh + elems;
  float* absmax = reinterpret_cast<float*>(Xl + elems);
  m->Xh = Xh;
  cudaError_t e = cudaMemsetAsync(absmax, 0, 16, stream);          // [0]: max |y X| (float), [2..3]: sum of squares (double)
  if (e != cudaSuccess) { delete m; return set_cuda_error(e); }
  fast_prepare_x_kernel<<<sm_count() * 8, 256, 0, stream>>>(X, ldx, y, N, d, m->numTiles, m->d_pad, Xh, Xl, absmax);
  e = cudaGetLastError();
  if (e != cudaSuccess) { delete m; return set_cuda_error(e); }
  float amax = 0.0f;
  float stats[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  {
    e = cudaMemcpyAsync(stats, absmax, 16, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) { delete m; return set_cuda_error(e); }
    amax = stats[0];
    if (absmax_host) *absmax_host = amax;
    if (!(amax < 3.0e4f)) {             // also a NaN or infinite entry of y*X
      delete m;
      return set_error(VB_ERR_UNSUPPORTED, "glm_fast: |y*X| exceeds the fp16 operand range or is not finite; use the float64 path");
    }
  }
  {
    // fp8 correction operands: static power-of-two scales from the TYPICAL magnitude of the data (r = round(log2 rms),
    // not the maximum: one outlier must not push the other entries' residuals below e5m2's range): X_l 2^ax sits near
    // 2^-10 and X_h 2^-bx near 2^-8 for typical entries, which leaves e5m2's 30 binades to Theta on the other side
    // (|theta| ~ 1 / (rms sqrt(d)) for logits of order one); clamped so that the largest entry cannot overflow e5m2.
    double sumsq;
    memcpy(&sumsq, stats + 2, sizeof(double));
    const double rms = sqrt(sumsq / ((double)N * (double)d));
    int r = 0, sexp = 0;
    if (rms > 0.0) r = (int)lrint(log2(rms));
    if (amax > 0.0f) frexpf(amax, &sexp);                       // amax < 2^sexp
    m->ax = 2 - r;
    m->bx = 8 + r;
    if (m->ax > 26 - sexp) m->ax = 26 - sexp;                    // |X_l| <= 2^-11 max|X|:  X_l 2^ax < 2^15
    if (m->bx < sexp - 15) m->bx = sexp - 15;                    // X_h 2^-bx < 2^15
    uint8_t* X8 = reinterpret_cast<uint8_t*>(model_mem) + (size_t)elems * 4 + 1024;
    m->X8 = X8;
    fast_prepare_x8_kernel<<<sm_count() * 8, 256, 0, stream>>>(Xh, Xl, m->numTiles, m->d_pad, exp2f((float)m->ax),
                                                               exp2f((float)-m->bx), X8);
    e = cudaGetLastError();
    if (e != cudaSuccess) { delete m; return set_cuda_error(e); }
  }
  const uint64_t x16d[4] = {64, (uint64_t)m->d_pad, 2, (uint64_t)m->numTiles};
  const uint64_t x16s[3] = {128, (uint64_t)m->d_pad * 128, (uint64_t)m->d_pad * 256};
  const uint32_t x16b[4] = {64, 32, 2, 1};
  const uint64_t x8d[4] = {128, (uint64_t)m->d_pad, (uint64_t)m->numTiles, 2};
  const uint64_t x8s[3] = {128, (uint64_t)m->d_pad * 128, (uint64_t)elems};
  const uint32_t x8b[4] = {128, 32, 1, 2};
  if (!encode_nd(&m->tmXP16, Xh, 4, x16d, x16s, x16b) ||
      !encode_nd(&m->tmXP8, m->X8, 4, x8d, x8s, x8b, CU_TENSOR_MAP_DATA_TYPE_UINT8)) {
    delete m;
    return set_error(VB_ERR_CUDA, "glm_fast_create: cuTensorMapEncodeTiled failed");
  }
  *handle = m;
  return VB_OK;
}

extern "C" int vb_glm_fast_destroy(void* handle) {
  delete static_cast<FastModel*>(handle);
  return VB_OK;
}

// ---- internal interface shared with engine.cu (fast_internal.cuh) ----------------------------------------------
namespace vb {
namespace fast {

int fast_dims(void* handle, int64_t* N, int* d, int* d_pad) {
  FastModel* m = static_cast<FastModel*>(handle);
  if (!m) return set_error(VB_ERR_INVALID_ARG, "glm_fast: null handle");
  if (N) *N = m->N;
  if (d) *d = m->d;
  if (d_pad) *d_pad = m->d_pad;
  return VB_OK;
}

int fast_operands(void* handle, void* workspace, size_t workspace_bytes, FastOperands* ops) {
  FastModel* m = static_cast<FastModel*>(handle);
  if (!m || !ops) return set_error(VB_ERR_INVALID_ARG, "glm_fast: null handle");
  FastLayout L;
  fast_layout(m->N, m->d_pad, L);
  if (!workspace || workspace_bytes < L.total) return set_error(VB_ERR_WORKSPACE, "glm_fast_sweep: workspace too small");
  if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0)
    return set_error(VB_ERR_INVALID_ARG, "glm_fast_sweep: workspace must be 1024-byte aligned");
  char* ws = static_cast<char*>(workspace);
  ops->Th = reinterpret_cast<__half*>(ws + L.off_Th);
  ops->E = reinterpret_cast<__half*>(ws + L.off_E);
  ops->wf = reinterpret_cast<float*>(ws + L.off_w);
  ops->T8 = reinterpret_cast<uint8_t*>(ws + L.off_T8);
  ops->ax = m->ax;
  ops->bx = m->bx;
  return VB_OK;
}

// Launches the sweep kernel on operands already packed into the workspace (Th, E, wf, T8); the per-CTA / per-pair
// partial sums stay in the workspace and are described by `parts` (ll partials are sums of softplus: sign -1).
int fast_launch(void* handle, void* workspace, size_t workspace_bytes, int S, int want_grad, int ll_total_only,
                int uniform_w, float* debug, cudaStream_t stream, FastPartials* parts) {
  FastModel* m = static_cast<FastModel*>(handle);
  FastOperands ops;
  int rc = fast_operands(handle, workspace, workspace_bytes, &ops);
  if (rc) return rc;
  if (S <= 0 || S > kSP) return set_error(VB_ERR_UNSUPPORTED, "glm_fast_sweep: at most 256 samples per sweep");
  FastLayout L;
  fast_layout(m->N, m->d_pad, L);
  char* ws = static_cast<char*>(workspace);

  // The maps are keyed on everything they encode: the workspace address, d_pad and the T8 address.  T8 follows the
  // per-CTA partial sums, so its offset also depends on the grid, i.e. on N: two models with the same d_pad that
  // share a workspace address place their e5m2 Theta copies at different offsets.
  static thread_local const void* cached_ws = nullptr;
  static thread_local const void* cached_t8 = nullptr;
  static thread_local int cached_dpad = 0;
  static thread_local CUtensorMap tmTP16, tmEP, tmTP8;
  if (cached_ws != workspace || cached_dpad != m->d_pad || cached_t8 != ops.T8) {
    cached_ws = nullptr;           // a failed encode below leaves no valid entry behind
    const uint64_t dp = (uint64_t)m->d_pad;
    const uint64_t t16d[3] = {64, dp, 4}, t16s[2] = {128, dp * 128};
    const uint32_t t16b[3] = {64, 32, 2};
    const uint64_t ed[3] = {64, (uint64_t)kSP, dp / 64}, es[2] = {128, (uint64_t)kSP * 128};
    const uint32_t eb[3] = {64, 64, 2};
    const uint64_t t8d[4] = {128, dp, 2, 2}, t8s[3] = {128, dp * 128, dp * 256};
    const uint32_t t8b[4] = {128, 32, 1, 2};
    if (!encode_nd(&tmTP16, ops.Th, 3, t16d, t16s, t16b) || !encode_nd(&tmEP, ops.E, 3, ed, es, eb) ||
        !encode_nd(&tmTP8, ops.T8, 4, t8d, t8s, t8b, CU_TENSOR_MAP_DATA_TYPE_UINT8))
      return set_error(VB_ERR_CUDA, "glm_fast_sweep: cuTensorMapEncodeTiled failed");
    cached_ws = workspace;
    cached_t8 = ops.T8;
    cached_dpad = m->d_pad;
  }

  Params p;
  p.N = m->N;
  p.d_pad = m->d_pad;
  p.S = S;
  p.numTiles = (int)m->numTiles;
  p.want_grad = want_grad;
  p.ll_total_only = ll_total_only;
  p.w = ops.wf;
  p.ll_part = reinterpret_cast<double*>(ws + L.off_ll);
  p.gmu_part = reinterpret_cast<double*>(ws + L.off_gmu);
  p.ge_part = reinterpret_cast<double*>(ws + L.off_ge);
  p.tim = debug ? reinterpret_cast<long long*>(debug + (size_t)49152 * L.grid) : nullptr;
  p.Xh = m->Xh;
  p.Xl8 = m->X8;
  p.xl_scale = exp2f((float)-m->ax);
  p.uniform_w = uniform_w;
  int pair_clusters = 0;
  {
    // function attributes and the cluster occupancy are per device: cache them per device ordinal, under a lock
    static std::mutex mu;
    static int cached[64];
    static bool ready[64] = {false};
    int dev = 0;
    VB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return set_error(VB_ERR_UNSUPPORTED, "glm_fast_sweep: device ordinal out of range");
    std::lock_guard<std::mutex> lock(mu);
    if (!ready[dev]) {
      VB_CUDA(cudaFuncSetAttribute(glm_fast_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
      int nc = 0;
      cudaLaunchConfig_t qc = {};
      qc.gridDim = dim3(sm_count() & ~1);
      qc.blockDim = dim3(kThreadsP);
      qc.dynamicSmemBytes = kSmemBytes;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = 2;
      qa[0].val.clusterDim.y = 1;
      qa[0].val.clusterDim.z = 1;
      qc.attrs = qa;
      qc.numAttrs = 1;
      if (cudaOccupancyMaxActiveClusters(&nc, glm_fast_pair_kernel, &qc) != cudaSuccess) {
        cudaGetLastError();
        nc = 0;
      }
      cached[dev] = nc;
      ready[dev] = true;
    }
    pair_clusters = cached[dev];
  }
  if (pair_clusters <= 0)
    return set_error(VB_ERR_UNSUPPORTED, "glm_fast_sweep: the CTA-pair kernel cannot be scheduled on this device; use the float64 path");
  const int64_t numSuper = m->numTiles / 2;
  int clusters = pair_clusters < L.grid / 2 ? pair_clusters : L.grid / 2;
  if (clusters < 1) clusters = 1;
  if (numSuper < clusters) clusters = (int)numSuper;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * clusters);
  cfg.blockDim = dim3(kThreadsP);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 2;
  VB_CUDA(cudaLaunchKernelEx(&cfg, glm_fast_pair_kernel, m->tmXP16, tmTP16, tmEP, m->tmXP8, tmTP8, p));
  if (parts) {
    parts->ll_part = p.ll_part;
    parts->gmu_part = p.gmu_part;
    parts->ge_part = p.ge_part;
    parts->nblk_ll = 2 * clusters;
    parts->nblk_g = clusters;       // one row of gradient partials per pair (a CTA owns half of the columns)
    parts->stride_ll = kSP;
    parts->stride_g = m->d_pad;
  }
  return VB_OK;
}

}  // namespace fast
}  // namespace vb

extern "C" int vb_glm_fast_sweep(void* handle, const double* theta, const double* base, const double* w, int64_t S,
                                 int want_grad, double* out_ll, double* out_gmu, double* out_ge, void* workspace,
                                 size_t workspace_bytes, float* debug, cudaStream_t stream) {
  // want_grad bit 0: gradients wanted; bit 1: only sum_s ll[s] is needed (each out_ll[s] receives the mean)
  // (when debug is given, debug + 49152*grid floats holds 128 int64 clock64 timestamp slots of CTA 0)
  FastModel* m = static_cast<FastModel*>(handle);
  const int ll_total_only = (want_grad >> 1) & 1;
  want_grad &= 1;
  if (!m || !theta || !out_ll || S <= 0) return set_error(VB_ERR_INVALID_ARG, "glm_fast_sweep: bad arguments");
  if (S > kSP) return set_error(VB_ERR_UNSUPPORTED, "glm_fast_sweep: at most 256 samples per sweep");
  if (want_grad && (!base || !out_gmu || !out_ge)) return set_error(VB_ERR_INVALID_ARG, "glm_fast_sweep: want_grad needs base, out_gmu, out_ge");
  FastOperands ops;
  int rc = fast_operands(handle, workspace, workspace_bytes, &ops);
  if (rc) return rc;
  VB_CUDA(launch_pdl(fast_prepare_theta_kernel, dim3(128), dim3(256), stream, theta, want_grad ? base : nullptr, w, S, m->d, m->d_pad,
                     ops.Th, ops.E, ops.wf, ops.T8, ops.ax, ops.bx));
  FastPartials parts;
  rc = fast_launch(handle, workspace, workspace_bytes, (int)S, want_grad, ll_total_only, w ? 0 : 1, debug, stream, &parts);
  if (rc) return rc;
  // ll = -sum softplus; gradient partials summed over the pairs -- one launch for the three arrays
  Reduce3 r;
  r.part[0] = parts.ll_part;  r.out[0] = out_ll;  r.nblk[0] = parts.nblk_ll; r.stride[0] = kSP;      r.n[0] = S;                    r.sign[0] = -1.0;
  r.part[1] = parts.gmu_part; r.out[1] = out_gmu; r.nblk[1] = parts.nblk_g;  r.stride[1] = m->d_pad; r.n[1] = want_grad ? m->d : 0; r.sign[1] = 1.0;
  r.part[2] = parts.ge_part;  r.out[2] = out_ge;  r.nblk[2] = parts.nblk_g;  r.stride[2] = m->d_pad; r.n[2] = want_grad ? m->d : 0; r.sign[2] = 1.0;
  const int64_t nmax = want_grad && m->d > S ? m->d : S;
  VB_CUDA(launch_pdl(reduce_partials3_kernel, dim3((unsigned)((nmax + 31) / 32), want_grad ? 3 : 1), dim3(256), stream, r));
  return VB_OK;
}
