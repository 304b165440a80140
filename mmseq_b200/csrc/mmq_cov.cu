/* mmq_cov.cu — the consumer side of the Gibbs trace: mmcollapse's per-sample trace covariance and its
 * mean-correlation scan (SURVEY.md section 8, row f3).
 *
 *   get_corrs(),  src/mmcollapse.cpp:514-561:  R.slice(s) = cov(myM) of the 1024 x C matrix of posterior traces of
 *                 the C collapse candidates of sample s (Armadillo cov(): centred columns, X^T X / (L - 1)),
 *                 non-finite entries -> 0 (:556-558);
 *   mean_corrs(), src/mmcollapse.cpp:483-511:  mean / sd over the samples of the correlation of a pair.
 *
 * This is the ONE dense contraction of the package, so it is the one place tensor cores are used:
 *
 *   k_cov_prep   one block per feature: mean and centred sum of squares in fp64, z = (x - mean) / sqrt(ssq)
 *                (so that the Gram matrix of z IS the correlation matrix, |z| <= 1), split into 1..3 bf16 terms
 *                z = z0 + z1 + z2 with fp64 residuals, stored K-major: Z[c][split * L + s];
 *   k_cov_gemm2  the 256 x 256 tiles of Z Z^T on or above the diagonal, on the 5th-generation tensor cores, one tile per
 *                CTA PAIR.  Persistent, clusters of two CTAs, warp-specialised: warp 0 = TMA producer (cp.async.bulk.tensor,
 *                128-byte swizzle, SASS UTMALDG.2D.2CTA; each CTA loads its 128 rows of both operands, both signalling the
 *                leader's mbarrier) into a 4-stage shared-memory ring; warp 1 of the leader = one thread issuing
 *                tcgen05.mma.cta_group::2 (kind::f16, bf16 x bf16 -> fp32, M 256 x N 256 x K 16 per pair, SASS UTCHMMA.2CTA)
 *                into one of TWO 256-column TMEM accumulators per SM, stage release and accumulator hand-over through
 *                tcgen05.commit multicast to both CTAs (UTCBAR.2CTA.MULTICAST); warps 2..9 = epilogue of the previous tile
 *                while the next one accumulates: tcgen05.ld (SASS LDTM), back to covariance in fp64 (r * sd_i * sd_j), a
 *                32 x 32 transposition through shared memory so that BOTH triangles are stored with full 256-byte warp
 *                stores (streaming), the diagonal exactly var_i, exactly symmetric; the accumulator goes back to the leader
 *                by a remote mbarrier arrive from the epilogue warps of both CTAs.  The split terms z_a z_b with
 *                a + b < nsplit are extra K-segments of the same accumulation (smallest terms first).
 *   k_mean_corrs the scan over samples, one thread per (row of ts, column) pair.
 *
 * Accuracy, in correlation units |cov_gpu - cov_exact| / (sd_i sd_j), for traces of length L: at most A + 1.5e-8 L, A =
 * 6e-3 / 1.2e-5 / 2e-7 for nsplit = 1 / 2 (the default) / 3 (include/mmq.h; tests/test_gpu_cov_accuracy.py asserts it
 * at L = 64 .. 65536).  A is the bf16 split, each term keeping 8 significant bits of what the previous ones left.  The
 * L term is the fp32 accumulation in TMEM: the tensor cores truncate the running sum towards zero, L / 16 times per
 * split product, so the error is a bias towards r = 0 that grows linearly with L, largest for a near-collinear pair
 * whose sum reaches |r| ~ 1 early.  At mmcollapse's L = 1024 that is 2.7e-5 for nsplit = 2, against a Monte-Carlo
 * error of a correlation estimated from 1024 draws of >= 1e-2.
 *
 * What bounds it: 0.91-0.93 ms at C = 16384, nsplit = 2 (0.54 of the measured cuBLAS bf16 peak; 0.66 with nsplit = 3).
 * Per MMA an SM reads 8 KB of operands from shared memory and receives 32 KB of TMA writes per stage, where one CTA alone
 * (M 128) needs 12 KB and 48 KB: together with the epilogue's transposition that is more than the 128 B/clk of
 * shared-memory bandwidth an SM has (a single-CTA version measured 0.99 ms; removed).  Taken apart with the stores and / or
 * the MMAs switched off (same pipeline otherwise): neither 0.45 ms, stores only 0.78, MMAs only 0.76, both 0.93-0.96.
 * The floor is the operand
 * traffic: 6.4 GB of tiles from the L2-resident Z per launch at the L2's ~12 TB/s (131 flop per byte for a 256 x 256 pair
 * tile caps the MMAs at 1.5 PFLOP/s, which is what each further split product costs: 0.18 ms), plus the epilogue's own
 * work (TMEM loads, the fp64 scaling, the transposition: ~0.25 ms) and the 2.1 GB of stores.  Both split terms of a K block
 * in one stage (every operand tile loaded once: 1.5x less L2 traffic, but only two stages fit) measured 0.90 against
 * 0.94 ms: not kept.  Next: clusters of two pairs with the shared operand multicast.
 */
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>
#include <stdint.h>

#include <algorithm>
#include <mutex>
#include <string>

#include "mmq_device.cuh"
#include "mmq_internal.h"

namespace {

constexpr int COV_BM = 128, COV_BN = 256, COV_BK = 64; /* one SM's part of a tile: 128 x 256 outputs, 64 bf16 (= one 128-byte swizzle row) of K per stage */
constexpr int COV_UMMA_K = 16;
constexpr int COV_A_BYTES = COV_BM * COV_BK * 2;
constexpr int COV_TMEM_COLS = 2 * COV_BN; /* two fp32 accumulators of COV_BN columns: all 512 columns, one CTA per SM */
constexpr int COV_THREADS = 320; /* warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2..9: epilogue (two per TMEM lane quarter) */
constexpr int COV_EPI_WARPS = 8;
constexpr int COV_EPI_BYTES = (33 * 32 + 32) * 8; /* per epilogue warp: 33 x 32 transposition buffer + sd of 32 columns */

/* ---- small PTX wrappers (tcgen05 / TMA tensor copies; the mbarrier basics are in mmq_device.cuh) ---- */
__device__ __forceinline__ void mbar_wait_trap(uint64_t* b, uint32_t parity) {
  /* a wrong descriptor or byte count must end in an error, not in a hung GPU */
  uint32_t ok;
  for (uint32_t spin = 0;; ++spin) {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok)
                 : "r"(smem_u32(b)), "r"(parity)
                 : "memory");
    if (ok) return;
    if (spin > (1u << 22)) __trap();
  }
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
/* shared-memory matrix descriptor of a K-major tile whose rows are 128 bytes, 128-byte swizzle (what TMA wrote):
 * start address >> 4 | leading byte offset (unused with swizzle: 1) << 16 | stride byte offset (8 rows = 1024 B) >> 4 << 32 |
 * descriptor version 1 (sm_100) << 46 | layout type 2 (SWIZZLE_128B) << 61 */
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, "
      "%21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
        "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
        "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

/* ---- k_cov_prep ---- */
__device__ __forceinline__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  double s = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i]; /* same order in every thread */
  return s;
}

/* feature c: x[s] = src[off[c] + s * stride], s < L.  Z: [C][nsplit * L] bf16.  sd[c] = sqrt(ssq / (L - 1)), 0 for a feature with a
 * non-finite value (its covariances are 0, as :556-558 leaves them). */
__global__ void __launch_bounds__(256) k_cov_prep(const double* __restrict__ src, const int64_t* __restrict__ off, int64_t off_step, int64_t stride,
                                                  int L, int64_t C, int nsplit, __nv_bfloat16* __restrict__ Z, double* __restrict__ sd) {
  __shared__ double red[8];
  const int64_t c = blockIdx.x;
  if (c >= C) return;
  const double* x = src + (off ? off[c] : c * off_step);
  double s = 0.0;
  for (int i = threadIdx.x; i < L; i += blockDim.x) s += x[(int64_t)i * stride];
  s = block_sum(s, red);
  const double mean = s / (double)L;
  double q = 0.0;
  for (int i = threadIdx.x; i < L; i += blockDim.x) {
    const double d = x[(int64_t)i * stride] - mean;
    q += d * d;
  }
  q = block_sum(q, red);
  const bool ok = isfinite(q) && q > 0.0;
  const double inv = ok ? 1.0 / sqrt(q) : 0.0;
  if (threadIdx.x == 0) sd[c] = ok ? sqrt(q / (double)(L > 1 ? L - 1 : 1)) : 0.0;
  __nv_bfloat16* z = Z + c * (int64_t)nsplit * L;
  for (int i = threadIdx.x; i < L; i += blockDim.x) {
    double r = ok ? (x[(int64_t)i * stride] - mean) * inv : 0.0;
    for (int t = 0; t < nsplit; ++t) {
      const __nv_bfloat16 b = __float2bfloat16_rn((float)r);
      z[(int64_t)t * L + i] = b;
      r -= (double)__bfloat162float(b);
    }
  }
}

/* ---- k_cov_gemm2: Z Z^T on CTA PAIRS (tcgen05.mma.cta_group::2) ----
 * A cluster of two CTAs (two SMs of one TPC) computes one 256 x 256 tile: CTA r of the pair holds rows 128 r .. of the A
 * operand and rows 128 r .. of the B operand (each loaded by its own TMA producer, both signalling the LEADER's mbarrier),
 * the leader's elected thread issues M 256 x N 256 x K 16 MMAs for both SMs, every SM accumulates its own 128 x 256 half in
 * its own TMEM and drains it with its own epilogue warps.  Per MMA an SM reads 8 KB of operands from shared memory instead
 * of the 12 KB of a single-CTA M 128 MMA, and receives 32 KB per stage instead of 48 KB: shared-memory bandwidth is what
 * bounds a single CTA (DESIGN.md).  Persistent: pair p walks the tiles p, p + pairs, ...  Stage release and accumulator
 * hand-over: tcgen05.commit with .multicast::cluster to both CTAs; the accumulator is handed back to the leader by the
 * epilogue warps of BOTH CTAs (remote mbarrier arrive through mapa). */
constexpr int COV2_STAGES = 4;
constexpr int COV2_STAGE_BYTES = 2 * COV_A_BYTES; /* this CTA's 128 rows of A and its 128 rows of B */
constexpr int COV2_SMEM = COV2_STAGES * COV2_STAGE_BYTES + COV_EPI_WARPS * COV_EPI_BYTES + 256 /* barriers, TMEM slot */ + 1024 /* alignment */;
/* instruction descriptor of the pair: fp32 accumulator (1 << 4), A and B bf16 (1 << 7, 1 << 10), both K-major (bits 15,
 * 16 zero), N >> 3 at bit 17, M >> 4 at bit 24; M = 256 */
constexpr uint32_t COV2_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
/* the address of the same shared-memory location in CTA `rank` of the cluster */
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, int c0, int c1, uint32_t leader_bar) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
               "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) { /* arrives on this barrier in BOTH CTAs of the pair */
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"((uint16_t)3)
               : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(COV_THREADS, 1)
    k_cov_gemm2(const __grid_constant__ CUtensorMap zmap, const double* __restrict__ sd, double* __restrict__ R, int64_t C, int L, int nsplit,
                int64_t tiles) {
  extern __shared__ uint8_t cov_smem_raw[];
  uint8_t* smem = cov_smem_raw + ((1024u - (smem_u32(cov_smem_raw) & 1023u)) & 1023u);
  uint8_t* epi = smem + COV2_STAGES * COV2_STAGE_BYTES;
  uint64_t* full = (uint64_t*)(epi + COV_EPI_WARPS * COV_EPI_BYTES); /* used in the leader only: both producers' bytes land there */
  uint64_t* empty = full + COV2_STAGES;
  uint64_t* tfull = empty + COV2_STAGES;
  uint64_t* tempty = tfull + 2; /* used in the leader only: 8 epilogue warps of each CTA arrive */
  uint32_t* tmem_slot = (uint32_t*)(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_rank();
  const bool leader = rank == 0;
  const int64_t pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&zmap) : "memory");
    for (int s = 0; s < COV2_STAGES; ++s) {
      mbar_init(full + s, 1);
      mbar_init(empty + s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull + b, 1);
      mbar_init(tempty + b, 2 * COV_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  cluster_sync_all(); /* nobody signals a barrier of the peer before it is initialised */
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(COV_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int kb_per_seg = L / COV_BK;
  const int iters = (nsplit * (nsplit + 1) / 2) * kb_per_seg;

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;
      for (int64_t t = pair; t < tiles; t += npairs) {
        int64_t nb = (int64_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
        while (nb * (nb + 1) / 2 > t) --nb;
        while ((nb + 1) * (nb + 2) / 2 <= t) ++nb;
        const int64_t mb = t - nb * (nb + 1) / 2;
        const int row_a = (int)(mb * 256 + rank * 128), row_b = (int)(nb * 256 + rank * 128);
        for (int sum = nsplit - 1; sum >= 0; --sum)
          for (int a = 0; a <= sum; ++a) {
            const int b = sum - a;
            for (int kb = 0; kb < kb_per_seg; ++kb, ++it) {
              const int stage = it % COV2_STAGES;
              const uint32_t phase = (uint32_t)(it / COV2_STAGES) & 1u;
              mbar_wait_trap(empty + stage, phase ^ 1u);
              uint8_t* dst = smem + stage * COV2_STAGE_BYTES;
              if (leader) mbar_expect_tx(full + stage, 2 * COV2_STAGE_BYTES); /* the bytes of both CTAs */
              const uint32_t lbar = mapa_u32(smem_u32(full + stage), 0);
              tma_load_2d_pair(dst, &zmap, a * L + kb * COV_BK, row_a, lbar);
              tma_load_2d_pair(dst + COV_A_BYTES, &zmap, b * L + kb * COV_BK, row_b, lbar);
            }
          }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      int it = 0, n = 0;
      for (int64_t t = pair; t < tiles; t += npairs, ++n) {
        const int buf = n & 1;
        mbar_wait_trap(tempty + buf, ((uint32_t)(n >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t acc = tmem + (uint32_t)(buf * COV_BN);
        for (int i = 0; i < iters; ++i, ++it) {
          const int stage = it % COV2_STAGES;
          const uint32_t phase = (uint32_t)(it / COV2_STAGES) & 1u;
          mbar_wait_trap(full + stage, phase);
          tc_fence_after();
          const uint32_t a0 = smem_u32(smem + stage * COV2_STAGE_BYTES), b0 = a0 + COV_A_BYTES;
#pragma unroll
          for (int k = 0; k < COV_BK / COV_UMMA_K; ++k)
            tc_mma_bf16_pair(acc, smem_desc_sw128(a0 + k * COV_UMMA_K * 2), smem_desc_sw128(b0 + k * COV_UMMA_K * 2), COV2_IDESC, (uint32_t)((i | k) != 0));
          tc_commit_pair(empty + stage);
        }
        tc_commit_pair(tfull + buf);
      }
    }
    __syncwarp();
  } else {
    const int q = warp & 3, half = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    double* tp = (double*)(epi + (warp - 2) * COV_EPI_BYTES);
    double* sdw = tp + 33 * 32;
    int n = 0;
    for (int64_t t = pair; t < tiles; t += npairs, ++n) {
      int64_t nb = (int64_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
      while (nb * (nb + 1) / 2 > t) --nb;
      while ((nb + 1) * (nb + 2) / 2 <= t) ++nb;
      const int64_t mb = t - nb * (nb + 1) / 2;
      const int64_t row_a = mb * 256 + (int64_t)rank * 128, row_b = nb * 256;
      const int64_t gi = row_a + row, gi0 = row_a + q * 32;
      const double si = gi < C ? sd[gi] : 0.0;
      const bool diag_tile = mb == nb;
      const bool edge = diag_tile || row_a + COV_BM > C || row_b + COV_BN > C;
      const int buf = n & 1;
      mbar_wait_trap(tfull + buf, (uint32_t)(n >> 1) & 1u);
      tc_fence_after();
      for (int c0 = half * (COV_BN / 2); c0 < (half + 1) * (COV_BN / 2); c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * COV_BN + c0), v);
        if (c0 + 32 == (half + 1) * (COV_BN / 2)) {
          tc_fence_before();
          if (lane == 0) {
            const uint32_t lb = mapa_u32(smem_u32(tempty + buf), 0);
            asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(lb) : "memory");
          }
        }
        const int64_t gj0 = row_b + c0;
        sdw[lane] = gj0 + lane < C ? sd[gj0 + lane] : 0.0;
        __syncwarp();
        if (!edge) {
          double* dp = R + gi + C * gj0;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const double val = (double)__uint_as_float(v[j]) * (si * sdw[j]);
            tp[j * 33 + lane] = val;
            __stcs(dp, val);
            dp += C;
          }
          __syncwarp();
          double* mp = R + gj0 + lane + C * gi0;
#pragma unroll
          for (int ii = 0; ii < 32; ++ii) {
            __stcs(mp, tp[lane * 33 + ii]);
            mp += C;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int64_t gj = gj0 + j;
            const double val = gi == gj ? si * si : (double)__uint_as_float(v[j]) * (si * sdw[j]);
            tp[j * 33 + lane] = val;
            if (gi < C && gj < C && !(diag_tile && gj < gi)) __stcs(R + gi + C * gj, val);
          }
          __syncwarp();
          const int64_t gj = gj0 + lane;
          if (gj < C) {
#pragma unroll 8
            for (int ii = 0; ii < 32; ++ii) {
              const int64_t gr = gi0 + ii;
              if (gr >= C) break;
              if (diag_tile ? gj > gr : true) __stcs(R + gj + C * gr, tp[lane * 33 + ii]);
            }
          }
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  cluster_sync_all(); /* the leader's MMAs write the peer's TMEM and barriers: nobody leaves before everybody is done */
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(COV_TMEM_COLS) : "memory");
  }
}

/* ---- k_mean_corrs: src/mmcollapse.cpp:483-511 ---- */
__global__ void __launch_bounds__(256) k_mean_corrs(const double* __restrict__ R, const uint8_t* __restrict__ S, int64_t C, int ns,
                                                    const int32_t* __restrict__ ts, int64_t nts, double sdpenalty, double* __restrict__ V,
                                                    double* __restrict__ W) {
  const int64_t CC = C * C;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nts * C; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = ts[p / C], v = p % C;
    double su = 0.0, sr = 0.0, sr2 = 0.0;
    for (int s = 0; s < ns; ++s) {
      const double* Rs = R + (int64_t)s * CC;
      double r = Rs[v + C * t]; /* = Rs[t + C v]: the slices are symmetric; this way a warp reads consecutive addresses */
      r = r / sqrt(Rs[t + C * t]);
      r = r / sqrt(Rs[v + C * v]);
      const double u = (double)(S[t + C * s] * S[v + C * s]);
      if (u == 0.0) r = 0.0;
      su += u;
      sr += u * r;
      sr2 += u * (r * r);
    }
    double mean = sr / su, sdv = 0.0;
    if (ns > 1) {
      sdv = sqrt((su / (su - 1.0)) * (sr2 / su - mean * mean));
      if (!isfinite(sdv)) sdv = 0.0;
    }
    mean = mean + sdpenalty * sdv;
    V[t + C * v] = mean;
    V[v + C * t] = mean;
    W[t + C * v] = sdv;
    W[v + C * t] = sdv;
  }
}

/* ---- host side ---- */
typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

encode_tiled_fn get_encode_tiled() {
  static encode_tiled_fn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      fn = (encode_tiled_fn)p;
  });
  return fn;
}

thread_local std::string g_cov_err;
int cov_fail(int code, const std::string& msg) {
  g_cov_err = msg;
  g_mmq_create_err = msg; /* mmq_last_error(NULL) */
  return code;
}
#define COV_CUDA(call)                                                                                                   \
  do {                                                                                                                   \
    cudaError_t e__ = (call);                                                                                            \
    if (e__ != cudaSuccess) return cov_fail(MMQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));          \
  } while (0)

size_t cov_ws_bytes(int L, int64_t C, int nsplit) {
  const size_t z = ((size_t)C * (size_t)nsplit * (size_t)L * 2 + 255) & ~(size_t)255;
  return z + (size_t)C * 8 + 256;
}

int cov_check(int L, int64_t C, int nsplit) {
  if (L < COV_BK || L % COV_BK != 0 || L > 65536) return cov_fail(MMQ_ERR_ARG, "mmq_trace_cov: the trace length must be a multiple of 64 (mmcollapse: 1024)");
  if (C < 1 || C > (int64_t)1 << 20) return cov_fail(MMQ_ERR_ARG, "mmq_trace_cov: 1 <= C <= 2^20 features");
  if (nsplit < 1 || nsplit > 3) return cov_fail(MMQ_ERR_ARG, "mmq_trace_cov: nsplit must be 1, 2 or 3");
  return MMQ_OK;
}

/* src_dev: fp64 on the device; feature c is src[off[c] + s * stride] (off_dev == NULL: src[c * off_step + s * stride]). */
int cov_run(const double* src_dev, const int64_t* off_dev, int64_t off_step, int64_t stride, int L, int64_t C, int nsplit, double* R_dev,
            void* ws_dev, cudaStream_t st) {
  encode_tiled_fn enc = get_encode_tiled();
  if (!enc) return cov_fail(MMQ_ERR_CUDA, "mmq_trace_cov: cuTensorMapEncodeTiled not available from the driver");
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] { attr_err = cudaFuncSetAttribute(k_cov_gemm2, cudaFuncAttributeMaxDynamicSharedMemorySize, COV2_SMEM); });
  if (attr_err != cudaSuccess) return cov_fail(MMQ_ERR_CUDA, std::string("mmq_trace_cov: shared-memory attribute: ") + cudaGetErrorString(attr_err));
  __nv_bfloat16* Z = (__nv_bfloat16*)ws_dev;
  const size_t zbytes = ((size_t)C * (size_t)nsplit * (size_t)L * 2 + 255) & ~(size_t)255;
  double* sd = (double*)((char*)ws_dev + zbytes);
  k_cov_prep<<<(unsigned)C, 256, 0, st>>>(src_dev, off_dev, off_step, stride, L, C, nsplit, Z, sd);
  g_mmq_launches.fetch_add(1, std::memory_order_relaxed);
  COV_CUDA(cudaGetLastError());
  CUtensorMap map;
  const cuuint64_t dims[2] = {(cuuint64_t)nsplit * (cuuint64_t)L, (cuuint64_t)C};
  const cuuint64_t strides[1] = {(cuuint64_t)nsplit * (cuuint64_t)L * 2};
  const cuuint32_t box[2] = {(cuuint32_t)COV_BK, 128u};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult cr = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)Z, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return cov_fail(MMQ_ERR_CUDA, "mmq_trace_cov: cuTensorMapEncodeTiled failed (" + std::to_string((int)cr) + ")");
  const int64_t T = (C + COV_BN - 1) / COV_BN;
  const int64_t tiles = T * (T + 1) / 2; /* 256 x 256 tiles of the upper triangle, one per CTA pair */
  int dev = 0, sms = 148;
  COV_CUDA(cudaGetDevice(&dev));
  COV_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int64_t pairs = std::max<int64_t>(1, std::min<int64_t>(tiles, sms / 2));
  k_cov_gemm2<<<(unsigned)(2 * pairs), COV_THREADS, COV2_SMEM, st>>>(map, sd, R_dev, C, L, nsplit, tiles);
  g_mmq_launches.fetch_add(1, std::memory_order_relaxed);
  COV_CUDA(cudaGetLastError());
  return MMQ_OK;
}

} /* namespace */

extern "C" {

int64_t mmq_trace_cov_workspace_bytes(int L, int64_t C, int nsplit) {
  if (cov_check(L, C, nsplit) != MMQ_OK) return -1;
  return (int64_t)cov_ws_bytes(L, C, nsplit);
}

int mmq_trace_cov_dev(const double* M_dev, int L, int64_t C, int nsplit, double* R_dev, void* workspace_dev, void* cuda_stream) {
  if (!M_dev || !R_dev || !workspace_dev) return cov_fail(MMQ_ERR_ARG, "mmq_trace_cov_dev: NULL argument");
  if (int rc = cov_check(L, C, nsplit)) return rc;
  return cov_run(M_dev, nullptr, L, 1, L, C, nsplit, R_dev, workspace_dev, (cudaStream_t)cuda_stream);
}

int mmq_trace_cov(int device, const double* M, int L, int64_t C, int nsplit, double* R) {
  if (!M || !R) return cov_fail(MMQ_ERR_ARG, "mmq_trace_cov: NULL argument");
  if (int rc = cov_check(L, C, nsplit)) return rc;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return cov_fail(MMQ_ERR_CUDA, "mmq_trace_cov: no CUDA device (there is no CPU fallback)");
  COV_CUDA(cudaSetDevice(device));
  double *dM = nullptr, *dR = nullptr;
  void* ws = nullptr;
  cudaStream_t st = nullptr;
  const size_t mb = (size_t)L * (size_t)C * 8, rb = (size_t)C * (size_t)C * 8;
  int rc = MMQ_OK;
  auto cleanup = [&] { /* the blocks go back to the device block cache (mmq_internal.h): per-sample calls pay cudaMalloc once */
    if (st) cudaStreamSynchronize(st);
    mmq_cache_free(dM);
    mmq_cache_free(dR);
    mmq_cache_free(ws);
    if (st) cudaStreamDestroy(st);
  };
#define COV_TRY(call)                                                                                    \
  do {                                                                                                   \
    cudaError_t e__ = (call);                                                                            \
    if (e__ != cudaSuccess) {                                                                            \
      cleanup();                                                                                         \
      return cov_fail(MMQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));                \
    }                                                                                                    \
  } while (0)
  COV_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  COV_TRY(mmq_cache_malloc(&dM, mb));
  COV_TRY(mmq_cache_malloc(&dR, rb));
  COV_TRY(mmq_cache_malloc(&ws, cov_ws_bytes(L, C, nsplit)));
  COV_TRY(cudaMemcpyAsync(dM, M, mb, cudaMemcpyHostToDevice, st));
  rc = cov_run(dM, nullptr, L, 1, L, C, nsplit, dR, ws, st);
  if (rc == MMQ_OK) {
    COV_TRY(cudaMemcpyAsync(R, dR, rb, cudaMemcpyDeviceToHost, st));
    COV_TRY(cudaStreamSynchronize(st));
  }
  cleanup();
  return rc;
}

int mmq_handle_trace_cov(mmq_handle* h, const int32_t* features, int64_t C, int nsplit, double* R_out, double* R_dev_out) {
  if (!h || !features || (!R_out && !R_dev_out)) return mmq_fail(h, MMQ_ERR_ARG, "mmq_handle_trace_cov: NULL argument");
  if (!h->trace || h->trace_len < 1) return mmq_fail(h, MMQ_ERR_STATE, "mmq_handle_trace_cov: no trace recorded (run mmq_gibbs with trace_len > 0)");
  const int L = h->trace_len;
  if (cov_check(L, C, nsplit) != MMQ_OK) return mmq_fail(h, MMQ_ERR_ARG, g_cov_err);
  MMQ_CUDA(h, cudaSetDevice(h->device));
  /* features >= 0: observed transcript t (trace[t * L + s]); features < 0: identical set -(f + 1) (group trace, slot-major) */
  bool need_sets = false;
  for (int64_t c = 0; c < C; ++c) {
    const int64_t f = features[c];
    if (f >= h->n) return mmq_fail(h, MMQ_ERR_ARG, "mmq_handle_trace_cov: transcript index out of range");
    if (f < 0) {
      need_sets = true;
      if (-(f + 1) >= h->groups[MMQ_GROUP_IDENTICAL].ngroups) return mmq_fail(h, MMQ_ERR_ARG, "mmq_handle_trace_cov: identical-set index out of range");
    }
  }
  if (need_sets) return mmq_fail(h, MMQ_ERR_ARG, "mmq_handle_trace_cov: identical-set features are read through mmq_get_group_trace + mmq_trace_cov (their trace is slot-major)");
  std::vector<int64_t> off((size_t)C);
  for (int64_t c = 0; c < C; ++c) off[(size_t)c] = (int64_t)features[c] * L;
  int64_t* off_dev = nullptr;
  void* ws = nullptr;
  double* dR = R_dev_out;
  const size_t rb = (size_t)C * (size_t)C * 8;
  auto cleanup = [&] {
    cudaStreamSynchronize(h->stream);
    mmq_cache_free(off_dev);
    mmq_cache_free(ws);
    if (dR != R_dev_out) mmq_cache_free(dR);
  };
#define COVH_TRY(call)                                                          \
  do {                                                                          \
    cudaError_t e__ = (call);                                                   \
    if (e__ != cudaSuccess) {                                                   \
      cleanup();                                                                \
      return mmq_cuda_fail(h, e__, #call, __FILE__, __LINE__);                  \
    }                                                                           \
  } while (0)
  COVH_TRY(mmq_cache_malloc(&off_dev, (size_t)C * 8));
  COVH_TRY(mmq_cache_malloc(&ws, cov_ws_bytes(L, C, nsplit)));
  if (!dR) COVH_TRY(mmq_cache_malloc(&dR, rb));
  COVH_TRY(cudaMemcpyAsync(off_dev, off.data(), (size_t)C * 8, cudaMemcpyHostToDevice, h->stream));
  const int rc = cov_run(h->trace, off_dev, 0, 1, L, C, nsplit, dR, ws, h->stream);
  if (rc != MMQ_OK) {
    cleanup();
    return mmq_fail(h, rc, g_cov_err);
  }
  if (R_out) COVH_TRY(cudaMemcpyAsync(R_out, dR, rb, cudaMemcpyDeviceToHost, h->stream));
  COVH_TRY(cudaStreamSynchronize(h->stream));
  cleanup();
  return MMQ_OK;
}

int mmq_mean_corrs_dev(const double* R_dev, const uint8_t* S_dev, int64_t C, int ns, const int32_t* ts_dev, int64_t nts, double sdpenalty,
                       double* V_dev, double* W_dev, void* cuda_stream) {
  if (!R_dev || !S_dev || !ts_dev || !V_dev || !W_dev) return cov_fail(MMQ_ERR_ARG, "mmq_mean_corrs_dev: NULL argument");
  if (C < 1 || ns < 1 || nts < 0) return cov_fail(MMQ_ERR_ARG, "mmq_mean_corrs_dev: bad sizes");
  if (nts == 0) return MMQ_OK;
  const int64_t pairs = nts * C;
  const int grid = (int)std::min<int64_t>((pairs + 255) / 256, 148 * 32);
  k_mean_corrs<<<grid, 256, 0, (cudaStream_t)cuda_stream>>>(R_dev, S_dev, C, ns, ts_dev, nts, sdpenalty, V_dev, W_dev);
  g_mmq_launches.fetch_add(1, std::memory_order_relaxed);
  COV_CUDA(cudaGetLastError());
  return MMQ_OK;
}

int mmq_mean_corrs(int device, const double* R, const uint8_t* S, int64_t C, int ns, const int32_t* ts, int64_t nts, double sdpenalty, double* V,
                   double* W) {
  if (!R || !S || !ts || !V || !W) return cov_fail(MMQ_ERR_ARG, "mmq_mean_corrs: NULL argument");
  if (C < 1 || ns < 1 || nts < 0) return cov_fail(MMQ_ERR_ARG, "mmq_mean_corrs: bad sizes");
  for (int64_t i = 0; i < nts; ++i)
    if (ts[i] < 0 || ts[i] >= C) return cov_fail(MMQ_ERR_ARG, "mmq_mean_corrs: row index out of range");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return cov_fail(MMQ_ERR_CUDA, "mmq_mean_corrs: no CUDA device (there is no CPU fallback)");
  COV_CUDA(cudaSetDevice(device));
  const size_t cc = (size_t)C * (size_t)C * 8;
  double *dR = nullptr, *dV = nullptr, *dW = nullptr;
  uint8_t* dS = nullptr;
  int32_t* dts = nullptr;
  cudaStream_t st = nullptr;
  auto cleanup = [&] {
    if (st) cudaStreamSynchronize(st);
    mmq_cache_free(dR);
    mmq_cache_free(dV);
    mmq_cache_free(dW);
    mmq_cache_free(dS);
    mmq_cache_free(dts);
    if (st) cudaStreamDestroy(st);
  };
  COV_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  COV_TRY(mmq_cache_malloc(&dR, cc * (size_t)ns));
  COV_TRY(mmq_cache_malloc(&dV, cc));
  COV_TRY(mmq_cache_malloc(&dW, cc));
  COV_TRY(mmq_cache_malloc(&dS, (size_t)C * (size_t)ns));
  COV_TRY(mmq_cache_malloc(&dts, (size_t)(nts > 0 ? nts : 1) * 4));
  COV_TRY(cudaMemcpyAsync(dR, R, cc * (size_t)ns, cudaMemcpyHostToDevice, st));
  COV_TRY(cudaMemcpyAsync(dV, V, cc, cudaMemcpyHostToDevice, st));
  COV_TRY(cudaMemcpyAsync(dW, W, cc, cudaMemcpyHostToDevice, st));
  COV_TRY(cudaMemcpyAsync(dS, S, (size_t)C * (size_t)ns, cudaMemcpyHostToDevice, st));
  COV_TRY(cudaMemcpyAsync(dts, ts, (size_t)nts * 4, cudaMemcpyHostToDevice, st));
  const int rc = mmq_mean_corrs_dev(dR, dS, C, ns, dts, nts, sdpenalty, dV, dW, st);
  if (rc == MMQ_OK) {
    COV_TRY(cudaMemcpyAsync(V, dV, cc, cudaMemcpyDeviceToHost, st));
    COV_TRY(cudaMemcpyAsync(W, dW, cc, cudaMemcpyDeviceToHost, st));
    COV_TRY(cudaStreamSynchronize(st));
  }
  cleanup();
  return rc;
}

} /* extern "C" */
