/* mmq_cls.cu — K2 for COLLAPSED shards (distinct hit classes with fragment counts k, the
 * reference's own representation: src/mmseq.cpp:395-441 builds it, :862-891 allocates it).
 *
 * The general kernel (k_alloc, mmq_core.cu) gives every class to one lane and lets that lane
 * run whatever mmq_alloc_row needs; with k between 1 and 10^5 and 2..30 members in one warp the
 * lanes diverge and the sweep is an order of magnitude away from the memory roofline.  The
 * plan below (built once in mmq_create) sorts the classes by what a sweep has to do for them:
 *
 *   d == 1              nothing: x = k is deterministic, summed once into seg_base[] (the Gamma
 *                       kernel restarts counts[] from it);
 *   k <= mmq_cat_limit(d),  the "small" set: k categorical draws, four per Philox block
 *   d <= MMQ_CLS_DMAX   (include/mmq_sampler.h).  A class becomes ceil(k / 64) SLOTS of at most 64
 *                       draws (16 blocks), so a class with thousands of fragments is shared out
 *                       between lanes.  Slots are ordered by (d, blocks, first member) and packed
 *                       in chunks of 32 — one slot per lane, member-major inside the chunk
 *                       (entry (j, lane) at chunk_base + 32 j + lane), so that every column load
 *                       of a warp is one fully used 128-byte line and no row pointers, no
 *                       shared-memory staging and no shuffles are needed.  A lane gathers its d
 *                       mu once, keeps the running sums S_j in registers and, per draw, counts
 *                       A_j += (u S_{d-1} < S_j); x_j = A_j - A_{j-1} (S is non-decreasing, so
 *                       that is "first j with target < S_j").  All lanes of a warp have the same
 *                       d and (almost always) the same number of blocks: no divergence.  The
 *                       order by first member keeps the mu gathers of a warp, and of the warps of
 *                       an SM, in neighbouring cache lines;
 *   the rest            (k > mmq_cat_limit(d): conditional-binomial chain; or more than 64 members) a
 *                       small sub-CSR handed to k_alloc, one class per warp, on a second stream.
 *
 * Two instances of the kernel (class sizes 2..8 in 64 registers, 9..16 and a generic loop up to 64
 * in 96) run concurrently on two streams.
 *
 * The integers are those of mmq_alloc_row on the same (seed, class id, sweep) — bit for bit
 * (tests/test_gpu_parity.py) — because the order of the floating-point sums is the same.
 *
 * Algorithmic HBM bytes per sweep: 4 B per packed column slot + 6 B per slot (draw count and slot
 * number in two bytes, low word of the class id) of the small set + the sub-CSR of the rest.
 */
#include <cub/cub.cuh>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "mmq_cls_plan.h"
#include "mmq_device.cuh"
#include "mmq_internal.h"

/* Philox block b of a class's own ALLOC stream */
__device__ __forceinline__ void cls_block(uint32_t (&wd)[4], uint32_t cid, uint32_t cid_hi, uint32_t sweep, uint32_t b, uint32_t seed) {
  wd[0] = cid; wd[1] = cid_hi; wd[2] = sweep; wd[3] = b;
  mmq_philox4x32_10(wd, seed, MMQ_STREAM_ALLOC);
}
/* the 32-bit word of a k == 1 class: word cid & 3 of the CAT stream's block cid >> 2 (shared by four classes) */
__device__ __forceinline__ uint32_t cls_word1(uint32_t cid, uint32_t cid_hi, uint32_t sweep, uint32_t seed) {
  uint32_t wd[4] = {(cid >> 2) | (cid_hi << 30), cid_hi >> 2, sweep, 0u};
  mmq_philox4x32_10(wd, seed, MMQ_STREAM_CAT);
  const uint32_t s = cid & 3u;
  return s == 0 ? wd[0] : s == 1 ? wd[1] : s == 2 ? wd[2] : wd[3];
}

/* One chunk: 32 slots of compile-time class size D, everything in registers.  A slot is a class
 * with its first block b0 and the number of draws kq <= 64 it makes (classes with more than 64
 * fragments occupy several slots). */
/* plan streams are read once per sweep and are as large as the L2: ask the L2 to evict them first, so that mu and counts stay
 * (measured on the config-2 shard: 8900 -> 9100 sweeps/s) */
__device__ __forceinline__ uint32_t ld_plan_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile(
      "{\n\t"
      ".reg .b64 pol;\n\t"
      "createpolicy.fractional.L2::evict_first.b64 pol, 1.0;\n\t"
      "ld.global.nc.L2::cache_hint.u32 %0, [%1], pol;\n\t"
      "}\n"
      : "=r"(v)
      : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ld_plan_u16(const uint16_t* p) {
  uint16_t v;
  asm volatile(
      "{\n\t"
      ".reg .b64 pol;\n\t"
      "createpolicy.fractional.L2::evict_first.b64 pol, 1.0;\n\t"
      "ld.global.nc.L2::cache_hint.u16 %0, [%1], pol;\n\t"
      "}\n"
      : "=h"(v)
      : "l"(p));
  return v;
}
__device__ __forceinline__ int32_t ld_plan(const int32_t* p) {
  int32_t v;
  asm volatile(
      "{\n\t"
      ".reg .b64 pol;\n\t"
      "createpolicy.fractional.L2::evict_first.b64 pol, 1.0;\n\t"
      "ld.global.nc.L2::cache_hint.s32 %0, [%1], pol;\n\t"
      "}\n"
      : "=r"(v)
      : "l"(p));
  return v;
}
template <int D>
__device__ __forceinline__ void cls_chunk(const int32_t* __restrict__ pc, int kq, uint32_t b0, uint32_t cid, uint32_t cid_hi,
                                          const double* __restrict__ mu, int32_t* __restrict__ counts, uint32_t seed,
                                          uint32_t sweep, int lane) {
  /* the columns are not kept: the few that receive fragments are re-read (L1 hits) at the end,
   * which leaves the registers to the running sums and buys resident warps */
  double S[D];
#pragma unroll
  for (int j = 0; j < D; ++j) S[j] = mu[ld_plan(pc + 32 * j)];
#pragma unroll
  for (int j = 1; j < D; ++j) S[j] = S[j - 1] + S[j];
  const double norm = S[D - 1];
  int A[D - 1];
#pragma unroll
  for (int j = 0; j < D - 1; ++j) A[j] = 0;
  const int nb = (kq + 3) >> 2;
  const int nbmax = __reduce_max_sync(0xffffffffu, nb);
#pragma unroll 1
  for (int b = 0; b < nbmax; ++b) {
    if (b < nb) {
      uint32_t wd[4];
      cls_block(wd, cid, cid_hi, sweep, b0 + (uint32_t)b, seed);
      const int nd = kq - 4 * b; /* draws of this block: min(4, nd) */
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const double target = mmq_uniform32(wd[r]) * norm;
        const bool live = r < nd;
#pragma unroll
        for (int j = 0; j < D - 1; ++j) A[j] += (live && target < S[j]) ? 1 : 0;
      }
    }
  }
  int prev = 0;
#pragma unroll
  for (int j = 0; j < D - 1; ++j) {
    const int x = A[j] - prev;
    prev = A[j];
    if (x) atomicAdd(counts + __ldg(pc + 32 * j), x);
  }
  if (kq - prev) atomicAdd(counts + __ldg(pc + 32 * (D - 1)), kq - prev);
}

/* any class size: members are re-read (L1/L2 hits) for every block of four draws */
__device__ __noinline__ void cls_chunk_any(const int32_t* __restrict__ pc, int D, int kq, uint32_t b0, uint32_t cid, uint32_t cid_hi,
                                           const double* __restrict__ mu, int32_t* __restrict__ counts, uint32_t seed,
                                           uint32_t sweep) {
  double norm = 0.0;
  {
    int j = 0;
    for (; j + 4 <= D; j += 4) { /* four independent gathers in flight; the sum stays left to right */
      const double a0 = mu[pc[32 * j]], a1 = mu[pc[32 * (j + 1)]], a2 = mu[pc[32 * (j + 2)]], a3 = mu[pc[32 * (j + 3)]];
      norm += a0; norm += a1; norm += a2; norm += a3;
    }
    for (; j < D; ++j) norm += mu[pc[32 * j]];
  }
  const int nb = (kq + 3) >> 2;
  for (int b = 0; b < nb; ++b) {
    uint32_t wd[4];
    cls_block(wd, cid, cid_hi, sweep, b0 + (uint32_t)b, seed);
    const int nd = min(4, kq - 4 * b);
    double t[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) t[r] = mmq_uniform32(wd[r]) * norm;
    double s = 0.0;
    int prev = 0;
    auto member = [&](int j, int32_t cj, double pj) {
      s += pj;
      int a = 0;
#pragma unroll
      for (int r = 0; r < 4; ++r) a += (r < nd && t[r] < s) ? 1 : 0;
      if (j == D - 1) a = nd;
      if (a - prev) atomicAdd(counts + cj, a - prev);
      prev = a;
    };
    int j = 0;
    for (; j + 4 <= D && prev < nd; j += 4) {
      const int32_t c0 = pc[32 * j], c1 = pc[32 * (j + 1)], c2 = pc[32 * (j + 2)], c3 = pc[32 * (j + 3)];
      const double a0 = mu[c0], a1 = mu[c1], a2 = mu[c2], a3 = mu[c3];
      member(j, c0, a0); member(j + 1, c1, a1); member(j + 2, c2, a2); member(j + 3, c3, a3);
    }
    for (; j < D && prev < nd; ++j) { /* prev == nd: every draw of the block has found its member */
      const int32_t cj = pc[32 * j];
      member(j, cj, mu[cj]);
    }
  }
}

/* LO: the instance for class sizes 2..MMQ_CLS_DLO (chunks [0, total_chunks) are all such runs);
 * otherwise sizes above MMQ_CLS_DLO. */
/* Where a chunk lies and its class size come from one 8-byte descriptor per chunk (fetched a chunk ahead like the slot
 * metadata): no shared memory, no run lookup, no 64-bit multiply. */
template <bool LO, int MINB>
__global__ void __launch_bounds__(MMQ_CLS_WARPS * 32, MINB)
k_alloc_cls(int chunk_begin, int chunk_end, const int32_t* __restrict__ pcol, const uint16_t* __restrict__ pk, const uint32_t* __restrict__ pcid,
            const unsigned long long* __restrict__ cdesc, uint32_t cid_hi, const double* __restrict__ mu, int32_t* __restrict__ counts,
            uint32_t seed, uint32_t sweep, const uint32_t* __restrict__ sweep_base) {
  if (sweep_base) sweep += *sweep_base; /* CUDA-graph replays: the sweep counter lives on the device */
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * MMQ_CLS_WARPS;
  const int count = chunk_end - chunk_begin;
  /* the long classes (the generic path above all) first in the 9..16 instance: they must not be the tail of the launch */
  auto chunk_of = [&](int i) { return LO ? chunk_begin + i : chunk_end - 1 - i; };
  int i = blockIdx.x * MMQ_CLS_WARPS + (threadIdx.x >> 5);
  /* draw counts and class ids are fetched one chunk ahead (two registers): their latency is off the critical path */
  uint32_t meta_n = 0, cid_n = 0;
  unsigned long long desc_n = 0ull;
  if (i < count) {
    meta_n = ld_plan_u16(pk + (int64_t)chunk_of(i) * 32 + lane);
    cid_n = ld_plan_u32(pcid + (int64_t)chunk_of(i) * 32 + lane);
    desc_n = cdesc[chunk_of(i)];
  }
  for (; i < count; i += nwarps) {
    const int D = (int)(desc_n & 0xffull);
    const int32_t* pc = pcol + (desc_n >> 8) + lane;
    const uint32_t meta = meta_n; /* draws of the slot | slot number within its class << 8 */
    const uint32_t cid = cid_n;
    if (i + nwarps < count) {
      meta_n = ld_plan_u16(pk + (int64_t)chunk_of(i + nwarps) * 32 + lane);
      cid_n = ld_plan_u32(pcid + (int64_t)chunk_of(i + nwarps) * 32 + lane);
      desc_n = cdesc[chunk_of(i + nwarps)];
    }
    const int kq = (int)(meta & 0xffu);
    const uint32_t b0 = (meta >> 8) * (uint32_t)(MMQ_CLS_GROUP(D) / 4);
#define MMQ_CLS_CASE(DD) case DD: cls_chunk<DD>(pc, kq, b0, cid, cid_hi, mu, counts, seed, sweep, lane); break;
    if (LO) {
      switch (D) {
        MMQ_CLS_CASE(2) MMQ_CLS_CASE(3) MMQ_CLS_CASE(4) MMQ_CLS_CASE(5) MMQ_CLS_CASE(6) MMQ_CLS_CASE(7) MMQ_CLS_CASE(8)
        default: break;
      }
    } else {
      switch (D) {
        MMQ_CLS_CASE(9) MMQ_CLS_CASE(10) MMQ_CLS_CASE(11) MMQ_CLS_CASE(12) MMQ_CLS_CASE(13) MMQ_CLS_CASE(14)
        MMQ_CLS_CASE(15) MMQ_CLS_CASE(16)
        default: cls_chunk_any(pc, D, kq, b0, cid, cid_hi, mu, counts, seed, sweep); break;
      }
    }
#undef MMQ_CLS_CASE
  }
}

/* ---- single-fragment classes (k == 1): 64 % of the classes and 70 % of the entries of the config-2 sample ----
 * Their chunks form the tail of the plan ([chunks_gen, chunks)) and have a kernel of their own: one categorical draw
 * per class needs the running sums only (no per-member counters, no block loop), so every class size up to 16 fits
 * 56 registers — twice the resident warps of the general 9..16 instance, which is what hides the column load -> mu
 * gather -> sum chain of two memory latencies. */
template <int D>
__device__ __forceinline__ void cls1_chunk(const int32_t* __restrict__ pc, bool live, uint32_t cid, uint32_t cid_hi, const double* __restrict__ mu,
                                           int32_t* __restrict__ counts, uint32_t seed, uint32_t sweep, int lane) {
  double S[D];
#pragma unroll
  for (int j = 0; j < D; ++j) S[j] = mu[ld_plan(pc + 32 * j)];
  const uint32_t word = cls_word1(cid, cid_hi, sweep, seed); /* independent of the loads in flight */
#pragma unroll
  for (int j = 1; j < D; ++j) S[j] = S[j - 1] + S[j];
  const double target = mmq_uniform32(word) * S[D - 1];
  int chosen = D - 1;
#pragma unroll
  for (int j = 0; j < D - 1; ++j) chosen -= (target < S[j]) ? 1 : 0; /* S is non-decreasing: first j with target < S_j */
  cat_red(counts, live ? __ldg(pc + 32 * chosen) : -1, lane);
}
/* any class size: the members are read twice (the second time from L1) */
__device__ __noinline__ void cls1_chunk_any(const int32_t* __restrict__ pc, int D, bool live, uint32_t cid, uint32_t cid_hi,
                                            const double* __restrict__ mu, int32_t* __restrict__ counts, uint32_t seed, uint32_t sweep, int lane) {
  double norm = 0.0;
  for (int j = 0; j < D; ++j) norm += mu[pc[32 * j]];
  const double target = mmq_uniform32(cls_word1(cid, cid_hi, sweep, seed)) * norm;
  double s = 0.0;
  int chosen = D - 1;
  for (int j = 0; j < D - 1; ++j) {
    s += mu[pc[32 * j]];
    if (target < s) { chosen = j; break; }
  }
  cat_red(counts, live ? pc[32 * chosen] : -1, lane);
}
__global__ void __launch_bounds__(MMQ_CLS_WARPS * 32, 9)
k_alloc_cls1(int chunk_begin, int chunk_end, const int32_t* __restrict__ pcol, const uint16_t* __restrict__ pk, const uint32_t* __restrict__ pcid,
             const unsigned long long* __restrict__ cdesc, uint32_t cid_hi, const double* __restrict__ mu, int32_t* __restrict__ counts,
             uint32_t seed, uint32_t sweep, const uint32_t* __restrict__ sweep_base) {
  if (sweep_base) sweep += *sweep_base;
  const int lane = threadIdx.x & 31;
  const int nwarps = gridDim.x * MMQ_CLS_WARPS;
  const int count = chunk_end - chunk_begin;
  /* the largest classes first (the plan orders the chunks by ascending size) */
  auto chunk_of = [&](int i) { return chunk_end - 1 - i; };
  int i = blockIdx.x * MMQ_CLS_WARPS + (threadIdx.x >> 5);
  uint32_t meta_n = 0, cid_n = 0;
  unsigned long long desc_n = 0ull;
  if (i < count) {
    meta_n = ld_plan_u16(pk + (int64_t)chunk_of(i) * 32 + lane);
    cid_n = ld_plan_u32(pcid + (int64_t)chunk_of(i) * 32 + lane);
    desc_n = cdesc[chunk_of(i)];
  }
  for (; i < count; i += nwarps) {
    const int D = (int)(desc_n & 0xffull);
    const int32_t* pc = pcol + (desc_n >> 8) + lane;
    const bool live = (meta_n & 0xffu) != 0u; /* padding lanes make no draw */
    const uint32_t cid = cid_n;
    if (i + nwarps < count) { /* metadata one chunk ahead: its latency is off the critical path */
      meta_n = ld_plan_u16(pk + (int64_t)chunk_of(i + nwarps) * 32 + lane);
      cid_n = ld_plan_u32(pcid + (int64_t)chunk_of(i + nwarps) * 32 + lane);
      desc_n = cdesc[chunk_of(i + nwarps)];
    }
#define MMQ_CLS1_CASE(DD) case DD: cls1_chunk<DD>(pc, live, cid, cid_hi, mu, counts, seed, sweep, lane); break;
    switch (D) {
      MMQ_CLS1_CASE(2) MMQ_CLS1_CASE(3) MMQ_CLS1_CASE(4) MMQ_CLS1_CASE(5) MMQ_CLS1_CASE(6) MMQ_CLS1_CASE(7) MMQ_CLS1_CASE(8)
      MMQ_CLS1_CASE(9) MMQ_CLS1_CASE(10) MMQ_CLS1_CASE(11) MMQ_CLS1_CASE(12) MMQ_CLS1_CASE(13) MMQ_CLS1_CASE(14) MMQ_CLS1_CASE(15)
      MMQ_CLS1_CASE(16)
      default: cls1_chunk_any(pc, D, live, cid, cid_hi, mu, counts, seed, sweep, lane); break;
    }
#undef MMQ_CLS1_CASE
  }
}

/* The chain set: classes with more than mmq_cat_limit(d) fragments — the multinomial by conditional binomials
 * (gsl_ran_multinomial, src/mmseq.cpp:880), O(d) binomials per class whatever k is, in the balanced splitting order of
 * mmq_alloc_chain (include/mmq_sampler.h): ceil(log2 d) levels, the binomials of a level independent of each other.
 * One class per lane of the block's first warps, 32 classes of equal size per chunk (member-major like the small set, so
 * every column load of a warp is one 128-byte line), longest classes first.  Three instances, one per splitting depth
 * (class sizes 5..16, 3..4 and 2), each over its contiguous chunk range: 91 % of the chain classes of the config-2
 * sample need one or two levels and no longer carry the shared memory and the level loop of the 16-member classes.
 *
 * A binomial is a rejection sampler (BTRS above a mean of 10) or an inversion loop of data-dependent length (BINV
 * below): with every lane running its own, a warp pays for the union of the regimes and for its slowest lane — the first
 * version of this kernel (a left-to-right chain per lane) kept 5.5 of 32 lanes busy (ncu, round 2) and took 117 us for
 * the 49k classes of the config-2 sample.  An attempt being a pure function of (class, sweep, node, attempt number),
 * the block instead QUEUES the binomials of a level in shared memory by regime and runs each queue densely: the BTRS
 * attempts in rounds, MMQ_CHAIN_SPEC attempts of every open draw side by side (the lowest accepted one counts), the
 * rejected ones re-queued; the inversions on the remaining threads of the first round.  Same integers as the CPU
 * replay's mmq_alloc_chain. */
#define MMQ_CHAIN_THREADS 256 /* threads per block */
#define MMQ_CHAIN_SPEC 2      /* attempts of an open BTRS draw evaluated side by side per round */
/* a queued draw, p <= 1/2; owner: class slot | node << 8 | flip << 16 (x = n - x' for p > 1/2).  BTRS draws fill the
 * queue from the front, inversions from the back.  (Keeping each draw's BTRS / BINV constants here instead of
 * recomputing them per attempt grows an entry from 16 to 72 bytes and did not pay: DESIGN.md, "Tried and measured out".) */
struct chain_req { double p; int n, owner; };
/* One instance per splitting depth: LV levels at most (class sizes up to 2^LV), C classes per block pass (the lanes of
 * the first C / 32 warps own them; every warp works in the dense phases).  The arrays are sized by the deepest class the
 * instance serves, so the shallow classes, most of the chain set, do not carry the footprint of the deep ones. */
template <int LV, int C>
struct chain_smem {
  static constexpr int NM = 1 << LV;         /* members of a class */
  static constexpr int NN = 1 << (LV - 1);   /* nodes of a class on its last level */
  static constexpr int QCAP = C * NN;        /* draws of a level */
  double p[NM][C];                           /* mu of the members */
  int cnt[NM][C];                            /* fragments of the nodes of the current level */
  int res[NN][C];                            /* left-half counts drawn on this level */
  chain_req q[QCAP];                         /* BTRS draws of this level from the front, inversions from the back */
  int open[2][QCAP];                         /* BTRS draws not yet accepted (indices into q), ping-pong over rounds */
  int att[MMQ_CHAIN_THREADS];                /* this pass's attempts: x, or -1 rejected */
  uint32_t cid[C];
  int d[C];                                  /* class size, 0 for a padding lane */
  int n[4];                                  /* BTRS draws, inversions, open[0], open[1] */
  int dmax;
};
template <int LV, int C, int MINB>
__global__ void __launch_bounds__(MMQ_CHAIN_THREADS, MINB)
k_alloc_chain(int chunk_begin, int chunk_end, const int32_t* __restrict__ pcol, const int32_t* __restrict__ ck, const uint32_t* __restrict__ ccid,
              const unsigned long long* __restrict__ cdesc, uint32_t cid_hi, const double* __restrict__ mu,
              int32_t* __restrict__ counts, uint32_t seed, uint32_t sweep, const uint32_t* __restrict__ sweep_base) {
  using SM = chain_smem<LV, C>;
  constexpr int QCAP = SM::QCAP;
  static_assert(C % 32 == 0 && C <= MMQ_CHAIN_THREADS && C <= 256, "class slots: owner warps, 8 bits of the owner word");
  extern __shared__ __align__(16) unsigned char chain_raw[];
  SM& S = *reinterpret_cast<SM*>(chain_raw);
  if (sweep_base) sweep += *sweep_base;
  const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
  constexpr int CW = C / 32;
  const bool owner_warp = wib < CW;
  for (int chunk0 = chunk_begin + blockIdx.x * CW; chunk0 < chunk_end; chunk0 += gridDim.x * CW) {
    const int chunk = chunk0 + wib;
    int D = 0;
    const int32_t* pc = pcol;
    int kv = 0;
    uint32_t cid = 0;
    if (owner_warp && chunk < chunk_end) {
      const unsigned long long desc = cdesc[chunk];
      D = (int)(desc & 0xffull);
      pc = pcol + (desc >> 8) + lane;
      kv = ck[(int64_t)chunk * 32 + lane];
      cid = ccid[(int64_t)chunk * 32 + lane];
    }
    if (kv <= 0) D = 0; /* padding lane */
    __syncthreads();    /* the previous pass is done with S */
    if (tid == 0) S.dmax = 0;
    if (owner_warp) {
      S.cid[tid] = cid;
      S.d[tid] = D;
      S.cnt[0][tid] = kv;
      for (int j = 0; j < D; ++j) S.p[j][tid] = mu[ld_plan(pc + 32 * j)];
    }
    __syncthreads();
    {
      const int dm = __reduce_max_sync(0xffffffffu, D);
      if (lane == 0 && dm > 0) atomicMax(&S.dmax, dm);
    }
    __syncthreads();
    int levels = 0;
    while ((1 << levels) < S.dmax) ++levels;
    for (int L = 0; L < LV && L < levels; ++L) {
      const int nodes = 1 << L;
      if (tid < 4) S.n[tid] = 0;
      __syncthreads();
      /* ---- the nodes of this level: what has to be drawn?  The (class, node) pairs are spread over all threads, 32
       * classes of one node per warp */
      for (int w0 = 0; w0 < C * nodes; w0 += MMQ_CHAIN_THREADS) {
        const int w = w0 + tid, c = w % C, i = w / C;
        bool pending = false, btrs = false;
        double pr = 0.0;
        int n = 0;
        const int dc = w < C * nodes ? S.d[c] : 0;
        if (dc > 0) {
          const int lo = MMQ_NODE_LO(i, L, dc), hi = MMQ_NODE_LO(i + 1, L, dc);
          n = S.cnt[i][c];
          if (hi - lo >= 2) {
            const int mid = MMQ_NODE_LO(2 * i + 1, L + 1, dc);
            if (mid == lo) S.res[i][c] = 0;
            else if (mid == hi) S.res[i][c] = n;
            else if (n == 0) S.res[i][c] = 0;
            else {
              double left = 0.0, right = 0.0;
              for (int j = lo; j < mid; ++j) left += S.p[j][c];
              for (int j = mid; j < hi; ++j) right += S.p[j][c];
              const double tot = left + right;
              pr = tot > 0.0 ? left / tot : 0.0;
              if (pr > 1.0) pr = 1.0;
              const double ph = pr > 0.5 ? 1.0 - pr : pr;
              if (n >= 2 && pr > 0.0 && pr < 1.0) {
                pending = true;
                btrs = (double)n * ph >= MMQ_BINV_MEAN;
              } else { /* p == 0 or 1, or a single fragment: mmq_binomial's first cases, here rather than queued */
                int x = pr >= 1.0 ? n : 0;
                if (n == 1 && pr > 0.0 && pr < 1.0) {
                  uint32_t wd[4];
                  cls_block(wd, S.cid[c], cid_hi, sweep, MMQ_CHAIN_BLOCK(nodes + i), seed);
                  x = mmq_uniform52(wd[0], wd[1]) < pr ? 1 : 0;
                }
                S.res[i][c] = x;
              }
            }
          }
        }
        const int owner = c | (i << 8) | (pr > 0.5 ? 1 << 16 : 0);
        const double ph = pr > 0.5 ? 1.0 - pr : pr;
        const int pt = queue_slot(&S.n[0], pending && btrs, lane);
        if (pt >= 0) { S.q[pt] = chain_req{ph, n, owner}; S.open[1][pt] = pt; }
        const int pi = queue_slot(&S.n[1], pending && !btrs, lane);
        if (pi >= 0) S.q[QCAP - 1 - pi] = chain_req{ph, n, owner};
      }
      __syncthreads();
      /* ---- round r: attempts SPEC r .. SPEC r + SPEC - 1 of every open BTRS draw, one per thread; in round 0 the
       * threads after them do the inversions (mean below 10) */
      const uint32_t heap = (uint32_t)nodes;
      const int ni = S.n[1];
      int nopen = S.n[0];
      uint32_t rr = 0; /* rounds: open[(rr + 1) & 1] is read, open[rr & 1] written */
      for (uint32_t r = 0; nopen > 0 || (r == 0 && ni > 0); ++r, ++rr) {
        /* attempts per open draw this round (speculation: only the lowest accepted attempt counts, so the result does not
         * depend on it): measured on the config-2 sample, 2 is the best trade between rounds and issue slots taken from the
         * concurrent class kernels (4 with 32-class blocks: 11.0 M instead of 7.1 M warp instructions, the sweep 15 % slower) */
        const int spec = MMQ_CHAIN_SPEC;
        const int work = nopen * spec, extra = r == 0 ? ni : 0;
        if (tid == 0) S.n[2 + (rr & 1)] = 0;
        for (int w0 = 0; w0 < work + extra; w0 += MMQ_CHAIN_THREADS) { /* passes of one work item per thread */
          const int wi = w0 + tid;
          if (wi < work) {
            const chain_req q = S.q[S.open[(rr + 1) & 1][wi / spec]];
            const int owner = q.owner;
            mmq_rng g;
            mmq_rng_init(&g, seed, MMQ_STREAM_ALLOC, ((uint64_t)cid_hi << 32) | S.cid[owner & 0xff], sweep);
            int64_t xb = 0;
            const bool ok = mmq_btrs_attempt(&g, MMQ_CHAIN_BLOCK(heap + ((owner >> 8) & 0xff)) + r + (uint32_t)(wi % spec), mmq_btrs_setup(q.n, q.p), &xb) != 0;
            S.att[tid] = ok ? (int)xb : -1;
          } else if (wi < work + extra) {
            const chain_req q = S.q[QCAP - 1 - (wi - work)];
            const int owner = q.owner, n = q.n;
            mmq_rng g;
            mmq_rng_init(&g, seed, MMQ_STREAM_ALLOC, ((uint64_t)cid_hi << 32) | S.cid[owner & 0xff], sweep);
            const uint32_t b0 = MMQ_CHAIN_BLOCK(heap + ((owner >> 8) & 0xff));
            int64_t x = 0;
            const mmq_binv_par bt = mmq_binv_setup(n, q.p);
            for (uint32_t att = 0; !mmq_binv_attempt(&g, b0 + att, n, bt, &x); ++att) { }
            S.res[(owner >> 8) & 0xff][owner & 0xff] = (owner >> 16) ? n - (int)x : (int)x;
          }
          __syncthreads();
          /* the first thread of each draw of this pass takes the lowest accepted attempt, or re-queues the draw */
          if ((w0 + (tid & ~31)) < work) {
            bool again = false;
            int req = 0;
            if (wi < work && tid % spec == 0) {
              req = S.open[(rr + 1) & 1][wi / spec];
              int xa = -1;
              for (int sp = spec - 1; sp >= 0; --sp) if (S.att[tid + sp] >= 0) xa = S.att[tid + sp];
              if (xa >= 0) {
                const chain_req q = S.q[req];
                S.res[(q.owner >> 8) & 0xff][q.owner & 0xff] = (q.owner >> 16) ? q.n - xa : xa;
              } else again = true;
            }
            const int pos = queue_slot(&S.n[2 + (rr & 1)], again, lane);
            if (pos >= 0) S.open[rr & 1][pos] = req;
          }
          __syncthreads();
        }
        r += (uint32_t)spec - 1u; /* the loop adds one more: r = attempts made so far */
        nopen = S.n[2 + (rr & 1)];
        __syncthreads();
      }
      /* ---- split: children 2 i and 2 i + 1 of node i (in place, from the top: 2 i >= i) */
      if (owner_warp && D > 0) {
        for (int i = nodes - 1; i >= 0; --i) {
          const int lo = MMQ_NODE_LO(i, L, D), hi = MMQ_NODE_LO(i + 1, L, D);
          const int n = S.cnt[i][tid];
          int nl = 0;
          if (hi - lo >= 2) nl = S.res[i][tid];
          else if (hi - lo == 1) nl = MMQ_NODE_LO(2 * i + 1, L + 1, D) == hi ? n : 0; /* a single member: it stays in the half that contains it */
          S.cnt[2 * i][tid] = nl;
          S.cnt[2 * i + 1][tid] = n - nl;
        }
      }
    }
    __syncthreads();
    if (owner_warp && D > 0) {
      const int nodes = 1 << levels;
      for (int i = 0; i < nodes; ++i) {
        const int lo = MMQ_NODE_LO(i, levels, D), hi = MMQ_NODE_LO(i + 1, levels, D);
        if (hi > lo) {
          const int x = S.cnt[i][tid];
          if (x != 0) atomicAdd(counts + __ldg(pc + 32 * lo), x);
        }
      }
    }
  }
}

__global__ void k_iota_u32(uint32_t* __restrict__ v, int64_t count) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) v[i] = (uint32_t)i;
}
__global__ void k_fill_i32_cls(int32_t* __restrict__ p, int64_t count, int32_t v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void k_cls_singletons(const int32_t* __restrict__ col1, const int32_t* __restrict__ k1, int64_t count,
                                 int32_t* __restrict__ base) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
    atomicAdd(base + col1[i], k1[i]);
}

/* ------------------------------------------------------------------ host */

template <typename T>
static int cls_upload(mmq_handle* h, T** dst, const std::vector<T>& v) {
  int rc = mmq_dev_alloc(h, (void**)dst, sizeof(T) * std::max<size_t>(v.size(), 1));
  if (rc) return rc;
  if (!v.empty()) MMQ_CUDA(h, cudaMemcpyAsync(*dst, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice, h->stream));
  return MMQ_OK;
}

/* ------------------------------------------------------------------ the plan, built on the device
 * The host builder of mmq_cls_plan.h (kept: the CPU tests replay it, MMQ_CLS_HOST_PLAN=1 selects it) takes ~100 ms for
 * the 3.6 M classes of the config-2 sample plus the upload of 124 MB from pageable memory — more than the 320 sweeps of
 * a default bench run.  The CSR is on the device already, so the same plan is made there:
 *   1. k_clsb_classify: per class its set, its number of slots; singletons are summed into seg_base[];
 *   2. exclusive scan of the slot counts; k_clsb_slots writes one 64-bit sort key per slot
 *      (pseudo size | 16 - Philox blocks | first member) — the chain set sorts behind the small set by descending size;
 *   3. one stable radix sort (cub); run boundaries of equal pseudo size come back to the host (<= 146 integers), which
 *      lays out runs and chunks;
 *   4. k_clsb_fill scatters columns, draw counts and class ids into the member-major chunks.
 * The few classes with more than MMQ_CLS_DMAX members (or above the chain kernel's size) are listed by the host. */
#define MMQ_CLSB_DPC0 MMQ_CLS_DP_END                         /* pseudo sizes of the chain set: DPC0 + (CHAIN_DMAX - d) */
#define MMQ_CLSB_NDP (MMQ_CLS_DP_END + MMQ_CLS_CHAIN_DMAX + 1)
struct clsb_run { long long e0; int first, chunk0, d, pad; }; /* per pseudo size: column offset, first sorted slot, first chunk */

__device__ __forceinline__ int clsb_set_of(int64_t d, int64_t kv) { /* 0 nothing to draw, 1 small, 2 chain, 3 rest */
  if (d == 1 || kv <= 0) return 0;
  if (d <= MMQ_CLS_DMAX && kv <= mmq_cat_limit((int)d)) return 1;
  return d <= MMQ_CLS_CHAIN_DMAX ? 2 : 3;
}
__global__ void k_clsb_classify(const int64_t* __restrict__ rp, const int32_t* __restrict__ col, const int32_t* __restrict__ kk,
                                const int64_t* __restrict__ class_id, int64_t cid_base, uint32_t cid_hi, int64_t m,
                                int32_t* __restrict__ nslots, int32_t* __restrict__ base, int* __restrict__ info) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t d = rp[i + 1] - rp[i], kv = kk[i];
    const uint64_t cid = (uint64_t)(class_id ? class_id[i] : cid_base + i);
    if ((uint32_t)(cid >> 32) != cid_hi || kv < 0) atomicOr(info, 1); /* the plan does not apply */
    const int set = clsb_set_of(d, kv);
    int ns = 0;
    if (set == 0) { if (d == 1 && kv > 0) { atomicAdd(base + col[rp[i]], (int32_t)kv); atomicOr(info + 1, 1); } }
    else if (set == 1) ns = kv == 1 ? 1 : (int)((kv + MMQ_CLS_GROUP(d) - 1) / MMQ_CLS_GROUP(d));
    else if (set == 2) ns = 1;
    else { atomicAdd(info + 2, 1); }
    nslots[i] = ns;
  }
}
__global__ void k_clsb_slots(const int64_t* __restrict__ rp, const int32_t* __restrict__ col, const int32_t* __restrict__ kk,
                             const int32_t* __restrict__ nslots, const int32_t* __restrict__ off, int64_t m,
                             unsigned long long* __restrict__ keys, uint32_t* __restrict__ slot_class, uint8_t* __restrict__ slot_no) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int ns = nslots[i];
    if (ns == 0) continue;
    const int64_t d = rp[i + 1] - rp[i], kv = kk[i];
    const unsigned long long first = (unsigned long long)(uint32_t)col[rp[i]];
    const int set = clsb_set_of(d, kv);
    for (int s = 0; s < ns; ++s) {
      unsigned long long dp, q;
      if (set == 2) { dp = MMQ_CLSB_DPC0 + (MMQ_CLS_CHAIN_DMAX - d); q = 0; }
      else if (kv == 1) { dp = MMQ_CLS_DP1(d); q = 16; }
      else {
        const int64_t grp = MMQ_CLS_GROUP(d);
        const int64_t draws = (s + 1) * grp <= kv ? grp : kv - s * grp;
        dp = (unsigned long long)d; q = (unsigned long long)(16 - (draws + 3) / 4);
      }
      const int64_t slot = (int64_t)off[i] + s;
      keys[slot] = (dp << 36) | (q << 31) | first;
      slot_class[slot] = (uint32_t)i;
      slot_no[slot] = (uint8_t)s;
    }
  }
}
/* first[dp] = first sorted position with that pseudo size */
__global__ void k_clsb_bounds(const unsigned long long* __restrict__ keys, int64_t S, int* __restrict__ first) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < S; p += (int64_t)gridDim.x * blockDim.x) {
    const int dp = (int)(keys[p] >> 36);
    if (p == 0 || (int)(keys[p - 1] >> 36) != dp) first[dp] = (int)p;
  }
}
__global__ void k_clsb_fill(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ vals, int64_t S,
                            const clsb_run* __restrict__ runs, const uint32_t* __restrict__ slot_class, const uint8_t* __restrict__ slot_no,
                            const int64_t* __restrict__ rp, const int32_t* __restrict__ col, const int32_t* __restrict__ kk,
                            const int64_t* __restrict__ class_id, int64_t cid_base, int32_t* __restrict__ pcol, uint16_t* __restrict__ pk,
                            uint32_t* __restrict__ pcid, int32_t* __restrict__ c_pcol, int32_t* __restrict__ c_k, uint32_t* __restrict__ c_cid) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < S; p += (int64_t)gridDim.x * blockDim.x) {
    const int dp = (int)(keys[p] >> 36);
    const clsb_run R = runs[dp];
    const uint32_t slot = vals[p];
    const int64_t i = slot_class[slot];
    const int sno = slot_no[slot];
    const int li = (int)p - R.first, d = R.d;
    const int64_t chunk = R.chunk0 + (li >> 5);
    const int32_t* src = col + rp[i];
    const uint32_t cid = (uint32_t)(class_id ? class_id[i] : cid_base + i);
    const int64_t kv = kk[i];
    if (dp >= MMQ_CLSB_DPC0) {
      int32_t* dst = c_pcol + R.e0 + (int64_t)(li >> 5) * 32 * d + (li & 31);
      for (int j = 0; j < d; ++j) dst[32 * j] = src[j];
      c_k[chunk * 32 + (li & 31)] = (int32_t)kv;
      c_cid[chunk * 32 + (li & 31)] = cid;
    } else {
      int32_t* dst = pcol + R.e0 + (int64_t)(li >> 5) * 32 * d + (li & 31);
      for (int j = 0; j < d; ++j) dst[32 * j] = src[j];
      const int64_t grp = MMQ_CLS_GROUP(d);
      const int64_t draws = kv == 1 ? 1 : ((sno + 1) * grp <= kv ? grp : kv - sno * grp);
      pk[chunk * 32 + (li & 31)] = (uint16_t)(draws | (sno << 8));
      pcid[chunk * 32 + (li & 31)] = cid;
    }
  }
}
__global__ void k_clsb_desc(const clsb_run* __restrict__ runs, int ndp, const int* __restrict__ nchunks, unsigned long long* __restrict__ cdesc,
                            unsigned long long* __restrict__ c_desc) {
  const int dp = blockIdx.x;
  if (dp >= ndp || nchunks[dp] == 0) return;
  const clsb_run R = runs[dp];
  unsigned long long* out = dp >= MMQ_CLSB_DPC0 ? c_desc : cdesc;
  for (int c = threadIdx.x; c < nchunks[dp]; c += blockDim.x)
    out[R.chunk0 + c] = ((unsigned long long)(R.e0 + (long long)c * 32 * R.d) << 8) | (unsigned long long)R.d;
}

/* Returns MMQ_OK with h->cls_ready set, or with it unset when the plan does not apply (the general kernel then). */
static int cls_plan_device(mmq_handle* h, const mmq_problem* p) {
  const int64_t m = h->m, n = h->n;
  const uint64_t cid0 = (uint64_t)(p->class_id ? p->class_id[0] : p->class_id_base);
  const uint32_t cid_hi = (uint32_t)(cid0 >> 32);
  int rc;
  int32_t *nslots = nullptr, *off = nullptr;
  unsigned long long *keys = nullptr, *keys2 = nullptr;
  uint32_t *vals = nullptr, *vals2 = nullptr, *slot_class = nullptr;
  uint8_t* slot_no = nullptr;
  int *info = nullptr, *first = nullptr, *nch_dev = nullptr;
  clsb_run* runs_dev = nullptr;
  void* temp = nullptr;
  auto cleanup = [&] {
    cudaStreamSynchronize(h->stream); /* the temporaries go back to the block cache: nothing queued may still touch them */
    for (void* q : {(void*)nslots, (void*)off, (void*)keys, (void*)keys2, (void*)vals, (void*)vals2, (void*)slot_class, (void*)slot_no,
                    (void*)info, (void*)first, (void*)nch_dev, (void*)runs_dev, temp})
      if (q) mmq_cache_free(q);
  };
#define CLSB(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { cleanup(); return mmq_cuda_fail(h, e__, #call, __FILE__, __LINE__); } } while (0)
  CLSB(mmq_cache_malloc(&nslots, sizeof(int32_t) * (size_t)(m + 1)));
  CLSB(mmq_cache_malloc(&off, sizeof(int32_t) * (size_t)(m + 1)));
  CLSB(mmq_cache_malloc(&info, sizeof(int) * 4));
  CLSB(mmq_cache_malloc(&first, sizeof(int) * MMQ_CLSB_NDP));
  CLSB(mmq_cache_malloc(&nch_dev, sizeof(int) * MMQ_CLSB_NDP));
  CLSB(mmq_cache_malloc(&runs_dev, sizeof(clsb_run) * MMQ_CLSB_NDP));
  CLSB(cudaMemsetAsync(info, 0, sizeof(int) * 4, h->stream));
  CLSB(cudaMemsetAsync(nslots + m, 0, sizeof(int32_t), h->stream));
  if ((rc = mmq_dev_alloc(h, (void**)&h->seg_base, sizeof(int32_t) * (size_t)n))) { cleanup(); return rc; }
  CLSB(cudaMemsetAsync(h->seg_base, 0, sizeof(int32_t) * (size_t)n, h->stream));
  const int grid = mmq_grid_for(m, 256, h->num_sms * 8);
  k_clsb_classify<<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, h->class_id, h->class_id_base, cid_hi, m, nslots, h->seg_base, info);
  g_mmq_launches.fetch_add(1);
  size_t tb1 = 0, tb2 = 0;
  CLSB(cub::DeviceScan::ExclusiveSum(nullptr, tb1, nslots, off, (int)(m + 1), h->stream));
  int host_info[4] = {0, 0, 0, 0};
  {
    void* t1 = nullptr;
    CLSB(mmq_cache_malloc(&t1, tb1));
    cudaError_t e = cub::DeviceScan::ExclusiveSum(t1, tb1, nslots, off, (int)(m + 1), h->stream);
    int total = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&total, off + m, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(host_info, info, sizeof(host_info), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    mmq_cache_free(t1); /* the stream was synchronised just above */
    if (e != cudaSuccess) { cleanup(); return mmq_cuda_fail(h, e, "class plan scan", __FILE__, __LINE__); }
    host_info[3] = total;
  }
  if (host_info[0]) { cleanup(); mmq_dev_free(h, h->seg_base); h->seg_base = nullptr; return MMQ_OK; } /* class ids spread over several 2^32 blocks (or k < 0) */
  const int64_t S = host_info[3];
  std::vector<int> first_h(MMQ_CLSB_NDP, -1), nch(MMQ_CLSB_NDP, 0);
  std::vector<clsb_run> runs(MMQ_CLSB_NDP);
  int64_t chunks = 0, packed = 0, chunks_lo = 0, chunks_gen = 0, c_chunks = 0, c_packed = 0, small_slots = 0, n_chain = 0;
  int64_t c_end[3] = {0, 0, 0};
  if (S > 0) {
    CLSB(mmq_cache_malloc(&keys, sizeof(unsigned long long) * (size_t)S));
    CLSB(mmq_cache_malloc(&keys2, sizeof(unsigned long long) * (size_t)S));
    CLSB(mmq_cache_malloc(&vals, sizeof(uint32_t) * (size_t)S));
    CLSB(mmq_cache_malloc(&vals2, sizeof(uint32_t) * (size_t)S));
    CLSB(mmq_cache_malloc(&slot_class, sizeof(uint32_t) * (size_t)S));
    CLSB(mmq_cache_malloc(&slot_no, (size_t)S));
    k_clsb_slots<<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, nslots, off, m, keys, slot_class, slot_no);
    g_mmq_launches.fetch_add(1);
    k_iota_u32<<<mmq_grid_for(S, 256, h->num_sms * 8), 256, 0, h->stream>>>(vals, S);
    g_mmq_launches.fetch_add(1);
    CLSB(cub::DeviceRadixSort::SortPairs(nullptr, tb2, keys, keys2, vals, vals2, (int)S, 0, 44, h->stream));
    CLSB(mmq_cache_malloc(&temp, tb2));
    CLSB(cub::DeviceRadixSort::SortPairs(temp, tb2, keys, keys2, vals, vals2, (int)S, 0, 44, h->stream));
    CLSB(cudaMemsetAsync(first, 0xff, sizeof(int) * MMQ_CLSB_NDP, h->stream));
    k_clsb_bounds<<<mmq_grid_for(S, 256, h->num_sms * 8), 256, 0, h->stream>>>(keys2, S, first);
    g_mmq_launches.fetch_add(1);
    CLSB(cudaMemcpyAsync(first_h.data(), first, sizeof(int) * MMQ_CLSB_NDP, cudaMemcpyDeviceToHost, h->stream));
    CLSB(cudaStreamSynchronize(h->stream));
    /* runs: pseudo sizes in ascending order; the small set's chunks, then (numbered separately) the chain set's */
    int64_t next_first = S;
    std::vector<int64_t> cnt(MMQ_CLSB_NDP, 0);
    for (int dp = MMQ_CLSB_NDP - 1; dp >= 0; --dp)
      if (first_h[dp] >= 0) { cnt[dp] = next_first - first_h[dp]; next_first = first_h[dp]; }
    for (int dp = 0; dp < MMQ_CLSB_NDP; ++dp) {
      const bool chain = dp >= MMQ_CLSB_DPC0;
      const int d = chain ? MMQ_CLS_CHAIN_DMAX - (dp - MMQ_CLSB_DPC0) : MMQ_CLS_D_OF(dp);
      runs[dp].first = first_h[dp] < 0 ? 0 : first_h[dp];
      runs[dp].d = d; runs[dp].pad = 0;
      const int64_t nc = (cnt[dp] + 31) / 32;
      nch[dp] = (int)nc;
      if (!chain) {
        runs[dp].e0 = packed; runs[dp].chunk0 = (int)chunks;
        chunks += nc; packed += nc * 32 * d; small_slots += cnt[dp];
        if (dp <= MMQ_CLS_DLO) chunks_lo = chunks;
        if (dp <= MMQ_CLS_DMAX) chunks_gen = chunks;
      } else {
        runs[dp].e0 = c_packed; runs[dp].chunk0 = (int)c_chunks;
        c_chunks += nc; c_packed += nc * 32 * d; n_chain += cnt[dp];
        for (int v = 0; v < 3; ++v)
          if (d > (4 >> v)) c_end[v] = c_chunks;
      }
    }
    if (chunks > 0x7fff0000ll) { cleanup(); mmq_dev_free(h, h->seg_base); h->seg_base = nullptr; return MMQ_OK; }
    if ((rc = mmq_dev_alloc(h, (void**)&h->cls_pcol, sizeof(int32_t) * (size_t)std::max<int64_t>(packed, 1)))) { cleanup(); return rc; }
    if ((rc = mmq_dev_alloc(h, (void**)&h->cls_pk, sizeof(uint16_t) * (size_t)std::max<int64_t>(chunks * 32, 1)))) { cleanup(); return rc; }
    if ((rc = mmq_dev_alloc(h, (void**)&h->cls_pcid, sizeof(uint32_t) * (size_t)std::max<int64_t>(chunks * 32, 1)))) { cleanup(); return rc; }
    if ((rc = mmq_dev_alloc(h, (void**)&h->cls_cdesc, sizeof(unsigned long long) * (size_t)std::max<int64_t>(chunks, 1)))) { cleanup(); return rc; }
    if (c_chunks > 0) {
      if ((rc = mmq_dev_alloc(h, (void**)&h->cls_c_pcol, sizeof(int32_t) * (size_t)c_packed))) { cleanup(); return rc; }
      if ((rc = mmq_dev_alloc(h, (void**)&h->cls_c_k, sizeof(int32_t) * (size_t)c_chunks * 32))) { cleanup(); return rc; }
      if ((rc = mmq_dev_alloc(h, (void**)&h->cls_c_cid, sizeof(uint32_t) * (size_t)c_chunks * 32))) { cleanup(); return rc; }
      if ((rc = mmq_dev_alloc(h, (void**)&h->cls_c_desc, sizeof(unsigned long long) * (size_t)c_chunks))) { cleanup(); return rc; }
      k_fill_i32_cls<<<mmq_grid_for(c_packed, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->cls_c_pcol, c_packed, (int32_t)n);
      CLSB(cudaMemsetAsync(h->cls_c_k, 0, sizeof(int32_t) * (size_t)c_chunks * 32, h->stream));
      CLSB(cudaMemsetAsync(h->cls_c_cid, 0, sizeof(uint32_t) * (size_t)c_chunks * 32, h->stream));
    }
    /* padding lanes: the sentinel column (mu[n] == 0), no draws */
    if (packed > 0) k_fill_i32_cls<<<mmq_grid_for(packed, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->cls_pcol, packed, (int32_t)n);
    if (chunks > 0) {
      CLSB(cudaMemsetAsync(h->cls_pk, 0, sizeof(uint16_t) * (size_t)chunks * 32, h->stream));
      CLSB(cudaMemsetAsync(h->cls_pcid, 0, sizeof(uint32_t) * (size_t)chunks * 32, h->stream));
    }
    CLSB(cudaMemcpyAsync(runs_dev, runs.data(), sizeof(clsb_run) * MMQ_CLSB_NDP, cudaMemcpyHostToDevice, h->stream));
    CLSB(cudaMemcpyAsync(nch_dev, nch.data(), sizeof(int) * MMQ_CLSB_NDP, cudaMemcpyHostToDevice, h->stream));
    k_clsb_fill<<<mmq_grid_for(S, 256, h->num_sms * 8), 256, 0, h->stream>>>(keys2, vals2, S, runs_dev, slot_class, slot_no, h->row_ptr, h->col, h->k,
                                                                             h->class_id, h->class_id_base, h->cls_pcol, h->cls_pk, h->cls_pcid,
                                                                             h->cls_c_pcol, h->cls_c_k, h->cls_c_cid);
    k_clsb_desc<<<MMQ_CLSB_NDP, 128, 0, h->stream>>>(runs_dev, MMQ_CLSB_NDP, nch_dev, h->cls_cdesc, h->cls_c_desc);
    g_mmq_launches.fetch_add(4);
  }
  /* the rest (more members than the plan's kernels take): listed by the host from the caller's arrays, one class per tile */
  const int64_t n_rest = host_info[2];
  int64_t nnz_rest = 0;
  if (n_rest > 0) {
    std::vector<int64_t> o_rp(1, 0), o_cid, o_tiles;
    std::vector<int32_t> o_col, o_k;
    std::vector<int64_t> rest;
    for (int64_t i = 0; i < m; ++i) {
      const int64_t d = p->row_ptr[i + 1] - p->row_ptr[i], kv = p->k[i];
      if (d != 1 && kv > 0 && !(d <= MMQ_CLS_DMAX && kv <= mmq_cat_limit((int)d)) && d > MMQ_CLS_CHAIN_DMAX) rest.push_back(i);
    }
    std::stable_sort(rest.begin(), rest.end(), [&](int64_t a, int64_t b) { return p->row_ptr[a + 1] - p->row_ptr[a] > p->row_ptr[b + 1] - p->row_ptr[b]; });
    for (size_t q = 0; q < rest.size(); ++q) {
      const int64_t i = rest[q];
      o_col.insert(o_col.end(), p->col + p->row_ptr[i], p->col + p->row_ptr[i + 1]);
      o_rp.push_back((int64_t)o_col.size());
      o_k.push_back(p->k[i]);
      o_cid.push_back(p->class_id ? p->class_id[i] : p->class_id_base + i);
      o_tiles.push_back((int64_t)q);
    }
    o_tiles.push_back((int64_t)rest.size());
    nnz_rest = (int64_t)o_col.size();
    o_col.resize(o_col.size() + 4, 0);
    if ((rc = cls_upload(h, &h->cls_o_rp, o_rp)) || (rc = cls_upload(h, &h->cls_o_col, o_col)) || (rc = cls_upload(h, &h->cls_o_k, o_k)) ||
        (rc = cls_upload(h, &h->cls_o_cid, o_cid)) || (rc = cls_upload(h, &h->cls_o_tiles, o_tiles))) { cleanup(); return rc; }
    CLSB(cudaStreamSynchronize(h->stream)); /* host temporaries */
  }
  if (host_info[1]) { /* singleton classes: counts[] starts from their constant sums */
    CLSB(cudaMemcpyAsync(h->counts, h->seg_base, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToDevice, h->stream));
    h->seg_base_in_counts = true;
  } else {
    mmq_dev_free(h, h->seg_base);
    h->seg_base = nullptr;
  }
  CLSB(cudaStreamSynchronize(h->stream));
  cleanup();
#undef CLSB
  h->cls_nruns = 0;
  h->cls_chunks = chunks; h->cls_chunks_lo = chunks_lo; h->cls_chunks_gen = chunks_gen;
  h->cls_cid_hi = cid_hi;
  h->cls_small = small_slots; /* slots of the small set (a class above 64 fragments takes several) */
  h->cls_rest = n_rest; h->cls_rest_nnz = nnz_rest; h->cls_rest_tiles = n_rest;
  h->cls_packed = packed;
  h->cls_c_chunks = c_chunks; h->cls_c_packed = c_packed; h->cls_chain = n_chain;
  for (int v = 0; v < 3; ++v) h->cls_c_end[v] = c_end[v];
  h->cls_ready = true;
  return MMQ_OK;
}

int mmq_cls_plan(mmq_handle* h, const mmq_problem* p) {
  h->cls_ready = false;
  if (!h->has_k || h->has_w || h->m == 0) return MMQ_OK;
  const char* hp_env = getenv("MMQ_CLS_HOST_PLAN"); /* once per mmq_create: the host builder instead of the device one (tests compare the two) */
  const bool host_plan = hp_env && atoi(hp_env) != 0;
  if (!h->stream2) {
    MMQ_CUDA(h, cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking));
    MMQ_CUDA(h, cudaStreamCreateWithFlags(&h->stream3, cudaStreamNonBlocking));
    MMQ_CUDA(h, cudaStreamCreateWithFlags(&h->stream4, cudaStreamNonBlocking));
    MMQ_CUDA(h, cudaStreamCreateWithFlags(&h->stream5, cudaStreamNonBlocking));
    MMQ_CUDA(h, cudaStreamCreateWithFlags(&h->stream6, cudaStreamNonBlocking));
    MMQ_CUDA(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    MMQ_CUDA(h, cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    MMQ_CUDA(h, cudaEventCreateWithFlags(&h->ev_join3, cudaEventDisableTiming));
    MMQ_CUDA(h, cudaEventCreateWithFlags(&h->ev_join4, cudaEventDisableTiming));
    MMQ_CUDA(h, cudaEventCreateWithFlags(&h->ev_join5, cudaEventDisableTiming));
    MMQ_CUDA(h, cudaEventCreateWithFlags(&h->ev_fork6, cudaEventDisableTiming));
    MMQ_CUDA(h, cudaEventCreateWithFlags(&h->ev_join6, cudaEventDisableTiming));
  }
  if (!host_plan) return cls_plan_device(h, p);
  mmq_cls_host_plan P;
  if (!mmq_cls_build_host(h->n, h->m, p->row_ptr, p->col, p->k, p->class_id, p->class_id_base, P)) return MMQ_OK;
  const auto t_up = std::chrono::steady_clock::now();
  const std::vector<mmq_cls_run>& runs = P.runs;
  const std::vector<uint16_t>& pk = P.pk;
  const std::vector<uint32_t>& pcid = P.pcid;
  const std::vector<int64_t>&o_rp = P.o_rp, &o_cid = P.o_cid, &o_tiles = P.o_tiles;
  const std::vector<int32_t>&o_col = P.o_col, &o_k = P.o_k, &s_col = P.s_col, &s_k = P.s_k;
  const std::unique_ptr<int32_t[]>& pcol = P.pcol;
  const int64_t packed = P.packed, chunks = P.chunks, chunks_lo = P.chunks_lo, small_classes = P.small_classes, n_rest = P.n_rest, nnz_rest = P.nnz_rest;
  const uint32_t cid_hi = P.cid_hi;
  auto tick = [&](const char* what) {
    static const bool timing = [] { const char* e = getenv("MMQ_CREATE_TIMING"); return e && atoi(e) != 0; }();
    if (timing) fprintf(stderr, "[mmq_cls_plan] %-26s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_up).count());
  };
  int rc;
  if ((rc = mmq_dev_alloc(h, (void**)&h->cls_pcol, sizeof(int32_t) * (size_t)std::max<int64_t>(packed, 1)))) return rc;
  if (packed > 0) MMQ_CUDA(h, cudaMemcpyAsync(h->cls_pcol, pcol.get(), sizeof(int32_t) * (size_t)packed, cudaMemcpyHostToDevice, h->stream));
  if ((rc = cls_upload(h, &h->cls_pk, pk))) return rc;
  if ((rc = cls_upload(h, &h->cls_pcid, pcid))) return rc;
  if ((rc = cls_upload(h, (mmq_cls_run**)&h->cls_runs, runs))) return rc;
  if ((rc = cls_upload(h, &h->cls_cdesc, P.cdesc))) return rc;
  if (P.c_chunks > 0) {
    if ((rc = mmq_dev_alloc(h, (void**)&h->cls_c_pcol, sizeof(int32_t) * (size_t)P.c_packed))) return rc;
    MMQ_CUDA(h, cudaMemcpyAsync(h->cls_c_pcol, P.c_pcol.get(), sizeof(int32_t) * (size_t)P.c_packed, cudaMemcpyHostToDevice, h->stream));
    if ((rc = cls_upload(h, &h->cls_c_k, P.c_k))) return rc;
    if ((rc = cls_upload(h, &h->cls_c_cid, P.c_cid))) return rc;
    if ((rc = cls_upload(h, &h->cls_c_desc, P.c_desc))) return rc;
  }
  if (n_rest > 0) {
    if ((rc = cls_upload(h, &h->cls_o_rp, o_rp))) return rc;
    if ((rc = cls_upload(h, &h->cls_o_col, o_col))) return rc;
    if ((rc = cls_upload(h, &h->cls_o_k, o_k))) return rc;
    if ((rc = cls_upload(h, &h->cls_o_cid, o_cid))) return rc;
    if ((rc = cls_upload(h, &h->cls_o_tiles, o_tiles))) return rc;
  }
  if (!s_col.empty()) {
    int32_t *d_col = nullptr, *d_k = nullptr;
    if ((rc = cls_upload(h, &d_col, s_col))) return rc;
    if ((rc = cls_upload(h, &d_k, s_k))) return rc;
    if ((rc = mmq_dev_alloc(h, (void**)&h->seg_base, sizeof(int32_t) * (size_t)h->n))) return rc;
    MMQ_CUDA(h, cudaMemsetAsync(h->seg_base, 0, sizeof(int32_t) * (size_t)h->n, h->stream));
    k_cls_singletons<<<mmq_grid_for((int64_t)s_col.size(), 256, h->num_sms * 8), 256, 0, h->stream>>>(d_col, d_k, (int64_t)s_col.size(), h->seg_base);
    MMQ_LAUNCHED(h);
    MMQ_CUDA(h, cudaMemcpyAsync(h->counts, h->seg_base, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToDevice, h->stream));
    h->seg_base_in_counts = true;
    MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
    mmq_dev_free(h, d_col);
    mmq_dev_free(h, d_k);
  }
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream)); /* the vectors are host temporaries */
  tick("uploads");
  h->cls_nruns = (int)runs.size();
  h->cls_chunks = chunks;
  h->cls_chunks_lo = chunks_lo;
  h->cls_chunks_gen = P.chunks_gen;
  h->cls_cid_hi = cid_hi;
  h->cls_small = small_classes;
  h->cls_rest = n_rest;
  h->cls_rest_nnz = nnz_rest;
  h->cls_rest_tiles = n_rest;
  h->cls_packed = packed;
  h->cls_c_chunks = P.c_chunks;
  h->cls_c_packed = P.c_packed;
  h->cls_chain = P.n_chain;
  for (int v = 0; v < 3; ++v) h->cls_c_end[v] = P.c_end[v];
  h->cls_ready = true;
  return MMQ_OK;
}

extern "C" int mmq_cls_stats(const mmq_handle* h, int64_t out[8]) {
  if (!h || !out) return MMQ_ERR_ARG;
  out[0] = h->cls_ready ? 1 : 0;
  out[1] = h->cls_small;
  out[2] = h->cls_packed;
  out[3] = h->cls_chunks * 32;
  out[4] = h->cls_rest;
  out[5] = h->cls_rest_nnz;
  out[6] = h->cls_chain;
  out[7] = h->cls_c_packed;
  return MMQ_OK;
}

int mmq_cls_launch(mmq_handle* h, uint32_t seed, uint32_t sweep, const uint32_t* sweep_base) {
  int rc = mmq_seg_add_base(h, true);
  if (rc) return rc;
  const int skip = h->skip_mask;
  const bool do_one = h->cls_chunks > h->cls_chunks_gen && !(skip & 16);
  const bool do_chain = h->cls_c_chunks > 0 && !(skip & 8);
  const bool do_rest = h->cls_rest > 0 && !(skip & 2);
  const bool do_hi = h->cls_chunks_gen > h->cls_chunks_lo && !(skip & 4);
  const bool do_lo = h->cls_chunks_lo > 0 && !(skip & 1);
  /* grids are capped at this many resident CTAs per SM */
  constexpr int CHAIN_CTAS = 3, LARGE_CTAS = 5, SMALL_CTAS = 8, SINGLE_CTAS = 9;
  /* up to five independent pieces, concurrently on the handle's side streams; the main stream takes the last
   * one and waits for the others */
  MMQ_CUDA(h, cudaEventRecord(h->ev_fork, h->stream));
#define MMQ_CLS_ARGS(c0, c1) (int)(c0), (int)(c1), h->cls_pcol, h->cls_pk, h->cls_pcid, h->cls_cdesc, h->cls_cid_hi, h->mu, h->counts, seed, sweep, sweep_base
  /* the chain set: one k_alloc_chain instance per splitting depth over its contiguous chunk range */
  auto chain = [&](auto kern, int C, size_t smem, int64_t c0, int64_t c1, cudaStream_t st) -> int {
    const int cw = C / 32;
    const int grid = (int)std::min<int64_t>((c1 - c0 + cw - 1) / cw, (int64_t)h->num_sms * CHAIN_CTAS);
    MMQ_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, MMQ_CHAIN_THREADS, smem, st>>>((int)c0, (int)c1, h->cls_c_pcol, h->cls_c_k, h->cls_c_cid, h->cls_c_desc, h->cls_cid_hi,
                                                 h->mu, h->counts, seed, sweep, sweep_base);
    MMQ_LAUNCHED(h);
    return MMQ_OK;
  };
  const int64_t* ce = h->cls_c_end;
  const bool do_deep = do_chain && ce[0] > 0, do_shallow = do_chain && ce[2] > ce[0];
  if (do_deep) { /* the longest dependent chains: first in */
    MMQ_CUDA(h, cudaStreamWaitEvent(h->stream4, h->ev_fork, 0));
    if ((rc = chain(k_alloc_chain<4, 64, 2>, 64, sizeof(chain_smem<4, 64>), 0, ce[0], h->stream4))) return rc;
    MMQ_CUDA(h, cudaEventRecord(h->ev_join4, h->stream4));
  }
  if (do_shallow) { /* d 3..4, then d == 2, one after the other on their own stream */
    MMQ_CUDA(h, cudaEventRecord(h->ev_fork6, h->stream));
    MMQ_CUDA(h, cudaStreamWaitEvent(h->stream6, h->ev_fork6, 0));
    if (ce[1] > ce[0] && (rc = chain(k_alloc_chain<2, 128, 3>, 128, sizeof(chain_smem<2, 128>), ce[0], ce[1], h->stream6))) return rc;
    if (ce[2] > ce[1] && (rc = chain(k_alloc_chain<1, 128, 3>, 128, sizeof(chain_smem<1, 128>), ce[1], ce[2], h->stream6))) return rc;
    MMQ_CUDA(h, cudaEventRecord(h->ev_join6, h->stream6));
  }
  if (do_rest) {
    MMQ_CUDA(h, cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
    const int grid = (int)std::min<int64_t>((h->cls_rest_tiles + MMQ_ALLOC_WARPS - 1) / MMQ_ALLOC_WARPS, (int64_t)h->num_sms * 3);
    mmq_launch_alloc_general(h, h->stream2, grid, h->cls_o_rp, h->cls_o_col, h->cls_o_k, h->cls_rest, h->cls_o_tiles, h->cls_rest_tiles,
                             h->cls_o_cid, seed, sweep, sweep_base);
    MMQ_LAUNCHED(h);
    MMQ_CUDA(h, cudaEventRecord(h->ev_join, h->stream2));
  }
  if (do_hi) { /* 96 registers, no spills */
    MMQ_CUDA(h, cudaStreamWaitEvent(h->stream3, h->ev_fork, 0));
    const int64_t c0 = h->cls_chunks_lo, c1 = h->cls_chunks_gen;
    const int grid = (int)std::min<int64_t>((c1 - c0 + MMQ_CLS_WARPS - 1) / MMQ_CLS_WARPS, (int64_t)h->num_sms * LARGE_CTAS);
    k_alloc_cls<false, 5><<<grid, MMQ_CLS_WARPS * 32, 0, h->stream3>>>(MMQ_CLS_ARGS(c0, c1));
    MMQ_LAUNCHED(h);
    MMQ_CUDA(h, cudaEventRecord(h->ev_join3, h->stream3));
  }
  if (do_lo) { /* 64 registers, no spills, 32 warps per SM */
    MMQ_CUDA(h, cudaStreamWaitEvent(h->stream5, h->ev_fork, 0));
    const int64_t c0 = 0, c1 = h->cls_chunks_lo;
    const int grid = (int)std::min<int64_t>((c1 - c0 + MMQ_CLS_WARPS - 1) / MMQ_CLS_WARPS, (int64_t)h->num_sms * SMALL_CTAS);
    k_alloc_cls<true, 8><<<grid, MMQ_CLS_WARPS * 32, 0, h->stream5>>>(MMQ_CLS_ARGS(c0, c1));
    MMQ_LAUNCHED(h);
    MMQ_CUDA(h, cudaEventRecord(h->ev_join5, h->stream5));
  }
  if (do_one) { /* the bulk of the entries, on the main stream */
    const int64_t c0 = h->cls_chunks_gen, c1 = h->cls_chunks;
    const int grid = (int)std::min<int64_t>((c1 - c0 + MMQ_CLS_WARPS - 1) / MMQ_CLS_WARPS, (int64_t)h->num_sms * SINGLE_CTAS);
    k_alloc_cls1<<<grid, MMQ_CLS_WARPS * 32, 0, h->stream>>>(MMQ_CLS_ARGS(c0, c1));
    MMQ_LAUNCHED(h);
  }
#undef MMQ_CLS_ARGS
  if (do_lo) MMQ_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join5, 0));
  if (do_hi) MMQ_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join3, 0));
  if (do_rest) MMQ_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join, 0));
  if (do_shallow) MMQ_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join6, 0));
  if (do_deep) MMQ_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join4, 0));
  return MMQ_OK;
}
