/* mmq_seg.cu — K2 for k == 1 shards laid out BY LENGTH (the loader's
 * LAYOUT_PER_FRAGMENT_BY_LENGTH): the rows of the shard come in a few long runs of equal
 * class size d.  Replaces, for such shards, the allocation loop of src/mmseq.cpp:862-891.
 *
 * What the plan (built once in mmq_create) buys every sweep:
 *   - no row pointers are read at all: inside a run, row r starts at e0 + r*d;
 *   - classes with a single member (d == 1) are not visited: their allocation is
 *     deterministic (x = k, no random number — include/mmq_sampler.h), so their counts
 *     are summed once into seg_base[] and the Gamma kernel restarts counts[] from it;
 *   - a warp takes 128 consecutive classes of ONE size d, four per lane — one Philox block —
 *     whose 128*d contiguous columns arrive by one TMA bulk copy issued a chunk ahead
 *     (k_alloc_seg4 below).
 * Arithmetic and its order are those of the k == 1 branch of mmq_alloc_row, so the counts
 * equal the CPU replay's bit for bit (tests/test_gpu_parity.py).
 *
 * Algorithmic HBM bytes per sweep: 4 B (+4 B weight) per CSR entry of the classes with
 * d >= 2 — nothing else is streamed.
 */
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <thread>
#include <vector>

#include "mmq_device.cuh"
#include "mmq_internal.h"

#define MMQ_SEG_MAX 96    /* more runs than this: not a by-length layout, use the ragged kernel */


__global__ void k_fill_i32(int32_t* __restrict__ p, int64_t count, int32_t v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void k_axpy_i32(int32_t* __restrict__ y, const int32_t* __restrict__ x, int64_t count, int sign) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) y[i] += sign * x[i];
}
/* base[col[q]] += 1 over the CSR entries [q0, q1) of a run of singleton classes */
__global__ void k_count_singletons(const int32_t* __restrict__ col, int64_t q0, int64_t q1, int32_t* __restrict__ base) {
  for (int64_t q = q0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < q1; q += (int64_t)gridDim.x * blockDim.x) atomicAdd(base + col[q], 1);
}

/* One class of compile-time size D (7..12), everything in registers: D columns by vector loads,
 * D independent mu gathers, sum, scan.  The chosen column is re-read (an L1 hit) instead of being
 * selected from registers. */
template <int D, bool HAS_W>
__device__ __noinline__ int32_t seg_row_fixed(const int32_t* __restrict__ cp, const float* __restrict__ wq,
                                                 const double* __restrict__ mu, double u) {
  int32_t c[D];
  float wv[HAS_W ? D : 1];
  if (D % 2 == 0) { /* the row start is 8-byte aligned for even D (two rows of a lane start 16-byte aligned) */
#pragma unroll
    for (int j = 0; j < D; j += 2) {
      const int2 v = *reinterpret_cast<const int2*>(cp + j);
      c[j] = v.x; c[j + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int j = 0; j < D; ++j) c[j] = cp[j];
  }
  if (HAS_W) {
#pragma unroll
    for (int j = 0; j < D; ++j) wv[j] = wq[j];
  }
  double g[D];
#pragma unroll
  for (int j = 0; j < D; ++j) g[j] = HAS_W ? mu[c[j]] * (double)wv[j] : mu[c[j]];
  double norm = 0.0;
#pragma unroll
  for (int j = 0; j < D; ++j) norm += g[j];
  const double target = u * norm;
  double acc = 0.0;
  int chosen = -1, lastpos = -1;
#pragma unroll
  for (int j = 0; j < D; ++j) {
    acc += g[j];
    if (chosen < 0 && target < acc) chosen = j;
    if (g[j] > 0.0) lastpos = j;
  }
  if (chosen < 0) chosen = lastpos >= 0 ? lastpos : D - 1;
  return cp[chosen];
}

/* Any class size: two passes with batched gathers straight from global memory. */
template <bool HAS_W>
__device__ __noinline__ int32_t seg_row_generic(const int32_t* __restrict__ c, const float* __restrict__ wv, int d,
                                                   const double* __restrict__ mu, double u) {
#define MMQ_PG(j) (HAS_W ? mu[c[j]] * (double)wv[j] : mu[c[j]])
  double norm = 0.0;
  int j = 0;
  for (; j + 4 <= d; j += 4) {
    const double a0 = MMQ_PG(j), a1 = MMQ_PG(j + 1), a2 = MMQ_PG(j + 2), a3 = MMQ_PG(j + 3);
    norm += a0; norm += a1; norm += a2; norm += a3;
  }
  for (; j < d; ++j) norm += MMQ_PG(j);
  const double target = u * norm;
  double acc = 0.0;
  int chosen = -1;
  for (j = 0; j + 4 <= d && chosen < 0; j += 4) {
    const double a0 = MMQ_PG(j), a1 = MMQ_PG(j + 1), a2 = MMQ_PG(j + 2), a3 = MMQ_PG(j + 3);
    acc += a0; if (chosen < 0 && target < acc) chosen = j;
    acc += a1; if (chosen < 0 && target < acc) chosen = j + 1;
    acc += a2; if (chosen < 0 && target < acc) chosen = j + 2;
    acc += a3; if (chosen < 0 && target < acc) chosen = j + 3;
  }
  for (; j < d && chosen < 0; ++j) { acc += MMQ_PG(j); if (target < acc) chosen = j; }
  if (chosen < 0) {
    chosen = d - 1;
    for (j = d - 1; j >= 0; --j)
      if (MMQ_PG(j) > 0.0) { chosen = j; break; }
  }
#undef MMQ_PG
  return c[chosen];
}

/* ---- the kernel ----------------------------------------------------------------------------
 * A warp takes 128 consecutive classes of one size D, FOUR per lane — the four
 * classes of one Philox block (CAT stream: class c draws word c & 3 of block c >> 2), so the
 * generator runs once per four allocations.
 *
 * The chunk's 128*D contiguous columns (and weights) arrive by ONE TMA bulk copy into the
 * warp's shared-memory buffer, issued while the previous chunk is being processed:
 *   D <= 6:  the lane pulls its 4*D columns into registers (D 16-byte LDS), the warp releases the
 *            buffer at once and lane 0 issues the copy of the NEXT chunk before any mu is
 *            gathered, so the DRAM latency of the column stream is never on the critical path;
 *   D <= STAGE (12 unweighted, 6 weighted): rows are read from the buffer one at a time, the
 *            next copy is issued when the chunk is done;
 *   larger:  straight from global memory (rare: < 1 % of the classes of a transcriptome).
 * Rows are grouped by class, so a row usually has the members of the row before it: the running
 * sums S_j = p_0 + ... + p_j (left to right, the order of mmq_alloc_row) are then reused and the
 * row costs one multiply, D compares and no gather.  chosen = first j with u*S_{D-1} < S_j.
 * Rows past the end of a run (or the dummy rows in front of it) read whatever the packed array
 * holds there — always valid column indices or the sentinel — and are masked at the reduction. */
#define MMQ_SEG4_ROWS 128
#define MMQ_SEG4_REG_D 6

__device__ __forceinline__ uint32_t seg4_word(const uint32_t (&wd)[4], int r) {
  return r == 0 ? wd[0] : r == 1 ? wd[1] : r == 2 ? wd[2] : wd[3];
}

__device__ __forceinline__ void seg4_put(int32_t (&out)[4], int r, int32_t v) { /* out stays in registers */
  if (r == 0) out[0] = v;
  if (r == 1) out[1] = v;
  if (r == 2) out[2] = v;
  if (r == 3) out[3] = v;
}

/* rare: no running sum exceeded the target (all-zero row): last member with p > 0, else the last */
template <bool HAS_W>
__device__ __noinline__ int32_t seg4_fallback(const int32_t* __restrict__ c, const float* __restrict__ wv, int d,
                                              const double* __restrict__ mu) {
  int chosen = d - 1;
  for (int j = d - 1; j >= 0; --j) {
    const double pj = HAS_W ? mu[c[j]] * (double)wv[j] : mu[c[j]];
    if (pj > 0.0) { chosen = j; break; }
  }
  return c[chosen];
}

/* four rows of compile-time size D <= 6 from registers */
template <int D, bool HAS_W, typename Release, typename RowPtr>
__device__ __forceinline__ void seg4_small(const int32_t* __restrict__ sc, const float* __restrict__ sw, int lane,
                                           const uint32_t (&wd)[4], const double* __restrict__ mu, Release&& release,
                                           RowPtr&& row_offset, const int32_t* __restrict__ colp,
                                           const float* __restrict__ wp, int32_t (&out)[4]) {
  int32_t c[4 * D];
  float wv[HAS_W ? 4 * D : 1];
#pragma unroll
  for (int j = 0; j < D; ++j) { /* the lane's 4*D columns: 16*D bytes, 16-byte aligned */
    const int4 v = *reinterpret_cast<const int4*>(sc + lane * 4 * D + 4 * j);
    c[4 * j] = v.x; c[4 * j + 1] = v.y; c[4 * j + 2] = v.z; c[4 * j + 3] = v.w;
    if (HAS_W) {
      const float4 f = *reinterpret_cast<const float4*>(sw + lane * 4 * D + 4 * j);
      wv[4 * j] = f.x; wv[4 * j + 1] = f.y; wv[4 * j + 2] = f.z; wv[4 * j + 3] = f.w;
    }
  }
  release(); /* the buffer is free: the next chunk's copy starts now */
  double S[D]; /* unweighted: running sums of the current class; weighted: its mu */
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    bool same = r > 0;
    if (r > 0) {
#pragma unroll
      for (int j = 0; j < D; ++j) same &= c[r * D + j] == c[(r - 1) * D + j];
    }
    if (!same) {
#pragma unroll
      for (int j = 0; j < D; ++j) S[j] = mu[c[r * D + j]];
      if (!HAS_W) {
#pragma unroll
        for (int j = 1; j < D; ++j) S[j] = S[j - 1] + S[j];
      }
    }
    double R[D];
    if (HAS_W) {
      R[0] = S[0] * (double)wv[r * D];
#pragma unroll
      for (int j = 1; j < D; ++j) R[j] = R[j - 1] + S[j] * (double)wv[r * D + j];
    } else {
#pragma unroll
      for (int j = 0; j < D; ++j) R[j] = S[j];
    }
    const double target = mmq_uniform32(wd[r]) * R[D - 1];
    int32_t o = c[r * D + D - 1];
    bool hit = target < R[D - 1];
#pragma unroll
    for (int j = D - 2; j >= 0; --j)
      if (target < R[j]) { o = c[r * D + j]; if (HAS_W) hit = true; } /* descending: the smallest index wins */
    if (!hit) {
      const int64_t q = row_offset(r);
      o = seg4_fallback<HAS_W>(colp + q, wp + q, D, mu);
    }
    out[r] = o;
  }
}

/* two consecutive rows (a pair) of compile-time size D read from the shared-memory buffer:
 * 2*D contiguous columns, 8-byte aligned.  Row b reuses row a's mu when it has the same members. */
template <int D, bool HAS_W, typename RowPtr>
__device__ __forceinline__ void seg4_pair_staged(const int32_t* __restrict__ sp, const float* __restrict__ swp, uint32_t wa,
                                                 uint32_t wb, const double* __restrict__ mu, RowPtr&& row_offset, int r0,
                                                 const int32_t* __restrict__ colp, const float* __restrict__ wp,
                                                 int32_t& oa, int32_t& ob) {
  int32_t c[2 * D];
#pragma unroll
  for (int j = 0; j < 2 * D; j += 2) {
    const int2 v = *reinterpret_cast<const int2*>(sp + j);
    c[j] = v.x; c[j + 1] = v.y;
  }
  bool same = true;
#pragma unroll
  for (int j = 0; j < D; ++j) same &= c[j] == c[D + j];
  double R[D]; /* running sums of the current row; unweighted rows with the same members share them */
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (h == 0 || !same || HAS_W) {
#pragma unroll
      for (int j = 0; j < D; ++j) R[j] = HAS_W ? mu[c[h * D + j]] * (double)swp[h * D + j] : mu[c[h * D + j]];
#pragma unroll
      for (int j = 1; j < D; ++j) R[j] = R[j - 1] + R[j];
    }
    const double target = mmq_uniform32(h ? wb : wa) * R[D - 1];
    int32_t o = c[h * D + D - 1];
    bool hit = target < R[D - 1];
#pragma unroll
    for (int j = D - 2; j >= 0; --j)
      if (target < R[j]) { o = c[h * D + j]; if (HAS_W) hit = true; } /* descending: the smallest index wins */
    if (!hit) {
      const int64_t q = row_offset(r0 + h);
      o = seg4_fallback<HAS_W>(colp + q, wp + q, D, mu);
    }
    if (h) ob = o; else oa = o;
  }
}

template <bool HAS_W, int STAGE, int NW, int MINB>
__global__ void __launch_bounds__(NW * 32, MINB)
k_alloc_seg4(const mmq_seg* __restrict__ segs, int nsegs, int total_chunks, int nwarps, const int32_t* __restrict__ colp,
             const float* __restrict__ wp, const double* __restrict__ mu, int32_t* __restrict__ counts, uint32_t seed,
             uint32_t sweep, const uint32_t* __restrict__ sweep_base) {
  if (sweep_base) sweep += *sweep_base; /* CUDA-graph replays: the sweep counter lives on the device */
  constexpr int WARP_BYTES = MMQ_SEG4_ROWS * STAGE * 4 * (HAS_W ? 2 : 1);
  extern __shared__ __align__(16) unsigned char seg4_smem[];
  mmq_seg* s_seg = reinterpret_cast<mmq_seg*>(seg4_smem);
  uint64_t* bars = reinterpret_cast<uint64_t*>(seg4_smem + sizeof(mmq_seg) * MMQ_SEG_MAX);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  int32_t* sc = reinterpret_cast<int32_t*>(seg4_smem + sizeof(mmq_seg) * MMQ_SEG_MAX + 8 * NW + wib * WARP_BYTES);
  float* sw = reinterpret_cast<float*>(sc + MMQ_SEG4_ROWS * STAGE);
  uint64_t* bar = bars + wib;
  for (int i = threadIdx.x; i < nsegs; i += blockDim.x) s_seg[i] = segs[i];
  if (lane == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  int chunk = blockIdx.x * NW + wib;
  if (chunk >= total_chunks) return;
  /* lane 0: start the bulk copy of chunk ch (of run s) when its class size is staged */
  auto issue = [&](int ch, int s) {
    const int d = s_seg[s].d;
    if (d > STAGE || lane != 0) return;
    const int64_t e = s_seg[s].e_virtual + (int64_t)(ch - s_seg[s].chunk0) * (MMQ_SEG4_ROWS * d);
    const uint32_t bytes = (uint32_t)(MMQ_SEG4_ROWS * 4 * d); /* 512*d: a multiple of 16; the packed array has slack */
    mbar_expect_tx(bar, HAS_W ? 2 * bytes : bytes);
    bulk_g2s_stream(sc, colp + e, bytes, bar);
    if (HAS_W) bulk_g2s_stream(sw, wp + e, bytes, bar);
  };
  int si = 0;
  while (si + 1 < nsegs && chunk >= s_seg[si + 1].chunk0) ++si;
  issue(chunk, si);
  uint32_t phase = 0;
  for (; chunk < total_chunks; chunk += nwarps) {
    /* everything about the run is re-read from shared memory where it is needed: registers are
     * for the rows */
    const int D = s_seg[si].d;
    auto release = [&]() { /* all lanes are done with the buffer: fetch this warp's next chunk */
      __syncwarp();
      const int next = chunk + nwarps;
      if (next < total_chunks) {
        int sn = si;
        while (sn + 1 < nsegs && next >= s_seg[sn + 1].chunk0) ++sn; /* warp-uniform */
        issue(next, sn);
      }
    };
    auto row_offset = [&](int r) -> int64_t { /* packed-array offset of the lane's row r (rare paths only) */
      return s_seg[si].e_virtual + (int64_t)((chunk - s_seg[si].chunk0) * MMQ_SEG4_ROWS + 4 * lane + r) * s_seg[si].d;
    };
    unsigned vmask = 0; /* bit r: the lane's row r is a class of the run (not a dummy, not past the end) */
    uint32_t wd[4];
    {
      const int rv = (chunk - s_seg[si].chunk0) * MMQ_SEG4_ROWS + 4 * lane; /* virtual row of the lane's first class */
      const int row_lo = s_seg[si].row_lo, rows = s_seg[si].rows;
#pragma unroll
      for (int r = 0; r < 4; ++r) vmask |= (rv + r >= row_lo && rv + r < rows) ? (1u << r) : 0u;
      const uint64_t cid = (uint64_t)(s_seg[si].cid_virtual + rv); /* a multiple of 4: the lane's classes are one Philox block */
      uint32_t sw_ = sweep;
      asm volatile("" : "+r"(sw_)); /* keeps the first Philox round in the loop instead of in spilled registers */
      wd[0] = (uint32_t)(cid >> 2); wd[1] = (uint32_t)(cid >> 34); wd[2] = sw_; wd[3] = 0u;
      mmq_philox4x32_10(wd, seed, MMQ_STREAM_CAT);
    }
    int32_t out[4] = {-1, -1, -1, -1};
    constexpr bool skip = false;
    if (D <= STAGE) {
      mbar_wait(bar, phase);
      phase ^= 1u;
      if (skip) release();
      else if (D == 2) seg4_small<2, HAS_W>(sc, sw, lane, wd, mu, release, row_offset, colp, wp, out);
      else if (D == 3) seg4_small<3, HAS_W>(sc, sw, lane, wd, mu, release, row_offset, colp, wp, out);
      else if (D == 4) seg4_small<4, HAS_W>(sc, sw, lane, wd, mu, release, row_offset, colp, wp, out);
      else if (D == 5) seg4_small<5, HAS_W>(sc, sw, lane, wd, mu, release, row_offset, colp, wp, out);
      else if (D == 6) seg4_small<6, HAS_W>(sc, sw, lane, wd, mu, release, row_offset, colp, wp, out);
      else {
#define MMQ_SEG4_CASE(DD)                                                                                             \
  else if (STAGE >= DD && D == DD) {                                                                                  \
    constexpr int DX = STAGE >= DD ? DD : 7;                                                                          \
    seg4_pair_staged<DX, HAS_W>(sc + lane * 4 * DX, sw + lane * 4 * DX, wd[0], wd[1], mu, row_offset, 0, colp, wp, out[0], out[1]); \
    seg4_pair_staged<DX, HAS_W>(sc + lane * 4 * DX + 2 * DX, sw + lane * 4 * DX + 2 * DX, wd[2], wd[3], mu, row_offset, 2, colp, wp, \
                                out[2], out[3]);                                                                      \
  }
        if (false) {}
        MMQ_SEG4_CASE(7) MMQ_SEG4_CASE(8) MMQ_SEG4_CASE(9) MMQ_SEG4_CASE(10) MMQ_SEG4_CASE(11) MMQ_SEG4_CASE(12)
#undef MMQ_SEG4_CASE
        release();
      }
    } else {
      release(); /* the buffer is idle: it can already take the next staged chunk */
      if (!skip) {
#pragma unroll 1
        for (int r = 0; r < 4; ++r)
          if ((vmask >> r) & 1u) { /* no slack is promised beyond the staged sizes */
            const int64_t q = row_offset(r);
            const double u = mmq_uniform32(seg4_word(wd, r));
            int32_t o;
#define MMQ_SEG4_DIRECT(DD) else if (STAGE < DD && D == DD) o = seg_row_fixed<DD, HAS_W>(colp + q, wp + q, mu, u);
            if (false) {}
            MMQ_SEG4_DIRECT(7) MMQ_SEG4_DIRECT(8) MMQ_SEG4_DIRECT(9) MMQ_SEG4_DIRECT(10) MMQ_SEG4_DIRECT(11) MMQ_SEG4_DIRECT(12)
#undef MMQ_SEG4_DIRECT
            else o = seg_row_generic<HAS_W>(colp + q, wp + q, D, mu, u);
            seg4_put(out, r, o);
          }
      }
    }
    /* counts[c] += 1, one reduction per distinct column of the warp and row slot; the four matches are
     * issued back to back.  Masked rows share the key -1 (never reduced). */
    {
      unsigned grp[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        if (!((vmask >> r) & 1u) || skip) out[r] = -1;
        grp[r] = __match_any_sync(0xffffffffu, out[r]);
      }
      const unsigned lt_mask = (1u << lane) - 1u;
#pragma unroll
      for (int r = 0; r < 4; ++r)
        if (out[r] >= 0 && (grp[r] & lt_mask) == 0) atomicAdd(counts + out[r], __popc(grp[r]));
    }
    const int next = chunk + nwarps;
    while (si + 1 < nsegs && next >= s_seg[si + 1].chunk0) ++si; /* warp-uniform */
  }
}

/* ------------------------------------------------------------------ host */

int mmq_seg_add_base(mmq_handle* h, bool want_in_counts) {
  if (!h->seg_base || h->seg_base_in_counts == want_in_counts) return MMQ_OK;
  k_axpy_i32<<<mmq_grid_for(h->n, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->counts, h->seg_base, h->n, want_in_counts ? 1 : -1);
  MMQ_LAUNCHED(h);
  h->seg_base_in_counts = want_in_counts;
  return MMQ_OK;
}

/* Host-only part of the plan: runs of equal class size.  Called right after the H2D copies are
 * queued, so the scan overlaps the DMA. */
int mmq_seg_scan(mmq_handle* h, const int64_t* rp) {
  h->seg_runs.clear();
  h->seg_scan_ok = false;
  const int64_t m = h->m;
  if (m == 0 || h->has_k) return MMQ_OK;
  /* 8 bytes per class to read: split between host threads (the H2D copies of the shard are in flight meanwhile) */
  const int nt = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<unsigned>(std::thread::hardware_concurrency(), 16u), m / (1 << 20)));
  std::vector<std::vector<mmq_handle::seg_run>> part((size_t)nt);
  std::vector<char> bad((size_t)nt, 0);
  auto scan = [&](int t) {
    const int64_t a = m * t / nt, b = m * (t + 1) / nt;
    auto& out = part[(size_t)t];
    for (int64_t i = a; i < b;) {
      const int64_t d = rp[i + 1] - rp[i];
      if (d > 0x7fffffff || d <= 0) { bad[(size_t)t] = 1; return; }
      int64_t j = i + 1;
      while (j < b && rp[j + 1] - rp[j] == d) ++j;
      out.push_back({i, j, rp[i], (int)d});
      if ((int)out.size() > MMQ_SEG_MAX + 1) { bad[(size_t)t] = 2; return; } /* ragged shard */
      i = j;
    }
  };
  if (nt == 1) scan(0);
  else {
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t) th.emplace_back(scan, t);
    for (auto& x : th) x.join();
  }
  for (int t = 0; t < nt; ++t) {
    if (bad[(size_t)t]) { h->seg_runs.clear(); return MMQ_OK; } /* not a by-length layout: the row-pointer kernel handles it */
    for (const auto& r : part[(size_t)t]) {
      if (!h->seg_runs.empty() && h->seg_runs.back().d == r.d && h->seg_runs.back().r1 == r.r0) h->seg_runs.back().r1 = r.r1; /* a run cut by the split */
      else h->seg_runs.push_back(r);
      if ((int)h->seg_runs.size() > MMQ_SEG_MAX) { h->seg_runs.clear(); return MMQ_OK; }
    }
  }
  h->seg_scan_ok = true;
  return MMQ_OK;
}

int mmq_seg_plan(mmq_handle* h) {
  h->seg_ready = false;
  if (!h->seg_scan_ok) return MMQ_OK;
  struct Run { int64_t r0, r1, q0; int d; };
  std::vector<Run> runs;
  for (const auto& r : h->seg_runs) runs.push_back({r.r0, r.r1, r.q0, r.d});
  const int rows_per_chunk = MMQ_SEG4_ROWS;
  std::vector<mmq_seg> segs;
  int64_t packed = 0, chunks = 0, entries = 0, rows = 0, singles = 0;
  for (const Run& r : runs) {
    if (r.d == 1) { singles += r.r1 - r.r0; continue; }
    if ((r.r1 - r.r0 + 3) > 0x7ffffff0ll) return MMQ_OK;
    mmq_seg sg;
    const int lead = (int)((h->class_id_base + r.r0) & 3); /* dummy rows: the virtual first class id is a multiple of 4 */
    packed = (packed + 3) & ~(int64_t)3;
    sg.e_virtual = packed;
    sg.cid_virtual = h->class_id_base + r.r0 - lead;
    sg.row_lo = lead;
    sg.rows = (int32_t)(r.r1 - r.r0 + lead);
    sg.d = r.d;
    sg.chunk0 = (int32_t)chunks;
    packed += (int64_t)sg.rows * r.d;
    chunks += (sg.rows + rows_per_chunk - 1) / rows_per_chunk;
    if (chunks > 0x7fff0000ll) return MMQ_OK;
    entries += (r.r1 - r.r0) * r.d;
    rows += r.r1 - r.r0;
    segs.push_back(sg);
  }
  if (segs.empty() && singles == 0) return MMQ_OK;
  packed = ((packed + 3) & ~(int64_t)3) + MMQ_SEG4_ROWS * 12 + 64; /* slack: the bulk copy of a run's last chunk always moves 128 rows */
  h->seg_packed = packed;
  h->seg_host.assign(segs.begin(), segs.end());
  int rc;
  if (singles > 0) {
    if ((rc = mmq_dev_alloc(h, (void**)&h->seg_base, sizeof(int32_t) * (size_t)h->n))) return rc;
    MMQ_CUDA(h, cudaMemsetAsync(h->seg_base, 0, sizeof(int32_t) * (size_t)h->n, h->stream));
    for (const Run& r : runs)
      if (r.d == 1) {
        k_count_singletons<<<mmq_grid_for(r.r1 - r.r0, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->col, r.q0, r.q0 + (r.r1 - r.r0), h->seg_base);
        MMQ_LAUNCHED(h);
      }
    MMQ_CUDA(h, cudaMemcpyAsync(h->counts, h->seg_base, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToDevice, h->stream));
    h->seg_base_in_counts = true;
  }
  if (!segs.empty()) {
    if ((rc = mmq_dev_alloc(h, &h->seg_table, sizeof(mmq_seg) * segs.size()))) return rc;
    MMQ_CUDA(h, cudaMemcpyAsync(h->seg_table, segs.data(), sizeof(mmq_seg) * segs.size(), cudaMemcpyHostToDevice, h->stream));
  }
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream)); /* segs is a host temporary */
  h->seg_count = (int)segs.size();
  h->seg_chunks = chunks;
  h->seg_entries = entries;
  h->seg_rows = rows;
  h->seg_singletons = singles;
  h->seg_ready = true;
  return MMQ_OK;
}

/* The packed, aligned copies of col / weight the segment kernel streams: made by the first sweep that runs it, so a
 * handle that is only swept with MMQ_GIBBS_GENERIC_KERNEL, RAGGED_KERNEL or TRANSPOSED never holds them. */
int mmq_seg_pack(mmq_handle* h) {
  if (h->seg_col || h->seg_count == 0) return MMQ_OK;
  const int64_t packed = h->seg_packed;
  int rc;
  if ((rc = mmq_dev_alloc(h, (void**)&h->seg_col, sizeof(int32_t) * (size_t)packed))) return rc;
  k_fill_i32<<<mmq_grid_for(packed, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->seg_col, packed, (int32_t)h->n);
  MMQ_LAUNCHED(h);
  if (h->has_w) {
    if ((rc = mmq_dev_alloc(h, (void**)&h->seg_w, sizeof(float) * (size_t)packed))) return rc;
    MMQ_CUDA(h, cudaMemsetAsync(h->seg_w, 0, sizeof(float) * (size_t)packed, h->stream));
  }
  size_t si = 0;
  for (const auto& r : h->seg_runs) {
    if (r.d == 1) continue;
    const mmq_seg& sg = h->seg_host[si++];
    const int64_t dst = sg.e_virtual + (int64_t)sg.row_lo * r.d;
    const size_t cnt = (size_t)(r.r1 - r.r0) * (size_t)r.d;
    MMQ_CUDA(h, cudaMemcpyAsync(h->seg_col + dst, h->col + r.q0, sizeof(int32_t) * cnt, cudaMemcpyDeviceToDevice, h->stream));
    if (h->has_w) MMQ_CUDA(h, cudaMemcpyAsync(h->seg_w + dst, h->w + r.q0, sizeof(float) * cnt, cudaMemcpyDeviceToDevice, h->stream));
  }
  return MMQ_OK;
}

int mmq_seg_launch(mmq_handle* h, uint32_t seed, uint32_t sweep, const uint32_t* sweep_base) {
  int rc = mmq_seg_add_base(h, true);
  if (rc) return rc;
  if ((rc = mmq_seg_pack(h))) return rc;
  if (h->seg_count == 0) return MMQ_OK; /* only singletons: nothing random to do */
  const int chunks = (int)h->seg_chunks;
  /* W weights, ST largest staged class size, NW warps per CTA, MINB CTAs per SM (=> register budget) */
#define MMQ_SEG4_GO(W, ST, NW, MINB)                                                                                        \
  do {                                                                                                                      \
    constexpr int SM = (int)sizeof(mmq_seg) * MMQ_SEG_MAX + 8 * NW + NW * MMQ_SEG4_ROWS * ST * 4 * (W ? 2 : 1);             \
    const int grid = std::min((chunks + NW - 1) / NW, h->num_sms * MINB);                                                   \
    MMQ_CUDA(h, cudaFuncSetAttribute(k_alloc_seg4<W, ST, NW, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM));      \
    k_alloc_seg4<W, ST, NW, MINB><<<grid, NW * 32, SM, h->stream>>>((const mmq_seg*)h->seg_table, h->seg_count, chunks,     \
                                                                    grid * NW, h->seg_col, h->seg_w, h->mu, h->counts, seed, \
                                                                    sweep, sweep_base);                                 \
  } while (0)
  if (h->has_w) MMQ_SEG4_GO(true, 12, 4, 4); /* 12 KB per warp: 16 warps per SM, no spills */
  else MMQ_SEG4_GO(false, 12, 4, 6);         /* 80 registers, no spills, 24 warps per SM */
#undef MMQ_SEG4_GO
  return MMQ_OK;
}
