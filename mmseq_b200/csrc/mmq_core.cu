/* mmq_core.cu — device-resident hit-class CSR, EM and Gibbs kernels (sm_100a)
 * and the C ABI over them (include/mmq.h).
 *
 * Reference loops replaced (eturro/mmseq 1.0.11, /root/reference):
 *   k_init_acc / k_divide    src/mmseq.cpp:617-638  initial mu, unique hits
 *   k_rowterm                src/mmseq.cpp:745-754, :796-802 (log-lik), :787-791 (D_i)
 *   k_em_acc / k_em_apply    src/mmseq.cpp:781-794  EM update
 *   k_alloc                  src/mmseq.cpp:862-891  multinomial per hit class
 *   k_count_reduce           src/mmseq.cpp:887, :895-899  per-transcript counts
 *   k_gamma                  src/mmseq.cpp:904-917  Gamma update + trace capture
 * Compile with -fmad=false: the samplers of include/mmq_sampler.h must round
 * exactly like the gcc build of the CPU replay.
 */
#include <cub/cub.cuh>
#include <dlfcn.h>
#include <nccl.h> /* types only; the library is dlopen'ed */

#include <algorithm>
#include <chrono>
#include <map>
#include <mutex>
#include <type_traits>
#include <unordered_map>
#include <cstdio>
#include <cstring>

#include "../../include/mmq_sampler.h"
#include "mmq_internal.h"
#include "mmq_device.cuh"

std::atomic<long long> g_mmq_launches{0};
thread_local std::string g_mmq_create_err;

/* ------------------------------------------------------------------ errors */

int mmq_fail(mmq_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_mmq_create_err = msg;
  return code;
}

int mmq_cuda_fail(mmq_handle* h, cudaError_t e, const char* what, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  return mmq_fail(h, MMQ_ERR_CUDA, buf);
}

/* ---- the device block cache (mmq_internal.h) ---- */
namespace {
struct dev_cache {
  std::mutex mu;
  std::multimap<size_t, void*> free_blocks;       /* by size */
  std::unordered_map<void*, size_t> size_of;      /* every block handed out or cached */
  size_t cached = 0;
};
dev_cache g_cache[16];
size_t cache_limit() {
  static const size_t lim = [] { const char* e = getenv("MMQ_DEVICE_CACHE_MB"); return (size_t)(e ? atoll(e) : 16384) << 20; }();
  return lim;
}
void cache_drop_all(dev_cache& c) { /* c.mu held */
  for (auto& kv : c.free_blocks) { cudaFree(kv.second); c.size_of.erase(kv.second); }
  c.free_blocks.clear();
  c.cached = 0;
}
}  // namespace

cudaError_t mmq_cache_malloc_raw(void** p, size_t bytes) {
  *p = nullptr;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (bytes == 0) bytes = 16;
  /* small blocks in 512-byte steps, large ones in 2 MB steps (the driver's own granularity): more hits */
  const size_t want = bytes < ((size_t)1 << 20) ? (bytes + 511) & ~(size_t)511 : (bytes + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1);
  dev_cache& c = g_cache[dev & 15];
  std::lock_guard<std::mutex> lk(c.mu);
  auto it = c.free_blocks.lower_bound(want);
  if (it != c.free_blocks.end() && it->first <= want + want / 4 + ((size_t)4 << 20)) { /* close enough in size: no big waste */
    *p = it->second;
    c.cached -= it->first;
    c.free_blocks.erase(it);
    return cudaSuccess;
  }
  e = cudaMalloc(p, want);
  if (e != cudaSuccess && !c.free_blocks.empty()) { /* out of memory with blocks parked here: give them back and retry */
    cudaGetLastError();
    cache_drop_all(c);
    e = cudaMalloc(p, want);
  }
  if (e == cudaSuccess) c.size_of[*p] = want;
  return e;
}

void mmq_cache_free(void* p) {
  if (!p) return;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return;
  dev_cache& c = g_cache[dev & 15];
  std::lock_guard<std::mutex> lk(c.mu);
  auto it = c.size_of.find(p);
  if (it == c.size_of.end()) { cudaFree(p); return; } /* not ours (or another device's): plain free */
  if (c.cached + it->second > cache_limit()) { cudaFree(p); c.size_of.erase(it); return; }
  c.free_blocks.emplace(it->second, p);
  c.cached += it->second;
}

int mmq_dev_alloc(mmq_handle* h, void** p, size_t bytes) {
  *p = nullptr;
  if (bytes == 0) bytes = 16;
  const size_t rounded = (bytes + 255) & ~(size_t)255;
  if (h->arena && h->arena_off + rounded <= h->arena_cap) {
    *p = h->arena + h->arena_off;
    h->arena_off += rounded;
    h->bytes += (int64_t)bytes;
    return MMQ_OK;
  }
  cudaError_t e = mmq_cache_malloc_raw(p, bytes);
  if (e != cudaSuccess) return mmq_cuda_fail(h, e, "cudaMalloc", __FILE__, __LINE__);
  /* a recycled block holds what its last user left: every handle starts from zeroed memory, whatever ran before it in
   * the process (padding slots of the plans are read, if never used) */
  e = cudaMemsetAsync(*p, 0, bytes, h->stream);
  if (e != cudaSuccess) return mmq_cuda_fail(h, e, "cudaMemsetAsync", __FILE__, __LINE__);
  h->bytes += (int64_t)bytes;
  h->allocs.push_back(*p);
  return MMQ_OK;
}

void mmq_dev_free(mmq_handle* h, void* p) {
  if (!p) return;
  if (h->arena && (char*)p >= h->arena && (char*)p < h->arena + h->arena_cap) return; /* released with the arena */
  auto it = std::find(h->allocs.begin(), h->allocs.end(), p);
  if (it != h->allocs.end()) h->allocs.erase(it);
  if (h->stream) cudaStreamSynchronize(h->stream); /* nothing queued may still touch the block when it is handed out again */
  mmq_cache_free(p);
}

/* ------------------------------------------------------- device utilities */

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

/* Deterministic block sum (blockDim.x a multiple of 32, <= 1024); result valid in thread 0. */
__device__ __forceinline__ double block_sum(double v) {
  __shared__ double s_part[32];
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) s_part[wid] = v;
  __syncthreads();
  double r = 0.0;
  if (threadIdx.x == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    for (int i = 0; i < nw; ++i) r += s_part[i];
  }
  return r;
}

/* out[slot] = sum of partial[0..count) in index order (single block of 256). */
__global__ void k_sum_partials(const double* __restrict__ partial, int count, double* __restrict__ out, int slot) {
  double v = 0.0;
  for (int i = threadIdx.x; i < count; i += blockDim.x) v += partial[i];
  v = block_sum(v);
  if (threadIdx.x == 0) out[slot] = v;
}

/* flags[0] |= 1 for an empty / negative-length row, |= 2 for a column out of range,
 * |= 4 for columns not strictly ascending within a row */
__global__ void k_validate(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int64_t m,
                           int64_t n, int* __restrict__ flags) {
  int bad = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = row_ptr[i], e = row_ptr[i + 1];
    if (e <= b) { bad |= 1; continue; }
    int32_t prev = -1;
    for (int64_t q = b; q < e; ++q) {
      const int32_t c = col[q];
      if (c < 0 || c >= n) bad |= 2;
      if (c <= prev) bad |= 4;
      prev = c;
    }
  }
  if (bad) atomicOr(flags, bad);
}

/* ---------------------------------------------------- transpose building */

__global__ void k_iota(uint32_t* __restrict__ v, int64_t nnz) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x)
    v[q] = (uint32_t)q;
}

/* keys sorted ascending: tptr[t] = first q with keys[q] >= t, tptr[n] = nnz */
__global__ void k_tptr(const int32_t* __restrict__ keys, int64_t nnz, int64_t n, int64_t* __restrict__ tptr) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q <= nnz; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t prev = (q == 0) ? -1 : (int64_t)keys[q - 1];
    const int64_t cur = (q == nnz) ? n : (int64_t)keys[q];
    for (int64_t t = prev + 1; t <= cur; ++t) tptr[t] = q;
  }
}

/* trow[q'] = class whose CSR range contains position perm[q'] */
__global__ void k_trow(const uint32_t* __restrict__ perm, const int64_t* __restrict__ row_ptr, int64_t m, int64_t nnz,
                       int32_t* __restrict__ trow) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pos = (int64_t)perm[q];
    int64_t lo = 0, hi = m; /* row_ptr[lo] <= pos < row_ptr[hi] */
    while (hi - lo > 1) {
      const int64_t mid = (lo + hi) >> 1;
      if (row_ptr[mid] <= pos) lo = mid; else hi = mid;
    }
    trow[q] = (int32_t)lo;
  }
}

/* --------------------------------------------------------- init / EM */

/* acc[t] = sum_{i containing t} k[i]/|i| (ascending i), uh[t] = sum of k[i] over
 * singleton classes {t}.  One warp per transcript.  src/mmseq.cpp:625-635. */
template <bool HAS_K>
__global__ void k_init_acc(const int64_t* __restrict__ tptr, const int32_t* __restrict__ trow,
                           const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ kk,
                           double* __restrict__ acc, int32_t* __restrict__ uh, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t t = warp0; t < n; t += nwarps) {
    double s = 0.0;
    int u = 0;
    for (int64_t q = tptr[t] + lane; q < tptr[t + 1]; q += 32) {
      const int32_t i = trow[q];
      const int64_t d = row_ptr[i + 1] - row_ptr[i];
      const int32_t kv = HAS_K ? kk[i] : 1;
      s += (double)kv / (double)d;
      if (d == 1) u += kv;
    }
    s = warp_sum(s);
    u = warp_sum_i(u);
    if (lane == 0) { acc[t] = s; uh[t] = u; }
  }
}

__global__ void k_divide(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out, int64_t n) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
    out[t] = a[t] / b[t];
}

/* rterm[i] = k_i / D_i with D_i = sum_{s in i} w_is mu_s; partial[block] = sum_i k_i log D_i.
 * src/mmseq.cpp:748-751 and :797-800 (log-lik), :789-790 (k[row]/inner_prod). */
template <bool HAS_K, bool HAS_W>
__global__ void k_rowterm(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                          const int32_t* __restrict__ kk, const float* __restrict__ w,
                          const double* __restrict__ mu, double* __restrict__ rterm,
                          double* __restrict__ partial, int64_t m) {
  double ll = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = row_ptr[i], e = row_ptr[i + 1];
    double D = 0.0;
    for (int64_t q = b; q < e; ++q) D += HAS_W ? (double)w[q] * mu[col[q]] : mu[col[q]];
    const double kv = (double)(HAS_K ? kk[i] : 1);
    rterm[i] = kv / D;
    ll += kv * log(D);
  }
  ll = block_sum(ll);
  if (threadIdx.x == 0) partial[blockIdx.x] = ll;
}

/* acc[t] = sum_{i containing t} w_it k_i / D_i, one warp per transcript. src/mmseq.cpp:786-791. */
template <bool HAS_W>
__global__ void k_em_acc(const int64_t* __restrict__ tptr, const uint32_t* __restrict__ perm,
                         const int32_t* __restrict__ trow, const float* __restrict__ w,
                         const double* __restrict__ rterm, double* __restrict__ acc, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t t = warp0; t < n; t += nwarps) {
    double s = 0.0;
    for (int64_t q = tptr[t] + lane; q < tptr[t + 1]; q += 32)
      s += HAS_W ? (double)w[perm[q]] * rterm[trow[q]] : rterm[trow[q]];
    s = warp_sum(s);
    if (lane == 0) acc[t] = s;
  }
}

/* mu_out[t] = mu[t]*acc[t]/l[t] (src/mmseq.cpp:792); partial[block] = sum_t mu_out[t] l[t] (:802). */
__global__ void k_em_apply(const double* __restrict__ mu, const double* __restrict__ acc,
                           const double* __restrict__ len, double* __restrict__ mu_out,
                           double* __restrict__ partial, int64_t n) {
  double s = 0.0;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    const double v = mu[t] * acc[t] / len[t];
    mu_out[t] = v;
    s += v * len[t];
  }
  s = block_sum(s);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

/* out[t] = a[t] * b[t]: the expected counts mu * acc of one E-step (mmq_expected_counts). */
__global__ void k_mul(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out, int64_t n) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
    out[t] = a[t] * b[t];
}

__global__ void k_mul_sum(const double* __restrict__ a, const double* __restrict__ b,
                          double* __restrict__ partial, int64_t n) {
  double s = 0.0;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
    s += a[t] * b[t];
  s = block_sum(s);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

/* ------------------------------------------------------------- Gibbs */

/* x[j] = v on this proxy adds v to counts[col_j] (no X matrix is kept: the
 * reference's X is write-only, src/mmseq.cpp:884). */
struct XRed {
  const int32_t* c;
  int32_t* counts;
  struct Ref {
    int32_t* addr;
    __device__ __forceinline__ void operator=(int32_t v) const { if (v != 0) atomicAdd(addr, v); }
  };
  __device__ __forceinline__ Ref operator[](int j) const { return Ref{counts + c[j]}; }
};
__device__ __forceinline__ void mmq_x_zero(const XRed&, int) {}
__device__ __forceinline__ void mmq_x_add(const XRed& x, int j, int32_t v) { x[j] = v; }

/* p[j] straight from global memory, for tiles too large to stage. */
template <bool HAS_W>
struct PGlobal {
  const int32_t* c;
  const float* w;
  const double* mu;
  __device__ __forceinline__ double operator[](int j) const {
    return HAS_W ? mu[c[j]] * (double)w[j] : mu[c[j]];
  }
};

/* K2: allocate the k_i fragments of every hit class among its transcripts.
 * A warp takes a tile of consecutive classes (as many as fit its staging slab, at
 * most one per lane; boundaries precomputed in mmq_create), stages the tile's
 * contiguous CSR segment (columns, and p = mu[col] * weight gathered once) in
 * shared memory with coalesced loads, then one thread per class runs
 * mmq_alloc_row on its slice.  MATERIALIZE writes x into the X array (CSR
 * order) for k_count_reduce; otherwise each non-zero x goes straight to
 * counts[] as a reduction (the fused path).  Persistent over tiles. */
template <bool MATERIALIZE, bool HAS_K, bool HAS_W>
__global__ void __launch_bounds__(MMQ_ALLOC_WARPS * 32, 3)
k_alloc(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
        const int32_t* __restrict__ kk, const float* __restrict__ w, const double* __restrict__ mu,
        int32_t* __restrict__ counts, int32_t* __restrict__ xout, int64_t m, const int64_t* __restrict__ tile_start,
        int64_t n_tiles, uint32_t seed, uint32_t sweep, int64_t class_id_base, const int64_t* __restrict__ class_id,
        const uint32_t* __restrict__ sweep_base) {
  if (sweep_base) sweep += *sweep_base; /* CUDA-graph replays: the sweep counter lives on the device */
  /* every warp owns its tiles and its staging slab: no block-level barrier, the warps of an SM
   * overlap each other's load latency */
  __shared__ double s_p_all[MMQ_ALLOC_WARPS][MMQ_ALLOC_CAP];
  __shared__ int32_t s_c_all[MMQ_ALLOC_WARPS][MMQ_ALLOC_CAP];
  __shared__ int32_t s_x_all[MATERIALIZE ? MMQ_ALLOC_WARPS : 1][MATERIALIZE ? MMQ_ALLOC_CAP : 1];
  __shared__ int64_t s_rp_all[MMQ_ALLOC_WARPS][33];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  double* s_p = s_p_all[wib];
  int32_t* s_c = s_c_all[wib];
  int32_t* s_x = s_x_all[MATERIALIZE ? wib : 0];
  int64_t* s_rp = s_rp_all[wib];
  const int64_t warp0 = (int64_t)blockIdx.x * MMQ_ALLOC_WARPS + wib;
  const int64_t nwarps = (int64_t)gridDim.x * MMQ_ALLOC_WARPS;
  for (int64_t tile = warp0; tile < n_tiles; tile += nwarps) {
    const int64_t r0 = tile_start[tile];
    const int nrows = (int)(tile_start[tile + 1] - r0); /* <= 32 */
    if (lane <= nrows) s_rp[lane] = row_ptr[r0 + lane];
    if (lane == 0 && nrows == 32) s_rp[32] = row_ptr[r0 + 32];
    __syncwarp();
    const int64_t base = s_rp[0];
    const int64_t cnt = s_rp[nrows] - base;
    const bool staged = cnt <= MMQ_ALLOC_CAP;
    if (staged) {
      for (int q = lane; q < (int)cnt; q += 32) {
        const int32_t c = col[base + q];
        double p = mu[c];
        if (HAS_W) p *= (double)w[base + q];
        s_c[q] = c;
        s_p[q] = p;
      }
    }
    __syncwarp();
    if (lane < nrows) {
      const int64_t rb = s_rp[lane];
      const int d = (int)(s_rp[lane + 1] - rb);
      const int64_t kv = HAS_K ? (int64_t)kk[r0 + lane] : 1;
      const uint64_t cid = (uint64_t)(class_id ? class_id[r0 + lane] : class_id_base + r0 + lane);
      if (staged) {
        const int off = (int)(rb - base);
        if (MATERIALIZE) mmq_alloc_row(s_p + off, s_x + off, d, kv, seed, cid, sweep);
        else mmq_alloc_row(s_p + off, XRed{s_c + off, counts}, d, kv, seed, cid, sweep);
      } else {
        PGlobal<HAS_W> pg{col + rb, HAS_W ? w + rb : nullptr, mu};
        if (MATERIALIZE) mmq_alloc_row(pg, xout + rb, d, kv, seed, cid, sweep);
        else mmq_alloc_row(pg, XRed{col + rb, counts}, d, kv, seed, cid, sweep);
      }
    }
    __syncwarp();
    if (MATERIALIZE && staged)
      for (int q = lane; q < (int)cnt; q += 32) xout[base + q] = s_x[q];
    __syncwarp();
  }
}


/* ------------------------------------------------ K2 fast path: k == 1 rows */

#define MMQ_CAT_WARPS 8   /* warps per CTA; warps are autonomous (no block barrier) */
#define MMQ_CAT_ROWS 64   /* classes per warp chunk: two consecutive classes per lane */
#define MMQ_CAT_SLAB 640  /* staged CSR entries per warp and buffer (unweighted) */
#define MMQ_CAT_SLAB_W 384 /* ... with per-hit weights (two arrays are staged) */

/* The two k == 1 classes of one lane: categorical draws with the arithmetic, and its order,
 * of the k == 1 branch of mmq_alloc_row (include/mmq_sampler.h): running sums S_j = p_0 + ... + p_j
 * left to right, target = u * S_{d-1}, chosen = first j with target < S_j.
 * Control flow is warp-uniform (trip counts are warp maxima, lanes past their row gather the
 * sentinel mu[n] == 0, adding 0.0 is exact), and gathers are issued in independent batches.
 * Returns the chosen COLUMNS (or -1 for an absent class). */
template <bool HAS_W>
__device__ __forceinline__ void cat_draw2(const int32_t* ca, const float* wa, int da, double ua, const int32_t* cb,
                                          const float* wb, int db, double ub, const double* __restrict__ mu,
                                          int32_t sentinel, int32_t& out_a, int32_t& out_b) {
  /* singletons (d == 1) need no mu: they gather the sentinel and fall to chosen = 0 below */
  const int ga = da > 1 ? da : 0, gb = db > 1 ? db : 0;
#define MMQ_PJ(c, wv, g, j) (HAS_W ? mu[(j) < (g) ? (c)[j] : sentinel] * (double)((j) < (g) ? (wv)[j] : 0.f) \
                                   : mu[(j) < (g) ? (c)[j] : sentinel])
  double Sa[4], Sb[4];
  {
    double pa[4], pb[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { pa[j] = MMQ_PJ(ca, wa, ga, j); pb[j] = MMQ_PJ(cb, wb, gb, j); }
    Sa[0] = pa[0]; Sb[0] = pb[0];
#pragma unroll
    for (int j = 1; j < 4; ++j) { Sa[j] = Sa[j - 1] + pa[j]; Sb[j] = Sb[j - 1] + pb[j]; }
  }
  double na = Sa[3], nb = Sb[3];
  const int gmax = __reduce_max_sync(0xffffffffu, ga > gb ? ga : gb); /* warp-uniform */
  for (int j0 = 4; j0 < gmax; j0 += 4) {
    double pa[4], pb[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) { pa[q] = MMQ_PJ(ca, wa, ga, j0 + q); pb[q] = MMQ_PJ(cb, wb, gb, j0 + q); }
#pragma unroll
    for (int q = 0; q < 4; ++q) { na += pa[q]; nb += pb[q]; }
  }
  const double ta = ua * na, tb = ub * nb;
  int cha = -1, chb = -1;
#pragma unroll
  for (int j = 3; j >= 0; --j) { /* descending: the smallest hit index wins */
    if (j < ga && ta < Sa[j]) cha = j;
    if (j < gb && tb < Sb[j]) chb = j;
  }
  /* rows longer than 4 that were not decided in their first four members: rescan the tail */
  const bool more_a = cha < 0 && ga > 4, more_b = chb < 0 && gb > 4;
  if (__any_sync(0xffffffffu, more_a || more_b)) {
    double xa = Sa[3], xb = Sb[3];
    for (int j0 = 4; j0 < gmax; j0 += 4) {
      double pa[4], pb[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) { pa[q] = MMQ_PJ(ca, wa, ga, j0 + q); pb[q] = MMQ_PJ(cb, wb, gb, j0 + q); }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        xa += pa[q]; xb += pb[q];
        if (cha < 0 && j0 + q < ga && ta < xa) cha = j0 + q;
        if (chb < 0 && j0 + q < gb && tb < xb) chb = j0 + q;
      }
    }
  }
  /* d == 1; or rounding at the top end / all-zero row: last member with p > 0, else the last member */
  if (cha < 0 && da > 0) {
    cha = da - 1;
    if (da > 1)
      for (int j = da - 1; j >= 0; --j)
        if (MMQ_PJ(ca, wa, da, j) > 0.0) { cha = j; break; }
  }
  if (chb < 0 && db > 0) {
    chb = db - 1;
    if (db > 1)
      for (int j = db - 1; j >= 0; --j)
        if (MMQ_PJ(cb, wb, db, j) > 0.0) { chb = j; break; }
  }
#undef MMQ_PJ
  out_a = da > 0 ? ca[cha] : -1;
  out_b = db > 0 ? cb[chb] : -1;
}

/* K2 for the per-fragment layout (k == 1, no X kept).  A warp owns chunks of 64 consecutive
 * classes, two per lane.  Pipeline per warp, no block barrier anywhere:
 *   - row pointers of chunk i+2 are loaded into registers (one 128-bit load per lane),
 *   - the contiguous column (and weight) segment of chunk i+1 is fetched by ONE TMA bulk
 *     copy (cp.async.bulk, 16-byte aligned, completion on a per-warp mbarrier) into the
 *     other half of the warp's shared-memory double buffer,
 *   - chunk i is processed from shared memory: every lane gathers mu for its two classes,
 *     draws both from ONE Philox block (classes 4c .. 4c+3 share block c of the CAT stream)
 *     and the chosen columns are added to counts[], aggregated across the warp first.
 * Chunks whose segment exceeds the buffer are read straight from global memory. */
template <bool HAS_W, int SLAB>
__global__ void __launch_bounds__(MMQ_CAT_WARPS * 32, 3)
k_alloc_cat(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const float* __restrict__ w,
            const double* __restrict__ mu, int32_t* __restrict__ counts, int64_t m, int64_t n_chunks,
            uint32_t seed, uint32_t sweep, int64_t class_id_base, int32_t sentinel, const uint32_t* __restrict__ sweep_base) {
  if (sweep_base) sweep += *sweep_base;
  extern __shared__ __align__(16) unsigned char cat_smem[];
  constexpr int PER_WARP = 16 + 2 * SLAB * 4 * (HAS_W ? 2 : 1);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  unsigned char* wbase = cat_smem + wib * PER_WARP;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(wbase);            /* [2] */
  int32_t* sc = reinterpret_cast<int32_t*>(wbase + 16);           /* [2][SLAB] */
  float* sw = reinterpret_cast<float*>(wbase + 16 + 2 * SLAB * 4); /* [2][SLAB] when HAS_W */
  const int64_t chunk0 = (int64_t)blockIdx.x * MMQ_CAT_WARPS + wib;
  const int64_t nwarps = (int64_t)gridDim.x * MMQ_CAT_WARPS;
  if (chunk0 >= n_chunks) return;
  if (lane == 0) {
    mbar_init(&mbar[0], 1);
    mbar_init(&mbar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();

  /* raw row pointers of this lane's two classes in a chunk: q0, q1 (and q2 = next lane's q0) */
  auto load_rp = [&](int64_t chunk, int64_t& q0, int64_t& q1, int64_t& q2) {
    const int64_t r0 = chunk * MMQ_CAT_ROWS;
    const int64_t ia = r0 + 2 * lane;
    if (r0 + MMQ_CAT_ROWS <= m) {
      const longlong2 v = *reinterpret_cast<const longlong2*>(row_ptr + ia); /* 16-byte aligned: ia is even */
      q0 = v.x; q1 = v.y;
      q2 = (lane == 31) ? row_ptr[r0 + MMQ_CAT_ROWS] : 0;
    } else {
      q0 = row_ptr[ia < m ? ia : m];
      q1 = row_ptr[ia + 1 < m ? ia + 1 : m];
      q2 = row_ptr[ia + 2 < m ? ia + 2 : m];
    }
  };
  /* turn raw pointers into (start, offsets) and launch the bulk copy into buffer `buf` */
  struct ChunkState { int64_t start; int oa, ob, oe; bool staged; };
  uint32_t uses0 = 0, uses1 = 0; /* completed-phase counters of the two mbarriers */
  auto prepare = [&](int64_t chunk, int64_t q0, int64_t q1, int64_t q2, int buf) -> ChunkState {
    const int64_t r0 = chunk * MMQ_CAT_ROWS;
    if (r0 + MMQ_CAT_ROWS <= m) {
      const int64_t nx = __shfl_down_sync(0xffffffffu, q0, 1);
      if (lane != 31) q2 = nx;
    }
    const int64_t base = __shfl_sync(0xffffffffu, q0, 0);
    const int64_t end = __shfl_sync(0xffffffffu, q2, 31);
    ChunkState st;
    st.start = base & ~(int64_t)3; /* col / weight arrays are 256-byte aligned and padded by 4 entries */
    st.oa = (int)(q0 - st.start);
    st.ob = (int)(q1 - st.start);
    st.oe = (int)(q2 - st.start);
    const int span = (int)(end - st.start);
    st.staged = span <= SLAB && span > 0;
    if (st.staged && lane == 0) {
      const uint32_t bytes = (uint32_t)((span + 3) & ~3) * 4u;
      mbar_expect_tx(&mbar[buf], HAS_W ? 2 * bytes : bytes);
      bulk_g2s(sc + buf * SLAB, col + st.start, bytes, &mbar[buf]);
      if (HAS_W) bulk_g2s(sw + buf * SLAB, w + st.start, bytes, &mbar[buf]);
    }
    return st;
  };

  int64_t q0, q1, q2;
  load_rp(chunk0, q0, q1, q2);
  ChunkState cur = prepare(chunk0, q0, q1, q2, 0);
  if (chunk0 + nwarps < n_chunks) load_rp(chunk0 + nwarps, q0, q1, q2);
  int it = 0;
  for (int64_t chunk = chunk0; chunk < n_chunks; chunk += nwarps, ++it) {
    const int buf = it & 1;
    const int64_t nxt = chunk + nwarps;
    ChunkState next;
    next.staged = false; next.start = 0; next.oa = next.ob = next.oe = 0;
    if (nxt < n_chunks) next = prepare(nxt, q0, q1, q2, buf ^ 1);       /* bulk copy for chunk i+1 */
    if (nxt + nwarps < n_chunks) load_rp(nxt + nwarps, q0, q1, q2);     /* row pointers for chunk i+2 */

    /* uniforms of this lane's two classes (independent of the data in flight) */
    const uint64_t ca = (uint64_t)(class_id_base + chunk * MMQ_CAT_ROWS + 2 * lane);
    uint32_t wd[4] = {(uint32_t)(ca >> 2), (uint32_t)(ca >> 34), sweep, 0u};
    mmq_philox4x32_10(wd, seed, MMQ_STREAM_CAT);
    const uint32_t sa = (uint32_t)(ca & 3); /* word of class a in block ca >> 2; class b takes the next one */
    const double ua = mmq_uniform32(sa == 0 ? wd[0] : sa == 1 ? wd[1] : sa == 2 ? wd[2] : wd[3]);
    double ub;
    if (sa != 3) {
      ub = mmq_uniform32(sa == 0 ? wd[1] : sa == 1 ? wd[2] : wd[3]);
    } else { /* odd class_id_base only: class b opens the next block */
      const uint64_t cb = ca + 1;
      uint32_t w2[4] = {(uint32_t)(cb >> 2), (uint32_t)(cb >> 34), sweep, 0u};
      mmq_philox4x32_10(w2, seed, MMQ_STREAM_CAT);
      ub = mmq_uniform32(w2[0]);
    }
    const int da = cur.ob - cur.oa, db = cur.oe - cur.ob;
    int32_t ca_col, cb_col;
    if (cur.staged) {
      mbar_wait(&mbar[buf], (buf ? uses1 : uses0) & 1u);
      if (buf) ++uses1; else ++uses0;
      const int32_t* c0 = sc + buf * SLAB;
      const float* w0 = sw + buf * SLAB;
      cat_draw2<HAS_W>(c0 + cur.oa, w0 + cur.oa, da, ua, c0 + cur.ob, w0 + cur.ob, db, ub, mu, sentinel, ca_col, cb_col);
    } else {
      const int32_t* c0 = col + cur.start;
      const float* w0 = w + cur.start;
      cat_draw2<HAS_W>(c0 + cur.oa, w0 + cur.oa, da, ua, c0 + cur.ob, w0 + cur.ob, db, ub, mu, sentinel, ca_col, cb_col);
    }
    cat_red(counts, ca_col, lane);
    cat_red(counts, cb_col, lane);
    __syncwarp(); /* every lane is done with buffer `buf` before the next iteration refills it */
    cur = next;
  }
}

/* K3: counts[t] = sum over the transposed CSR of X — an atomic-free segmented
 * reduction, one warp per transcript.  src/mmseq.cpp:887, :895-899. */
__global__ void k_count_reduce(const int64_t* __restrict__ tptr, const uint32_t* __restrict__ perm,
                               const int32_t* __restrict__ x, int32_t* __restrict__ counts, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t t = warp0; t < n; t += nwarps) {
    int s = 0;
    for (int64_t q = tptr[t] + lane; q < tptr[t + 1]; q += 32) s += x[perm[q]];
    s = warp_sum_i(s);
    if (lane == 0) counts[t] = s;
  }
}

/* ---- K4: the Gamma update, 256 transcripts per block pass, rejections regrouped ----------------------------
 * Marsaglia-Tsang is a rejection sampler and the a < 1 boost an extra branch: with one transcript per lane running its
 * own loop, a warp pays for its slowest lane (measured in round 1: 13 of 32 lanes active on average).  Here an attempt
 * is a pure function of (transcript, sweep, attempt number) (include/mmq_sampler.h), so the block runs attempt 0 of all
 * its transcripts densely, queues the rejected ones (~5 %) in shared memory and runs attempt 1 of those densely, and so
 * on; the boosts (transcripts without fragments: shape alpha < 1) are queued and done densely too.  Same values, bit
 * for bit, as the sequential mmq_gamma of the CPU replay. */
#define MMQ_GAMMA_THREADS 256
struct gamma_smem {
  double d[MMQ_GAMMA_THREADS], c[MMQ_GAMMA_THREADS], v[MMQ_GAMMA_THREADS], boost[MMQ_GAMMA_THREADS];
  double lu[MMQ_GAMMA_THREADS], lx2[MMQ_GAMMA_THREADS], lv[MMQ_GAMMA_THREADS]; /* undecided attempts: the log test's inputs */
  int32_t id[MMQ_GAMMA_THREADS], cnt_t[MMQ_GAMMA_THREADS];
  int q[2][MMQ_GAMMA_THREADS], ql[MMQ_GAMMA_THREADS], qb[MMQ_GAMMA_THREADS];
  int n[4]; /* retry queues 0 / 1, boosts, log tests */
};
/* Every thread of the block calls this with its transcript t (or t < 0: none) and its count c; returns the new mu[t]. */
__device__ __forceinline__ double gamma_block(gamma_smem& S, int64_t t, int32_t c, double rate, double alpha, uint32_t seed, uint32_t sweep) {
  const int tid = threadIdx.x, lane = tid & 31;
  const bool valid = t >= 0;
  double a = alpha + (double)c;
  const bool boosted = valid && a < 1.0;
  if (a < 1.0) a += 1.0;
  const mmq_gamma_par par = mmq_gamma_setup(a);
  __syncthreads(); /* the previous pass is done with S */
  S.d[tid] = par.d; S.c[tid] = par.c; S.id[tid] = (int32_t)t; S.cnt_t[tid] = c; S.boost[tid] = 1.0;
  if (tid < 4) S.n[tid] = 0;
  __syncthreads();
  /* round r: attempt r of the transcripts still open (round 0: all of them, one per thread), then the log tests of
   * the attempts the squeeze did not decide, both densely; what is rejected goes to the other queue */
  for (uint32_t r = 0;; ++r) {
    const int ncur = r == 0 ? MMQ_GAMMA_THREADS : S.n[(r - 1) & 1];
    if (ncur == 0) break;
    if (r > 0) {
      __syncthreads();
      if (tid == 0) { S.n[r & 1] = 0; S.n[3] = 0; }
      __syncthreads();
    }
    if ((tid & ~31) < ncur) {
      int st = 1, item = tid;
      double v = 0.0, x2 = 0.0, u = 0.0;
      if (tid < ncur) {
        mmq_gamma_par q = par;
        if (r > 0) { item = S.q[(r - 1) & 1][tid]; q.d = S.d[item]; q.c = S.c[item]; }
        if (r > 0 || valid) {
          mmq_rng g;
          mmq_rng_init(&g, seed, MMQ_STREAM_GAMMA, (uint64_t)S.id[item], sweep);
          st = mmq_gamma_try(&g, r, q, &v, &x2, &u);
        }
        if (st == 1) S.v[item] = v;
      }
      const int pos = queue_slot(&S.n[r & 1], st == 0, lane);
      if (pos >= 0) S.q[r & 1][pos] = item;
      const int pl = queue_slot(&S.n[3], st == 2, lane);
      if (pl >= 0) { S.ql[pl] = item; S.lu[pl] = u; S.lx2[pl] = x2; S.lv[pl] = v; }
    }
    __syncthreads();
    const int nl = S.n[3];
    if ((tid & ~31) < nl) {
      bool rej = false;
      int item = 0;
      if (tid < nl) {
        item = S.ql[tid];
        const double v = S.lv[tid];
        if (mmq_gamma_logtest(S.lu[tid], S.lx2[tid], v, S.d[item])) S.v[item] = v;
        else rej = true;
      }
      const int pos = queue_slot(&S.n[r & 1], rej, lane);
      if (pos >= 0) S.q[r & 1][pos] = item;
    }
    __syncthreads();
  }
  const int pb = queue_slot(&S.n[2], boosted, lane);
  if (pb >= 0) S.qb[pb] = tid;
  __syncthreads();
  const int nb = S.n[2];
  if (tid < nb) {
    const int item = S.qb[tid];
    mmq_rng g;
    mmq_rng_init(&g, seed, MMQ_STREAM_GAMMA, (uint64_t)S.id[item], sweep);
    S.boost[item] = mmq_gamma_boost(&g, alpha + (double)S.cnt_t[item]);
  }
  __syncthreads();
  return S.boost[tid] * par.d * S.v[tid] / rate;
}

/* ---- posterior fragment-count moments (mmq_count_moments_begin) ----
 * Rows [0, n) of the accumulators are the transcripts, [n, n + groups) the identical sets and then the genes.  Every
 * sweep adds each row's count c to sum (u64) and c^2 to sq (u128): integer sums, so the result does not depend on the
 * order of the additions (GPU count, launch geometry, graph or not).  A group's count is summed within the sweep first
 * (gsum, int32, warp-aggregated atomics), since its square is not the sum of its members' squares. */
struct mmq_cnt_acc {
  unsigned long long* sum; /* [rows] */
  unsigned __int128* sq;   /* [rows] */
  const int2* group;       /* [n] (identical set, n_ident + gene) of each transcript, -1 = none; null: no groups */
  int32_t* gsum;           /* [groups] this sweep's group counts, zero between sweeps */
};

/* a group's share of the warp's counts: one atomic per distinct group in the warp.  All 32 lanes call it. */
__device__ __forceinline__ void count_group_add(int32_t* gsum, int key, int32_t c) {
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  const int s = __reduce_add_sync(peers, c);
  if (key >= 0 && s != 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(gsum + key, s);
}

/* Every thread of the block calls this with its transcript t (t < 0: none) and the count the Gamma step uses. */
__device__ __forceinline__ void count_acc(const mmq_cnt_acc& A, int64_t t, int32_t c) {
  if (t >= 0) {
    A.sum[t] += (unsigned long long)c;
    A.sq[t] += (unsigned __int128)((unsigned long long)c * (unsigned long long)c);
  }
  if (A.group) {
    const int2 g = t >= 0 ? A.group[t] : make_int2(-1, -1);
    count_group_add(A.gsum, g.x, c);
    count_group_add(A.gsum, g.y, c);
  }
}

/* The per-sweep group step: each group's sweep count and its square into rows n + g; gsum back to zero. */
__global__ void k_count_groups(mmq_cnt_acc A, int64_t n, int64_t groups) {
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < groups; g += (int64_t)gridDim.x * blockDim.x) {
    const int32_t c = A.gsum[g];
    if (c == 0) continue;
    A.gsum[g] = 0;
    A.sum[n + g] += (unsigned long long)c;
    A.sq[n + g] += (unsigned __int128)((unsigned long long)c * (unsigned long long)c);
  }
}

/* The trace rule of src/mmseq.cpp:911-917: sweep s is recorded in slot s / stride when s % stride == 0 and that slot is
 * < trace_len.  stride > 0. */
__host__ __device__ __forceinline__ bool trace_recorded(uint32_t sweep, int stride, int trace_len) {
  return sweep % (uint32_t)stride == 0 && sweep / (uint32_t)stride < (uint32_t)trace_len;
}

/* ---- peer memory (NVLink) ----------------------------------------------------------------------
 * Every rank owns a peer-mapped block (mmq_internal.h: MMQ_P2P_*): two flag arrays, the two parity
 * buffers of its count vector and its mu vector.  Flags are written with st.release.sys into the
 * peers' blocks and polled locally with ld.acquire.sys. */
__device__ __forceinline__ void p2p_publish(int32_t* flag, int32_t epoch) {
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
}
__device__ __forceinline__ void p2p_wait(const int32_t* flag, int32_t epoch) {
  int32_t v;
  do { asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory"); } while (v < epoch);
}
struct mmq_p2p_args {
  char* base[MMQ_P2P_MAX]; /* peer-mapped block of every rank (own block included) */
  int64_t off_counts;      /* this epoch's parity buffer inside a block */
  int64_t off_reset;       /* the other parity buffer (own block only) */
  int64_t off_mu;
  int nranks, rank;
  int32_t epoch;                /* + *epoch_base when replayed from a CUDA graph */
  const int32_t* epoch_base;
};

/* The exchange's barrier at the start of a Gamma kernel: block 0 tells every rank that this rank's allocation of the
 * epoch is done, and every block waits for the peers'.  One thread per peer polls that peer's flag (own allocation is
 * complete by stream order: no wait on self): the waits overlap instead of one system-scope round trip after the
 * other; the block barrier orders everybody else's loads behind them.  (& rather than &&: one predicate, and
 * threadIdx.x is read once for both tests.) */
__device__ __forceinline__ void p2p_arrive_and_wait(const mmq_p2p_args& a, int32_t epoch) {
  int32_t* own = reinterpret_cast<int32_t*>(a.base[a.rank]);
  if ((blockIdx.x == 0) & (threadIdx.x < a.nranks))
    p2p_publish(reinterpret_cast<int32_t*>(a.base[threadIdx.x]) + MMQ_P2P_FLAG_ALLOC + 8 * a.rank, epoch);
  if (threadIdx.x < a.nranks && (int)threadIdx.x != a.rank) p2p_wait(own + MMQ_P2P_FLAG_ALLOC + 8 * threadIdx.x, epoch);
  __syncthreads();
}

/* transcript t's count summed over the ranks: all ranks' counts in flight at once — with a run-time trip count the adds
 * serialise the peer loads, one NVLink round trip after the other */
__device__ __forceinline__ int32_t p2p_count(const mmq_p2p_args& a, int64_t t) {
  int32_t v[MMQ_P2P_MAX];
#pragma unroll
  for (int r = 0; r < MMQ_P2P_MAX; ++r) v[r] = r < a.nranks ? __ldcv(reinterpret_cast<const int32_t*>(a.base[r] + a.off_counts) + t) : 0;
  int32_t c = 0;
#pragma unroll
  for (int r = 0; r < MMQ_P2P_MAX; ++r) c += v[r];
  return c;
}

/* K4 (+K5 capture): mu[t] ~ Gamma(alpha + counts[t], rate beta + l[t]); counts are cleared for the next sweep (to
 * counts_base: classes the allocation kernels skip, the singletons); a recorded sweep stores mu into its trace slot.
 * src/mmseq.cpp:904-917.  Compile-time variants (the kernel is bound by the latency of one pass, so each one is the
 * machine code it would be on its own):
 *   P2P: src is the peer blocks (mmq_p2p_args), the all-reduce over peer memory that multi-GPU runs use by default.
 *        Every rank reads the count vectors of ALL ranks (parity buffer src.off_counts), draws every Gamma variate,
 *        keeps the summed counts and clears its own other parity buffer (src.off_reset).  One barrier.
 *        Else src is the own count vector, read and cleared in place.  One parameter whose type follows P2P, rather
 *        than both: the parameters after it then sit at the constant-bank alignment they would have in a kernel of
 *        either kind alone, and ptxas pairs their loads the same way.
 *   ACC: also add the counts into the moment accumulators A (mmq_count_moments_begin).  Without ACC, A is unused. */
template <bool ACC, bool P2P>
__global__ void __launch_bounds__(MMQ_GAMMA_THREADS, 5)
k_gamma(std::conditional_t<P2P, mmq_p2p_args, int32_t* __restrict__> src, const int32_t* __restrict__ counts_base,
        const double* __restrict__ len, double* __restrict__ mu, double* __restrict__ trace, int stride, int trace_len, int64_t n,
        double alpha, double beta, uint32_t seed, uint32_t sweep, int32_t* __restrict__ counts_copy,
        const uint32_t* __restrict__ sweep_base, mmq_cnt_acc A) {
  __shared__ gamma_smem S;
  if (sweep_base) sweep += *sweep_base;
  int32_t epoch = 0;
  if constexpr (P2P) {
    epoch = src.epoch + (src.epoch_base ? *src.epoch_base : 0);
    p2p_arrive_and_wait(src, epoch);
  }
  double* trace_col = nullptr;
  if (trace && stride > 0 && trace_recorded(sweep, stride, trace_len)) trace_col = trace + sweep / (uint32_t)stride;
  int32_t* reset;
  if constexpr (P2P) reset = reinterpret_cast<int32_t*>(src.base[src.rank] + src.off_reset);
  else reset = src;
  for (int64_t t0 = (int64_t)blockIdx.x * MMQ_GAMMA_THREADS; t0 < n; t0 += (int64_t)gridDim.x * MMQ_GAMMA_THREADS) {
    const int64_t t = t0 + threadIdx.x < n ? t0 + threadIdx.x : -1;
    int32_t c = 0;
    double rate = 1.0;
    if (t >= 0) {
      if constexpr (P2P) c = p2p_count(src, t);
      else c = src[t];
      reset[t] = counts_base ? counts_base[t] : 0;
      if (counts_copy) counts_copy[t] = c;
      rate = beta + len[t];
    }
    if (ACC) count_acc(A, t, c);
    const double v = gamma_block(S, t, c, rate, alpha, seed, sweep);
    if (t >= 0) {
      mu[t] = v;
      if (trace_col) trace_col[t * (int64_t)trace_len] = v;
    }
  }
  /* the mu flags advance too, so that a later k_gamma_rs (which waits for them) sees a monotone epoch: every rank
   * wrote its own mu, nothing to wait for */
  if constexpr (P2P)
    if (blockIdx.x == 0 && threadIdx.x < src.nranks)
      p2p_publish(reinterpret_cast<int32_t*>(src.base[threadIdx.x]) + MMQ_P2P_FLAG_MU + 8 * src.rank, epoch);
}

/* The reduce-scatter alternative to k_gamma<ACC, true> (mmq_tune knob 6; the all-reduce is the default, DESIGN §7):
 * reduce-scatter + Gamma + all-gather in ONE kernel.  Rank r owns the transcripts
 * [n r / N, n (r+1) / N): after the "allocation done" barrier it sums the N count vectors for its slice
 * only ((N-1) 4n/N bytes over NVLink instead of (N-1) 4n), draws n/N Gamma variates instead of n, and
 * stores each new mu into the mu vector of EVERY rank (P2P stores).  The last block to finish publishes
 * "mu slice written" to the peers and waits for theirs, so that when the kernel completes the whole mu
 * vector is in place on this rank: the next allocation kernel needs no other synchronisation than stream
 * order.  The other parity buffer of the own counts is reset for the next sweep (all of it, by all blocks). */
__global__ void __launch_bounds__(MMQ_GAMMA_THREADS)
k_gamma_rs(mmq_p2p_args a, const int32_t* __restrict__ counts_base, const double* __restrict__ len, int64_t n,
           double alpha, double beta, uint32_t seed, uint32_t sweep, const uint32_t* __restrict__ sweep_base) {
  __shared__ gamma_smem S;
  if (sweep_base) sweep += *sweep_base;
  const int32_t epoch = a.epoch + (a.epoch_base ? *a.epoch_base : 0);
  int32_t* own = reinterpret_cast<int32_t*>(a.base[a.rank]);
  p2p_arrive_and_wait(a, epoch);
  const int64_t s0 = n * a.rank / a.nranks, s1 = n * (a.rank + 1) / a.nranks;
  for (int64_t t0 = s0 + (int64_t)blockIdx.x * MMQ_GAMMA_THREADS; t0 < s1; t0 += (int64_t)gridDim.x * MMQ_GAMMA_THREADS) {
    const int64_t t = t0 + threadIdx.x < s1 ? t0 + threadIdx.x : -1;
    int32_t c = 0;
    double rate = 1.0;
    if (t >= 0) {
      c = p2p_count(a, t);
      rate = beta + len[t];
    }
    const double v = gamma_block(S, t, c, rate, alpha, seed, sweep);
    if (t >= 0)
      for (int r = 0; r < a.nranks; ++r) reinterpret_cast<double*>(a.base[r] + a.off_mu)[t] = v;
  }
  int32_t* reset = reinterpret_cast<int32_t*>(a.base[a.rank] + a.off_reset);
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
    reset[t] = counts_base ? counts_base[t] : 0;
  /* the block's peer stores are ordered before its sign-off: bar.sync makes them happen before thread 0's system-scope
   * fence (one fence per block; a fence per thread cost 8 us per sweep) */
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    unsigned int* done = reinterpret_cast<unsigned int*>(own + MMQ_P2P_DONE);
    if (atomicAdd(done, 1u) == gridDim.x - 1) { /* last block of this rank */
      *done = 0u;
      __threadfence_system();
      for (int r = 0; r < a.nranks; ++r)
        p2p_publish(reinterpret_cast<int32_t*>(a.base[r]) + MMQ_P2P_FLAG_MU + 8 * a.rank, epoch);
      for (int r = 0; r < a.nranks; ++r)
        if (r != a.rank) p2p_wait(own + MMQ_P2P_FLAG_MU + 8 * r, epoch);
    }
  }
}

/* trace capture of a multi-GPU sweep: after k_gamma_rs has completed mu holds the values of all ranks */
__global__ void k_trace_capture(const double* __restrict__ mu, double* __restrict__ trace, int stride, int trace_len, int64_t n,
                                uint32_t sweep, const uint32_t* __restrict__ sweep_base) {
  if (sweep_base) sweep += *sweep_base;
  if (!trace_recorded(sweep, stride, trace_len)) return;
  double* col = trace + sweep / (uint32_t)stride;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x)
    col[t * (int64_t)trace_len] = mu[t];
}

__global__ void k_set2_u32(uint32_t* p, uint32_t a, uint32_t b) { p[0] = a; p[1] = b; }
__global__ void k_add2_u32(uint32_t* p, uint32_t v) { p[0] += v; p[1] += v; }

/* -------------------------------------------------------------- NCCL */

namespace {
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi g_nccl;

const char* nccl_load() {
  if (g_nccl.lib) return nullptr;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* lib = nullptr;
  for (const char* nm : names) { lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
  if (!lib) return "cannot dlopen libnccl.so.2";
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(lib, "ncclCommInitRank");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(lib, "ncclAllReduce");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(lib, "ncclCommDestroy");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(lib, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy) return "libnccl lacks a required symbol";
  g_nccl.lib = lib;
  return nullptr;
}
}  // namespace

int mmq_allreduce(mmq_handle* h, void* buf, size_t count, int type) {
  if (h->nranks <= 1 || !h->comm) return MMQ_OK;
  const ncclDataType_t dt = type == 1 ? ncclFloat64 : type == 2 ? ncclInt64 : ncclInt32;
  ncclResult_t r = g_nccl.AllReduce(buf, buf, count, dt, ncclSum, (ncclComm_t)h->comm, h->stream);
  if (r != ncclSuccess)
    return mmq_fail(h, MMQ_ERR_NCCL, std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"));
  return MMQ_OK;
}

/* ---------------------------------------------------------------- C ABI */

extern "C" {

const char* mmq_version(void) { return "mmseq-b200 0.1 (hot path of eturro/mmseq 1.0.11)"; }
int mmq_release_cache(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess) return MMQ_ERR_CUDA;
  int cur = 0;
  cudaGetDevice(&cur);
  for (int d = 0; d < ndev && d < 16; ++d) {
    if (device >= 0 && d != device) continue;
    cudaSetDevice(d);
    std::lock_guard<std::mutex> lk(g_cache[d].mu); /* cached blocks are idle by contract (mmq_cache_free) */
    cache_drop_all(g_cache[d]);
  }
  cudaSetDevice(cur);
  return MMQ_OK;
}

int64_t mmq_launch_count(void) { return (int64_t)g_mmq_launches.load(); }

const char* mmq_last_error(const mmq_handle* h) { return h ? h->err.c_str() : g_mmq_create_err.c_str(); }

static void drop_graph(mmq_handle* h);
static int p2p_adopt(mmq_handle* h, int rank, int nranks);

static int upload(mmq_handle* h, void** dst, const void* src, size_t bytes, size_t pad = 0) {
  int rc = mmq_dev_alloc(h, dst, bytes + pad);
  if (rc) return rc;
  if (bytes) MMQ_CUDA(h, cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
  return MMQ_OK;
}

/* Tiles of the general allocation kernel: greedily as many consecutive classes as fit the
 * warp's staging slab (and one per lane); a class longer than the slab is a tile of its own.
 * rp_host may be null: the row pointers are then read back from the device. */
static int build_tiles(mmq_handle* h, const int64_t* rp_host) {
  if (h->tile_start) return MMQ_OK;
  std::vector<int64_t> tmp;
  if (!rp_host) {
    tmp.resize((size_t)h->m + 1);
    MMQ_CUDA(h, cudaMemcpyAsync(tmp.data(), h->row_ptr, sizeof(int64_t) * tmp.size(), cudaMemcpyDeviceToHost, h->stream));
    MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
    rp_host = tmp.data();
  }
  std::vector<int64_t> ts;
  ts.reserve((size_t)(h->m / 16 + 2));
  int64_t r = 0;
  while (r < h->m) {
    ts.push_back(r);
    int64_t e = r + 1;
    while (e < h->m && e - r < 32 && rp_host[e + 1] - rp_host[r] <= MMQ_ALLOC_CAP) ++e;
    r = e;
  }
  ts.push_back(h->m);
  h->n_tiles = (int64_t)ts.size() - 1;
  int rc = mmq_dev_alloc(h, (void**)&h->tile_start, sizeof(int64_t) * ts.size());
  if (rc) return rc;
  MMQ_CUDA(h, cudaMemcpyAsync(h->tile_start, ts.data(), sizeof(int64_t) * ts.size(), cudaMemcpyHostToDevice, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream)); /* ts is a host temporary */
  return MMQ_OK;
}

static int build_transpose(mmq_handle* h) {
  if (h->tptr) return MMQ_OK; /* built on first use: the fused Gibbs path never needs it */
  const int64_t nnz = h->nnz, n = h->n, m = h->m;
  int rc;
  if ((rc = mmq_dev_alloc(h, (void**)&h->tptr, sizeof(int64_t) * (size_t)(n + 1)))) return rc;
  if ((rc = mmq_dev_alloc(h, (void**)&h->perm, sizeof(uint32_t) * (size_t)nnz))) return rc;
  if ((rc = mmq_dev_alloc(h, (void**)&h->trow, sizeof(int32_t) * (size_t)nnz))) return rc;
  if (nnz == 0) {
    MMQ_CUDA(h, cudaMemsetAsync(h->tptr, 0, sizeof(int64_t) * (size_t)(n + 1), h->stream));
    return MMQ_OK;
  }
  int32_t* keys_out = nullptr;
  uint32_t* iota = nullptr;
  void* temp = nullptr;
  size_t temp_bytes = 0;
  MMQ_CUDA(h, mmq_cache_malloc(&keys_out, sizeof(int32_t) * (size_t)nnz));
  MMQ_CUDA(h, mmq_cache_malloc(&iota, sizeof(uint32_t) * (size_t)nnz));
  const int grid = mmq_grid_for(nnz, 256, h->num_sms * 8);
  k_iota<<<grid, 256, 0, h->stream>>>(iota, nnz);
  MMQ_LAUNCHED(h);
  int end_bit = 1;
  while (end_bit < 31 && ((int64_t)1 << end_bit) < n) ++end_bit;
  /* stable LSD radix sort of (column, position): positions stay ascending within a column */
  MMQ_CUDA(h, cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, h->col, keys_out, iota, h->perm, nnz, 0, end_bit, h->stream));
  MMQ_CUDA(h, mmq_cache_malloc(&temp, temp_bytes));
  MMQ_CUDA(h, cub::DeviceRadixSort::SortPairs(temp, temp_bytes, h->col, keys_out, iota, h->perm, nnz, 0, end_bit, h->stream));
  k_tptr<<<grid, 256, 0, h->stream>>>(keys_out, nnz, n, h->tptr);
  MMQ_LAUNCHED(h);
  k_trow<<<grid, 256, 0, h->stream>>>(h->perm, h->row_ptr, m, nnz, h->trow);
  MMQ_LAUNCHED(h);
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  mmq_cache_free(keys_out);
  mmq_cache_free(iota);
  mmq_cache_free(temp);
  return MMQ_OK;
}

int mmq_create(const mmq_problem* p, int device, mmq_handle** out) {
  if (!out) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_create: out is NULL");
  *out = nullptr;
  if (!p || p->n <= 0 || p->m < 0 || p->nnz < 0 || !p->row_ptr || (!p->col && p->nnz > 0) || !p->len)
    return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_create: bad problem (n <= 0, m < 0 or NULL arrays)");
  if (p->nnz >= (int64_t)0xffffffffll) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_create: nnz per shard must be < 2^32");
  if (p->n >= (int64_t)0x7fffffffll || p->m >= (int64_t)0x7fffffffll) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_create: n and m per shard must be < 2^31");
  if (p->row_ptr[0] != 0 || p->row_ptr[p->m] != p->nnz) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_create: row_ptr[0] != 0 or row_ptr[m] != nnz");
  if (!(p->alpha > 0.0) || !(p->beta >= 0.0)) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_create: alpha must be > 0 and beta >= 0");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    char buf[256];
    snprintf(buf, sizeof buf, "mmq_create: no CUDA device (%s); this library has no CPU path", cudaGetErrorString(e));
    return mmq_fail(nullptr, MMQ_ERR_CUDA, buf);
  }
  if (device < 0 || device >= ndev) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_create: device index out of range");
  mmq_handle* h = new mmq_handle();
  h->device = device;
  /* MMQ_CREATE_TIMING=1: host wall clock of the phases below on stderr (no extra synchronisation) */
  static const bool timing = [] { const char* e = getenv("MMQ_CREATE_TIMING"); return e && atoi(e) != 0; }();
  auto t_last = std::chrono::steady_clock::now();
  auto tick = [&](const char* what) {
    if (!timing) return;
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[mmq_create] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
    t_last = now;
  };
#define CREATE_TRY(expr)                      \
  do {                                        \
    int rc__ = (expr);                        \
    if (rc__) {                               \
      g_mmq_create_err = h->err;              \
      mmq_destroy(h);                         \
      return rc__;                            \
    }                                         \
  } while (0)
  auto cuda_try = [&](cudaError_t ce, const char* what) -> int {
    return ce == cudaSuccess ? MMQ_OK : mmq_cuda_fail(h, ce, what, __FILE__, __LINE__);
  };
  CREATE_TRY(cuda_try(cudaSetDevice(device), "cudaSetDevice"));
  CREATE_TRY(cuda_try(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking), "cudaStreamCreate"));
  h->own_stream = true;
  CREATE_TRY(cuda_try(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device), "cudaDeviceGetAttribute")); /* cudaGetDeviceProperties takes ~10 ms */
  tick("device, stream");
  h->n = p->n; h->m = p->m; h->nnz = p->nnz; h->class_id_base = p->class_id_base;
  h->alpha = p->alpha; h->beta = p->beta;
  h->has_k = p->k != nullptr; h->has_w = p->weight != nullptr;
  for (int64_t t = 0; t < p->n; ++t)
    if (!(p->len[t] > 0.0)) { h->err = "mmq_create: transcript length must be > 0 (src/mmseq.cpp:604-607)"; CREATE_TRY(MMQ_ERR_ARG); }
  tick("length check");
  {
    const size_t n = (size_t)p->n, m = (size_t)p->m, nnz = (size_t)p->nnz;
    size_t want = 8 * (m + 1) + 4 * nnz + 16 + (h->has_k ? 4 * m : 0) + (p->class_id ? 8 * m : 0) + (h->has_w ? 4 * nnz + 16 : 0) +
                  8 * n + 2 * 8 * (n + 1) + 8 * n + 4 * n + 4 * n + 8 * std::max<size_t>(m, 1) + 8 * (size_t)h->num_sms * 8 + 32;
    if (!h->has_k) want += (h->has_w ? 2 : 1) * 4 * (nnz + 128 * 12 + 128) + 4 * n + 4096; /* the segment plan's packed copies */
    else if (!h->has_w) want += 4 * (nnz + nnz / 8) + 6 * (m + m / 4) + 4 * n + (1 << 16);     /* the class plan's (an estimate: what does not fit is allocated separately) */
    want += 64 * 256;                                                                      /* alignment of the pieces */
    void* a = nullptr;
    if (mmq_cache_malloc_raw(&a, want) == cudaSuccess && cudaMemsetAsync(a, 0, want, h->stream) == cudaSuccess) { h->arena = (char*)a; h->arena_cap = want; }
    else cudaGetLastError(); /* fall back to separate allocations */
  }
  CREATE_TRY(upload(h, (void**)&h->row_ptr, p->row_ptr, sizeof(int64_t) * (size_t)(p->m + 1)));
  CREATE_TRY(upload(h, (void**)&h->col, p->col, sizeof(int32_t) * (size_t)p->nnz, 16)); /* +4 entries: aligned 128-bit staging may over-read */
  if (h->has_k) CREATE_TRY(upload(h, (void**)&h->k, p->k, sizeof(int32_t) * (size_t)p->m));
  if (p->class_id) {
    if (!h->has_k) { h->err = "mmq_create: class_id needs k (the k == 1 kernels pair consecutive class ids)"; CREATE_TRY(MMQ_ERR_ARG); }
    CREATE_TRY(upload(h, (void**)&h->class_id, p->class_id, sizeof(int64_t) * (size_t)p->m));
  }
  if (h->has_w) CREATE_TRY(upload(h, (void**)&h->w, p->weight, sizeof(float) * (size_t)p->nnz, 16));
  CREATE_TRY(upload(h, (void**)&h->len, p->len, sizeof(double) * (size_t)p->n));
  CREATE_TRY(mmq_dev_alloc(h, (void**)&h->mu, sizeof(double) * (size_t)(p->n + 1))); /* mu[n] == 0: gather sentinel */
  CREATE_TRY(mmq_dev_alloc(h, (void**)&h->mu_tmp, sizeof(double) * (size_t)(p->n + 1)));
  CREATE_TRY(mmq_dev_alloc(h, (void**)&h->acc, sizeof(double) * (size_t)p->n));
  CREATE_TRY(mmq_dev_alloc(h, (void**)&h->counts, sizeof(int32_t) * (size_t)p->n));
  CREATE_TRY(mmq_dev_alloc(h, (void**)&h->uh, sizeof(int32_t) * (size_t)p->n));
  CREATE_TRY(mmq_dev_alloc(h, (void**)&h->rterm, sizeof(double) * (size_t)std::max<int64_t>(p->m, 1)));
  h->partial_cap = h->num_sms * 8;
  CREATE_TRY(mmq_dev_alloc(h, (void**)&h->partial, sizeof(double) * (size_t)h->partial_cap));
  CREATE_TRY(mmq_dev_alloc(h, (void**)&h->scalars, sizeof(double) * 4));
  CREATE_TRY(cuda_try(cudaMemsetAsync(h->counts, 0, sizeof(int32_t) * (size_t)p->n, h->stream), "memset counts"));
  CREATE_TRY(cuda_try(cudaMemsetAsync(h->mu, 0, sizeof(double) * (size_t)(p->n + 1), h->stream), "memset mu"));
  CREATE_TRY(cuda_try(cudaMemsetAsync(h->mu_tmp, 0, sizeof(double) * (size_t)(p->n + 1), h->stream), "memset mu_tmp"));
  tick("allocations, copies queued");
  if (!h->has_k) CREATE_TRY(mmq_seg_scan(h, p->row_ptr)); /* host scan, overlapped with the queued H2D copies */
  tick("segment scan (host)");
  if (p->m > 0) { /* structural checks on the device: no O(nnz) host loop in front of the upload */
    int* d_flags = (int*)h->scalars;
    CREATE_TRY(cuda_try(cudaMemsetAsync(d_flags, 0, sizeof(int), h->stream), "memset flags"));
    k_validate<<<mmq_grid_for(p->m, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->row_ptr, h->col, p->m, p->n, d_flags);
    g_mmq_launches.fetch_add(1);
    int flags = 0;
    CREATE_TRY(cuda_try(cudaMemcpyAsync(&flags, d_flags, sizeof(int), cudaMemcpyDeviceToHost, h->stream), "copy flags"));
    CREATE_TRY(cuda_try(cudaStreamSynchronize(h->stream), "validate"));
    if (flags & 1) { h->err = "mmq_create: empty or negative-length class row"; CREATE_TRY(MMQ_ERR_ARG); }
    if (flags & 2) { h->err = "mmq_create: column index out of range"; CREATE_TRY(MMQ_ERR_ARG); }
    if (flags & 4) { h->err = "mmq_create: columns must be strictly ascending within a class (src/mmseq.cpp:412)"; CREATE_TRY(MMQ_ERR_ARG); }
  }
  tick("H2D copies + validation");
  if (!h->has_k) CREATE_TRY(mmq_seg_plan(h));
  if (h->has_k) CREATE_TRY(mmq_cls_plan(h, p));
  if (h->has_k && !h->cls_ready) CREATE_TRY(build_tiles(h, p->row_ptr)); /* the general kernel's tiles; otherwise on its first use */
  tick("tiles");
  CREATE_TRY(cuda_try(cudaStreamSynchronize(h->stream), "cudaStreamSynchronize"));
  tick("segment / class plan");
  h->arena_cap = h->arena_off; /* closed: later allocations (trace, transpose, peer buffers) are their own */
#undef CREATE_TRY
  *out = h;
  return MMQ_OK;
}

void mmq_destroy(mmq_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  drop_graph(h);
  for (void* p : h->p2p_opened) if (p) cudaIpcCloseMemHandle(p);
  for (cudaEvent_t e : h->ev_alloc) cudaEventDestroy(e);
  for (cudaEvent_t e : h->ev_gamma) cudaEventDestroy(e);
  if (h->stream2) { cudaStreamSynchronize(h->stream2); cudaStreamDestroy(h->stream2); }
  if (h->stream3) { cudaStreamSynchronize(h->stream3); cudaStreamDestroy(h->stream3); }
  if (h->stream4) { cudaStreamSynchronize(h->stream4); cudaStreamDestroy(h->stream4); }
  if (h->ev_join4) cudaEventDestroy(h->ev_join4);
  if (h->stream5) { cudaStreamSynchronize(h->stream5); cudaStreamDestroy(h->stream5); }
  if (h->ev_join5) cudaEventDestroy(h->ev_join5);
  if (h->stream6) { cudaStreamSynchronize(h->stream6); cudaStreamDestroy(h->stream6); }
  if (h->ev_fork6) cudaEventDestroy(h->ev_fork6);
  if (h->ev_join6) cudaEventDestroy(h->ev_join6);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_join3) cudaEventDestroy(h->ev_join3);
  if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy((ncclComm_t)h->comm);
  /* the blocks go back to the cache: nothing may still be running on them — every stream this handle ever launched on was
   * synchronised above (no cudaDeviceSynchronize: another thread may be capturing a graph on its own stream) */
  for (void* p : h->allocs) mmq_cache_free(p);
  if (h->arena) mmq_cache_free(h->arena);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int mmq_set_stream(mmq_handle* h, void* s) {
  if (!h) return MMQ_ERR_ARG;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  h->stream = (cudaStream_t)s;
  h->own_stream = false;
  return MMQ_OK;
}
void* mmq_get_stream(mmq_handle* h) { return h ? (void*)h->stream : nullptr; }

int mmq_synchronize(mmq_handle* h) {
  if (!h) return MMQ_ERR_ARG;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

int64_t mmq_device_bytes(const mmq_handle* h) { return h ? h->bytes : 0; }

int mmq_comm_id(char id[128]) {
  const char* e = nccl_load();
  if (e) return mmq_fail(nullptr, MMQ_ERR_NCCL, e);
  ncclUniqueId uid;
  static_assert(sizeof(uid) == 128, "ncclUniqueId is 128 bytes");
  ncclResult_t r = g_nccl.GetUniqueId(&uid);
  if (r != ncclSuccess) return mmq_fail(nullptr, MMQ_ERR_NCCL, "ncclGetUniqueId failed");
  memcpy(id, &uid, 128);
  return MMQ_OK;
}

int mmq_comm_init(mmq_handle* h, const char id[128], int rank, int nranks) {
  if (!h || !id || nranks < 1 || rank < 0 || rank >= nranks) return mmq_fail(h, MMQ_ERR_ARG, "mmq_comm_init: bad arguments");
  if (nranks == 1) { h->rank = 0; h->nranks = 1; return MMQ_OK; }
  const char* e = nccl_load();
  if (e) return mmq_fail(h, MMQ_ERR_NCCL, e);
  MMQ_CUDA(h, cudaSetDevice(h->device));
  ncclUniqueId uid;
  memcpy(&uid, id, 128);
  ncclComm_t comm;
  ncclResult_t r = g_nccl.CommInitRank(&comm, nranks, uid, rank);
  if (r != ncclSuccess)
    return mmq_fail(h, MMQ_ERR_NCCL, std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"));
  h->comm = comm; h->rank = rank; h->nranks = nranks;
  return MMQ_OK;
}

int mmq_comm_move(mmq_handle* from, mmq_handle* to) {
  if (!from || !to || from == to) return mmq_fail(to, MMQ_ERR_ARG, "mmq_comm_move: bad arguments");
  if (to->comm || to->p2p_n > 1) return mmq_fail(to, MMQ_ERR_STATE, "mmq_comm_move: destination already has a communicator");
  if (from->device != to->device) return mmq_fail(to, MMQ_ERR_ARG, "mmq_comm_move: handles are on different devices");
  MMQ_CUDA(from, cudaSetDevice(from->device));
  MMQ_CUDA(from, cudaStreamSynchronize(from->stream));
  to->comm = from->comm; to->rank = from->rank; to->nranks = from->nranks;
  from->comm = nullptr; from->rank = 0; from->nranks = 1;
  if (from->p2p_n > 1 && from->n == to->n) {
    /* the peer mapping goes along (no cudaIpc round trip per sample): the block, the peers' mappings and the epoch
     * counter move to `to`, whose counts and mu are copied into the block; `from` returns to its own buffers.
     * Every rank must make the same move between the same two sweeps. */
    drop_graph(from);
    MMQ_CUDA(to, cudaStreamSynchronize(to->stream));
    auto it = std::find(from->allocs.begin(), from->allocs.end(), from->p2p_buf);
    if (it != from->allocs.end()) { from->allocs.erase(it); to->allocs.push_back(from->p2p_buf); }
    if (to->p2p_buf) mmq_dev_free(to, to->p2p_buf);
    to->p2p_buf = from->p2p_buf;
    for (int r = 0; r < MMQ_P2P_MAX; ++r) { to->p2p_base[r] = from->p2p_base[r]; to->p2p_opened[r] = from->p2p_opened[r]; from->p2p_opened[r] = nullptr; from->p2p_base[r] = nullptr; }
    to->p2p_epoch = from->p2p_epoch;
    const int rank = from->p2p_rank, nranks = from->p2p_n;
    MMQ_CUDA(from, cudaMemcpyAsync(from->mu_own, from->mu, sizeof(double) * (size_t)(from->n + 1), cudaMemcpyDeviceToDevice, from->stream));
    MMQ_CUDA(from, cudaStreamSynchronize(from->stream));
    from->mu = from->mu_own; from->counts = from->counts_own;
    from->p2p_buf = nullptr; from->p2p_n = 0; from->p2p_rank = 0; from->p2p_epoch = 0;
    int rc = p2p_adopt(to, rank, nranks);
    if (rc) return rc;
  }
  return MMQ_OK;
}

/* ---- fused count exchange over peer memory ---- */
static inline size_t p2p_r256(size_t v) { return (v + 255) & ~(size_t)255; }
static inline size_t p2p_off_counts(const mmq_handle* h, int parity) { return MMQ_P2P_HEAD + (size_t)parity * p2p_r256(sizeof(int32_t) * (size_t)h->n); }
static inline size_t p2p_off_mu(const mmq_handle* h) { return MMQ_P2P_HEAD + 2 * p2p_r256(sizeof(int32_t) * (size_t)h->n); }

static int p2p_alloc(mmq_handle* h) {
  if (h->p2p_buf) return MMQ_OK;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  const size_t bytes = p2p_off_mu(h) + sizeof(double) * (size_t)(h->n + 1);
  /* a plain allocation, not one from the block cache: the block is exported to other processes (cudaIpcGetMemHandle), it
   * must not be handed out again under a mapping a peer still holds; mmq_cache_free() frees what it does not know */
  MMQ_CUDA(h, cudaMalloc(&h->p2p_buf, bytes));
  h->allocs.push_back(h->p2p_buf);
  h->bytes += (int64_t)bytes;
  MMQ_CUDA(h, cudaMemsetAsync(h->p2p_buf, 0, bytes, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

int mmq_p2p_export(mmq_handle* h, char ipc_handle[64]) {
  if (!h || !ipc_handle) return mmq_fail(h, MMQ_ERR_ARG, "mmq_p2p_export: NULL argument");
  int rc = p2p_alloc(h);
  if (rc) return rc;
  cudaIpcMemHandle_t mh;
  static_assert(sizeof(mh) == 64, "cudaIpcMemHandle_t is 64 bytes");
  MMQ_CUDA(h, cudaIpcGetMemHandle(&mh, h->p2p_buf));
  memcpy(ipc_handle, &mh, 64);
  return MMQ_OK;
}

/* Point the handle's counts and mu into its peer-mapped block (keeping their current contents). */
static int p2p_adopt(mmq_handle* h, int rank, int nranks) {
  drop_graph(h);
  char* own = (char*)h->p2p_buf;
  int32_t* c[2] = {(int32_t*)(own + p2p_off_counts(h, 0)), (int32_t*)(own + p2p_off_counts(h, 1))};
  double* pmu = (double*)(own + p2p_off_mu(h));
  /* both parity buffers start from the current counts (zero, or the constant base of a segment / class plan) */
  for (int b = 0; b < 2; ++b) MMQ_CUDA(h, cudaMemcpyAsync(c[b], h->counts, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToDevice, h->stream));
  MMQ_CUDA(h, cudaMemcpyAsync(pmu, h->mu, sizeof(double) * (size_t)(h->n + 1), cudaMemcpyDeviceToDevice, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  h->counts_own = h->counts; h->mu_own = h->mu;
  h->p2p_counts[0] = c[0]; h->p2p_counts[1] = c[1];
  h->p2p_rank = rank; h->p2p_n = nranks;
  h->counts = c[h->p2p_epoch & 1];
  h->mu = pmu;
  return MMQ_OK;
}

int mmq_p2p_attach(mmq_handle* h, const char* ipc_handles, int rank, int nranks) {
  if (!h || !ipc_handles || nranks < 1 || nranks > MMQ_P2P_MAX || rank < 0 || rank >= nranks) return mmq_fail(h, MMQ_ERR_ARG, "mmq_p2p_attach: bad arguments");
  if (h->p2p_n > 1) return mmq_fail(h, MMQ_ERR_STATE, "mmq_p2p_attach: already attached");
  int rc = p2p_alloc(h);
  if (rc) return rc;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  void* opened[MMQ_P2P_MAX] = {};
  for (int r = 0; r < nranks; ++r) { /* map every peer first: a failure leaves the handle detached */
    if (r == rank) continue;
    cudaIpcMemHandle_t mh;
    memcpy(&mh, ipc_handles + 64 * r, 64);
    cudaError_t e = cudaIpcOpenMemHandle(&opened[r], mh, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (int q = 0; q < r; ++q) if (opened[q]) cudaIpcCloseMemHandle(opened[q]);
      return mmq_cuda_fail(h, e, "cudaIpcOpenMemHandle", __FILE__, __LINE__);
    }
  }
  for (int r = 0; r < nranks; ++r) {
    h->p2p_opened[r] = opened[r];
    h->p2p_base[r] = r == rank ? (char*)h->p2p_buf : (char*)opened[r];
  }
  h->p2p_epoch = 0;
  return p2p_adopt(h, rank, nranks);
}

int mmq_p2p_attach_local(mmq_handle** hs, int nranks) {
  if (!hs || nranks < 1 || nranks > MMQ_P2P_MAX) return mmq_fail(nullptr, MMQ_ERR_ARG, "mmq_p2p_attach_local: bad arguments");
  for (int r = 0; r < nranks; ++r)
    if (!hs[r] || hs[r]->n != hs[0]->n) return mmq_fail(hs[0], MMQ_ERR_ARG, "mmq_p2p_attach_local: handles must share n");
  for (int r = 0; r < nranks; ++r)
    if (hs[r]->p2p_n > 1) return mmq_fail(hs[r], MMQ_ERR_STATE, "mmq_p2p_attach_local: already attached");
  /* two phases, all or nothing: peer access and buffers for EVERY rank first; only then are the handles switched
   * over (a rank attached while another one still uses NCCL would spin on flags that never come) */
  for (int r = 0; r < nranks; ++r) {
    mmq_handle* h = hs[r];
    MMQ_CUDA(h, cudaSetDevice(h->device));
    for (int q = 0; q < nranks; ++q)
      if (q != r && hs[q]->device != h->device) {
        cudaError_t e = cudaDeviceEnablePeerAccess(hs[q]->device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) return mmq_cuda_fail(hs[0], e, "cudaDeviceEnablePeerAccess", __FILE__, __LINE__);
      }
    int rc = p2p_alloc(h);
    if (rc) { if (h != hs[0]) hs[0]->err = h->err; return rc; }
  }
  for (int r = 0; r < nranks; ++r) {
    mmq_handle* h = hs[r];
    MMQ_CUDA(h, cudaSetDevice(h->device));
    for (int q = 0; q < nranks; ++q) h->p2p_base[q] = (char*)hs[q]->p2p_buf;
    h->p2p_epoch = 0;
    int rc = p2p_adopt(h, r, nranks);
    if (rc) return rc;
  }
  return MMQ_OK;
}

int mmq_p2p_attached(const mmq_handle* h) { return h && h->p2p_n > 1 ? h->p2p_n : 0; }

/* ---- initial mu ---- */
int mmq_init_mu(mmq_handle* h, int32_t* unique_hits_out) {
  if (!h) return MMQ_ERR_ARG;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  { int rc0 = build_transpose(h); if (rc0) return rc0; }
  const int grid = mmq_grid_for(h->n * 32, 256, h->num_sms * 8);
  if (h->has_k) k_init_acc<true><<<grid, 256, 0, h->stream>>>(h->tptr, h->trow, h->row_ptr, h->k, h->acc, h->uh, h->n);
  else k_init_acc<false><<<grid, 256, 0, h->stream>>>(h->tptr, h->trow, h->row_ptr, h->k, h->acc, h->uh, h->n);
  MMQ_LAUNCHED(h);
  int rc;
  if ((rc = mmq_allreduce(h, h->acc, (size_t)h->n, 1))) return rc;
  if ((rc = mmq_allreduce(h, h->uh, (size_t)h->n, 0))) return rc;
  k_divide<<<mmq_grid_for(h->n, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->acc, h->len, h->mu, h->n);
  MMQ_LAUNCHED(h);
  if (unique_hits_out) MMQ_CUDA(h, cudaMemcpyAsync(unique_hits_out, h->uh, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

int mmq_set_mu(mmq_handle* h, const double* mu) {
  if (!h || !mu) return mmq_fail(h, MMQ_ERR_ARG, "mmq_set_mu: NULL argument");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaMemcpyAsync(h->mu, mu, sizeof(double) * (size_t)h->n, cudaMemcpyHostToDevice, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

int mmq_get_mu(mmq_handle* h, double* mu_out) {
  if (!h || !mu_out) return mmq_fail(h, MMQ_ERR_ARG, "mmq_get_mu: NULL argument");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaMemcpyAsync(mu_out, h->mu, sizeof(double) * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

/* ---- log-likelihood and EM ---- */

/* scalars[0] = sum over this shard's classes of k log D (and rterm refreshed) from `mu_dev`. */
static int launch_rowterm(mmq_handle* h, const double* mu_dev) {
  const int grid = mmq_grid_for(h->m, 256, h->partial_cap);
  if (h->has_k) {
    if (h->has_w) k_rowterm<true, true><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, h->w, mu_dev, h->rterm, h->partial, h->m);
    else k_rowterm<true, false><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, h->w, mu_dev, h->rterm, h->partial, h->m);
  } else {
    if (h->has_w) k_rowterm<false, true><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, h->w, mu_dev, h->rterm, h->partial, h->m);
    else k_rowterm<false, false><<<grid, 256, 0, h->stream>>>(h->row_ptr, h->col, h->k, h->w, mu_dev, h->rterm, h->partial, h->m);
  }
  MMQ_LAUNCHED(h);
  k_sum_partials<<<1, 256, 0, h->stream>>>(h->partial, grid, h->scalars, 0);
  MMQ_LAUNCHED(h);
  return mmq_allreduce(h, h->scalars, 1, 1);
}

int mmq_loglik(mmq_handle* h, double* out) {
  if (!h || !out) return mmq_fail(h, MMQ_ERR_ARG, "mmq_loglik: NULL argument");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  int rc = launch_rowterm(h, h->mu);
  if (rc) return rc;
  const int grid = mmq_grid_for(h->n, 256, h->partial_cap);
  k_mul_sum<<<grid, 256, 0, h->stream>>>(h->mu, h->len, h->partial, h->n);
  MMQ_LAUNCHED(h);
  k_sum_partials<<<1, 256, 0, h->stream>>>(h->partial, grid, h->scalars, 1);
  MMQ_LAUNCHED(h);
  double s[2];
  MMQ_CUDA(h, cudaMemcpyAsync(s, h->scalars, sizeof s, cudaMemcpyDeviceToHost, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  *out = s[0] - s[1];
  return MMQ_OK;
}

int mmq_em(mmq_handle* h, int max_iter, double eps, int* iters_out, double* loglik_out, double* llr_out) {
  if (!h) return MMQ_ERR_ARG;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  double loglik = 0.0;
  int rc = build_transpose(h);
  if (rc) return rc;
  rc = mmq_loglik(h, &loglik); /* also leaves rterm = k/D(mu) */
  if (rc) return rc;
  double llr = eps + 1.0; /* src/mmseq.cpp:756 */
  if (!(llr > eps)) llr = INFINITY; /* eps so negative that eps + 1 == eps (callers stepping one iteration at a time) */
  int iter = 0;
  const int grid_w = mmq_grid_for(h->n * 32, 256, h->num_sms * 8);
  const int grid_t = mmq_grid_for(h->n, 256, h->partial_cap);
  while (iter < max_iter && llr > eps) {
    if (h->has_w) k_em_acc<true><<<grid_w, 256, 0, h->stream>>>(h->tptr, h->perm, h->trow, h->w, h->rterm, h->acc, h->n);
    else k_em_acc<false><<<grid_w, 256, 0, h->stream>>>(h->tptr, h->perm, h->trow, h->w, h->rterm, h->acc, h->n);
    MMQ_LAUNCHED(h);
    if ((rc = mmq_allreduce(h, h->acc, (size_t)h->n, 1))) return rc;
    k_em_apply<<<grid_t, 256, 0, h->stream>>>(h->mu, h->acc, h->len, h->mu_tmp, h->partial, h->n);
    MMQ_LAUNCHED(h);
    k_sum_partials<<<1, 256, 0, h->stream>>>(h->partial, grid_t, h->scalars, 1);
    MMQ_LAUNCHED(h);
    if ((rc = launch_rowterm(h, h->mu_tmp))) return rc;
    double s[2];
    MMQ_CUDA(h, cudaMemcpyAsync(s, h->scalars, sizeof s, cudaMemcpyDeviceToHost, h->stream));
    /* mu keeps its address for the life of the handle (captured CUDA graphs and the peers of a multi-GPU run hold it) */
    MMQ_CUDA(h, cudaMemcpyAsync(h->mu, h->mu_tmp, sizeof(double) * (size_t)h->n, cudaMemcpyDeviceToDevice, h->stream));
    MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
    const double ll2 = s[0] - s[1];
    llr = ll2 - loglik;
    loglik = ll2;
    ++iter;
  }
  if (iters_out) *iters_out = iter;
  if (loglik_out) *loglik_out = loglik;
  if (llr_out) *llr_out = llr;
  return MMQ_OK;
}

/* ---- Gibbs ---- */

static int ensure_x(mmq_handle* h) {
  if (h->x) return MMQ_OK;
  return mmq_dev_alloc(h, (void**)&h->x, sizeof(int32_t) * (size_t)std::max<int64_t>(h->nnz, 1));
}

} /* extern "C" */
template <bool MAT>
static void launch_alloc_t(mmq_handle* h, int grid, uint32_t seed, uint32_t sweep, const uint32_t* sweep_base) {
#define MMQ_ALLOC_ARGS h->row_ptr, h->col, h->k, h->w, h->mu, h->counts, h->x, h->m, h->tile_start, h->n_tiles, seed, sweep, h->class_id_base, h->class_id, sweep_base
  if (h->has_k) {
    if (h->has_w) k_alloc<MAT, true, true><<<grid, MMQ_ALLOC_WARPS * 32, 0, h->stream>>>(MMQ_ALLOC_ARGS);
    else k_alloc<MAT, true, false><<<grid, MMQ_ALLOC_WARPS * 32, 0, h->stream>>>(MMQ_ALLOC_ARGS);
  } else {
    if (h->has_w) k_alloc<MAT, false, true><<<grid, MMQ_ALLOC_WARPS * 32, 0, h->stream>>>(MMQ_ALLOC_ARGS);
    else k_alloc<MAT, false, false><<<grid, MMQ_ALLOC_WARPS * 32, 0, h->stream>>>(MMQ_ALLOC_ARGS);
  }
#undef MMQ_ALLOC_ARGS
}
void mmq_launch_alloc_general(mmq_handle* h, cudaStream_t stream, int grid, const int64_t* row_ptr, const int32_t* col, const int32_t* k,
                              int64_t m, const int64_t* tile_start, int64_t n_tiles, const int64_t* class_id, uint32_t seed,
                              uint32_t sweep, const uint32_t* sweep_base) {
  k_alloc<false, true, false><<<grid, MMQ_ALLOC_WARPS * 32, 0, stream>>>(row_ptr, col, k, nullptr, h->mu, h->counts, nullptr, m, tile_start, n_tiles,
                                                                        seed, sweep, 0, class_id, sweep_base);
}
static mmq_cnt_acc count_args(const mmq_handle* h) { return mmq_cnt_acc{h->cnt_sum, h->cnt_sq, h->cnt_group, h->cnt_gsum}; }
/* After the Gamma kernel of a sweep that accumulates count moments: the group step, and the sweep counted (a graph
 * capture launches nothing now: mmq_gibbs counts its replays). */
static int count_groups_step(mmq_handle* h, const uint32_t* sweep_base) {
  if (!h->cnt_block) return MMQ_OK;
  if (!sweep_base) ++h->cnt_sweeps;
  if (h->cnt_groups == 0) return MMQ_OK;
  k_count_groups<<<mmq_grid_for(h->cnt_groups, 256, h->num_sms * 4), 256, 0, h->stream>>>(count_args(h), h->n, h->cnt_groups);
  MMQ_LAUNCHED(h);
  return MMQ_OK;
}
/* K4 of a sweep: the k_gamma instantiation for the handle (accumulating or not, own counts or the peers' in a), or the
 * reduce-scatter kernel and its trace capture. */
static int launch_gamma(mmq_handle* h, const mmq_p2p_args& a, uint32_t seed, uint32_t sweep, int stride, int32_t* counts_copy,
                        const uint32_t* sweep_base) {
  const bool p2p = h->p2p_n > 1;
  if (p2p && !counts_copy && h->exchange_rs == 1) { /* mmq_tune(h, 6, 1): reduce-scatter + Gamma + all-gather */
    /* the all-reduce is the default: the Gamma kernel is bound by the latency of one pass, not by throughput, so
     * drawing n / N variates instead of n saves nothing, while this variant pays a second barrier and the peer stores
     * (DESIGN §7) */
    const int64_t slice = (h->n + h->p2p_n - 1) / h->p2p_n;
    k_gamma_rs<<<mmq_grid_for(std::max<int64_t>(slice, h->n / 8), MMQ_GAMMA_THREADS, h->num_sms * 4), MMQ_GAMMA_THREADS, 0, h->stream>>>(a, h->seg_base, h->len, h->n, h->alpha, h->beta, seed, sweep, sweep_base);
    MMQ_LAUNCHED(h);
    /* is this sweep recorded?  plain launch: the host knows; graph capture: sweep = j, the replays start at
     * sweeps congruent to capture_phase modulo the stride (the kernel re-checks against the real sweep number) */
    if (stride > 0 && h->trace &&
        (sweep_base ? ((uint32_t)h->capture_phase + sweep) % (uint32_t)stride == 0 : trace_recorded(sweep, stride, h->trace_len))) {
      k_trace_capture<<<mmq_grid_for(h->n, 256, h->num_sms * 4), 256, 0, h->stream>>>(h->mu, h->trace, stride, h->trace_len, h->n, sweep, sweep_base);
      MMQ_LAUNCHED(h);
    }
    return MMQ_OK;
  }
  const int grid = mmq_grid_for(h->n, MMQ_GAMMA_THREADS, h->num_sms * 5);
  auto go = [&](auto kernel, const auto& src) {
    kernel<<<grid, MMQ_GAMMA_THREADS, 0, h->stream>>>(src, h->seg_base, h->len, h->mu, stride > 0 ? h->trace : nullptr, stride, h->trace_len, h->n,
                                                      h->alpha, h->beta, seed, sweep, counts_copy, sweep_base, count_args(h));
  };
  if (p2p) h->cnt_block ? go(k_gamma<true, true>, a) : go(k_gamma<false, true>, a);
  else h->cnt_block ? go(k_gamma<true, false>, h->counts) : go(k_gamma<false, false>, h->counts);
  MMQ_LAUNCHED(h);
  return count_groups_step(h, sweep_base);
}
/* The peer-memory exchange of the next sweep: this epoch's parity buffers; advances the epoch. */
static mmq_p2p_args p2p_args(mmq_handle* h, const int32_t* epoch_base) {
  const int b = h->p2p_epoch & 1;
  mmq_p2p_args a;
  for (int r = 0; r < MMQ_P2P_MAX; ++r) a.base[r] = r < h->p2p_n ? h->p2p_base[r] : nullptr;
  a.off_counts = (int64_t)p2p_off_counts(h, b);
  a.off_reset = (int64_t)p2p_off_counts(h, b ^ 1);
  a.off_mu = (int64_t)p2p_off_mu(h);
  a.nranks = h->p2p_n; a.rank = h->p2p_rank;
  ++h->p2p_epoch;
  /* inside a graph capture the epoch is relative to the device counter that the graph advances */
  a.epoch = epoch_base ? (int32_t)(h->p2p_epoch - h->graph_epoch0) : (int32_t)h->p2p_epoch;
  a.epoch_base = epoch_base;
  return a;
}
/* K2 on the per-fragment layout without multiplicities (k_alloc_cat); it visits the singletons itself. */
template <bool HAS_W>
static int launch_alloc_cat(mmq_handle* h, uint32_t seed, uint32_t sweep, const uint32_t* sweep_base) {
  constexpr int SLAB = HAS_W ? MMQ_CAT_SLAB_W : MMQ_CAT_SLAB;
  constexpr int SM = MMQ_CAT_WARPS * (16 + 2 * SLAB * 4 * (HAS_W ? 2 : 1));
  MMQ_CUDA(h, cudaFuncSetAttribute(k_alloc_cat<HAS_W, SLAB>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM));
  const int64_t n_chunks = (h->m + MMQ_CAT_ROWS - 1) / MMQ_CAT_ROWS;
  const int cgrid = (int)std::min<int64_t>((n_chunks + MMQ_CAT_WARPS - 1) / MMQ_CAT_WARPS, (int64_t)h->num_sms * 3);
  k_alloc_cat<HAS_W, SLAB><<<cgrid, MMQ_CAT_WARPS * 32, SM, h->stream>>>(h->row_ptr, h->col, h->w, h->mu, h->counts, h->m, n_chunks, seed, sweep,
                                                                       h->class_id_base, (int32_t)h->n, sweep_base);
  return MMQ_OK;
}
extern "C" {

/* State a sweep builds on first use (synchronising copies, allocations): done ahead of a graph capture. */
static int prepare_sweep(mmq_handle* h, int flags) {
  if (h->m <= 0) return MMQ_OK;
  int rc;
  const bool transposed = (flags & MMQ_GIBBS_TRANSPOSED) != 0;
  if ((transposed || (h->has_k && !h->cls_ready) || (flags & MMQ_GIBBS_GENERIC_KERNEL)) && (rc = build_tiles(h, nullptr))) return rc;
  if (transposed) {
    if ((rc = ensure_x(h))) return rc;
    if ((rc = build_transpose(h))) return rc;
  }
  const bool fast = !transposed && !(flags & (MMQ_GIBBS_GENERIC_KERNEL | MMQ_GIBBS_RAGGED_KERNEL));
  if (fast && h->seg_ready && (rc = mmq_seg_pack(h))) return rc; /* allocations: not inside a capture */
  return MMQ_OK;
}

/* One sweep on the stream: the allocation launch, the count exchange, the Gamma launch. */
static int enqueue_sweep(mmq_handle* h, uint32_t seed, uint32_t sweep, int flags, int stride, int32_t* counts_copy, const uint32_t* sweep_base,
                         const int32_t* epoch_base = nullptr) {
  const bool transposed = (flags & MMQ_GIBBS_TRANSPOSED) != 0;
  const bool timed = (flags & MMQ_GIBBS_TIME_KERNELS) != 0;
  int rc;
  auto mark = [&](std::vector<cudaEvent_t>& v) {
    if (!timed) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, h->stream);
    v.push_back(e);
  };
  if (h->m > 0) {
    if (!sweep_base && (rc = prepare_sweep(h, flags))) return rc; /* (a graph capture prepares before it begins) */
    const int grid = (int)std::min<int64_t>(std::max<int64_t>((h->n_tiles + MMQ_ALLOC_WARPS - 1) / MMQ_ALLOC_WARPS, 1), (int64_t)h->num_sms * 3);
    if (transposed) {
      if ((rc = ensure_x(h))) return rc;
      if ((rc = build_transpose(h))) return rc;
      mark(h->ev_alloc);
      launch_alloc_t<true>(h, grid, seed, sweep, sweep_base);
      MMQ_LAUNCHED(h);
      mark(h->ev_alloc);
      k_count_reduce<<<mmq_grid_for(h->n * 32, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->tptr, h->perm, h->x, h->counts, h->n);
      MMQ_LAUNCHED(h);
    } else {
      mark(h->ev_alloc);
      if (h->seg_ready && !(flags & (MMQ_GIBBS_GENERIC_KERNEL | MMQ_GIBBS_RAGGED_KERNEL))) {
        if ((rc = mmq_seg_launch(h, seed, sweep, sweep_base))) return rc;
      } else if (h->cls_ready && !(flags & (MMQ_GIBBS_GENERIC_KERNEL | MMQ_GIBBS_RAGGED_KERNEL))) {
        if ((rc = mmq_cls_launch(h, seed, sweep, sweep_base))) return rc;
        g_mmq_launches.fetch_sub(1, std::memory_order_relaxed); /* counted inside; MMQ_LAUNCHED below adds one */
      } else if (!h->has_k && !(flags & MMQ_GIBBS_GENERIC_KERNEL)) {
        if ((rc = mmq_seg_add_base(h, false))) return rc; /* this kernel visits the singletons itself */
        if ((rc = h->has_w ? launch_alloc_cat<true>(h, seed, sweep, sweep_base) : launch_alloc_cat<false>(h, seed, sweep, sweep_base))) return rc;
      } else {
        if ((rc = mmq_seg_add_base(h, false))) return rc;
        launch_alloc_t<false>(h, grid, seed, sweep, sweep_base);
      }
      MMQ_LAUNCHED(h);
      mark(h->ev_alloc);
    }
  }
  /* the count exchange: fused into the Gamma kernel over peer memory, else an all-reduce (a no-op on one GPU) */
  const bool p2p = h->p2p_n > 1;
  mmq_p2p_args a{};
  if (p2p) a = p2p_args(h, epoch_base);
  else if ((rc = mmq_allreduce(h, h->counts, (size_t)h->n, 0))) return rc;
  mark(h->ev_gamma);
  if ((rc = launch_gamma(h, a, seed, sweep, stride, counts_copy, sweep_base))) return rc;
  mark(h->ev_gamma);
  if (p2p) h->counts = h->p2p_counts[h->p2p_epoch & 1]; /* the next sweep reduces into the other parity buffer */
  if (h->seg_base) h->seg_base_in_counts = true; /* the Gamma kernel restarted counts[] from seg_base */
  return MMQ_OK;
}

static int ensure_trace(mmq_handle* h, int trace_len) {
  if (trace_len <= 0) return MMQ_OK;
  if (h->trace && h->trace_len == trace_len) return MMQ_OK;
  if (h->trace) { mmq_dev_free(h, h->trace); h->bytes -= (int64_t)sizeof(double) * h->n * h->trace_len; h->trace = nullptr; }
  int rc = mmq_dev_alloc(h, (void**)&h->trace, sizeof(double) * (size_t)h->n * (size_t)trace_len);
  if (rc) return rc;
  h->trace_len = trace_len;
  MMQ_CUDA(h, cudaMemsetAsync(h->trace, 0, sizeof(double) * (size_t)h->n * (size_t)trace_len, h->stream));
  for (auto& g : h->groups) g.trace_valid = false;
  return MMQ_OK;
}

static void drop_graph(mmq_handle* h) {
  if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
  if (h->graph) { cudaGraphDestroy(h->graph); h->graph = nullptr; }
  h->graph_flags = -1;
}

/* Capture MMQ_GRAPH_SWEEPS sweeps (sweep = graph_base[0] + j; peer-memory epoch = graph_base[1] + j + 1) followed by
 * graph_base[0..1] += MMQ_GRAPH_SWEEPS.  `phase` = first sweep of a replay modulo the trace stride (decides which of the
 * captured sweeps carry the multi-GPU trace-capture kernel). */
static int capture_graph(mmq_handle* h, uint32_t seed, int flags, int stride, int phase) {
  drop_graph(h);
  if (!h->graph_base) {
    int rc = mmq_dev_alloc(h, (void**)&h->graph_base, 2 * sizeof(uint32_t));
    if (rc) return rc;
  }
  const long long launches_before = g_mmq_launches.load();
  const int32_t epoch0 = h->p2p_epoch;
  int32_t* const counts0 = h->counts;
  h->graph_epoch0 = epoch0;
  h->capture_phase = phase;
  MMQ_CUDA(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  int rc = MMQ_OK;
  for (int j = 0; j < MMQ_GRAPH_SWEEPS && rc == MMQ_OK; ++j)
    rc = enqueue_sweep(h, seed, (uint32_t)j, flags, stride, nullptr, h->graph_base, h->p2p_n > 1 ? (const int32_t*)(h->graph_base + 1) : nullptr);
  if (rc == MMQ_OK) {
    k_add2_u32<<<1, 1, 0, h->stream>>>(h->graph_base, MMQ_GRAPH_SWEEPS);
    g_mmq_launches.fetch_add(1);
  }
  cudaGraph_t g = nullptr;
  cudaError_t e = cudaStreamEndCapture(h->stream, &g);
  h->capture_phase = -1;
  h->p2p_epoch = epoch0; /* nothing ran: the host mirror of the epoch and the parity buffer go back */
  h->counts = counts0;
  h->graph_launches = g_mmq_launches.load() - launches_before; /* kernel nodes of one replay */
  g_mmq_launches.store(launches_before);                       /* capturing launched nothing */
  if (rc != MMQ_OK) { if (g) cudaGraphDestroy(g); return rc; }
  if (e != cudaSuccess) return mmq_cuda_fail(h, e, "cudaStreamEndCapture", __FILE__, __LINE__);
  h->graph = g;
  e = cudaGraphInstantiate(&h->graph_exec, g, 0);
  if (e != cudaSuccess) { drop_graph(h); return mmq_cuda_fail(h, e, "cudaGraphInstantiate", __FILE__, __LINE__); }
  h->graph_seed = seed; h->graph_flags = flags; h->graph_stride = stride; h->graph_trace_len = h->trace_len;
  h->graph_trace = h->trace; h->graph_stream = h->stream; h->graph_phase = phase; h->graph_mu = h->mu; h->graph_counts = h->counts;
  return MMQ_OK;
}

int mmq_gibbs(mmq_handle* h, uint32_t seed, int64_t first_sweep, int64_t n_sweeps, int stride, int trace_len, int flags) {
  if (!h) return MMQ_ERR_ARG;
  if (first_sweep < 0 || n_sweeps < 0 || first_sweep + n_sweeps > (int64_t)0xffffffffll) return mmq_fail(h, MMQ_ERR_ARG, "mmq_gibbs: sweep range out of bounds");
  if (trace_len > 0 && stride <= 0) return mmq_fail(h, MMQ_ERR_ARG, "mmq_gibbs: stride must be > 0");
  if (h->cnt_block && h->p2p_n > 1 && h->exchange_rs == 1)
    return mmq_fail(h, MMQ_ERR_STATE, "mmq_gibbs: count moments are not accumulated under the reduce-scatter exchange (mmq_tune knob 6), "
                                      "where each rank sums only its own slice of the counts; set knob 6 back to 0");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  int rc = ensure_trace(h, trace_len);
  if (rc) return rc;
  for (auto& g : h->groups) g.trace_valid = false;
  const int st = trace_len > 0 ? stride : 0;
  int64_t s = first_sweep;
  const int64_t end = first_sweep + n_sweeps;
  /* CUDA graph of MMQ_GRAPH_SWEEPS sweeps for every call that long — single GPU and the fused peer-memory exchange
   * (the NCCL exchange and the per-kernel timing mode go out as plain launches): whole graphs first, the remainder as
   * plain launches.  Sweep number and peer-memory epoch are read from graph_base on the device, so one instantiated
   * graph serves the whole chain and later calls. */
  const bool p2p = h->p2p_n > 1;
  const bool use_graph = !(flags & (MMQ_GIBBS_NO_GRAPH | MMQ_GIBBS_TIME_KERNELS)) && (h->nranks == 1 || p2p) && n_sweeps >= MMQ_GRAPH_SWEEPS + (p2p ? 1 : 0);
  if (use_graph) {
    if ((rc = prepare_sweep(h, flags))) return rc;
    if (p2p && (h->p2p_epoch & 1)) { /* the captured sweeps alternate the parity buffers starting from an even epoch */
      if ((rc = enqueue_sweep(h, seed, (uint32_t)s, flags, st, nullptr, nullptr))) return rc;
      ++s;
    }
    const int phase = st > 0 ? (int)(s % st) : 0;
    const bool reuse = h->graph_exec && h->graph_seed == seed && h->graph_flags == flags && h->graph_stride == st &&
                       h->graph_trace_len == h->trace_len && h->graph_trace == h->trace && h->graph_stream == h->stream &&
                       h->graph_mu == h->mu && h->graph_counts == h->counts && (!p2p || st == 0 || h->graph_phase == phase);
    if (!reuse && (rc = capture_graph(h, seed, flags, st, phase))) return rc;
    k_set2_u32<<<1, 1, 0, h->stream>>>(h->graph_base, (uint32_t)s, (uint32_t)h->p2p_epoch);
    MMQ_LAUNCHED(h);
    while (end - s >= MMQ_GRAPH_SWEEPS) {
      if (p2p && st > 0 && (int)(s % st) != h->graph_phase) break; /* stride does not divide the graph length: plain launches */
      MMQ_CUDA(h, cudaGraphLaunch(h->graph_exec, h->stream));
      g_mmq_launches.fetch_add(h->graph_launches, std::memory_order_relaxed);
      if (h->cnt_block) h->cnt_sweeps += MMQ_GRAPH_SWEEPS;
      s += MMQ_GRAPH_SWEEPS;
      if (p2p) h->p2p_epoch += MMQ_GRAPH_SWEEPS;
    }
  }
  for (; s < end; ++s)
    if ((rc = enqueue_sweep(h, seed, (uint32_t)s, flags, st, nullptr, nullptr))) return rc;
  return MMQ_OK;
}

int mmq_sweep_debug(mmq_handle* h, uint32_t seed, int64_t sweep, int flags, int32_t* x_out, int32_t* counts_out, double* mu_out) {
  if (!h) return MMQ_ERR_ARG;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  if (x_out && !(flags & MMQ_GIBBS_TRANSPOSED)) return mmq_fail(h, MMQ_ERR_ARG, "mmq_sweep_debug: x_out needs MMQ_GIBBS_TRANSPOSED (the fused path keeps no X)");
  int32_t* counts_copy = nullptr;
  MMQ_CUDA(h, cudaMalloc(&counts_copy, sizeof(int32_t) * (size_t)h->n));
  int rc = enqueue_sweep(h, seed, (uint32_t)sweep, flags, 0, counts_copy, nullptr);
  if (rc) { cudaFree(counts_copy); return rc; }
  cudaError_t e = cudaSuccess;
  if (x_out) e = cudaMemcpyAsync(x_out, h->x, sizeof(int32_t) * (size_t)h->nnz, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess && counts_out) e = cudaMemcpyAsync(counts_out, counts_copy, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess && mu_out) e = cudaMemcpyAsync(mu_out, h->mu, sizeof(double) * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(counts_copy);
  if (e != cudaSuccess) return mmq_cuda_fail(h, e, "mmq_sweep_debug copies", __FILE__, __LINE__);
  return MMQ_OK;
}

static void drain_events(std::vector<cudaEvent_t>& v, double* ms_total, int64_t* launches) {
  double tot = 0.0;
  int64_t cnt = 0;
  for (size_t i = 0; i + 1 < v.size(); i += 2) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, v[i], v[i + 1]) == cudaSuccess) { tot += ms; ++cnt; }
  }
  for (cudaEvent_t e : v) cudaEventDestroy(e);
  v.clear();
  if (ms_total) *ms_total = tot;
  if (launches) *launches = cnt;
}

int mmq_kernel_times(mmq_handle* h, double* alloc_ms, int64_t* alloc_launches, double* gamma_ms, int64_t* gamma_launches) {
  if (!h) return MMQ_ERR_ARG;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  drain_events(h->ev_alloc, alloc_ms, alloc_launches);
  drain_events(h->ev_gamma, gamma_ms, gamma_launches);
  return MMQ_OK;
}

int mmq_trace_len(const mmq_handle* h) { return h ? h->trace_len : 0; }

int mmq_tune(mmq_handle* h, int knob, int value) {
  if (!h || (knob != 0 && knob != 6)) return mmq_fail(h, MMQ_ERR_ARG, "mmq_tune: bad knob");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  drop_graph(h); /* a captured graph has the old launches baked in */
  if (knob == 0) h->skip_mask = value;
  else h->exchange_rs = value;
  return MMQ_OK;
}

int mmq_warmup(int device) {
  if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return MMQ_ERR_CUDA; }
  return cudaFree(nullptr) == cudaSuccess ? MMQ_OK : MMQ_ERR_CUDA;
}

int mmq_get_trace(mmq_handle* h, double* out) {
  if (!h || !out) return mmq_fail(h, MMQ_ERR_ARG, "mmq_get_trace: NULL argument");
  if (!h->trace) return mmq_fail(h, MMQ_ERR_STATE, "mmq_get_trace: no trace recorded (run mmq_gibbs with trace_len > 0)");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaMemcpyAsync(out, h->trace, sizeof(double) * (size_t)h->n * (size_t)h->trace_len, cudaMemcpyDeviceToHost, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

/* ---- posterior fragment counts ---- */

/* bytes of the accumulator block: sq, sum, group map, group sums (mmq_internal.h) */
static void count_layout(int64_t n, int64_t groups, size_t b[4]) {
  b[0] = sizeof(unsigned __int128) * (size_t)(n + groups);
  b[1] = sizeof(unsigned long long) * (size_t)(n + groups);
  b[2] = groups > 0 ? sizeof(int2) * (size_t)n : 0;
  b[3] = sizeof(int32_t) * (size_t)groups;
}

static void count_free(mmq_handle* h) {
  if (!h->cnt_block) return;
  size_t b[4];
  count_layout(h->n, h->cnt_groups, b);
  h->bytes -= (int64_t)(b[0] + b[1] + b[2] + b[3]);
  mmq_dev_free(h, h->cnt_block); /* synchronises the stream first */
  h->cnt_block = nullptr; h->cnt_sq = nullptr; h->cnt_sum = nullptr; h->cnt_group = nullptr; h->cnt_gsum = nullptr;
  h->cnt_ident = h->cnt_groups = 0;
  h->cnt_sweeps = 0;
}

int mmq_count_moments_begin(mmq_handle* h, const int32_t* ident_of, int64_t n_ident, const int32_t* gene_of, int64_t n_gene) {
  if (!h) return MMQ_ERR_ARG;
  if (n_ident < 0 || n_gene < 0 || n_ident + n_gene > INT32_MAX)
    return mmq_fail(h, MMQ_ERR_ARG, "mmq_count_moments_begin: group counts out of range");
  if ((n_ident > 0 && !ident_of) || (n_gene > 0 && !gene_of))
    return mmq_fail(h, MMQ_ERR_ARG, "mmq_count_moments_begin: ident_of / gene_of is NULL but its group count is not 0");
  const int64_t n = h->n, groups = n_ident + n_gene;
  std::vector<int2> grp;
  if (groups > 0) {
    grp.resize((size_t)n);
    for (int64_t t = 0; t < n; ++t) {
      const int32_t i = n_ident > 0 ? ident_of[t] : -1, g = n_gene > 0 ? gene_of[t] : -1;
      if (i < -1 || i >= n_ident || g < -1 || g >= n_gene)
        return mmq_fail(h, MMQ_ERR_ARG, "mmq_count_moments_begin: transcript " + std::to_string(t) + " names a group out of range");
      grp[(size_t)t] = make_int2(i, g < 0 ? -1 : (int)(n_ident + g));
    }
  }
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  drop_graph(h); /* a captured graph has the other Gamma kernel baked in */
  count_free(h);
  size_t b[4];
  count_layout(n, groups, b);
  const size_t b_sq = b[0], b_sum = b[1], b_grp = b[2], bytes = b[0] + b[1] + b[2] + b[3];
  /* from the block cache, not the arena: a handle that never asks for counts pays nothing */
  void* blk = nullptr;
  MMQ_CUDA(h, mmq_cache_malloc(&blk, bytes));
  h->allocs.push_back(blk);
  h->bytes += (int64_t)bytes;
  h->cnt_block = blk;
  char* p = static_cast<char*>(blk);
  h->cnt_sq = reinterpret_cast<unsigned __int128*>(p);
  h->cnt_sum = reinterpret_cast<unsigned long long*>(p + b_sq);
  h->cnt_group = groups > 0 ? reinterpret_cast<int2*>(p + b_sq + b_sum) : nullptr;
  h->cnt_gsum = reinterpret_cast<int32_t*>(p + b_sq + b_sum + b_grp);
  h->cnt_ident = n_ident;
  h->cnt_groups = groups;
  h->cnt_sweeps = 0;
  MMQ_CUDA(h, cudaMemsetAsync(blk, 0, bytes, h->stream));
  if (groups > 0) MMQ_CUDA(h, cudaMemcpyAsync(h->cnt_group, grp.data(), b_grp, cudaMemcpyHostToDevice, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

int mmq_count_moments_end(mmq_handle* h) {
  if (!h) return MMQ_ERR_ARG;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  drop_graph(h);
  count_free(h);
  return MMQ_OK;
}

int mmq_get_count_moments(mmq_handle* h, int which, int64_t* sweeps, uint64_t* sum, uint64_t* sumsq_lo, uint64_t* sumsq_hi) {
  if (!h) return MMQ_ERR_ARG;
  if (!h->cnt_block) return mmq_fail(h, MMQ_ERR_STATE, "mmq_get_count_moments: no count moments (call mmq_count_moments_begin first)");
  if (which < 0 || which > 2) return mmq_fail(h, MMQ_ERR_ARG, "mmq_get_count_moments: which must be 0, 1 or 2");
  const int64_t r0 = which == 0 ? 0 : which == 1 ? h->n : h->n + h->cnt_ident;
  const int64_t rows = which == 0 ? h->n : which == 1 ? h->cnt_ident : h->cnt_groups - h->cnt_ident;
  MMQ_CUDA(h, cudaSetDevice(h->device));
  if (sweeps) *sweeps = (int64_t)h->cnt_sweeps;
  if (rows > 0 && sum)
    MMQ_CUDA(h, cudaMemcpyAsync(sum, h->cnt_sum + r0, sizeof(uint64_t) * (size_t)rows, cudaMemcpyDeviceToHost, h->stream));
  std::vector<unsigned __int128> sq;
  if (rows > 0 && (sumsq_lo || sumsq_hi)) {
    sq.resize((size_t)rows);
    MMQ_CUDA(h, cudaMemcpyAsync(sq.data(), h->cnt_sq + r0, sizeof(unsigned __int128) * (size_t)rows, cudaMemcpyDeviceToHost, h->stream));
  }
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  for (size_t r = 0; r < sq.size(); ++r) {
    if (sumsq_lo) sumsq_lo[r] = (uint64_t)sq[r];
    if (sumsq_hi) sumsq_hi[r] = (uint64_t)(sq[r] >> 64);
  }
  return MMQ_OK;
}

/* One E-step at the current mu (src/mmseq.cpp:781-794): acc = the EM accumulation of all shards, out = mu * acc. */
int mmq_expected_counts(mmq_handle* h, double* out) {
  if (!h || !out) return mmq_fail(h, MMQ_ERR_ARG, "mmq_expected_counts: NULL argument");
  MMQ_CUDA(h, cudaSetDevice(h->device));
  int rc = build_transpose(h);
  if (rc) return rc;
  if ((rc = launch_rowterm(h, h->mu))) return rc; /* rterm = k / D(mu) */
  const int grid_w = mmq_grid_for(h->n * 32, 256, h->num_sms * 8);
  if (h->has_w) k_em_acc<true><<<grid_w, 256, 0, h->stream>>>(h->tptr, h->perm, h->trow, h->w, h->rterm, h->acc, h->n);
  else k_em_acc<false><<<grid_w, 256, 0, h->stream>>>(h->tptr, h->perm, h->trow, h->w, h->rterm, h->acc, h->n);
  MMQ_LAUNCHED(h);
  if ((rc = mmq_allreduce(h, h->acc, (size_t)h->n, 1))) return rc;
  k_mul<<<mmq_grid_for(h->n, 256, h->num_sms * 8), 256, 0, h->stream>>>(h->mu, h->acc, h->mu_tmp, h->n);
  MMQ_LAUNCHED(h);
  MMQ_CUDA(h, cudaMemcpyAsync(out, h->mu_tmp, sizeof(double) * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
  MMQ_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMQ_OK;
}

} /* extern "C" */
