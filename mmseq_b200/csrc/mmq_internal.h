/* mmq_internal.h — state behind the opaque mmq_handle and small launch helpers.
 * Internal to libmmseq_b200.so; the public surface is include/mmq.h. */
#ifndef MMQ_INTERNAL_H
#define MMQ_INTERNAL_H

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/mmq.h"

/* Tiling of the general allocation kernel: each of the MMQ_ALLOC_WARPS warps of a CTA
 * stages up to MMQ_ALLOC_CAP CSR entries of up to 32 consecutive classes. */
#define MMQ_ALLOC_THREADS 256
#define MMQ_ALLOC_WARPS 8
#define MMQ_ALLOC_CAP 320 /* staged CSR entries per warp tile */
#define MMQ_GRAPH_SWEEPS 16 /* sweeps per captured CUDA graph */
#define MMQ_P2P_MAX 8      /* ranks of one NVSwitch box */
/* head of a rank's peer-mapped block, in int32 units: one flag per rank, each in its own 32-byte sector */
#define MMQ_P2P_HEAD 1024         /* bytes */
#define MMQ_P2P_FLAG_ALLOC 0      /* [8 r]: rank r has finished the allocation of epoch e */
#define MMQ_P2P_FLAG_MU 64        /* [64 + 8 r]: rank r has stored its slice of mu of epoch e everywhere */
#define MMQ_P2P_DONE 128          /* blocks of the own Gamma kernel that have finished */

/* one run of equal class size of the segment plan (mmq_seg.cu) */
struct mmq_seg {
  int64_t e_virtual;   /* packed-array offset of the (possibly dummy) virtual first row; multiple of 4 */
  int64_t cid_virtual; /* class id of the virtual first row; a MULTIPLE OF 4, so a lane's classes are one Philox block */
  int32_t row_lo;      /* 0..3: the virtual rows in front of the run's first class are dummies */
  int32_t rows;        /* virtual row count (dummies included) */
  int32_t d;           /* class size of the run */
  int32_t chunk0;      /* first chunk of this run in the global chunk numbering */
};

struct mmq_group_set {
  int64_t ngroups = 0;
  int64_t* ptr_dev = nullptr;     /* [ngroups+1] */
  int32_t* members_dev = nullptr; /* [ptr[ngroups]] */
  double* extra_dev = nullptr;    /* [ngroups*trace_len] or null */
  double* trace_dev = nullptr;    /* [trace_len * ngroups] slot-major, built lazily */
  bool trace_valid = false;
};

struct mmq_handle {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int num_sms = 148;

  int64_t n = 0, m = 0, nnz = 0, class_id_base = 0;
  double alpha = 0.1, beta = 0.1;
  bool has_k = false, has_w = false;
  int64_t* tile_start = nullptr; /* [n_tiles+1] class ranges of the general allocation kernel */
  int64_t n_tiles = 0;

  /* class-major CSR */
  int64_t* row_ptr = nullptr; /* [m+1] */
  int32_t* col = nullptr;     /* [nnz] */
  int32_t* k = nullptr;       /* [m] or null */
  int64_t* class_id = nullptr; /* [m] or null */
  float* w = nullptr;         /* [nnz] or null */
  double* len = nullptr;      /* [n] */
  /* transcript-major transpose */
  int64_t* tptr = nullptr;  /* [n+1] */
  uint32_t* perm = nullptr; /* [nnz] position in the class-major arrays */
  int32_t* trow = nullptr;  /* [nnz] class (row) of that position */

  /* state */
  double* mu = nullptr;      /* [n] */
  double* mu_tmp = nullptr;  /* [n] */
  double* acc = nullptr;     /* [n] fp64 per-transcript partial sums (EM, init) */
  int32_t* counts = nullptr; /* [n] zero between sweeps */
  int32_t* uh = nullptr;     /* [n] */
  int32_t* x = nullptr;      /* [nnz], only for the transposed / debug path */
  double* rterm = nullptr;   /* [m] k_i / D_i */
  double* partial = nullptr; /* block partial sums */
  int partial_cap = 0;
  double* scalars = nullptr; /* [4] device scalars */

  double* trace = nullptr; /* [trace_len * n] slot-major: trace[s*n + t] */
  int trace_len = 0;

  mmq_group_set groups[2];

  /* multi-GPU */
  void* comm = nullptr; /* ncclComm_t */
  int rank = 0, nranks = 1;

  /* segmented plan for k == 1 shards whose rows come in few runs of equal length
   * (the loader's by-length layout): packed, aligned copies of col / weight, a segment
   * table, and the constant counts of the singleton classes the sweep kernel skips */
  struct seg_run { int64_t r0, r1, q0; int d; };
  std::vector<seg_run> seg_runs; /* host scan of the row pointers */
  bool seg_scan_ok = false;
  bool seg_ready = false;
  void* seg_table = nullptr; /* mmq_seg[] on the device */
  int seg_count = 0;
  int64_t seg_chunks = 0;
  int32_t* seg_col = nullptr;
  float* seg_w = nullptr;
  int32_t* seg_base = nullptr; /* [n] or null */
  bool seg_base_in_counts = true; /* counts[] currently starts from seg_base */
  int64_t seg_entries = 0, seg_rows = 0, seg_singletons = 0, seg_packed = 0;
  std::vector<mmq_seg> seg_host; /* the table, kept for the lazy packing (mmq_seg_pack) */

  /* class plan for collapsed shards (mmq_cls.cu): the classes with few fragments packed in
   * member-major chunks of 32, the rest as a sub-CSR for the general kernel on stream2 */
  bool cls_ready = false;
  void* cls_runs = nullptr; /* mmq_cls_run[] on the device */
  int cls_nruns = 0;
  int64_t cls_chunks_gen = 0; /* chunks [cls_chunks_gen, cls_chunks): single-fragment classes (k_alloc_cls1) */
  int64_t cls_chunks = 0, cls_chunks_lo = 0, cls_small = 0, cls_packed = 0, cls_rest = 0, cls_rest_nnz = 0, cls_rest_tiles = 0;
  uint32_t cls_cid_hi = 0;
  int32_t* cls_pcol = nullptr;
  uint16_t* cls_pk = nullptr; /* draws of the slot | slot number within its class << 8 */
  uint32_t* cls_pcid = nullptr;
  unsigned long long* cls_cdesc = nullptr; /* [chunks] offset of the chunk in cls_pcol << 8 | class size */
  int64_t *cls_o_rp = nullptr, *cls_o_cid = nullptr, *cls_o_tiles = nullptr;
  int32_t *cls_o_col = nullptr, *cls_o_k = nullptr;
  /* the chain set (more than mmq_cat_limit(d) fragments): k_alloc_chain, one class per lane */
  int32_t* cls_c_pcol = nullptr;
  int32_t* cls_c_k = nullptr;
  uint32_t* cls_c_cid = nullptr;
  unsigned long long* cls_c_desc = nullptr;
  int64_t cls_c_chunks = 0, cls_c_packed = 0, cls_chain = 0;
  int64_t cls_c_end[3] = {0, 0, 0}; /* chain chunks [0, end[0]): d > 4; [end[0], end[1]): d 3..4; [end[1], end[2]): d == 2 */
  cudaStream_t stream2 = nullptr, stream3 = nullptr, stream4 = nullptr, stream5 = nullptr, stream6 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join3 = nullptr, ev_join4 = nullptr, ev_join5 = nullptr;
  cudaEvent_t ev_fork6 = nullptr, ev_join6 = nullptr;

  /* fused count exchange over peer memory: one peer-mapped block per rank, laid out as
   * [flags MMQ_P2P_HEAD bytes | counts parity 0 | counts parity 1 | mu] (offsets: p2p_off_* in mmq_core.cu) */
  void* p2p_buf = nullptr;
  int32_t* p2p_counts[2] = {nullptr, nullptr};
  char* p2p_base[MMQ_P2P_MAX] = {};   /* block of every rank as mapped here (own block included) */
  void* p2p_opened[MMQ_P2P_MAX] = {}; /* cudaIpcOpenMemHandle mappings to close */
  int p2p_n = 0, p2p_rank = 0;
  int32_t p2p_epoch = 0;              /* host mirror: sweeps exchanged so far */
  int32_t* counts_own = nullptr;      /* the single-GPU buffers (counts / mu point into p2p_buf when attached) */
  double* mu_own = nullptr;

  /* CUDA graph of MMQ_GRAPH_SWEEPS consecutive sweeps; the sweep counter is read from
   * graph_base on the device, so one instantiated graph serves the whole chain */
  uint32_t* graph_base = nullptr;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  long long graph_launches = 0; /* kernels one replay of the graph launches */
  int32_t graph_epoch0 = 0;     /* p2p_epoch when the capture began */
  int capture_phase = -1, graph_phase = 0; /* first sweep of a replay modulo the trace stride */
  const double* graph_mu = nullptr;
  const int32_t* graph_counts = nullptr;
  uint32_t graph_seed = 0;
  int graph_flags = -1, graph_stride = 0, graph_trace_len = 0;
  const double* graph_trace = nullptr;
  cudaStream_t graph_stream = nullptr;

  /* posterior fragment-count moments (mmq_count_moments_begin; cnt_block null when not accumulating): one block-cache
   * allocation holding sq (u128) and sum (u64) of rows [0, n) transcripts, [n, n + cnt_ident) identical sets and
   * [n + cnt_ident, n + cnt_groups) genes, then cnt_group (int2[n], or none without groups) and cnt_gsum (int32[cnt_groups]) */
  void* cnt_block = nullptr;
  unsigned __int128* cnt_sq = nullptr;
  unsigned long long* cnt_sum = nullptr;
  int2* cnt_group = nullptr;
  int32_t* cnt_gsum = nullptr;
  int64_t cnt_ident = 0, cnt_groups = 0;
  uint64_t cnt_sweeps = 0; /* sweeps accumulated (graph replays counted by mmq_gibbs) */

  /* MMQ_GIBBS_TIME_KERNELS: (start, stop) event pairs around each launch */
  std::vector<cudaEvent_t> ev_alloc, ev_gamma;

  /* mmq_tune: knob 0, pieces of the class-plan sweep not launched (bit mask); knob 6, 1 = the reduce-scatter exchange */
  int skip_mask = 0;
  int exchange_rs = 0;

  int64_t bytes = 0;
  std::string err;
  std::vector<void*> allocs;
  /* one device allocation behind the arrays mmq_create makes (a dozen cudaMalloc calls cost
   * milliseconds each at these sizes); later allocations are separate */
  char* arena = nullptr;
  size_t arena_cap = 0, arena_off = 0;
};

extern std::atomic<long long> g_mmq_launches;
extern thread_local std::string g_mmq_create_err;

int mmq_fail(mmq_handle* h, int code, const std::string& msg);
int mmq_cuda_fail(mmq_handle* h, cudaError_t e, const char* what, const char* file, int line);
/* Device blocks through a process-wide cache (per device, mmq_core.cu): cudaMalloc / cudaFree cost 1-100 ms each at these
 * sizes and vary wildly from call to call (measured: the class plan's dozen temporaries made mmq_create take anywhere from 8
 * to 1900 ms), so blocks that are given back are kept and handed out again.  mmq_cache_free: the caller guarantees that no
 * queued GPU work still touches the block (synchronise the stream first).  mmq_release_cache (mmq.h) returns them to the driver. */
cudaError_t mmq_cache_malloc_raw(void** p, size_t bytes);
void mmq_cache_free(void* p);
template <class T>
static inline cudaError_t mmq_cache_malloc(T** p, size_t bytes) { return mmq_cache_malloc_raw((void**)p, bytes); }
int mmq_dev_alloc(mmq_handle* h, void** p, size_t bytes);
void mmq_dev_free(mmq_handle* h, void* p);
/* in-place sum over the ranks of h's communicator (none: no-op); type 0 int32, 1 fp64, 2 int64 */
int mmq_allreduce(mmq_handle* h, void* buf, size_t count, int type);
int mmq_ensure_trace_groups(mmq_handle* h);
int mmq_seg_scan(mmq_handle* h, const int64_t* row_ptr_host);
int mmq_seg_plan(mmq_handle* h);
int mmq_seg_launch(mmq_handle* h, uint32_t seed, uint32_t sweep, const uint32_t* sweep_base);
int mmq_seg_pack(mmq_handle* h);
int mmq_seg_add_base(mmq_handle* h, bool want_in_counts);
int mmq_cls_plan(mmq_handle* h, const mmq_problem* p);
int mmq_cls_launch(mmq_handle* h, uint32_t seed, uint32_t sweep, const uint32_t* sweep_base);
/* the general allocation kernel (fused reduction, with k, no weights) on an arbitrary sub-CSR and stream */
void mmq_launch_alloc_general(mmq_handle* h, cudaStream_t stream, int grid, const int64_t* row_ptr, const int32_t* col, const int32_t* k,
                              int64_t m, const int64_t* tile_start, int64_t n_tiles, const int64_t* class_id, uint32_t seed,
                              uint32_t sweep, const uint32_t* sweep_base);

#define MMQ_CUDA(h, call)                                                              \
  do {                                                                                 \
    cudaError_t e__ = (call);                                                          \
    if (e__ != cudaSuccess) return mmq_cuda_fail((h), e__, #call, __FILE__, __LINE__); \
  } while (0)

#define MMQ_LAUNCHED(h)                                                                       \
  do {                                                                                        \
    g_mmq_launches.fetch_add(1, std::memory_order_relaxed);                                   \
    cudaError_t e__ = cudaGetLastError();                                                     \
    if (e__ != cudaSuccess) return mmq_cuda_fail((h), e__, "kernel launch", __FILE__, __LINE__); \
  } while (0)

static inline int mmq_grid_for(int64_t work_items, int per_block, int max_blocks) {
  int64_t b = (work_items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return (int)b;
}

#endif
