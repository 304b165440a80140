/* mmq.h — C ABI of libmmseq_b200.so: the B200 (sm_100a) implementation of
 * mmseq's expression-estimation hot path (EM initialisation + Gibbs sampler
 * over hit classes), eturro/mmseq 1.0.11 src/mmseq.cpp:593-918 and the
 * summaries of :938-1395.
 *
 * The reference has no plugin or FFI interface for this path: it is one
 * main() (src/mmseq.cpp:179-1728).  The seams this ABI cuts are therefore the
 * loop nests of that function; every entry point cites the lines it replaces.
 * The host program (`mmseq`, mmseq_b200/csrc/mmseq_main.cpp) keeps the
 * reference's command line and file formats and calls only these functions.
 *
 * Conventions
 *   - plain C: pointers and sizes, no C++ or torch types;
 *   - all array arguments are HOST pointers unless the name ends in _dev;
 *     the library owns every device allocation behind the opaque handle;
 *   - every function returns 0 on success, non-zero on failure;
 *     mmq_last_error() gives the message (the reference prints to cerr and
 *     exit(1)s, e.g. src/mmseq.cpp:278-296, :595-607 — the CLI wrapper does that);
 *   - a handle is used from one host thread at a time; handles are independent;
 *   - results do not depend on the GPU count or launch geometry: every random
 *     draw is a pure function of (seed, stream, class or transcript id, sweep)
 *     through Philox4x32-10 (include/mmq_sampler.h).
 * There is no CPU fallback: without a CUDA device mmq_create fails.
 */
#ifndef MMQ_H
#define MMQ_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMQ_OK 0
#define MMQ_ERR_ARG 1
#define MMQ_ERR_CUDA 2
#define MMQ_ERR_STATE 3
#define MMQ_ERR_NCCL 4

typedef struct mmq_handle mmq_handle;

/* The hit-class matrix M of src/mmseq.cpp:117 (boolean, m x n, row-major
 * compressed) in CSR form, with the per-class fragment counts k (:385, :440)
 * and the scaled lengths l (:593-608).  One mmq_problem is one GPU's shard:
 * a contiguous block of classes (rows) and ALL n transcripts (columns). */
typedef struct mmq_problem {
  int64_t n;              /* transcripts with at least one hit (columns), :388 */
  int64_t m;              /* hit classes in this shard (rows), :387            */
  int64_t nnz;            /* row_ptr[m]                                        */
  const int64_t* row_ptr; /* [m+1]                                             */
  const int32_t* col;     /* [nnz] ascending within a row (:412 sort(comb))    */
  const int32_t* k;       /* [m] fragments per class, or NULL meaning all 1
                             (the per-fragment layout)                         */
  const float* weight;    /* [nnz] per-hit weights or NULL.  NULL = reference
                             semantics (M is boolean, :72, :437-438).          */
  const double* len;      /* [n] l[t] = effective_length[t]*N/1e9, :603        */
  double alpha, beta;     /* Gamma prior on mu, :184-185                       */
  int64_t class_id_base;  /* global index of this shard's row 0: the Philox
                             counter of row i is class_id_base + i             */
  const int64_t* class_id; /* [m] explicit Philox counters, or NULL.  Lets the caller
                             hand the classes over in any order (e.g. sorted by cost so
                             that a warp's classes do similar work) and still get the
                             chain of the canonical order.  k != NULL only.       */
} mmq_problem;

/* Upload a shard (H2D) and validate it on the device.  The transcript-major transpose
 * (replaces Mt = trans(M), src/mmseq.cpp:578, and Mrowsum/Mcolsum :582-589) is built on the
 * device by the first call that needs it (mmq_init_mu, mmq_em, a TRANSPOSED sweep). */
int mmq_create(const mmq_problem* problem, int device, mmq_handle** out);
void mmq_destroy(mmq_handle* h);
/* Message of the last failure on h (h may be NULL: failure of mmq_create). */
const char* mmq_last_error(const mmq_handle* h);
/* Run every later call on this cudaStream_t (default: a stream owned by h). */
int mmq_set_stream(mmq_handle* h, void* cuda_stream);
void* mmq_get_stream(mmq_handle* h);
int mmq_synchronize(mmq_handle* h);
/* Device memory held by the handle, bytes. */
int64_t mmq_device_bytes(const mmq_handle* h);

/* Multi-GPU: one process (or thread) per GPU, each with its own shard.  Rank 0
 * calls mmq_comm_id and ships the 128 bytes to the others (torch.distributed,
 * MPI, a file — the caller's plumbing); everyone calls mmq_comm_init.  After
 * that mmq_init_mu / mmq_em / mmq_gibbs end each pass with one NCCL all-reduce
 * over NVLink of the per-transcript vector (int32 counts for Gibbs — the
 * reference's thread-partials sum, src/mmseq.cpp:895-899 — fp64 partial sums
 * for EM).  libnccl.so.2 is dlopen'ed on first use. */
int mmq_comm_id(char id[128]);
int mmq_comm_init(mmq_handle* h, const char id[128], int rank, int nranks);
/* Hand the communicator of `from` (which keeps none) to `to`: lets a long-lived process load
 * the next sample's shard without paying NCCL initialisation again.  A peer-memory attachment
 * (mmq_p2p_attach*) moves along when both handles have the same n; every rank must then make the
 * same move between the same two sweeps. */
int mmq_comm_move(mmq_handle* from, mmq_handle* to);

/* Fused count exchange over NVLink peer memory (optional, on top of the communicator).
 * After mmq_p2p_attach the Gibbs sweep makes no NCCL call: the Gamma kernel of every rank
 * signals "my allocation is done" into its peers' flag words, waits for theirs, then reads the
 * count vectors of ALL ranks straight from peer memory (P2P loads), sums them and draws —
 * the all-reduce (src/mmseq.cpp:895-899) and the Gamma update (:904-908) are ONE kernel.
 * Counts are double-buffered by sweep parity so no second barrier is needed.
 *   multi-process: every rank calls mmq_p2p_export (64-byte cudaIpcMemHandle), the caller
 *     gathers the handles of all ranks (rank order) and passes them to mmq_p2p_attach;
 *   single process, one handle per GPU: mmq_p2p_attach_local with the handles in rank order.
 * All ranks must then issue the same sequence of sweeps (they already must, for NCCL). */
int mmq_p2p_export(mmq_handle* h, char ipc_handle[64]);
int mmq_p2p_attach(mmq_handle* h, const char* ipc_handles, int rank, int nranks);
int mmq_p2p_attach_local(mmq_handle** handles, int nranks);
/* Ranks attached through mmq_p2p_attach*(), 0 when the handle exchanges counts through NCCL (or is alone). */
int mmq_p2p_attached(const mmq_handle* h);

/* mu0[t] = (sum_{i containing t} k[i]/|i|)/l[t] and unique_hits[t] =
 * counts_shared[t][0]; src/mmseq.cpp:617-638.  Leaves mu0 as the current mu.
 * unique_hits_out (int32[n]) may be NULL. */
int mmq_init_mu(mmq_handle* h, int32_t* unique_hits_out);
int mmq_set_mu(mmq_handle* h, const double* mu);
int mmq_get_mu(mmq_handle* h, double* mu_out);

/* sum_i k[i] log(sum_{s in i} mu[s]) - sum_t mu[t] l[t]; src/mmseq.cpp:745-754. */
int mmq_loglik(mmq_handle* h, double* loglik_out);

/* EM from the current mu; src/mmseq.cpp:756-811: llr starts at eps+1, loop
 * while iter < max_iter && llr > eps.  Outputs may be NULL. */
int mmq_em(mmq_handle* h, int max_iter, double eps, int* iters_out, double* loglik_out,
           double* llr_out);

/* Gibbs sweeps first_sweep .. first_sweep+n_sweeps-1 from the current mu;
 * src/mmseq.cpp:851-918.  Sweep s with s % stride == 0 stores mu into trace
 * slot s/stride (slots >= trace_len are dropped), :911-917.  Asynchronous on
 * the handle's stream; mmq_synchronize / mmq_get_* wait for it.
 * flags: MMQ_GIBBS_* below. */
#define MMQ_GIBBS_DEFAULT 0
#define MMQ_GIBBS_TRANSPOSED 1 /* materialise X, reduce over the transposed CSR
                                  (atomic-free); default is the fused path   */
#define MMQ_GIBBS_NO_GRAPH 2   /* plain launches instead of a CUDA graph      */
#define MMQ_GIBBS_TIME_KERNELS 4 /* bracket every k_alloc / k_gamma launch with
                                  CUDA events on the handle's stream; read the
                                  totals with mmq_kernel_times               */
#define MMQ_GIBBS_GENERIC_KERNEL 8 /* k == 1 shards: use the general multinomial
                                  kernel instead of the categorical fast path
                                  (same results; for tests and comparison)   */
#define MMQ_GIBBS_RAGGED_KERNEL 16 /* k == 1 shards: use the row-pointer driven (TMA-staged)
                                  kernel even when the by-length segment plan exists */
int mmq_gibbs(mmq_handle* h, uint32_t seed, int64_t first_sweep, int64_t n_sweeps, int stride,
              int trace_len, int flags);

/* What the class plan of a collapsed shard (classes with counts k; built by mmq_create) holds:
 * out[0] 1 if the plan is in use, out[1] classes of the small set (k <= mmq_cat_limit(d) fragments, at most
 * 64 members: categorical draws, stands in for the multinomial of src/mmseq.cpp:880 for those classes), out[2] packed column
 * slots and out[3] class slots streamed per sweep for them, out[4] classes and out[5] CSR entries
 * left to the general kernel (more than 64 members), out[6] classes of the chain set (more than
 * mmq_cat_limit(d) fragments: gsl_ran_multinomial's conditional-binomial chain, one class per lane) and out[7]
 * their packed column slots.  Used by bench.py for the algorithmic-bytes figure. */
int mmq_cls_stats(const mmq_handle* h, int64_t out[8]);

/* Measurement switches; value 0 restores the default, any knob other than 0 and 6 is MMQ_ERR_ARG.
 * knob 0: bit mask of pieces of the class-plan sweep NOT launched (1 k >= 2 small classes, 2 rest, 4 k >= 2 large
 * classes, 8 chain, 16 single-fragment classes), to time the others alone (tools/gpu_tune_cls.py); the chain is then
 * wrong.  knob 6: 1 = the multi-GPU count exchange as reduce-scatter + all-gather (k_gamma_rs) instead of the all-reduce
 * inside the Gamma kernel (all ranks must set it alike); results do not depend on it. */
int mmq_tune(mmq_handle* h, int knob, int value);

/* Device time of the launches made under MMQ_GIBBS_TIME_KERNELS since the last
 * call (waits for the stream): total milliseconds and launch count of the
 * allocation kernel and of the Gamma kernel.  Any output may be NULL. */
int mmq_kernel_times(mmq_handle* h, double* alloc_ms, int64_t* alloc_launches, double* gamma_ms,
                     int64_t* gamma_launches);

/* One sweep with its integer state exposed, for bit-exact parity against the
 * CPU replay: x_out int32[nnz] (CSR order; the X matrix of :842-847, :884),
 * counts_out int32[n] (Xcolsum, :895-899; the all-reduced vector when a
 * communicator is attached), mu_out fp64[n] after the Gamma step.  Any may be
 * NULL.  flags as mmq_gibbs (TRANSPOSED or fused); both give the same integers. */
int mmq_sweep_debug(mmq_handle* h, uint32_t seed, int64_t sweep, int flags, int32_t* x_out,
                    int32_t* counts_out, double* mu_out);

/* ---- posterior fragment counts per transcript, identical set and gene ----------------------------------
 * (none — the reference reports log_mu and unique hits only; these are the counts Salmon's NumReads, kallisto's
 * est_counts and RSEM's expected_count give.)  c_t(s) is the count of transcript t that the Gamma step of sweep s
 * uses (Xcolsum, src/mmseq.cpp:895-899, singleton classes and all shards included); a group's count is the sum of its
 * members' counts within the sweep, so its variance is not derived from theirs.
 *
 * Start (or restart) accumulating: zeroes the accumulators; every later sweep (mmq_gibbs, graph or not, and
 * mmq_sweep_debug) adds c and c^2 of every row, as exact integers.  ident_of / gene_of: int32[n], the identical set /
 * gene of each observed transcript or -1 (may be NULL when the group count is 0).  Call it with the same arguments on
 * every rank; no communication is added.  mmq_gibbs refuses to accumulate under mmq_tune knob 6 (MMQ_ERR_STATE). */
int mmq_count_moments_begin(mmq_handle* h, const int32_t* ident_of, int64_t n_ident, const int32_t* gene_of, int64_t n_gene);
/* Stop accumulating and free the accumulators. */
int mmq_count_moments_end(mmq_handle* h);
/* which: 0 transcripts (n rows), 1 identical sets, 2 genes.  sweeps: sweeps accumulated (S); sum u64[rows] = sum_s c;
 * sumsq_lo / sumsq_hi u64[rows]: the low and high words of the 128-bit sum_s c^2.  Any output may be NULL.
 * Posterior mean sum / S; sd sqrt((S sumsq - sum^2) / (S (S - 1))) (the S - 1 of src/sokal.cc:63), 0 when S < 2.
 * The moments of several chains (mmseq -chains C -pool) are their exact sums: the caller adds sweeps, sum and the
 * 128-bit sumsq of the handles as integers and finishes with the same expressions (no library call does it). */
int mmq_get_count_moments(mmq_handle* h, int which, int64_t* sweeps, uint64_t* sum, uint64_t* sumsq_lo, uint64_t* sumsq_hi);
/* EM expected counts: one E-step at the current mu, src/mmseq.cpp:781-794: out[t] = mu[t] * sum_{i containing t}
 * k[i] w[i,t] / D_i with D_i = sum_{s in i} mu[s] w[i,s] (w = 1 without weights), summed over all shards (the fp64
 * all-reduce of mmq_em).  sum_t out[t] = N up to rounding.  out fp64[n].  Leaves mu unchanged. */
int mmq_expected_counts(mmq_handle* h, double* out);

/* trace_out[t*trace_len + s] = mu[t] at slot s — the layout of mu_trace,
 * src/mmseq.cpp:827, :914. */
int mmq_get_trace(mmq_handle* h, double* trace_out);
int mmq_trace_len(const mmq_handle* h);

/* ---- posterior summaries on the device (src/mmseq.cpp:938-1363) ---------- */

/* Groups of transcripts whose traces are summed: identical-transcript sets
 * (:938-954) and genes (:959-982).  member ids index the n observed
 * transcripts; `extra` (fp64[ngroups*trace_len], may be NULL) is added to the
 * group trace — the prior-simulated Gamma draws of hit-less isoforms, :971-978. */
#define MMQ_GROUP_IDENTICAL 0
#define MMQ_GROUP_GENE 1
int mmq_set_groups(mmq_handle* h, int kind, int64_t ngroups, const int64_t* group_ptr,
                   const int32_t* members, const double* extra);

/* Per-feature summaries of a trace matrix.  which: 0 transcripts (n rows),
 * 1 identical sets, 2 genes.  All outputs fp64[rows] unless noted; NULL skips.
 *   log_mean   mean of log(trace)                                  :1203-1227
 *   var,tau,win  sokal() on the log trace (win int32)        :1308-1363, sokal.cc:33-87
 *   pct        fp64[rows*npct], sorted raw trace at index pct_idx[j]   :1111-1172 */
int mmq_summarize(mmq_handle* h, int which, double* log_mean, double* var, double* tau,
                  int32_t* win, int32_t* sokal_status, int npct, const int32_t* pct_idx, double* pct);
/* Group traces back to the host, [g*trace_len + s]; which = 1 or 2 as above. */
int mmq_get_group_trace(mmq_handle* h, int which, double* out);

/* Proportion summaries of the observed transcripts (:985-1008, :1236-1265):
 * prop = mu_t / gene trace; mean_prop; sum and sum of squares of
 * Phi^-1(clamp(prop, 1e-9, 1-1e-9)) (callers finish :1261-1265 on the host);
 * pct of the sorted proportion trace.  gene_of[t] = gene index of transcript t
 * (int32[n]); multi_iso[t] != 0 when the gene has more than one isoform. */
int mmq_prop_summaries(mmq_handle* h, const int32_t* gene_of, const uint8_t* multi_iso,
                       double* mean_prop, double* sum_probit, double* sumsq_probit, int npct,
                       const int32_t* pct_idx, double* pct, double* prop_trace_out);

/* uh(): unique hits of transcript sets, src/uh.cpp:3-26 — sum of k[i] over the
 * classes all of whose members lie in one set.  set_of int32[n]: the set of
 * each transcript or -1.  out int32[nsets] (all-reduced over shards). */
int mmq_unique_hits_sets(mmq_handle* h, const int32_t* set_of, int64_t nsets, int32_t* out);

/* Prior draws for transcripts without hits, src/mmseq.cpp:971-978:
 * out[u*trace_len + s] ~ Gamma(alpha, rate[u]) with rate[u] = beta + len*N/1e9, from the
 * PRIOR Philox stream keyed by (seed, ids[u], s) — the reference draws them from rg[0]. */
int mmq_prior_draws(int device, int64_t count, const int64_t* ids, const double* rate, double alpha,
                    uint32_t seed, int trace_len, double* out);

/* Stand-alone batched Sokal on host data: rows x len fp64 (len a power of two,
 * 4..2048); src/sokal.cc:33-87. */
int mmq_sokal_batch(int device, int64_t rows, int len, const double* x, double* var, double* tau,
                    int32_t* win, int32_t* status);

/* ---- convergence of several independent chains (none in the reference; mmseq -chains) -----------------------------
 * Seed of chain `chain` (0 <= chain < 8) of a run with seed `seed`: chain 0 is `seed` itself; chain c >= 1 is word 0 of
 * Philox4x32-10 at counter (c, j, 0, 0) under key (seed, 0x4348414e "CHAN") for the first j whose value differs from the
 * seeds of chains 0 .. c-1, so the seeds of one run are distinct.  Outside the range: `seed`.  (include/mmq_sampler.h
 * defines the same function inline for host and device code.) */
#ifndef MMQ_SAMPLER_H
uint32_t mmq_chain_seed(uint32_t seed, int chain);
#endif
/* Rank-normalised split-R-hat and bulk / tail effective sample size per feature (Vehtari, Gelman, Simpson, Carpenter,
 * Buerkner 2021, as Stan, ArviZ and the `posterior` R package report them).  chain_dev[c] (a host array of device
 * pointers): chain c's draws [row * L + s], the mmq_get_trace layout, all on the calling device; 2 <= nchains <= 8, L a
 * power of two in [8, 2048], nchains * L <= 8192, else MMQ_ERR_ARG.  out_dev: fp64[5 * rows], [q * rows + row] for
 * q = 0 rhat, 1 ess_bulk, 2 ess_tail, 3 log_mean, 4 log_sd.  Asynchronous on cuda_stream, no allocation; one CTA per
 * feature, grid min(rows, 2 x SMs); every value is fp64 and independent of the grid and of the row order.
 * Definitions, for one feature's draws x[c][s] (S = nchains L draws), split into M = 2 nchains chains of N = L/2,
 * y[2c+h][i] = x[c][h N + i]:
 *   any x NaN or +-inf: all five outputs NaN;
 *   z(v) = Phi^-1((r - 3/8) / (S + 1/4)), r the average rank of each value among all S (ties share the mean rank);
 *   split R-hat(y): m_j, w_j the split chains' means and variances (ddof 1; a chain of equal values: that value and 0),
 *     W = mean w_j, B = N var(m_j, ddof 1), R-hat = sqrt(((N-1)/N W + B/N) / W), NaN when W = 0;
 *   rhat = max(R-hat(z(x)), R-hat(z(|x - med|))), med the median of all S draws; NaN when either is NaN;
 *   ess(y): Geyer's initial monotone sequence over the split chains' autocovariances, as Stan and ArviZ compute it
 *     (tests/chain_reference.py spells it out), NaN when all S values of y are equal;
 *   ess_bulk = ess(z(x)); ess_tail = min(ess(1[x <= q_0.05]), ess(1[x <= q_0.95])), q_p the type-7 quantile of all S
 *     draws, NaN when either is NaN;
 *   log_mean, log_sd: mean and sd (S - 1) of log x over all S draws, plain IEEE (a zero draw gives -inf / NaN). */
int mmq_chain_diagnostics_dev(const double* const* chain_dev, int nchains, int64_t rows, int L, double* out_dev, void* cuda_stream);
/* The same on the traces the handles recorded (mmq_gibbs with trace_len = L): which 0 transcripts, 1 identical sets,
 * 2 genes (groups set alike on every handle, mmq_set_groups).  Runs on chains[0]'s device and stream; traces of handles
 * on other devices are copied there (cudaMemcpyPeerAsync, a workspace of rows L 8 bytes per such chain).  Same n,
 * trace_len and group counts on every handle, else MMQ_ERR_ARG.  Outputs fp64[rows] on the host; any may be NULL. */
int mmq_chain_diagnostics(mmq_handle* const* chains, int nchains, int which, double* rhat, double* ess_bulk,
                          double* ess_tail, double* log_mean, double* log_sd);

/* Posterior summaries over the pooled draws of several chains (none in the reference; mmseq -chains C -pool): the
 * columns of the .mmseq tables over all S = nchains L draws of a feature instead of one chain's L.  chain_dev, nchains,
 * L and their limits as mmq_chain_diagnostics_dev, else MMQ_ERR_ARG.  pct_idx_dev: int32[npct] on the device, indices
 * into the S sorted draws (an index outside [0, S) gives NaN); pct_dev: fp64[rows * npct], [row * npct + j]; both may be
 * NULL when npct = 0.  out_dev: fp64[3 * rows], [q * rows + row].  Asynchronous on cuda_stream, no allocation; one CTA
 * per feature, grid min(rows, 2 x SMs); every value is fp64, summed in a fixed order, and independent of the grid and
 * of the row order.  Definitions, for one feature's draws x[c][s] (tests/pool_reference.py restates them):
 *   pct[j] = the draws sorted ascending (NaN last), at index pct_idx[j] (the host program: round(p / 100 (S - 1)));
 *   mode 0 (draws of mu):
 *     q = 0 log mean and q = 1 sd (S - 1) of log x over all S draws, plain IEEE (a zero draw gives -inf / NaN), NaN
 *       when any x is NaN or +-inf: the bits of mmq_chain_diagnostics_dev's log_mean and log_sd;
 *     q = 2 ess_mean: the ESS of mmq_chain_diagnostics_dev (Geyer's initial monotone sequence over the 2 nchains split
 *       chains) applied to log x itself, not to its ranks; NaN when any log x is not finite or all are equal.
 *     The tables' mcse = sd / sqrt(ess_mean) and iact = S / ess_mean (NaN with ess_mean).
 *   mode 1 (proportion draws): q = 0 the mean of x over all S draws; q = 1, 2 are not written. */
int mmq_pooled_summaries_dev(const double* const* chain_dev, int nchains, int64_t rows, int L, int mode, int npct,
                             const int32_t* pct_idx_dev, double* out_dev, double* pct_dev, void* cuda_stream);
/* The same on the traces the handles recorded (mmq_gibbs with trace_len = L), on chains[0]'s device and stream, traces of
 * other devices copied there (cudaMemcpyPeerAsync, as mmq_chain_diagnostics).  which 0 transcripts, 1 identical sets,
 * 2 genes: mode 0 into mean (log mean), sd and ess_mean.  which 3, the proportions of the observed transcripts: every
 * chain's proportion draws are mu_t over that chain's own gene trace (mmq_prop_summaries' k_prop, run on each chain's
 * device; gene_of, multi_iso as there), mode 1 into mean; sum_probit / sumsq_probit receive each chain's sum and sum of
 * squares of the probits added in chain order (the host finishes them as src/mmseq.cpp:1260-1265 with S draws);
 * sd and ess_mean are not written.  gene_of / multi_iso are read for which 3 only.  pct_idx host int32[npct] in [0, S),
 * else MMQ_ERR_ARG.  Same n, trace_len and group counts on every handle, else MMQ_ERR_ARG.  Outputs fp64[rows] (pct
 * fp64[rows * npct]) on the host; any may be NULL. */
int mmq_pooled_summaries(mmq_handle* const* chains, int nchains, int which, const int32_t* gene_of, const uint8_t* multi_iso,
                         int npct, const int32_t* pct_idx, double* mean, double* sd, double* ess_mean, double* sum_probit,
                         double* sumsq_probit, double* pct);

/* ---- transcripts per million (none in the reference; mmseq -tpm) ------------------------------------------------------
 * The abundance unit Salmon, kallisto and RSEM report, with its posterior over the recorded draws.  mu is a rate per
 * scaled length (l_t = efflen_t N / 1e9, so exp(log_mu) is on the FPKM scale), and TPM is mu normalised within each draw.
 * tests/tpm_reference.py restates these definitions in numpy.  x_c[t][s]: chain c's recorded draw of mu for observed
 * transcript t < n at slot s < L (the mmq_get_trace layout [t * L + s]); C chains, S = C L draws per feature.
 *   1. Totals: D_c[s] = sum_{t < n} x_c[t][s] in fp64 over the observed transcripts only (hit-less isoforms' prior draws
 *      are not included).  Order: tiles of 512 rows, each summed in row order per slot from 0.0, then the tile sums in
 *      tile order from 0.0.  It depends on (n, L) only, so the bits are the same on any grid, device or repeat, and the
 *      relative error is at most about (512 + n / 512) eps: within 1e-12 of the exact sum of positive draws.
 *   2. Draws of a feature: its members are itself (a transcript) or its observed members in the CSR order given to
 *      mmq_set_groups (an identical set or a gene; the group's `extra` is NOT added).  Per draw, w = the sum of the
 *      members' draws in that order from 0.0, and tpm_c[s] = (w / D_c[s]) * 1e6, in plain IEEE in exactly that order.  A
 *      feature without members has w = 0 and so TPM 0 in every draw.  Sum over transcripts, or over genes, is 1e6.
 *   3. Over the S draws: mean = sum tpm / S (fixed order); sd = sqrt(sum (tpm - mean)^2 / (S - 1)), two-pass; both NaN
 *      when any draw is not finite.  pct[j] = the draws sorted ascending (NaN last) at index pct_idx[j]; an index outside
 *      [0, S) gives NaN (the host program: round(p / 100 (S - 1)), as -pool).
 *   4. EM (computed by the caller): tpm_em_f = (sum_{members} mu_em[t] / sum_{t < n} mu_em[t]) * 1e6, both sums in index
 *      order; 0 for a feature without members.
 * Limits: 1 <= nchains <= 8, L a power of two in [4, 2048], nchains L <= 8192; otherwise MMQ_ERR_ARG. */
/* Bytes of workspace mmq_draw_totals_dev needs for a trace of `rows` rows (8 L ceil(rows / 512); 0 for bad arguments). */
int64_t mmq_draw_totals_workspace_bytes(int64_t rows, int L);
/* totals_dev fp64[L] = D[s] of definition 1 over the trace trace_dev [row * L + s] (rows >= 0; rows = 0 gives 0.0).
 * Asynchronous on cuda_stream, no allocation: workspace_dev holds mmq_draw_totals_workspace_bytes(rows, L) bytes. */
int mmq_draw_totals_dev(const double* trace_dev, int64_t rows, int L, double* totals_dev, void* workspace_dev, void* cuda_stream);
/* Summaries 2-3 per feature.  chain_dev[c] (a host array of device pointers): chain c's transcript trace [t * L + s];
 * totals_dev fp64[nchains L], chain-major (chain c's D at [c L + s]); group_ptr_dev int64[rows + 1] / members_dev int32
 * both given (feature r = members[group_ptr[r] .. group_ptr[r + 1]) ) or both NULL (feature r = transcript r).  out_dev
 * fp64[2 rows]: [r] mean, [rows + r] sd; pct_dev fp64[rows npct], [r npct + j]; pct_idx_dev int32[npct] (both may be NULL
 * when npct = 0).  All on the calling device; asynchronous on cuda_stream, no allocation; one CTA per feature, grid
 * min(rows, 2 x SMs); results independent of the grid and of the row order. */
int mmq_tpm_summaries_dev(const double* const* chain_dev, const double* totals_dev, int nchains, int64_t rows, int L,
                          const int64_t* group_ptr_dev, const int32_t* members_dev, int npct, const int32_t* pct_idx_dev,
                          double* out_dev, double* pct_dev, void* cuda_stream);
/* The same on the traces the handles recorded (mmq_gibbs with trace_len = L): which 0 transcripts, 1 identical sets,
 * 2 genes, with the groups of chains[0] (mmq_set_groups).  Each chain is normalised by its own totals.  Runs on
 * chains[0]'s device and stream; transcript traces of handles on other devices are copied there (cudaMemcpyPeerAsync,
 * as mmq_chain_diagnostics); the workspace comes from the block cache.  Same n, trace_len and group counts on every
 * handle, and pct_idx (host int32[npct]) in [0, S), else MMQ_ERR_ARG.  mean, sd fp64[rows], pct fp64[rows npct] and
 * totals_out fp64[nchains L] (the D_c, chain-major) on the host; any may be NULL. */
int mmq_tpm_summaries(mmq_handle* const* chains, int nchains, int which, int npct, const int32_t* pct_idx, double* mean, double* sd,
                      double* pct, double* totals_out);

/* ---- allelic fraction of haplotype pairs (none in the reference; mmseq -allelic) ---------------------------------------
 * A haplotype-aware reference lists every transcript twice, STEM_A and STEM_B.  The two copies share most of their
 * fragments, so their draws are anti-correlated and the sd of a ratio cannot be formed from the .mmseq columns; these
 * functions compute it per draw.  tests/allelic_reference.py restates the definitions in numpy.
 *   1. Pairs (the caller's, mmseq_main.cpp): header transcripts named STEM_A and STEM_B (fixed suffixes) in one gene,
 *      with or without hits; id STEM; in the header order of the _A copy.  A transcript named *_A / *_B whose partner is
 *      missing or in another gene is not paired.  Genes: a gene's A side is the _A copies of the pairs inside it, its B
 *      side their _B copies (in pair order); isoforms outside a pair are ignored.
 *   2. Members (column space): an id m < n is observed transcript m, a row of the chain's trace; an id n + j is row j of
 *      the caller's prior draws of that chain, laid out [j L + s] as mmq_prior_draws writes them.  The host program
 *      passes, as prior rows, exactly the hit-less copies that belong to a pair, in header order: the draws that chain
 *      already uses for them, the exact posterior of a copy without fragments.
 *   3. Per draw (chain c, slot s): a = the sum of the A members' draws in CSR order from 0.0, b the same for the B
 *      members, phi = a / (a + b) in plain IEEE.  No fraction trace is stored.
 *   4. Over the S = C L draws: mean = sum phi / S; sd = sqrt(sum (phi - mean)^2 / (S - 1)), two-pass; prob_a =
 *      (#{a > b} + #{a = b} / 2) / S; pct[j] = phi sorted ascending (NaN last) at index pct_idx[j] (the host program:
 *      round(p / 100 (S - 1)), as -tpm).  If any phi is not finite (a + b = 0 in some draw, as for a unit without
 *      members) every one of these is NaN.
 *   5. EM (the caller's): em_fraction_a = sum_A mu_em / (sum_A mu_em + sum_B mu_em) over the observed members in index
 *      order, hit-less copies counting 0; NaN when both sums are 0.
 *   6. Allele-only fragments: a_only[u] = sum of k_i over the hit classes i that contain an A member of unit u and no B
 *      member of u; b_only[u] the same with A and B swapped.  A per-fragment layout (k = NULL, also a weighted file)
 *      counts 1 per row: set membership decides, the weights are ignored (as for unique hits).  Exact int32 counts. */
/* unit_of int32[n]: the unit of each observed transcript or -1; side uint8[n]: 0 (A) or 1 (B).  a_only, b_only
 * int32[nunits] on the host, all-reduced over the shards of a communicator (every rank calls it, as mmq_unique_hits_sets).
 * A unit index outside [-1, nunits) or a side other than 0 / 1 is MMQ_ERR_ARG. */
int mmq_allele_only_counts(mmq_handle* h, const int32_t* unit_of, const uint8_t* side, int64_t nunits, int32_t* a_only,
                           int32_t* b_only);
/* Summaries 3-4 per unit.  chain_dev[c] (a host array of device pointers): chain c's transcript trace [t L + s] over n
 * observed transcripts; prior_dev[c]: chain c's nprior prior rows [j L + s] (prior_dev, or each prior_dev[c], may be NULL
 * when nprior = 0); a_ptr_dev int64[rows + 1] / a_mem_dev int32 and b_ptr_dev / b_mem_dev: the A and B members of every
 * unit, ids in [0, n + nprior) (not checked here: the handle form checks them).  out_dev fp64[3 rows]: [r] mean,
 * [rows + r] sd, [2 rows + r] prob_a; pct_dev fp64[rows npct], [r npct + j].  All on the calling device; asynchronous on
 * cuda_stream, no allocation; one CTA per unit, grid min(rows, 2 x SMs); results independent of the grid and of the row
 * order.  Limits those of -tpm: 1 <= nchains <= 8, L a power of two in [4, 2048], nchains L <= 8192; else MMQ_ERR_ARG. */
int mmq_allelic_summaries_dev(const double* const* chain_dev, const double* const* prior_dev, int nchains, int64_t n, int64_t nprior,
                              int64_t rows, int L, const int64_t* a_ptr_dev, const int32_t* a_mem_dev, const int64_t* b_ptr_dev,
                              const int32_t* b_mem_dev, int npct, const int32_t* pct_idx_dev, double* out_dev, double* pct_dev,
                              void* cuda_stream);
/* The same on the transcript traces the handles recorded (same n and trace_len on every handle), on chains[0]'s device
 * and stream; traces of handles on other devices are copied there with cudaMemcpyPeerAsync, the prior rows prior_host[c]
 * (host fp64[nprior L] per chain) and the CSRs with cudaMemcpyAsync into block-cache memory.  A member id outside
 * [0, n + nprior), a CSR that does not start at 0 or decreases, or pct_idx outside [0, S) is MMQ_ERR_ARG.  mean, sd,
 * prob_a fp64[rows] and pct fp64[rows npct] on the host; any may be NULL. */
int mmq_allelic_summaries(mmq_handle* const* chains, int nchains, const double* const* prior_host, int64_t nprior, int64_t rows,
                          const int64_t* a_ptr, const int32_t* a_mem, const int64_t* b_ptr, const int32_t* b_mem, int npct,
                          const int32_t* pct_idx, double* mean, double* sd, double* prob_a, double* pct);

/* ---- isoform pairs within a gene (none in the reference; mmseq -isocorr) ------------------------------------------------
 * Isoforms that share most of their fragments get strongly anti-correlated draws: their marginal log_mu and sd look
 * confident while their split is not.  mmcollapse thresholds the correlation of the mu draws (src/mmcollapse.cpp:514-561);
 * these functions give it per sample and gene, with P(first > second) and the shared fragments, without the trace files.
 * tests/isocorr_reference.py restates the definitions in numpy.
 *   1. Pairs: for every gene, its observed isoforms (members with hits) in the CSR order given to
 *      mmq_set_groups(MMQ_GROUP_GENE) (the host program: header order), m_0 .. m_{k-1}.  Every (a, b) with a < b is one
 *      pair, a-major within the gene; genes in group order.  pair_base[g] = sum_{g' < g} k'(k' - 1) / 2, and the pair
 *      index is pair_base[g] + a (2k - a - 1) / 2 + (b - a - 1).  Hit-less isoforms (their prior draws are independent of
 *      everything by construction) and isoforms of different genes are not pairs.
 *   2. Draws: x_i[c, s] = chain c's recorded mu of member i at slot s, over S = C L draws; a pair's two values always come
 *      from the same (c, s).
 *   3. Per pair (i, j): corr_mu = sum (x_i - m_i)(x_j - m_j) / sqrt(sum (x_i - m_i)^2 sum (x_j - m_j)^2), two-pass, m the
 *      mean over all S draws (pooled, not per chain), clamped to [-1, 1]; corr_log_mu the same on log x; prob_1_gt_2 =
 *      (#{x_i > x_j} + #{x_i = x_j} / 2) / S.  A correlation is NaN when either member has a draw that is not finite (for
 *      the log, also a draw <= 0) or a centred sum of squares of 0; all three are NaN when either member has a NaN draw.
 *      Order: a member's mean and sum of squares over the draws in 32 lane-strided partial sums and a fixed shuffle tree;
 *      a pair's cross sum in draw order (fma) by one thread.  Nothing depends on the grid, the device, the gene order or
 *      a repeat.
 *   4. Shared fragments: shared[p] = sum of k_r over the hit classes r that contain both members of pair p.  A
 *      per-fragment layout (k = NULL, also a weighted file) counts 1 per row: the weights are ignored (as for unique
 *      hits), so a weighted file gives the counts of the unweighted file with the same records.  Exact int64.
 * Limits of the summaries those of -tpm: 1 <= nchains <= 8, L a power of two in [4, 2048], nchains L <= 8192. */
/* gene_of / local_of int32[n]: the gene and the local index a of every observed transcript, both -1 for one whose gene
 * has fewer than 2 observed isoforms; pair_base int64[ngenes] (definition 1; gene g's pairs end at pair_base[g + 1], the
 * last gene's at npairs).  out int64[npairs] on the host, all-reduced over the shards of a communicator (every rank
 * calls it, as mmq_allele_only_counts).  A gene index outside [-1, ngenes), a local index outside [0, k), a pair_base
 * that does not start at 0, decreases, exceeds npairs or gives a gene a pair count other than k (k - 1) / 2 is
 * MMQ_ERR_ARG. */
int mmq_pair_shared_counts(mmq_handle* h, const int32_t* gene_of, const int32_t* local_of, const int64_t* pair_base, int64_t ngenes,
                           int64_t npairs, int64_t* out);
/* Bytes of workspace mmq_isocorr_summaries_dev needs: 40 nmembers + 8 (ngenes + 1) (0 for bad arguments). */
int64_t mmq_isocorr_workspace_bytes(int64_t ngenes, int64_t nmembers);
/* Summaries 3 per pair.  chain_dev[c] (a host array of device pointers): chain c's transcript trace [t L + s];
 * gene_ptr_dev int64[ngenes + 1] / members_dev int32[nmembers]: every gene's observed members (trace rows, not checked
 * here: the handle form's come from mmq_set_groups), nmembers = gene_ptr[ngenes]; pair_base_dev int64[ngenes]
 * (definition 1, npairs in all).  out_dev fp64[3 npairs]: [p] corr_mu, [npairs + p] corr_log_mu, [2 npairs + p]
 * prob_1_gt_2.  All on the calling device; asynchronous on cuda_stream, no allocation: workspace_dev holds
 * mmq_isocorr_workspace_bytes(ngenes, nmembers) bytes.  Work items (gene, pair of 32-member tiles), grid
 * min(npairs, 2 x SMs); every member's trace row is read once per item.  Bad limits are MMQ_ERR_ARG. */
int mmq_isocorr_summaries_dev(const double* const* chain_dev, int nchains, int64_t ngenes, int64_t nmembers, int L,
                              const int64_t* gene_ptr_dev, const int32_t* members_dev, const int64_t* pair_base_dev, int64_t npairs,
                              double* out_dev, void* workspace_dev, void* cuda_stream);
/* The same on the transcript traces the handles recorded (same n, trace_len and group counts on every handle), with
 * chains[0]'s gene groups; pair_base is derived from that CSR.  Runs on chains[0]'s device and stream; traces of handles
 * on other devices are copied there with cudaMemcpyPeerAsync; the workspace comes from the block cache.  npairs other
 * than the groups' pair count is MMQ_ERR_ARG.  corr_mu, corr_log_mu, prob_gt fp64[npairs] on the host; any may be NULL. */
int mmq_isocorr_summaries(mmq_handle* const* chains, int nchains, int64_t npairs, double* corr_mu, double* corr_log_mu, double* prob_gt);

/* ---- the consumer of the traces: mmcollapse's covariance step (src/mmcollapse.cpp:483-561) ----------
 * The one dense contraction of the package: tensor cores (tcgen05, bf16 split products, fp32 accumulation in
 * TMEM), everything around it fp64.  nsplit = bf16 terms per value (2: the default of the callers here).  Error in
 * correlation units, |cov - cov_exact| / (sd_i sd_j), for traces of length L: at most A + 1.5e-8 L with A = 6e-3 /
 * 1.2e-5 / 2e-7 for nsplit = 1 / 2 / 3.  A is the bf16 split; 1.5e-8 L is the fp32 accumulation, which truncates
 * towards zero (|r| comes out a little small) and so grows linearly with L.  At L = 1024: 6e-3 / 2.7e-5 / 1.6e-5; at
 * the longest L, 65536: 7e-3 / 1e-3 / 1e-3.  (Fitted with a margin of 1.5x or more over the largest error measured on
 * a B200, tests/collapse_case.py.)
 * A feature whose centred sum of squares is not finite (a non-finite value, or |x - mean| of ~1e154 and more) gets a
 * zero row and column, its variance included.  Armadillo's cov() keeps the finite off-diagonal entries of such a
 * feature, but mmcollapse divides them by its variance, which :556-558 sets to 0: its correlations are not finite
 * either way. */

/* get_corrs()'s per-sample step, src/mmcollapse.cpp:553-558: R = cov(M) of the L x C trace matrix (column c =
 * the L posterior draws of feature c, contiguous: Armadillo's layout of myM and the layout of mmq_get_trace),
 * non-finite -> 0.  R: C x C fp64, both triangles, exactly symmetric, diagonal = the columns' variances.
 * L a multiple of 64 (mmcollapse: TRACELEN 1024).  Host pointers; H2D, kernels and D2H inside. */
int mmq_trace_cov(int device, const double* M, int L, int64_t C, int nsplit, double* R);
/* Same on device-resident data, asynchronous on cuda_stream, no allocation inside: workspace_dev must hold
 * mmq_trace_cov_workspace_bytes(L, C, nsplit) bytes (256-byte aligned). */
int64_t mmq_trace_cov_workspace_bytes(int L, int64_t C, int nsplit);
int mmq_trace_cov_dev(const double* M_dev, int L, int64_t C, int nsplit, double* R_dev, void* workspace_dev, void* cuda_stream);
/* Straight from the trace a handle recorded (mmq_gibbs with trace_len = L): features[c] = index of an observed
 * transcript; no trace file round trip (the reference re-reads *.trace_gibbs.gz, src/mmcollapse.cpp:530-551).
 * R_out (host) and / or R_dev_out (device, C x C fp64) receive the matrix; either may be NULL. */
int mmq_handle_trace_cov(mmq_handle* h, const int32_t* features, int64_t C, int nsplit, double* R_out, double* R_dev_out);

/* mean_corrs(), src/mmcollapse.cpp:483-511.  R: C x C x ns cube (slice s at R + s C C, symmetric slices as
 * mmq_trace_cov writes them), S: C x ns column-major, 1 where feature c was observed in sample s (:686-695);
 * for every t in ts[0..nts) and v in 0..C-1: V(t,v) = V(v,t) = mean over the samples with S(t,s) S(v,s) = 1 of
 * R(t,v,s)/sqrt(R(t,t,s))/sqrt(R(v,v,s)) + sdpenalty * W(t,v), W = their sd (0 for one sample or if not finite).
 * V, W: C x C fp64, read and written (entries outside the rows / columns of ts stay). */
int mmq_mean_corrs(int device, const double* R, const uint8_t* S, int64_t C, int ns, const int32_t* ts, int64_t nts, double sdpenalty,
                   double* V, double* W);
int mmq_mean_corrs_dev(const double* R_dev, const uint8_t* S_dev, int64_t C, int ns, const int32_t* ts_dev, int64_t nts, double sdpenalty,
                       double* V_dev, double* W_dev, void* cuda_stream);

/* Device memory given back by mmq_destroy and by the set-up steps' temporaries is kept in a per-device cache and handed
 * out again (cudaMalloc / cudaFree of these sizes cost 1-100 ms each and made mmq_create vary between 8 ms and 2 s; a
 * process that runs one sample after another — config 5 — now pays them once).  At most MMQ_DEVICE_CACHE_MB (environment,
 * default 16384; 0 disables) are held per device; this call returns them to the driver (device < 0: every device). */
int mmq_release_cache(int device);

/* Kernel launches issued by this process through the library so far. */
int64_t mmq_launch_count(void);
/* Bring up the CUDA context of `device` (the first CUDA call of a process costs 1-2 s): a host
 * program calls this from a side thread while it parses its input.  No reference counterpart. */
int mmq_warmup(int device);

const char* mmq_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MMQ_H */
