/* hits_loader.h — host-side loader: .hits file (text schema 0 or zlib-binary
 * schema 1) -> header tables + hit-class CSR, ready for mmq_create.
 *
 * Replaces, for the path, the reference's HitsfileReader (src/hitsio.cpp:250-447)
 * and the class-construction loop of src/mmseq.cpp:395-441, with the header
 * validation of :342-379 and the length scaling of :593-608.
 * Semantics kept: column index = order of first appearance of a transcript in
 * the record stream (:403); a transcript repeated inside one record is counted
 * once and tallied in doublehits (:404-409); the sorted column set is the class
 * key (:412-413); class index = order of first appearance (:417-418); N counts
 * records (:400); transcripts never hit are not columns. */
#ifndef MMQ_HITS_LOADER_H
#define MMQ_HITS_LOADER_H

#include <cstdint>
#include <stdint.h>
#include <string>
#include <vector>

namespace mmq {

struct HitsHeader {
  int schema = 0;                              /* 0 text, 1 binary, 2 binary with per-hit weights */
  std::vector<std::string> names;              /* header order = transcriptList */
  std::vector<double> efflen;                  /* sidLen */
  std::vector<int32_t> truelen;                /* sidSeqLen */
  std::vector<std::string> gene_names;         /* std::map order (byte-wise ascending) */
  std::vector<std::vector<int32_t>> gene_members;  /* header indices, listed order */
  std::vector<std::vector<int32_t>> identical;     /* header indices, listed order */
  std::vector<int32_t> gene_of;                /* [T] index into gene_names */
};

enum Layout {
  LAYOUT_COLLAPSED = 0,        /* reference semantics: distinct sets + k */
  LAYOUT_PER_FRAGMENT = 1,     /* one row per record, record order, k == 1 */
  LAYOUT_PER_FRAGMENT_SORTED = 2, /* one row per record, rows grouped by class */
  LAYOUT_PER_FRAGMENT_BY_LENGTH = 3, /* one row per record, rows grouped by class size, then by
                                        class: the device layout of choice (runs of equal length
                                        need no row pointers, singletons are skipped) */
  /* OR-ed in: columns are header transcript indices (n = T) instead of
   * first-appearance indices — a column space shared by independently loaded
   * shards of one transcriptome (multi-GPU harness) */
  LAYOUT_IDENTITY_COLUMNS = 16,
  /* OR-ed in: the n observed transcripts are numbered in HEADER order instead of
   * first-appearance order.  Headers list a gene's isoforms together, so the mu of
   * co-mapping transcripts share cache lines on the device.  (The reference's .M / .k
   * dumps use first-appearance numbering; the host program writes those from a
   * first-appearance load.) */
  LAYOUT_HEADER_ORDER_COLUMNS = 32
};

struct HitClasses {
  int layout = LAYOUT_COLLAPSED;
  int64_t N = 0;   /* numbermappedreads */
  int64_t n = 0;   /* observed transcripts */
  int64_t m = 0;   /* rows */
  int64_t n_classes = 0; /* distinct sets (== m when collapsed) */
  std::vector<int64_t> row_ptr;
  std::vector<int32_t> col;
  std::vector<int32_t> k;      /* empty in the per-fragment layouts */
  std::vector<float> w;        /* empty without per-hit weights */
  std::vector<int32_t> col2hdr, hdr2col, doublehits;
  /* per-fragment layouts: the distinct sets behind the rows, in first-appearance order — what a
   * LAYOUT_COLLAPSED load of the same records returns as row_ptr / col / k (.k, .M, unique hits).
   * Empty in the collapsed layout, whose rows are the sets. */
  std::vector<int64_t> set_ptr;
  std::vector<int32_t> set_col;
  std::vector<int32_t> set_k;
  /* weighted per-fragment layouts: the first record (0-based, record order) whose weights are all
   * zero — its likelihood is 0 under every mu — or -1 */
  int64_t first_zero_weight_record = -1;
};

/* Both return 0 on success; on failure err holds the reference's message where it has one.
 * weighted_layout >= 0: the layout a file with per-hit weights (schema 2) is loaded in instead of
 * `layout`; hdr.schema tells the caller which one it got.  -1: such a file is loaded in `layout`,
 * which must then be a per-fragment one. */
int load_hits_file(const std::string& path, int layout, HitsHeader& hdr, HitClasses& cls, std::string& err,
                   int weighted_layout = -1);
int validate_header(const HitsHeader& hdr, std::string& err);

/* Streaming class builder (also the in-memory entry point used by the harness). */
class ClassBuilder {
 public:
  ClassBuilder(int64_t n_header_transcripts, int layout, bool weighted);
  /* one record: header transcript indices (and weights) of one fragment */
  void add_record(const int32_t* tids, const float* w, int cnt);
  /* All records at once, on all host threads (nothing added before): either the inflated binary file —
   * off[r] = offset of record r's uint32 hit count, the uint32 transcript indices follow — or the harness's arrays.
   * Same classes, numbering and counts as add_record() record by record.  Return 1 on an index out of range, 2 on a weight that is negative or not finite
   * (weights: schema 2 — one fp32 per hit after a record's indices — or frag_w). */
  bool parallel_ready() const;
  int add_records_binary(const uint8_t* base, const uint64_t* off, int64_t nrec);
  int add_records_csr(const int64_t* frag_ptr, const int32_t* frag_tid, const float* frag_w, int64_t nrec);
  void finish(HitClasses& out);
 private:
  struct Impl;
  Impl* p_;
 public:
  ~ClassBuilder();
};

/* l[t] = efflen * N / 1e9 for the n observed transcripts (src/mmseq.cpp:603). */
int scaled_lengths(const HitsHeader& hdr, const HitClasses& cls, std::vector<double>& l, std::string& err);

}  // namespace mmq


/* host_special.cpp */
extern "C" {
double mmq_host_ndtri(double p);
double mmq_host_digamma(double x);
double mmq_host_trigamma(double x);
}

#endif
