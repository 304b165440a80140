/* mmseq_main.cpp — the `mmseq` host program: the reference's command line and
 * file formats (src/mmseq.cpp:156-296, :1469-1694 of eturro/mmseq 1.0.11) over
 * the CUDA hot path behind include/mmq.h.
 *
 *   mmseq [OPTIONS...] hits_file output_base
 *
 * Same flags, defaults, validation messages and exit codes as the reference;
 * same output files and column layouts.  Everything numeric runs on the GPU
 * through the C ABI: initial mu and unique hits, EM, the Gibbs sweeps, the
 * prior draws of hit-less isoforms, trace aggregation, Sokal, percentiles and
 * proportion summaries.  The host only parses, formats and writes.
 * Additive options: -gpus INT (shard hit classes over GPUs of this box),
 * -notraces (skip the four *.trace_gibbs.gz text dumps), -batch FILE / -per_gpu INT (many
 * samples dealt to the GPUs, independent chains: BASELINE config 5), -counts (posterior and EM fragment counts per
 * transcript, identical set and gene: *.counts, *.identical.counts, *.gene.counts), -chains INT (independent chains
 * from the EM estimate, split-R-hat and bulk / tail ESS per transcript, identical set and gene: *.convergence,
 * *.identical.convergence, *.gene.convergence), -pool (with -chains: the three tables and the -counts files over the draws
 * of all chains), -tpm (posterior and EM transcripts per million per transcript, identical set and gene: *.tpm,
 * *.identical.tpm, *.gene.tpm), -allelic (posterior and EM allelic fraction per haplotype pair STEM_A / STEM_B and gene:
 * *.allelic, *.gene.allelic), -isocorr (posterior correlation, P(first > second) and shared fragments of every isoform
 * pair within a gene: *.isocorr).
 */
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <charconv>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <functional>
#include <iostream>
#include <limits>
#include <map>
#include <sstream>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/mmq.h"
#include "fmt_g6.h"
#include "huff_gz.h"
#include "trace_writer.h"
#include "hits_loader.h"

#define QUOTE_(x) #x
#define QUOTE(x) QUOTE_(x)
#ifndef VERSION
#define VERSION 1.0.11-b200
#endif

using namespace std;

/* The usage text of the reference (src/mmseq.cpp:156-177) plus the additive options. */
static void printUsage(ostream& out) {
  out << "Usage: mmseq [OPTIONS...] hits_file output_base" << endl
      << endl
      << "Mandatory arguments:" << endl
      << "  hits_file          hits file generated with `bam2hits`\n"
      << "  output_base        base name for output files" << endl
      << endl
      << "Optional arguments:\n"
      << "  -alpha FLOAT       value of alpha in Gamma prior for mu (default: 0.1)" << endl
      << "  -beta FLOAT        value of beta in Gamma prior for mu (default: 0.1)" << endl
      << "  -max_em_iter INT   maximum number of EM iterations (default: 1000)" << endl
      << "  -epsilon FLOAT     minimum loglik ratio between successive EM iterations (default: 0.1)" << endl
      << "  -gibbs_iter INT    number of Gibbs iterations (default: 16384)" << endl
      << "  -gibbs_ss INT      subsampling interval for Gibbs output (default: gibbs_iter/1024)" << endl
      << "  -seed INT          seed for the PRNG in thread 0 (default: 1234)" << endl
      << "  -percentiles STR   comma-separated list of real-scale marginal posterior percentiles to output (default: \"5,25,50,75,95\")" << endl
      << "  -debug             output additional diagnostic files" << endl
      << "  -help              print this help message" << endl
      << "  -version           print the version" << endl
      << "  -gpus INT          (B200 build) shard hit classes over this many GPUs (default: 1)" << endl
      << "  -notraces          (B200 build) do not write the *.trace_gibbs.gz text dumps" << endl
      << "  -batch FILE        (B200 build) many samples: FILE lists one \"hits_file output_base\" pair per line (no positional arguments)" << endl
      << "  -per_gpu INT       (B200 build) batch mode: samples in flight per GPU (default: 4)" << endl
      << "  -counts            (B200 build) also write posterior and EM fragment counts (*.counts, *.identical.counts, *.gene.counts)" << endl
      << "  -chains INT        (B200 build) run INT independent chains (1..8, default: 1) and write split-R-hat and ESS per feature (*.convergence, *.identical.convergence, *.gene.convergence)" << endl
      << "  -pool              (B200 build) with -chains 2 or more: the *.mmseq tables and -counts files summarise the draws of all chains (default: chain 1's); trace files stay chain 1's" << endl
      << "  -tpm               (B200 build) also write posterior and EM transcripts per million (*.tpm, *.identical.tpm, *.gene.tpm)" << endl
      << "  -allelic           (B200 build) also write the posterior and EM allelic fraction of every haplotype pair STEM_A / STEM_B and gene (*.allelic, *.gene.allelic)" << endl
      << "  -isocorr           (B200 build) also write the posterior correlation, P(first > second) and shared fragments of every isoform pair within a gene (*.isocorr)" << endl
      << endl;
}

[[noreturn]] static void die(const string& msg) {
  cerr << msg << endl;
  exit(1);
}

static void check(int rc, mmq_handle* h, const char* what) {
  if (rc) die(string("Error: ") + what + ": " + mmq_last_error(h));
}

/* "%g" of a double (== operator<< at the stream's default precision 6, what the reference writes).  General case:
 * std::to_chars, which the standard specifies to give printf's characters in the C locale (libstdc++: 2.5x faster than
 * snprintf).  The trace files hold 4e8 of them, so the common case gets a direct path (fmt_g6.h). */
static inline char* fmt_g(char (&buf)[40], double v) { return fmt_g6(buf, v); }

/* gzip text writer with the reference's stream formatting ("%g" == operator<< at precision 6) */
struct GzText {
  gzFile f = nullptr;
  string buf;
  explicit GzText(const string& path) {
    f = gzopen(path.c_str(), "wb");
    if (!f) die("Error: cannot open " + path + " for writing.");
    buf.reserve(1 << 20);
  }
  void put(const string& s) { buf += s; flush_if(); }
  void put(double v) {
    char t[40];
    buf.append(t, (size_t)(fmt_g(t, v) - t));
    flush_if();
  }
  void flush_if() { if (buf.size() > (1 << 20) - 64) flush(); }
  void flush() { if (!buf.empty()) { gzwrite(f, buf.data(), (unsigned)buf.size()); buf.clear(); } }
  ~GzText() { flush(); if (f) gzclose(f); }
};

/* the *.trace_gibbs.gz writer lives in trace_writer.h (shared with the test-support library) */
static void write_trace_gz(const string& path, const vector<string>& ids, const vector<char>& keep, const double* tr, int L) {
  const string err = mmq::write_trace_gz(path, ids, keep, tr, L);
  if (!err.empty()) die(err);
}

static void write_pcts(ostream& ofs, const double* v, size_t np, char last) {
  for (size_t i = 0; i < np; ++i) {
    ofs << v[i];
    ofs << (i == np - 1 ? last : ',');
  }
}

/* Rows of a table formatted by all host threads (each into a string stream with the file stream's
 * formatting state), written in order: the bytes are those of one loop over `ofs`. */
static void write_rows(ostream& ofs, int64_t rows, const function<void(ostream&, int64_t)>& row) {
  const int T = (int)max<int64_t>(1, min<int64_t>(min(32u, max(1u, thread::hardware_concurrency())), rows / 64));
  if (T == 1) { for (int64_t r = 0; r < rows; ++r) row(ofs, r); return; }
  vector<ostringstream> part((size_t)T);
  vector<thread> th;
  for (int t = 0; t < T; ++t) {
    part[(size_t)t].copyfmt(ofs);
    th.emplace_back([&, t] { for (int64_t r = rows * t / T; r < rows * (t + 1) / T; ++r) row(part[(size_t)t], r); });
  }
  for (auto& x : th) x.join();
  for (auto& p : part) { const string blk = p.str(); ofs.write(blk.data(), (streamsize)blk.size()); }
}

/* posterior sd of a count from its moments over S sweeps: sqrt((S sum c^2 - (sum c)^2) / (S (S - 1))), the numerator
 * exact in 128 bits (it can pass 2^64 long before the end of a chain) and the S - 1 of the sd column (src/sokal.cc:63) */
static double count_sd(int64_t S, uint64_t sum, uint64_t sumsq_lo, uint64_t sumsq_hi) {
  if (S < 2) return 0.0;
  const unsigned __int128 sq = ((unsigned __int128)sumsq_hi << 64) | sumsq_lo;
  const unsigned __int128 num = (unsigned __int128)(uint64_t)S * sq - (unsigned __int128)sum * sum;
  return sqrt((double)num / ((double)S * (double)(S - 1)));
}

struct Shard {
  int device = 0;
  int64_t row0 = 0, row1 = 0;
  mmq_handle* h = nullptr;
};

/* MMQ_TIMING=1: wall-clock of the host program's phases on stderr */
static void phase(const char* name) {
  static const bool on = getenv("MMQ_TIMING") != nullptr;
  static auto t_start = chrono::steady_clock::now();
  static auto t_last = t_start;
  if (!on) return;
  const auto now = chrono::steady_clock::now();
  fprintf(stderr, "[mmseq timing] %-28s %8.3f s  (+%.3f)\n", name, chrono::duration<double>(now - t_start).count(),
          chrono::duration<double>(now - t_last).count());
  t_last = now;
}

/* ---- command line (src/mmseq.cpp:183-296): one table of options, the reference's messages and exit codes ---- */
struct Options {
  double alpha = 0.1, beta = 0.1, epsilon = 0.1;
  int max_em_iter = 1000, gibbs_iter = 16384, trace_length = 1024, gibbs_ss = 16384 / 1024, seed = 1234;
  vector<double> percentiles{5.0, 25.0, 50.0, 75.0, 95.0};
  bool debug = false, notraces = false, counts = false;
  bool pool = false; /* -pool: the tables and -counts over the draws of all chains */
  bool tpm = false;  /* -tpm: the .tpm files */
  bool allelic = false; /* -allelic: the .allelic files */
  bool isocorr = false; /* -isocorr: the .isocorr file */
  int ngpus = 1;
  string batch;     /* -batch FILE: one "hits_file output_base" pair per line */
  int per_gpu = 4;  /* -per_gpu INT: samples in flight per GPU in batch mode */
  int chains = 1;   /* -chains INT: independent chains per sample */
  vector<string> positional;
};

[[noreturn]] static void usage_error(const string& msg) {
  if (!msg.empty()) cerr << msg << "\n";
  printUsage(cerr);
  exit(1);
}

#define MMQ_CHAINS 8 /* chains per sample: the limit of mmq_chain_diagnostics */

static bool is_power_of_two(int v) { return v > 0 && (v & (v - 1)) == 0; }

static void parse_percentiles(const string& list, vector<double>& out) {
  out.clear();
  size_t pos = 0;
  while (pos <= list.size()) {
    const size_t comma = list.find(',', pos);
    const string item = list.substr(pos, comma == string::npos ? string::npos : comma - pos);
    if (!item.empty()) {
      const double v = strtod(item.c_str(), NULL);
      if (!(v >= 0 && v <= 100)) { cerr << "Percentiles must be in (0,100)\n"; exit(1); }
      out.push_back(v);
    }
    if (comma == string::npos) break;
    pos = comma + 1;
  }
}

static Options parse_command_line(int argc, char** argv) {
  Options o;
  enum Kind { REAL, INT, TEXT, FLAG };
  struct Spec { const char* name; Kind kind; void* target; };
  string pct;
  const Spec specs[] = {
      {"-alpha", REAL, &o.alpha},         {"-beta", REAL, &o.beta},           {"-max_em_iter", INT, &o.max_em_iter},
      {"-epsilon", REAL, &o.epsilon},     {"-gibbs_iter", INT, &o.gibbs_iter}, {"-gibbs_ss", INT, &o.gibbs_ss},
      {"-seed", INT, &o.seed},            {"-percentiles", TEXT, &pct},       {"-gpus", INT, &o.ngpus},
      {"-batch", TEXT, &o.batch},         {"-per_gpu", INT, &o.per_gpu},      {"-notraces", FLAG, &o.notraces},
      {"-debug", FLAG, &o.debug},         {"-counts", FLAG, &o.counts},       {"-chains", INT, &o.chains},
      {"-pool", FLAG, &o.pool},           {"-tpm", FLAG, &o.tpm},            {"-allelic", FLAG, &o.allelic},
      {"-isocorr", FLAG, &o.isocorr},
  };
  /* options come first; what is left must be the mandatory arguments (none in batch mode) */
  int i = 1;
  for (; i < argc; ++i) {
    const string arg = argv[i];
    if (arg == "-h" || arg == "--help" || arg == "-help") { cerr << "Calculate mmseq expression estimates.\n"; usage_error(""); }
    if (arg == "-v" || arg == "--version" || arg == "-version") { cerr << "mmseq-" << QUOTE(VERSION) << endl; exit(1); }
    const Spec* hit = nullptr;
    for (const Spec& sp : specs) if (arg == sp.name) { hit = &sp; break; }
    if (!hit) break;
    if (hit->kind == FLAG) { *static_cast<bool*>(hit->target) = true; continue; }
    if (i + 1 >= argc) usage_error("Error: option " + arg + " needs a value.");
    const char* val = argv[++i];
    if (hit->kind == REAL) *static_cast<double*>(hit->target) = strtod(val, NULL);
    else if (hit->kind == INT) *static_cast<int*>(hit->target) = atoi(val);
    else *static_cast<string*>(hit->target) = val;
    if (hit->target == &pct) parse_percentiles(pct, o.percentiles);
  }
  for (; i < argc; ++i) o.positional.push_back(argv[i]);
  const size_t want = o.batch.empty() ? 2 : 0;
  if (o.positional.size() != want) {
    if (!o.positional.empty() && o.positional[0][0] == '-') usage_error("Error: unrecognised option " + o.positional[0] + ".");
    usage_error("Error: mandatory arguments missing.");
  }
  /* src/mmseq.cpp:278-296 (a zero -gibbs_ss would divide by zero there; rejected here) */
  if (o.gibbs_ss == 0 || o.gibbs_iter % o.gibbs_ss != 0) usage_error("Error: gibbs_iter must be divisible by gibbs_ss.");
  o.gibbs_ss = o.gibbs_iter / o.trace_length; /* forced, as the reference does (:284) */
  if (o.gibbs_iter <= 0 || o.trace_length <= 0)
    usage_error("Error: no. of iteratons or trace length <= 0. Possible integer overflow - is gibbs_iter too high?");
  if (!is_power_of_two(o.trace_length)) usage_error("Error: gibbs_iter/gibbs_ss must be a power of 2.");
  if (o.gibbs_ss <= 0) usage_error("Error: gibbs_iter must be at least " + to_string(o.trace_length) + " (the trace length).");
  if (o.ngpus < 1) die("Error: -gpus must be >= 1.");
  if (o.per_gpu < 1) die("Error: -per_gpu must be >= 1.");
  if (o.chains < 1 || o.chains > MMQ_CHAINS) die("Error: -chains must be in 1.." + to_string(MMQ_CHAINS) + ".");
  if (o.pool && o.chains < 2) die("Error: -pool needs -chains 2 or more.");
  return o;
}

/* -allelic: the haplotype pairs of a header (include/mmq.h, allelic fraction): header transcripts STEM_A and STEM_B of one
 * gene, with or without hits, in the header order of the _A copy.  `lonely` counts the transcripts named *_A / *_B whose
 * partner is missing or in another gene. */
struct HaploPairs {
  vector<int32_t> a, b; /* header indices of the two copies of every pair */
  vector<string> stem;  /* the pair's feature id */
  vector<char> paired;  /* per header transcript */
  int64_t lonely = 0;
};

static HaploPairs find_pairs(const mmq::HitsHeader& hdr) {
  HaploPairs hp;
  const int64_t T = (int64_t)hdr.names.size();
  unordered_map<string, int32_t> index;
  for (int64_t t = 0; t < T; ++t) index.emplace(hdr.names[(size_t)t], (int32_t)t);
  auto named = [&](int64_t t, char copy) {
    const string& s = hdr.names[(size_t)t];
    return s.size() >= 2 && s[s.size() - 2] == '_' && s.back() == copy;
  };
  hp.paired.assign((size_t)T, 0);
  for (int64_t t = 0; t < T; ++t) {
    if (!named(t, 'A')) continue;
    const string& s = hdr.names[(size_t)t];
    const string stem = s.substr(0, s.size() - 2);
    const auto it = index.find(stem + "_B");
    if (it == index.end() || hdr.gene_of[(size_t)it->second] != hdr.gene_of[(size_t)t]) continue;
    hp.a.push_back((int32_t)t);
    hp.b.push_back(it->second);
    hp.stem.push_back(stem);
    hp.paired[(size_t)t] = hp.paired[(size_t)it->second] = 1;
  }
  for (int64_t t = 0; t < T; ++t) hp.lonely += (named(t, 'A') || named(t, 'B')) && !hp.paired[(size_t)t];
  return hp;
}

/* One sample: hits file in, the nine output files out (src/mmseq.cpp:312-1694).  first_device: the GPU of a
 * single-GPU run, or the first of o.ngpus consecutive devices.  Messages go to out / err (the terminal for a
 * single sample, the sample's log in batch mode). */
static void run_sample(const Options& o, const string& hits_file, const string& output_base, int first_device, ostream& out, ostream& err) {
  const double alpha = o.alpha, beta = o.beta, epsilon = o.epsilon;
  const int max_em_iter = o.max_em_iter, gibbs_iter = o.gibbs_iter, trace_length = o.trace_length, gibbs_ss = o.gibbs_ss, seed = o.seed;
  const vector<double>& percentiles = o.percentiles;
  const bool debug = o.debug, notraces = o.notraces;
  /* with several chains every chain runs whole on one GPU: chain c (0-based) on first_device + c mod o.ngpus */
  const int nchains = o.chains;
  const int ngpus = nchains > 1 ? 1 : o.ngpus; /* shards of chain 1 (the chain of the tables) */
  const int ndev = nchains > 1 ? min(o.ngpus, nchains) : o.ngpus;
  auto chain_device = [&](int c) { return first_device + c % o.ngpus; };

  /* the CUDA contexts come up (1-2 s) while the hits file is being parsed */
  thread warmup([ndev, first_device] { for (int g = 0; g < ndev; ++g) mmq_warmup(first_device + g); });

  /* ---- load: header + records -> hit classes (src/hitsio.cpp, src/mmseq.cpp:312-441).  A file with per-hit
   * weights (schema 2) cannot be collapsed: two fragments with the same transcript set differ in their weights.
   * It is loaded one row per fragment, grouped by set size and set (the segment kernel's layout), and the loader
   * also returns the distinct sets, from which .k, .M and the debug files are written as for an unweighted file. */
  mmq::HitsHeader hdr;
  mmq::HitClasses cls;
  {
    string err;
    if (mmq::load_hits_file(hits_file, mmq::LAYOUT_COLLAPSED, hdr, cls, err, mmq::LAYOUT_PER_FRAGMENT_BY_LENGTH)) { warmup.join(); die(err); }
  }
  warmup.join();
  const bool weighted = hdr.schema == 2;
  if (cls.first_zero_weight_record >= 0) /* its likelihood term is log 0: EM would turn mu into NaN */
    die("Error: fragment record " + to_string(cls.first_zero_weight_record + 1) + " of \"" + hits_file +
        "\" has per-hit weights that are all zero: its likelihood is zero whatever the abundances.");
  HaploPairs hp;
  if (o.allelic) {
    hp = find_pairs(hdr);
    if (hp.a.empty()) die("Error: -allelic found no pair of transcripts STEM_A / STEM_B in one gene.");
    if (hp.lonely > 0) err << "Note: -allelic: " << hp.lonely << " transcripts named *_A / *_B have no partner in their gene." << endl;
  }
  out << "Running mmseq with parameters:\n"
       << "  alpha:         " << alpha << endl
       << "  beta:          " << beta << endl
       << "  max_em_iter:   " << max_em_iter << endl
       << "  epsilon:       " << epsilon << endl
       << "  gibbs_iter:    " << gibbs_iter << endl
       << "  gibbs_ss:      " << gibbs_ss << endl
       << "  seed[0]:       " << seed << endl
       << "  debug:         " << debug << endl
       << "  threads:       " << o.ngpus << " GPU(s)" << endl;
  if (nchains > 1) out << "  chains:        " << nchains << endl;
  if (o.pool) out << "  pooled:        yes" << endl;
  const int64_t T = (int64_t)hdr.names.size();
  const int64_t n = cls.n, m = cls.m; /* m: rows on the GPUs (sets, or fragments of a weighted file) */
  const int64_t N = cls.N;
  const int64_t G = (int64_t)hdr.gene_names.size(), I = (int64_t)hdr.identical.size();
  const int L = trace_length;
  /* the distinct transcript sets in first-appearance order, with their fragment counts */
  const vector<int64_t>& set_ptr = weighted ? cls.set_ptr : cls.row_ptr;
  const vector<int32_t>& set_col = weighted ? cls.set_col : cls.col;
  const vector<int32_t>& set_k = weighted ? cls.set_k : cls.k;
  const int64_t n_sets = weighted ? cls.n_classes : m;
  phase("hits file loaded");
  out << "Found " << n << " transcripts in " << n_sets << " transcript combinations.\r" << endl;
  if (n == 0 || n_sets == 0) die("Error: no mapped fragments in the hits file.");

  vector<double> l;
  {
    string err;
    if (mmq::scaled_lengths(hdr, cls, l, err)) die(err);
  }

  /* ---- the groups in column space: each observed transcript's identical set (-1: none) and gene, whether that gene
   * has other isoforms, and the observed members of every identical set and gene (CSR, in header order) */
  vector<int32_t> ident_of((size_t)n, -1), gene_of((size_t)n);
  vector<uint8_t> multi((size_t)n);
  vector<int64_t> iptr{0}, gptr{0};
  vector<int32_t> imem, gmem;
  for (int64_t s = 0; s < I; ++s) {
    for (int32_t hidx : hdr.identical[(size_t)s]) { const int32_t c = cls.hdr2col[(size_t)hidx]; if (c >= 0) { ident_of[(size_t)c] = (int32_t)s; imem.push_back(c); } }
    iptr.push_back((int64_t)imem.size());
  }
  for (int64_t g = 0; g < G; ++g) {
    for (int32_t hidx : hdr.gene_members[(size_t)g]) { const int32_t c = cls.hdr2col[(size_t)hidx]; if (c >= 0) gmem.push_back(c); }
    gptr.push_back((int64_t)gmem.size());
  }
  for (int64_t t = 0; t < n; ++t) {
    gene_of[(size_t)t] = hdr.gene_of[(size_t)cls.col2hdr[(size_t)t]];
    multi[(size_t)t] = hdr.gene_members[(size_t)gene_of[(size_t)t]].size() > 1;
  }

  /* ---- shards.  The library orders the classes of a shard itself (class plan, mmq_cls.cu), so the
   * host hands them over as they are: one GPU takes the loader's arrays in place; several GPUs take
   * every ngpus-th class (first-appearance order is unrelated to the cost of a class, so the deal is
   * an equal mix).  The Philox counter of a class is its first-appearance index either way
   * (mmq_problem.class_id): the chain does not depend on the number of GPUs.
   * The fragment rows of a weighted file (k = NULL, where explicit class ids are not accepted) are cut
   * into contiguous ranges with equal numbers of hits instead; the Philox counter of a row is its index
   * in the whole row order (mmq_problem.class_id_base), so again the chain does not depend on the cut. */
  vector<Shard> shards((size_t)ngpus);
  vector<vector<int64_t>> shard_rp((size_t)ngpus), shard_id((size_t)ngpus);
  vector<vector<int32_t>> shard_col((size_t)ngpus), shard_k((size_t)ngpus);
  mmq_problem whole; /* the problem of the unsharded chain 1, for chains 2.. (-chains) */
  for (int g = 0; g < ngpus; ++g) {
    Shard& S = shards[(size_t)g];
    S.device = first_device + g;
    mmq_problem p;
    memset(&p, 0, sizeof p);
    p.n = n;
    if (weighted) {
      const int64_t nnz = cls.row_ptr[(size_t)m];
      auto row_at = [&](int64_t gi) { /* first row whose hits start at or after gi/ngpus of all hits */
        if (gi == ngpus) return m;
        return (int64_t)(lower_bound(cls.row_ptr.begin(), cls.row_ptr.begin() + m, nnz * gi / ngpus) - cls.row_ptr.begin());
      };
      const int64_t r0 = row_at(g), r1 = row_at(g + 1), q0 = cls.row_ptr[(size_t)r0];
      auto& rp = shard_rp[(size_t)g];
      rp.resize((size_t)(r1 - r0 + 1));
      for (int64_t i = r0; i <= r1; ++i) rp[(size_t)(i - r0)] = cls.row_ptr[(size_t)i] - q0;
      p.m = r1 - r0; p.nnz = rp.back();
      p.row_ptr = rp.data();
      p.col = cls.col.data() + q0;
      p.weight = cls.w.data() + q0;
      p.k = nullptr;
      p.class_id = nullptr;
      p.class_id_base = r0;
    } else if (ngpus == 1) {
      p.m = m; p.nnz = cls.row_ptr[(size_t)m];
      p.row_ptr = cls.row_ptr.data();
      p.col = cls.col.data();
      p.k = cls.k.data();
      p.class_id = nullptr; /* class i is row i */
    } else {
      auto& rp = shard_rp[(size_t)g];
      auto& id = shard_id[(size_t)g];
      auto& cc = shard_col[(size_t)g];
      auto& kk = shard_k[(size_t)g];
      rp.push_back(0);
      for (int64_t i = g; i < m; i += ngpus) {
        id.push_back(i);
        kk.push_back(cls.k[(size_t)i]);
        for (int64_t q = cls.row_ptr[(size_t)i]; q < cls.row_ptr[(size_t)i + 1]; ++q) cc.push_back(cls.col[(size_t)q]);
        rp.push_back((int64_t)cc.size());
      }
      p.m = (int64_t)id.size(); p.nnz = rp.back();
      p.row_ptr = rp.data();
      p.col = cc.data();
      p.k = kk.data();
      p.class_id = id.data();
    }
    S.row0 = 0; S.row1 = p.m;
    p.len = l.data();
    p.alpha = alpha; p.beta = beta;
    if (g == 0) whole = p;
    int rc = mmq_create(&p, S.device, &S.h);
    if (rc) die(string("Error: mmq_create: ") + mmq_last_error(nullptr));
  }
  auto on_all = [&](auto fn) { /* run fn(shard index) on every shard concurrently (collectives need all ranks) */
    if (ngpus == 1) { fn(0); return; }
    vector<thread> th;
    for (int g = 0; g < ngpus; ++g) th.emplace_back([&, g] { fn(g); });
    for (auto& t : th) t.join();
  };
  if (ngpus > 1) {
    char uid[128];
    if (mmq_comm_id(uid)) die(string("Error: mmq_comm_id: ") + mmq_last_error(nullptr));
    on_all([&](int g) { check(mmq_comm_init(shards[(size_t)g].h, uid, g, ngpus), shards[(size_t)g].h, "mmq_comm_init"); });
  }
  if (ngpus > 1) { /* Gibbs: all-reduce + Gamma update fused over NVLink peer memory (no NCCL call per sweep) */
    vector<mmq_handle*> hs;
    for (auto& S : shards) hs.push_back(S.h);
    if (mmq_p2p_attach_local(hs.data(), ngpus)) err << "Note: peer access unavailable (" << mmq_last_error(hs[0]) << "); using NCCL for the count exchange." << endl;
  }
  mmq_handle* H0 = shards[0].h;

  /* ---- initial mu, unique hits (src/mmseq.cpp:610-638) */
  vector<int32_t> unique_hits((size_t)n);
  on_all([&](int g) { check(mmq_init_mu(shards[(size_t)g].h, g == 0 ? unique_hits.data() : nullptr), shards[(size_t)g].h, "mmq_init_mu"); });

  /* ---- unique hits of identical sets and genes (src/mmseq.cpp:643-680, src/uh.cpp) */
  vector<int32_t> identical_unique_hits((size_t)I, 0), gene_unique_hits((size_t)G, 0);
  {
    phase("shards on the GPUs");
    err << "Counting unique hits to sets of identical transcripts...";
    if (I > 0) on_all([&](int g) { check(mmq_unique_hits_sets(shards[(size_t)g].h, ident_of.data(), I, g == 0 ? identical_unique_hits.data() : vector<int32_t>((size_t)I).data()), shards[(size_t)g].h, "mmq_unique_hits_sets"); });
    err << "done." << endl;
    err << "Counting unique hits to genes...";
    on_all([&](int g) { check(mmq_unique_hits_sets(shards[(size_t)g].h, gene_of.data(), G, g == 0 ? gene_unique_hits.data() : vector<int32_t>((size_t)G).data()), shards[(size_t)g].h, "mmq_unique_hits_sets"); });
    err << "done." << endl;
  }

  /* ---- .k and .M (src/mmseq.cpp:682-695): one integer per line / "row<TAB>col" per nonzero.  The
   * reference streams them through operator<< with endl; the same bytes are formatted here by all
   * host threads into blocks that are written in order. */
  {
    auto put_int = [](string& out, int64_t v) {
      char buf[24];
      int len = 0;
      if (v < 0) { out.push_back('-'); v = -v; }
      do { buf[len++] = (char)('0' + v % 10); v /= 10; } while (v);
      while (len) out.push_back(buf[--len]);
    };
    auto write_blocks = [&](const string& path, const string& head, int64_t rows, const function<void(string&, int64_t)>& row) {
      FILE* f = fopen(path.c_str(), "wb");
      if (!f) die("Error: cannot write " + path);
      if (!head.empty()) fwrite(head.data(), 1, head.size(), f);
      const int nt = (int)max<int64_t>(1, min<int64_t>(min(32u, max(1u, thread::hardware_concurrency())), rows / 65536));
      vector<string> part((size_t)nt);
      vector<thread> th;
      for (int t = 0; t < nt; ++t)
        th.emplace_back([&, t] {
          string& out = part[(size_t)t];
          const int64_t a = rows * t / nt, b = rows * (t + 1) / nt;
          for (int64_t i = a; i < b; ++i) row(out, i);
        });
      for (auto& x : th) x.join();
      for (const string& blk : part) fwrite(blk.data(), 1, blk.size(), f);
      fclose(f);
    };
    write_blocks(output_base + ".k", "", n_sets, [&](string& out, int64_t i) { put_int(out, set_k[(size_t)i]); out.push_back('\n'); });
    string head = "#";
    for (int64_t t = 0; t < n; t++) { head += "\t"; head += hdr.names[(size_t)cls.col2hdr[(size_t)t]]; }
    head += "\n";
    write_blocks(output_base + ".M", head, n_sets, [&](string& out, int64_t i) {
      for (int64_t q = set_ptr[(size_t)i]; q < set_ptr[(size_t)i + 1]; ++q) {
        put_int(out, i); out.push_back('\t'); put_int(out, set_col[(size_t)q]); out.push_back('\n');
      }
    });
  }
  ofstream ofs;

  phase(".k and .M written");
  if (debug) { /* src/mmseq.cpp:697-731 */
    vector<vector<int>> counts_shared((size_t)n, vector<int>(100, 0));
    for (int64_t i = 0; i < n_sets; ++i) {
      const int64_t d = set_ptr[(size_t)i + 1] - set_ptr[(size_t)i];
      for (int64_t q = set_ptr[(size_t)i]; q < set_ptr[(size_t)i + 1]; ++q)
        counts_shared[(size_t)set_col[(size_t)q]][(size_t)min<int64_t>(d, 100) - 1] += set_k[(size_t)i];
    }
    ofs.open((output_base + ".sharedcounts").c_str());
    for (int64_t hI = 0; hI < T; ++hI) {
      ofs << hdr.names[(size_t)hI] << "\t";
      const int32_t c = cls.hdr2col[(size_t)hI];
      for (int i = 0; i < 100; i++) { if (c >= 0) ofs << counts_shared[(size_t)c][(size_t)i] << "\t"; else ofs << "0\t"; }
      ofs << endl;
    }
    ofs.close(); ofs.clear();
    ofs.open((output_base + ".doublehits").c_str());
    for (int64_t i = 0; i < n; i++) ofs << cls.doublehits[(size_t)i] << endl;
    ofs.close(); ofs.clear();
    /* Mt rows (transcripts) equal to the previous row are listed in .dupIDs, the others dumped */
    vector<vector<int32_t>> Mt((size_t)n);
    for (int64_t i = 0; i < n_sets; ++i)
      for (int64_t q = set_ptr[(size_t)i]; q < set_ptr[(size_t)i + 1]; ++q) Mt[(size_t)set_col[(size_t)q]].push_back((int32_t)i);
    ofs.open((output_base + ".Mt-nodups").c_str());
    ofstream ofs2((output_base + ".dupIDs").c_str());
    for (int64_t t = 0; t < n; ++t) {
      if (t > 0 && Mt[(size_t)t] == Mt[(size_t)t - 1]) ofs2 << hdr.names[(size_t)cls.col2hdr[(size_t)t]] << endl;
      else for (int32_t i : Mt[(size_t)t]) ofs << t << "\t" << i << endl;
    }
    ofs.close(); ofs.clear();
    ofs2.close();
  }

  /* ---- EM (src/mmseq.cpp:741-820) */
  vector<double> mu_em((size_t)n);
  {
    out.precision(5);
    out.setf(ios::fixed, ios::floatfield);
    auto t0 = chrono::steady_clock::now();
    int iters = 0;
    double loglik = 0, llr = 0;
    if (!debug) {
      vector<int> it_g((size_t)ngpus); vector<double> ll_g((size_t)ngpus), llr_g((size_t)ngpus);
      on_all([&](int g) { check(mmq_em(shards[(size_t)g].h, max_em_iter, epsilon, &it_g[(size_t)g], &ll_g[(size_t)g], &llr_g[(size_t)g]), shards[(size_t)g].h, "mmq_em"); });
      iters = it_g[0]; loglik = ll_g[0]; llr = llr_g[0];
      if (iters > 0) out << "EM iteration " << iters - 1 << ", log likelihood ratio: " << llr << "            \r";
    } else { /* one iteration per call so that every mu can be dumped (.trace_em.gz, :764-768) */
      GzText g(output_base + ".trace_em.gz");
      for (int64_t t = 0; t < n; t++) { g.put(hdr.names[(size_t)cls.col2hdr[(size_t)t]]); g.put(" "); }
      g.put("\n");
      vector<double> mu((size_t)n);
      vector<double> ll_g((size_t)ngpus);
      on_all([&](int gi) { check(mmq_loglik(shards[(size_t)gi].h, &ll_g[(size_t)gi]), shards[(size_t)gi].h, "mmq_loglik"); });
      loglik = ll_g[0];
      llr = epsilon + 1;
      while (iters < max_em_iter && llr > epsilon) {
        out << "EM iteration " << iters << flush;
        check(mmq_get_mu(H0, mu.data()), H0, "mmq_get_mu");
        for (int64_t t = 0; t < n; t++) { g.put(mu[(size_t)t]); g.put(" "); }
        g.put("\n");
        vector<double> l2((size_t)ngpus);
        on_all([&](int gi) { check(mmq_em(shards[(size_t)gi].h, 1, -numeric_limits<double>::infinity(), nullptr, &l2[(size_t)gi], nullptr), shards[(size_t)gi].h, "mmq_em"); });
        llr = l2[0] - loglik;
        loglik = l2[0];
        out << ", log likelihood ratio: " << llr << "            \r";
        iters++;
      }
    }
    out << endl;
    out.unsetf(ios::floatfield);
    out.precision(6);
    const double sec = chrono::duration<double>(chrono::steady_clock::now() - t0).count();
    err << "EM: " << iters << " iterations in " << sec << " s" << endl;
    check(mmq_get_mu(H0, mu_em.data()), H0, "mmq_get_mu");
  }

  /* ---- -counts: EM expected counts at mu_em (one E-step, all shards), and from here on every Gibbs sweep adds its
   * counts of transcripts, identical sets and genes into the accumulators of every shard (with -pool, of every chain) */
  vector<double> em_count;
  if (o.counts) {
    em_count.resize((size_t)n);
    vector<vector<double>> other((size_t)ngpus);
    on_all([&](int g) {
      mmq_handle* h = shards[(size_t)g].h;
      if (g > 0) other[(size_t)g].resize((size_t)n);
      check(mmq_expected_counts(h, g == 0 ? em_count.data() : other[(size_t)g].data()), h, "mmq_expected_counts");
    });
    on_all([&](int g) {
      mmq_handle* h = shards[(size_t)g].h;
      check(mmq_count_moments_begin(h, ident_of.data(), I, gene_of.data(), G), h, "mmq_count_moments_begin");
    });
  }

  /* ---- -chains: chains 2..C, each whole on its GPU from mu_em with its own seed, concurrently with chain 1 */
  vector<mmq_handle*> chain_h((size_t)nchains, nullptr);
  chain_h[0] = H0;
  vector<thread> chain_th;
  for (int c = 1; c < nchains; ++c)
    chain_th.emplace_back([&, c] {
      mmq_handle*& h = chain_h[(size_t)c];
      if (mmq_create(&whole, chain_device(c), &h)) die(string("Error: mmq_create: ") + mmq_last_error(nullptr));
      check(mmq_set_mu(h, mu_em.data()), h, "mmq_set_mu");
      if (o.counts && o.pool) check(mmq_count_moments_begin(h, ident_of.data(), I, gene_of.data(), G), h, "mmq_count_moments_begin");
      check(mmq_gibbs(h, mmq_chain_seed((uint32_t)seed, c), 0, gibbs_iter, gibbs_ss, L, MMQ_GIBBS_DEFAULT), h, "mmq_gibbs");
      check(mmq_synchronize(h), h, "mmq_synchronize");
    });

  /* ---- Gibbs (src/mmseq.cpp:822-918) */
  {
    auto t0 = chrono::steady_clock::now();
    out << "Gibbs iteration " << gibbs_iter - 1 << "       \r";
    on_all([&](int g) {
      mmq_handle* h = shards[(size_t)g].h;
      check(mmq_gibbs(h, (uint32_t)seed, 0, gibbs_iter, gibbs_ss, L, MMQ_GIBBS_DEFAULT), h, "mmq_gibbs");
      check(mmq_synchronize(h), h, "mmq_synchronize");
    });
    out << endl;
    const double sec = chrono::duration<double>(chrono::steady_clock::now() - t0).count();
    err << "Gibbs: " << gibbs_iter << " sweeps in " << sec << " s (" << gibbs_iter / sec << " sweeps/s, " << (double)m * gibbs_iter / sec
         << (weighted ? " fragment allocations/s)" : " hit-class allocations/s)") << endl;
  }
  for (auto& t : chain_th) t.join();

  phase("EM + Gibbs");
  out << "Amalgamating transcripts and calculating summary statistics..." << flush;

  /* the Gamma prior's rate for a feature of effective length len, and the closed-form log_mu of a feature without
   * hits (:971-978, :1372-1395) */
  auto prior_rate = [&](double len) { return beta + len * (double)N / 1000000000.0; };
  const double digalpha = mmq_host_digamma(alpha);
  const double sqrtpolygalpha = sqrt(mmq_host_trigamma(alpha));
  auto closed_log_mu = [&](double len) { return digalpha - log(prior_rate(len)); };

  /* ---- prior-simulated traces for isoforms without hits (src/mmseq.cpp:971-978), on the device */
  vector<int64_t> unobs;           /* header indices */
  vector<int64_t> unobs_slot((size_t)T, -1);
  for (int64_t hI = 0; hI < T; ++hI)
    if (cls.hdr2col[(size_t)hI] < 0) { unobs_slot[(size_t)hI] = (int64_t)unobs.size(); unobs.push_back(hI); }
  const int64_t U = (int64_t)unobs.size();
  vector<double> simu((size_t)U * (size_t)L);
  vector<double> rate((size_t)U);
  for (int64_t u = 0; u < U; ++u) rate[(size_t)u] = prior_rate(hdr.efflen[(size_t)unobs[(size_t)u]]);
  if (U > 0 && mmq_prior_draws(shards[0].device, U, unobs.data(), rate.data(), alpha, (uint32_t)seed, L, simu.data()))
    die(string("Error: mmq_prior_draws: ") + mmq_last_error(nullptr));

  /* ---- groups: identical sets (:938-954) and genes (:959-982); with -chains, on every chain, the gene extras from
   * each chain's own prior draws (built one chain at a time in one host buffer; kept under -pool for the hit-less
   * isoforms' pooled columns) */
  vector<vector<double>> simu_pool((size_t)nchains); /* [c >= 1]: chain c's prior draws, under -pool */
  {
    vector<double> extra((size_t)G * (size_t)L), simu_c;
    for (int c = 0; c < nchains; ++c) {
      mmq_handle* h = chain_h[(size_t)c];
      const double* sim = simu.data();
      if (c > 0) {
        vector<double>& dst = o.pool ? simu_pool[(size_t)c] : simu_c;
        dst.resize(simu.size());
        if (U > 0 && mmq_prior_draws(chain_device(c), U, unobs.data(), rate.data(), alpha, mmq_chain_seed((uint32_t)seed, c), L, dst.data()))
          die(string("Error: mmq_prior_draws: ") + mmq_last_error(nullptr));
        sim = dst.data();
      }
      fill(extra.begin(), extra.end(), 0.0);
      for (int64_t g = 0; g < G; ++g)
        for (int32_t hidx : hdr.gene_members[(size_t)g])
          if (cls.hdr2col[(size_t)hidx] < 0) {
            const double* sv = sim + (size_t)unobs_slot[(size_t)hidx] * (size_t)L;
            for (int i = 0; i < L; ++i) extra[(size_t)g * (size_t)L + (size_t)i] += sv[i];
          }
      check(mmq_set_groups(h, MMQ_GROUP_IDENTICAL, I, iptr.data(), imem.data(), nullptr), h, "mmq_set_groups");
      check(mmq_set_groups(h, MMQ_GROUP_GENE, G, gptr.data(), gmem.data(), extra.data()), h, "mmq_set_groups");
    }
  }

  /* ---- the three levels of every per-feature output, in the order of the C ABI's `which`: transcripts (a table row
   * per header transcript, a device row per observed one), identical sets and genes (one row per group in both) */
  struct Summ { vector<double> mean, sd, mcse, iact, pct; }; /* the .mmseq columns of every device row */
  Summ summ[3];
  vector<char> ident_obs((size_t)I); /* the identical sets' `observed`: chain 1's log mean is finite (:1567) */
  /* an identical set's columns follow its members named as the last member (:1560-1565); "+" follows the others */
  auto named_last = [&](const vector<int32_t>& mem, size_t j) { return hdr.names[(size_t)mem[j]].compare(hdr.names[(size_t)mem.back()]) == 0; };
  auto identical_id = [&](int64_t s) {
    const auto& mem = hdr.identical[(size_t)s];
    string id;
    for (size_t j = 0; j < mem.size(); ++j) { id += hdr.names[(size_t)mem[j]]; if (!named_last(mem, j)) id += "+"; }
    return id;
  };
  struct Level {
    const char* suffix;         /* of the level's output files */
    const char* name;
    int which;
    int64_t rows, dev_rows;     /* table rows, device rows */
    const vector<int64_t>* ptr; /* groups: the observed members of each (iptr / imem, gptr / gmem) */
    const vector<int32_t>* mem;
    function<string(int64_t)> id;       /* table row -> feature id */
    function<int64_t(int64_t)> dev_row; /* table row -> device row, -1 for a transcript without hits */
    function<bool(int64_t)> observed;   /* device row -> the `observed` column of the .mmseq and .convergence tables */
    function<pair<double, double>(int64_t)> unobserved; /* table row -> log_mu and sd of a row that is not observed */
    bool has_hits(int64_t q) const { return !ptr || (*ptr)[(size_t)q + 1] > (*ptr)[(size_t)q]; }
    double sum(int64_t q, const vector<double>& x) const { /* a group's: its members' in header order */
      if (!ptr) return x[(size_t)q];
      double s = 0.0;
      for (int64_t k = (*ptr)[(size_t)q]; k < (*ptr)[(size_t)q + 1]; ++k) s += x[(size_t)(*mem)[(size_t)k]];
      return s;
    }
  };
  auto same_row = [](int64_t r) { return r; };
  const Level levels[3] = {
      {"", "transcripts", 0, T, n, nullptr, nullptr, [&](int64_t hI) { return hdr.names[(size_t)hI]; },
       [&](int64_t hI) { return (int64_t)cls.hdr2col[(size_t)hI]; }, [](int64_t) { return true; },
       [&](int64_t hI) { return make_pair(closed_log_mu(hdr.efflen[(size_t)hI]), sqrtpolygalpha); }},
      {".identical", "identical sets", 1, I, I, &iptr, &imem, identical_id, same_row, [&](int64_t s) { return ident_obs[(size_t)s] != 0; },
       [&](int64_t s) {
         const auto& mem = hdr.identical[(size_t)s];
         size_t j = 0;
         while (!named_last(mem, j)) ++j;
         return make_pair(log(mem.size()) + digalpha - log(prior_rate(hdr.efflen[(size_t)mem[j]])), sqrtpolygalpha);
       }},
      {".gene", "genes", 2, G, G, &gptr, &gmem, [&](int64_t g) { return hdr.gene_names[(size_t)g]; }, same_row,
       [&](int64_t g) { return gptr[(size_t)g + 1] > gptr[(size_t)g]; },
       [&](int64_t g) { return make_pair(summ[2].mean[(size_t)g], summ[2].sd[(size_t)g]); }}, /* chain 1's, as the reference */
  };

  /* ---- -isocorr: the isoform pairs of every gene (include/mmq.h, isoform pairs): a gene's observed members in the CSR
   * order of gptr / gmem, m_0 .. m_{k-1}, and every (a, b) with a < b, a-major; genes in .gene.mmseq order.  iso_gene /
   * iso_local: the gene and local index a of every observed isoform of a gene with two or more, else -1; pair_gene /
   * pair_a / pair_b: the gene and the two local indices of every pair. */
  vector<int32_t> iso_gene, iso_local, pair_gene, pair_a, pair_b;
  vector<int64_t> pair_base;
  if (o.isocorr) {
    iso_gene.assign((size_t)n, -1);
    iso_local.assign((size_t)n, -1);
    pair_base.resize((size_t)G);
    for (int64_t g = 0; g < G; ++g) {
      pair_base[(size_t)g] = (int64_t)pair_gene.size();
      const int64_t b = gptr[(size_t)g], k = gptr[(size_t)g + 1] - b;
      for (int64_t a = 0; a < k && k >= 2; ++a) {
        iso_gene[(size_t)gmem[(size_t)(b + a)]] = (int32_t)g;
        iso_local[(size_t)gmem[(size_t)(b + a)]] = (int32_t)a;
        for (int64_t c = a + 1; c < k; ++c) { pair_gene.push_back((int32_t)g); pair_a.push_back((int32_t)a); pair_b.push_back((int32_t)c); }
      }
    }
  }

  /* ---- the two levels of -allelic: haplotype pairs (a row per pair) and genes (a row per gene of .gene.mmseq, its A side
   * the _A copies of the pairs inside it, its B side their _B copies, in pair order).  Members are in column space: an
   * observed copy is its column, a hit-less copy n + j, j its row among the prior rows (the hit-less paired copies in
   * header order).  unit_of / side: the unit of every observed copy (-1: none) and its side (0 A, 1 B). */
  struct AlleleLevel {
    const char* suffix; /* of the level's .allelic file */
    int64_t rows;
    function<string(int64_t)> id;
    vector<int64_t> npairs, a_ptr{0}, b_ptr{0};
    vector<int32_t> a_mem, b_mem, unit_of;
    vector<uint8_t> side;
    int64_t n_obs; /* member ids below it have hits */
    bool observed(int64_t u) const { /* a member with hits on either side */
      for (int64_t q = a_ptr[(size_t)u]; q < a_ptr[(size_t)u + 1]; ++q) if (a_mem[(size_t)q] < n_obs) return true;
      for (int64_t q = b_ptr[(size_t)u]; q < b_ptr[(size_t)u + 1]; ++q) if (b_mem[(size_t)q] < n_obs) return true;
      return false;
    }
  };
  vector<AlleleLevel> allele_levels;
  vector<int32_t> prior_hdr; /* header index of prior row j */
  if (o.allelic) {
    vector<int32_t> col_of((size_t)T);
    for (int64_t hI = 0; hI < T; ++hI) {
      col_of[(size_t)hI] = cls.hdr2col[(size_t)hI];
      if (hp.paired[(size_t)hI] && col_of[(size_t)hI] < 0) { col_of[(size_t)hI] = (int32_t)(n + (int64_t)prior_hdr.size()); prior_hdr.push_back((int32_t)hI); }
    }
    vector<vector<int32_t>> by_gene((size_t)G);
    const int64_t P = (int64_t)hp.a.size();
    for (int64_t p = 0; p < P; ++p) by_gene[(size_t)hdr.gene_of[(size_t)hp.a[(size_t)p]]].push_back((int32_t)p);
    allele_levels = {{"", P, [&](int64_t p) { return hp.stem[(size_t)p]; }}, {".gene", G, [&](int64_t g) { return hdr.gene_names[(size_t)g]; }}};
    for (int lvl = 0; lvl < 2; ++lvl) {
      AlleleLevel& al = allele_levels[(size_t)lvl];
      al.n_obs = n;
      al.unit_of.assign((size_t)n, -1);
      al.side.assign((size_t)n, 0);
      for (int64_t u = 0; u < al.rows; ++u) {
        const vector<int32_t> one{(int32_t)u};
        const vector<int32_t>& ps = lvl == 0 ? one : by_gene[(size_t)u];
        for (int32_t p : ps)
          for (int sd = 0; sd < 2; ++sd) {
            const int32_t c = col_of[(size_t)(sd ? hp.b : hp.a)[(size_t)p]];
            (sd ? al.b_mem : al.a_mem).push_back(c);
            if (c < n) { al.unit_of[(size_t)c] = (int32_t)u; al.side[(size_t)c] = (uint8_t)sd; }
          }
        al.npairs.push_back((int64_t)ps.size());
        al.a_ptr.push_back((int64_t)al.a_mem.size());
        al.b_ptr.push_back((int64_t)al.b_mem.size());
      }
    }
  }

  /* ---- summaries on the device: chain 1's (sd, mcse, iact: :1308-1363).  With -pool the observed rows come from
   * mmq_pooled_summaries over the draws of all chains, `draws` of them per feature, with the percentile rule of :1113
   * for `draws` draws: mcse = sd / sqrt(ess_mean), iact = draws / ess_mean.  What survives of chain 1's summaries: the
   * unobserved rows of the identical-set and gene tables (as in the .convergence files) and ident_obs. */
  const size_t NP = percentiles.size();
  const int npool = o.pool ? nchains : 1;
  const int64_t draws = (int64_t)npool * L;
  vector<int32_t> pidx(NP), pidx_all(NP);
  for (size_t i = 0; i < NP; i++) {
    pidx[i] = static_cast<int>(round(percentiles[i] / 100.0 * (trace_length - 1))); /* :1113 */
    pidx_all[i] = static_cast<int>(round(percentiles[i] / 100.0 * (draws - 1)));
  }
  for (const Level& lv : levels) {
    Summ& S = summ[lv.which];
    const size_t R = (size_t)lv.dev_rows;
    vector<double> var(R), tau(R);
    vector<int32_t> win(R), status(R);
    S.mean.resize(R); S.sd.resize(R); S.mcse.resize(R); S.iact.resize(R); S.pct.resize(R * NP);
    if (R > 0 && !(o.pool && lv.which == 0)) /* -pool: every transcript row comes from mmq_pooled_summaries */
      check(mmq_summarize(H0, lv.which, S.mean.data(), var.data(), tau.data(), win.data(), status.data(), (int)NP, pidx.data(), S.pct.data()), H0, "mmq_summarize");
    for (size_t r = 0; r < R; ++r) {
      if (status[r] != 0) { S.mcse[r] = trace_length; S.iact[r] = NAN; }
      else { S.mcse[r] = sqrt(tau[r] * var[r] / trace_length); S.iact[r] = tau[r]; }
      S.sd[r] = sqrt(var[r]);
    }
    if (lv.which == 1) for (size_t s = 0; s < R; ++s) ident_obs[s] = isfinite(S.mean[s]) != 0;
    if (!o.pool || R == 0) continue;
    vector<double> mean(R), psd(R), ess(R), pct(R * NP);
    check(mmq_pooled_summaries(chain_h.data(), nchains, lv.which, nullptr, nullptr, (int)NP, pidx_all.data(), mean.data(), psd.data(), ess.data(),
                               nullptr, nullptr, pct.data()), H0, "mmq_pooled_summaries");
    for (size_t r = 0; r < R; ++r) {
      if (!lv.observed((int64_t)r)) continue;
      S.mean[r] = mean[r];
      S.sd[r] = psd[r];
      S.mcse[r] = psd[r] / sqrt(ess[r]);
      S.iact[r] = (double)draws / ess[r];
      copy(pct.begin() + (ptrdiff_t)(r * NP), pct.begin() + (ptrdiff_t)((r + 1) * NP), S.pct.begin() + (ptrdiff_t)(r * NP));
    }
  }

  /* proportions of observed transcripts (:985-1008, :1236-1265) */
  vector<double> meanprop((size_t)n), meanprobitprop((size_t)n), ssprobitprop((size_t)n), sdprobitprop((size_t)n), pct_prop((size_t)n * NP);
  vector<double> prop_trace;
  if (!notraces) prop_trace.resize((size_t)n * (size_t)L);
  if (!o.pool)
    check(mmq_prop_summaries(H0, gene_of.data(), multi.data(), meanprop.data(), meanprobitprop.data(), ssprobitprop.data(), (int)NP, pidx.data(),
                             pct_prop.data(), notraces ? nullptr : prop_trace.data()), H0, "mmq_prop_summaries");
  else if (!notraces) /* chain 1's proportion trace for its trace file; the summaries come from all chains below */
    check(mmq_prop_summaries(H0, gene_of.data(), multi.data(), nullptr, nullptr, nullptr, 0, nullptr, nullptr, prop_trace.data()), H0,
          "mmq_prop_summaries");
  if (o.pool) /* every chain's proportions over its own gene trace; the probit sums added over the chains */
    check(mmq_pooled_summaries(chain_h.data(), nchains, 3, gene_of.data(), multi.data(), (int)NP, pidx_all.data(), meanprop.data(), nullptr,
                               nullptr, meanprobitprop.data(), ssprobitprop.data(), pct_prop.data()), H0, "mmq_pooled_summaries");
  for (int64_t t = 0; t < n; t++) /* :1260-1265, same expression order */
    sdprobitprop[(size_t)t] = sqrt((ssprobitprop[(size_t)t] - meanprobitprop[(size_t)t] * meanprobitprop[(size_t)t] / draws) / (draws - 1.0));
  for (int64_t t = 0; t < n; t++) meanprobitprop[(size_t)t] /= draws;

  /* gene traces are needed on the host for the hit-less isoforms' proportions and the trace file */
  vector<double> gene_trace((size_t)G * (size_t)L);
  if (G > 0) check(mmq_get_group_trace(H0, 2, gene_trace.data()), H0, "mmq_get_group_trace");

  /* hit-less isoforms: percentiles of the simulated trace, proportion summaries (:1174-1192, :1267-1305); with -pool over
   * the prior draws of all chains, each chain's proportions over its own gene trace and its probit sums added in chain
   * order */
  vector<double> pct_simu((size_t)U * NP), pct_prop_simu((size_t)U * NP), meanprop_simu((size_t)U), meanprobitprop_simu((size_t)U), sdprobitprop_simu((size_t)U);
  {
    vector<const double*> sim_c((size_t)npool), gtr_c((size_t)npool);
    vector<vector<double>> gtr_other((size_t)npool);
    for (int c = 0; c < npool; ++c) {
      sim_c[(size_t)c] = c == 0 ? simu.data() : simu_pool[(size_t)c].data();
      if (c == 0) { gtr_c[0] = gene_trace.data(); continue; }
      gtr_other[(size_t)c].resize((size_t)G * (size_t)L);
      if (U > 0) check(mmq_get_group_trace(chain_h[(size_t)c], 2, gtr_other[(size_t)c].data()), chain_h[(size_t)c], "mmq_get_group_trace");
      gtr_c[(size_t)c] = gtr_other[(size_t)c].data();
    }
    /* isoforms u0 .. u1 - 1; every isoform's values are its own, so the host threads split the isoforms freely */
    auto isoforms = [&](int64_t u0, int64_t u1) {
      vector<double> v((size_t)draws), pv((size_t)draws);
      for (int64_t u = u0; u < u1; ++u) {
        const int32_t g = hdr.gene_of[(size_t)unobs[(size_t)u]];
        const bool multi_iso = hdr.gene_members[(size_t)g].size() > 1;
        double mp = 0.0, s1 = 0.0, s2 = 0.0;
        for (int c = 0; c < npool; ++c) {
          const double* sv = sim_c[(size_t)c] + (size_t)u * (size_t)L;
          const double* gt = gtr_c[(size_t)c] + (size_t)g * (size_t)L;
          double c1 = 0.0, c2 = 0.0;
          for (int i = 0; i < L; ++i) {
            const double p = sv[i] / gt[i];
            v[(size_t)c * (size_t)L + (size_t)i] = sv[i];
            pv[(size_t)c * (size_t)L + (size_t)i] = p;
            mp += p;
            double temp;
            if (multi_iso) temp = mmq_host_ndtri(min(max(p, 0.000000001), 0.999999999));
            else temp = numeric_limits<double>::infinity();
            c1 += temp;
            c2 += temp * temp;
          }
          s1 = c == 0 ? c1 : s1 + c1;
          s2 = c == 0 ? c2 : s2 + c2;
        }
        sort(v.begin(), v.end());
        sort(pv.begin(), pv.end());
        for (size_t j = 0; j < NP; ++j) {
          pct_simu[(size_t)u * NP + j] = v[(size_t)pidx_all[j]];
          pct_prop_simu[(size_t)u * NP + j] = pv[(size_t)pidx_all[j]];
        }
        meanprop_simu[(size_t)u] = mp / draws;
        sdprobitprop_simu[(size_t)u] = sqrt((s2 - s1 * s1 / draws) / (draws - 1.0));
        meanprobitprop_simu[(size_t)u] = s1 / draws;
      }
    };
    const int nt = (int)max<int64_t>(1, min<int64_t>(min(32u, max(1u, thread::hardware_concurrency())), U * npool / 256));
    vector<thread> th;
    for (int t = 0; t < nt; ++t) th.emplace_back(isoforms, U * t / nt, U * (t + 1) / nt);
    for (auto& x : th) x.join();
  }

  phase("summaries");
  /* ---- trace dumps (:829-831, :911-917, :1033-1108) */
  if (!notraces) {
    vector<double> tr((size_t)n * (size_t)L);
    check(mmq_get_trace(H0, tr.data()), H0, "mmq_get_trace");
    vector<string> ids((size_t)n);
    for (int64_t t = 0; t < n; ++t) ids[(size_t)t] = hdr.names[(size_t)cls.col2hdr[(size_t)t]];
    write_trace_gz(output_base + ".trace_gibbs.gz", ids, {}, tr.data(), L);
    write_trace_gz(output_base + ".prop.trace_gibbs.gz", ids, {}, prop_trace.data(), L);
    vector<double> itr((size_t)I * (size_t)L);
    if (I > 0) check(mmq_get_group_trace(H0, 1, itr.data()), H0, "mmq_get_group_trace");
    vector<string> iids((size_t)I);
    vector<char> keep((size_t)I);
    for (int64_t s = 0; s < I; ++s) {
      iids[(size_t)s] = identical_id(s);
      keep[(size_t)s] = isfinite(log(itr[(size_t)s * (size_t)L])) != 0; /* :1045 */
    }
    write_trace_gz(output_base + ".identical.trace_gibbs.gz", iids, keep, itr.data(), L);
    vector<char> gkeep((size_t)G);
    for (int64_t g = 0; g < G; ++g) gkeep[(size_t)g] = isfinite(log(gene_trace[(size_t)g * (size_t)L])) != 0; /* :1074 */
    write_trace_gz(output_base + ".gene.trace_gibbs.gz", hdr.gene_names, gkeep, gene_trace.data(), L);
  }

  phase("trace files");
  const Summ &St = summ[0], &Si = summ[1], &Sg = summ[2];
  /* ---- gene lengths (:1372-1395) */
  vector<double> gene_lengths((size_t)G, 0.0);
  for (int64_t g = 0; g < G; ++g) {
    if (isfinite(Sg.mean[(size_t)g]) != 0) {
      double sum = 0;
      for (int32_t hidx : hdr.gene_members[(size_t)g]) {
        const int32_t c = cls.hdr2col[(size_t)hidx];
        const double len = hdr.efflen[(size_t)hidx];
        if (c >= 0) {
          gene_lengths[(size_t)g] += len * exp(St.mean[(size_t)c]);
          sum += exp(St.mean[(size_t)c]);
        } else {
          gene_lengths[(size_t)g] += len * exp(closed_log_mu(len));
          sum += exp(closed_log_mu(len));
        }
      }
      gene_lengths[(size_t)g] /= sum;
    }
  }

  /* ---- .mmseq (:1469-1554) */
  ofs.open((output_base + ".mmseq").c_str());
  ofs << "# Mapped fragments: " << N << endl;
  ofs << "feature_id\tlog_mu\tsd\tmcse\tiact\teffective_length\ttrue_length\tunique_hits\tmean_proportion\tmean_probit_proportion\tsd_probit_proportion\tlog_mu_em\tobserved\tntranscripts\t";
  ofs << "percentiles";
  write_pcts(ofs, percentiles.data(), NP, '\t');
  ofs << "percentiles_proportion";
  write_pcts(ofs, percentiles.data(), NP, '\n');
  write_rows(ofs, T, [&](ostream& ofs, int64_t hI) {
    const string& name = hdr.names[(size_t)hI];
    const int32_t c = cls.hdr2col[(size_t)hI];
    const size_t ntr = hdr.gene_members[(size_t)hdr.gene_of[(size_t)hI]].size();
    if (c >= 0) {
      ofs << name << "\t" << St.mean[(size_t)c] << "\t" << St.sd[(size_t)c] << "\t" << St.mcse[(size_t)c] << "\t" << St.iact[(size_t)c] << "\t"
          << hdr.efflen[(size_t)hI] << "\t" << hdr.truelen[(size_t)hI] << "\t" << unique_hits[(size_t)c] << "\t" << meanprop[(size_t)c] << "\t"
          << meanprobitprop[(size_t)c] << "\t" << sdprobitprop[(size_t)c] << "\t" << log(mu_em[(size_t)c]) << "\t"
          << "1" << "\t" << ntr << "\t";
      write_pcts(ofs, St.pct.data() + (size_t)c * NP, NP, '\t');
      write_pcts(ofs, pct_prop.data() + (size_t)c * NP, NP, '\n');
    } else {
      const size_t u = (size_t)unobs_slot[(size_t)hI];
      ofs << name << "\t" << closed_log_mu(hdr.efflen[(size_t)hI]) << "\t" << sqrtpolygalpha << "\t"
          << "0" << "\t" << "1" << "\t" << hdr.efflen[(size_t)hI] << "\t" << hdr.truelen[(size_t)hI] << "\t" << 0 << "\t" << meanprop_simu[u] << "\t"
          << meanprobitprop_simu[u] << "\t" << sdprobitprop_simu[u] << "\t" << "NA" << "\t" << "0" << "\t" << ntr << "\t";
      write_pcts(ofs, pct_simu.data() + u * NP, NP, '\t');
      write_pcts(ofs, pct_prop_simu.data() + u * NP, NP, '\n');
    }
  });
  ofs.close(); ofs.clear();

  /* ---- .identical.mmseq (:1556-1613) */
  ofs.open((output_base + ".identical.mmseq").c_str());
  ofs << "# Mapped fragments: " << N << endl;
  ofs << "feature_id\tlog_mu\tsd\tmcse\tiact\teffective_length\ttrue_length\tunique_hits\tobserved\tntranscripts\t";
  ofs << "percentiles";
  write_pcts(ofs, percentiles.data(), NP, '\n');
  for (int64_t s = 0; s < I; ++s) {
    const auto& mem = hdr.identical[(size_t)s];
    const int32_t first = mem.front();
    const bool obs = ident_obs[(size_t)s] != 0;
    for (size_t j = 0; j < mem.size(); ++j) {
      ofs << hdr.names[(size_t)mem[j]];
      if (!named_last(mem, j)) { ofs << "+"; continue; }
      if (obs) ofs << "\t" << Si.mean[(size_t)s] << "\t" << Si.sd[(size_t)s] << "\t" << Si.mcse[(size_t)s] << "\t" << Si.iact[(size_t)s];
      else { const auto u = levels[1].unobserved(s); ofs << "\t" << u.first << "\t" << u.second << "\t" << "0" << "\t" << "NA"; }
      ofs << "\t" << hdr.efflen[(size_t)first] << "\t" << hdr.truelen[(size_t)first] << "\t" << (obs ? identical_unique_hits[(size_t)s] : 0) << "\t"
          << (obs ? "1" : "0") << "\t" << mem.size() << "\t";
    }
    if (obs) write_pcts(ofs, Si.pct.data() + (size_t)s * NP, NP, '\n');
    else for (size_t i = 0; i < NP; i++) ofs << "NA" << (i == NP - 1 ? "\n" : ",");
  }
  ofs.close(); ofs.clear();

  /* ---- .gene.mmseq (:1615-1669) */
  ofs.open((output_base + ".gene.mmseq").c_str());
  ofs << "# Mapped fragments: " << N << endl;
  ofs << "feature_id\tlog_mu\tsd\tmcse\tiact\teffective_length\ttrue_length\tunique_hits\tntranscripts\tobserved\t";
  ofs << "percentiles";
  write_pcts(ofs, percentiles.data(), NP, '\n');
  write_rows(ofs, G, [&](ostream& ofs, int64_t g) {
    const size_t ntr = hdr.gene_members[(size_t)g].size();
    ofs << hdr.gene_names[(size_t)g] << "\t" << Sg.mean[(size_t)g] << "\t" << Sg.sd[(size_t)g] << "\t";
    if (levels[2].observed(g))
      ofs << Sg.mcse[(size_t)g] << "\t" << Sg.iact[(size_t)g] << "\t" << gene_lengths[(size_t)g] << "\t" << "NA" << "\t" << gene_unique_hits[(size_t)g] << "\t"
          << ntr << "\t" << "1" << "\t";
    else
      ofs << Sg.sd[(size_t)g] / sqrt(trace_length) << "\t" << 1 << "\t" << gene_lengths[(size_t)g] << "\t" << "NA" << "\t" << "0" << "\t" << ntr << "\t" << "0" << "\t";
    write_pcts(ofs, Sg.pct.data() + (size_t)g * NP, NP, '\n');
  });
  ofs.close(); ofs.clear();

  /* output_base + suffix + ext: the mapped-fragments line, `head`, then one line per table row: its id and
   * cols(table row, device row) */
  auto write_table = [&](const string& suffix, const string& head, int64_t rows, const function<string(int64_t)>& id,
                         const function<void(ostream&, int64_t)>& cols) {
    ofs.open((output_base + suffix).c_str());
    ofs << "# Mapped fragments: " << N << endl << head;
    write_rows(ofs, rows, [&](ostream& os, int64_t r) { os << id(r) << "\t"; cols(os, r); });
    ofs.close(); ofs.clear();
  };
  auto write_level = [&](const Level& lv, const char* ext, const string& head, const function<void(ostream&, int64_t, int64_t)>& cols) {
    write_table(string(lv.suffix) + ext, head, lv.rows, lv.id, [&](ostream& os, int64_t r) { cols(os, r, lv.dev_row(r)); });
  };

  /* ---- -counts: .counts, .identical.counts, .gene.counts — posterior mean and sd over the chain's sweeps, EM expected
   * count (a group's: the sum of its members').  Every shard holds the same moments.  With -pool the moments of all
   * chains are added exactly: sweeps, sums and 128-bit sums of squares. */
  if (o.counts)
    for (const Level& lv : levels) {
      int64_t S = 0;
      const size_t R = (size_t)lv.dev_rows;
      vector<uint64_t> sum(R), lo(R), hi(R);
      check(mmq_get_count_moments(H0, lv.which, &S, sum.data(), lo.data(), hi.data()), H0, "mmq_get_count_moments");
      for (int c = 1; c < npool; ++c) {
        mmq_handle* h = chain_h[(size_t)c];
        int64_t Sc = 0;
        vector<uint64_t> sc(R), lc(R), hc(R);
        check(mmq_get_count_moments(h, lv.which, &Sc, sc.data(), lc.data(), hc.data()), h, "mmq_get_count_moments");
        S += Sc;
        for (size_t q = 0; q < R; ++q) {
          sum[q] += sc[q];
          const uint64_t l = lo[q] + lc[q];
          hi[q] += hc[q] + (l < lo[q]);
          lo[q] = l;
        }
      }
      write_level(lv, ".counts", "feature_id\tposterior_mean_count\tposterior_sd_count\tem_count\n", [&](ostream& os, int64_t, int64_t q) {
        if (q < 0 || S == 0) os << 0.0 << "\t" << 0.0 << "\t" << 0.0 << "\n";
        else os << (double)sum[(size_t)q] / (double)S << "\t" << count_sd(S, sum[(size_t)q], lo[(size_t)q], hi[(size_t)q]) << "\t" << lv.sum(q, em_count) << "\n";
      });
    }

  /* ---- -tpm: .tpm, .identical.tpm, .gene.tpm — posterior mean, sd and percentiles of TPM over chain 1's draws (with
   * -pool over every chain's, each chain normalised by its own totals; mmq_tpm_summaries), and the EM TPM from mu_em.
   * The totals are over the observed transcripts only, so TPM sums to 1e6 over the observed features; a feature without
   * an observed member reports 0 in every column. */
  if (o.tpm) {
    double em_total = 0.0;
    for (int64_t t = 0; t < n; ++t) em_total += mu_em[(size_t)t];
    ostringstream head;
    head << "feature_id\tposterior_mean_tpm\tposterior_sd_tpm\tem_tpm\tpercentiles_tpm";
    write_pcts(head, percentiles.data(), NP, '\n');
    if (NP == 0) head << '\n';
    const vector<double> zeros(NP, 0.0);
    for (const Level& lv : levels) {
      const size_t R = (size_t)lv.dev_rows;
      vector<double> mean(R), sdv(R), pct(R * NP);
      if (R > 0)
        check(mmq_tpm_summaries(chain_h.data(), npool, lv.which, (int)NP, pidx_all.data(), mean.data(), sdv.data(), pct.data(), nullptr), H0,
              "mmq_tpm_summaries");
      write_level(lv, ".tpm", head.str(), [&](ostream& os, int64_t, int64_t q) {
        const bool obs = q >= 0 && lv.has_hits(q);
        if (!obs) os << 0 << "\t" << 0 << "\t" << 0 << "\t";
        else os << mean[(size_t)q] << "\t" << sdv[(size_t)q] << "\t" << (lv.sum(q, mu_em) / em_total) * 1000000.0 << "\t";
        write_pcts(os, obs ? pct.data() + (size_t)q * NP : zeros.data(), NP, '\n');
        if (NP == 0) os << '\n';
      });
    }
  }

  /* ---- -allelic: .allelic, .gene.allelic — per unit the fragments only one side explains (mmq_allele_only_counts, all
   * shards), the EM fraction from mu_em, and the posterior mean, sd, P(a > b) and percentiles of phi = a / (a + b) over
   * chain 1's draws (with -pool over every chain's; mmq_allelic_summaries).  The hit-less copies of a pair enter as the
   * prior draws their chain already uses.  A unit without an observed member reports NA in every posterior and EM
   * column; NaN is written NA. */
  if (o.allelic) {
    const int64_t nprior = (int64_t)prior_hdr.size();
    vector<vector<double>> prior_rows((size_t)npool, vector<double>((size_t)nprior * (size_t)L));
    vector<const double*> prior_ptr((size_t)npool);
    for (int c = 0; c < npool; ++c) {
      const double* sim = c == 0 ? simu.data() : simu_pool[(size_t)c].data();
      for (int64_t j = 0; j < nprior; ++j)
        copy_n(sim + (size_t)unobs_slot[(size_t)prior_hdr[(size_t)j]] * (size_t)L, L, prior_rows[(size_t)c].begin() + (ptrdiff_t)(j * L));
      prior_ptr[(size_t)c] = prior_rows[(size_t)c].data();
    }
    ostringstream head;
    head << "feature_id\tpairs\ta_only_fragments\tb_only_fragments\tem_fraction_a\tposterior_mean_fraction_a\tposterior_sd_fraction_a"
            "\tprob_a_gt_b\tpercentiles_fraction_a";
    write_pcts(head, percentiles.data(), NP, '\n');
    if (NP == 0) head << '\n';
    auto put = [](ostream& os, double v) -> ostream& { if (std::isnan(v)) os << "NA"; else os << v; return os; };
    for (const AlleleLevel& al : allele_levels) {
      const size_t R = (size_t)al.rows;
      vector<int32_t> a_only(R), b_only(R);
      on_all([&](int g) {
        mmq_handle* h = shards[(size_t)g].h;
        vector<int32_t> oa(g == 0 ? 0 : R), ob(g == 0 ? 0 : R);
        check(mmq_allele_only_counts(h, al.unit_of.data(), al.side.data(), al.rows, g == 0 ? a_only.data() : oa.data(), g == 0 ? b_only.data() : ob.data()),
              h, "mmq_allele_only_counts");
      });
      vector<double> mean(R), sdv(R), prob(R), pct(R * NP);
      check(mmq_allelic_summaries(chain_h.data(), npool, prior_ptr.data(), nprior, al.rows, al.a_ptr.data(), al.a_mem.data(), al.b_ptr.data(),
                                  al.b_mem.data(), (int)NP, pidx_all.data(), mean.data(), sdv.data(), prob.data(), pct.data()), H0,
            "mmq_allelic_summaries");
      write_table(string(al.suffix) + ".allelic", head.str(), al.rows, al.id, [&](ostream& os, int64_t u) {
        const bool obs = al.observed(u);
        double sa = 0.0, sb = 0.0; /* EM: the observed members in index order; a hit-less copy counts 0 */
        for (int64_t q = al.a_ptr[(size_t)u]; q < al.a_ptr[(size_t)u + 1]; ++q) if (al.a_mem[(size_t)q] < n) sa += mu_em[(size_t)al.a_mem[(size_t)q]];
        for (int64_t q = al.b_ptr[(size_t)u]; q < al.b_ptr[(size_t)u + 1]; ++q) if (al.b_mem[(size_t)q] < n) sb += mu_em[(size_t)al.b_mem[(size_t)q]];
        const double na = NAN, em = sa == 0.0 && sb == 0.0 ? na : sa / (sa + sb);
        os << al.npairs[(size_t)u] << "\t" << a_only[(size_t)u] << "\t" << b_only[(size_t)u] << "\t";
        put(os, obs ? em : na) << "\t";
        put(os, obs ? mean[(size_t)u] : na) << "\t";
        put(os, obs ? sdv[(size_t)u] : na) << "\t";
        put(os, obs ? prob[(size_t)u] : na) << "\t";
        for (size_t j = 0; j < NP; ++j) put(os, obs ? pct[(size_t)u * NP + j] : na) << (j == NP - 1 ? '\n' : ',');
        if (NP == 0) os << '\n';
      });
    }
  }

  /* ---- -isocorr: .isocorr — per isoform pair of a gene the fragments both explain (mmq_pair_shared_counts, all shards)
   * and the correlation of mu and of log mu and P(first > second) over chain 1's draws (with -pool over every chain's;
   * mmq_isocorr_summaries).  NaN is written NA. */
  if (o.isocorr) {
    const int64_t P = (int64_t)pair_gene.size();
    vector<int64_t> shared((size_t)P);
    on_all([&](int g) {
      mmq_handle* h = shards[(size_t)g].h;
      vector<int64_t> other(g == 0 ? 0 : (size_t)P);
      check(mmq_pair_shared_counts(h, iso_gene.data(), iso_local.data(), pair_base.data(), G, P, g == 0 ? shared.data() : other.data()), h,
            "mmq_pair_shared_counts");
    });
    vector<double> cmu((size_t)P), clog((size_t)P), pgt((size_t)P);
    check(mmq_isocorr_summaries(chain_h.data(), npool, P, cmu.data(), clog.data(), pgt.data()), H0, "mmq_isocorr_summaries");
    auto put = [](ostream& os, double v) -> ostream& { if (std::isnan(v)) os << "NA"; else os << v; return os; };
    auto name = [&](int64_t p, int32_t a) { return hdr.names[(size_t)cls.col2hdr[(size_t)gmem[(size_t)(gptr[(size_t)pair_gene[(size_t)p]] + a)]]]; };
    write_table(".isocorr", "gene_id\ttranscript_1\ttranscript_2\tshared_fragments\tcorr_mu\tcorr_log_mu\tprob_1_gt_2\n", P,
                [&](int64_t p) { return hdr.gene_names[(size_t)pair_gene[(size_t)p]]; }, [&](ostream& os, int64_t p) {
                  os << name(p, pair_a[(size_t)p]) << "\t" << name(p, pair_b[(size_t)p]) << "\t" << shared[(size_t)p] << "\t";
                  put(os, cmu[(size_t)p]) << "\t";
                  put(os, clog[(size_t)p]) << "\t";
                  put(os, pgt[(size_t)p]) << "\n";
                });
  }

  /* ---- -chains: .convergence, .identical.convergence, .gene.convergence — log_mu and sd pooled over the draws of all
   * chains, split-R-hat and bulk / tail ESS (mmq_chain_diagnostics); a row whose `observed` column is 0 in the tables
   * above carries that table's closed-form log_mu and sd, and NA. */
  if (nchains > 1)
    for (const Level& lv : levels) {
      const size_t R = (size_t)lv.dev_rows;
      vector<double> rh(R), eb(R), et(R), lm(R), ls(R);
      if (R > 0)
        check(mmq_chain_diagnostics(chain_h.data(), nchains, lv.which, rh.data(), eb.data(), et.data(), lm.data(), ls.data()), H0,
              "mmq_chain_diagnostics");
      auto put = [](ostream& os, double v) -> ostream& { if (std::isnan(v)) os << "NA"; else os << v; return os; };
      write_level(lv, ".convergence", "feature_id\tlog_mu\tsd\trhat\tess_bulk\tess_tail\n", [&](ostream& os, int64_t r, int64_t q) {
        if (q < 0 || !lv.observed(q)) { const auto u = lv.unobserved(r); put(os, u.first) << "\t"; put(os, u.second) << "\tNA\tNA\tNA\n"; return; }
        put(os, lm[(size_t)q]) << "\t"; put(os, ls[(size_t)q]) << "\t"; put(os, rh[(size_t)q]) << "\t"; put(os, eb[(size_t)q]) << "\t"; put(os, et[(size_t)q]) << "\n";
      });
      double max_rhat = NAN, min_ess = NAN;
      int64_t over = 0;
      for (int64_t r = 0; r < lv.rows; ++r) {
        const int64_t q = lv.dev_row(r);
        if (q < 0 || !lv.observed(q)) continue;
        if (!std::isnan(rh[(size_t)q])) { max_rhat = std::isnan(max_rhat) ? rh[(size_t)q] : max(max_rhat, rh[(size_t)q]); over += rh[(size_t)q] > 1.01; }
        if (!std::isnan(eb[(size_t)q])) min_ess = std::isnan(min_ess) ? eb[(size_t)q] : min(min_ess, eb[(size_t)q]);
      }
      err << "Convergence of the " << lv.name << " over " << nchains << " chains: largest rhat " << max_rhat << ", " << over
          << " with rhat > 1.01, smallest ess_bulk " << min_ess << endl;
    }

  out << "done." << endl;
  for (auto& S : shards) mmq_destroy(S.h);
  for (int c = 1; c < nchains; ++c) mmq_destroy(chain_h[(size_t)c]);

  phase("tables");
  out << "Output files: " << endl;
  auto list = [&](const char* ext) { for (const Level& lv : levels) out << "  " << output_base << lv.suffix << ext << endl; };
  list(".mmseq");
  if (o.counts) list(".counts");
  if (o.tpm) list(".tpm");
  for (const AlleleLevel& al : allele_levels) out << "  " << output_base << al.suffix << ".allelic" << endl;
  if (o.isocorr) out << "  " << output_base << ".isocorr" << endl;
  if (nchains > 1) list(".convergence");
  out << "  " << output_base << ".M" << endl << "  " << output_base << ".k" << endl << endl;
  if (!notraces) {
    list(".trace_gibbs.gz");
    out << "  " << output_base << ".prop.trace_gibbs.gz" << endl << endl;
  }
  if (debug) {
    out << endl
         << "  " << output_base << ".trace_em.gz" << endl
         << "  " << output_base << ".sharedcounts" << endl
         << "  " << output_base << ".Mt-nodups" << endl
         << "  " << output_base << ".doublehits" << endl
         << "  " << output_base << ".dupIDs" << endl;
  }
}

/* -batch FILE (config 5: many samples, independent chains): every line of FILE names a hits file and an output base.
 * Samples are dealt to the GPUs of the box, per_gpu of them in flight per GPU (their parsing, host-side formatting
 * and device work overlap); each runs as a single-GPU sample and writes its messages to <output_base>.log. */
static int run_batch(const Options& o) {
  vector<pair<string, string>> samples;
  {
    ifstream f(o.batch.c_str());
    if (!f) die("Error: cannot open batch file " + o.batch + ".");
    string a, b;
    while (f >> a >> b) samples.emplace_back(a, b);
  }
  if (samples.empty()) die("Error: no samples in " + o.batch + ".");
  Options one = o;
  one.ngpus = 1;
  const int workers = (int)min<size_t>(samples.size(), (size_t)o.ngpus * (size_t)o.per_gpu);
  cout << "Batch of " << samples.size() << " samples on " << o.ngpus << " GPU(s), " << o.per_gpu << " in flight per GPU." << endl;
  const auto t0 = chrono::steady_clock::now();
  atomic<size_t> next{0};
  vector<thread> th;
  for (int w = 0; w < workers; ++w)
    th.emplace_back([&, w] {
      for (size_t i = next.fetch_add(1); i < samples.size(); i = next.fetch_add(1)) {
        ostringstream log;
        const auto s0 = chrono::steady_clock::now();
        run_sample(one, samples[i].first, samples[i].second, w % o.ngpus, log, log);
        log << "wall " << chrono::duration<double>(chrono::steady_clock::now() - s0).count() << " s on GPU " << w % o.ngpus << endl;
        ofstream lf((samples[i].second + ".log").c_str());
        lf << log.str();
      }
    });
  for (auto& t : th) t.join();
  const double wall = chrono::duration<double>(chrono::steady_clock::now() - t0).count();
  cout << "Batch done: " << samples.size() << " samples in " << wall << " s (" << samples.size() / wall << " samples/s, "
       << (double)samples.size() * o.gibbs_iter / wall << " Gibbs sweeps/s over all samples)." << endl;
  return 0;
}

int main(int argc, char** argv) {
  phase("start");
  const Options o = parse_command_line(argc, argv);
  if (!o.batch.empty()) {
    run_batch(o);
  } else {
    run_sample(o, o.positional[0], o.positional[1], 0, cout, cerr);
  }
  /* every output file is closed: leave without unwinding gigabytes of host vectors and the CUDA
   * contexts (1-2 s at 30M fragments); exit status 0 as src/mmseq.cpp:1727 */
  cout.flush();
  cerr.flush();
  fflush(nullptr);
  _exit(0);
}
