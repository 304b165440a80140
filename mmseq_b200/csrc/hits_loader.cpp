/* hits_loader.cpp — see hits_loader.h.  Format facts follow the reference's
 * writer/reader pair: src/hitsio.cpp:162-240 (writer), :250-447 (reader),
 * README.md:388-403. */
#include "hits_loader.h"
#include "inflate_par.h"
#include "fmt_g6.h"
#include "huff_gz.h"
#include "trace_writer.h"

#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <sstream>
#include <thread>
#include <unordered_map>

namespace mmq {

namespace {

/* Buffered byte stream over a file, transparently zlib-inflated when the file
 * starts with 0x78 (src/hitsio.cpp:258: "lazy but sufficient" detection).  Reading and
 * inflating run in a producer thread that hands 4 MB blocks to the parser through a small
 * queue, so decompression overlaps parsing and class building. */
class ByteSource {
 public:
  ~ByteSource() { close(); }
  bool open(const std::string& path) {
    f_ = fopen(path.c_str(), "rb");
    if (!f_) return false;
    int c = fgetc(f_);
    if (c == EOF) { compressed_ = false; }
    else { ungetc(c, f_); compressed_ = (c == 0x78); }
    pos_ = len_ = 0;
    base_ = nullptr;
    if (compressed_ && !getenv("MMQ_LOADER_SERIAL_INFLATE")) {
      /* the whole stream on all host threads (inflate_par.h); anything it cannot handle falls through to zlib below,
       * which also produces the proper diagnosis for a corrupt or truncated file */
      fseek(f_, 0, SEEK_END);
      const long sz = ftell(f_);
      fseek(f_, 0, SEEK_SET);
      long par_min = 4 << 20; /* smaller files are not worth the threads */
      if (const char* e = getenv("MMQ_LOADER_PAR_MIN_BYTES")) par_min = atol(e);
      if (sz > par_min) {
        const bool tm = getenv("MMQ_LOADER_TIMING") != nullptr;
        auto clk = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        const double t0 = clk();
        std::unique_ptr<uint8_t[]> rawp(new uint8_t[(size_t)sz]);
        struct { uint8_t* p; size_t n; uint8_t* data() { return p; } size_t size() { return n; } } raw{rawp.get(), (size_t)sz};
        if (fread(raw.data(), 1, (size_t)sz, f_) == (size_t)sz) {
          const double t1 = clk();
          unsigned hc = std::thread::hardware_concurrency();
          if (const char* e = getenv("MMQ_LOADER_INFLATE_THREADS")) hc = (unsigned)atoi(e);
          const bool okp = ipar::inflate_parallel(raw.data(), raw.size(), (int)std::max(1u, hc), whole_);
          if (tm) fprintf(stderr, "[loader] file read %.2f s, parallel inflate (%u threads) %.2f s%s\n", t1 - t0, hc, clk() - t1, okp ? "" : " FAILED: serial zlib instead");
          if (okp) {
            base_ = (const char*)whole_.data();
            len_ = whole_.size();
            whole_mode_ = true;
            return true;
          }
        }
        fseek(f_, 0, SEEK_SET);
      }
    }
    if (compressed_) {
      memset(&zs_, 0, sizeof zs_);
      if (inflateInit(&zs_) != Z_OK) return false;
      zinit_ = true;
      in_.resize(1 << 20);
    }
    producer_done_ = false;
    stop_ = false;
    whole_mode_ = false;
    prod_ = std::thread([this] { produce(); });
    return true;
  }
  void close() {
    if (prod_.joinable()) {
      { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
      cv_.notify_all();
      prod_.join();
    }
    if (zinit_) { inflateEnd(&zs_); zinit_ = false; }
    if (f_) { fclose(f_); f_ = nullptr; }
  }
  bool corrupt() const { return corrupt_; }
  /* the whole inflated file is in memory (parallel inflate): the record walk can then hand offsets to parallel builders */
  bool whole() const { return whole_mode_; }
  const char* whole_base() const { return base_; }
  size_t whole_pos() const { return pos_; }
  size_t whole_size() const { return len_; }
  int peek() {
    if (pos_ == len_ && !fill()) return EOF;
    return (unsigned char)base_[pos_];
  }
  int get() {
    if (pos_ == len_ && !fill()) return EOF;
    return (unsigned char)base_[pos_++];
  }
  /* like std::getline: false only when nothing at all could be read */
  bool getline(std::string& out) {
    out.clear();
    bool any = false;
    for (;;) {
      if (pos_ == len_ && !fill()) return any;
      any = true;
      const char* b = base_ + pos_;
      const char* nl = (const char*)memchr(b, '\n', len_ - pos_);
      if (nl) {
        out.append(b, (size_t)(nl - b));
        pos_ += (size_t)(nl - b) + 1;
        return true;
      }
      out.append(b, len_ - pos_);
      pos_ = len_;
    }
  }
  /* a line as a view into the current block (no copy) unless it straddles two blocks */
  bool getline_view(const char*& p, size_t& n) {
    if (pos_ == len_ && !fill()) return false;
    const char* b = base_ + pos_;
    const char* nl = (const char*)memchr(b, '\n', len_ - pos_);
    if (nl) { p = b; n = (size_t)(nl - b); pos_ += n + 1; return true; }
    if (!getline(carry_)) return false;
    p = carry_.data(); n = carry_.size();
    return true;
  }
  bool read_bytes(void* dst, size_t n) {
    char* d = (char*)dst;
    while (n) {
      if (pos_ == len_ && !fill()) return false;
      size_t c = std::min(n, len_ - pos_);
      memcpy(d, base_ + pos_, c);
      pos_ += c; d += c; n -= c;
    }
    return true;
  }
  bool read_u32(uint32_t& v) { /* raw little-endian, src/hitsio.cpp:22-34 */
    if (len_ - pos_ >= 4) { memcpy(&v, base_ + pos_, 4); pos_ += 4; return true; }
    return read_bytes(&v, 4);
  }
  /* one byte, or 0xFF followed by a uint32 (src/hitsio.cpp:36-55) */
  bool read_small(uint32_t& v) {
    int c = get();
    if (c == EOF) return false;
    if (c == 255) return read_u32(v);
    v = (uint32_t)c;
    return true;
  }

 private:
  static constexpr size_t BLOCK = (size_t)4 << 20;
  /* producer thread: read (and inflate) the file into blocks */
  void produce() {
    for (;;) {
      std::vector<char> blk(BLOCK);
      size_t got = 0;
      bool last = false;
      if (!compressed_) {
        got = fread(blk.data(), 1, blk.size(), f_);
        last = got < blk.size();
      } else {
        while (got < blk.size() && !last) {
          if (zs_.avail_in == 0) {
            size_t r = fread(in_.data(), 1, in_.size(), f_);
            if (r == 0) { corrupt_ = true; last = true; break; } /* the file ends before the zlib stream does: truncated */
            zs_.next_in = (Bytef*)in_.data();
            zs_.avail_in = (uInt)r;
          }
          zs_.next_out = (Bytef*)blk.data() + got;
          zs_.avail_out = (uInt)(blk.size() - got);
          int rc = inflate(&zs_, Z_NO_FLUSH);
          got = blk.size() - zs_.avail_out;
          if (rc == Z_STREAM_END) { last = true; break; }
          if (rc != Z_OK && rc != Z_BUF_ERROR) { corrupt_ = true; last = true; break; }
        }
      }
      blk.resize(got);
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return q_.size() < 4 || stop_; });
        if (stop_) return;
        if (got) q_.push_back(std::move(blk));
        if (last) producer_done_ = true;
      }
      cv_.notify_all();
      if (last) return;
    }
  }
  bool fill() {
    if (whole_mode_) return false; /* the whole file is already in memory */
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [&] { return !q_.empty() || producer_done_; });
    if (q_.empty()) return false;
    buf_ = std::move(q_.front());
    q_.pop_front();
    lk.unlock();
    cv_.notify_all();
    pos_ = 0;
    len_ = buf_.size();
    base_ = buf_.data();
    return len_ > 0;
  }
  FILE* f_ = nullptr;
  bool compressed_ = false, zinit_ = false, corrupt_ = false;
  z_stream zs_;
  std::vector<char> buf_, in_;
  const char* base_ = nullptr; /* the current block (or the whole inflated file) */
  ipar::Bytes whole_;
  bool whole_mode_ = false;
  std::string carry_;
  size_t pos_ = 0, len_ = 0;
  std::thread prod_;
  std::mutex mu_;
  std::condition_variable cv_;
  std::deque<std::vector<char>> q_;
  bool producer_done_ = false, stop_ = false;
};

inline uint64_t mix64(uint64_t x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
  return x;
}

}  // namespace

/* ------------------------------------------------------------ class builder */

struct ClassBuilder::Impl {
  int layout;
  bool header_order = false, identity_cols = false;
  bool weighted;
  int builders = 1; /* threads of ingest_parallel */
  int64_t N = 0;
  std::vector<int32_t> hdr2col, col2hdr, doublehits;
  /* distinct classes in first-appearance order */
  std::vector<int64_t> cls_ptr{0};
  std::vector<int32_t> cls_col;
  std::vector<int32_t> cls_k;
  /* open-addressing table of class ids keyed by the sorted column set */
  std::vector<int32_t> table;
  std::vector<uint64_t> cls_hash;
  /* per-fragment layouts: class of each record and (weighted) the weights in class column order */
  std::vector<int32_t> rec_class;
  std::vector<float> rec_w;
  std::vector<int64_t> rec_wptr{0};
  std::vector<std::pair<int32_t, float>> comb;

  /* ---- parallel ingestion (unweighted): add_record() does the sequential part (column
   * numbering, de-duplication, sort, hash) and hands the class key to one of K shard workers
   * chosen by the hash; each worker owns a hash table.  finish() merges the shards' classes in
   * order of their first record, which is exactly the sequential first-appearance numbering. */
  struct Batch {
    std::vector<int64_t> rec;
    std::vector<uint64_t> hash;
    std::vector<uint32_t> off{0};
    std::vector<int32_t> cols;
    void clear() { rec.clear(); hash.clear(); off.assign(1, 0); cols.clear(); }
  };
  struct Shard {
    std::mutex mu;
    std::condition_variable cv;
    std::deque<std::unique_ptr<Batch>> q;
    bool done = false;
    std::thread th;
    std::unique_ptr<Batch> cur;
    /* worker-owned */
    std::vector<int32_t> table;
    std::vector<uint64_t> hash;
    std::vector<int64_t> ptr{0};
    std::vector<int32_t> col, k;
    std::vector<int64_t> first_rec;
    std::vector<std::pair<int64_t, int32_t>> rec_cls; /* per-fragment layouts */
  };
  std::vector<std::unique_ptr<Shard>> shards;
  int64_t n_records_keyed = 0; /* records that carry a class (non-empty) */
  static constexpr size_t BATCH_RECORDS = 16384;

  void worker(Shard& S, bool keep_rec) {
    S.table.assign((size_t)1 << 16, -1);
    for (;;) {
      std::unique_ptr<Batch> b;
      {
        std::unique_lock<std::mutex> lk(S.mu);
        S.cv.wait(lk, [&] { return !S.q.empty() || S.done; });
        if (S.q.empty()) return;
        b = std::move(S.q.front());
        S.q.pop_front();
      }
      S.cv.notify_all();
      const size_t nb = b->rec.size();
      for (size_t i = 0; i < nb; ++i) {
        const int32_t* c = b->cols.data() + b->off[i];
        const size_t d = b->off[i + 1] - b->off[i];
        const uint64_t hsh = b->hash[i];
        size_t mask = S.table.size() - 1, s = (size_t)hsh & mask;
        int32_t cid = -1;
        for (;;) {
          const int32_t t = S.table[s];
          if (t < 0) break;
          if (S.hash[(size_t)t] == hsh && (size_t)(S.ptr[(size_t)t + 1] - S.ptr[(size_t)t]) == d &&
              std::memcmp(S.col.data() + S.ptr[(size_t)t], c, d * sizeof(int32_t)) == 0) { cid = t; break; }
          s = (s + 1) & mask;
        }
        if (cid < 0) {
          cid = (int32_t)S.hash.size();
          S.col.insert(S.col.end(), c, c + d);
          S.ptr.push_back((int64_t)S.col.size());
          S.k.push_back(0);
          S.hash.push_back(hsh);
          S.first_rec.push_back(b->rec[i]);
          S.table[s] = cid;
          if (S.hash.size() * 2 > S.table.size()) {
            const size_t nsz = S.table.size() * 2;
            std::vector<int32_t> nt(nsz, -1);
            for (size_t t = 0; t < S.hash.size(); ++t) {
              size_t z = (size_t)S.hash[t] & (nsz - 1);
              while (nt[z] >= 0) z = (z + 1) & (nsz - 1);
              nt[z] = (int32_t)t;
            }
            S.table.swap(nt);
          }
        }
        else if (b->rec[i] < S.first_rec[(size_t)cid]) S.first_rec[(size_t)cid] = b->rec[i]; /* batches of several builders arrive in any order */
        S.k[(size_t)cid]++;
        if (keep_rec) S.rec_cls.emplace_back(b->rec[i], cid);
      }
    }
  }
  void push(Shard& S) {
    {
      std::unique_lock<std::mutex> lk(S.mu);
      S.cv.wait(lk, [&] { return S.q.size() < 8; }); /* bounded: the parser cannot run away from the workers */
      S.q.push_back(std::move(S.cur));
    }
    S.cv.notify_all();
    S.cur.reset(new Batch());
  }
  void start_workers(int K) {
    const bool keep_rec = layout != LAYOUT_COLLAPSED;
    for (int i = 0; i < K; ++i) {
      shards.emplace_back(new Shard());
      shards.back()->cur.reset(new Batch());
    }
    for (auto& sp : shards) { Shard* S = sp.get(); S->th = std::thread([this, S, keep_rec] { worker(*S, keep_rec); }); }
  }
  /* drain the workers and lay the classes out in first-appearance order (cls_*, rec_class) */
  void merge_shards() {
    for (auto& sp : shards) { if (!sp->cur->rec.empty()) push(*sp); }
    for (auto& sp : shards) { { std::lock_guard<std::mutex> lk(sp->mu); sp->done = true; } sp->cv.notify_all(); }
    for (auto& sp : shards) sp->th.join();
    /* global order = ascending first record.  Every shard sorts its own classes (in parallel), a K-way merge interleaves
     * them, and the copies into the merged arrays run in parallel again: the sequential part is one pass over the classes. */
    const size_t K = shards.size();
    struct Ref { int64_t first; int32_t local; };
    std::vector<std::vector<Ref>> sorted(K);
    {
      std::vector<std::thread> th;
      for (size_t s = 0; s < K; ++s)
        th.emplace_back([&, s] {
          const Shard& S = *shards[s];
          std::vector<Ref>& v = sorted[s];
          v.resize(S.hash.size());
          for (size_t c = 0; c < v.size(); ++c) v[c] = {S.first_rec[c], (int32_t)c};
          std::sort(v.begin(), v.end(), [](const Ref& a, const Ref& b) { return a.first < b.first; });
        });
      for (auto& t : th) t.join();
    }
    size_t total = 0;
    for (size_t s = 0; s < K; ++s) total += sorted[s].size();
    std::vector<int32_t> g_shard(total), g_local(total);
    std::vector<std::vector<int32_t>> l2g(K);
    for (size_t s = 0; s < K; ++s) l2g[s].resize(sorted[s].size());
    cls_ptr.assign(total + 1, 0);
    {
      std::vector<size_t> head(K, 0);
      for (size_t g = 0; g < total; ++g) {
        size_t best = K;
        int64_t bf = 0;
        for (size_t s = 0; s < K; ++s)
          if (head[s] < sorted[s].size() && (best == K || sorted[s][head[s]].first < bf)) { best = s; bf = sorted[s][head[s]].first; }
        const int32_t c = sorted[best][head[best]++].local;
        g_shard[g] = (int32_t)best;
        g_local[g] = c;
        l2g[best][(size_t)c] = (int32_t)g;
        const Shard& S = *shards[best];
        cls_ptr[g + 1] = cls_ptr[g] + (S.ptr[(size_t)c + 1] - S.ptr[(size_t)c]);
      }
    }
    cls_col.resize((size_t)cls_ptr[total]);
    cls_k.resize(total);
    cls_hash.resize(total);
    {
      const int W = (int)std::max<size_t>(1, std::min<size_t>(16, std::thread::hardware_concurrency()));
      auto copy = [&](int w) {
        for (size_t g = total * (size_t)w / (size_t)W; g < total * (size_t)(w + 1) / (size_t)W; ++g) {
          const Shard& S = *shards[(size_t)g_shard[g]];
          const size_t c = (size_t)g_local[g];
          std::memcpy(cls_col.data() + cls_ptr[g], S.col.data() + S.ptr[c], sizeof(int32_t) * (size_t)(S.ptr[c + 1] - S.ptr[c]));
          cls_k[g] = S.k[c];
          cls_hash[g] = S.hash[c];
        }
      };
      std::vector<std::thread> th;
      for (int w = 1; w < W; ++w) th.emplace_back(copy, w);
      copy(0);
      for (auto& t : th) t.join();
    }
    if (layout != LAYOUT_COLLAPSED) {
      /* records were numbered densely over the keyed ones, in stream order; a record belongs to one shard only */
      rec_class.assign((size_t)n_records_keyed, -1);
      std::vector<std::thread> th;
      for (size_t s = 0; s < K; ++s)
        th.emplace_back([&, s] { for (auto& rc : shards[s]->rec_cls) rec_class[(size_t)rc.first] = l2g[s][(size_t)rc.second]; });
      for (auto& t : th) t.join();
    }
    shards.clear();
  }

  void stop_workers() { /* records come one by one with weights: the sequential tables below take over */
    for (auto& sp : shards) { { std::lock_guard<std::mutex> lk(sp->mu); sp->done = true; } sp->cv.notify_all(); }
    for (auto& sp : shards) sp->th.join();
    shards.clear();
  }
  void push_batch(Shard& S, std::unique_ptr<Batch> b) {
    {
      std::unique_lock<std::mutex> lk(S.mu);
      S.cv.wait(lk, [&] { return S.q.size() < 16; });
      S.q.push_back(std::move(b));
    }
    S.cv.notify_all();
  }

  /* Records handed over all at once (the inflated file in memory, or the harness's arrays): W builder threads take
   * contiguous ranges of records and do what add_record() does per record — de-duplication, sort, hash — but in HEADER index
   * space, so that nothing depends on the order in which records are seen; the class keys go to the hash-sharded workers
   * as before.  The numbering the reference derives from the stream order (column = first appearance of the transcript,
   * src/mmseq.cpp:403; class = first appearance of the set, :417-418) is reconstructed afterwards from the smallest
   * (record, position) each transcript was seen at and the smallest record of each class: same result as the sequential
   * walk, checked against it in tests/test_loader.py.
   * acc(r, p, cnt): record r's cnt little-endian uint32 transcript indices at p (unaligned).  Returns 0, or 1 when an index
   * is out of range. */
  template <class Acc>
  int ingest_parallel(int64_t nrec, int64_t T, const Acc& acc, int W) {
    const int K = (int)shards.size();
    const uint64_t NONE = ~0ull;
    std::vector<std::vector<uint64_t>> fa((size_t)W);
    std::vector<std::vector<int32_t>> dh((size_t)W);
    /* weighted: every builder keeps the weights of its (contiguous) record range, in header-sorted member order */
    std::vector<std::vector<float>> bw((size_t)W);
    std::vector<std::vector<int32_t>> bcnt((size_t)W);
    std::atomic<int> bad(0);
    auto build = [&](int w) {
      std::vector<uint64_t>& first = fa[(size_t)w];
      std::vector<int32_t>& dbl = dh[(size_t)w];
      first.assign((size_t)T, NONE);
      dbl.assign((size_t)T, 0);
      std::vector<std::unique_ptr<Batch>> cur((size_t)K);
      for (auto& c : cur) c.reset(new Batch());
      std::vector<int32_t> ids;
      std::vector<std::pair<int32_t, float>> pw;
      const int64_t r0 = nrec * w / W, r1 = nrec * (w + 1) / W;
      if (weighted) { bw[(size_t)w].reserve((size_t)(r1 - r0) * 4); bcnt[(size_t)w].reserve((size_t)(r1 - r0)); }
      for (int64_t r = r0; r < r1; ++r) {
        const uint8_t* p;
        const float* wp = nullptr;
        int cnt;
        acc(r, p, cnt, wp);
        ids.clear();
        if (!weighted) {
          for (int j = 0; j < cnt; ++j) {
            uint32_t v;
            memcpy(&v, p + 4 * (size_t)j, 4);
            if (v >= (uint32_t)T) { bad.store(1); return; }
            if (first[v] == NONE) first[v] = ((uint64_t)r << 24) | (uint64_t)std::min(j, 0xffffff);
            bool dup = false;
            if (ids.size() <= 32) {
              for (int32_t e : ids) if (e == (int32_t)v) { dup = true; break; }
              if (dup) { dbl[v]++; continue; } /* src/mmseq.cpp:404-409 */
            }
            ids.push_back((int32_t)v);
          }
          std::sort(ids.begin(), ids.end());
          if (ids.size() > 33) { /* long records: duplicates removed after the sort */
            size_t o = 1;
            for (size_t j = 1; j < ids.size(); ++j) {
              if (ids[j] == ids[o - 1]) dbl[(size_t)ids[j]]++;
              else ids[o++] = ids[j];
            }
            ids.resize(o);
          }
        } else {
          /* (transcript, weight) pairs; a repeated transcript adds its weight to the first occurrence, in record order */
          pw.clear();
          for (int j = 0; j < cnt; ++j) {
            uint32_t v;
            float wj;
            memcpy(&v, p + 4 * (size_t)j, 4);
            memcpy(&wj, (const uint8_t*)wp + 4 * (size_t)j, 4);
            if (v >= (uint32_t)T) { bad.store(1); return; }
            if (!(wj >= 0.f) || !std::isfinite(wj)) { bad.store(2); return; }
            if (first[v] == NONE) first[v] = ((uint64_t)r << 24) | (uint64_t)std::min(j, 0xffffff);
            bool dup = false;
            for (auto& e : pw) if (e.first == (int32_t)v) { dup = true; e.second += wj; break; }
            if (dup) dbl[v]++;
            else pw.emplace_back((int32_t)v, wj);
          }
          std::sort(pw.begin(), pw.end(), [](const std::pair<int32_t, float>& a, const std::pair<int32_t, float>& b) { return a.first < b.first; });
          for (auto& e : pw) { ids.push_back(e.first); bw[(size_t)w].push_back(e.second); }
          bcnt[(size_t)w].push_back((int32_t)pw.size());
        }
        uint64_t hsh = 0x9e3779b97f4a7c15ull ^ (uint64_t)ids.size();
        for (int32_t e : ids) hsh = mix64(hsh ^ (uint64_t)(uint32_t)e) + 0x632be59bd9b4e019ull;
        const int sh = (int)((hsh >> 40) % (uint64_t)K);
        Batch& B = *cur[(size_t)sh];
        B.rec.push_back(r);
        B.hash.push_back(hsh);
        B.cols.insert(B.cols.end(), ids.begin(), ids.end());
        B.off.push_back((uint32_t)B.cols.size());
        if (B.rec.size() >= BATCH_RECORDS) {
          push_batch(*shards[(size_t)sh], std::move(cur[(size_t)sh]));
          cur[(size_t)sh].reset(new Batch());
        }
      }
      for (int sh = 0; sh < K; ++sh)
        if (!cur[(size_t)sh]->rec.empty()) push_batch(*shards[(size_t)sh], std::move(cur[(size_t)sh]));
    };
    const double tb0 = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    {
      std::vector<std::thread> th;
      for (int w = 1; w < W; ++w) th.emplace_back(build, w);
      build(0);
      for (auto& t : th) t.join();
    }
    if (getenv("MMQ_LOADER_TIMING")) fprintf(stderr, "[loader]   builders done after %.2f s\n", std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count() - tb0);
    N += nrec;
    n_records_keyed += nrec;
    const bool tm = getenv("MMQ_LOADER_TIMING") != nullptr;
    auto clk = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double tb = clk();
    merge_shards(); /* classes in order of their first record, members still header indices */
    if (tm) fprintf(stderr, "[loader]   %d builders + %d class-table workers; drain + merge %.2f s\n", W, K, clk() - tb);
    if (bad.load()) return bad.load();
    /* columns: transcripts in order of first appearance */
    const bool identity = identity_cols;
    std::vector<uint64_t>& first = fa[0];
    for (int w = 1; w < W; ++w)
      for (int64_t h = 0; h < T; ++h) first[(size_t)h] = std::min(first[(size_t)h], fa[(size_t)w][(size_t)h]);
    if (!identity) {
      std::vector<int32_t> seen;
      for (int64_t h = 0; h < T; ++h) if (first[(size_t)h] != NONE) seen.push_back((int32_t)h);
      std::sort(seen.begin(), seen.end(), [&](int32_t a, int32_t b) { return first[(size_t)a] < first[(size_t)b]; });
      col2hdr = seen;
      doublehits.assign(seen.size(), 0);
      for (size_t c = 0; c < seen.size(); ++c) hdr2col[(size_t)seen[c]] = (int32_t)c;
    }
    for (int w = 0; w < W; ++w)
      for (int64_t h = 0; h < T; ++h)
        if (dh[(size_t)w][(size_t)h]) doublehits[(size_t)hdr2col[(size_t)h]] += dh[(size_t)w][(size_t)h];
    /* members: header index -> column, ascending again (the reference sorts the column indices, :412); weighted: where
     * each member came from, so that every record's weights can follow */
    const int64_t C = (int64_t)cls_hash.size();
    std::vector<int32_t> perm; /* [entry of cls_col] position of that member in the header-sorted class */
    if (weighted) perm.resize(cls_col.size());
    if (!identity) {
      auto renum = [&](int w) {
        std::vector<std::pair<int32_t, int32_t>> tmp;
        for (int64_t c = C * w / W; c < C * (w + 1) / W; ++c) {
          int32_t* b = cls_col.data() + cls_ptr[(size_t)c];
          int32_t* e = cls_col.data() + cls_ptr[(size_t)c + 1];
          for (int32_t* q = b; q < e; ++q) *q = hdr2col[(size_t)*q];
          if (!weighted) { std::sort(b, e); continue; }
          tmp.clear();
          for (int32_t* q = b; q < e; ++q) tmp.emplace_back(*q, (int32_t)(q - b));
          std::sort(tmp.begin(), tmp.end());
          int32_t* pm = perm.data() + cls_ptr[(size_t)c];
          for (size_t j = 0; j < tmp.size(); ++j) { b[j] = tmp[j].first; pm[j] = tmp[j].second; }
        }
      };
      std::vector<std::thread> th;
      for (int w = 1; w < W; ++w) th.emplace_back(renum, w);
      renum(0);
      for (auto& t : th) t.join();
    } else if (weighted) {
      for (int64_t c = 0; c < C; ++c)
        for (int64_t q = cls_ptr[(size_t)c]; q < cls_ptr[(size_t)c + 1]; ++q) perm[(size_t)q] = (int32_t)(q - cls_ptr[(size_t)c]);
    }
    if (weighted) {
      /* the records' weights, in the column order of their class */
      rec_wptr.assign((size_t)nrec + 1, 0);
      {
        int64_t r = 0;
        for (int w = 0; w < W; ++w)
          for (int32_t c : bcnt[(size_t)w]) { rec_wptr[(size_t)r + 1] = rec_wptr[(size_t)r] + c; ++r; }
      }
      rec_w.resize((size_t)rec_wptr[(size_t)nrec]);
      auto place = [&](int w) {
        const int64_t r0 = nrec * w / W, r1 = nrec * (w + 1) / W;
        const float* src = bw[(size_t)w].data();
        for (int64_t r = r0; r < r1; ++r) {
          const int64_t d = rec_wptr[(size_t)r + 1] - rec_wptr[(size_t)r];
          const int32_t* pm = perm.data() + cls_ptr[(size_t)rec_class[(size_t)r]];
          float* dst = rec_w.data() + rec_wptr[(size_t)r];
          for (int64_t j = 0; j < d; ++j) dst[j] = src[pm[j]];
          src += d;
        }
      };
      std::vector<std::thread> th;
      for (int w = 1; w < W; ++w) th.emplace_back(place, w);
      place(0);
      for (auto& t : th) t.join();
    }
    return 0;
  }

  void grow_table() {
    size_t nsz = table.empty() ? (size_t)1 << 16 : table.size() * 2;
    std::vector<int32_t> nt(nsz, -1);
    for (size_t c = 0; c < cls_hash.size(); ++c) {
      size_t s = (size_t)cls_hash[c] & (nsz - 1);
      while (nt[s] >= 0) s = (s + 1) & (nsz - 1);
      nt[s] = (int32_t)c;
    }
    table.swap(nt);
  }
};

ClassBuilder::ClassBuilder(int64_t T, int layout, bool weighted) : p_(new Impl()) {
  p_->layout = layout & 15;
  p_->header_order = (layout & LAYOUT_HEADER_ORDER_COLUMNS) != 0 && !(layout & LAYOUT_IDENTITY_COLUMNS);
  p_->weighted = weighted;
  p_->hdr2col.assign((size_t)T, -1);
  p_->identity_cols = (layout & LAYOUT_IDENTITY_COLUMNS) != 0;
  if (layout & LAYOUT_IDENTITY_COLUMNS) {
    p_->col2hdr.resize((size_t)T);
    p_->doublehits.assign((size_t)T, 0);
    for (int64_t t = 0; t < T; ++t) { p_->hdr2col[(size_t)t] = (int32_t)t; p_->col2hdr[(size_t)t] = (int32_t)t; }
  }
  p_->grow_table();
  {
    /* hash-shard workers (they own the class tables) and, for records handed over all at once, as many builder threads */
    const unsigned hc = std::thread::hardware_concurrency();
    int K = hc >= 8 ? std::min(12, (int)hc / 2) : 3; /* measured on 8 threads: 4 builders + 4 workers 0.91 s, 5 + 3 1.09 s, 6 + 2 1.92 s */
    if (const char* e = getenv("MMQ_LOADER_THREADS")) K = atoi(e);
    if (hc && (int)hc - 2 < K) K = std::max(0, (int)hc - 2);
    if (K > 0) p_->start_workers(K);
    p_->builders = std::max(1, std::min(16, (int)hc - K));
    if (const char* e = getenv("MMQ_LOADER_BUILDERS")) p_->builders = std::max(1, atoi(e));
  }
}
ClassBuilder::~ClassBuilder() {
  if (!p_->shards.empty()) p_->merge_shards();
  delete p_;
}

bool ClassBuilder::parallel_ready() const { return !p_->shards.empty() && p_->N == 0; }
int ClassBuilder::add_records_binary(const uint8_t* base, const uint64_t* off, int64_t nrec) {
  Impl& P = *p_;
  const bool wt = P.weighted;
  auto acc = [base, off, wt](int64_t r, const uint8_t*& p, int& cnt, const float*& w) {
    uint32_t c;
    memcpy(&c, base + off[r], 4);
    cnt = (int)c;
    p = base + off[r] + 4;
    w = wt ? (const float*)(p + 4 * (size_t)c) : nullptr; /* schema 2: the weights follow the indices (unaligned: read with memcpy) */
  };
  return P.ingest_parallel(nrec, (int64_t)P.hdr2col.size(), acc, P.builders);
}
int ClassBuilder::add_records_csr(const int64_t* frag_ptr, const int32_t* frag_tid, const float* frag_w, int64_t nrec) {
  Impl& P = *p_;
  auto acc = [frag_ptr, frag_tid, frag_w](int64_t r, const uint8_t*& p, int& cnt, const float*& w) {
    cnt = (int)(frag_ptr[r + 1] - frag_ptr[r]);
    p = (const uint8_t*)(frag_tid + frag_ptr[r]);
    w = frag_w ? frag_w + frag_ptr[r] : nullptr;
  };
  return P.ingest_parallel(nrec, (int64_t)P.hdr2col.size(), acc, P.builders);
}

void ClassBuilder::add_record(const int32_t* tids, const float* w, int cnt) {
  Impl& P = *p_;
  if (P.weighted && !P.shards.empty()) P.stop_workers();
  P.N++;
  auto& comb = P.comb;
  comb.clear();
  for (int j = 0; j < cnt; ++j) {
    const int32_t h = tids[j];
    int32_t c = P.hdr2col[(size_t)h];
    if (c < 0) { /* first appearance: new column (src/mmseq.cpp:403) */
      c = (int32_t)P.col2hdr.size();
      P.hdr2col[(size_t)h] = c;
      P.col2hdr.push_back(h);
      P.doublehits.push_back(0);
    }
    bool dup = false;
    for (auto& e : comb)
      if (e.first == c) { dup = true; if (w) e.second += w[j]; break; }
    if (dup) P.doublehits[(size_t)c]++; /* :404-409 */
    else comb.emplace_back(c, w ? w[j] : 1.0f);
  }
  if (comb.empty()) return; /* a record without hits adds to N only */
  std::sort(comb.begin(), comb.end(), [](const std::pair<int32_t, float>& a, const std::pair<int32_t, float>& b) { return a.first < b.first; });
  uint64_t hsh = 0x9e3779b97f4a7c15ull ^ (uint64_t)comb.size();
  for (auto& e : comb) hsh = mix64(hsh ^ (uint64_t)(uint32_t)e.first) + 0x632be59bd9b4e019ull;
  if (!P.shards.empty()) { /* parallel ingestion: the table work happens in the shard's worker */
    Impl::Shard& S = *P.shards[(size_t)((hsh >> 40) % P.shards.size())];
    Impl::Batch& B = *S.cur;
    B.rec.push_back(P.n_records_keyed++);
    B.hash.push_back(hsh);
    for (auto& e : comb) B.cols.push_back(e.first);
    B.off.push_back((uint32_t)B.cols.size());
    if (B.rec.size() >= Impl::BATCH_RECORDS) P.push(S);
    return;
  }
  size_t mask = P.table.size() - 1;
  size_t s = (size_t)hsh & mask;
  int32_t cid = -1;
  for (;;) {
    const int32_t c = P.table[s];
    if (c < 0) break;
    if (P.cls_hash[(size_t)c] == hsh) {
      const int64_t b = P.cls_ptr[(size_t)c], e = P.cls_ptr[(size_t)c + 1];
      if (e - b == (int64_t)comb.size()) {
        bool same = true;
        for (size_t j = 0; j < comb.size(); ++j)
          if (P.cls_col[(size_t)b + j] != comb[j].first) { same = false; break; }
        if (same) { cid = c; break; }
      }
    }
    s = (s + 1) & mask;
  }
  if (cid < 0) { /* new class, index = order of first appearance (:417-418) */
    cid = (int32_t)P.cls_hash.size();
    for (auto& e : comb) P.cls_col.push_back(e.first);
    P.cls_ptr.push_back((int64_t)P.cls_col.size());
    P.cls_k.push_back(0);
    P.cls_hash.push_back(hsh);
    P.table[s] = cid;
    if (P.cls_hash.size() * 2 > P.table.size()) P.grow_table();
  }
  P.cls_k[(size_t)cid]++; /* :440 */
  if (P.layout != LAYOUT_COLLAPSED) {
    P.rec_class.push_back(cid);
    if (P.weighted) {
      for (auto& e : comb) P.rec_w.push_back(e.second);
      P.rec_wptr.push_back((int64_t)P.rec_w.size());
    }
  }
}

void ClassBuilder::finish(HitClasses& out) {
  Impl& P = *p_;
  const bool tm = getenv("MMQ_LOADER_TIMING") != nullptr;
  auto clk = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double t_last = clk();
  auto tick = [&](const char* what) { if (tm) { const double t = clk(); fprintf(stderr, "[loader]   finish: %-28s %.2f s\n", what, t - t_last); t_last = t; } };
  if (!P.shards.empty()) P.merge_shards();
  if (P.header_order) {
    /* renumber the observed transcripts by header index; members of a class stay ascending */
    const int64_t n0 = (int64_t)P.col2hdr.size();
    std::vector<int32_t> by((size_t)n0), newcol((size_t)n0);
    for (int64_t c = 0; c < n0; ++c) by[(size_t)c] = (int32_t)c;
    std::sort(by.begin(), by.end(), [&](int32_t a, int32_t b) { return P.col2hdr[(size_t)a] < P.col2hdr[(size_t)b]; });
    for (int64_t i = 0; i < n0; ++i) newcol[(size_t)by[(size_t)i]] = (int32_t)i;
    std::vector<int32_t> c2h((size_t)n0), dh((size_t)n0);
    for (int64_t c = 0; c < n0; ++c) { c2h[(size_t)newcol[(size_t)c]] = P.col2hdr[(size_t)c]; dh[(size_t)newcol[(size_t)c]] = P.doublehits[(size_t)c]; }
    P.col2hdr.swap(c2h);
    P.doublehits.swap(dh);
    for (size_t hI = 0; hI < P.hdr2col.size(); ++hI) if (P.hdr2col[hI] >= 0) P.hdr2col[hI] = newcol[(size_t)P.hdr2col[hI]];
    const int64_t C = (int64_t)P.cls_hash.size();
    const int W = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    auto par = [&](int64_t count, const std::function<void(int64_t, int64_t)>& body) { /* body(begin, end) on W threads */
      std::vector<std::thread> th;
      for (int w = 1; w < W; ++w) th.emplace_back([&, w] { body(count * w / W, count * (w + 1) / W); });
      body(0, count / W);
      for (auto& t : th) t.join();
    };
    std::vector<int32_t> perm; /* weighted: [entry of cls_col] old position of the member now at that place */
    if (P.weighted) perm.resize(P.cls_col.size());
    par(C, [&](int64_t c0, int64_t c1) {
      std::vector<std::pair<int32_t, int32_t>> tmp; /* (new column, old position) */
      for (int64_t c = c0; c < c1; ++c) {
        const int64_t b = P.cls_ptr[(size_t)c], e = P.cls_ptr[(size_t)c + 1];
        tmp.clear();
        for (int64_t q = b; q < e; ++q) tmp.emplace_back(newcol[(size_t)P.cls_col[(size_t)q]], (int32_t)(q - b));
        std::sort(tmp.begin(), tmp.end());
        for (int64_t q = b; q < e; ++q) P.cls_col[(size_t)q] = tmp[(size_t)(q - b)].first;
        if (P.weighted) for (int64_t q = b; q < e; ++q) perm[(size_t)q] = tmp[(size_t)(q - b)].second;
      }
    });
    if (P.weighted)
      par((int64_t)P.rec_class.size(), [&](int64_t r0, int64_t r1) {
        std::vector<float> t2;
        for (int64_t r = r0; r < r1; ++r) {
          const int64_t cb = P.cls_ptr[(size_t)P.rec_class[(size_t)r]];
          const size_t d = (size_t)(P.cls_ptr[(size_t)P.rec_class[(size_t)r] + 1] - cb);
          float* wr = P.rec_w.data() + P.rec_wptr[(size_t)r];
          t2.assign(wr, wr + d);
          for (size_t j = 0; j < d; ++j) wr[j] = t2[(size_t)perm[(size_t)cb + j]];
        }
      });
  }
  tick("header-order renumbering");
  out.layout = P.layout;
  out.N = P.N;
  out.n = (int64_t)P.col2hdr.size();
  out.n_classes = (int64_t)P.cls_hash.size();
  out.col2hdr = P.col2hdr;
  out.hdr2col = P.hdr2col;
  out.doublehits = P.doublehits;
  out.w.clear();
  out.set_ptr.clear(); out.set_col.clear(); out.set_k.clear();
  out.first_zero_weight_record = -1;
  if (P.layout == LAYOUT_COLLAPSED) {
    out.m = out.n_classes;
    out.row_ptr.swap(P.cls_ptr);
    out.col.swap(P.cls_col);
    out.k.swap(P.cls_k);
    return;
  }
  const int64_t R = (int64_t)P.rec_class.size();
  std::vector<int64_t> order((size_t)R);
  if (P.layout == LAYOUT_PER_FRAGMENT_SORTED || P.layout == LAYOUT_PER_FRAGMENT_BY_LENGTH) {
    /* stable counting sort of records by class, classes ranked by (size,) first appearance */
    std::vector<int64_t> rank((size_t)out.n_classes);
    for (int64_t c = 0; c < out.n_classes; ++c) rank[(size_t)c] = c;
    if (P.layout == LAYOUT_PER_FRAGMENT_BY_LENGTH) {
      std::vector<int64_t> by((size_t)out.n_classes);
      for (int64_t c = 0; c < out.n_classes; ++c) by[(size_t)c] = c;
      /* by class size, then by the member columns lexicographically: neighbouring rows gather
       * the same or neighbouring mu entries */
      auto less = [&](int64_t a, int64_t b) {
        const int64_t da = P.cls_ptr[(size_t)a + 1] - P.cls_ptr[(size_t)a], db = P.cls_ptr[(size_t)b + 1] - P.cls_ptr[(size_t)b];
        if (da != db) return da < db;
        const int32_t* pa = P.cls_col.data() + P.cls_ptr[(size_t)a];
        const int32_t* pb = P.cls_col.data() + P.cls_ptr[(size_t)b];
        for (int64_t j = 0; j < da; ++j)
          if (pa[j] != pb[j]) return pa[j] < pb[j];
        return a < b; /* distinct classes never tie; a total order anyway */
      };
      {
        /* sorted chunks on all threads, then pairwise merges */
        const int64_t nC = out.n_classes;
        int W = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        while (W > 1 && nC / W < 64) W /= 2;
        std::vector<int64_t> cut((size_t)W + 1);
        for (int w = 0; w <= W; ++w) cut[(size_t)w] = nC * w / W;
        {
          std::vector<std::thread> th;
          for (int w = 0; w < W; ++w) th.emplace_back([&, w] { std::sort(by.begin() + cut[(size_t)w], by.begin() + cut[(size_t)w + 1], less); });
          for (auto& t : th) t.join();
        }
        for (int step = 1; step < W; step *= 2) {
          std::vector<std::thread> th;
          for (int w = 0; w + step < W; w += 2 * step)
            th.emplace_back([&, w, step] {
              std::inplace_merge(by.begin() + cut[(size_t)w], by.begin() + cut[(size_t)(w + step)], by.begin() + cut[(size_t)std::min(W, w + 2 * step)], less);
            });
          for (auto& t : th) t.join();
        }
      }
      for (int64_t i = 0; i < out.n_classes; ++i) rank[(size_t)by[(size_t)i]] = i;
      tick("classes by size and members");
    }
    std::vector<int64_t> start((size_t)out.n_classes + 1, 0);
    for (int64_t r = 0; r < R; ++r) start[(size_t)rank[(size_t)P.rec_class[(size_t)r]] + 1]++;
    for (int64_t c = 0; c < out.n_classes; ++c) start[(size_t)c + 1] += start[(size_t)c];
    for (int64_t r = 0; r < R; ++r) order[(size_t)start[(size_t)rank[(size_t)P.rec_class[(size_t)r]]]++] = r;
  } else {
    for (int64_t r = 0; r < R; ++r) order[(size_t)r] = r;
  }
  tick("records by class");
  out.m = R;
  out.k.clear();
  out.row_ptr.assign((size_t)R + 1, 0);
  int64_t total = 0;
  for (int64_t i = 0; i < R; ++i) {
    const int32_t c = P.rec_class[(size_t)order[(size_t)i]];
    total += P.cls_ptr[(size_t)c + 1] - P.cls_ptr[(size_t)c];
    out.row_ptr[(size_t)i + 1] = total;
  }
  tick("row pointers");
  out.col.resize((size_t)total);
  if (P.weighted) out.w.resize((size_t)total);
  {
    const int W = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<int64_t> zero_rec((size_t)W, R); /* per thread: first record whose weights are all zero */
    auto copy = [&](int w) {
      for (int64_t i = R * w / W; i < R * (w + 1) / W; ++i) {
        const int64_t r = order[(size_t)i];
        const int32_t c = P.rec_class[(size_t)r];
        const int64_t b = P.cls_ptr[(size_t)c], d = P.cls_ptr[(size_t)c + 1] - b;
        std::memcpy(out.col.data() + out.row_ptr[(size_t)i], P.cls_col.data() + b, sizeof(int32_t) * (size_t)d);
        if (P.weighted) {
          const float* wr = P.rec_w.data() + P.rec_wptr[(size_t)r];
          std::memcpy(out.w.data() + out.row_ptr[(size_t)i], wr, sizeof(float) * (size_t)d);
          if (r < zero_rec[(size_t)w] && std::all_of(wr, wr + d, [](float x) { return x == 0.f; })) zero_rec[(size_t)w] = r;
        }
      }
    };
    std::vector<std::thread> th;
    for (int w = 1; w < W; ++w) th.emplace_back(copy, w);
    copy(0);
    for (auto& t : th) t.join();
    const int64_t z = *std::min_element(zero_rec.begin(), zero_rec.end());
    if (z < R) out.first_zero_weight_record = z;
  }
  tick("rows copied");
  /* the sets the rows were built from, for what is defined per set (.k, .M, unique hits) */
  out.set_ptr.swap(P.cls_ptr);
  out.set_col.swap(P.cls_col);
  out.set_k.swap(P.cls_k);
}

/* ------------------------------------------------------------------ header */

int validate_header(const HitsHeader& hdr, std::string& err) {
  /* src/mmseq.cpp:342-379 */
  const size_t T = hdr.names.size();
  {
    std::vector<std::string> s = hdr.names;
    std::sort(s.begin(), s.end());
    if (std::unique(s.begin(), s.end()) != s.end()) { err = "Error: duplicate transcripts in @TranscriptMetaData entries."; return 1; }
  }
  std::vector<int> seen(T, 0);
  for (size_t g = 0; g < hdr.gene_members.size(); ++g)
    for (int32_t h : hdr.gene_members[g]) {
      if (seen[(size_t)h]) { err = "Error: transcripts must be nested within genes in GeneIsoforms metadata."; return 1; }
      seen[(size_t)h] = 1;
    }
  for (size_t t = 0; t < T; ++t)
    if (!seen[t]) { err = "Error: " + hdr.names[t] + " does not belong to a gene in the @GeneIsoforms header entries."; return 1; }
  return 0;
}

namespace {

struct NameIndex {
  std::unordered_map<std::string, int32_t> map;
  int32_t find(const std::string& s) const {
    auto it = map.find(s);
    return it == map.end() ? -1 : it->second;
  }
  /* allocation-free lookup for the record loop of the text schema (one call per alignment):
   * open addressing over FNV-1a, names compared in place */
  const std::vector<std::string>* names = nullptr;
  std::vector<uint32_t> slots; /* header index + 1, 0 = empty */
  static uint64_t fnv(const char* p, size_t n) {
    uint64_t h = 0xcbf29ce484222325ull;
    for (size_t i = 0; i < n; ++i) { h ^= (unsigned char)p[i]; h *= 0x100000001b3ull; }
    return h ^ (h >> 29);
  }
  void build_fast(const std::vector<std::string>& nm) {
    names = &nm;
    size_t sz = 64;
    while (sz < nm.size() * 2 + 8) sz <<= 1;
    slots.assign(sz, 0);
    for (size_t i = 0; i < nm.size(); ++i) {
      size_t s = (size_t)fnv(nm[i].data(), nm[i].size()) & (sz - 1);
      bool dup = false;
      while (slots[s]) { if ((*names)[slots[s] - 1] == nm[i]) { dup = true; break; } s = (s + 1) & (sz - 1); }
      if (!dup) slots[s] = (uint32_t)i + 1; /* first wins, as map::insert */
    }
  }
  int32_t find_fast(const char* p, size_t n) const {
    const size_t mask = slots.size() - 1;
    size_t s = (size_t)fnv(p, n) & mask;
    while (slots[s]) {
      const std::string& cand = (*names)[slots[s] - 1];
      if (cand.size() == n && memcmp(cand.data(), p, n) == 0) return (int32_t)slots[s] - 1;
      s = (s + 1) & mask;
    }
    return -1;
  }
};

int finish_header(HitsHeader& hdr, const std::vector<std::pair<std::string, std::vector<std::string>>>& genes_raw,
                  const std::vector<std::vector<std::string>>& ident_raw, NameIndex& idx, std::string& err) {
  for (size_t t = 0; t < hdr.names.size(); ++t) idx.map.emplace(hdr.names[t], (int32_t)t); /* first wins, as map::insert */
  std::map<std::string, std::vector<std::string>> gmap; /* std::map: byte-wise order, insert keeps the first */
  for (auto& g : genes_raw) gmap.insert(g);
  hdr.gene_of.assign(hdr.names.size(), -1);
  for (auto& g : gmap) {
    std::vector<int32_t> mem;
    for (auto& nm : g.second) {
      int32_t h = idx.find(nm);
      if (h < 0) { err = "Error: transcript '" + nm + "' of gene '" + g.first + "' has no @TranscriptMetaData entry."; return 1; }
      mem.push_back(h);
      if (hdr.gene_of[(size_t)h] < 0) hdr.gene_of[(size_t)h] = (int32_t)hdr.gene_names.size();
    }
    hdr.gene_names.push_back(g.first);
    hdr.gene_members.push_back(mem);
  }
  for (auto& s : ident_raw) {
    std::vector<int32_t> mem;
    for (auto& nm : s) {
      int32_t h = idx.find(nm);
      if (h < 0) { err = "Error: transcript '" + nm + "' in @IdenticalTranscripts has no @TranscriptMetaData entry."; return 1; }
      mem.push_back(h);
    }
    hdr.identical.push_back(mem);
  }
  return validate_header(hdr, err);
}

double parse_double_like_istream(const std::string& s) { /* string_to_double, src/hitsio.cpp:14-20 */
  std::istringstream i(s);
  double x;
  if (!(i >> x)) return 0;
  return x;
}

}  // namespace

int load_hits_file(const std::string& path, int layout, HitsHeader& hdr, HitClasses& cls, std::string& err, int weighted_layout) {
  ByteSource src;
  const double t_open0 = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
  if (!src.open(path)) { err = "Error reading hits file \"" + path + "\"."; return 1; }
  hdr = HitsHeader();
  std::vector<std::pair<std::string, std::vector<std::string>>> genes_raw;
  std::vector<std::vector<std::string>> ident_raw;
  NameIndex idx;
  std::string line;
  /* schema detection on the first line, src/hitsio.cpp:261-275 */
  if (!src.getline(line)) { err = "Input file \"" + path + "\" does not seem to be a hits file."; return 1; }
  {
    std::istringstream tok(line);
    std::string t1;
    tok >> t1;
    if (t1 == "@TranscriptMetaData") hdr.schema = 0;
    else if (line == "MMSEQ_HITSFILE") {
      /* schema 1: the reference's binary format (src/hitsio.cpp:403-410 accepts nothing else); schema 2 (this
       * package's extension, SURVEY section 8 f4): the same stream with one fp32 weight per hit after a record's
       * transcript indices — likelihood x insert-size x bias weight of the alignment, what bam2hits computes and then
       * throws away (src/bam2hits.cpp:778-801, :992-1003) */
      uint32_t s = 99;
      if (!src.read_u32(s) || (s != 1 && s != 2)) { err = "Input file \"" + path + "\" does not seem to be a hits file."; return 1; }
      hdr.schema = (int)s;
    } else { err = "Input file \"" + path + "\" does not seem to be a hits file."; return 1; }
  }
  if (hdr.schema == 0) {
    /* text header, src/hitsio.cpp:286-329; `line` already holds the first header line */
    bool have_line = true;
    for (;;) {
      if (!have_line) {
        int c = src.peek();
        if (c == EOF || c == '>') break;
        if (!src.getline(line)) break;
      }
      have_line = false;
      std::istringstream tok(line);
      std::string t1;
      tok >> t1;
      if (t1 == "@TranscriptMetaData") {
        std::string nm; double el = 0; int tl = 0;
        tok >> nm >> el >> tl;
        hdr.names.push_back(nm);
        hdr.efflen.push_back(el);
        hdr.truelen.push_back(tl);
      } else if (t1 == "@GeneIsoforms") {
        std::string gid, tid;
        std::vector<std::string> mem;
        tok >> gid;
        while (tok >> tid) mem.push_back(tid);
        genes_raw.emplace_back(gid, mem);
      } else if (t1 == "@IdenticalTranscripts") {
        std::string tid;
        std::vector<std::string> mem;
        while (tok >> tid) mem.push_back(tid);
        ident_raw.push_back(mem);
      } else { err = "Hits file looks malformed."; return 1; }
    }
  } else {
    /* binary header, src/hitsio.cpp:349-398 */
    uint32_t T = 0;
    if (!src.read_u32(T)) { err = "Hits file looks malformed."; return 1; }
    for (uint32_t i = 0; i < T; ++i) {
      std::string nm, el; uint32_t tl = 0;
      if (!src.getline(nm) || !src.getline(el) || !src.read_u32(tl)) { err = "Hits file looks malformed."; return 1; }
      hdr.names.push_back(nm);
      hdr.efflen.push_back(parse_double_like_istream(el));
      hdr.truelen.push_back((int32_t)tl);
    }
    uint32_t G = 0;
    if (!src.read_u32(G)) { err = "Hits file looks malformed."; return 1; }
    for (uint32_t g = 0; g < G; ++g) {
      std::string gid; uint32_t c = 0;
      if (!src.getline(gid) || !src.read_u32(c)) { err = "Hits file looks malformed."; return 1; }
      std::vector<std::string> mem;
      for (uint32_t j = 0; j < c; ++j) { std::string nm; if (!src.getline(nm)) { err = "Hits file looks malformed."; return 1; } mem.push_back(nm); }
      genes_raw.emplace_back(gid, mem);
    }
    uint32_t I = 0;
    if (!src.read_u32(I)) { err = "Hits file looks malformed."; return 1; }
    for (uint32_t s = 0; s < I; ++s) {
      uint32_t c = 0;
      if (!src.read_u32(c)) { err = "Hits file looks malformed."; return 1; }
      std::vector<std::string> mem;
      for (uint32_t j = 0; j < c; ++j) { std::string nm; if (!src.getline(nm)) { err = "Hits file looks malformed."; return 1; } mem.push_back(nm); }
      ident_raw.push_back(mem);
    }
  }
  /* the binary header may repeat a name: the reference's maps keep the first entry but
   * headerTranscriptName keeps every slot, so record indices address the full list */
  std::vector<std::string> all_names = hdr.names;
  if (finish_header(hdr, genes_raw, ident_raw, idx, err)) return 1;
  const int64_t T = (int64_t)hdr.names.size();
  const bool timing = getenv("MMQ_LOADER_TIMING") != nullptr;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  const double t_hdr = now();
  if (timing) fprintf(stderr, "[loader] open%s + header %.2f s\n", src.whole() ? " (file inflated on all threads)" : "", t_hdr - t_open0);
  if (hdr.schema == 2 && weighted_layout >= 0) layout = weighted_layout;
  if (hdr.schema == 2 && (layout & 15) == LAYOUT_COLLAPSED) {
    err = "Error: \"" + path + "\" carries per-hit weights (schema 2): it needs a per-fragment layout.";
    return 1;
  }
  ClassBuilder cb(T, layout, hdr.schema == 2);
  std::vector<int32_t> tids;
  std::vector<float> wts;
  if (hdr.schema == 0) {
    /* records, src/hitsio.cpp:331-347 */
    idx.build_fast(hdr.names);
    const char* lp; size_t ln;
    for (;;) {
      if (src.peek() == EOF) break;
      if (!src.getline_view(lp, ln)) break;
      if (ln == 0 || lp[0] != '>') { err = "Hits file looks malformed."; return 1; }
      if (src.peek() == EOF) {
        fprintf(stderr, "Warning: read record without any mapping transcripts found at the end of the hits file. The hits file may be corrupted.\n");
        break;
      }
      tids.clear();
      while (src.peek() != EOF && src.peek() != '>') {
        if (!src.getline_view(lp, ln)) break;
        int32_t h = idx.find_fast(lp, ln);
        if (h < 0) { err = "Error: transcript '" + std::string(lp, ln) + "' has no length."; return 1; } /* src/mmseq.cpp:599-601 */
        tids.push_back(h);
      }
      if (tids.empty()) { /* the reference would open a hit class with no transcripts (src/mmseq.cpp:401-440): refused here */
        err = "Error: a read record without any mapping transcripts in the hits file.";
        return 1;
      }
      cb.add_record(tids.data(), nullptr, (int)tids.size());
    }
  } else {
    /* records, src/hitsio.cpp:413-439; read names are delta-coded (:101-115) and unused here */
    std::string mid;
    if (src.whole() && cb.parallel_ready() && !getenv("MMQ_LOADER_SERIAL_RECORDS")) {
      /* the inflated file is in memory: one cheap sequential walk finds where each record's hit list starts (the delta-coded
       * names make record boundaries sequential), the rest — de-duplication, sort, hash, class tables — runs on all threads */
      const uint8_t* b = (const uint8_t*)src.whole_base();
      const size_t end = src.whole_size();
      size_t p = src.whole_pos();
      const std::string malformed = "Hits file looks malformed.";
      std::vector<uint64_t> off;
      off.reserve((end - p) / 24 + 16);
      const uint32_t Tn = (uint32_t)all_names.size();
      auto line_end = [&](size_t q) { while (q < end && b[q] != '\n') ++q; return q; }; /* names are a few bytes: no memchr call */
      auto small = [&](size_t& q) { /* one byte, or 0xFF + uint32 (src/hitsio.cpp:36-55) */
        if (q >= end) return false;
        if (b[q] == 255) { if (q + 5 > end) return false; q += 5; } else q += 1;
        return true;
      };
      while (p < end) {
        size_t nl = line_end(p);
        if (nl == p) { /* empty line: delta form */
          ++p;
          if (!small(p)) { err = malformed; return 1; }
          nl = line_end(p);
          if (nl >= end) { err = malformed; return 1; }
          p = nl + 1;
          if (!small(p)) { err = malformed; return 1; }
        } else {
          p = nl < end ? nl + 1 : end;
        }
        if (p + 4 > end) { err = malformed; return 1; }
        uint32_t cnt;
        memcpy(&cnt, b + p, 4);
        if (cnt == 0) { err = "Error: a read record without any mapping transcripts in the hits file."; return 1; }
        const size_t per_hit = hdr.schema == 2 ? 8 : 4; /* schema 2: one fp32 weight per hit after the indices */
        if (cnt > Tn || p + 4 + per_hit * (size_t)cnt > end) { err = malformed; return 1; }
        off.push_back((uint64_t)p);
        p += 4 + per_hit * (size_t)cnt;
      }
      const double t_scan = now();
      if (int brc = cb.add_records_binary(b, off.data(), (int64_t)off.size())) {
        err = brc == 2 ? "Error: per-hit weights must be finite and non-negative." : malformed;
        return 1;
      }
      const double t_rec = now();
      cb.finish(cls);
      if (timing) fprintf(stderr, "[loader] record walk %.2f s, classes (parallel) %.2f s, finish (layout) %.2f s\n", t_scan - t_hdr, t_rec - t_scan, now() - t_rec);
      return 0;
    }
    for (;;) {
      const char* lp; size_t ln;
      if (!src.getline_view(lp, ln)) break;
      /* the stream may end between records only: anything missing inside one is a malformed (truncated) file */
      const std::string malformed = "Hits file looks malformed.";
      if (ln == 0) {
        uint32_t nb = 0, ne = 0;
        if (!src.read_small(nb) || !src.getline_view(lp, ln) || !src.read_small(ne)) { err = src.corrupt() ? "Error: zlib stream of \"" + path + "\" is corrupt." : malformed; return 1; }
      }
      uint32_t cnt = 0;
      if (!src.read_u32(cnt)) { err = src.corrupt() ? "Error: zlib stream of \"" + path + "\" is corrupt." : malformed; return 1; }
      if (cnt == 0) { err = "Error: a read record without any mapping transcripts in the hits file."; return 1; }
      if (cnt > (uint32_t)all_names.size()) { err = malformed; return 1; } /* more hits than transcripts: not a count */
      tids.resize(cnt);
      for (uint32_t j = 0; j < cnt; ++j) {
        uint32_t v = 0;
        if (!src.read_u32(v)) { err = src.corrupt() ? "Error: zlib stream of \"" + path + "\" is corrupt." : malformed; return 1; }
        if (v >= (uint32_t)all_names.size()) { err = malformed; return 1; }
        tids[j] = (int32_t)v;
      }
      if (hdr.schema == 2) {
        wts.resize(cnt);
        if (!src.read_bytes(wts.data(), sizeof(float) * cnt)) { err = src.corrupt() ? "Error: zlib stream of \"" + path + "\" is corrupt." : malformed; return 1; }
        for (uint32_t j = 0; j < cnt; ++j)
          if (!(wts[j] >= 0.f) || !std::isfinite(wts[j])) { err = "Error: per-hit weights must be finite and non-negative."; return 1; }
      }
      cb.add_record(tids.data(), hdr.schema == 2 ? wts.data() : nullptr, (int)cnt);
    }
  }
  if (src.corrupt()) { err = "Error: zlib stream of \"" + path + "\" is corrupt."; return 1; }
  const double t_rec = now();
  cb.finish(cls);
  if (timing) fprintf(stderr, "[loader] records %.2f s, finish (merge + layout) %.2f s\n", t_rec - t_hdr, now() - t_rec);
  return 0;
}

int scaled_lengths(const HitsHeader& hdr, const HitClasses& cls, std::vector<double>& l, std::string& err) {
  l.resize((size_t)cls.n);
  for (int64_t t = 0; t < cls.n; ++t) {
    const int32_t h = cls.col2hdr[(size_t)t];
    l[(size_t)t] = hdr.efflen[(size_t)h] * (double)cls.N / 1000000000.0;
    if (l[(size_t)t] <= 0) { err = "Error: transcript '" + hdr.names[(size_t)h] + "' has a length of zero."; return 1; }
  }
  return 0;
}

}  // namespace mmq

/* ---------------------------------------------------------------- C ABI
 * (for the Python harness; the host program links the C++ API directly) */
extern "C" {

struct mmqh_hits {
  mmq::HitsHeader hdr;
  mmq::HitClasses cls;
  std::vector<int64_t> gene_ptr, ident_ptr;
  std::vector<int32_t> gene_mem, ident_mem;
};

static void set_err(char* err, int errlen, const std::string& s) {
  if (err && errlen > 0) { snprintf(err, (size_t)errlen, "%s", s.c_str()); }
}

static void flatten(mmqh_hits* H) {
  H->gene_ptr.assign(1, 0);
  for (auto& g : H->hdr.gene_members) { for (int32_t h : g) H->gene_mem.push_back(h); H->gene_ptr.push_back((int64_t)H->gene_mem.size()); }
  H->ident_ptr.assign(1, 0);
  for (auto& g : H->hdr.identical) { for (int32_t h : g) H->ident_mem.push_back(h); H->ident_ptr.push_back((int64_t)H->ident_mem.size()); }
}

mmqh_hits* mmqh_load(const char* path, int layout, char* err, int errlen) {
  mmqh_hits* H = new mmqh_hits();
  std::string e;
  if (mmq::load_hits_file(path, layout, H->hdr, H->cls, e)) { set_err(err, errlen, e); delete H; return nullptr; }
  flatten(H);
  return H;
}

/* In-memory records (header transcript indices), no names or genes. */
mmqh_hits* mmqh_from_records(int64_t T, const double* efflen, int64_t N, const int64_t* frag_ptr, const int32_t* frag_tid,
                             const float* frag_w, int layout, char* err, int errlen) {
  if (frag_w && (layout & 15) == mmq::LAYOUT_COLLAPSED) { set_err(err, errlen, "per-hit weights need a per-fragment layout"); return nullptr; }
  mmqh_hits* H = new mmqh_hits();
  H->hdr.efflen.assign(efflen, efflen + T);
  H->hdr.names.resize((size_t)T);
  mmq::ClassBuilder cb(T, layout, frag_w != nullptr);
  bool any_empty = false;
  for (int64_t f = 0; f < N && !any_empty; ++f) any_empty = frag_ptr[f + 1] == frag_ptr[f];
  if (!any_empty && N > 0 && cb.parallel_ready() && !getenv("MMQ_LOADER_SERIAL_RECORDS")) {
    /* all records at once on all host threads (a negative index reads as a huge unsigned one: out of range) */
    if (int brc = cb.add_records_csr(frag_ptr, frag_tid, frag_w, N)) {
      set_err(err, errlen, brc == 2 ? "per-hit weights must be finite and non-negative" : "transcript index out of range");
      delete H;
      return nullptr;
    }
  } else {
    for (int64_t f = 0; f < N; ++f) {
      const int64_t b = frag_ptr[f], e = frag_ptr[f + 1];
      for (int64_t q = b; q < e; ++q)
        if (frag_tid[q] < 0 || frag_tid[q] >= T) { set_err(err, errlen, "transcript index out of range"); delete H; return nullptr; }
      cb.add_record(frag_tid + b, frag_w ? frag_w + b : nullptr, (int)(e - b));
    }
  }
  cb.finish(H->cls);
  flatten(H);
  return H;
}

void mmqh_free(mmqh_hits* H) { delete H; }

/* test support: fmt_g6.h on an array of doubles, the texts separated by single spaces; returns the bytes written */
int64_t mmqh_fmt_g6(const double* v, int64_t n, char* out) {
  char* p = out;
  for (int64_t i = 0; i < n; ++i) { p = fmt_g6(p, v[i]); *p++ = ' '; }
  return (int64_t)(p - out);
}

/* test support: trace_writer.h — ids separated by '\n' in one string, keep (may be NULL) one flag per feature; 0 on success */
int mmqh_write_trace_gz(const char* path, const char* ids_nl, int64_t nfeat, const uint8_t* keep, const double* tr, int L) {
  std::vector<std::string> ids;
  const char* p = ids_nl;
  for (int64_t i = 0; i < nfeat; ++i) {
    const char* e = strchr(p, '\n');
    ids.emplace_back(p, e ? (size_t)(e - p) : strlen(p));
    p = e ? e + 1 : p + strlen(p);
  }
  std::vector<char> kp;
  if (keep) kp.assign(keep, keep + nfeat);
  return mmq::write_trace_gz(path, ids, kp, tr, L).empty() ? 0 : 1;
}

/* test support: huff_gz.h, one gzip member for the n bytes; returns its size (out must hold n + 1024 bytes) */
int64_t mmqh_gz_huffman(const void* in, int64_t n, void* out) {
  std::vector<uint8_t> z;
  mmq::hgz::gz_member((const char*)in, (size_t)n, z);
  memcpy(out, z.data(), z.size());
  return (int64_t)z.size();
}

/* test support: inflate_par.h on a zlib stream in memory; bytes written to out (capacity cap), -1 when the stream is
 * refused (the loader then uses serial zlib), -2 when out is too small */
int64_t mmqh_inflate_parallel(const void* in, int64_t n, int threads, void* out, int64_t cap) {
  mmq::ipar::Bytes b;
  if (!mmq::ipar::inflate_parallel((const uint8_t*)in, (size_t)n, threads, b)) return -1;
  if ((int64_t)b.size() > cap) return -2;
  memcpy(out, b.data(), b.size());
  return (int64_t)b.size();
}

int64_t mmqh_dim(const mmqh_hits* H, int which) {
  switch (which) {
    case 0: return (int64_t)H->hdr.names.size();
    case 1: return (int64_t)H->hdr.gene_names.size();
    case 2: return (int64_t)H->hdr.identical.size();
    case 3: return H->cls.N;
    case 4: return H->cls.n;
    case 5: return H->cls.m;
    case 6: return (int64_t)H->cls.col.size();
    case 7: return H->cls.n_classes;
    case 8: return H->hdr.schema;
    case 9: return (int64_t)H->cls.set_col.size();
    case 10: return H->cls.first_zero_weight_record;
    default: return -1;
  }
}
const int64_t* mmqh_row_ptr(const mmqh_hits* H) { return H->cls.row_ptr.data(); }
const int32_t* mmqh_col(const mmqh_hits* H) { return H->cls.col.data(); }
const int32_t* mmqh_k(const mmqh_hits* H) { return H->cls.k.empty() ? nullptr : H->cls.k.data(); }
const float* mmqh_w(const mmqh_hits* H) { return H->cls.w.empty() ? nullptr : H->cls.w.data(); }
const int64_t* mmqh_set_ptr(const mmqh_hits* H) { return H->cls.set_ptr.empty() ? nullptr : H->cls.set_ptr.data(); }
const int32_t* mmqh_set_col(const mmqh_hits* H) { return H->cls.set_ptr.empty() ? nullptr : H->cls.set_col.data(); }
const int32_t* mmqh_set_k(const mmqh_hits* H) { return H->cls.set_ptr.empty() ? nullptr : H->cls.set_k.data(); }
const int32_t* mmqh_col2hdr(const mmqh_hits* H) { return H->cls.col2hdr.data(); }
const int32_t* mmqh_hdr2col(const mmqh_hits* H) { return H->cls.hdr2col.data(); }
const int32_t* mmqh_doublehits(const mmqh_hits* H) { return H->cls.doublehits.data(); }
const double* mmqh_efflen(const mmqh_hits* H) { return H->hdr.efflen.data(); }
const int32_t* mmqh_truelen(const mmqh_hits* H) { return H->hdr.truelen.data(); }
const int32_t* mmqh_gene_of(const mmqh_hits* H) { return H->hdr.gene_of.data(); }
const char* mmqh_name(const mmqh_hits* H, int64_t t) { return H->hdr.names[(size_t)t].c_str(); }
const char* mmqh_gene_name(const mmqh_hits* H, int64_t g) { return H->hdr.gene_names[(size_t)g].c_str(); }
const int64_t* mmqh_gene_ptr(const mmqh_hits* H) { return H->gene_ptr.data(); }
const int32_t* mmqh_gene_members(const mmqh_hits* H) { return H->gene_mem.data(); }
const int64_t* mmqh_ident_ptr(const mmqh_hits* H) { return H->ident_ptr.data(); }
const int32_t* mmqh_ident_members(const mmqh_hits* H) { return H->ident_mem.data(); }
int mmqh_scaled_len(const mmqh_hits* H, double* l_out) {
  std::vector<double> l;
  std::string e;
  if (mmq::scaled_lengths(H->hdr, H->cls, l, e)) return 1;
  std::memcpy(l_out, l.data(), sizeof(double) * l.size());
  return 0;
}

} /* extern "C" */
