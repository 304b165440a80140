/* mmq_cls_plan.h — host side of the class plan of a collapsed shard (see mmq_cls.cu): pure C++,
 * no CUDA, so that the plan can also be built and replayed on the CPU by the tests
 * (hits_loader.cpp: mmqh_cls_replay; tests/test_cls_plan_cpu.py).  Included by mmq_cls.cu, which
 * uploads what mmq_cls_build_host produced. */
#ifndef MMQ_CLS_PLAN_H
#define MMQ_CLS_PLAN_H

#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/mmq_sampler.h"

#define MMQ_CLS_DMAX 64  /* longer classes go to the general kernel */
#define MMQ_CLS_DLO 8    /* class sizes 2..8: the 64-register instance (32 warps per SM) */
#define MMQ_CLS_DREG 16  /* class sizes up to this are register-resident template instances */
#define MMQ_CLS_CHAIN_DMAX 16 /* classes with more fragments than mmq_cat_limit(d): up to this size k_alloc_chain, above it the general kernel */
#define MMQ_CLS_WARPS 4
/* draws per slot of a class with d members: 64 (16 Philox blocks) for the small sizes; 16 for the larger ones, whose
 * slots cost 4 (d - 1) compare-and-add pairs per block — a 64-draw slot of a 16-member class is ~16 us of dependent work
 * for its warp, and the few such chunks then decide when the launch ends (measured in round 2: 26 us for 3.4 M warp
 * instructions).  Which draws a slot makes is a plan detail: draw t of a class always reads word t & 3 of block t >> 2. */
#define MMQ_CLS_GROUP(d) ((d) <= MMQ_CLS_DLO ? MMQ_CAT_GROUP : 16)
#define MMQ_CLS_NQ 17    /* sort positions inside a run of equal d: 16 - blocks (k >= 2); 16: k == 1 (those form runs of their own) */
/* runs are numbered by a "pseudo size": d for the classes with k >= 2, MMQ_CLS_DMAX + 1 + d for the single-fragment
 * classes — their chunks come after all the others and are swept by their own kernel (k_alloc_cls1) */
#define MMQ_CLS_DP1(d) (MMQ_CLS_DMAX + 1 + (d))
#define MMQ_CLS_DP_END (2 * MMQ_CLS_DMAX + 2)
#define MMQ_CLS_D_OF(dp) ((dp) > MMQ_CLS_DMAX ? (dp) - (MMQ_CLS_DMAX + 1) : (dp))

struct mmq_cls_run {
  int64_t e0;     /* offset in pcol of the run's first chunk */
  int32_t chunk0; /* first chunk of the run in the global numbering */
  int32_t d;      /* class size */
};


struct mmq_cls_host_plan {
  std::vector<mmq_cls_run> runs;
  std::unique_ptr<int32_t[]> pcol; /* [packed] member-major chunks of 32 slots */
  std::vector<uint16_t> pk;        /* [chunks * 32] draws of the slot | slot number within its class << 8 */
  std::vector<uint32_t> pcid;      /* [chunks * 32] low word of the class id */
  std::vector<unsigned long long> cdesc; /* [chunks] offset of the chunk in pcol << 8 | class size */
  int64_t chunks = 0, chunks_lo = 0, chunks_gen = 0, packed = 0, small_classes = 0, n_rest = 0, nnz_rest = 0;
  /* chunks [0, chunks_lo): k >= 2, d <= MMQ_CLS_DLO; [chunks_lo, chunks_gen): k >= 2, larger d; [chunks_gen, chunks): k == 1 */
  uint32_t cid_hi = 0;
  /* the chain set: classes with more than mmq_cat_limit(d) fragments and at most MMQ_CLS_DMAX members (conditional-binomial
   * chains, one class per lane of k_alloc_chain): member-major chunks of 32 like the small set, longest classes first */
  std::unique_ptr<int32_t[]> c_pcol;       /* [c_packed] */
  std::vector<int32_t> c_k;                /* [c_chunks * 32] fragments of the class (0: padding lane) */
  std::vector<uint32_t> c_cid;             /* [c_chunks * 32] low word of the class id */
  std::vector<unsigned long long> c_desc;  /* [c_chunks] offset of the chunk in c_pcol << 8 | class size */
  int64_t c_chunks = 0, c_packed = 0, n_chain = 0;
  int64_t c_end[3] = {0, 0, 0};            /* chain chunks of the classes above 4 members, above 2, all (k_alloc_chain's instances) */
  std::vector<int64_t> o_rp, o_cid, o_tiles; /* the rest: sub-CSR for the general kernel, one class per tile */
  std::vector<int32_t> o_col, o_k;
  std::vector<int32_t> s_col, s_k;           /* singleton classes: column and count */
};

/* host threads for a loop over `count` items (MMQ_PLAN_THREADS overrides: the tests run the threaded paths on small shards) */
static int cls_threads(int64_t count) {
  const char* e = getenv("MMQ_PLAN_THREADS");
  if (e && atoi(e) > 0) return (int)std::max<int64_t>(1, std::min<int64_t>(atoi(e), count));
  return (int)std::max<int64_t>(1, std::min<int64_t>(std::min<unsigned>(std::thread::hardware_concurrency(), 16u), count / 65536));
}

template <typename F>
static void cls_parallel_for(int64_t count, F&& f) {
  const int nt = cls_threads(count);
  if (nt <= 1) { f((int64_t)0, count); return; }
  std::vector<std::thread> th;
  for (int t = 0; t < nt; ++t) th.emplace_back([&, t] { f(count * t / nt, count * (t + 1) / nt); });
  for (auto& x : th) x.join();
}


/* Builds the plan of one shard (n transcripts, m classes: CSR rp / col, counts kk, Philox ids
 * class_id[] or class_id_base + row).  Returns false when the plan does not apply (class ids spread
 * over several 2^32 blocks, negative counts, too many chunks): the general kernel handles the shard. */
static bool mmq_cls_build_host(int64_t n, int64_t m, const int64_t* rp, const int32_t* col, const int32_t* kk, const int64_t* class_id,
                               int64_t class_id_base, mmq_cls_host_plan& P) {
  if (m <= 0) return false;
  static const bool timing = [] { const char* e = getenv("MMQ_CREATE_TIMING"); return e && atoi(e) != 0; }();
  auto t_last = std::chrono::steady_clock::now();
  auto tick = [&](const char* what) {
    if (!timing) return;
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[mmq_cls_plan] %-26s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
    t_last = now;
  };
  auto cid_of = [&](int64_t i) -> uint64_t { return (uint64_t)(class_id ? class_id[i] : class_id_base + i); };
  const uint32_t cid_hi = (uint32_t)(cid_of(0) >> 32);

  /* classify (host threads).  Slots of the small set are keyed (d, q): q = 16 - blocks for classes with
   * k >= 2 (a run of equal d starts with its most expensive slots), q = 16 for single-fragment classes
   * (whole warps of them take the one-draw path).  key16[i]: the key of the class's last (partial) slot,
   * or of its full slots when k is a multiple of 64; -1 singleton / empty, -2 rest. */
  const int NKEY = MMQ_CLS_DP_END * MMQ_CLS_NQ;
  std::vector<int16_t> key16(m);
  struct Tally { std::vector<int64_t> key_count; int64_t n_single = 0, n_rest = 0, nnz_rest = 0, small = 0, n_chain = 0; bool ok = true; };
  /* thread t owns classes [m t / T, m (t+1) / T) in this pass and in the placement pass below; it also counts
   * its small classes per first member (the buckets of the counting sort) */
  const int T = cls_threads(m);
  auto on_threads = [&](auto&& fn) {
    if (T == 1) { fn(0); return; }
    std::vector<std::thread> th;
    for (int t = 0; t < T; ++t) th.emplace_back([&, t] { fn(t); });
    for (auto& x : th) x.join();
  };
  const size_t nb = (size_t)n + 1;
  std::vector<int64_t> hist((size_t)T * nb, 0); /* [thread][first member] */
  std::vector<Tally> tally((size_t)T);
  on_threads([&](int tt) {
    Tally& t = tally[(size_t)tt];
    int64_t* hc = hist.data() + (size_t)tt * nb;
    t.key_count.assign(NKEY + 1, 0);
    for (int64_t i = m * tt / T; i < m * (tt + 1) / T; ++i) {
      const int64_t d = rp[i + 1] - rp[i];
      const int64_t kv = kk[i];
      if ((uint32_t)(cid_of(i) >> 32) != cid_hi || kv < 0) t.ok = false;
      if (d == 1 || kv <= 0) { key16[i] = -1; ++t.n_single; } /* k == 0: nothing to allocate */
      else if (d <= MMQ_CLS_DMAX && kv <= mmq_cat_limit((int)d)) {
        ++t.small;
        ++hc[col[rp[i]]];
        if (kv == 1) { key16[i] = (int16_t)(MMQ_CLS_DP1(d) * MMQ_CLS_NQ + 16); ++t.key_count[key16[i]]; }
        else {
          const int64_t grp = MMQ_CLS_GROUP(d);
          const int64_t full = kv / grp, tail = kv % grp;
          t.key_count[d * MMQ_CLS_NQ + (16 - grp / 4)] += full; /* full slots */
          key16[i] = (int16_t)(d * MMQ_CLS_NQ + (tail ? 16 - (int)((tail + 3) >> 2) : 16 - (int)(grp / 4)));
          if (tail) ++t.key_count[key16[i]];
        }
      } else if (d <= MMQ_CLS_CHAIN_DMAX) { key16[i] = -3; ++t.n_chain; }
      else { key16[i] = -2; ++t.n_rest; t.nnz_rest += d; }
    }
  });
  tick("classify");
  std::vector<int64_t> key_count(NKEY + 1, 0);
  int64_t n_single = 0, n_rest = 0, nnz_rest = 0, small_classes = 0, n_chain = 0;
  for (const Tally& t : tally) {
    n_chain += t.n_chain;
    if (!t.ok) return false; /* class ids spread over several 2^32 blocks (or k < 0): the general kernel handles it */
    for (int q = 0; q <= NKEY; ++q) key_count[q] += t.key_count[q];
    n_single += t.n_single; n_rest += t.n_rest; nnz_rest += t.nnz_rest; small_classes += t.small;
  }

  /* runs of equal d, chunks of 32 slots */
  std::vector<mmq_cls_run>& runs = P.runs;
  std::vector<int64_t> key_slot(NKEY + 1, 0); /* first slot (global numbering, 32 per chunk) of each key */
  std::vector<int64_t> run_slots; /* slots in use per run: the rest of its last chunk is padding */
  int64_t chunks = 0, packed = 0, chunks_lo = 0, chunks_gen = 0;
  std::vector<int32_t> run_of_d(MMQ_CLS_DP_END, -1); /* by pseudo size */
  for (int dp = 2; dp < MMQ_CLS_DP_END; ++dp) {
    const int d = MMQ_CLS_D_OF(dp);
    int64_t cnt = 0;
    for (int q = 0; q < MMQ_CLS_NQ; ++q) { key_slot[dp * MMQ_CLS_NQ + q] = chunks * 32 + cnt; cnt += key_count[dp * MMQ_CLS_NQ + q]; }
    if (cnt > 0) {
      mmq_cls_run r;
      r.e0 = packed; r.chunk0 = (int32_t)chunks; r.d = d;
      run_of_d[dp] = (int32_t)runs.size();
      runs.push_back(r);
      run_slots.push_back(cnt);
      const int64_t nch = (cnt + 31) / 32;
      chunks += nch;
      packed += nch * 32 * d;
      if (chunks > 0x7fff0000ll) return false;
    }
    if (dp <= MMQ_CLS_DLO) chunks_lo = chunks;
    if (dp <= MMQ_CLS_DMAX) chunks_gen = chunks;
  }
  P.cdesc.assign((size_t)chunks, 0ull);
  for (size_t r = 0; r < runs.size(); ++r) {
    const int64_t c1 = r + 1 < runs.size() ? runs[r + 1].chunk0 : chunks;
    for (int64_t c = runs[r].chunk0; c < c1; ++c)
      P.cdesc[(size_t)c] = ((unsigned long long)(runs[r].e0 + (c - runs[r].chunk0) * 32 * runs[r].d) << 8) | (unsigned long long)runs[r].d;
  }

  /* Within a key the classes are placed by their first member (a stable counting sort): members are
   * ascending and the isoforms of a gene are neighbours in the header, so the lanes of a warp and the
   * warps of an SM gather neighbouring mu — L1 hits instead of one L2 sector per 8-byte gather. */
  static_assert(MMQ_CAT_KMAX / 16 <= 255 && MMQ_CAT_GROUP <= 255, "slot counts are kept in bytes");
  struct Ord { int32_t i; int16_t key; uint8_t full, tail; }; /* key: of the partial slot (tail draws) when there is one */
  std::vector<Ord> order((size_t)small_classes);
  /* parallel stable counting sort (counts taken in the classification pass): per first member, thread t gets
   * a contiguous piece of that member's bucket */
  {
    int64_t run = 0;
    for (size_t v = 0; v < nb; ++v) /* exclusive prefix in (member, thread) order */
      for (int t = 0; t < T; ++t) { const int64_t c = hist[(size_t)t * nb + v]; hist[(size_t)t * nb + v] = run; run += c; }
    on_threads([&](int t) {
      int64_t* c = hist.data() + (size_t)t * nb;
      for (int64_t i = m * t / T; i < m * (t + 1) / T; ++i)
        if (key16[i] >= 0) order[(size_t)c[col[rp[i]]]++] = Ord{(int32_t)i, key16[i], (uint8_t)(kk[i] / MMQ_CLS_GROUP(rp[i + 1] - rp[i])), (uint8_t)(kk[i] % MMQ_CLS_GROUP(rp[i + 1] - rp[i]))};
    });
  }
  tick("order by first member");
  /* first slot of every small class within each of its (at most two) keys, in placement order: thread t
   * takes a contiguous piece of the order; the keys' running positions are prefixed over the threads */
  std::vector<int64_t> slot_full((size_t)small_classes), slot_tail((size_t)small_classes);
  {
    std::vector<int64_t> used((size_t)T * (NKEY + 1), 0); /* [thread][key]: slots the piece needs */
    on_threads([&](int t) {
      int64_t* u = used.data() + (size_t)t * (NKEY + 1);
      for (int64_t o = small_classes * t / T; o < small_classes * (t + 1) / T; ++o) {
        const Ord& e = order[(size_t)o];
        const int dpu = e.key / MMQ_CLS_NQ;
        u[dpu * MMQ_CLS_NQ + (16 - MMQ_CLS_GROUP(MMQ_CLS_D_OF(dpu)) / 4)] += e.full;
        if (e.tail) ++u[e.key];
      }
    });
    for (int q = 0; q <= NKEY; ++q) {
      int64_t run = key_slot[q];
      for (int t = 0; t < T; ++t) { const int64_t c = used[(size_t)t * (NKEY + 1) + q]; used[(size_t)t * (NKEY + 1) + q] = run; run += c; }
    }
    on_threads([&](int t) {
      int64_t* next = used.data() + (size_t)t * (NKEY + 1);
      for (int64_t o = small_classes * t / T; o < small_classes * (t + 1) / T; ++o) {
        const Ord& e = order[(size_t)o];
        const int dp = e.key / MMQ_CLS_NQ;
        const int qf = 16 - MMQ_CLS_GROUP(MMQ_CLS_D_OF(dp)) / 4; /* the key of the class's full slots */
        slot_full[(size_t)o] = next[dp * MMQ_CLS_NQ + qf];
        next[dp * MMQ_CLS_NQ + qf] += e.full;
        slot_tail[(size_t)o] = e.tail ? next[e.key]++ : -1; /* -1: k is a multiple of 64, no partial slot */
      }
    });
  }
  tick("slots");
  P.pcol.reset(new int32_t[(size_t)std::max<int64_t>(packed, 1)]); /* every entry is written below */
  std::unique_ptr<int32_t[]>& pcol = P.pcol;
  std::vector<uint16_t>& pk = P.pk;
  std::vector<uint32_t>& pcid = P.pcid;
  pk.assign((size_t)chunks * 32, 0);
  pcid.assign((size_t)chunks * 32, 0u);
  for (size_t r = 0; r < runs.size(); ++r) { /* padding slots of a run's last chunk: the sentinel column (mu[n] == 0), no draws */
    const int d = runs[r].d;
    const int64_t used = run_slots[r], nch = (used + 31) / 32;
    int32_t* last = pcol.get() + runs[r].e0 + (nch - 1) * 32 * d;
    for (int lane = (int)(used - (nch - 1) * 32); lane < 32; ++lane)
      for (int j = 0; j < d; ++j) last[32 * j + lane] = (int32_t)n;
  }
  cls_parallel_for(small_classes, [&](int64_t a0, int64_t b0) {
    for (int64_t o = a0; o < b0; ++o) {
      const Ord& e = order[(size_t)o];
      const int64_t i = e.i;
      const mmq_cls_run& r = runs[run_of_d[e.key / MMQ_CLS_NQ]];
      const int d = r.d;
      const int32_t* src = col + rp[i];
      const uint32_t cid = (uint32_t)cid_of(i);
      auto put = [&](int64_t s, int draws, int slot_no) {
        const int64_t ch = s >> 5;
        int32_t* dst = pcol.get() + r.e0 + (ch - r.chunk0) * 32 * d + (s & 31);
        for (int j = 0; j < d; ++j) dst[32 * j] = src[j];
        pk[s] = (uint16_t)(draws | (slot_no << 8));
        pcid[s] = cid;
      };
      for (int q = 0; q < (int)e.full; ++q) put(slot_full[(size_t)o] + q, MMQ_CLS_GROUP(d), q);
      if (e.tail) put(slot_tail[(size_t)o], (int)e.tail, (int)e.full);
    }
  });

  tick("fill");
  /* the chain set: by class size (longest first: a chain is serial in its members, the long ones must not be the tail of
   * the launch), then by first member; 32 classes per chunk, member-major, padding lanes have k = 0 and the sentinel column */
  {
    std::vector<int64_t> chain;
    chain.reserve((size_t)n_chain);
    for (int64_t i = 0; i < m; ++i)
      if (key16[i] == -3) chain.push_back(i);
    std::stable_sort(chain.begin(), chain.end(), [&](int64_t a, int64_t b) {
      const int64_t da = rp[a + 1] - rp[a], db = rp[b + 1] - rp[b];
      return da != db ? da > db : col[rp[a]] < col[rp[b]];
    });
    int64_t c_chunks = 0, c_packed = 0;
    for (size_t a = 0; a < chain.size();) { /* runs of equal d */
      const int64_t d = rp[chain[a] + 1] - rp[chain[a]];
      size_t b = a;
      while (b < chain.size() && rp[chain[b] + 1] - rp[chain[b]] == d) ++b;
      const int64_t nch = ((int64_t)(b - a) + 31) / 32;
      for (int64_t c = 0; c < nch; ++c) P.c_desc.push_back(((unsigned long long)(c_packed + c * 32 * d) << 8) | (unsigned long long)d);
      c_chunks += nch;
      c_packed += nch * 32 * d;
      for (int v = 0; v < 3; ++v)
        if (d > (4 >> v)) P.c_end[v] = c_chunks;
      a = b;
    }
    P.c_pcol.reset(new int32_t[(size_t)std::max<int64_t>(c_packed, 1)]);
    for (int64_t q = 0; q < c_packed; ++q) P.c_pcol[(size_t)q] = (int32_t)n;
    P.c_k.assign((size_t)c_chunks * 32, 0);
    P.c_cid.assign((size_t)c_chunks * 32, 0u);
    int64_t chunk = 0;
    for (size_t a = 0; a < chain.size();) {
      const int64_t d = rp[chain[a] + 1] - rp[chain[a]];
      size_t b = a;
      while (b < chain.size() && rp[chain[b] + 1] - rp[chain[b]] == d) ++b;
      for (size_t q = a; q < b; ++q) {
        const int64_t i = chain[q], s = chunk * 32 + (int64_t)(q - a);
        int32_t* dst = P.c_pcol.get() + (P.c_desc[(size_t)(s >> 5)] >> 8) + (s & 31);
        for (int64_t j = 0; j < d; ++j) dst[32 * j] = col[rp[i] + j];
        P.c_k[(size_t)s] = kk[i];
        P.c_cid[(size_t)s] = (uint32_t)cid_of(i);
      }
      chunk += ((int64_t)(b - a) + 31) / 32;
      a = b;
    }
    P.c_chunks = c_chunks; P.c_packed = c_packed; P.n_chain = n_chain;
  }
  tick("chain set");
  /* the rest: a sub-CSR for the general kernel, longest chains first, ONE class per warp tile (a
   * chain of binomials is serial: what matters is when the slowest warp ends, not lane use) */
  std::vector<int64_t> rest;
  rest.reserve((size_t)n_rest);
  for (int64_t i = 0; i < m; ++i)
    if (key16[i] == -2) rest.push_back(i);
  std::stable_sort(rest.begin(), rest.end(), [&](int64_t a, int64_t b) { return rp[a + 1] - rp[a] > rp[b + 1] - rp[b]; });
  std::vector<int64_t>&o_rp = P.o_rp, &o_cid = P.o_cid, &o_tiles = P.o_tiles;
  std::vector<int32_t>&o_col = P.o_col, &o_k = P.o_k;
  o_rp.assign((size_t)n_rest + 1, 0); o_cid.assign((size_t)n_rest, 0); o_tiles.assign((size_t)n_rest + 1, 0);
  o_col.assign((size_t)nnz_rest + 4, 0); o_k.assign((size_t)n_rest, 0);
  for (int64_t q = 0; q < n_rest; ++q) {
    const int64_t i = rest[q];
    const int64_t d = rp[i + 1] - rp[i];
    memcpy(o_col.data() + o_rp[q], col + rp[i], sizeof(int32_t) * (size_t)d);
    o_rp[q + 1] = o_rp[q] + d;
    o_k[q] = kk[i];
    o_cid[q] = (int64_t)cid_of(i);
    o_tiles[q] = q;
  }
  o_tiles[n_rest] = n_rest;

  /* singletons: constant counts */
  std::vector<int32_t>&s_col = P.s_col, &s_k = P.s_k;
  s_col.clear(); s_k.clear();
  s_col.reserve((size_t)n_single); s_k.reserve((size_t)n_single);
  for (int64_t i = 0; i < m; ++i)
    if (key16[i] == -1 && kk[i] > 0) { s_col.push_back(col[rp[i]]); s_k.push_back(kk[i]); }

  tick("rest, singletons");
  P.chunks = chunks; P.chunks_lo = chunks_lo; P.chunks_gen = chunks_gen; P.packed = packed; P.cid_hi = cid_hi;
  P.small_classes = small_classes; P.n_rest = n_rest; P.nnz_rest = nnz_rest;
  return true;
}

/* CPU replay of one sweep over a plan: what k_alloc_cls + k_alloc + seg_base add up to.  The draws
 * and the order of the floating-point sums are those of the kernels (and of mmq_alloc_row). */
static void mmq_cls_replay_host(const mmq_cls_host_plan& P, int64_t n, const double* mu, uint32_t seed, uint32_t sweep, int32_t* counts) {
  for (int64_t t = 0; t < n; ++t) counts[t] = 0;
  for (size_t i = 0; i < P.s_col.size(); ++i) counts[P.s_col[i]] += P.s_k[i];
  std::vector<double> S;
  for (size_t r = 0; r < P.runs.size(); ++r) {
    const int d = P.runs[r].d;
    const int64_t c0 = P.runs[r].chunk0, c1 = r + 1 < P.runs.size() ? P.runs[r + 1].chunk0 : P.chunks;
    S.assign((size_t)d, 0.0);
    for (int64_t ch = c0; ch < c1; ++ch)
      for (int lane = 0; lane < 32; ++lane) {
        const int32_t* pc = P.pcol.get() + P.runs[r].e0 + (ch - c0) * 32 * d + lane;
        const uint32_t meta = P.pk[(size_t)(ch * 32 + lane)];
        const int kq = (int)(meta & 0xffu);
        const uint32_t b0 = (meta >> 8) * (uint32_t)(MMQ_CLS_GROUP(d) / 4);
        const uint32_t cid = P.pcid[(size_t)(ch * 32 + lane)];
        if (kq == 0) continue;
        for (int j = 0; j < d; ++j) S[(size_t)j] = (pc[32 * j] == (int32_t)n ? 0.0 : mu[pc[32 * j]]) + (j ? S[(size_t)j - 1] : 0.0);
        const double norm = S[(size_t)d - 1];
        const bool is1 = kq == 1 && b0 == 0u;
        for (int t = 0; t < kq; ++t) {
          uint32_t wd[4];
          uint32_t word;
          if (is1) {
            wd[0] = (cid >> 2) | (P.cid_hi << 30); wd[1] = P.cid_hi >> 2; wd[2] = sweep; wd[3] = 0u;
            mmq_philox4x32_10(wd, seed, MMQ_STREAM_CAT);
            word = wd[cid & 3u];
          } else {
            wd[0] = cid; wd[1] = P.cid_hi; wd[2] = sweep; wd[3] = b0 + (uint32_t)(t >> 2);
            mmq_philox4x32_10(wd, seed, MMQ_STREAM_ALLOC);
            word = wd[t & 3];
          }
          const double target = mmq_uniform32(word) * norm;
          int chosen = d - 1;
          for (int j = 0; j < d - 1; ++j)
            if (target < S[(size_t)j]) { chosen = j; break; }
          counts[pc[32 * chosen]] += 1;
        }
      }
  }
  std::vector<double> p;
  std::vector<int32_t> x;
  for (int64_t s = 0; s < P.c_chunks * 32; ++s) { /* the chain set, lane by lane */
    const int64_t kv = P.c_k[(size_t)s];
    if (kv <= 0) continue;
    const int d = (int)(P.c_desc[(size_t)(s >> 5)] & 0xffull);
    const int32_t* pc = P.c_pcol.get() + (P.c_desc[(size_t)(s >> 5)] >> 8) + (s & 31);
    p.resize((size_t)d); x.assign((size_t)d, 0);
    for (int j = 0; j < d; ++j) p[(size_t)j] = mu[pc[32 * j]];
    mmq_alloc_row(p.data(), x.data(), d, kv, seed, ((uint64_t)P.cid_hi << 32) | P.c_cid[(size_t)s], sweep);
    for (int j = 0; j < d; ++j) counts[pc[32 * j]] += x[(size_t)j];
  }
  for (int64_t q = 0; q < P.n_rest; ++q) {
    const int d = (int)(P.o_rp[(size_t)q + 1] - P.o_rp[(size_t)q]);
    p.resize((size_t)d); x.assign((size_t)d, 0);
    for (int j = 0; j < d; ++j) p[(size_t)j] = mu[P.o_col[(size_t)P.o_rp[(size_t)q] + (size_t)j]];
    mmq_alloc_row(p.data(), x.data(), d, (int64_t)P.o_k[(size_t)q], seed, (uint64_t)P.o_cid[(size_t)q], sweep);
    for (int j = 0; j < d; ++j) counts[P.o_col[(size_t)P.o_rp[(size_t)q] + (size_t)j]] += x[(size_t)j];
  }
}

#endif /* MMQ_CLS_PLAN_H */
