/* oracle/oracle.cc -- TEST INFRASTRUCTURE ONLY: CPU restatement of the BreakID hot path.
 *
 * Every function restates one reference function on the struct-of-arrays record batch the
 * product's C-ABI consumes, and cites the reference lines it follows (paths relative to
 * /root/reference).  PINNING: the reference ships no tests or golden vectors (SURVEY.md §4), so
 * this restatement is pinned against the reference ITSELF, compiled here from its own sources
 * (oracle/Makefile -> oracle/_ref/libbreakid_ref.so + BreakID_ref): tests/test_oracle_vs_ref.py
 * diffs every orc_* entry point against the corresponding ref_* wrapper (oracle/ref_shim.cc) in
 * this container, and the committed fixtures under tests/golden/ (made by
 * tests/golden/make_golden.py with the reference binary) pin it where /root/reference is absent.
 *
 * Two kinds of functions live here:
 *   orc_*        literal restatements (sorted linked lists, N x N matrix, std::sort ...).
 *   orc_model_*  CPU models of the *device formulations* (parallel introsort replay, AHC by
 *                components with the closed-form tie rule).  They exist so that the formulation
 *                is proven equal to the literal restatement / the reference on the CPU before it
 *                is trusted on the GPU.  The CUDA kernels in breakid_b200/csrc follow them.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this library.
 */
#include "oracle.h"

#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <unordered_map>
#include <vector>

namespace {

enum { F_PAIRED = 0x1, F_PROPER = 0x2, F_UNMAP = 0x4, F_REVERSE = 0x10, F_SECONDARY = 0x100,
       F_QCFAIL = 0x200, F_DUP = 0x400 };

struct H128 {
  uint64_t lo, hi;
  bool operator==(const H128 &o) const { return lo == o.lo && hi == o.hi; }
};
struct H128Hash { size_t operator()(const H128 &h) const { return (size_t)(h.lo ^ (h.hi * 0x9E3779B97F4A7C15ULL)); } };

/* src/util_bam.cc:57-68 -- uint32 wrap-around sum of target_len[0..tid) + pos */
uint32_t genome_pos(const uint32_t *target_len, int tid, int32_t pos)
{
  uint32_t p = 0;
  for (int i = 0; i < tid; ++i) p += target_len[i];
  p += (uint32_t)pos;
  return p;
}

struct KeyIdx { uint32_t key; uint32_t idx; };
bool cmp_key(KeyIdx a, KeyIdx b) { return a.key < b.key; }   /* src/BreakID.h:170-183 shape */

}  // namespace

extern "C" {

void orc_free(void *p) { free(p); }

/* ------------------------------------------------------------------------------------------
 * a1. insert-size statistics -- src/BreakID.cc:1909-1954.
 * The sd accumulator is a `long` that is converted to double, added to d*d and truncated back on
 * every element (src/BreakID.cc:1913,1944); sd = sqrt(total/(double)n) (population sd).
 * Also returns the integer intermediates so the device path can be compared exactly. */
void orc_insert_stats(long n, const uint16_t *flag, const int32_t *isize, double *mean, double *sd,
                      int64_t *sum_out, int64_t *count_out, int64_t *sd_total_out)
{
  const uint32_t filter = F_UNMAP | F_SECONDARY | F_QCFAIL | F_DUP;
  long total = 0, cnt = 0;
  for (long i = 0; i < n; ++i)
    if ((flag[i] & F_PAIRED) && (flag[i] & F_PROPER) && !(flag[i] & filter)) { total += abs(isize[i]); ++cnt; }
  double m = (double)total / (double)cnt;
  long sd_total = 0;
  for (long i = 0; i < n; ++i)
    if ((flag[i] & F_PAIRED) && (flag[i] & F_PROPER) && !(flag[i] & filter)) {
      double x = (double)abs(isize[i]);
      sd_total += (x - m) * (x - m);      /* long += double: convert, add, truncate */
    }
  *mean = m;
  *sd = sqrt(sd_total / (double)cnt);
  if (sum_out) *sum_out = total;
  if (count_out) *count_out = cnt;
  if (sd_total_out) *sd_total_out = sd_total;
}

/* src/BreakID.cc:103 -- one distance used by scan, mask, span and cluster stages */
/* src/BreakID.cc:103.  The literal 3 is the only thing the extension flag -s replaces (include/breakid_b200.h: bkid_params.sd_mult);
 * its reference counterpart is the same binary with that one literal read from the environment (oracle/Makefile: ref_s). */
static int g_sd_mult = 3;
void orc_set_sd_mult(int m) { g_sd_mult = m; }
double orc_dist(double mean, double sd, int times) { return times * sqrt(times) * (mean + g_sd_mult * sd); }

/* the breakpoint vote window (src/BreakID.cc:444-445, literal 2) and the complementary-cigar tolerance (:891, literal 10)
 * of every refinement entry point; the device reads them from bkid_params.bp_pos_error / mismatch_num */
static int g_bp_err = 2, g_mismatch = 10;
void orc_set_refine_consts(int bp_err, int mismatch) { g_bp_err = bp_err; g_mismatch = mismatch; }

/* ------------------------------------------------------------------------------------------
 * a2/a3. discordant-pair scan -- src/BreakID.cc:1362-1515, src/util_bam.cc:7-47,57-68.
 * names[t] = header target name of tid t.  Output: pairs bucket by bucket in std::map<string>
 * order of "p1chr_p2chr", inside a bucket in emission order. */
long orc_scan(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos,
              const int32_t *mtid, const int32_t *mpos, const uint64_t *name_hash /* [2n] lo,hi */,
              int n_targets, const uint32_t *target_len, const char *const *names,
              long qual, double w, orc_pair **out)
{
  std::unordered_map<H128, long, H128Hash> store;      /* readname_2_alignment (:1379) */
  std::vector<orc_pair> emitted;
  for (long i = 0; i < n; ++i) {
    /* :1419-1420 -- SUPPLEMENTARY, UNMAP, QCFAIL are NOT tested */
    if (!((long)mapq[i] >= qual && !(flag[i] & F_DUP) && !(flag[i] & F_SECONDARY) &&
          (flag[i] & F_PAIRED) && !(flag[i] & F_PROPER)))
      continue;
    H128 h{name_hash[2 * i], name_hash[2 * i + 1]};
    auto it = store.find(h);
    if (it == store.end()) { store[h] = i; continue; }       /* first mate (:1485-1494) */
    long j = it->second;
    int ti = tid[i] < 0 ? -1 : tid[i], tj = tid[j] < 0 ? -1 : tid[j];   /* rname "*" for tid<0 */
    long pi = (long)pos[i] + 1, pj = (long)pos[j] + 1;
    if (ti != tj || (double)labs(pi - pj) >= w) {             /* :1428 */
      uint32_t c1 = genome_pos(target_len, tid[i], pos[i]);   /* :1431 -- the CURRENT record's own fields */
      uint32_t c2 = genome_pos(target_len, mtid[i], mpos[i]); /* :1432 -- and its MATE fields           */
      orc_pair p;
      memset(&p, 0, sizeof p);
      p.name_lo = h.lo; p.name_hi = h.hi;
      if (c1 <= c2) {                                          /* :1434-1448 */
        p.p1_flag = flag[i]; p.p1_tid = ti; p.p1_pos = (uint32_t)pi; p.p1_mapq = mapq[i];
        p.p1_chr_pos = c1; p.p2_chr_pos = c2;
        p.p2_flag = flag[j]; p.p2_tid = tj; p.p2_pos = (uint32_t)pj; p.p2_mapq = mapq[j];
      } else {                                                 /* :1449-1465 */
        p.p2_flag = flag[i]; p.p2_tid = ti; p.p2_pos = (uint32_t)pi; p.p2_mapq = mapq[i];
        p.p1_chr_pos = c2; p.p2_chr_pos = c1;
        p.p1_flag = flag[j]; p.p1_tid = tj; p.p1_pos = (uint32_t)pj; p.p1_mapq = mapq[j];
      }
      p.p1_strand = (p.p1_flag & F_REVERSE) ? '-' : '+';       /* :1467-1478 */
      p.p2_strand = (p.p2_flag & F_REVERSE) ? '-' : '+';
      p.cluster = -1;
      emitted.push_back(p);
    }
    store.erase(it);                                           /* :1482 -- always */
  }
  /* :1500-1512 -- bucket by "p1chr_p2chr", std::map<string> iteration order */
  auto nm = [&](int t) { return t < 0 ? std::string("*") : std::string(names[t]); };
  std::map<std::string, std::vector<long>> buckets;
  for (size_t k = 0; k < emitted.size(); ++k)
    buckets[nm(emitted[k].p1_tid) + "_" + nm(emitted[k].p2_tid)].push_back((long)k);
  orc_pair *o = (orc_pair *)calloc(emitted.size() ? emitted.size() : 1, sizeof(orc_pair));
  long k = 0; int b = 0;
  for (auto &kv : buckets) {
    for (long e : kv.second) { o[k] = emitted[e]; o[k].bucket = b; o[k].orig = (uint32_t)k; ++k; }
    ++b;
  }
  *out = o;
  return (long)emitted.size();
}

/* rank of every possible "chrA_chrB" bucket name in std::map<string> order (what the product's
 * host computes once per header and hands to the device).  rank[(a+1)*(n_targets+1)+(b+1)],
 * index 0 = "*".  Dense: equal strings ("scaf" + "1_2", "scaf_1" + "2") share a rank, as they share
 * one key of orc_scan's map. */
void orc_bucket_rank_table(int n_targets, const char *const *names, int32_t *rank)
{
  int m = n_targets + 1;
  std::vector<std::pair<std::string, int>> v;
  for (int a = 0; a < m; ++a)
    for (int b = 0; b < m; ++b) {
      std::string sa = a ? names[a - 1] : "*", sb = b ? names[b - 1] : "*";
      v.push_back({sa + "_" + sb, a * m + b});
    }
  std::sort(v.begin(), v.end());
  int32_t r = -1;
  for (size_t k = 0; k < v.size(); ++k) {
    if (k == 0 || v[k].first != v[k - 1].first) ++r;
    rank[v[k].second] = r;
  }
}

/* ------------------------------------------------------------------------------------------
 * A2. the unstable std::sort the pipeline depends on (src/BreakID.cc:1274,1278,1282,144,1091,
 * 1127): literal = libstdc++ std::sort with a key-only comparator.  perm[i] = original index. */
void orc_std_sort_perm(long n, const uint32_t *key, uint32_t *perm)
{
  std::vector<KeyIdx> v(n);
  for (long i = 0; i < n; ++i) v[i] = KeyIdx{key[i], (uint32_t)i};
  std::sort(v.begin(), v.end(), cmp_key);
  for (long i = 0; i < n; ++i) perm[i] = v[i].idx;
}

/* MODEL of the device formulation of the same sort ("parallel introsort replay"):
 * libstdc++ introsort = recursive {median-of-3 to front, unguarded Hoare partition} until a
 * segment has <= 16 elements or the depth budget 2*floor(log2 n) is spent (then heapsort), followed
 * by one insertion sort over the whole array.  Facts used:
 *  (1) a partition step is data-parallel: with L = positions (ascending) holding key >= pivot and
 *      R = positions (descending) holding key <= pivot inside [first+1,last), the sequential
 *      pointer walk swaps L[k] <-> R[k] for k < K = #{k : L[k] < R[k]} and returns
 *      cut = min(L[K], R[K-1]) (R[-1] = last);
 *  (2) the final insertion sort is stable and never moves an element across a partition cut, so
 *      it equals an independent stable sort of every terminal segment.
 * So the permutation is: level-synchronous partitions over all segments, then a stable sort of
 * each terminal (<=16) segment.  Depth-exhausted segments fall back to the literal heapsort. */
static long g_model_heapsorts = 0;
static void model_heapsort(KeyIdx *a, long n)
{
  ++g_model_heapsorts;
  /* std::__partial_sort(first,last,last) = __heap_select (make_heap; nothing to select) +
   * __sort_heap -- libstdc++ bits/stl_heap.h semantics */
  auto adjust = [&](long hole, long len, KeyIdx value) {
    const long top = hole;
    long child = hole;
    while (child < (len - 1) / 2) {
      child = 2 * (child + 1);
      if (a[child].key < a[child - 1].key) child--;
      a[hole] = a[child];
      hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
      child = 2 * (child + 1);
      a[hole] = a[child - 1];
      hole = child - 1;
    }
    long parent = (hole - 1) / 2;                      /* __push_heap */
    while (hole > top && a[parent].key < value.key) {
      a[hole] = a[parent];
      hole = parent;
      parent = (hole - 1) / 2;
    }
    a[hole] = value;
  };
  if (n < 2) return;
  for (long parent = (n - 2) / 2;; --parent) {         /* __make_heap */
    KeyIdx v = a[parent];
    adjust(parent, n, v);
    if (parent == 0) break;
  }
  for (long last = n - 1; last > 0; --last) {          /* __sort_heap / __pop_heap */
    KeyIdx v = a[last];
    a[last] = a[0];
    adjust(0, last, v);
  }
}

long orc_model_heapsort_count(void) { return g_model_heapsorts; }

void orc_model_sort_perm(long n, const uint32_t *key, uint32_t *perm)
{
  std::vector<KeyIdx> a(n);
  for (long i = 0; i < n; ++i) a[i] = KeyIdx{key[i], (uint32_t)i};
  struct Seg { long f, l; int depth; };
  std::vector<Seg> cur, nxt, terminal;
  if (n > 1) {
    int lg = 0;
    for (long t = n; t > 1; t >>= 1) ++lg;              /* std::__lg(n) */
    cur.push_back({0, n, 2 * lg});
  }
  std::vector<long> L, R;
  while (!cur.empty()) {
    nxt.clear();
    for (const Seg &s : cur) {
      long f = s.f, l = s.l;
      if (l - f <= 16) { terminal.push_back(s); continue; }
      if (s.depth == 0) { model_heapsort(&a[f], l - f); continue; }
      /* __move_median_to_first(first, first+1, mid, last-1) */
      long mid = f + (l - f) / 2, A = f + 1, B = mid, C = l - 1;
      uint32_t ka = a[A].key, kb = a[B].key, kc = a[C].key;
      long med;
      if (ka < kb) { if (kb < kc) med = B; else if (ka < kc) med = C; else med = A; }
      else if (ka < kc) med = A;
      else if (kb < kc) med = C;
      else med = B;
      std::swap(a[f], a[med]);
      uint32_t p = a[f].key;
      /* data-parallel form of __unguarded_partition(first+1, last, first) */
      L.clear(); R.clear();
      for (long i = f + 1; i < l; ++i) if (!(a[i].key < p)) L.push_back(i);
      for (long i = l - 1; i > f; --i) if (!(p < a[i].key)) R.push_back(i);
      size_t K = 0;
      while (K < L.size() && K < R.size() && L[K] < R[K]) ++K;
      for (size_t k = 0; k < K; ++k) std::swap(a[L[k]], a[R[k]]);
      long rprev = K ? R[K - 1] : l;
      long cut = (K < L.size() && L[K] < rprev) ? L[K] : rprev;
      nxt.push_back({cut, l, s.depth - 1});
      nxt.push_back({f, cut, s.depth - 1});
    }
    cur.swap(nxt);
  }
  if (n <= 16 && n > 0) terminal.push_back({0, n, 0});
  for (const Seg &s : terminal)                          /* stable sort of each terminal segment */
    std::stable_sort(a.begin() + s.f, a.begin() + s.l, cmp_key);
  for (long i = 0; i < n; ++i) perm[i] = a[i].idx;
}

/* ------------------------------------------------------------------------------------------
 * a4. isolated-pair removal -- src/BreakID.cc:1271-1285, mask_pairs_chr_pos :1813-1877.
 * Works on indices; returns surviving original indices in final order (may contain the index
 * that sat at position 1 twice; never positions 0 and np-1 of either pass). */
static void mask_pass(std::vector<KeyIdx> &v, const uint32_t *p1, const uint32_t *p2, long distance)
{
  long np = (long)v.size();
  if (np <= 2) { v.clear(); return; }
  auto gap = [](uint32_t a, uint32_t b) { return (long)abs((int32_t)(a - b)); };
  std::vector<KeyIdx> out;
  long Lx = gap(p1[v[1].idx], p1[v[2].idx]), Ly = gap(p2[v[1].idx], p2[v[2].idx]);
  if (!(Lx > distance || Ly > distance)) out.push_back(v[1]);            /* :1830-1835 */
  for (long i = 1; i < np - 1; ++i) {                                    /* :1845-1870 */
    long ll = gap(p1[v[i - 1].idx], p1[v[i].idx]), lr = gap(p1[v[i + 1].idx], p1[v[i].idx]);
    Lx = ll < lr ? ll : lr;
    ll = gap(p2[v[i - 1].idx], p2[v[i].idx]); lr = gap(p2[v[i + 1].idx], p2[v[i].idx]);
    Ly = ll < lr ? ll : lr;
    if (!(Lx > distance || Ly > distance)) out.push_back(v[i]);
  }
  v.swap(out);
}

long orc_remove_isolated(long n, const uint32_t *p1, const uint32_t *p2, double w, uint32_t *out_idx)
{
  std::vector<KeyIdx> v(n);
  for (long i = 0; i < n; ++i) v[i] = KeyIdx{p1[i], (uint32_t)i};
  std::sort(v.begin(), v.end(), cmp_key);                                /* :1274 */
  mask_pass(v, p1, p2, (long)w);                                         /* double -> long at the call */
  if (!v.empty()) {
    for (auto &e : v) e.key = p2[e.idx];
    std::sort(v.begin(), v.end(), cmp_key);                              /* :1278 */
    mask_pass(v, p1, p2, (long)w);
    if (!v.empty()) {
      for (auto &e : v) e.key = p1[e.idx];
      std::sort(v.begin(), v.end(), cmp_key);                            /* :1282 */
    }
  }
  for (size_t i = 0; i < v.size(); ++i) out_idx[i] = v[i].idx;
  return (long)v.size();
}

/* ------------------------------------------------------------------------------------------
 * a6. -fast clustering -- src/BreakID.cc:1046-1160.  Input order = order after a4.
 * Output: surviving original indices + cluster id (1-based, first appearance in p1 order). */
long orc_cluster_fast(long n, const uint32_t *p1, const uint32_t *p2, double w,
                      uint32_t *out_idx, int32_t *out_cluster, int *roots)
{
  struct E { uint32_t idx; int k1, k2; };
  std::vector<E> e(n), tmp;
  for (long i = 0; i < n; ++i) e[i] = E{(uint32_t)i, 0, 0};
  const size_t min_reads = 2;
  auto sweep = [&](const uint32_t *pp, bool second) {
    tmp.clear();
    long m = (long)e.size();
    if (m == 0) return;                     /* the reference reads enspan[0] of an empty vector here (:1095) */
    std::vector<long> cl{0};
    int k = 1;
    long pre = pp[e[0].idx];
    for (long i = 1; i < m; ++i) {
      if ((double)pp[e[i].idx] <= (double)pre + w && i != m - 1) cl.push_back(i);   /* :1064,:1100 */
      else {
        if (cl.size() >= min_reads) {
          for (long j : cl) { if (second) e[j].k2 = k; else e[j].k1 = k; tmp.push_back(e[j]); }
          ++k;
        }
        pre = pp[e[i].idx];
        cl.clear(); cl.push_back(i);
      }
    }
    e = tmp;
  };
  auto sort_by = [&](const uint32_t *pp) {
    std::vector<KeyIdx> v(e.size());
    for (size_t i = 0; i < e.size(); ++i) v[i] = KeyIdx{pp[e[i].idx], (uint32_t)i};
    std::sort(v.begin(), v.end(), cmp_key);
    std::vector<E> r(e.size());
    for (size_t i = 0; i < e.size(); ++i) r[i] = e[v[i].idx];
    e.swap(r);
  };
  sweep(p1, false);
  sort_by(p2);                                                             /* :1091 */
  sweep(p2, true);
  sort_by(p1);                                                             /* :1127 */
  std::map<std::pair<int, int>, int> cnt, cl;                              /* key / key_cl (:1129-1157) */
  for (auto &x : e) cnt[{x.k1, x.k2}]++;
  int k = 0; long m = 0;
  for (auto &x : e) {
    if (cnt[{x.k1, x.k2}] >= (int)min_reads) {
      auto it = cl.find({x.k1, x.k2});
      int id;
      if (it == cl.end()) { id = ++k; cl[{x.k1, x.k2}] = id; } else id = it->second;
      out_idx[m] = x.idx; out_cluster[m] = id; ++m;
    }
  }
  *roots = k;
  return m;
}

/* ------------------------------------------------------------------------------------------
 * a5. AHC, literal -- src/util_cluster.cc:7-396 + src/BreakID.cc:1304-1352.
 * Average linkage (distance_type hard-wired to 1, src/BreakID.cc:33,135). */
namespace {
struct Nb { int target; double d; Nb *prev, *next; };
struct LNode { int is_root; std::vector<int> pts; Nb *nbs; int ma, mb; };
struct Lit {
  long N; std::vector<LNode> nodes; int roots; std::vector<double> mat; std::vector<Nb *> pool;
  double m(int a, int b) const { return mat[(size_t)a * N + b]; }
  double dist(int cur, int tgt) const {                                     /* get_distance :158-199 */
    if (cur < N && tgt < N) return m(cur, tgt);
    const std::vector<int> &a = nodes[cur].pts, &b = nodes[tgt].pts;
    double total = 0.0;                                                      /* average_linkage :201-215 */
    for (size_t i = 0; i < a.size(); ++i) for (size_t j = 0; j < b.size(); ++j) total += m(a[i], b[j]);
    return total / (int)(a.size() * b.size());
  }
  void insert_sorted(Nb *cn, int cur) {                                      /* :249-297 */
    Nb *t = nodes[cur].nbs;
    auto before = [&](Nb *tt) {
      cn->next = tt;
      if (tt->prev) { tt->prev->next = cn; cn->prev = tt->prev; } else nodes[cur].nbs = cn;
      tt->prev = cn;
    };
    while (t->next) { if (t->d >= cn->d) { before(t); return; } t = t->next; }
    if (t->d > cn->d) before(t); else { cn->prev = t; t->next = cn; }
  }
  void update_neighbours() {                                                 /* :112-134 */
    int cur = (int)nodes.size() - 1, seen = 1, tgt = cur;
    while (seen < roots) {
      --tgt;
      if (nodes[tgt].is_root) {
        ++seen;
        Nb *cn = (Nb *)calloc(1, sizeof(Nb)); pool.push_back(cn);
        cn->target = tgt; cn->d = dist(cur, tgt);
        if (nodes[cur].nbs) insert_sorted(cn, cur); else nodes[cur].nbs = cn;
      }
    }
  }
};
}  // namespace

/* returns number of nodes; fills is_root / merged children (size 2n) */
long orc_ahc_tree(long n, const double *x, const double *y, long thr,
                  int32_t *is_root, int32_t *merged_a, int32_t *merged_b)
{
  Lit c; c.N = n; c.roots = 0;
  c.mat.resize((size_t)n * n);
  for (long i = 0; i < n; ++i) for (long j = 0; j < n; ++j) {
    double dx = x[i] - x[j], dy = y[i] - y[j];
    c.mat[(size_t)i * n + j] = sqrt(dx * dx + dy * dy);                      /* :79-84, pow(.,2) folds to a product */
  }
  for (long i = 0; i < n; ++i) {                                             /* add_leaves :86-110 */
    c.nodes.push_back(LNode{1, {(int)i}, nullptr, -1, -1}); c.roots++;
    c.update_neighbours();
  }
  while (c.roots > 1) {                                                      /* merge_clusters :299-318 */
    double best = DBL_MAX; int first = -1, second = 0;
    int seen = 0, j = (int)c.nodes.size();
    while (seen < c.roots) {                                                 /* :320-334 */
      --j;
      if (!c.nodes[j].is_root) continue;
      ++seen;
      for (Nb *q = c.nodes[j].nbs; q; q = q->next)                           /* :337-355 */
        if (c.nodes[q->target].is_root) {
          if (first == -1 || q->d < best) { first = j; second = q->target; best = q->d; }
          break;
        }
    }
    if (first != -1 && best <= (double)thr) {                                /* :308 */
      LNode nn{1, {}, nullptr, first, second};                               /* merge :357-396 */
      c.nodes[first].is_root = 0; c.nodes[second].is_root = 0;
      nn.pts = c.nodes[first].pts;
      nn.pts.insert(nn.pts.end(), c.nodes[second].pts.begin(), c.nodes[second].pts.end());
      c.nodes.push_back(nn); c.roots--;
      c.update_neighbours();
    } else break;
  }
  long nn = (long)c.nodes.size();
  for (long i = 0; i < nn; ++i) { is_root[i] = c.nodes[i].is_root; merged_a[i] = c.nodes[i].ma; merged_b[i] = c.nodes[i].mb; }
  for (Nb *p : c.pool) free(p);
  return nn;
}

/* from a merge tree to the reference's pair re-emission (src/BreakID.cc:1328-1352): roots with
 * >= 2 points in node order get k = 0,1,..; points in `points` order (first.points ++ second.points) */
static long tree_to_clusters(long n, long nn, const int32_t *is_root, const int32_t *ma, const int32_t *mb,
                             uint32_t *out_idx, int32_t *out_cluster, int *roots)
{
  std::vector<std::vector<int>> pts(nn);
  for (long i = 0; i < nn; ++i) {
    if (i < n) pts[i] = {(int)i};
    else { pts[i] = pts[ma[i]]; pts[i].insert(pts[i].end(), pts[mb[i]].begin(), pts[mb[i]].end()); }
  }
  long m = 0; int k = 0, r = 0;
  for (long i = 0; i < nn; ++i) {
    if (is_root[i]) ++r;
    if (is_root[i] && pts[i].size() >= 2) {
      for (int p : pts[i]) { out_idx[m] = (uint32_t)p; out_cluster[m] = k; ++m; }
      ++k;
    }
  }
  *roots = r;                                                                 /* print_root_nodes :398-417 */
  return m;
}

long orc_cluster_ahc(long n, const uint32_t *p1, const uint32_t *p2, double thr,
                     uint32_t *out_idx, int32_t *out_cluster, int *roots)
{
  std::vector<double> x(n), y(n);
  for (long i = 0; i < n; ++i) { x[i] = p1[i]; y[i] = p2[i]; }             /* build_pair_array :1795-1806 */
  std::vector<int32_t> r(2 * n + 1), a(2 * n + 1), b(2 * n + 1);
  long nn = orc_ahc_tree(n, x.data(), y.data(), (long)thr, r.data(), a.data(), b.data());
  return tree_to_clusters(n, nn, r.data(), a.data(), b.data(), out_idx, out_cluster, roots);
}

/* ------------------------------------------------------------------------------------------
 * MODEL of the device AHC formulation (SURVEY.md App. A4 + the closed-form tie rule below).
 *
 *  * Components: sort by x, cut at x-gaps > thr; inside a piece sort by y, cut at y-gaps > thr.
 *    Points of different components are farther apart than thr, so no linkage across components
 *    can ever be <= thr and only in-component neighbour rows are kept.
 *  * Node j keeps a ROW D(j,t) over the in-component roots t < j that existed when j was created
 *    (leaf rows are recomputed from coordinates).  The reference's sorted list is replaced by:
 *      winner(j) = among still-root t with minimal D: let T = {t : D(j,t) == dmin} over the whole
 *      row (root or not), t1 > t2 its two highest indices.  The list holds T in ascending index
 *      order, except that t1 precedes t2 iff, when t2 was inserted, t1 was the list tail:
 *      every row entry with index in (t2, j) other than t1 has D < dmin AND no out-of-component
 *      root with index in (t2, j) existed when j was created ("sentinel", insert_sorted's tail
 *      exception src/util_cluster.cc:266-273).  So winner = min(S) unless min(S)==t2 && t1 in S &&
 *      exception -> t1.
 *  * Sentinel arithmetic: every merged node stores its global creation rank g and its rank l
 *      inside its component.  For merged j and t2: if t2 is merged, an out-of-component root in
 *      (t2,j) exists iff (g_j-g_t2) > (l_j-l_t2); if t2 is a leaf it exists iff g_j > l_j (some
 *      other component has merged before) or an out-of-component leaf index > t2 exists.
 *      For leaf j: static -- an out-of-component leaf with index in (t2, j).
 *  * Global loop: repeatedly take the component whose head event is minimal (ties -> higher global
 *      index of `first`), stop when it exceeds thr.
 * Output identical in shape to orc_ahc_tree (global node numbering).
 */
namespace {
struct MNode {
  int is_root, comp, lrank;       /* lrank: creation rank inside the component (merged only) */
  long grank;                     /* global creation rank (merged only) */
  int gidx;                       /* global node index */
  std::vector<int> pts;           /* global leaf indices */
  std::vector<int> row_t;         /* local target ids (descending) */
  std::vector<double> row_d;
  int best_t; double best_d;      /* cached winner (local id) or -1 */
};
struct Comp {
  std::vector<int> leaves;        /* global leaf indices ascending = local ids 0..c-1 */
  std::vector<MNode> nodes;       /* local id order */
  int merges;
  int hi_oc_leaf;                 /* highest global leaf index NOT in this component (-1 if none) */
  int head_j; double head_d;      /* current best event */
  long flag_decisions;            /* decisions the device's speculative pass flags (orc_model_ahc_flags) */
};
}  // namespace

static long g_model_exc_taken = 0, g_model_exc_blocked = 0;
void orc_model_ahc_counters(long *taken, long *blocked) { *taken = g_model_exc_taken; *blocked = g_model_exc_blocked; }

/* Flag predictor.  The device's speculative pass (bkid_cluster.cuh ahc_find_best<false>) flags a component when a tail
 * exception needs the out-of-component sentinel and that cannot be settled statically: j is a merged node, unless t2 is a
 * leaf and some out-of-component leaf index lies above it.  Up to its first such decision a component takes the same path
 * here and on the device, so "flagged" == "at least one such decision in the model".  Counts of the last
 * orc_model_ahc_tree call: components flagged, and all such decisions. */
static long g_model_flag_comps = 0, g_model_flag_decisions = 0;
void orc_model_ahc_flags(long *flagged_comps, long *decisions) { *flagged_comps = g_model_flag_comps; *decisions = g_model_flag_decisions; }

long orc_model_ahc_tree(long n, const double *x, const double *y, long thr,
                        int32_t *is_root, int32_t *merged_a, int32_t *merged_b)
{
  /* ---- components ---- */
  std::vector<int> comp_of(n, -1);
  std::vector<Comp> comps;
  {
    std::vector<int> ox(n);
    for (long i = 0; i < n; ++i) ox[i] = (int)i;
    std::stable_sort(ox.begin(), ox.end(), [&](int a, int b) { return x[a] < x[b]; });
    long s = 0;
    while (s < n) {
      long e = s + 1;
      while (e < n && !(x[ox[e]] - x[ox[e - 1]] > (double)thr)) ++e;
      std::vector<int> oy(ox.begin() + s, ox.begin() + e);
      std::stable_sort(oy.begin(), oy.end(), [&](int a, int b) { return y[a] < y[b]; });
      size_t s2 = 0;
      while (s2 < oy.size()) {
        size_t e2 = s2 + 1;
        while (e2 < oy.size() && !(y[oy[e2]] - y[oy[e2 - 1]] > (double)thr)) ++e2;
        Comp c; c.merges = 0; c.head_j = -1; c.head_d = DBL_MAX; c.hi_oc_leaf = -1; c.flag_decisions = 0;
        c.leaves.assign(oy.begin() + s2, oy.begin() + e2);
        std::sort(c.leaves.begin(), c.leaves.end());
        for (int l : c.leaves) comp_of[l] = (int)comps.size();
        comps.push_back(c);
        s2 = e2;
      }
      s = e;
    }
  }
  auto euclid = [&](int a, int b) { double dx = x[a] - x[b], dy = y[a] - y[b]; return sqrt(dx * dx + dy * dy); };
  /* lo_oc[j] = highest leaf index < j not in j's component (-1 if none) */
  std::vector<int> lo_oc(n, -1);
  for (long j = 0; j < n; ++j) { long r = j - 1; while (r >= 0 && comp_of[r] == comp_of[j]) --r; lo_oc[j] = (int)r; }
  for (size_t ci = 0; ci < comps.size(); ++ci) {
    Comp &c = comps[ci];
    long r = n - 1; while (r >= 0 && comp_of[r] == (int)ci) --r;
    c.hi_oc_leaf = (int)r;
    for (size_t k = 0; k < c.leaves.size(); ++k) {
      MNode nd; nd.is_root = 1; nd.comp = (int)ci; nd.lrank = -1; nd.grank = -1; nd.gidx = c.leaves[k];
      nd.pts = {c.leaves[k]}; nd.best_t = -1; nd.best_d = 0;
      c.nodes.push_back(nd);
    }
  }
  long total_merges = 0;
  /* distance from node j (local) to target t (local): row lookup or recompute */
  auto rowd = [&](Comp &c, int j, int t) -> double {
    int cl = (int)c.leaves.size();
    if (j < cl) return euclid(c.leaves[j], c.leaves[t]);
    MNode &nj = c.nodes[j];
    for (size_t k = 0; k < nj.row_t.size(); ++k) if (nj.row_t[k] == t) return nj.row_d[k];
    return DBL_MAX;
  };
  /* winner among still-root targets of node j */
  auto find_best = [&](Comp &c, int j) {
    int cl = (int)c.leaves.size();
    MNode &nj = c.nodes[j];
    std::vector<int> ts;                    /* row targets (roots at creation), any order */
    if (j < cl) { for (int t = j - 1; t >= 0; --t) ts.push_back(t); }
    else ts = nj.row_t;
    double dmin = DBL_MAX; int tmin = -1;
    for (int t : ts) if (c.nodes[t].is_root) { double d = rowd(c, j, t); if (d < dmin || (d == dmin && t < tmin)) { dmin = d; tmin = t; } }
    nj.best_t = tmin; nj.best_d = dmin;
    if (tmin < 0) return;
    int t1 = -1, t2 = -1;                   /* two highest indices in the row with D == dmin */
    for (int t : ts) if (rowd(c, j, t) == dmin) { if (t > t1) { t2 = t1; t1 = t; } else if (t > t2) t2 = t; }
    if (t2 < 0 || tmin != t2 || !c.nodes[t1].is_root) return;
    /* in-component part of the tail test */
    for (int t : ts) if (t > t2 && t != t1 && !(rowd(c, j, t) < dmin)) return;
    /* out-of-component sentinel */
    if (j >= cl && !(t2 < cl && c.hi_oc_leaf > c.leaves[t2])) ++c.flag_decisions;
    bool sentinel;
    if (j < cl) sentinel = lo_oc[c.leaves[j]] > c.leaves[t2];
    else if (t2 >= cl) sentinel = (nj.grank - c.nodes[t2].grank) > (long)(nj.lrank - c.nodes[t2].lrank);
    else sentinel = (nj.grank > (long)nj.lrank) || (c.hi_oc_leaf > c.leaves[t2]);
    if (!sentinel) { nj.best_t = t1; ++g_model_exc_taken; } else ++g_model_exc_blocked;
  };
  auto comp_head = [&](Comp &c) {
    c.head_j = -1; c.head_d = DBL_MAX;
    for (int j = (int)c.nodes.size() - 1; j >= 0; --j) {
      MNode &nj = c.nodes[j];
      if (!nj.is_root || nj.best_t < 0) continue;
      if (c.head_j == -1 || nj.best_d < c.head_d) { c.head_j = j; c.head_d = nj.best_d; }
    }
  };
  for (Comp &c : comps) {
    for (size_t j = 0; j < c.nodes.size(); ++j) find_best(c, (int)j);
    comp_head(c);
  }
  /* ---- global loop ---- */
  struct GNode { int a, b, root; };
  std::vector<GNode> g(n, GNode{-1, -1, 1});
  for (;;) {
    int bc = -1; double bd = DBL_MAX; int bg = -1;
    for (size_t ci = 0; ci < comps.size(); ++ci) {
      Comp &c = comps[ci];
      if (c.head_j < 0) continue;
      int gi = c.nodes[c.head_j].gidx;
      if (bc < 0 || c.head_d < bd || (c.head_d == bd && gi > bg)) { bc = (int)ci; bd = c.head_d; bg = gi; }
    }
    if (bc < 0 || !(bd <= (double)thr)) break;
    Comp &c = comps[bc];
    int first = c.head_j, second = c.nodes[first].best_t;
    MNode nn; nn.is_root = 1; nn.comp = bc; nn.lrank = c.merges; nn.grank = total_merges;
    nn.gidx = (int)(n + total_merges); nn.best_t = -1; nn.best_d = 0;
    c.merges++; total_merges++;
    nn.pts = c.nodes[first].pts;
    nn.pts.insert(nn.pts.end(), c.nodes[second].pts.begin(), c.nodes[second].pts.end());
    c.nodes[first].is_root = 0; c.nodes[second].is_root = 0;
    g[c.nodes[first].gidx].root = 0; g[c.nodes[second].gidx].root = 0;
    g.push_back(GNode{c.nodes[first].gidx, c.nodes[second].gidx, 1});
    int jn = (int)c.nodes.size();
    for (int t = jn - 1; t >= 0; --t) {
      if (!c.nodes[t].is_root) continue;
      const std::vector<int> &a = nn.pts, &b = c.nodes[t].pts;
      double total = 0.0;
      for (size_t i = 0; i < a.size(); ++i) for (size_t k = 0; k < b.size(); ++k) total += euclid(a[i], b[k]);
      nn.row_t.push_back(t); nn.row_d.push_back(total / (int)(a.size() * b.size()));
    }
    c.nodes.push_back(nn);
    find_best(c, jn);
    for (int j = 0; j < jn; ++j)
      if (c.nodes[j].is_root && (c.nodes[j].best_t == first || c.nodes[j].best_t == second)) find_best(c, j);
    comp_head(c);
  }
  g_model_flag_comps = g_model_flag_decisions = 0;
  for (const Comp &c : comps) { g_model_flag_comps += c.flag_decisions > 0; g_model_flag_decisions += c.flag_decisions; }
  long nn = (long)g.size();
  for (long i = 0; i < nn; ++i) { is_root[i] = g[i].root; merged_a[i] = g[i].a; merged_b[i] = g[i].b; }
  return nn;
}

long orc_model_cluster_ahc(long n, const uint32_t *p1, const uint32_t *p2, double thr,
                           uint32_t *out_idx, int32_t *out_cluster, int *roots)
{
  std::vector<double> x(n), y(n);
  for (long i = 0; i < n; ++i) { x[i] = p1[i]; y[i] = p2[i]; }
  std::vector<int32_t> r(2 * n + 1), a(2 * n + 1), b(2 * n + 1);
  long nn = orc_model_ahc_tree(n, x.data(), y.data(), (long)thr, r.data(), a.data(), b.data());
  return tree_to_clusters(n, nn, r.data(), a.data(), b.data(), out_idx, out_cluster, roots);
}


/* Per-bucket AHC of orc_run and orc_shard_bucket_clusters: the literal restatement by default; orc_set_ahc_model(1) switches
 * to the component model, which is pinned to the literal form by the CPU suite and is the only one fast enough for buckets
 * of thousands of points (the literal form is O(N^3)). */
static int g_ahc_model = 0;
void orc_set_ahc_model(int on) { g_ahc_model = on != 0; }
static long bucket_ahc(long n, const uint32_t *p1, const uint32_t *p2, double thr, uint32_t *out_idx, int32_t *out_cluster, int *roots)
{
  return g_ahc_model ? orc_model_cluster_ahc(n, p1, p2, thr, out_idx, out_cluster, roots)
                     : orc_cluster_ahc(n, p1, p2, thr, out_idx, out_cluster, roots);
}

/* ==========================================================================================
 * Refinement: a7 cluster summary, a8 split-read evidence, a9 vote, a10 depth/AF/type, a11 nib.
 * ========================================================================================== */
}  /* extern "C" (reopened below) */

namespace {

/* CigarRoller semantics (src/CigarRoller.cc:26-136,187-205; src/Cigar.cc:80-144; src/Cigar.h:215-228).
 * op codes: 1 match 3 insert 4 del 5 skip 6 softClip 7 hardClip 8 pad (enum src/Cigar.h:66-77). */
struct Roller {
  std::vector<std::pair<int, uint32_t>> ops;
  void add(int op, int count) {                                /* operator+= :26-46 */
    if ((uint32_t)count == 0) return;
    if (ops.empty() || ops.back().first != op) ops.push_back({op, (uint32_t)count});
    else ops.back().second += (uint32_t)count;
  }
  void add_char(int ch, int count) {                           /* Add(char,int) :67-117 */
    switch (ch) {
      case 0: case 'M': add(1, count); break;
      case 1: case 'I': add(3, count); break;
      case 2: case 'D': add(4, count); break;
      case 3: case 'N': add(5, count); break;
      case 4: case 'S': add(6, count); break;
      case 5: case 'H': add(7, count); break;
      case 6: case 'P': add(8, count); break;
      case 7: case '=': add(1, count); break;
      case 8: case 'X': add(1, count); break;
      default: break;                                          /* reference prints an error and continues */
    }
  }
  void set_text(const std::string &t) {                        /* Add(const char*) :120-136: the count is NOT reset */
    ops.clear();
    int cnt = 0;
    const char *c = t.c_str();
    while (*c) {
      if (isdigit((unsigned char)*c)) { char *e; cnt = (int)strtol(c, &e, 10); c = e; }
      else { add_char((unsigned char)*c, cnt); ++c; }
    }
  }
  void set_bam(const uint32_t *b, int n) { ops.clear(); for (int i = 0; i < n; ++i) add_char(b[i] & 0xF, (int)(b[i] >> 4)); }
  std::string str() const {                                    /* Cigar::getCigarString :22-38 */
    static const char ch[] = "?MMIDNSHP";
    std::string s;
    for (auto &o : ops) s += std::to_string(o.second) + ch[o.first];
    return s;
  }
  int matches() const { int n = 0; for (auto &o : ops) if (o.first == 1) n += o.second; return n; }
  int begin_clips() const { int n = 0; for (auto &o : ops) { if (o.first == 6 || o.first == 7) n += o.second; else break; } return n; }
  int end_clips() const { int n = 0; for (size_t i = ops.size(); i-- > 0;) { if (ops[i].first == 6 || ops[i].first == 7) n += ops[i].second; else break; } return n; }
  int ref_count() const { int n = 0; for (auto &o : ops) if (o.first == 1 || o.first == 2 || o.first == 4 || o.first == 5) n += o.second; return n; }
  uint32_t aln_end(uint32_t start) const { return start + ref_count() - 1; }   /* :316-321 */
};

/* full match of ([0-9]+[MS]){2} (src/CigarRoller.cc:326) */
bool regex_2ms(const std::string &s)
{
  size_t i = 0;
  for (int g = 0; g < 2; ++g) {
    size_t d = i;
    while (i < s.size() && s[i] >= '0' && s[i] <= '9') ++i;
    if (i == d || i >= s.size() || (s[i] != 'M' && s[i] != 'S')) return false;
    ++i;
  }
  return i == s.size();
}

/* src/CigarRoller.cc:323-346 */
bool complementary(const Roller &c1, const std::string &c2, int err)
{
  Roller r2; r2.set_text(c2);
  if (!(regex_2ms(c1.str()) && regex_2ms(c2))) return false;
  int c1_m = c1.matches(), c2_m = r2.matches();
  int c1_s = c1.begin_clips() + c1.end_clips(), c2_s = r2.end_clips() + r2.begin_clips();
  return (c1_m <= c2_s + err && c1_m >= c2_s - err) && (c1_m + c1_s == c2_m + c2_s);
}

std::vector<std::string> split_nonempty(const std::string &s, char delim)   /* src/util_bed.cc:194-222 */
{
  std::vector<std::string> r; std::string cur;
  for (char c : s) { if (c == delim) { if (!cur.empty()) r.push_back(cur); cur.clear(); } else cur += c; }
  if (!cur.empty()) r.push_back(cur);
  return r;
}

std::string chrom_id_name(int t)                                            /* src/util_bam.cc:128-142 */
{
  if (t == 23) return "chrY";
  if (t == 22) return "chrX";
  if (t >= 0 && t < 22) return "chr" + std::to_string(t + 1);
  return "";
}

struct Ev {
  uint64_t lo, hi; std::string pchr, schr, pcig, scig;
  uint32_t pstart, sstart, pend, send, pbp, sbp; bool secondary; uint16_t flag;
};

struct Recs {
  long n; const uint16_t *flag; const uint8_t *mapq; const int32_t *tid, *pos, *endpos; const uint64_t *nh;
  long n_sa; const uint32_t *sa_rec, *cig_off, *cig_ops, *sa_off; const uint8_t *sa_txt; const uint32_t *oc_off; const uint8_t *oc_txt;
  std::vector<long> sa_slot_of;   /* filled lazily: record -> sa slot or -1 */
};

int g_cigar_error = 0;

/* src/BreakID.cc:868-1037.  Region semantics of the index iterator (htslib hts.c:1776-1777,1963-1965):
 * same tid, pos0 < end, bam_endpos > max(beg,0). */
void find_sa_reads(const Recs &R, int tid, uint32_t region_start, uint32_t region_end,
                   std::map<std::pair<uint64_t, uint64_t>, std::vector<Ev>> &out, std::vector<Ev> *flat, int mismatch)
{
  out.clear();
  int beg = (int)region_start, end = (int)region_end;
  if (beg < 0) beg = 0;
  int total_cov = 0, total_ev = 0;
  if (end < beg) return;     /* NULL iterator: the reference then reads the rest of the file; out of domain here */
  /* records are coordinate sorted: binary search the first record of tid, then walk */
  long lo = 0, hi = R.n;
  while (lo < hi) { long m = (lo + hi) / 2; if ((uint32_t)R.tid[m] < (uint32_t)tid) lo = m + 1; else hi = m; }
  for (long i = lo; i < R.n && R.tid[i] == tid && R.pos[i] < end; ++i) {
    if (!(R.endpos[i] > beg)) continue;
    ++total_cov;                                                          /* :894 every record counts */
    long k = R.sa_slot_of[i];
    if (k < 0) continue;
    std::string sa((const char *)R.sa_txt + R.sa_off[k], R.sa_off[k + 1] - R.sa_off[k]);
    if (!(!sa.empty() && !(R.flag[i] & F_DUP) && (R.flag[i] & F_PAIRED))) continue;   /* :898 */
    std::string oc((const char *)R.oc_txt + R.oc_off[k], R.oc_off[k + 1] - R.oc_off[k]);
    std::vector<std::string> f = split_nonempty(sa, ',');
    if (f.size() < 4) continue;                                           /* reference: UB; out of domain */
    Roller sa_c, c1, rec_c;
    sa_c.set_text(f[3]);
    rec_c.set_bam(R.cig_ops + R.cig_off[k], (int)(R.cig_off[k + 1] - R.cig_off[k]));
    if (!oc.empty()) c1.set_text(oc); else c1 = rec_c;                    /* :906-913 */
    if (!complementary(c1, f[3], mismatch)) continue;                     /* :915 */
    ++total_ev;
    Ev e; e.lo = R.nh[2 * i]; e.hi = R.nh[2 * i + 1]; e.flag = R.flag[i];
    e.secondary = (R.flag[i] & F_SECONDARY) != 0;
    uint32_t sa_start = (uint32_t)atoi(f[1].c_str());                     /* stoi :929 */
    uint32_t sa_end = sa_c.aln_end(sa_start);
    uint32_t a_start = (uint32_t)((long)R.pos[i] + 1);                    /* getAlignmentStart */
    int alen = rec_c.ref_count();
    uint32_t a_end = (uint32_t)((long)(alen == 0 ? R.pos[i] : R.pos[i] + alen - 1) + 1);   /* getAlignmentEnd */
    std::string rec_str = rec_c.str();
    std::string own_chr = chrom_id_name(R.tid[i]);
    uint32_t own_end = !oc.empty() ? c1.aln_end(a_start) : a_end;
    std::string own_cig = !oc.empty() ? oc : rec_str;
    uint32_t own_bp, sa_bp;
    if (c1.begin_clips() != 0) own_bp = a_start; else if (c1.end_clips() != 0) own_bp = a_end; else { g_cigar_error = 1; continue; }
    if (sa_c.begin_clips() != 0) sa_bp = sa_start; else if (sa_c.end_clips() != 0) sa_bp = sa_end; else { g_cigar_error = 1; continue; }
    if (!e.secondary) {                                                   /* :933-973 */
      e.pchr = own_chr; e.pstart = a_start; e.pend = own_end; e.pcig = own_cig; e.pbp = own_bp;
      e.schr = f[0]; e.sstart = sa_start; e.send = sa_end; e.scig = f[3]; e.sbp = sa_bp;
    } else {                                                              /* :974-1016 */
      e.pchr = f[0]; e.pstart = sa_start; e.pend = sa_end; e.pcig = f[3]; e.pbp = sa_bp;
      e.schr = own_chr; e.sstart = a_start; e.send = own_end; e.scig = own_cig; e.sbp = own_bp;
    }
    out[{e.lo, e.hi}].push_back(e);
    if (flat) flat->push_back(e);
  }
  if (total_cov < 5 || total_ev < 2) { out.clear(); if (flat) flat->clear(); }   /* :1032-1035 */
}

/* src/BreakID.cc:577-857 (the "update version" vote, :797-855) */
int find_bp_pair(const std::map<std::pair<uint64_t, uint64_t>, std::vector<Ev>> &m1,
                 const std::map<std::pair<uint64_t, uint64_t>, std::vector<Ev>> &m2,
                 const std::string &p1_chr, int bp_err, int32_t *p1_bp, int32_t *p2_bp)
{
  std::vector<std::pair<int32_t, int32_t>> upd;
  for (auto &kv : m1) {
    auto it = m2.find(kv.first);
    if (it == m2.end()) continue;
    for (const Ev &a : kv.second) for (const Ev &b : it->second) {
      bool c = a.secondary != b.secondary && a.pchr == b.pchr && a.schr == b.schr && a.pstart == b.pstart &&
               a.sstart == b.sstart && a.pend == b.pend && a.send == b.send && a.pcig == b.pcig && a.scig == b.scig &&
               a.pbp == b.pbp && a.sbp == b.sbp;                           /* new_condition :627-637 */
      if (!c) continue;
      if (a.pchr == p1_chr) upd.push_back({(int32_t)a.pbp, (int32_t)a.sbp});  /* :647,671-672 */
      else upd.push_back({(int32_t)a.sbp, (int32_t)a.pbp});                   /* :717-718 */
    }
  }
  std::map<std::string, int> cnt;
  for (auto &u : upd) cnt[std::to_string(u.first) + "," + std::to_string(u.second)] = 0;
  for (auto &kv : cnt) {
    size_t c = kv.first.find(',');
    uint32_t k1 = (uint32_t)strtoull(kv.first.substr(0, c).c_str(), nullptr, 10);
    uint32_t k2 = (uint32_t)strtoull(kv.first.substr(c + 1).c_str(), nullptr, 10);
    for (auto &u : upd)                                                     /* mixed int32/uint32 compares :820-821 */
      if (((uint32_t)u.first <= k1 + bp_err && (uint32_t)u.first >= k1 - bp_err) &&
          ((uint32_t)u.second <= k2 + bp_err && (uint32_t)u.second >= k2 - bp_err)) kv.second++;
  }
  int best = 0; *p1_bp = -1; *p2_bp = -1;
  for (auto &kv : cnt)
    if (best < kv.second) {                                                 /* first strict max in string order :841-855 */
      best = kv.second;
      size_t c = kv.first.find(',');
      *p1_bp = (int32_t)(uint32_t)strtoull(kv.first.substr(0, c).c_str(), nullptr, 10);
      *p2_bp = (int32_t)(uint32_t)strtoull(kv.first.substr(c + 1).c_str(), nullptr, 10);
    }
  return best;
}

/* src/util_bed.cc:154-192: records overlapping 0-based [pos-1,pos) with qual>0, !DUP, PAIRED */
double single_base_depth(const Recs &R, int tid, uint64_t pos)
{
  int beg = (int)(pos - 1), end = (int)pos;
  if (beg < 0) beg = 0;
  if (end < beg) return 0;
  long lo = 0, hi = R.n;
  while (lo < hi) { long m = (lo + hi) / 2; if ((uint32_t)R.tid[m] < (uint32_t)tid) lo = m + 1; else hi = m; }
  int depth = 0;
  for (long i = lo; i < R.n && R.tid[i] == tid && R.pos[i] < end; ++i)
    if (R.endpos[i] > beg && R.mapq[i] > 0 && !(R.flag[i] & F_DUP) && (R.flag[i] & F_PAIRED)) ++depth;
  return depth;
}

/* src/nibtools.cc:38-64 + src/nibtools.h:23-59 */
char nib_base(const uint8_t *packed, uint64_t nbases, long pos, char prev)
{
  if (pos < 0 || (uint64_t)pos >= nbases) return prev;           /* reference leaves `base` untouched (status 4) */
  int b = packed[pos / 2];
  int v = (pos % 2 == 0) ? (b >> 4) : (b & 0xf);
  switch (v) { case 0: case 8: return 'T'; case 1: case 9: return 'C'; case 2: case 10: return 'A'; case 3: case 11: return 'G'; default: return 'N'; }
}

int longest_run(const char *s)                                    /* src/util_bed.cc:224-261 */
{
  int best = 0;
  for (int i = 0; s[i];) { int j = i; while (s[j] == s[i]) ++j; if (j - i > best) best = j - i; i = j; }
  return best;
}

}  // namespace

extern "C" {

int orc_is_complementary(const char *c1, const char *c2, int err)
{
  Roller r; r.set_text(c1);
  return complementary(r, c2, err) ? 1 : 0;
}

static void fill_recs(Recs &R, long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos,
                      const int32_t *endpos, const uint64_t *nh, long n_sa, const uint32_t *sa_rec, const uint32_t *cig_off,
                      const uint32_t *cig_ops, const uint32_t *sa_off, const uint8_t *sa_txt, const uint32_t *oc_off, const uint8_t *oc_txt)
{
  R.n = n; R.flag = flag; R.mapq = mapq; R.tid = tid; R.pos = pos; R.endpos = endpos; R.nh = nh;
  R.n_sa = n_sa; R.sa_rec = sa_rec; R.cig_off = cig_off; R.cig_ops = cig_ops; R.sa_off = sa_off; R.sa_txt = sa_txt;
  R.oc_off = oc_off; R.oc_txt = oc_txt;
  R.sa_slot_of.assign(n, -1);
  for (long k = 0; k < n_sa; ++k) R.sa_slot_of[sa_rec[k]] = k;
}

static void ev_to_pod(const Ev &s, orc_evidence &e, std::vector<std::string> &others)
{
  auto cid = [&](const std::string &x) -> int {
    if (x.empty()) return -1;
    for (int t = 0; t < 24; ++t) if (chrom_id_name(t) == x) return t;
    for (size_t k = 0; k < others.size(); ++k) if (others[k] == x) return -2 - (int)k;
    others.push_back(x); return -2 - (int)(others.size() - 1);
  };
  memset(&e, 0, sizeof e);
  e.name_lo = s.lo; e.name_hi = s.hi;
  e.primary_chr = cid(s.pchr); e.secondary_chr = cid(s.schr);
  e.primary_start = s.pstart; e.secondary_start = s.sstart; e.primary_end = s.pend; e.secondary_end = s.send;
  e.primary_bp = s.pbp; e.secondary_bp = s.sbp;
  e.primary_cigar_h = orc_str_hash(s.pcig.c_str()); e.secondary_cigar_h = orc_str_hash(s.scig.c_str());
  e.flag = s.flag; e.secondary = s.secondary;
}

/* evidence rows of one region in std::map<name> ... the reference iterates names in string order which
 * the hashes cannot reproduce, so rows are returned in RECORD order (tests sort both sides). */
long orc_find_sa_reads(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos,
                       const int32_t *endpos, const uint64_t *nh, long n_sa, const uint32_t *sa_rec, const uint32_t *cig_off,
                       const uint32_t *cig_ops, const uint32_t *sa_off, const uint8_t *sa_txt, const uint32_t *oc_off,
                       const uint8_t *oc_txt, int q_tid, uint32_t start, uint32_t end, orc_evidence **out)
{
  Recs R; fill_recs(R, n, flag, mapq, tid, pos, endpos, nh, n_sa, sa_rec, cig_off, cig_ops, sa_off, sa_txt, oc_off, oc_txt);
  std::map<std::pair<uint64_t, uint64_t>, std::vector<Ev>> m; std::vector<Ev> flat;
  find_sa_reads(R, q_tid, start, end, m, &flat, g_mismatch);
  orc_evidence *o = (orc_evidence *)calloc(flat.size() ? flat.size() : 1, sizeof(orc_evidence));
  std::vector<std::string> others;
  for (size_t k = 0; k < flat.size(); ++k) ev_to_pod(flat[k], o[k], others);
  *out = o;
  return (long)flat.size();
}

int orc_find_bp(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos,
                const int32_t *endpos, const uint64_t *nh, long n_sa, const uint32_t *sa_rec, const uint32_t *cig_off,
                const uint32_t *cig_ops, const uint32_t *sa_off, const uint8_t *sa_txt, const uint32_t *oc_off,
                const uint8_t *oc_txt, int tid1, const char *chr1, uint32_t s1, uint32_t e1, int tid2, uint32_t s2, uint32_t e2,
                int32_t *p1_bp, int32_t *p2_bp)
{
  Recs R; fill_recs(R, n, flag, mapq, tid, pos, endpos, nh, n_sa, sa_rec, cig_off, cig_ops, sa_off, sa_txt, oc_off, oc_txt);
  std::map<std::pair<uint64_t, uint64_t>, std::vector<Ev>> m1, m2;
  *p1_bp = -1; *p2_bp = -1;
  find_sa_reads(R, tid1, s1, e1, m1, nullptr, g_mismatch);
  if (!m1.empty()) find_sa_reads(R, tid2, s2, e2, m2, nullptr, g_mismatch);
  if (m1.empty() || m2.empty()) return 0;
  return find_bp_pair(m1, m2, chr1, g_bp_err, p1_bp, p2_bp);
}

double orc_single_base_depth(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos,
                             const int32_t *endpos, int q_tid, uint64_t q_pos)
{
  Recs R; R.n = n; R.flag = flag; R.mapq = mapq; R.tid = tid; R.pos = pos; R.endpos = endpos;
  return single_base_depth(R, q_tid, q_pos);
}

/* src/BreakID.cc:554-561: 41-mer = 1-based [bp-20, bp+20] */
void orc_neighbor_41(const uint8_t *packed, uint64_t nbases, int32_t bp, char *out42)
{
  memset(out42, 0, 42);
  char prev = 'N';
  int k = 0;
  for (int32_t i = bp - 20; i < bp; ++i) { prev = nib_base(packed, nbases, (long)i - 1, prev); out42[k++] = prev; }
  for (int32_t i = bp - 1; i < bp - 1 + 21; ++i) { prev = nib_base(packed, nbases, (long)i, prev); out42[k++] = prev; }
}
int orc_longest_repeat(const char *s) { return longest_run(s); }

/* ------------------------------------------------------------------------------------------
 * Whole hot path on one record batch -- what reference main() computes between
 * src/BreakID.cc:98 and :167, minus gene annotation and file writing.  Output: the valid clusters in
 * the order main() appends them (bucket order, then cluster id).
 * mode 0 = AHC (default), 1 = -fast.  nib_packed[t] may be NULL (41-mers left empty).
 * Returns the number of clusters, or -1 when the reference's fatal "error cigar" path was hit. */
long orc_run(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos,
             const int32_t *mtid, const int32_t *mpos, const int32_t *isize, const int32_t *endpos, const uint64_t *nh,
             long n_sa, const uint32_t *sa_rec, const uint32_t *cig_off, const uint32_t *cig_ops, const uint32_t *sa_off,
             const uint8_t *sa_txt, const uint32_t *oc_off, const uint8_t *oc_txt,
             int n_targets, const uint32_t *target_len, const char *const *names,
             const uint8_t *const *nib_packed, const uint64_t *nib_len,
             int qual, int times, int mode, double *mean_out, double *sd_out, double *dist_out, orc_cluster **out)
{
  g_cigar_error = 0;
  double mean, sd;
  orc_insert_stats(n, flag, isize, &mean, &sd, nullptr, nullptr, nullptr);
  double dist = orc_dist(mean, sd, times);
  if (mean_out) *mean_out = mean;
  if (sd_out) *sd_out = sd;
  if (dist_out) *dist_out = dist;
  orc_pair *pairs = nullptr;
  long np = orc_scan(n, flag, mapq, tid, pos, mtid, mpos, nh, n_targets, target_len, names, qual, dist, &pairs);
  Recs R; fill_recs(R, n, flag, mapq, tid, pos, endpos, nh, n_sa, sa_rec, cig_off, cig_ops, sa_off, sa_txt, oc_off, oc_txt);
  std::vector<orc_cluster> result;
  long s = 0;
  while (s < np) {
    long e = s;
    while (e < np && pairs[e].bucket == pairs[s].bucket) ++e;
    long nb = e - s;
    std::vector<uint32_t> p1(nb), p2(nb), idx(nb + 2);
    for (long i = 0; i < nb; ++i) { p1[i] = pairs[s + i].p1_chr_pos; p2[i] = pairs[s + i].p2_chr_pos; }
    long nm = orc_remove_isolated(nb, p1.data(), p2.data(), dist, idx.data());          /* :123 */
    if (nm >= 2) {                                                                       /* :125 */
      std::vector<uint32_t> q1(nm), q2(nm), cidx(nm + 2); std::vector<int32_t> cl(nm + 2);
      for (long i = 0; i < nm; ++i) { q1[i] = p1[idx[i]]; q2[i] = p2[idx[i]]; }
      int roots = 0;
      long nc = mode ? orc_cluster_fast(nm, q1.data(), q2.data(), dist, cidx.data(), cl.data(), &roots)
                     : bucket_ahc(nm, q1.data(), q2.data(), dist, cidx.data(), cl.data(), &roots);
      /* a7: per-cluster summary (src/BreakID.cc:222-352); order inside a cluster does not matter */
      std::map<long, std::vector<long>> members;
      for (long i = 0; i < nc; ++i) members[cl[i]].push_back(s + idx[cidx[i]]);
      for (auto &kv : members) {
        orc_cluster c; memset(&c, 0, sizeof c);
        const orc_pair &f = pairs[kv.second[0]];
        c.bucket = f.bucket; c.id = (int32_t)kv.first; c.p1_tid = f.p1_tid; c.p2_tid = f.p2_tid;
        uint64_t s1 = 0, s2 = 0; uint32_t mn1 = UINT32_MAX, mx1 = 0, mn2 = UINT32_MAX, mx2 = 0;
        bool t_diff = false, t_rev = false, t_same = false, t_def = false;
        for (long m : kv.second) {
          const orc_pair &p = pairs[m];
          s1 += p.p1_pos; s2 += p.p2_pos;
          mn1 = std::min(mn1, p.p1_pos); mx1 = std::max(mx1, p.p1_pos); mn2 = std::min(mn2, p.p2_pos); mx2 = std::max(mx2, p.p2_pos);
          if (p.p1_tid != p.p2_tid) t_diff = true;                                       /* :231-253 */
          else {
            if (p.p1_strand == '-' && p.p2_strand == '+') t_rev = true;
            if (p.p1_strand == p.p2_strand) t_same = true;
            if (p.p1_strand == '+' && p.p2_strand == '-') t_def = true;
          }
        }
        c.n_discordant_pair = (int64_t)kv.second.size();
        c.p1_mean_pos = (uint32_t)((double)s1 / (double)c.n_discordant_pair);            /* :342-343 */
        c.p2_mean_pos = (uint32_t)((double)s2 / (double)c.n_discordant_pair);
        c.p1_min_pos = mn1; c.p1_max_pos = mx1; c.p2_min_pos = mn2; c.p2_max_pos = mx2;
        int64_t md = (int64_t)(c.p1_mean_pos - c.p2_mean_pos);                            /* :345 */
        if (c.p1_tid == c.p2_tid && md <= 2 * dist && md >= -2 * dist) continue;          /* :348 */
        /* a8-a10 (src/BreakID.cc:421-485) */
        int w = (int)dist;                                                                /* const int w, :390 */
        uint32_t r1s = (uint32_t)(c.p1_mean_pos - w), r1e = (uint32_t)(c.p1_mean_pos + w);
        uint32_t r2s = (uint32_t)(c.p2_mean_pos - w), r2e = (uint32_t)(c.p2_mean_pos + w);
        std::map<std::pair<uint64_t, uint64_t>, std::vector<Ev>> m1, m2;
        find_sa_reads(R, c.p1_tid, r1s, r1e, m1, nullptr, g_mismatch);
        if (!m1.empty()) find_sa_reads(R, c.p2_tid, r2s, r2e, m2, nullptr, g_mismatch);
        if (m1.empty() || m2.empty()) continue;
        int32_t b1, b2;
        std::string p1name = c.p1_tid >= 0 ? names[c.p1_tid] : "*";
        int votes = find_bp_pair(m1, m2, p1name, g_bp_err, &b1, &b2);
        if (votes < 2) continue;                                                          /* :446 */
        c.p1_exact_pos = (uint32_t)b1; c.p2_exact_pos = b2; c.n_split_read = votes;
        c.p1_bp_depth = single_base_depth(R, c.p1_tid, (uint64_t)c.p1_exact_pos);
        c.p2_bp_depth = single_base_depth(R, c.p2_tid, (uint64_t)(int64_t)c.p2_exact_pos);
        c.p1_alle_freq = (float)c.n_split_read / (float)c.p1_bp_depth;                    /* :475-478 */
        c.p2_alle_freq = (float)c.n_split_read / (float)c.p2_bp_depth;
        c.fusion_type = 0;                                                                /* :1888-1907 */
        if (t_diff) c.fusion_type = 1;
        if (t_same) c.fusion_type = 2;
        if (t_rev) c.fusion_type = 3;
        if (t_def) c.fusion_type = 4;
        if (nib_packed) {
          if (c.p1_tid >= 0 && nib_packed[c.p1_tid]) orc_neighbor_41(nib_packed[c.p1_tid], nib_len[c.p1_tid], (int32_t)c.p1_exact_pos, c.p1_rpt);
          if (c.p2_tid >= 0 && nib_packed[c.p2_tid]) orc_neighbor_41(nib_packed[c.p2_tid], nib_len[c.p2_tid], c.p2_exact_pos, c.p2_rpt);
          c.is_rpt = (longest_run(c.p1_rpt) > 10 || longest_run(c.p2_rpt) > 10) ? 1 : 0;
        }
        result.push_back(c);
      }
    }
    s = e;
  }
  free(pairs);
  orc_cluster *o = (orc_cluster *)calloc(result.size() ? result.size() : 1, sizeof(orc_cluster));
  for (size_t i = 0; i < result.size(); ++i) o[i] = result[i];
  *out = o;
  if (g_cigar_error) return -1;
  return (long)result.size();
}


/* ==========================================================================================
 * Sharded decomposition of the same path (mirrors the bkid_shard_* entry points of the C ABI): the
 * records are cut into contiguous slices of the coordinate-sorted stream, candidates are exchanged by
 * name hash, pairs by bucket owner, coverage / depth are partial counts that get summed, and the
 * split-read evidence table is global.  tests/test_multi_gloo.py runs these pieces in two processes
 * over gloo and requires the result to equal orc_run on the unsplit input.
 * ========================================================================================== */
typedef struct {
  uint64_t name_lo, name_hi;
  int32_t tid, pos, mtid, mpos;
  uint64_t gidx;
  uint16_t flag;
  uint8_t mapq;
  uint8_t _pad[5];
} orc_cand;

typedef struct {
  uint64_t pchr, schr, pcig, scig, name_lo, name_hi;
  uint32_t pstart, sstart, pend, send, pbp, sbp;
  int32_t tid, pos, endpos;
  uint8_t ok, fatal, secondary, _pad;
} orc_sarow;

static uint64_t chr_code_str(const std::string &x)
{
  if (x.empty()) return ~0ull;
  for (int t = 0; t < 24; ++t) if (chrom_id_name(t) == x) return (uint64_t)t;
  return orc_str_hash(x.c_str()) | (1ull << 63);
}

long orc_shard_sd_partial(long n, const uint16_t *flag, const int32_t *isize, double mean, long t_in)
{
  const uint32_t filter = F_UNMAP | F_SECONDARY | F_QCFAIL | F_DUP;
  long t = t_in;
  for (long i = 0; i < n; ++i)
    if ((flag[i] & F_PAIRED) && (flag[i] & F_PROPER) && !(flag[i] & filter)) {
      double x = (double)abs(isize[i]);
      t += (x - mean) * (x - mean);
    }
  return t;
}

long orc_shard_candidates(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos, const int32_t *mtid,
                          const int32_t *mpos, const uint64_t *nh, long qual, uint64_t index_offset, orc_cand **out)
{
  std::vector<orc_cand> v;
  for (long i = 0; i < n; ++i)
    if ((long)mapq[i] >= qual && !(flag[i] & F_DUP) && !(flag[i] & F_SECONDARY) && (flag[i] & F_PAIRED) && !(flag[i] & F_PROPER)) {
      orc_cand c; memset(&c, 0, sizeof c);
      c.name_lo = nh[2 * i]; c.name_hi = nh[2 * i + 1]; c.tid = tid[i]; c.pos = pos[i]; c.mtid = mtid[i]; c.mpos = mpos[i];
      c.gidx = index_offset + (uint64_t)i; c.flag = flag[i]; c.mapq = mapq[i];
      v.push_back(c);
    }
  orc_cand *o = (orc_cand *)calloc(v.size() ? v.size() : 1, sizeof(orc_cand));
  for (size_t i = 0; i < v.size(); ++i) o[i] = v[i];
  *out = o;
  return (long)v.size();
}

/* join over candidates given in global file order; pairs carry bucket = rank of "chrA_chrB" among ALL possible
 * names (rank table as in orc_bucket_rank_table) and the second-seen mate's global index in orig | _pad<<32 */
long orc_shard_join(long n, const orc_cand *cand, int n_targets, const uint32_t *target_len, const int32_t *rank_table, double w, orc_pair **out)
{
  std::unordered_map<H128, long, H128Hash> store;
  std::vector<orc_pair> emitted;
  for (long i = 0; i < n; ++i) {
    H128 h{cand[i].name_lo, cand[i].name_hi};
    auto it = store.find(h);
    if (it == store.end()) { store[h] = i; continue; }
    const orc_cand &I = cand[i], &J = cand[it->second];
    int ti = I.tid < 0 ? -1 : I.tid, tj = J.tid < 0 ? -1 : J.tid;
    long pi = (long)I.pos + 1, pj = (long)J.pos + 1;
    if (ti != tj || (double)labs(pi - pj) >= w) {
      uint32_t c1 = genome_pos(target_len, I.tid, I.pos), c2 = genome_pos(target_len, I.mtid, I.mpos);
      orc_pair p; memset(&p, 0, sizeof p);
      p.name_lo = h.lo; p.name_hi = h.hi;
      if (c1 <= c2) {
        p.p1_flag = I.flag; p.p1_tid = ti; p.p1_pos = (uint32_t)pi; p.p1_mapq = I.mapq; p.p1_chr_pos = c1; p.p2_chr_pos = c2;
        p.p2_flag = J.flag; p.p2_tid = tj; p.p2_pos = (uint32_t)pj; p.p2_mapq = J.mapq;
      } else {
        p.p2_flag = I.flag; p.p2_tid = ti; p.p2_pos = (uint32_t)pi; p.p2_mapq = I.mapq; p.p1_chr_pos = c2; p.p2_chr_pos = c1;
        p.p1_flag = J.flag; p.p1_tid = tj; p.p1_pos = (uint32_t)pj; p.p1_mapq = J.mapq;
      }
      p.p1_strand = (p.p1_flag & F_REVERSE) ? '-' : '+';
      p.p2_strand = (p.p2_flag & F_REVERSE) ? '-' : '+';
      p.bucket = rank_table[(p.p1_tid + 1) * (n_targets + 1) + (p.p2_tid + 1)];
      p.cluster = -1;
      p.orig = (uint32_t)(I.gidx & 0xffffffffull); p._pad = (uint32_t)((I.gidx >> 32) & 0xff);
      emitted.push_back(p);
    }
    store.erase(it);
  }
  orc_pair *o = (orc_pair *)calloc(emitted.size() ? emitted.size() : 1, sizeof(orc_pair));
  for (size_t i = 0; i < emitted.size(); ++i) o[i] = emitted[i];
  *out = o;
  return (long)emitted.size();
}

/* mask + cluster + summary of the buckets present in `pairs` (sorted by (bucket rank, second-mate index)); cluster
 * records keep bucket = global rank and are not refined yet (exact positions -1) */
long orc_shard_bucket_clusters(long np, const orc_pair *pairs, double dist, int mode, orc_cluster **out)
{
  std::vector<orc_cluster> result;
  long s = 0;
  while (s < np) {
    long e = s;
    while (e < np && pairs[e].bucket == pairs[s].bucket) ++e;
    long nb = e - s;
    std::vector<uint32_t> p1(nb), p2(nb), idx(nb + 2);
    for (long i = 0; i < nb; ++i) { p1[i] = pairs[s + i].p1_chr_pos; p2[i] = pairs[s + i].p2_chr_pos; }
    long nm = orc_remove_isolated(nb, p1.data(), p2.data(), dist, idx.data());
    if (nm >= 2) {
      std::vector<uint32_t> q1(nm), q2(nm), cidx(nm + 2); std::vector<int32_t> cl(nm + 2);
      for (long i = 0; i < nm; ++i) { q1[i] = p1[idx[i]]; q2[i] = p2[idx[i]]; }
      int roots = 0;
      long nc = mode ? orc_cluster_fast(nm, q1.data(), q2.data(), dist, cidx.data(), cl.data(), &roots)
                     : bucket_ahc(nm, q1.data(), q2.data(), dist, cidx.data(), cl.data(), &roots);
      std::map<long, std::vector<long>> members;
      for (long i = 0; i < nc; ++i) members[cl[i]].push_back(s + idx[cidx[i]]);
      for (auto &kv : members) {
        orc_cluster c; memset(&c, 0, sizeof c);
        const orc_pair &f = pairs[kv.second[0]];
        c.bucket = f.bucket; c.id = (int32_t)kv.first; c.p1_tid = f.p1_tid; c.p2_tid = f.p2_tid;
        uint64_t s1 = 0, s2 = 0; uint32_t mn1 = UINT32_MAX, mx1 = 0, mn2 = UINT32_MAX, mx2 = 0;
        bool t_diff = false, t_rev = false, t_same = false, t_def = false;
        for (long m : kv.second) {
          const orc_pair &p = pairs[m];
          s1 += p.p1_pos; s2 += p.p2_pos;
          mn1 = std::min(mn1, p.p1_pos); mx1 = std::max(mx1, p.p1_pos); mn2 = std::min(mn2, p.p2_pos); mx2 = std::max(mx2, p.p2_pos);
          if (p.p1_tid != p.p2_tid) t_diff = true;
          else {
            if (p.p1_strand == '-' && p.p2_strand == '+') t_rev = true;
            if (p.p1_strand == p.p2_strand) t_same = true;
            if (p.p1_strand == '+' && p.p2_strand == '-') t_def = true;
          }
        }
        c.n_discordant_pair = (int64_t)kv.second.size();
        c.p1_mean_pos = (uint32_t)((double)s1 / (double)c.n_discordant_pair);
        c.p2_mean_pos = (uint32_t)((double)s2 / (double)c.n_discordant_pair);
        c.p1_min_pos = mn1; c.p1_max_pos = mx1; c.p2_min_pos = mn2; c.p2_max_pos = mx2;
        int64_t md = (int64_t)(c.p1_mean_pos - c.p2_mean_pos);
        if (c.p1_tid == c.p2_tid && md <= 2 * dist && md >= -2 * dist) continue;
        c.fusion_type = 0;
        if (t_diff) c.fusion_type = 1;
        if (t_same) c.fusion_type = 2;
        if (t_rev) c.fusion_type = 3;
        if (t_def) c.fusion_type = 4;
        c.p1_exact_pos = 0xffffffffu; c.p2_exact_pos = -1;
        result.push_back(c);
      }
    }
    s = e;
  }
  orc_cluster *o = (orc_cluster *)calloc(result.size() ? result.size() : 1, sizeof(orc_cluster));
  for (size_t i = 0; i < result.size(); ++i) o[i] = result[i];
  *out = o;
  return (long)result.size();
}

/* one self-contained evidence row per SA-tagged record of the slice (same layout as the device's EvRow) */
void orc_shard_sa_rows(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos, const int32_t *endpos,
                       const uint64_t *nh, long n_sa, const uint32_t *sa_rec, const uint32_t *cig_off, const uint32_t *cig_ops,
                       const uint32_t *sa_off, const uint8_t *sa_txt, const uint32_t *oc_off, const uint8_t *oc_txt, orc_sarow *rows)
{
  for (long k = 0; k < n_sa; ++k) {
    orc_sarow r; memset(&r, 0, sizeof r);
    long i = sa_rec[k];
    r.tid = tid[i]; r.pos = pos[i]; r.endpos = endpos[i]; r.name_lo = nh[2 * i]; r.name_hi = nh[2 * i + 1];
    rows[k] = r;
    std::string sa((const char *)sa_txt + sa_off[k], sa_off[k + 1] - sa_off[k]);
    if (!(!sa.empty() && !(flag[i] & F_DUP) && (flag[i] & F_PAIRED))) continue;
    std::string oc((const char *)oc_txt + oc_off[k], oc_off[k + 1] - oc_off[k]);
    std::vector<std::string> f = split_nonempty(sa, ',');
    if (f.size() < 4) continue;
    Roller sa_c, c1, rec_c;
    sa_c.set_text(f[3]);
    rec_c.set_bam(cig_ops + cig_off[k], (int)(cig_off[k + 1] - cig_off[k]));
    if (!oc.empty()) c1.set_text(oc); else c1 = rec_c;
    if (!complementary(c1, f[3], g_mismatch)) continue;
    r.ok = 1; r.secondary = (flag[i] & F_SECONDARY) ? 1 : 0;
    uint32_t sa_start = (uint32_t)atoi(f[1].c_str()), sa_end = sa_c.aln_end(sa_start);
    uint32_t a_start = (uint32_t)((long)pos[i] + 1);
    int alen = rec_c.ref_count();
    uint32_t a_end = (uint32_t)((long)(alen == 0 ? pos[i] : pos[i] + alen - 1) + 1);
    uint64_t own_chr = chr_code_str(chrom_id_name(tid[i])), sa_chr = chr_code_str(f[0]);
    uint32_t own_end = !oc.empty() ? c1.aln_end(a_start) : a_end;
    uint64_t own_cig = orc_str_hash((!oc.empty() ? oc : rec_c.str()).c_str()), sa_cig = orc_str_hash(f[3].c_str());
    uint32_t own_bp = 0, sa_bp = 0;
    if (c1.begin_clips() != 0) own_bp = a_start; else if (c1.end_clips() != 0) own_bp = a_end; else r.fatal = 1;
    if (sa_c.begin_clips() != 0) sa_bp = sa_start; else if (sa_c.end_clips() != 0) sa_bp = sa_end; else r.fatal = 1;
    if (!r.secondary) {
      r.pchr = own_chr; r.pstart = a_start; r.pend = own_end; r.pcig = own_cig; r.pbp = own_bp;
      r.schr = sa_chr; r.sstart = sa_start; r.send = sa_end; r.scig = sa_cig; r.sbp = sa_bp;
    } else {
      r.pchr = sa_chr; r.pstart = sa_start; r.pend = sa_end; r.pcig = sa_cig; r.pbp = sa_bp;
      r.schr = own_chr; r.sstart = a_start; r.send = own_end; r.scig = own_cig; r.sbp = own_bp;
    }
    rows[k] = r;
  }
}

static void cluster_regions(const orc_cluster &c, double dist, int *b1, int *e1, int *b2, int *e2)
{
  int w = (int)dist;
  *b1 = (int)(uint32_t)(c.p1_mean_pos - w); *e1 = (int)(uint32_t)(c.p1_mean_pos + w);
  *b2 = (int)(uint32_t)(c.p2_mean_pos - w); *e2 = (int)(uint32_t)(c.p2_mean_pos + w);
  if (*b1 < 0) *b1 = 0;
  if (*b2 < 0) *b2 = 0;
}

static uint32_t count_overlaps(long n, const int32_t *tid, const int32_t *pos, const int32_t *endpos, const uint16_t *flag, const uint8_t *mapq,
                               int t, int beg, int end, bool depth_only)
{
  if (end < beg || t < 0) return 0;
  uint32_t c = 0;
  for (long i = 0; i < n; ++i)
    if (tid[i] == t && pos[i] < end && endpos[i] > beg && (!depth_only || (mapq[i] > 0 && !(flag[i] & F_DUP) && (flag[i] & F_PAIRED)))) ++c;
  return c;
}

/* partial coverage of both regions of every cluster on one slice of records */
void orc_shard_coverage(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos, const int32_t *endpos,
                        long ncl, const orc_cluster *cl, double dist, uint32_t *cov)
{
  for (long c = 0; c < ncl; ++c) {
    int b1, e1, b2, e2;
    cluster_regions(cl[c], dist, &b1, &e1, &b2, &e2);
    cov[2 * c] = count_overlaps(n, tid, pos, endpos, flag, mapq, cl[c].p1_tid, b1, e1, false);
    cov[2 * c + 1] = count_overlaps(n, tid, pos, endpos, flag, mapq, cl[c].p2_tid, b2, e2, false);
  }
}

/* gate + pairing + vote on the GLOBAL row table with TOTAL coverage; returns -1 on the fatal cigar path */
long orc_shard_vote(long n_rows, const orc_sarow *rows, long ncl, orc_cluster *cl, const uint32_t *cov, int n_targets, const char *const *names,
                    double dist, uint32_t *valid)
{
  bool fatal = false;
  for (long c = 0; c < ncl; ++c) {
    valid[c] = 0;
    int b1, e1, b2, e2;
    cluster_regions(cl[c], dist, &b1, &e1, &b2, &e2);
    auto collect = [&](int t, int beg, int end, uint32_t coverage, std::vector<long> &ev) {
      ev.clear();
      if (end < beg || t < 0) return;
      for (long k = 0; k < n_rows; ++k)
        if (rows[k].tid == t && rows[k].pos < end && rows[k].endpos > beg && rows[k].ok) { ev.push_back(k); if (rows[k].fatal) fatal = true; }
      if (coverage < 5 || ev.size() < 2) ev.clear();
    };
    std::vector<long> l1, l2;
    collect(cl[c].p1_tid, b1, e1, cov[2 * c], l1);
    if (!l1.empty()) collect(cl[c].p2_tid, b2, e2, cov[2 * c + 1], l2);
    if (l1.empty() || l2.empty()) continue;
    uint64_t p1code = chr_code_str(cl[c].p1_tid >= 0 && cl[c].p1_tid < n_targets ? names[cl[c].p1_tid] : "*");
    std::vector<std::pair<int32_t, int32_t>> upd;
    for (long a : l1) for (long b : l2) {
      const orc_sarow &A = rows[a], &B = rows[b];
      if (A.name_lo == B.name_lo && A.name_hi == B.name_hi && A.secondary != B.secondary && A.pchr == B.pchr && A.schr == B.schr &&
          A.pstart == B.pstart && A.sstart == B.sstart && A.pend == B.pend && A.send == B.send && A.pcig == B.pcig && A.scig == B.scig &&
          A.pbp == B.pbp && A.sbp == B.sbp) {
        if (A.pchr == p1code) upd.push_back({(int32_t)A.pbp, (int32_t)A.sbp}); else upd.push_back({(int32_t)A.sbp, (int32_t)A.pbp});
      }
    }
    std::map<std::string, int> cnt;
    for (auto &u : upd) cnt[std::to_string(u.first) + "," + std::to_string(u.second)] = 0;
    int best = 0; int32_t bx = -1, by = -1;
    for (auto &kv : cnt) {
      size_t q = kv.first.find(',');
      uint32_t k1 = (uint32_t)strtoull(kv.first.substr(0, q).c_str(), nullptr, 10), k2 = (uint32_t)strtoull(kv.first.substr(q + 1).c_str(), nullptr, 10);
      for (auto &u : upd)
        if (((uint32_t)u.first <= k1 + g_bp_err && (uint32_t)u.first >= k1 - g_bp_err) &&
            ((uint32_t)u.second <= k2 + g_bp_err && (uint32_t)u.second >= k2 - g_bp_err)) kv.second++;
      if (best < kv.second) { best = kv.second; bx = (int32_t)k1; by = (int32_t)k2; }
    }
    if (best >= 2) { valid[c] = 1; cl[c].p1_exact_pos = (uint32_t)bx; cl[c].p2_exact_pos = by; cl[c].n_split_read = best; }
  }
  return fatal ? -1 : 0;
}

void orc_shard_depth(long n, const uint16_t *flag, const uint8_t *mapq, const int32_t *tid, const int32_t *pos, const int32_t *endpos,
                     long ncl, const orc_cluster *cl, const uint32_t *valid, uint32_t *depth)
{
  for (long c = 0; c < ncl; ++c) {
    depth[2 * c] = depth[2 * c + 1] = 0;
    if (!valid[c]) continue;
    uint64_t p1 = (uint64_t)cl[c].p1_exact_pos, p2 = (uint64_t)(int64_t)cl[c].p2_exact_pos;
    int b1 = (int)(p1 - 1), e1 = (int)p1, b2 = (int)(p2 - 1), e2 = (int)p2;
    if (b1 < 0) b1 = 0;
    if (b2 < 0) b2 = 0;
    depth[2 * c] = count_overlaps(n, tid, pos, endpos, flag, mapq, cl[c].p1_tid, b1, e1, true);
    depth[2 * c + 1] = count_overlaps(n, tid, pos, endpos, flag, mapq, cl[c].p2_tid, b2, e2, true);
  }
}

/* depth (totals), AF, 41-mers; compacts the valid clusters to the front and returns their number */
long orc_shard_finish(long ncl, orc_cluster *cl, const uint32_t *valid, const uint32_t *depth, const uint8_t *const *nib_packed, const uint64_t *nib_len)
{
  long m = 0;
  for (long c = 0; c < ncl; ++c) {
    if (!valid[c]) continue;
    orc_cluster x = cl[c];
    x.p1_bp_depth = depth[2 * c]; x.p2_bp_depth = depth[2 * c + 1];
    x.p1_alle_freq = (float)x.n_split_read / (float)x.p1_bp_depth;
    x.p2_alle_freq = (float)x.n_split_read / (float)x.p2_bp_depth;
    if (nib_packed) {
      if (x.p1_tid >= 0 && nib_packed[x.p1_tid]) orc_neighbor_41(nib_packed[x.p1_tid], nib_len[x.p1_tid], (int32_t)x.p1_exact_pos, x.p1_rpt);
      if (x.p2_tid >= 0 && nib_packed[x.p2_tid]) orc_neighbor_41(nib_packed[x.p2_tid], nib_len[x.p2_tid], x.p2_exact_pos, x.p2_rpt);
      x.is_rpt = (longest_run(x.p1_rpt) > 10 || longest_run(x.p2_rpt) > 10) ? 1 : 0;
    }
    cl[m++] = x;
  }
  return m;
}

}  /* extern "C" */

// ---- extension: banded edit distance (checker of bkid_op_banded_align) ------------------------------------------
extern "C" int orc_banded_edit(const unsigned char *q, int nq, const unsigned char *r, int nr, int w)
{
  if (nr - nq > w || nq - nr > w) return -1;
  const int INF = 1 << 20;
  std::vector<int> prev((size_t)nr + 1, INF), cur((size_t)nr + 1, INF);
  for (int j = 0; j <= nr && j <= w; ++j) prev[j] = j;
  for (int i = 1; i <= nq; ++i) {
    std::fill(cur.begin(), cur.end(), INF);
    int lo = i - w < 0 ? 0 : i - w, hi = i + w > nr ? nr : i + w;
    for (int j = lo; j <= hi; ++j) {
      if (j == 0) { cur[j] = i; continue; }
      int sub = (q[i - 1] == r[j - 1] && q[i - 1] != 'N') ? 0 : 1;
      int best = prev[j - 1] + sub;                          // (i-1, j-1) is always inside the band
      if (j - (i - 1) <= w && prev[j] + 1 < best) best = prev[j] + 1;          // (i-1, j) inside the band?
      if (j - 1 >= lo && cur[j - 1] + 1 < best) best = cur[j - 1] + 1;         // (i, j-1) inside the band?
      cur[j] = best > INF ? INF : best;
    }
    prev.swap(cur);
  }
  return prev[nr];
}
