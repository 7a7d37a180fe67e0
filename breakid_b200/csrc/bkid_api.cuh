// bkid_api.cuh -- context, host orchestration and the exported C ABI.  Included by bkid_core.cu.
#pragma once

#define GRID1(n, t) (unsigned)div_up((long long)(n), (t))

// slots (in 32-bit words) of the context's small device counter block `counters` (1 KB); 64-bit values are 8-byte aligned
enum CounterSlot {
  CS_G = 0,             // K1 results: 6 x u64 (G_SUM .. G_SPAN), 16 words reserved
  CS_SD_OUT = 16,       // sd_resolve: [0] total (i64), [1] out-of-regime flag (i64)
  CS_SDF = 20,          // sd_fast: sum floor(a), E, out-of-regime (u64 x 3)
  CS_SORT = 28,         // std::sort replay: active / terminal / small work-list sizes
  CS_TOTAL = 32,        // grand totals of the exclusive scans (u64 x 2)
  CS_HASH_ERR = 40,     // mate join: a mixed group beyond the fix-up cap
  CS_MAXSPAN = 44,      // max_span_kernel result
  CS_FATAL = 46,        // the reference's fatal "error cigar" condition was met
  CS_ROOTS = 48,        // AHC: number of final roots
  CS_MISSING = 50,      // an SA record is missing from the sparse mate/name table
  CS_DECODE = 52,       // device decode: totals of the six per-chunk scans (u64 x 6)
  CS_NC = 64,           // number of candidates found through the sparse table (u32)
  CS_XBAD = 65,         // the sparse table is not strictly ascending / points outside the batch
  CS_RG_TICKET = 66,    // AHC tie groups: the next group to hand out
  CS_SORT_HEAP = 67     // std::sort replay: depth-exhausted segments waiting for is_heap
};

struct Scratch {          // reusable device scratch for sorts / scans over `cap` elements
  DBuf keys, keys_alt, vals, vals_alt, hist, scan_tmp, a32, b32, c32, d32, e32;
  int ensure(long long n, cudaStream_t st)
  {
    size_t m = (size_t)std::max<long long>(n, 1);
    BK_TRY(keys.ensure(m * 8, 0, st)); BK_TRY(keys_alt.ensure(m * 8, 0, st));
    BK_TRY(vals.ensure(m * 4, 0, st)); BK_TRY(vals_alt.ensure(m * 4, 0, st));
    BK_TRY(hist.ensure(bk::radix_hist_elems(n) * 4, 0, st));
    BK_TRY(scan_tmp.ensure((bk::scan_tmp_elems(std::max<long long>((long long)bk::radix_hist_elems(n), n)) + 8) * 8, 0, st));
    BK_TRY(a32.ensure(m * 4 + 16, 0, st)); BK_TRY(b32.ensure(m * 4 + 16, 0, st)); BK_TRY(c32.ensure(m * 4 + 16, 0, st));
    BK_TRY(d32.ensure(m * 4 + 16, 0, st)); BK_TRY(e32.ensure(m * 4 + 16, 0, st));
    return 0;
  }
  bk::RadixTmp rt() { return bk::RadixTmp{keys_alt.as<uint64_t>(), vals_alt.as<uint32_t>(), hist.as<uint32_t>(), scan_tmp.as<unsigned long long>()}; }
  void release() { for (DBuf *b : {&keys, &keys_alt, &vals, &vals_alt, &hist, &scan_tmp, &a32, &b32, &c32, &d32, &e32}) b->release(); }
};

struct bkid_decoder;
static void decoder_free(bkid_ctx *c);

struct bkid_ctx {
  bkid_decoder *dec = nullptr;              // streaming BGZF/BAM decode state (bkid_bamdec.cuh)
  std::vector<int32_t> ex_iv;               // exclude intervals: merged, sorted (tid, beg, end) triples
  DBuf ex_tab, ex_lo, ex_len, ex_pre;
  long long n_excluded = 0;
  int device = 0, n_sm = 148;
  cudaStream_t st = nullptr, st2 = nullptr, st3 = nullptr;     // st2: side stream for the sd replay (overlaps the join); st3: max span (needed only by the refinement)
  bkid_params prm;
  int nt = 0;
  std::vector<uint32_t> target_len;
  std::vector<std::string> names;
  std::string err;
  // header tables
  DBuf d_cum, d_bucket_rank, d_canon;
  // resident record columns (file order)
  long long n = 0, cap_n = 0;
  bool borrowed = false;
  DBuf flag, mapq, tid, pos, isize, endpos, cls, cand_bits;
  DBuf isize16, span16;                     // narrow forms of the insert-size / span columns (kept narrow in HBM when the batches have them)
  int form_isize = 0, form_span = 0;        // 0 = undecided (empty context), 1 = wide (isize / endpos), 2 = narrow (isize16 / span16)
  long long reserve_hint = 0;               // bkid_reserve on an empty context: applied once the column forms are known
  const int16_t *p_isize16 = nullptr; const uint16_t *p_span16 = nullptr;
  long long n_x = 0;
  DBuf x_rec, x_mtid, x_mpos, x_nh;
  const uint16_t *p_flag = nullptr; const uint8_t *p_mapq = nullptr;
  const int32_t *p_tid = nullptr, *p_pos = nullptr, *p_isize = nullptr, *p_endpos = nullptr;
  const uint32_t *p_x_rec = nullptr; const int32_t *p_x_mtid = nullptr, *p_x_mpos = nullptr; const uint64_t *p_x_nh = nullptr;
  // SA side table
  long long n_sa = 0, n_cig = 0, sa_bytes = 0, oc_bytes = 0;
  DBuf sa_rec, cig_off, cig_ops, sa_off, sa_txt, oc_off, oc_txt;
  DBuf seq_off, seq4, seq_len; long long seq_bytes = 0; bool have_seq = false;      // optional read bases of the SA records
  const uint32_t *p_seq_off = nullptr; const uint8_t *p_seq4 = nullptr; const int32_t *p_seq_len = nullptr;
  const uint32_t *p_sa_rec = nullptr, *p_cig_off = nullptr, *p_cig_ops = nullptr, *p_sa_off = nullptr, *p_oc_off = nullptr;
  const uint8_t *p_sa_txt = nullptr, *p_oc_txt = nullptr;
  // nib
  std::vector<DBuf> nib;
  std::vector<uint64_t> nib_len;
  DBuf d_nib_ptr, d_nib_len;
  // state
  bool classified = false, have_stats = false, scanned = false, clustered = false, refined = false;
  double mean = 0, sd = 0;
  long long sum_abs = 0, cnt_insert = 0;
  unsigned long long sum_sq = 0, xmax = 0;  // K1: sum of isize^2 and max |isize| over the insert records
  long long n_cand_k1 = 0;                  // candidates counted by K1 (the sparse table must list every one of them)
  int sd_kub = 0;                           // upper bound of the binade of the sd accumulator (sd_fast)
  cudaStream_t sd_fast_st = nullptr;        // stream of the sd_fast pass in flight (sd_fast_launch .. stats_collect), null when none
  DBuf tile_cand, counters, cand_idx, cand, bucket_rank_of;
  long long n_cand = 0;
  // pairs (stage 0)
  DBuf pairs0, pairs_tmp, bucket_off0;
  long long np0 = 0; int nb = 0;
  DBuf X, Y, bucket_of_pair;
  // stage 1 (after isolated-pair removal): pair ids in order + bucket offsets
  DBuf cur1, curb1, seg1;
  long long n1 = 0;
  // stage 2 (after clustering): members grouped by (bucket, cluster)
  DBuf mem_pair, mem_bucket, mem_cluster;
  long long n2 = 0;
  std::vector<int32_t> roots_per_bucket;
  // clusters
  DBuf sdtab, sdlut; bool sd_prepared = false; double sd_mean = 0;
  DBuf clusters, clusters_out, sarows, work, cov, depth, evoff, valid, name_key, name_row;
  const void *rows_ptr = nullptr; long long n_rows = 0, n_evcap = 0; int maxspan = 1; bool clusters_ranked = false;
  long long n_clusters = 0, n_called = 0;
  Scratch sc;
  DBuf tmpA, tmpB, tmpC, tmpD, tmpE, tmpF, tmpG, tmpH;
  DBuf dist_send, dist_recv, dist_rows;     // multi-GPU exchanges (bkid_dist.cuh)
  DBuf sortheap;                            // depth-exhausted segments of the std::sort replay
  DBuf sortbig;                             // big-segment lists / tile status of the std::sort replay (exact_sort_segments)
  DBuf dist_scalars;                        // all-reduce operands of one bkid_dist_run: never shared with a stage's scratch (those are re-sized under it)
  bkid_timings tm;
  cudaEvent_t ev[16];
  cudaEvent_t ev_run[2];
  cudaEvent_t ev_side[2];
  cudaEvent_t ev_w[4];                   // push_batch: narrow column copied (st) -> widened (st3) -> joined (st)
  bool k8_attr_set = false;
  bool maxspan_cached = false, maxspan_pending = false;   // pending: max_span_kernel in flight on st3
  long long launches0 = 0;
};

// optional sub-stage timing (env BKID_DEBUG_TIMING=1): CUDA events on the context stream, printed to stderr
struct SubTimer {
  cudaStream_t st; bool on; std::vector<std::pair<std::string, cudaEvent_t>> ev;
  explicit SubTimer(cudaStream_t s) : st(s), on(getenv("BKID_DEBUG_TIMING") != nullptr) { mark("start"); }
  void mark(const char *name) { if (!on) return; cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); ev.push_back({name, e}); }
  ~SubTimer() {
    if (!on) return;
    cudaStreamSynchronize(st);
    for (size_t i = 1; i < ev.size(); ++i) { float ms = 0; cudaEventElapsedTime(&ms, ev[i - 1].second, ev[i].second); fprintf(stderr, "[bkid-timing] %-28s %8.3f ms\n", ev[i].first.c_str(), ms); }
    for (auto &e : ev) cudaEventDestroy(e.second);
  }
};

static int fail(bkid_ctx *c, int code, const std::string &msg)
{
  if (c) c->err = msg;
  else g_create_err = msg;
  return code;
}
#define CU(c, x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) { bk_set_cuda_error(e__, __FILE__, __LINE__); return fail((c), e__ == cudaErrorMemoryAllocation ? BKID_ERR_NOMEM : BKID_ERR_CUDA, g_last_cuda_err); } } while (0)
#define TRY(c, x) do { int rc__ = (x); if (rc__ != 0) { if ((c)->err.empty()) (c)->err = g_last_cuda_err; return rc__; } } while (0)

static int sync_check(bkid_ctx *c)
{
  CU(c, cudaStreamSynchronize(c->st));
  CU(c, cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// std::sort replay over segments (buckets).  key/val are permuted in place.
// ---------------------------------------------------------------------------------------------
static int exact_sort_segments(bkid_ctx *c, uint32_t *key, uint32_t *val, const uint32_t *seg_off, int nseg, long long n)
{
  if (n < 2 || nseg <= 0) return 0;
  cudaStream_t st = c->st;
  size_t seg_bytes = ((size_t)n / 2 + 16) * sizeof(Seg);
  TRY(c, c->tmpA.ensure(seg_bytes, 0, st));
  TRY(c, c->tmpB.ensure(seg_bytes, 0, st));
  TRY(c, c->tmpC.ensure(seg_bytes, 0, st));
  TRY(c, c->tmpD.ensure((size_t)n * 4 + 16, 0, st));
  TRY(c, c->tmpE.ensure((size_t)n * 4 + 16, 0, st));
  TRY(c, c->counters.ensure(256, 0, st));
  unsigned *cnt = c->counters.as<unsigned>() + CS_SORT;     // [0]=act A, [1]=act B, [2]=terminal, [3]=small
  CU(c, cudaMemsetAsync(cnt, 0, 16, st));
  Seg *act[2] = {c->tmpA.as<Seg>(), c->tmpB.as<Seg>()};
  Seg *term = c->tmpC.as<Seg>();
  TRY(c, c->tmpH.ensure(seg_bytes, 0, st));
  Seg *small = c->tmpH.as<Seg>();
  // depth-exhausted segments above the small size (each > 1024 elements, disjoint): finished by is_heap after the last level
  TRY(c, c->sortheap.ensure(((size_t)n / IS_SMALL + 16) * sizeof(Seg), 0, st));
  Seg *heapl = c->sortheap.as<Seg>();
  unsigned *n_heap = c->counters.as<unsigned>() + CS_SORT_HEAP;
  CU(c, cudaMemsetAsync(n_heap, 0, 4, st));
  // big segments (> IS_BIG elements, several CTAs each): two lists, their packed sizes (count << 32 | tiles), two tickets, tile status words
  const bool big_possible = n > (long long)IS_BIG;
  const size_t maxbig = (size_t)(n / IS_BIG) + 2, maxtiles = (size_t)(n / IS_BTILE) + maxbig + 2;
  BigSeg *big[2] = {nullptr, nullptr};
  unsigned long long *bigcnt = nullptr, *status = nullptr;
  unsigned *tickets = nullptr;
  if (big_possible) {
    TRY(c, c->sortbig.ensure(64 + 2 * maxbig * sizeof(BigSeg) + maxtiles * 8, 0, st));
    char *base = (char *)c->sortbig.p;
    bigcnt = (unsigned long long *)base; tickets = (unsigned *)(base + 16);
    big[0] = (BigSeg *)(base + 64); big[1] = big[0] + maxbig;
    status = (unsigned long long *)(big[1] + maxbig);
    CU(c, cudaMemsetAsync(base, 0, 64, st));
    CU(c, cudaMemsetAsync(status, 0, maxtiles * 8, st));
  }
  BK_LAUNCH(is_init_roots, GRID1(nseg, 256), 256, 0, st, seg_off, nseg, act[0], cnt + 0, small, cnt + 3, term, cnt + 2, big[0], bigcnt);
  int lg = 0;
  for (long long t = n; t > 1; t >>= 1) ++lg;
  int max_levels = 2 * lg + 2;
  int cur = 0;
  bool any_big = big_possible;                              // until a poll shows the big lists have drained (children are never larger than their parent)
  for (int level = 0; level < max_levels; ++level) {
    if (level > 0 && (level % 4) == 0) {                          // early exit once no segment is above the small-segment size (polled every 4th level: a poll is a host round trip)
      unsigned h = 0;
      unsigned long long hb = 0;
      CU(c, cudaMemcpyAsync(&h, cnt + cur, 4, cudaMemcpyDeviceToHost, st));
      if (any_big) CU(c, cudaMemcpyAsync(&hb, bigcnt + cur, 8, cudaMemcpyDeviceToHost, st));
      CU(c, cudaStreamSynchronize(st));
      if (hb == 0) any_big = false;
      if (h == 0 && !any_big) break;
    }
    CU(c, cudaMemsetAsync(cnt + (cur ^ 1), 0, 4, st));
    if (any_big) {                                             // the two kernels reset each other's counters: no memsets between levels
      BK_LAUNCH(is_big_part, 592, IS_THREADS, 0, st, key, val, big[cur], bigcnt + cur, tickets, status, c->tmpD.as<uint32_t>(), c->tmpE.as<uint32_t>(),
                bigcnt + (cur ^ 1), tickets + 1, heapl, n_heap);
      BK_LAUNCH(is_big_swap, 592, IS_THREADS, 0, st, key, val, big[cur], bigcnt + cur, tickets + 1, c->tmpD.as<uint32_t>(), c->tmpE.as<uint32_t>(),
                act[cur ^ 1], cnt + (cur ^ 1), small, cnt + 3, term, cnt + 2, big[cur ^ 1], bigcnt + (cur ^ 1), tickets, status);
    }
    BK_LAUNCH(is_level, 592, IS_THREADS, 0, st, key, val, act[cur], cnt + cur, act[cur ^ 1], cnt + (cur ^ 1), small, cnt + 3, term, cnt + 2,
              c->tmpD.as<uint32_t>(), c->tmpE.as<uint32_t>(), heapl, n_heap);
    cur ^= 1;
  }
  BK_LAUNCH(is_heap, 148, 256, IS_HEAP_SMEM_ELEMS * 8 + 16, st, key, val, heapl, n_heap);
  BK_LAUNCH(is_small, 2368, ISS_WARPS * 32, 0, st, key, val, small, cnt + 3);
  BK_LAUNCH(is_terminal, 592, 128, 0, st, key, val, term, cnt + 2);
  return 0;
}

// sort the current order of every bucket by coord[cur[p]] with std::sort semantics
static int sort_current_by(bkid_ctx *c, uint32_t *cur, long long n, const uint32_t *coord, const uint32_t *seg_off, int nseg)
{
  if (n < 2) return 0;
  TRY(c, c->tmpF.ensure((size_t)n * 4 + 16, 0, c->st));
  uint32_t *key = c->tmpF.as<uint32_t>();
  BK_LAUNCH(gather_u32, GRID1(n, 256), 256, 0, c->st, coord, cur, n, key);
  return exact_sort_segments(c, key, cur, seg_off, nseg, n);
}

// one isolated-pair mask pass: (cur, curb, seg) -> (cur_out, curb_out, seg_out); returns new count
static int mask_pass(bkid_ctx *c, const uint32_t *cur, const uint32_t *curb, const uint32_t *seg, long long n, int nseg, const uint32_t *X, const uint32_t *Y,
                     long long distance, uint32_t *cur_out, uint32_t *curb_out, uint32_t *seg_out, long long *n_out)
{
  cudaStream_t st = c->st;
  if (n == 0) { CU(c, cudaMemsetAsync(seg_out, 0, (size_t)(nseg + 1) * 4, st)); *n_out = 0; return 0; }
  TRY(c, c->sc.ensure(n, st));
  uint32_t *cnt = c->sc.a32.as<uint32_t>(), *off = c->sc.b32.as<uint32_t>();
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  BK_LAUNCH(k4_mask_count, GRID1(n, 256), 256, 0, st, cur, curb, seg, n, X, Y, distance, cnt);
  bk::exclusive_scan<uint32_t, uint32_t>(cnt, off, n, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
  unsigned long long h = 0;
  CU(c, cudaMemcpyAsync(&h, tot, 8, cudaMemcpyDeviceToHost, st));
  CU(c, cudaStreamSynchronize(st));
  BK_LAUNCH(k4_mask_write, GRID1(n, 256), 256, 0, st, cur, curb, n, cnt, off, cur_out, curb_out);
  BK_LAUNCH(k4_new_offsets, GRID1(nseg + 1, 256), 256, 0, st, seg, nseg, off, n, h, seg_out);
  *n_out = (long long)h;
  return 0;
}

// generic keep-compaction of (cur, curb) with new segment offsets
static int compact_pass(bkid_ctx *c, const uint32_t *cur, const uint32_t *curb, const uint32_t *seg, long long n, int nseg, const uint32_t *keep,
                        uint32_t *cur_out, uint32_t *curb_out, uint32_t *seg_out, uint32_t *off_keep /* n scratch */, long long *n_out)
{
  cudaStream_t st = c->st;
  if (n == 0) { CU(c, cudaMemsetAsync(seg_out, 0, (size_t)(nseg + 1) * 4, st)); *n_out = 0; return 0; }
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  bk::exclusive_scan<uint32_t, uint32_t>(keep, off_keep, n, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
  unsigned long long h = 0;
  CU(c, cudaMemcpyAsync(&h, tot, 8, cudaMemcpyDeviceToHost, st));
  CU(c, cudaStreamSynchronize(st));
  BK_LAUNCH(compact_write, GRID1(n, 256), 256, 0, st, cur, curb, keep, off_keep, n, cur_out, curb_out);
  BK_LAUNCH(k4_new_offsets, GRID1(nseg + 1, 256), 256, 0, st, seg, nseg, off_keep, n, h, seg_out);
  *n_out = (long long)h;
  return 0;
}

// remove_isolated_pairs (src/BreakID.cc:1271-1285) for all buckets; result in c->cur1/curb1/seg1/n1
static int remove_isolated_all(bkid_ctx *c, const uint32_t *cur0, const uint32_t *curb0, const uint32_t *seg0, long long n0, int nseg,
                               const uint32_t *X, const uint32_t *Y, double w)
{
  cudaStream_t st = c->st;
  long long distance = (long long)w;                     // double -> long at the call (src/BreakID.cc:1275)
  size_t m = (size_t)std::max<long long>(n0, 1) * 4 + 64, sb = (size_t)(nseg + 2) * 4;
  TRY(c, c->cur1.ensure(m, 0, st)); TRY(c, c->curb1.ensure(m, 0, st)); TRY(c, c->seg1.ensure(sb, 0, st));
  DBuf &ca = c->sc.c32, &cb = c->sc.d32;
  TRY(c, c->sc.ensure(n0 + 8, st));
  TRY(c, c->tmpG.ensure(3 * sb + m * 2, 0, st));
  uint32_t *segA = c->tmpG.as<uint32_t>(), *segB = segA + (nseg + 2);
  uint32_t *curA = ca.as<uint32_t>(), *curbA = cb.as<uint32_t>();
  uint32_t *work_cur = c->tmpG.as<uint32_t>() + 3 * (nseg + 2);
  uint32_t *work_curb = work_cur + std::max<long long>(n0, 1) + 8;
  if (n0 > 0) {
    CU(c, cudaMemcpyAsync(work_cur, cur0, (size_t)n0 * 4, cudaMemcpyDeviceToDevice, st));
    CU(c, cudaMemcpyAsync(work_curb, curb0, (size_t)n0 * 4, cudaMemcpyDeviceToDevice, st));
  }
  TRY(c, sort_current_by(c, work_cur, n0, X, seg0, nseg));                                  // :1274
  long long na = 0, nb2 = 0;
  TRY(c, mask_pass(c, work_cur, work_curb, seg0, n0, nseg, X, Y, distance, curA, curbA, segA, &na));   // :1275
  TRY(c, sort_current_by(c, curA, na, Y, segA, nseg));                                       // :1278
  TRY(c, mask_pass(c, curA, curbA, segA, na, nseg, X, Y, distance, c->cur1.as<uint32_t>(), c->curb1.as<uint32_t>(), segB, &nb2));   // :1279
  TRY(c, sort_current_by(c, c->cur1.as<uint32_t>(), nb2, X, segB, nseg));                    // :1282
  CU(c, cudaMemcpyAsync(c->seg1.p, segB, (size_t)(nseg + 1) * 4, cudaMemcpyDeviceToDevice, st));
  c->n1 = nb2;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// clustering of the stage-1 order; fills mem_pair / mem_bucket / mem_cluster grouped by (bucket, cluster)
// ---------------------------------------------------------------------------------------------
static int cluster_ahc(bkid_ctx *c, const uint32_t *cur, const uint32_t *curb, const uint32_t *seg, long long n, int nseg, const uint32_t *X, const uint32_t *Y, double thr_d)
{
  cudaStream_t st = c->st;
  c->n2 = 0;
  c->roots_per_bucket.assign(nseg, 0);
  if (n == 0) return 0;
  long long thr = (long long)thr_d;                      // long distance_threshold (src/util_cluster.cc:7)
  SubTimer T_(st);
  TRY(c, c->sc.ensure(n + 8, st));
  // coordinates in leaf order
  DBuf &LX = c->tmpA, &LY = c->tmpB;
  TRY(c, LX.ensure((size_t)n * 4 + 16, 0, st)); TRY(c, LY.ensure((size_t)n * 4 + 16, 0, st));
  BK_LAUNCH(gather_u32, GRID1(n, 256), 256, 0, st, X, cur, n, LX.as<uint32_t>());
  BK_LAUNCH(gather_u32, GRID1(n, 256), 256, 0, st, Y, cur, n, LY.as<uint32_t>());
  uint64_t *key = c->sc.keys.as<uint64_t>();
  uint32_t *val = c->sc.vals.as<uint32_t>();
  uint32_t *head = c->sc.a32.as<uint32_t>(), *hex = c->sc.b32.as<uint32_t>();
  unsigned long long *stmp = c->sc.scan_tmp.as<unsigned long long>();
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  int bbits = 1; while ((1ll << bbits) < nseg + 1) ++bbits;
  // pieces: sort by (bucket, x), cut at x gaps
  BK_LAUNCH(ahc_key_bx, GRID1(n, 256), 256, 0, st, curb, LX.as<uint32_t>(), n, key, val);
  bk::radix_sort_pairs(key, val, n, 0, 32 + bbits, c->sc.rt(), st);
  BK_LAUNCH(ahc_gap_heads, GRID1(n, 256), 256, 0, st, key, n, thr, head);
  bk::exclusive_scan<uint32_t, uint32_t>(head, hex, n, stmp, tot, st);
  unsigned long long npiece = 0;
  CU(c, cudaMemcpyAsync(&npiece, tot, 8, cudaMemcpyDeviceToHost, st)); CU(c, cudaStreamSynchronize(st));
  int pbits = 1; while ((1ull << pbits) < npiece + 1) ++pbits;
  // components: sort by (piece, y), cut at y gaps
  BK_LAUNCH(ahc_key_group, GRID1(n, 256), 256, 0, st, head, hex, val, LY.as<uint32_t>(), n, key);
  bk::radix_sort_pairs(key, val, n, 0, 32 + pbits, c->sc.rt(), st);
  BK_LAUNCH(ahc_gap_heads, GRID1(n, 256), 256, 0, st, key, n, thr, head);
  bk::exclusive_scan<uint32_t, uint32_t>(head, hex, n, stmp, tot, st);
  unsigned long long ncomp64 = 0;
  CU(c, cudaMemcpyAsync(&ncomp64, tot, 8, cudaMemcpyDeviceToHost, st)); CU(c, cudaStreamSynchronize(st));
  uint32_t ncomp = (uint32_t)ncomp64;
  int cbits = 1; while ((1ull << cbits) < ncomp64 + 1) ++cbits;
  // leaves of a component in ascending leaf index: sort by (comp, p)
  BK_LAUNCH(ahc_key_group, GRID1(n, 256), 256, 0, st, head, hex, val, (const uint32_t *)nullptr, n, key);
  bk::radix_sort_pairs(key, val, n, 0, 32 + cbits, c->sc.rt(), st);
  BK_LAUNCH(ahc_comp_heads, GRID1(n, 256), 256, 0, st, key, n, head);
  T_.mark("ahc: component sorts");
  // component tables
  DBuf &T = c->tmpC;
  size_t nc1 = (size_t)ncomp + 2;
  size_t bytes = nc1 * (4 + 4 + 4 + 8 + 8 + 8 + 8 + 4 + 8 + 8 + 4 + 8 + 4 + 4) + (size_t)n * (4 + 4 + 4) + (size_t)(nseg + 2) * (4 + 4 + 4 + 4) + 4096;
  TRY(c, T.ensure(bytes, 0, st));
  CU(c, cudaMemsetAsync(T.p, 0, bytes, st));
  char *bp = (char *)T.p;
  auto take = [&](size_t b) { char *r = bp; bp += (b + 15) & ~(size_t)15; return r; };
  uint32_t *comp_off = (uint32_t *)take(nc1 * 4), *comp_bucket = (uint32_t *)take(nc1 * 4);
  int32_t *hi_oc = (int32_t *)take(nc1 * 4);
  unsigned long long *pts_sz = (unsigned long long *)take(nc1 * 8), *row_sz = (unsigned long long *)take(nc1 * 8);
  unsigned long long *pts_off = (unsigned long long *)take(nc1 * 8), *row_off = (unsigned long long *)take(nc1 * 8);
  uint32_t *comp_nnodes = (uint32_t *)take(nc1 * 4);
  unsigned long long *comp_pts_used = (unsigned long long *)take(nc1 * 8), *comp_row_used = (unsigned long long *)take(nc1 * 8);
  int32_t *comp_head_j = (int32_t *)take(nc1 * 4);
  double *comp_head_d = (double *)take(nc1 * 8);
  int32_t *comp_flag = (int32_t *)take(nc1 * 4);
  uint32_t *comp_cursor = (uint32_t *)take(nc1 * 4);
  uint32_t *comp_of_point = (uint32_t *)take((size_t)n * 4);
  uint32_t *comp_leaf = (uint32_t *)take((size_t)n * 4);
  int32_t *lo_oc = (int32_t *)take((size_t)n * 4);
  uint32_t *bucket_comp_off = (uint32_t *)take((size_t)(nseg + 2) * 4);
  int32_t *bucket_flag = (int32_t *)take((size_t)(nseg + 2) * 4);
  unsigned *merges_pb = (unsigned *)take((size_t)(nseg + 2) * 4);
  uint32_t *bucket_first_root = (uint32_t *)take((size_t)(nseg + 2) * 4);
  BK_LAUNCH(ahc_comp_fill, GRID1(n, 256), 256, 0, st, key, head, val, n, curb, comp_off, comp_bucket, comp_of_point);
  CU(c, cudaMemcpyAsync(comp_leaf, val, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
  { uint32_t nn = (uint32_t)n; CU(c, cudaMemcpyAsync(comp_off + ncomp, &nn, 4, cudaMemcpyHostToDevice, st)); CU(c, cudaStreamSynchronize(st)); }
  BK_LAUNCH(ahc_comp_static, GRID1(ncomp, 128), 128, 0, st, comp_off, comp_leaf, comp_bucket, comp_of_point, seg, ncomp, lo_oc, hi_oc, pts_sz, row_sz);
  unsigned long long *tot2 = tot + 1;
  bk::exclusive_scan<unsigned long long, unsigned long long>(pts_sz, pts_off, ncomp, stmp, tot, st);
  bk::exclusive_scan<unsigned long long, unsigned long long>(row_sz, row_off, ncomp, stmp, tot2, st);
  unsigned long long pool[2] = {0, 0};
  std::vector<uint32_t> seg_h((size_t)nseg + 1);
  CU(c, cudaMemcpyAsync(seg_h.data(), seg, (size_t)(nseg + 1) * 4, cudaMemcpyDeviceToHost, st));
  CU(c, cudaMemcpyAsync(pool, tot, 16, cudaMemcpyDeviceToHost, st)); CU(c, cudaStreamSynchronize(st));
  bool have_large = false;                               // any bucket beyond the shared-memory replay classes?
  // unflagged buckets from RG_LO points up take the sort-based rank form in global memory.  On the 30x single-GPU workload
  // this is time-neutral against the O(M^2) counting kernel in shared memory; with deeper coverage (100x, or N ranks' slices
  // of one genome meeting on a bucket owner) the counting kernel grows quadratically and was the longest kernel of the step.
  const uint32_t RG_LO = 512u;
  for (int b = 0; b < nseg; ++b) have_large |= seg_h[b + 1] - seg_h[b] >= RG_LO;
  if ((pool[0] * 4 + pool[1] * 12) > (100ull << 30)) return fail(c, BKID_ERR_NOMEM, "AHC component too large for the row pools");
  BK_LAUNCH(ahc_bucket_comp_off, GRID1(nseg + 1, 128), 128, 0, st, comp_bucket, ncomp, (uint32_t)nseg, bucket_comp_off);
  // node arrays + pools + events
  DBuf &NB = c->tmpD;
  size_t nn2 = (size_t)2 * n + 2;
  size_t nbytes = nn2 * (1 + 4 + 8 + 8 + 4 + 4 + 8 + 4 + 4 + 4) + (size_t)n * (8 + 4) + pool[0] * 4 + pool[1] * 12 + 8192;
  TRY(c, NB.ensure(nbytes, 0, st));
  bp = (char *)NB.p;
  AhcView v;
  memset(&v, 0, sizeof v);
  v.seg_off = seg; v.X = LX.as<uint32_t>(); v.Y = LY.as<uint32_t>();
  v.comp_off = comp_off; v.comp_leaf = comp_leaf; v.comp_bucket = comp_bucket; v.lo_oc = lo_oc; v.hi_oc = hi_oc;
  v.pts_off = pts_off; v.row_off = row_off;
  v.node_best_d = (double *)take(nn2 * 8);
  v.node_pts = (unsigned long long *)take(nn2 * 8); v.node_row = (unsigned long long *)take(nn2 * 8);
  v.row_d = (double *)take(pool[1] * 8 + 8);
  v.ev_d = (double *)take((size_t)n * 8 + 8);
  v.node_npts = (uint32_t *)take(nn2 * 4); v.node_rowlen = (uint32_t *)take(nn2 * 4);
  v.node_best_t = (int32_t *)take(nn2 * 4); v.node_grank = (int32_t *)take(nn2 * 4);
  v.node_ma = (int32_t *)take(nn2 * 4); v.node_mb = (int32_t *)take(nn2 * 4);
  v.pts_pool = (uint32_t *)take(pool[0] * 4 + 8); v.row_t = (int32_t *)take(pool[1] * 4 + 8);
  v.ev_first = (int32_t *)take((size_t)n * 4 + 8);
  v.node_root = (uint8_t *)take(nn2);
  v.comp_nnodes = comp_nnodes; v.comp_pts_used = comp_pts_used; v.comp_row_used = comp_row_used;
  v.comp_head_j = comp_head_j; v.comp_head_d = comp_head_d; v.comp_flag = comp_flag; v.comp_cursor = comp_cursor;
  v.thr = (double)thr;
  T_.mark("ahc: tables+alloc");
  BK_LAUNCH(ahc_components, GRID1(ncomp, 4), 128, 0, st, v, ncomp);
  T_.mark("ahc: components kernel");
  BK_LAUNCH(ahc_bucket_flags, GRID1(ncomp, 128), 128, 0, st, comp_flag, comp_bucket, ncomp, bucket_flag);
  // replay: shared-memory form for buckets up to 4096 points (two smem classes), global form above that
  T_.mark("ahc: bucket flags");
  if (T_.on) {
    std::vector<int32_t> hf(ncomp); std::vector<uint32_t> hoff(ncomp + 1), hnn(ncomp);
    cudaMemcpyAsync(hf.data(), comp_flag, (size_t)ncomp * 4, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(hoff.data(), comp_off, (size_t)(ncomp + 1) * 4, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(hnn.data(), comp_nnodes, (size_t)ncomp * 4, cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    long nf = 0, maxc = 0, merges = 0, fl_pts = 0;
    for (uint32_t i = 0; i < ncomp; ++i) { uint32_t cs = hoff[i + 1] - hoff[i]; nf += hf[i] != 0; if (hf[i]) fl_pts += cs; maxc = std::max<long>(maxc, cs); merges += hnn[i] - cs; }
    fprintf(stderr, "[bkid-timing] ncomp %u flagged %ld (points %ld) max comp %ld merges %ld points %lld buckets %d\n", ncomp, nf, fl_pts, maxc, merges, n, nseg);
  }
  BK_LAUNCH(ahc_replay_rank, (unsigned)nseg, RK_THREADS, 49 * 512, st, v, bucket_comp_off, (uint32_t)nseg, bucket_flag, 0u, RG_LO);
  T_.mark("ahc: replay rank form");
  BK_LAUNCH(ahc_replay_smem, (unsigned)nseg, 32, 49 * 900, st, v, bucket_comp_off, (uint32_t)nseg, bucket_flag, 0u, 900u);
  BK_LAUNCH(ahc_replay_smem, (unsigned)nseg, 32, 49 * 4096, st, v, bucket_comp_off, (uint32_t)nseg, bucket_flag, 900u, 4096u);
  T_.mark("ahc: replay smem (flagged)");
  if (have_large) {
    // buckets >= RG_LO points without flagged components: rank form in global memory
    DBuf &RG = c->tmpF;
    size_t nn = (size_t)n + 8;
    TRY(c, RG.ensure(nn * (8 + 4 + 4 + 4 + 4 + 4 + 4 + 1) + (size_t)(nseg + 2) * 4 + 256, 0, st));
    char *q = (char *)RG.p;
    RankGlobal g;
    g.pm = (double *)q; q += nn * 8;
    g.slot_comp = (uint32_t *)q; q += nn * 4;
    g.first = (int32_t *)q; q += nn * 4;
    g.rank = (uint32_t *)q; q += nn * 4;
    g.order = (uint32_t *)q; q += nn * 4;
    g.is_head = (uint32_t *)q; q += nn * 4;
    uint32_t *head_excl = (uint32_t *)q; q += nn * 4;
    uint32_t *bucket_events = (uint32_t *)q; q += (size_t)(nseg + 2) * 4;
    g.tie = (uint8_t *)q;
    uint32_t *head_pos = c->sc.e32.as<uint32_t>();
    CU(c, cudaMemsetAsync(bucket_events, 0, (size_t)(nseg + 2) * 4, st));
    CU(c, cudaMemsetAsync(g.is_head, 0, nn * 4, st));
    BK_LAUNCH(ahc_rg_bucket_events, GRID1(ncomp, 128), 128, 0, st, v, ncomp, bucket_events);
    BK_LAUNCH(ahc_rg_prepare, GRID1(ncomp, 128), 128, 0, st, v, g, ncomp, bucket_flag, RG_LO);
    {
      uint64_t *rk = c->sc.keys.as<uint64_t>();
      uint32_t *rv = c->sc.vals.as<uint32_t>();
      BK_LAUNCH(ahc_rg_sortkeys, GRID1(n, 256), 256, 0, st, v, g, curb, n, bucket_flag, RG_LO, rk, rv);
      bk::radix_sort_pairs(rk, rv, n, 0, 64, c->sc.rt(), st);
      BK_LAUNCH(ahc_rg_bucketkeys, GRID1(n, 256), 256, 0, st, curb, rv, n, rk);
      bk::radix_sort_pairs(rk, rv, n, 0, bbits, c->sc.rt(), st);
      BK_LAUNCH(ahc_rg_rank_sorted, GRID1(n, 256), 256, 0, st, v, g, curb, n, bucket_flag, RG_LO, rv);
    }
    BK_LAUNCH(ahc_rg_heads, GRID1(n, 256), 256, 0, st, v, g, curb, n, bucket_flag, RG_LO, bucket_events);
    bk::exclusive_scan<uint32_t, uint32_t>(g.is_head, head_excl, n, stmp, tot, st);
    BK_LAUNCH(ahc_rg_head_list, GRID1(n, 256), 256, 0, st, g.is_head, head_excl, n, head_pos);
    unsigned *rg_ticket = c->counters.as<unsigned>() + CS_RG_TICKET;
    CU(c, cudaMemsetAsync(rg_ticket, 0, 4, st));
    BK_LAUNCH(ahc_rg_ties, 148 * 4, 128, 0, st, v, g, curb, bucket_flag, RG_LO, bucket_events, head_pos, tot, rg_ticket);      // one warp per tie group, ticket order
    BK_LAUNCH(ahc_rg_write, GRID1(n, 256), 256, 0, st, v, g, curb, n, bucket_flag, RG_LO);
  }
  T_.mark("ahc: replay rank form (global)");
  BK_LAUNCH(ahc_bucket_exact, (unsigned)nseg, 32, 0, st, v, bucket_comp_off, (uint32_t)nseg, bucket_flag, 4096u);
  T_.mark("ahc: replay+exact");
  // final roots -> clusters
  unsigned *cnt = c->counters.as<unsigned>() + CS_ROOTS;
  CU(c, cudaMemsetAsync(cnt, 0, 4, st));
  uint64_t *rkey = c->sc.keys.as<uint64_t>();
  uint32_t *rnode = c->sc.vals.as<uint32_t>();
  BK_LAUNCH(ahc_final_roots, GRID1(ncomp, 128), 128, 0, st, v, ncomp, rkey, rnode, cnt, merges_pb);
  unsigned nroot = 0;
  CU(c, cudaMemcpyAsync(&nroot, cnt, 4, cudaMemcpyDeviceToHost, st)); CU(c, cudaStreamSynchronize(st));
  std::vector<unsigned> merges(nseg);
  std::vector<uint32_t> segh(nseg + 1);
  CU(c, cudaMemcpyAsync(merges.data(), merges_pb, (size_t)nseg * 4, cudaMemcpyDeviceToHost, st));
  CU(c, cudaMemcpyAsync(segh.data(), seg, (size_t)(nseg + 1) * 4, cudaMemcpyDeviceToHost, st));
  CU(c, cudaStreamSynchronize(st));
  for (int b = 0; b < nseg; ++b) c->roots_per_bucket[b] = (int32_t)(segh[b + 1] - segh[b]) - (int32_t)merges[b];   // print_root_nodes
  if (nroot == 0) return sync_check(c);
  bk::radix_sort_pairs(rkey, rnode, nroot, 0, 32 + bbits, c->sc.rt(), st);
  uint32_t *rsize = c->sc.a32.as<uint32_t>(), *roff = c->sc.b32.as<uint32_t>(), *rhead = c->sc.e32.as<uint32_t>();
  BK_LAUNCH(ahc_root_sizes, GRID1(nroot, 128), 128, 0, st, v, rkey, rnode, nroot, rsize, rhead);
  BK_LAUNCH(ahc_root_firsts, GRID1(nroot, 128), 128, 0, st, rhead, nroot, rkey, bucket_first_root);
  bk::exclusive_scan<uint32_t, uint32_t>(rsize, roff, nroot, stmp, tot, st);
  unsigned long long nm = 0;
  CU(c, cudaMemcpyAsync(&nm, tot, 8, cudaMemcpyDeviceToHost, st)); CU(c, cudaStreamSynchronize(st));
  size_t mb = (size_t)std::max<unsigned long long>(nm, 1) * 4 + 16;
  TRY(c, c->mem_pair.ensure(mb, 0, st)); TRY(c, c->mem_bucket.ensure(mb, 0, st)); TRY(c, c->mem_cluster.ensure(mb, 0, st));
  TRY(c, c->tmpE.ensure(mb, 0, st));
  BK_LAUNCH(ahc_emit, GRID1(nroot, 4), 128, 0, st, v, rkey, rnode, roff, bucket_first_root, nroot, c->tmpE.as<uint32_t>(), c->mem_cluster.as<int32_t>(), c->mem_bucket.as<uint32_t>());
  // members are positions in the stage-1 order; translate to pair ids
  BK_LAUNCH(gather_u32, GRID1(nm, 256), 256, 0, st, cur, c->tmpE.as<uint32_t>(), (long long)nm, c->mem_pair.as<uint32_t>());
  c->n2 = (long long)nm;
  T_.mark("ahc: final roots+emit");
  return sync_check(c);
}

__global__ void fast_member_keys(const uint32_t *__restrict__ curb, const int32_t *__restrict__ cl, long long n, uint64_t *__restrict__ key, uint32_t *__restrict__ val)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) { key[p] = ((uint64_t)curb[p] << 32) | (uint32_t)cl[p]; val[p] = (uint32_t)p; }
}
__global__ void fast_member_write(const uint64_t *__restrict__ key, const uint32_t *__restrict__ val, const uint32_t *__restrict__ cur, long long n,
                                  uint32_t *__restrict__ mem_pair, uint32_t *__restrict__ mem_bucket, int32_t *__restrict__ mem_cluster)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) { mem_pair[p] = cur[val[p]]; mem_bucket[p] = (uint32_t)(key[p] >> 32); mem_cluster[p] = (int32_t)(key[p] & 0xffffffffu); }
}

static int cluster_fast(bkid_ctx *c, const uint32_t *cur, const uint32_t *curb, const uint32_t *seg, long long n, int nseg, const uint32_t *X, const uint32_t *Y, double w,
                        long long np0)
{
  cudaStream_t st = c->st;
  c->n2 = 0;
  c->roots_per_bucket.assign(nseg, 0);
  if (n == 0) return 0;
  int min_reads = c->prm.min_reads;
  TRY(c, c->sc.ensure(std::max(n, np0) + 8, st));
  size_t m = (size_t)n * 4 + 64, sb = (size_t)(nseg + 2) * 4;
  // tmpA..tmpF belong to the sort replay; the sweep state lives in tmpG
  TRY(c, c->tmpG.ensure(4 * m + 4 * sb + (size_t)np0 * 8 + 64, 0, st));
  uint32_t *curA = c->tmpG.as<uint32_t>(), *curbA = curA + n + 8, *curB = curbA + n + 8, *curbB = curB + n + 8;
  uint32_t *segA = curbB + n + 8, *segB = segA + nseg + 2;
  uint32_t *k1 = segB + nseg + 2, *k2 = k1 + np0;
  uint32_t *keep = c->sc.a32.as<uint32_t>(), *off = c->sc.b32.as<uint32_t>();
  long long na = 0, nb2 = 0, nc = 0;
  BK_LAUNCH(fast_sweep, GRID1(nseg, 64), 64, 0, st, cur, seg, (uint32_t)nseg, X, w, min_reads, k1, keep);                       // :1056-1087
  TRY(c, compact_pass(c, cur, curb, seg, n, nseg, keep, curA, curbA, segA, off, &na));
  TRY(c, sort_current_by(c, curA, na, Y, segA, nseg));                                                                         // :1091
  if (na > 0) BK_LAUNCH(fast_sweep, GRID1(nseg, 64), 64, 0, st, curA, segA, (uint32_t)nseg, Y, w, min_reads, k2, keep);         // :1093-1123
  TRY(c, compact_pass(c, curA, curbA, segA, na, nseg, keep, curB, curbB, segB, off, &nb2));
  TRY(c, sort_current_by(c, curB, nb2, X, segB, nseg));                                                                        // :1127
  if (nb2 == 0) return sync_check(c);
  int32_t *cl = (int32_t *)c->sc.c32.as<uint32_t>();
  int32_t *ncl = (int32_t *)c->sc.d32.as<uint32_t>();
  BK_LAUNCH(fast_number, GRID1(nseg, 64), 64, 0, st, curB, segB, (uint32_t)nseg, k1, k2, min_reads, cl, keep, ncl);             // :1129-1157
  CU(c, cudaMemcpyAsync(c->roots_per_bucket.data(), ncl, (size_t)nseg * 4, cudaMemcpyDeviceToHost, st));
  // drop ids seen fewer than min_reads times, group the rest by (bucket, cluster)
  uint32_t *curC = curA, *curbC = curbA;     // reuse
  // compact the cluster ids alongside: write cl through the same offsets
  bk::exclusive_scan<uint32_t, uint32_t>(keep, off, nb2, c->sc.scan_tmp.as<unsigned long long>(), (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL), st);
  unsigned long long h = 0;
  CU(c, cudaMemcpyAsync(&h, c->counters.as<unsigned>() + CS_TOTAL, 8, cudaMemcpyDeviceToHost, st)); CU(c, cudaStreamSynchronize(st));
  nc = (long long)h;
  if (nc == 0) return 0;
  BK_LAUNCH(compact_write, GRID1(nb2, 256), 256, 0, st, curB, curbB, keep, off, nb2, curC, curbC);
  uint32_t *clC = c->sc.e32.as<uint32_t>();
  BK_LAUNCH(compact_write, GRID1(nb2, 256), 256, 0, st, (const uint32_t *)cl, curbB, keep, off, nb2, clC, c->sc.vals_alt.as<uint32_t>() /* unused copy */);
  uint64_t *key = c->sc.keys.as<uint64_t>();
  uint32_t *val = c->sc.vals.as<uint32_t>();
  BK_LAUNCH(fast_member_keys, GRID1(nc, 256), 256, 0, st, curbC, (const int32_t *)clC, nc, key, val);
  int bbits = 1; while ((1ll << bbits) < nseg + 1) ++bbits;
  bk::radix_sort_pairs(key, val, nc, 0, 32 + bbits, c->sc.rt(), st);
  size_t mb = (size_t)nc * 4 + 16;
  TRY(c, c->mem_pair.ensure(mb, 0, st)); TRY(c, c->mem_bucket.ensure(mb, 0, st)); TRY(c, c->mem_cluster.ensure(mb, 0, st));
  BK_LAUNCH(fast_member_write, GRID1(nc, 256), 256, 0, st, key, val, curC, nc, c->mem_pair.as<uint32_t>(), c->mem_bucket.as<uint32_t>(), c->mem_cluster.as<int32_t>());
  c->n2 = nc;
  return sync_check(c);
}

// =============================================================================================
// exported C ABI
// =============================================================================================
extern "C" {

int bkid_abi_version(void) { return BKID_ABI_VERSION; }

const char *bkid_last_error(const bkid_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

void bkid_default_params(bkid_params *p)
{
  p->qual = 20; p->times = 2; p->fast = 0; p->min_reads = 2; p->bp_pos_error = 2; p->mismatch_num = 10; p->sd_mult = 3; p->validate_align = 0;
}

bkid_ctx *bkid_create(int device, const bkid_header *hdr, const bkid_params *params)
{
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) { g_create_err = std::string("no usable CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e); return nullptr; }
  if (device < 0 || device >= ndev) { g_create_err = "device index out of range"; return nullptr; }
  if (!hdr || hdr->n_targets < 0) { g_create_err = "bad header"; return nullptr; }
  if (cudaSetDevice(device) != cudaSuccess) { g_create_err = "cudaSetDevice failed"; return nullptr; }
  bkid_ctx *c = new bkid_ctx();
  c->device = device;
  cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, device);
  if (params) c->prm = *params; else bkid_default_params(&c->prm);
  if (cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking) != cudaSuccess) { g_create_err = "cudaStreamCreate failed"; delete c; return nullptr; }
  cudaStreamCreateWithFlags(&c->st2, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&c->st3, cudaStreamNonBlocking);
  for (auto &ev : c->ev) cudaEventCreate(&ev);
  for (auto &ev : c->ev_run) cudaEventCreate(&ev);
  for (auto &ev : c->ev_side) cudaEventCreate(&ev);
  for (auto &ev : c->ev_w) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  c->nt = hdr->n_targets;
  for (int i = 0; i < c->nt; ++i) { c->target_len.push_back(hdr->target_len[i]); c->names.emplace_back(hdr->target_name[i]); }
  int nt = c->nt, m = nt + 1;
  std::vector<uint32_t> cum(nt + 1, 0);
  for (int i = 0; i < nt; ++i) cum[i + 1] = cum[i] + c->target_len[i];                 // uint32 wrap, src/util_bam.cc:61-64
  // rank of every "A_B" bucket name in std::map<string> order (src/BreakID.cc:1500-1512); index 0 = "*"
  std::vector<std::pair<std::string, int>> bn;
  for (int a = 0; a < m; ++a)
    for (int b = 0; b < m; ++b) bn.push_back({(a ? c->names[a - 1] : std::string("*")) + "_" + (b ? c->names[b - 1] : std::string("*")), a * m + b});
  std::sort(bn.begin(), bn.end());
  std::vector<int32_t> rank((size_t)m * m);
  for (size_t r = 0; r < bn.size(); ++r) rank[bn[r].second] = (int32_t)r;
  std::vector<uint64_t> canon(nt ? nt : 1);
  for (int i = 0; i < nt; ++i) canon[i] = chr_code((const uint8_t *)c->names[i].data(), (uint32_t)c->names[i].size());
  bool ok = c->d_cum.ensure((size_t)(nt + 1) * 4, 0, c->st) == 0 && c->d_bucket_rank.ensure(rank.size() * 4, 0, c->st) == 0 &&
            c->d_canon.ensure(canon.size() * 8, 0, c->st) == 0 && c->counters.ensure(1024, 0, c->st) == 0 &&
            c->d_nib_ptr.ensure((size_t)(nt + 1) * 8, 0, c->st) == 0 && c->d_nib_len.ensure((size_t)(nt + 1) * 8, 0, c->st) == 0;
  if (!ok) { g_create_err = "device allocation failed: " + g_last_cuda_err; delete c; return nullptr; }
  cudaMemcpy(c->d_cum.p, cum.data(), (size_t)(nt + 1) * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(c->d_bucket_rank.p, rank.data(), rank.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(c->d_canon.p, canon.data(), canon.size() * 8, cudaMemcpyHostToDevice);
  cudaMemset(c->d_nib_ptr.p, 0, (size_t)(nt + 1) * 8);
  cudaMemset(c->d_nib_len.p, 0, (size_t)(nt + 1) * 8);
  c->nib.resize(nt); c->nib_len.assign(nt, 0);
  cudaFuncSetAttribute(sd_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, SD_BLOCK * 9);
  cudaFuncSetAttribute(is_heap, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(IS_HEAP_SMEM_ELEMS * 8 + 16));
  cudaFuncSetAttribute(ahc_replay_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, 49 * 4096);
  cudaFuncSetAttribute(ahc_replay_rank, cudaFuncAttributeMaxDynamicSharedMemorySize, 49 * 4096);
  memset(&c->tm, 0, sizeof c->tm);
  if (cudaGetLastError() != cudaSuccess) { g_create_err = "CUDA error during create"; delete c; return nullptr; }
  return c;
}

void bkid_destroy(bkid_ctx *c)
{
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->st);
  decoder_free(c);
  for (DBuf *b : {&c->d_cum, &c->d_bucket_rank, &c->d_canon, &c->flag, &c->mapq, &c->tid, &c->pos, &c->isize, &c->endpos, &c->isize16, &c->span16, &c->cand_bits, &c->x_rec, &c->x_mtid, &c->x_mpos, &c->x_nh, &c->cls,
                  &c->sa_rec, &c->cig_off, &c->cig_ops, &c->sa_off, &c->sa_txt, &c->oc_off, &c->oc_txt, &c->seq_off, &c->seq4, &c->seq_len, &c->d_nib_ptr, &c->d_nib_len, &c->tile_cand, &c->counters,
                  &c->cand_idx, &c->cand, &c->bucket_rank_of, &c->pairs0, &c->pairs_tmp, &c->bucket_off0, &c->X, &c->Y, &c->bucket_of_pair, &c->cur1, &c->curb1, &c->seg1, &c->mem_pair,
                  &c->mem_bucket, &c->mem_cluster, &c->sdtab, &c->sdlut, &c->clusters, &c->clusters_out, &c->sarows, &c->name_key, &c->name_row, &c->ex_tab, &c->ex_lo, &c->ex_len, &c->ex_pre, &c->work, &c->cov, &c->depth, &c->evoff, &c->valid, &c->tmpA, &c->tmpB, &c->tmpC, &c->tmpD, &c->tmpE, &c->tmpF, &c->tmpG, &c->tmpH, &c->dist_send, &c->dist_recv, &c->dist_rows, &c->dist_scalars, &c->sortbig, &c->sortheap})
    b->release();
  for (auto &b : c->nib) b.release();
  c->sc.release();
  for (auto &ev : c->ev) cudaEventDestroy(ev);
  for (auto &ev : c->ev_run) cudaEventDestroy(ev);
  for (auto &ev : c->ev_side) cudaEventDestroy(ev);
  for (auto &ev : c->ev_w) cudaEventDestroy(ev);
  cudaStreamDestroy(c->st2);
  cudaStreamDestroy(c->st3);
  cudaStreamDestroy(c->st);
  delete c;
}

static void invalidate(bkid_ctx *c)
{
  if (c->sd_fast_st) { cudaStreamSynchronize(c->sd_fast_st); c->sd_fast_st = nullptr; }
  if (c->maxspan_pending) { cudaStreamSynchronize(c->st3); c->maxspan_pending = false; }
  c->classified = c->have_stats = c->scanned = c->clustered = c->refined = false; c->sd_prepared = false; c->maxspan_cached = false;
}

// capacity for n records in the column forms the context currently has (an undecided form allocates nothing yet)
static int reserve_impl(bkid_ctx *c, long long n, long long n_x, long long n_sa, long long n_cig, long long sa_b, long long oc_b)
{
  cudaStream_t st = c->st;
  if (c->borrowed) return fail(c, BKID_ERR_ARG, "context holds borrowed device columns; bkid_reset first");
  size_t k = (size_t)c->n;
  TRY(c, c->flag.ensure((size_t)n * 2 + 64, k * 2, st)); TRY(c, c->mapq.ensure((size_t)n + 64, k, st));
  TRY(c, c->tid.ensure((size_t)n * 4 + 64, k * 4, st)); TRY(c, c->pos.ensure((size_t)n * 4 + 64, k * 4, st));
  if (c->form_isize == 1) TRY(c, c->isize.ensure((size_t)n * 4 + 64, k * 4, st));
  if (c->form_isize == 2) TRY(c, c->isize16.ensure((size_t)n * 2 + 64, k * 2, st));
  if (c->form_span == 1) TRY(c, c->endpos.ensure((size_t)n * 4 + 64, k * 4, st));
  if (c->form_span == 2) TRY(c, c->span16.ensure((size_t)n * 2 + 64, k * 2, st));
  size_t kx = (size_t)c->n_x;
  TRY(c, c->x_rec.ensure((size_t)n_x * 4 + 64, kx * 4, st)); TRY(c, c->x_mtid.ensure((size_t)n_x * 4 + 64, kx * 4, st));
  TRY(c, c->x_mpos.ensure((size_t)n_x * 4 + 64, kx * 4, st)); TRY(c, c->x_nh.ensure((size_t)n_x * 16 + 64, kx * 16, st));
  size_t s = (size_t)c->n_sa;
  TRY(c, c->sa_rec.ensure((size_t)n_sa * 4 + 64, s * 4, st));
  TRY(c, c->cig_off.ensure((size_t)(n_sa + 1) * 4 + 64, (s + 1) * 4, st));
  TRY(c, c->sa_off.ensure((size_t)(n_sa + 1) * 4 + 64, (s + 1) * 4, st));
  TRY(c, c->oc_off.ensure((size_t)(n_sa + 1) * 4 + 64, (s + 1) * 4, st));
  TRY(c, c->cig_ops.ensure((size_t)n_cig * 4 + 64, (size_t)c->n_cig * 4, st));
  TRY(c, c->sa_txt.ensure((size_t)sa_b + 64, (size_t)c->sa_bytes, st));
  TRY(c, c->oc_txt.ensure((size_t)oc_b + 64, (size_t)c->oc_bytes, st));
  return 0;
}

int bkid_reserve(bkid_ctx *c, int64_t n, int64_t n_x, int64_t n_sa, int64_t n_cig, int64_t sa_b, int64_t oc_b)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->reserve_hint = std::max<long long>(c->reserve_hint, n);
  return reserve_impl(c, std::max<long long>(n, c->n), std::max<long long>(n_x, c->n_x), std::max<long long>(n_sa, c->n_sa), std::max<long long>(n_cig, c->n_cig),
                      std::max<long long>(sa_b, c->sa_bytes), std::max<long long>(oc_b, c->oc_bytes));
}

__global__ void add_offset_u32(uint32_t *p, long long n, uint32_t d)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] += d;
}

// widening of the narrow host encodings (include/breakid_b200.h: isize16 / span16 / tid runs)
__global__ void widen_isize16(const int16_t *__restrict__ src, long long n, int32_t *__restrict__ dst)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (int32_t)src[i];
}
__global__ void widen_span16(const int32_t *__restrict__ pos, const uint16_t *__restrict__ span, long long n, int32_t *__restrict__ endpos)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) endpos[i] = pos[i] + (int32_t)span[i];
}
__global__ void widen_tid_runs(const uint32_t *__restrict__ start, const int32_t *__restrict__ rtid, int nruns, long long n, int32_t *__restrict__ tid)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int a = 0, b = nruns;                         // last run with start <= i
  while (b - a > 1) { int m = (a + b) >> 1; if ((long long)start[m] <= i) a = m; else b = m; }
  tid[i] = rtid[a];
}

static void set_ptrs(bkid_ctx *c)
{
  c->p_flag = c->flag.as<uint16_t>(); c->p_mapq = c->mapq.as<uint8_t>(); c->p_tid = c->tid.as<int32_t>(); c->p_pos = c->pos.as<int32_t>();
  c->p_isize = c->form_isize == 2 ? nullptr : c->isize.as<int32_t>(); c->p_isize16 = c->form_isize == 2 ? c->isize16.as<int16_t>() : nullptr;
  c->p_endpos = c->form_span == 2 ? nullptr : c->endpos.as<int32_t>(); c->p_span16 = c->form_span == 2 ? c->span16.as<uint16_t>() : nullptr;
  c->p_x_rec = c->x_rec.as<uint32_t>(); c->p_x_mtid = c->x_mtid.as<int32_t>(); c->p_x_mpos = c->x_mpos.as<int32_t>(); c->p_x_nh = c->x_nh.as<uint64_t>();
  c->p_sa_rec = c->sa_rec.as<uint32_t>(); c->p_cig_off = c->cig_off.as<uint32_t>(); c->p_cig_ops = c->cig_ops.as<uint32_t>();
  c->p_seq_off = c->seq_off.as<uint32_t>(); c->p_seq4 = c->seq4.as<uint8_t>(); c->p_seq_len = c->seq_len.as<int32_t>();
  c->p_sa_off = c->sa_off.as<uint32_t>(); c->p_sa_txt = c->sa_txt.as<uint8_t>(); c->p_oc_off = c->oc_off.as<uint32_t>(); c->p_oc_txt = c->oc_txt.as<uint8_t>();
}

// The context keeps the insert-size and span columns in ONE form each.  An empty context adopts the form of its first batch;
// a wide batch arriving at a narrow context widens the records already held (one pass), a narrow batch arriving at a wide
// context is widened on the way in.  want = 1 wide, 2 narrow.
static int settle_forms(bkid_ctx *c, int want_isize, int want_span, long long n_new)
{
  cudaStream_t st = c->st;
  long long n0 = c->n;
  size_t cap = (size_t)std::max<long long>(n0 + n_new, c->reserve_hint);
  if (c->form_isize == 0) c->form_isize = want_isize;
  else if (c->form_isize == 2 && want_isize == 1) {
    TRY(c, c->isize.ensure(cap * 4 + 64, 0, st));
    if (n0) BK_LAUNCH(widen_isize16, GRID1(n0, 256), 256, 0, st, c->isize16.as<int16_t>(), n0, c->isize.as<int32_t>());
    c->form_isize = 1;
  }
  if (c->form_span == 0) c->form_span = want_span;
  else if (c->form_span == 2 && want_span == 1) {
    TRY(c, c->endpos.ensure(cap * 4 + 64, 0, st));
    if (n0) BK_LAUNCH(widen_span16, GRID1(n0, 256), 256, 0, st, c->pos.as<int32_t>(), c->span16.as<uint16_t>(), n0, c->endpos.as<int32_t>());
    c->form_span = 1;
  }
  return 0;
}

static int push_impl(bkid_ctx *c, const bkid_batch *b, cudaMemcpyKind kind)
{
  if (!c || !b || b->n < 0 || b->n_sa < 0 || b->n_x < 0) return c ? fail(c, BKID_ERR_ARG, "bad batch") : BKID_ERR_ARG;
  if (b->n > 0 && ((!b->isize && !b->isize16) || (!b->endpos && !b->span16) || (!b->tid && (b->n_tid_runs <= 0 || !b->tid_run_start || !b->tid_run_tid))))
    return fail(c, BKID_ERR_ARG, "bad batch: a dense column is missing in both its wide and its narrow form");
  cudaSetDevice(c->device);
  cudaStream_t st = c->st;
  if ((unsigned long long)(c->n + b->n) >= 0xffffffffull) return fail(c, BKID_ERR_ARG, "more than 2^32-1 records per context");
  invalidate(c);
  cudaEventRecord(c->ev[0], st);
  long long n0 = c->n, s0 = c->n_sa, x0 = c->n_x;
  // side-table sizes need the last offsets of the incoming batch
  uint32_t ncig = 0, nsa_b = 0, noc_b = 0;
  if (b->n_sa > 0) {
    if (kind == cudaMemcpyHostToDevice) { ncig = b->cig_off[b->n_sa]; nsa_b = b->sa_off[b->n_sa]; noc_b = b->oc_off[b->n_sa]; }
    else {
      CU(c, cudaMemcpy(&ncig, b->cig_off + b->n_sa, 4, cudaMemcpyDeviceToHost));
      CU(c, cudaMemcpy(&nsa_b, b->sa_off + b->n_sa, 4, cudaMemcpyDeviceToHost));
      CU(c, cudaMemcpy(&noc_b, b->oc_off + b->n_sa, 4, cudaMemcpyDeviceToHost));
    }
  }
  if (b->n > 0) TRY(c, settle_forms(c, b->isize ? 1 : 2, b->endpos ? 1 : 2, b->n));
  TRY(c, reserve_impl(c, std::max<long long>(n0 + b->n, c->reserve_hint), x0 + b->n_x, s0 + b->n_sa, c->n_cig + ncig, c->sa_bytes + nsa_b, c->oc_bytes + noc_b));
  size_t n = (size_t)b->n;
  if (n) {
    // Narrow columns that the context keeps narrow are plain copies.  Those it holds wide (and the tid runs, always) are
    // staged in scratch and widened on a second stream, so that the widening kernels overlap the copies of the
    // remaining columns instead of standing between them on the copy stream.
    cudaStream_t sw = c->st3;
    const bool widen_i = b->isize16 && !b->isize && c->form_isize == 1, widen_s = b->span16 && !b->endpos && c->form_span == 1;
    size_t stage = (widen_i ? n * 2 : 0) + (widen_s ? n * 2 : 0) + (b->tid ? 0 : (size_t)b->n_tid_runs * 8) + 64;
    TRY(c, c->tmpH.ensure(stage, 0, st));
    char *sp = (char *)c->tmpH.p;
    bool widened = false;
    if (b->tid) CU(c, cudaMemcpyAsync(c->tid.as<int32_t>() + n0, b->tid, n * 4, kind, st));
    else {
      uint32_t *rs = (uint32_t *)sp; sp += (size_t)b->n_tid_runs * 4;
      int32_t *rt = (int32_t *)sp; sp += (size_t)b->n_tid_runs * 4;
      CU(c, cudaMemcpyAsync(rs, b->tid_run_start, (size_t)b->n_tid_runs * 4, kind, st));
      CU(c, cudaMemcpyAsync(rt, b->tid_run_tid, (size_t)b->n_tid_runs * 4, kind, st));
      CU(c, cudaEventRecord(c->ev_w[0], st)); CU(c, cudaStreamWaitEvent(sw, c->ev_w[0], 0));
      BK_LAUNCH(widen_tid_runs, GRID1(n, 256), 256, 0, sw, rs, rt, (int)b->n_tid_runs, (long long)n, c->tid.as<int32_t>() + n0);
      widened = true;
    }
    if (c->form_isize == 2) CU(c, cudaMemcpyAsync(c->isize16.as<int16_t>() + n0, b->isize16, n * 2, kind, st));
    else if (b->isize) CU(c, cudaMemcpyAsync(c->isize.as<int32_t>() + n0, b->isize, n * 4, kind, st));
    else {
      int16_t *s16 = (int16_t *)sp; sp += n * 2;
      CU(c, cudaMemcpyAsync(s16, b->isize16, n * 2, kind, st));
      CU(c, cudaEventRecord(c->ev_w[1], st)); CU(c, cudaStreamWaitEvent(sw, c->ev_w[1], 0));
      BK_LAUNCH(widen_isize16, GRID1(n, 256), 256, 0, sw, s16, (long long)n, c->isize.as<int32_t>() + n0);
      widened = true;
    }
    CU(c, cudaMemcpyAsync(c->pos.as<int32_t>() + n0, b->pos, n * 4, kind, st));
    if (c->form_span == 2) CU(c, cudaMemcpyAsync(c->span16.as<uint16_t>() + n0, b->span16, n * 2, kind, st));
    else if (b->endpos) CU(c, cudaMemcpyAsync(c->endpos.as<int32_t>() + n0, b->endpos, n * 4, kind, st));
    else {
      uint16_t *e16 = (uint16_t *)sp; sp += n * 2;
      CU(c, cudaMemcpyAsync(e16, b->span16, n * 2, kind, st));
      CU(c, cudaEventRecord(c->ev_w[2], st)); CU(c, cudaStreamWaitEvent(sw, c->ev_w[2], 0));
      BK_LAUNCH(widen_span16, GRID1(n, 256), 256, 0, sw, c->pos.as<int32_t>() + n0, e16, (long long)n, c->endpos.as<int32_t>() + n0);
      widened = true;
    }
    CU(c, cudaMemcpyAsync(c->flag.as<uint16_t>() + n0, b->flag, n * 2, kind, st));
    CU(c, cudaMemcpyAsync(c->mapq.as<uint8_t>() + n0, b->mapq, n, kind, st));
    if (widened) { CU(c, cudaEventRecord(c->ev_w[3], sw)); CU(c, cudaStreamWaitEvent(st, c->ev_w[3], 0)); }
  }
  size_t nx = (size_t)b->n_x;
  if (nx) {
    CU(c, cudaMemcpyAsync(c->x_rec.as<uint32_t>() + x0, b->x_rec, nx * 4, kind, st));
    CU(c, cudaMemcpyAsync(c->x_mtid.as<int32_t>() + x0, b->x_mtid, nx * 4, kind, st));
    CU(c, cudaMemcpyAsync(c->x_mpos.as<int32_t>() + x0, b->x_mpos, nx * 4, kind, st));
    CU(c, cudaMemcpyAsync(c->x_nh.as<uint64_t>() + 2 * x0, b->x_name_hash, nx * 16, kind, st));
    if (n0) BK_LAUNCH(add_offset_u32, GRID1(nx, 256), 256, 0, st, c->x_rec.as<uint32_t>() + x0, (long long)nx, (uint32_t)n0);
  }
  size_t ns = (size_t)b->n_sa;
  if (ns) {
    CU(c, cudaMemcpyAsync(c->sa_rec.as<uint32_t>() + s0, b->sa_rec, ns * 4, kind, st));
    CU(c, cudaMemcpyAsync(c->cig_off.as<uint32_t>() + s0, b->cig_off, (ns + 1) * 4, kind, st));
    CU(c, cudaMemcpyAsync(c->sa_off.as<uint32_t>() + s0, b->sa_off, (ns + 1) * 4, kind, st));
    CU(c, cudaMemcpyAsync(c->oc_off.as<uint32_t>() + s0, b->oc_off, (ns + 1) * 4, kind, st));
    if (ncig) CU(c, cudaMemcpyAsync(c->cig_ops.as<uint32_t>() + c->n_cig, b->cig_ops, (size_t)ncig * 4, kind, st));
    if (nsa_b) CU(c, cudaMemcpyAsync(c->sa_txt.as<uint8_t>() + c->sa_bytes, b->sa_txt, nsa_b, kind, st));
    if (noc_b) CU(c, cudaMemcpyAsync(c->oc_txt.as<uint8_t>() + c->oc_bytes, b->oc_txt, noc_b, kind, st));
    if (n0) BK_LAUNCH(add_offset_u32, GRID1(ns, 256), 256, 0, st, c->sa_rec.as<uint32_t>() + s0, (long long)ns, (uint32_t)n0);
    if (c->n_cig) BK_LAUNCH(add_offset_u32, GRID1(ns + 1, 256), 256, 0, st, c->cig_off.as<uint32_t>() + s0, (long long)ns + 1, (uint32_t)c->n_cig);
    if (c->sa_bytes) BK_LAUNCH(add_offset_u32, GRID1(ns + 1, 256), 256, 0, st, c->sa_off.as<uint32_t>() + s0, (long long)ns + 1, (uint32_t)c->sa_bytes);
    if (c->oc_bytes) BK_LAUNCH(add_offset_u32, GRID1(ns + 1, 256), 256, 0, st, c->oc_off.as<uint32_t>() + s0, (long long)ns + 1, (uint32_t)c->oc_bytes);
  } else if (s0 == 0) {
    CU(c, cudaMemsetAsync(c->cig_off.p, 0, 4, st)); CU(c, cudaMemsetAsync(c->sa_off.p, 0, 4, st)); CU(c, cudaMemsetAsync(c->oc_off.p, 0, 4, st));
  }
  if (ns) {                                             // optional read bases of the SA records
    if (b->seq_off && b->seq4 && b->seq_len && (s0 == 0 || c->have_seq)) {
      uint32_t nseq_b = 0;
      if (kind == cudaMemcpyHostToDevice) nseq_b = b->seq_off[ns];
      else CU(c, cudaMemcpy(&nseq_b, b->seq_off + ns, 4, cudaMemcpyDeviceToHost));
      TRY(c, c->seq_off.ensure((size_t)(s0 + ns + 1) * 4 + 64, (size_t)(s0 + 1) * 4, st));
      TRY(c, c->seq_len.ensure((size_t)(s0 + ns) * 4 + 64, (size_t)s0 * 4, st));
      TRY(c, c->seq4.ensure((size_t)c->seq_bytes + nseq_b + 64, (size_t)c->seq_bytes, st));
      CU(c, cudaMemcpyAsync(c->seq_off.as<uint32_t>() + s0, b->seq_off, (ns + 1) * 4, kind, st));
      CU(c, cudaMemcpyAsync(c->seq_len.as<int32_t>() + s0, b->seq_len, ns * 4, kind, st));
      if (nseq_b) CU(c, cudaMemcpyAsync(c->seq4.as<uint8_t>() + c->seq_bytes, b->seq4, nseq_b, kind, st));
      if (c->seq_bytes) BK_LAUNCH(add_offset_u32, GRID1(ns + 1, 256), 256, 0, st, c->seq_off.as<uint32_t>() + s0, (long long)ns + 1, (uint32_t)c->seq_bytes);
      c->seq_bytes += nseq_b; c->have_seq = true;
    } else c->have_seq = false;
  }
  c->n += b->n; c->n_x += b->n_x; c->n_sa += b->n_sa; c->n_cig += ncig; c->sa_bytes += nsa_b; c->oc_bytes += noc_b;
  set_ptrs(c);
  cudaEventRecord(c->ev[1], st);
  TRY(c, sync_check(c));
  float ms = 0; cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
  c->tm.h2d += ms;
  return 0;
}

int bkid_push_batch(bkid_ctx *c, const bkid_batch *b) { return push_impl(c, b, cudaMemcpyHostToDevice); }

int bkid_push_batch_device(bkid_ctx *c, const bkid_batch *b)
{
  if (!c || !b) return BKID_ERR_ARG;
  if (c->n == 0 && !c->borrowed && c->flag.p == nullptr) {
    // adopt the caller's device columns without copying (already-resident input), in whichever form they are
    cudaSetDevice(c->device);
    if ((unsigned long long)b->n >= 0xffffffffull) return fail(c, BKID_ERR_ARG, "more than 2^32-1 records per context");
    if (b->n > 0 && (!b->tid || (!b->isize && !b->isize16) || (!b->endpos && !b->span16)))
      return fail(c, BKID_ERR_ARG, "bkid_push_batch_device needs tid and the insert-size / span columns (wide or narrow) resident on the device");
    invalidate(c);
    c->borrowed = true;
    c->n = b->n; c->n_sa = b->n_sa; c->n_x = b->n_x;
    c->p_flag = b->flag; c->p_mapq = b->mapq; c->p_tid = b->tid; c->p_pos = b->pos;
    c->p_isize = b->isize; c->p_isize16 = b->isize ? nullptr : b->isize16;
    c->p_endpos = b->endpos; c->p_span16 = b->endpos ? nullptr : b->span16;
    c->form_isize = b->isize ? 1 : 2; c->form_span = b->endpos ? 1 : 2;
    c->p_x_rec = b->x_rec; c->p_x_mtid = b->x_mtid; c->p_x_mpos = b->x_mpos; c->p_x_nh = b->x_name_hash;
    c->p_sa_rec = b->sa_rec; c->p_cig_off = b->cig_off; c->p_cig_ops = b->cig_ops; c->p_sa_off = b->sa_off; c->p_sa_txt = b->sa_txt;
    c->p_oc_off = b->oc_off; c->p_oc_txt = b->oc_txt;
    c->p_seq_off = b->seq_off; c->p_seq4 = b->seq4; c->p_seq_len = b->seq_len; c->have_seq = b->seq_off && b->seq4 && b->seq_len;
    return 0;
  }
  return push_impl(c, b, cudaMemcpyDeviceToDevice);
}

int bkid_reset(bkid_ctx *c)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->st);
  invalidate(c);
  c->n = c->n_x = c->n_sa = c->n_cig = c->sa_bytes = c->oc_bytes = 0;
  c->seq_bytes = 0; c->have_seq = false;
  c->borrowed = false;
  c->form_isize = c->form_span = 0;         // the next first batch decides again (allocations are kept)
  set_ptrs(c);
  memset(&c->tm, 0, sizeof c->tm);
  c->launches0 = g_bk_launches;
  return 0;
}

int bkid_set_exclude(bkid_ctx *c, int64_t n_iv, const int32_t *tid, const int32_t *beg, const int32_t *end)
{
  if (!c || n_iv < 0 || (n_iv > 0 && (!tid || !beg || !end))) return c ? fail(c, BKID_ERR_ARG, "bad exclude intervals") : BKID_ERR_ARG;
  cudaSetDevice(c->device);
  std::vector<std::array<int32_t, 3>> v;
  for (int64_t k = 0; k < n_iv; ++k) {
    if (tid[k] < 0 || tid[k] >= c->nt) return fail(c, BKID_ERR_ARG, "exclude interval on an unknown target");
    int32_t b = beg[k] < 0 ? 0 : beg[k];
    if (end[k] > b) v.push_back({tid[k], b, end[k]});
  }
  std::sort(v.begin(), v.end());
  c->ex_iv.clear();
  for (auto &x : v) {                                   // merge overlapping / touching intervals
    size_t m = c->ex_iv.size();
    if (m && c->ex_iv[m - 3] == x[0] && x[1] <= c->ex_iv[m - 1]) { if (x[2] > c->ex_iv[m - 1]) c->ex_iv[m - 1] = x[2]; }
    else { c->ex_iv.push_back(x[0]); c->ex_iv.push_back(x[1]); c->ex_iv.push_back(x[2]); }
  }
  invalidate(c);
  return 0;
}

static ISizeCol isize_col(const bkid_ctx *c) { return ISizeCol{c->p_isize, c->p_isize16}; }

static int classify_impl(bkid_ctx *c)
{
  if (c->classified) return 0;
  cudaStream_t st = c->st;
  long long n = c->n;
  int ntiles = div_up(std::max<long long>(n, 1), K1_TILE);
  TRY(c, c->cls.ensure((size_t)n + 64, 0, st));
  TRY(c, c->cand_bits.ensure((size_t)n / 8 + 64, 0, st));
  unsigned long long *g = (unsigned long long *)(c->counters.as<unsigned>() + CS_G);
  CU(c, cudaMemsetAsync(g, 0, 64, st));
  cudaEventRecord(c->ev[2], st);
  const bool i16 = c->p_isize16 != nullptr, s16 = c->p_span16 != nullptr;
  if (n > 0) {
    uint8_t *cls = c->cls.as<uint8_t>();
    // persistent grid = exactly what is resident at once (a partial second wave of persistent CTAs would idle most SMs)
    int occ = 0;
    if (i16 && s16) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k1_classify<true, true>, K1_THREADS, 0);
    else if (i16) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k1_classify<true, false>, K1_THREADS, 0);
    else if (s16) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k1_classify<false, true>, K1_THREADS, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k1_classify<false, false>, K1_THREADS, 0);
    ntiles = std::min(ntiles, c->n_sm * std::max(occ, 1));
    if (i16 && s16) BK_LAUNCH((k1_classify<true, true>), (unsigned)ntiles, K1_THREADS, 0, st, c->p_flag, c->p_mapq, c->p_isize, c->p_isize16, c->p_span16, n, c->prm.qual, cls, c->cand_bits.as<uint8_t>(), g);
    else if (i16) BK_LAUNCH((k1_classify<true, false>), (unsigned)ntiles, K1_THREADS, 0, st, c->p_flag, c->p_mapq, c->p_isize, c->p_isize16, c->p_span16, n, c->prm.qual, cls, c->cand_bits.as<uint8_t>(), g);
    else if (s16) BK_LAUNCH((k1_classify<false, true>), (unsigned)ntiles, K1_THREADS, 0, st, c->p_flag, c->p_mapq, c->p_isize, c->p_isize16, c->p_span16, n, c->prm.qual, cls, c->cand_bits.as<uint8_t>(), g);
    else BK_LAUNCH((k1_classify<false, false>), (unsigned)ntiles, K1_THREADS, 0, st, c->p_flag, c->p_mapq, c->p_isize, c->p_isize16, c->p_span16, n, c->prm.qual, cls, c->cand_bits.as<uint8_t>(), g);
  }
  cudaEventRecord(c->ev[3], st);
  int n_iv = (int)(c->ex_iv.size() / 3);
  c->n_excluded = 0;
  unsigned long long ne = 0;
  if (n_iv > 0 && n > 0) {
    TRY(c, c->ex_tab.ensure((size_t)n_iv * 12 + 64, 0, st)); TRY(c, c->ex_lo.ensure((size_t)n_iv * 4 + 64, 0, st));
    TRY(c, c->ex_len.ensure((size_t)n_iv * 4 + 64, 0, st)); TRY(c, c->ex_pre.ensure((size_t)(n_iv + 1) * 8 + 64, 0, st));
    CU(c, cudaMemcpyAsync(c->ex_tab.p, c->ex_iv.data(), (size_t)n_iv * 12, cudaMemcpyHostToDevice, st));
    BK_LAUNCH(ex_ranges, GRID1(n_iv, 128), 128, 0, st, c->p_tid, c->p_pos, n, c->ex_tab.as<int32_t>(), n_iv, c->ex_lo.as<uint32_t>(), c->ex_len.as<uint32_t>());
    BK_LAUNCH(ex_prefix, 1, 32, 0, st, c->ex_len.as<uint32_t>(), n_iv, c->ex_pre.as<unsigned long long>());
    BK_LAUNCH(ex_apply, 148 * 8, 256, 0, st, c->ex_lo.as<uint32_t>(), c->ex_pre.as<unsigned long long>(), n_iv, isize_col(c), c->cls.as<uint8_t>(), c->cand_bits.as<uint8_t>(), g);
    CU(c, cudaMemcpyAsync(&ne, c->ex_pre.as<unsigned long long>() + n_iv, 8, cudaMemcpyDeviceToHost, st));
  }
  unsigned long long h[6] = {0, 0, 0, 0, 0, 0};
  CU(c, cudaMemcpyAsync(h, g, 48, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  c->n_excluded = (long long)ne;
  float ms = 0; cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]);
  c->tm.classify = ms;
  c->sum_abs = (long long)h[G_SUM]; c->cnt_insert = (long long)h[G_CNT]; c->sum_sq = h[G_SQ]; c->n_cand_k1 = (long long)h[G_CAND]; c->xmax = h[G_XMAX];
  if (s16) { c->maxspan = (int)h[G_SPAN] + 1; c->maxspan_cached = true; }    // the narrow span column was read by K1 anyway
  c->classified = true;
  c->tm.n_records = n;
  return 0;
}

// Upper bound K of the binade of the truncating sd accumulator (sd_fast): the final total is at most
// sum (x - mean)^2 + N (every element adds floor(a) and at most 1), and sum (x - S/N)^2 = (N sum x^2 - S^2) / N exactly.
// The slack covers the rounding of the mean, of the per-element products and the division.  51 = no useful bound
// (the sum of squares may have wrapped): every correction candidate then counts and the general path decides.
static int sd_upper_binade(unsigned long long sum_abs, unsigned long long cnt, unsigned long long sum_sq, unsigned long long xmax)
{
  if (cnt == 0) return 0;
  if (xmax > 65535ull) return 51;
  unsigned __int128 V = (unsigned __int128)sum_sq * cnt - (unsigned __int128)sum_abs * sum_abs;
  unsigned __int128 T = V / cnt + 1;
  T += (T >> 30) + 2 * (unsigned __int128)cnt + 1024;
  if (T >> 51) return 51;
  int k = 0;
  while ((T >> (k + 1)) != 0) ++k;
  return k;
}

// The insert-size statistics (src/BreakID.cc:1909-1954) on every path, single-GPU and sharded:
//   stats_begin   mean = S / N, the binade bound, and the one-pass form sd_fast launched asynchronously;
//   stats_collect joins it: F = sum floor(a) is the exact total when E == 0;
//   stats_replay  otherwise the exact, order-dependent replay (chained through the ranks when sharded);
//   stats_set     sd = sqrt(total / N).
// E as stats_collect reports it saturates at SD_E_SAT, which stays far from overflow when summed over the ranks.
static const unsigned long long SD_E_SAT = 1ull << 40;

// exact continuation of the truncating sd accumulator over the local records, starting from t_in:
// stats_prepare = the streaming pass that builds the per-block tables for `mean` (independent of t_in),
// stats_replay = the single-CTA exact walk from t_in.
static int stats_prepare(bkid_ctx *c, double mean)
{
  cudaStream_t st = c->st;
  long long n = c->n;
  c->sd_prepared = false;
  if (n <= 0 || c->cnt_insert <= 0) return 0;
  int nb = div_up(std::max<long long>(n, 1), SD_BLOCK);
  TRY(c, c->sdtab.ensure((size_t)nb * (8 + SD_K * 4 + 4 + 8) + 256, 0, st));
  TRY(c, c->sdlut.ensure((size_t)SD_LUT * 8, 0, st));
  char *bp = (char *)c->sdtab.p;
  long long *blkF = (long long *)bp; bp += (size_t)nb * 8;
  double *blkA = (double *)bp; bp += (size_t)nb * 8;
  uint32_t *blkCum = (uint32_t *)bp; bp += (size_t)nb * SD_K * 4;
  uint32_t *blkN = (uint32_t *)bp;
  BK_LAUNCH(sd_build_lut, SD_LUT / 256, 256, 0, st, mean, c->sdlut.as<unsigned long long>());
  BK_LAUNCH(sd_block_stats, (unsigned)nb, SD_THREADS, 0, st, c->cls.as<uint8_t>(), isize_col(c), n, mean, c->sdlut.as<unsigned long long>(), blkF, blkCum, blkN, blkA);
  c->sd_prepared = true; c->sd_mean = mean;
  return 0;
}

static int stats_replay(bkid_ctx *c, double mean, long long t_in, long long *t_out)
{
  cudaStream_t st = c->st;
  long long n = c->n;
  *t_out = t_in;
  if (n <= 0 || c->cnt_insert <= 0) return 0;
  SubTimer T_(st);
  if (!c->sd_prepared || c->sd_mean != mean) TRY(c, stats_prepare(c, mean));
  T_.mark("sd: block stats");
  int nb = div_up(std::max<long long>(n, 1), SD_BLOCK);
  char *bp = (char *)c->sdtab.p;
  long long *blkF = (long long *)bp; bp += (size_t)nb * 8;
  double *blkA = (double *)bp; bp += (size_t)nb * 8;
  uint32_t *blkCum = (uint32_t *)bp; bp += (size_t)nb * SD_K * 4;
  uint32_t *blkN = (uint32_t *)bp;
  long long *out = (long long *)(c->counters.as<unsigned>() + CS_SD_OUT);
  BK_LAUNCH(sd_resolve, 1, SDR_T, SD_BLOCK * 9, st, c->cls.as<uint8_t>(), isize_col(c), n, mean, nb, blkF, blkCum, blkN, blkA, t_in, out);
  T_.mark("sd: resolve");
  long long h[2] = {0, 0};
  CU(c, cudaMemcpyAsync(h, out, 16, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  if (h[1]) {                                                              // total left the closed-form regime: literal replay
    BK_LAUNCH(sd_sequential, 1, 1, 0, st, c->cls.as<uint8_t>(), isize_col(c), n, mean, t_in, out);
    CU(c, cudaMemcpyAsync(h, out, 16, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
  }
  *t_out = h[0];
  return 0;
}

// the one-pass form over the local records for `mean`: asynchronous on `st`, between ev_side[0] and ev_side[1]
static int sd_fast_launch(bkid_ctx *c, double mean, int kub, cudaStream_t st)
{
  long long n = c->n;
  unsigned long long *out = (unsigned long long *)(c->counters.as<unsigned>() + CS_SDF);
  c->sd_kub = kub;
  cudaEventRecord(c->ev_side[0], st);
  CU(c, cudaMemsetAsync(out, 0, 24, st));
  c->sd_fast_st = st;
  if (n > 0 && c->cnt_insert > 0) {
    double thr = 1.0 - ldexp(1.0, kub - 53);                                  // corrections need frac(a) >= 1 - 2^(k-53), k <= kub
    int occ = 0;
    if (c->p_isize16) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, sd_fast<true>, 256, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, sd_fast<false>, 256, 0);
    const int grid = c->n_sm * std::max(occ, 1);
    if (c->p_isize16) BK_LAUNCH((sd_fast<true>), grid, 256, 0, st, c->cls.as<uint8_t>(), c->p_isize, c->p_isize16, n, mean, thr, out);
    else BK_LAUNCH((sd_fast<false>), grid, 256, 0, st, c->cls.as<uint8_t>(), c->p_isize, c->p_isize16, n, mean, thr, out);
  }
  cudaEventRecord(c->ev_side[1], st);
  return 0;
}

// S, N, SQ, XM: K1's sums over the insert records, local on one GPU, all-reduced when sharded
static int stats_begin(bkid_ctx *c, unsigned long long S, unsigned long long N, unsigned long long SQ, unsigned long long XM, cudaStream_t st)
{
  c->mean = (double)(long long)S / (double)(long long)N;                      // src/BreakID.cc:1941 (0/0 = NaN like the reference)
  return sd_fast_launch(c, c->mean, sd_upper_binade(S, N, SQ, XM), st);
}

// F = sum floor(a), E = records that could need a correction.  E is forced to SD_E_SAT (the replay decides) when the pass
// left its regime, when the binade bound is useless (kub >= 51), or under BKID_SD_GENERAL (tests: force the replay).
// A context without insert records gives (0, 0).
static int stats_collect(bkid_ctx *c, unsigned long long *F, unsigned long long *E)
{
  cudaStream_t st = c->sd_fast_st;
  if (!st) return fail(c, BKID_ERR_ARG, "the one-pass sd form was collected before it was launched");
  unsigned long long h[3] = {0, 0, 0};
  CU(c, cudaMemcpyAsync(h, c->counters.as<unsigned>() + CS_SDF, 24, cudaMemcpyDeviceToHost, st));
  CU(c, cudaStreamSynchronize(st));
  CU(c, cudaGetLastError());
  c->sd_fast_st = nullptr;
  const bool force = h[2] || c->sd_kub >= 51 || getenv("BKID_SD_GENERAL") != nullptr;
  *F = h[0];
  *E = c->cnt_insert <= 0 ? 0 : force ? SD_E_SAT : std::min(h[1], SD_E_SAT);
  return 0;
}

static void stats_set(bkid_ctx *c, long long total, long long N)
{
  c->sd = sqrt((double)total / (double)N);                                   // :1946
  c->have_stats = true;
}

// one GPU: collect, replay when the one-pass form may be inexact, set.  tm.insert_stats = device time of the pass + the replay
static int stats_finish(bkid_ctx *c)
{
  unsigned long long F = 0, E = 0;
  TRY(c, stats_collect(c, &F, &E));
  float ms = 0; cudaEventElapsedTime(&ms, c->ev_side[0], c->ev_side[1]);
  long long total = (long long)F;
  if (E != 0) {
    cudaEventRecord(c->ev[4], c->st);
    TRY(c, stats_replay(c, c->mean, 0, &total));
    cudaEventRecord(c->ev[5], c->st);
    TRY(c, sync_check(c));
    float ms2 = 0; cudaEventElapsedTime(&ms2, c->ev[4], c->ev[5]);
    ms += ms2;
  }
  c->tm.insert_stats = ms;
  stats_set(c, total, c->cnt_insert);
  return 0;
}

// bkid_run: the sd pass on st2 (and, for a wide span column, the max-span reduction on st3) overlaps candidate
// extraction and the join's sort; scan_impl finishes the statistics before the join's emit needs the distance
static int side_launch(bkid_ctx *c)
{
  long long n = c->n;
  TRY(c, stats_begin(c, c->sum_abs, c->cnt_insert, c->sum_sq, c->xmax, c->st2));
  if (!c->maxspan_cached) {
    // the max reference span bounds the region-query windows of the refinement only: its own stream, collected there
    int *mx = (int *)(c->counters.as<unsigned>() + CS_MAXSPAN);
    CU(c, cudaMemsetAsync(mx, 0, 4, c->st3));
    if (n > 0) BK_LAUNCH(max_span_kernel, 1184, 256, 0, c->st3, c->p_pos, c->p_endpos, n, mx);
    c->maxspan_pending = true;
  }
  return 0;
}

static int maxspan_collect(bkid_ctx *c)
{
  if (!c->maxspan_pending) return 0;
  int maxspan = 0;
  CU(c, cudaMemcpyAsync(&maxspan, c->counters.as<unsigned>() + CS_MAXSPAN, 4, cudaMemcpyDeviceToHost, c->st3));
  CU(c, cudaStreamSynchronize(c->st3));
  CU(c, cudaGetLastError());
  c->maxspan = maxspan + 1; c->maxspan_cached = true; c->maxspan_pending = false;
  return 0;
}

int bkid_insert_stats(bkid_ctx *c, double *mean, double *sd)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->err.clear();
  TRY(c, classify_impl(c));
  if (!c->have_stats) {
    TRY(c, stats_begin(c, c->sum_abs, c->cnt_insert, c->sum_sq, c->xmax, c->st));
    TRY(c, stats_finish(c));
  }
  if (mean) *mean = c->mean;
  if (sd) *sd = c->sd;
  return 0;
}

// ---- scan, in three reusable pieces (the multi-GPU path runs them around two exchanges) -------------
// (1) local candidates in file order -> c->cand, straight from the sparse mate/name table (no host round trip: the
// count stays on the device in CS_NC; K1's count n_cand_k1 sizes everything and is checked against it later).
// with_keys: also write the join's (name_lo, index) sort pairs.
static int extract_candidates(bkid_ctx *c, unsigned long long index_offset, bool with_keys)
{
  TRY(c, classify_impl(c));
  cudaStream_t st = c->st;
  long long n = c->n, nx = c->n_x;
  long long cap = std::min<long long>(c->n_cand_k1, nx);      // every candidate is listed: more than n_x cannot be found
  c->n_cand = cap;
  unsigned *cs = c->counters.as<unsigned>();
  CU(c, cudaMemsetAsync(cs + CS_NC, 0, 8, st));
  TRY(c, c->cand.ensure((size_t)(cap + 1) * sizeof(bkid_cand), 0, st));
  if (nx <= 0 || n <= 0) return 0;
  int ntiles = div_up(nx, KX_TILE);
  TRY(c, c->sc.ensure(std::max<long long>(cap, ntiles) + 8, st));
  TRY(c, c->tile_cand.ensure((size_t)(ntiles + 1) * 4 * 2 + (size_t)ntiles * KX_THREADS + 64, 0, st));       // one flag byte per kx thread
  uint32_t *tile_cnt = c->tile_cand.as<uint32_t>(), *tile_off = tile_cnt + ntiles + 1;
  uint8_t *is_cand = (uint8_t *)(tile_off + ntiles + 1);                 // 4 candidate bits per kx thread
  unsigned long long *tot = (unsigned long long *)(cs + CS_TOTAL);
  BK_LAUNCH(kx_count, (unsigned)ntiles, KX_THREADS, 0, st, c->p_x_rec, nx, c->cand_bits.as<uint8_t>(), n, tile_cnt, is_cand, (int *)(cs + CS_XBAD));
  bk::exclusive_scan<uint32_t, uint32_t>(tile_cnt, tile_off, ntiles, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
  CU(c, cudaMemcpyAsync(cs + CS_NC, tot, 4, cudaMemcpyDeviceToDevice, st));
  if (cap > 0)     // a table that lists more candidates than K1 counted cannot exist (same predicate, same class bytes)
    BK_LAUNCH(kx_write, (unsigned)ntiles, KX_THREADS, 0, st, c->p_x_rec, nx, is_cand, n, tile_off, c->p_flag, c->p_mapq, c->p_tid, c->p_pos, c->p_x_mtid, c->p_x_mpos, c->p_x_nh,
              index_offset, c->cand.as<bkid_cand>(), with_keys ? c->sc.keys.as<uint64_t>() : (uint64_t *)nullptr, c->sc.vals.as<uint32_t>());
  return 0;
}
// the deferred check of (1): called at the next host synchronisation
static int check_candidates(bkid_ctx *c, const unsigned *h_nc_bad)
{
  if (h_nc_bad[1]) return fail(c, BKID_ERR_ARG, "the sparse mate/name table is not strictly ascending or points outside the batch (x_rec)");
  if ((long long)h_nc_bad[0] != c->n_cand_k1)
    return fail(c, BKID_ERR_ARG, "a discordant-scan candidate is missing from the sparse mate/name table (x_rec must list every record that is not a proper pair)");
  return 0;
}

// (2) mate join on a candidate array that is in global file order -> pairs in emission order in c->pairs_tmp.
// join_presort needs no distance (sort on 32 bits of the name hash); join_emit applies the discordance test.
// nc_dev: exact candidate count on the device (or nullptr: nc is exact).
static int join_presort(bkid_ctx *c, const bkid_cand *cand, long long nc, const uint32_t *nc_dev, bool keys_ready)
{
  cudaStream_t st = c->st;
  if (nc <= 0) return 0;
  TRY(c, c->sc.ensure(nc + 8, st));
  uint64_t *key = c->sc.keys.as<uint64_t>();
  uint32_t *val = c->sc.vals.as<uint32_t>();
  if (!keys_ready) BK_LAUNCH(k2_cand_keys, GRID1(nc, 256), 256, 0, st, cand, nc, key, val);
  if (bk::radix_sort_pairs(key, val, nc, 0, 32, c->sc.rt(), st, nc_dev) < 0) return fail(c, BKID_ERR_ARG, "more than 2^30 candidates");
  size_t maxp = (size_t)nc / 2 + 1;
  TRY(c, c->pairs_tmp.ensure(maxp * sizeof(bkid_pair), 0, st));
  return 0;
}

static int join_emit(bkid_ctx *c, const bkid_cand *cand, long long nc, const uint32_t *nc_dev, double w, bool check_table, long long *np_out)
{
  cudaStream_t st = c->st;
  *np_out = 0;
  unsigned *cs = c->counters.as<unsigned>();
  unsigned long long *tot = (unsigned long long *)(cs + CS_TOTAL);
  uint64_t *key = c->sc.keys.as<uint64_t>();
  uint32_t *val = c->sc.vals.as<uint32_t>();
  uint32_t *flag = c->sc.a32.as<uint32_t>(), *off = c->sc.b32.as<uint32_t>(), *mate = c->sc.c32.as<uint32_t>();
  int *big = (int *)(cs + CS_HASH_ERR);
  unsigned long long np = 0; int hbig = 0; unsigned hnc[2] = {0, 0};
  for (int attempt = 0; attempt < 2 && nc > 0; ++attempt) {
    CU(c, cudaMemsetAsync(big, 0, 4, st));
    CU(c, cudaMemsetAsync(mate, 0xff, (size_t)nc * 4, st));
    // attempt 0: groups = equal low 32 bits of the name hash, mixed groups up to 64 records are put in order in place;
    // attempt 1 (a larger mixed group exists): the remaining 32 bits are sorted too, groups = equal name_lo
    if (attempt == 1 && bk::radix_sort_pairs(key, val, nc, 32, 64, c->sc.rt(), st, nc_dev) < 0) return fail(c, BKID_ERR_ARG, "more than 2^30 candidates");
    BK_LAUNCH(k2_join, GRID1(nc, 256), 256, 0, st, key, val, nc_dev, (uint32_t)nc, cand, attempt == 0 ? 32 : 64, attempt == 0 ? 64u : 4096u, w, mate, big);
    BK_LAUNCH(k2_mate_flags, GRID1(nc, 256), 256, 0, st, mate, nc, flag);
    bk::exclusive_scan<uint32_t, uint32_t>(flag, off, nc, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
    BK_LAUNCH(k2_build_pairs, GRID1(nc, 256), 256, 0, st, mate, off, nc, cand, c->d_cum.as<uint32_t>(), c->nt, c->d_bucket_rank.as<int32_t>(), c->pairs_tmp.as<bkid_pair>());
    CU(c, cudaMemcpyAsync(&np, tot, 8, cudaMemcpyDeviceToHost, st));
    CU(c, cudaMemcpyAsync(&hbig, big, 4, cudaMemcpyDeviceToHost, st));
    CU(c, cudaMemcpyAsync(hnc, cs + CS_NC, 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    if (!hbig) break;
    if (attempt == 1) return fail(c, BKID_ERR_HASH, "more than 4096 records share a 64-bit read-name hash without sharing the name");
  }
  if (check_table) { if (nc <= 0) { CU(c, cudaMemcpyAsync(hnc, cs + CS_NC, 8, cudaMemcpyDeviceToHost, st)); TRY(c, sync_check(c)); } TRY(c, check_candidates(c, hnc)); }
  *np_out = (long long)np;
  return 0;
}

static int join_candidates(bkid_ctx *c, const bkid_cand *cand, long long nc, double w, long long *np_out)
{
  TRY(c, join_presort(c, cand, nc, nullptr, false));
  return join_emit(c, cand, nc, nullptr, w, false, np_out);
}

// (3) group the pairs by bucket, build buckets -> c->pairs0 ...  ordered: the pairs arrive in emission order (one GPU's
// join) and only need the stable grouping by bucket rank; otherwise they are ordered by (bucket rank, second-mate index)
static int set_pairs(bkid_ctx *c, const bkid_pair *pairs, long long np, bool ordered)
{
  cudaStream_t st = c->st;
  c->np0 = np; c->nb = 0;
  if (np <= 0) return 0;
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  TRY(c, c->sc.ensure(np + 8, st));
  TRY(c, c->pairs0.ensure((size_t)np * sizeof(bkid_pair), 0, st));
  unsigned long long *pkey = (unsigned long long *)c->sc.keys.as<uint64_t>();
  uint32_t *pslot = c->sc.vals.as<uint32_t>();
  BK_LAUNCH(k2_pair_keys, GRID1(np, 256), 256, 0, st, pairs, np, ordered ? 1 : 0, pkey, pslot);
  int rbits = 1; while ((1ll << rbits) < (long long)(c->nt + 1) * (c->nt + 1) + 1) ++rbits;
  if (bk::radix_sort_pairs((uint64_t *)pkey, pslot, np, ordered ? PAIR_IDX_BITS : 0, PAIR_IDX_BITS + rbits, c->sc.rt(), st) < 0) return fail(c, BKID_ERR_ARG, "more than 2^30 pairs");
  uint32_t *bh = c->sc.a32.as<uint32_t>(), *bhx = c->sc.b32.as<uint32_t>();
  BK_LAUNCH(k2_gather_pairs, GRID1(np, 256), 256, 0, st, pairs, pslot, pkey, np, c->pairs0.as<bkid_pair>(), bh);
  bk::exclusive_scan<uint32_t, uint32_t>(bh, bhx, np, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
  unsigned long long nbk = 0;
  CU(c, cudaMemcpyAsync(&nbk, tot, 8, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  c->nb = (int)nbk;
  TRY(c, c->bucket_off0.ensure((size_t)(nbk + 2) * 4, 0, st));
  TRY(c, c->bucket_rank_of.ensure((size_t)(nbk + 2) * 4, 0, st));
  BK_LAUNCH(k2_bucket_ids, GRID1(np, 256), 256, 0, st, c->pairs0.as<bkid_pair>(), bh, bhx, np, c->bucket_off0.as<uint32_t>(), c->bucket_rank_of.as<int32_t>());
  uint32_t npu = (uint32_t)np;
  CU(c, cudaMemcpyAsync(c->bucket_off0.as<uint32_t>() + nbk, &npu, 4, cudaMemcpyHostToDevice, st));
  TRY(c, c->X.ensure((size_t)np * 4 + 64, 0, st)); TRY(c, c->Y.ensure((size_t)np * 4 + 64, 0, st)); TRY(c, c->bucket_of_pair.ensure((size_t)np * 4 + 64, 0, st));
  BK_LAUNCH(pair_xy, GRID1(np, 256), 256, 0, st, c->pairs0.as<bkid_pair>(), np, c->X.as<uint32_t>(), c->Y.as<uint32_t>(), c->bucket_of_pair.as<uint32_t>());
  return sync_check(c);
}

// (1) + (2) + (3) on one GPU.  w_from_stats (bkid_run): insert statistics begun by side_launch are finished between the
// join's distance-independent presort and its emit, and *w becomes the reference's distance from them
static int scan_impl(bkid_ctx *c, double *w, bool w_from_stats)
{
  cudaStream_t st = c->st;
  const uint32_t *nc_dev = c->counters.as<unsigned>() + CS_NC;
  cudaEventRecord(c->ev[6], st);
  TRY(c, extract_candidates(c, 0ull, true));
  TRY(c, join_presort(c, c->cand.as<bkid_cand>(), c->n_cand, nc_dev, true));
  if (w_from_stats) {
    if (!c->have_stats) TRY(c, stats_finish(c));
    const int times = c->prm.times;
    *w = times * sqrt((double)times) * (c->mean + c->prm.sd_mult * c->sd);    // src/BreakID.cc:103
  }
  long long np = 0;
  TRY(c, join_emit(c, c->cand.as<bkid_cand>(), c->n_cand, nc_dev, *w, true, &np));
  cudaEventRecord(c->ev[7], st);
  TRY(c, set_pairs(c, c->pairs_tmp.as<bkid_pair>(), np, true));
  cudaEventRecord(c->ev[8], st);
  TRY(c, sync_check(c));
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]); c->tm.join = ms;
  cudaEventElapsedTime(&ms, c->ev[7], c->ev[8]); c->tm.bucket_sort = ms;
  c->tm.n_candidates = c->n_cand; c->tm.n_pairs = c->np0;
  c->scanned = true; c->clustered = c->refined = false;
  return 0;
}

int bkid_scan(bkid_ctx *c, double w, int64_t *n_pairs)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->err.clear();
  TRY(c, classify_impl(c));
  TRY(c, scan_impl(c, &w, false));
  if (n_pairs) *n_pairs = c->np0;
  return 0;
}

// K6: one summary record per cluster of the member list (c->mem_pair / mem_bucket / mem_cluster index c->pairs0, grouped by
// (bucket, cluster id)); clusters whose mean positions are closer than 2*dist on one chromosome are dropped (src/BreakID.cc:300-350)
static int summarize_impl(bkid_ctx *c, double dist)
{
  cudaStream_t st = c->st;
  if (c->n2 > 0) {
    long long nm = c->n2;
    TRY(c, c->sc.ensure(nm + 8, st));
    uint32_t *head = c->sc.a32.as<uint32_t>(), *hex = c->sc.b32.as<uint32_t>(), *start = c->sc.c32.as<uint32_t>(), *keep = c->sc.d32.as<uint32_t>(), *koff = c->sc.e32.as<uint32_t>();
    unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
    BK_LAUNCH(k6_cluster_heads, GRID1(nm, 256), 256, 0, st, c->mem_bucket.as<uint32_t>(), c->mem_cluster.as<int32_t>(), nm, head);
    bk::exclusive_scan<uint32_t, uint32_t>(head, hex, nm, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
    unsigned long long ncl = 0;
    CU(c, cudaMemcpyAsync(&ncl, tot, 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    BK_LAUNCH(k6_cluster_starts, GRID1(nm, 256), 256, 0, st, head, hex, nm, start);
    TRY(c, c->clusters.ensure((size_t)(ncl + 1) * sizeof(bkid_cluster_rec), 0, st));
    TRY(c, c->clusters_out.ensure((size_t)(ncl + 1) * sizeof(bkid_cluster_rec), 0, st));
    BK_LAUNCH(k6_summarize, GRID1(ncl, 128), 128, 0, st, c->pairs0.as<bkid_pair>(), c->mem_pair.as<uint32_t>(), c->mem_cluster.as<int32_t>(), start, (uint32_t)ncl, nm, dist,
              c->clusters_out.as<bkid_cluster_rec>(), keep);
    bk::exclusive_scan<uint32_t, uint32_t>(keep, koff, (long long)ncl, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
    unsigned long long nk = 0;
    CU(c, cudaMemcpyAsync(&nk, tot, 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    BK_LAUNCH(compact_clusters, GRID1(ncl, 128), 128, 0, st, c->clusters_out.as<bkid_cluster_rec>(), keep, koff, (uint32_t)ncl, c->clusters.as<bkid_cluster_rec>());
    c->n_clusters = (long long)nk;
    c->tm.n_clustered = nm;
  }
  return 0;
}

int bkid_cluster(bkid_ctx *c, double dist, int mode, int64_t *n_clusters)
{
  if (!c) return BKID_ERR_ARG;
  if (!c->scanned) return fail(c, BKID_ERR_ARG, "bkid_cluster before bkid_scan");
  cudaSetDevice(c->device);
  c->err.clear();
  cudaStream_t st = c->st;
  c->n1 = c->n2 = 0; c->n_clusters = 0; c->clusters_ranked = false;
  cudaEventRecord(c->ev[9], st);
  if (c->np0 > 0) {
    long long np = c->np0;
    TRY(c, c->sc.ensure(np + 8, st));
    // initial order = scan emission order (already grouped by bucket)
    TRY(c, c->tmpB.ensure((size_t)np * 4 + 64, 0, st));
    uint32_t *cur0 = c->tmpB.as<uint32_t>();
    BK_LAUNCH(iota_u32, GRID1(np, 256), 256, 0, st, cur0, np);
    // tmpB is used by nothing inside remove_isolated_all except via explicit arguments
    TRY(c, remove_isolated_all(c, cur0, c->bucket_of_pair.as<uint32_t>(), c->bucket_off0.as<uint32_t>(), np, c->nb, c->X.as<uint32_t>(), c->Y.as<uint32_t>(), dist));
  }
  cudaEventRecord(c->ev[10], st);
  if (c->n1 > 0) {
    if (mode) TRY(c, cluster_fast(c, c->cur1.as<uint32_t>(), c->curb1.as<uint32_t>(), c->seg1.as<uint32_t>(), c->n1, c->nb, c->X.as<uint32_t>(), c->Y.as<uint32_t>(), dist, c->np0));
    else TRY(c, cluster_ahc(c, c->cur1.as<uint32_t>(), c->curb1.as<uint32_t>(), c->seg1.as<uint32_t>(), c->n1, c->nb, c->X.as<uint32_t>(), c->Y.as<uint32_t>(), dist));
  }
  cudaEventRecord(c->ev[11], st);
  TRY(c, summarize_impl(c, dist));
  cudaEventRecord(c->ev[12], st);
  TRY(c, sync_check(c));
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev[9], c->ev[10]); c->tm.mask = ms;
  cudaEventElapsedTime(&ms, c->ev[10], c->ev[11]); c->tm.cluster = ms;
  cudaEventElapsedTime(&ms, c->ev[11], c->ev[12]); c->tm.summarize = ms;
  c->tm.n_masked = c->n1; c->tm.n_clusters = c->n_clusters;
  c->clustered = true; c->refined = false;
  if (n_clusters) *n_clusters = c->n_clusters;
  return 0;
}

int bkid_set_nib(bkid_ctx *c, int32_t tid, const uint8_t *packed, uint64_t n_bases)
{
  if (!c || tid < 0 || tid >= c->nt) return c ? fail(c, BKID_ERR_ARG, "bad tid") : BKID_ERR_ARG;
  cudaSetDevice(c->device);
  size_t bytes = (size_t)((n_bases + 1) / 2);
  TRY(c, c->nib[tid].ensure(bytes + 64, 0, c->st));
  CU(c, cudaMemcpyAsync(c->nib[tid].p, packed, bytes, cudaMemcpyHostToDevice, c->st));
  c->nib_len[tid] = n_bases;
  void *p = c->nib[tid].p;
  CU(c, cudaMemcpyAsync((char *)c->d_nib_ptr.p + (size_t)tid * 8, &p, 8, cudaMemcpyHostToDevice, c->st));
  CU(c, cudaMemcpyAsync((char *)c->d_nib_len.p + (size_t)tid * 8, &n_bases, 8, cudaMemcpyHostToDevice, c->st));
  return sync_check(c);
}

// ---- refinement, in reusable pieces (the multi-GPU path all-reduces the two partial-count buffers) -----
static int refine_build_rows(bkid_ctx *c)
{
  cudaStream_t st = c->st;
  TRY(c, classify_impl(c));
  TRY(c, c->sarows.ensure((size_t)(c->n_sa + 1) * sizeof(EvRow), 0, st));
  {
    int *miss = (int *)(c->counters.as<unsigned>() + CS_MISSING);
    CU(c, cudaMemsetAsync(miss, 0, 4, st));
    if (c->n_sa > 0) {
      BK_LAUNCH(k7_evidence_rows, GRID1(c->n_sa, 128), 128, 0, st, c->p_sa_rec, c->n_sa, c->cls.as<uint8_t>(), c->p_flag, c->p_tid, c->p_pos, c->p_endpos, c->p_span16, c->p_x_rec, c->n_x, c->p_x_nh, miss,
                c->p_cig_off, c->p_cig_ops, c->p_sa_off, c->p_sa_txt, c->p_oc_off, c->p_oc_txt, c->prm.mismatch_num, c->sarows.as<EvRow>());
      int hm = 0;
      CU(c, cudaMemcpyAsync(&hm, miss, 4, cudaMemcpyDeviceToHost, st));
      TRY(c, sync_check(c));
      if (hm) return fail(c, BKID_ERR_ARG, "an SA-tagged record is missing from the sparse mate/name table");
      if (c->prm.validate_align) {
        if (!c->have_seq) return fail(c, BKID_ERR_ARG, "validate_align needs the read bases of the SA records (bkid_batch seq_off / seq4 / seq_len)");
        BK_LAUNCH(k7_validate_rows, GRID1(c->n_sa, AL_WARPS), AL_WARPS * 32, 0, st, c->p_sa_rec, c->n_sa, c->p_flag, c->p_cig_off, c->p_cig_ops, c->p_sa_off, c->p_sa_txt,
                  c->p_oc_off, c->p_seq_off, c->p_seq4, c->p_seq_len, c->d_canon.as<uint64_t>(), c->nt, (const uint8_t *const *)c->d_nib_ptr.p, c->d_nib_len.as<uint64_t>(),
                  c->sarows.as<EvRow>());
      }
    }
  }
  c->rows_ptr = c->sarows.as<EvRow>(); c->n_rows = c->n_sa;
  return 0;
}

static int refine_local_maxspan(bkid_ctx *c, int *out)
{
  cudaStream_t st = c->st;
  if (c->maxspan_pending) { TRY(c, maxspan_collect(c)); *out = c->maxspan; return 0; }
  if (c->p_span16) { TRY(c, classify_impl(c)); *out = c->maxspan; return 0; }     // K1 read the narrow span column
  int *mx = (int *)(c->counters.as<unsigned>() + CS_MAXSPAN);
  CU(c, cudaMemsetAsync(mx, 0, 4, st));
  if (c->n > 0) BK_LAUNCH(max_span_kernel, 1184, 256, 0, st, c->p_pos, c->p_endpos, c->n, mx);
  int maxspan = 0;
  CU(c, cudaMemcpyAsync(&maxspan, mx, 4, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  *out = maxspan + 1;
  return 0;
}

static RefineView refine_view(bkid_ctx *c)
{
  RefineView v;
  v.n = c->n; v.cls = c->cls.as<uint8_t>(); v.tid = c->p_tid; v.pos = c->p_pos; v.endpos = c->p_endpos; v.span16 = c->p_span16;
  v.n_sa = c->n_rows; v.rows = (const EvRow *)c->rows_ptr; v.maxspan = c->maxspan;
  v.name_key = c->name_key.as<uint64_t>(); v.name_row = c->name_row.as<uint32_t>();
  v.canon = c->d_canon.as<uint64_t>(); v.nt = c->nt;
  v.nib = (const uint8_t *const *)c->d_nib_ptr.p; v.nib_len = c->d_nib_len.as<uint64_t>();
  return v;
}

// regions + partial coverage of the local record shard -> c->cov [2*ncl]
static int refine_coverage(bkid_ctx *c, double dist)
{
  cudaStream_t st = c->st;
  uint32_t ncl = (uint32_t)c->n_clusters;
  TRY(c, classify_impl(c));
  TRY(c, c->sc.ensure((long long)ncl + 8, st));
  TRY(c, c->work.ensure((size_t)(ncl + 1) * sizeof(ClusterWork), 0, st));
  TRY(c, c->cov.ensure((size_t)(2 * ncl + 2) * 4, 0, st));
  TRY(c, c->depth.ensure((size_t)(2 * ncl + 2) * 4, 0, st));
  TRY(c, c->evoff.ensure((size_t)(ncl + 2) * 4, 0, st));
  if (ncl == 0) return 0;
  RefineView v = refine_view(c);
  int w = (int)dist;                                                       // const int w (src/BreakID.cc:390)
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  uint32_t *evcap = c->sc.a32.as<uint32_t>();
  BK_LAUNCH(k7_regions, GRID1(ncl, 128), 128, 0, st, v, c->clusters.as<bkid_cluster_rec>(), ncl, w, c->work.as<ClusterWork>(), evcap);
  bk::exclusive_scan<uint32_t, uint32_t>(evcap, c->evoff.as<uint32_t>(), ncl, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
  BK_LAUNCH(k7_coverage, GRID1(ncl, 4), 128, 0, st, v, c->work.as<ClusterWork>(), ncl, c->cov.as<uint32_t>());
  unsigned long long nev = 0;
  CU(c, cudaMemcpyAsync(&nev, tot, 8, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  c->n_evcap = (long long)nev;
  return 0;
}

// gate + evidence pairing + vote (needs TOTAL coverage in c->cov)
static int refine_vote(bkid_ctx *c)
{
  cudaStream_t st = c->st;
  uint32_t ncl = (uint32_t)c->n_clusters;
  if (ncl == 0) return 0;
  // evidence rows ordered by read-name hash (pairing looks a split read's other half up by name)
  TRY(c, c->sc.ensure(std::max<long long>(ncl, c->n_rows) + 8, st));
  TRY(c, c->name_key.ensure((size_t)(c->n_rows + 1) * 8, 0, st));
  TRY(c, c->name_row.ensure((size_t)(c->n_rows + 1) * 4, 0, st));
  if (c->n_rows > 0) {
    BK_LAUNCH(k7_name_keys, GRID1(c->n_rows, 256), 256, 0, st, (const EvRow *)c->rows_ptr, c->n_rows, c->name_key.as<uint64_t>(), c->name_row.as<uint32_t>());
    bk::radix_sort_pairs(c->name_key.as<uint64_t>(), c->name_row.as<uint32_t>(), c->n_rows, 0, 32, c->sc.rt(), st);
  }
  RefineView v = refine_view(c);
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  ClusterWork *work = c->work.as<ClusterWork>();
  uint32_t *entcnt = c->sc.c32.as<uint32_t>(), *entoff = c->sc.d32.as<uint32_t>();
  TRY(c, c->valid.ensure((size_t)(ncl + 2) * 4, 0, st));
  TRY(c, c->tmpC.ensure((size_t)(c->n_evcap + 1) * 4, 0, st));
  int *fatal = (int *)(c->counters.as<unsigned>() + CS_FATAL);
  CU(c, cudaMemsetAsync(fatal, 0, 4, st));
  BK_LAUNCH((k7_collect<false>), ncl, RF_THREADS, 0, st, v, c->clusters.as<bkid_cluster_rec>(), ncl, work, c->cov.as<uint32_t>(), c->evoff.as<uint32_t>(),
            c->tmpC.as<uint32_t>(), (const uint32_t *)nullptr, (int2 *)nullptr);
  BK_LAUNCH(k7_entry_counts, GRID1(ncl, 128), 128, 0, st, work, ncl, entcnt, fatal);
  bk::exclusive_scan<uint32_t, uint32_t>(entcnt, entoff, ncl, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
  unsigned long long nent = 0; int hf = 0;
  CU(c, cudaMemcpyAsync(&nent, tot, 8, cudaMemcpyDeviceToHost, st));
  CU(c, cudaMemcpyAsync(&hf, fatal, 4, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  if (hf) return fail(c, BKID_ERR_CIGAR, "error cigar: a complementary split alignment has no clip (reference exits at src/BreakID.cc:954-968)");
  TRY(c, c->tmpD.ensure((size_t)(nent + 1) * sizeof(int2), 0, st));
  BK_LAUNCH((k7_collect<true>), ncl, RF_THREADS, 0, st, v, c->clusters.as<bkid_cluster_rec>(), ncl, work, c->cov.as<uint32_t>(), c->evoff.as<uint32_t>(),
            c->tmpC.as<uint32_t>(), entoff, c->tmpD.as<int2>());
  BK_LAUNCH(k8_vote, ncl, RF_THREADS, 0, st, c->clusters.as<bkid_cluster_rec>(), ncl, work, entoff, c->tmpD.as<int2>(), c->prm.bp_pos_error, c->valid.as<uint32_t>());
  if (nent > K8_SMALL) {                                                   // only then can a cluster be heavy
    TRY(c, c->tmpE.ensure((size_t)(nent + 1) * 8, 0, st));
    TRY(c, c->tmpF.ensure((size_t)(nent + 1) * 4, 0, st));
    if (!c->k8_attr_set) { cudaFuncSetAttribute(k8_vote_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(K8_BIG_SMEM_KEYS * 8)); c->k8_attr_set = true; }   // per device: kept per context
    BK_LAUNCH(k8_vote_big, ncl, K8_BIG_THREADS, K8_BIG_SMEM_KEYS * 8, st, c->clusters.as<bkid_cluster_rec>(), ncl, work, entoff, c->tmpD.as<int2>(), c->tmpE.as<uint64_t>(),
              c->tmpF.as<uint32_t>(), c->prm.bp_pos_error, c->valid.as<uint32_t>());
  }
  c->tm.n_evidence = (long long)nent;
  return 0;
}

static int refine_depth(bkid_ctx *c)
{
  uint32_t ncl = (uint32_t)c->n_clusters;
  if (ncl == 0) return 0;
  RefineView v = refine_view(c);
  BK_LAUNCH(k9_depth, GRID1(ncl, 4), 128, 0, c->st, v, c->clusters.as<bkid_cluster_rec>(), c->valid.as<uint32_t>(), ncl, c->depth.as<uint32_t>());
  return 0;
}

static int refine_finish(bkid_ctx *c)
{
  cudaStream_t st = c->st;
  uint32_t ncl = (uint32_t)c->n_clusters;
  c->n_called = 0;
  if (ncl == 0) return 0;
  RefineView v = refine_view(c);
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  BK_LAUNCH(k10_finish, GRID1(ncl, 128), 128, 0, st, v, c->clusters.as<bkid_cluster_rec>(), c->valid.as<uint32_t>(), c->depth.as<uint32_t>(), ncl);
  uint32_t *voff = c->sc.b32.as<uint32_t>();
  bk::exclusive_scan<uint32_t, uint32_t>(c->valid.as<uint32_t>(), voff, ncl, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
  unsigned long long nv = 0;
  CU(c, cudaMemcpyAsync(&nv, tot, 8, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  TRY(c, c->clusters_out.ensure((size_t)(ncl + 1) * sizeof(bkid_cluster_rec), 0, st));
  BK_LAUNCH(compact_clusters, GRID1(ncl, 128), 128, 0, st, c->clusters.as<bkid_cluster_rec>(), c->valid.as<uint32_t>(), voff, ncl, c->clusters_out.as<bkid_cluster_rec>());
  c->n_called = (long long)nv;
  return sync_check(c);
}

int bkid_refine(bkid_ctx *c, double dist, int64_t *n_called)
{
  if (!c) return BKID_ERR_ARG;
  if (!c->clustered) return fail(c, BKID_ERR_ARG, "bkid_refine before bkid_cluster");
  cudaSetDevice(c->device);
  c->err.clear();
  cudaStream_t st = c->st;
  c->n_called = 0;
  cudaEventRecord(c->ev[13], st);
  if (c->n_clusters > 0) {
    TRY(c, refine_build_rows(c));
    TRY(c, maxspan_collect(c));
    if (!c->maxspan_cached) TRY(c, refine_local_maxspan(c, &c->maxspan));
    cudaEventRecord(c->ev[14], st);
    TRY(c, refine_coverage(c, dist));
    TRY(c, refine_vote(c));
    TRY(c, refine_depth(c));
    TRY(c, refine_finish(c));
  } else cudaEventRecord(c->ev[14], st);
  cudaEventRecord(c->ev[15], st);
  TRY(c, sync_check(c));
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev[13], c->ev[14]); c->tm.evidence = ms;
  cudaEventElapsedTime(&ms, c->ev[14], c->ev[15]); c->tm.refine = ms;
  c->tm.n_sa = c->n_sa; c->tm.n_called = c->n_called;
  c->refined = true;
  if (n_called) *n_called = c->n_called;
  return 0;
}

// =============================================================================================
// Shard entry points (multi-GPU; one context per rank, exchanges done by the caller -- see
// breakid_b200/dist.py).  Device pointers handed out stay valid until the next call on the context.
// =============================================================================================

int bkid_shard_insert_partial(bkid_ctx *c, int64_t *sum_abs, int64_t *count, uint64_t *sum_sq, uint64_t *max_abs)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, classify_impl(c));
  *sum_abs = c->sum_abs; *count = c->cnt_insert;
  if (sum_sq) *sum_sq = c->sum_sq;
  if (max_abs) *max_abs = c->xmax;
  return 0;
}

int bkid_sd_upper_binade(uint64_t sum_abs, uint64_t count, uint64_t sum_sq, uint64_t max_abs)
{
  return sd_upper_binade(sum_abs, count, sum_sq, max_abs);
}

// one-pass form over the local records with the GLOBAL mean and binade bound: asynchronous on the side stream, so it
// overlaps candidate extraction and the candidate all-to-all; bkid_shard_sd_fast_collect joins it
int bkid_shard_sd_fast(bkid_ctx *c, double mean, int32_t upper_binade)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, classify_impl(c));
  return sd_fast_launch(c, mean, upper_binade, c->st2);
}

int bkid_shard_sd_fast_collect(bkid_ctx *c, uint64_t *sum_floor, uint64_t *n_correctable)
{
  if (!c || !sum_floor || !n_correctable) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  unsigned long long F = 0, E = 0;
  TRY(c, stats_collect(c, &F, &E));
  *sum_floor = F; *n_correctable = E;
  return 0;
}

int bkid_shard_sd_prepare(bkid_ctx *c, double mean)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, classify_impl(c));
  return stats_prepare(c, mean);
}

int bkid_shard_sd_partial(bkid_ctx *c, double mean, int64_t t_in, int64_t *t_out)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, classify_impl(c));
  long long t = 0;
  TRY(c, stats_replay(c, mean, (long long)t_in, &t));
  *t_out = t;
  return 0;
}

int bkid_shard_set_stats(bkid_ctx *c, double mean, double sd)
{
  if (!c) return BKID_ERR_ARG;
  c->mean = mean; c->sd = sd; c->have_stats = true;
  return 0;
}

int bkid_shard_candidates(bkid_ctx *c, uint64_t index_offset, const bkid_cand **dev, int64_t *n)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, extract_candidates(c, index_offset, false));
  unsigned hnc[2] = {0, 0};
  CU(c, cudaMemcpyAsync(hnc, c->counters.as<unsigned>() + CS_NC, 8, cudaMemcpyDeviceToHost, c->st));
  TRY(c, sync_check(c));
  TRY(c, check_candidates(c, hnc));
  *dev = c->cand.as<bkid_cand>(); *n = c->n_cand;
  return 0;
}

int bkid_shard_join(bkid_ctx *c, const bkid_cand *dev_cand, int64_t n, double w, const bkid_pair **dev_pairs, int64_t *n_pairs)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  long long np = 0;
  TRY(c, join_candidates(c, dev_cand, n, w, &np));
  *dev_pairs = c->pairs_tmp.as<bkid_pair>(); *n_pairs = np;
  return 0;
}

int bkid_shard_set_pairs(bkid_ctx *c, const bkid_pair *dev_pairs, int64_t n)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, set_pairs(c, dev_pairs, n, false));
  c->tm.n_pairs = c->np0;
  c->scanned = true; c->clustered = c->refined = false;
  return 0;
}

__global__ void cluster_bucket_to_rank(bkid_cluster_rec *cl, uint32_t n, const int32_t *__restrict__ rank_of)
{
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) cl[i].bucket = rank_of[cl[i].bucket];
}

// local clusters after bkid_cluster, with `bucket` rewritten to the GLOBAL bucket-name rank
int bkid_shard_clusters(bkid_ctx *c, const bkid_cluster_rec **dev, int64_t *n)
{
  if (!c || !c->clustered) return c ? fail(c, BKID_ERR_ARG, "bkid_shard_clusters before bkid_cluster") : BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  if (c->n_clusters > 0 && !c->clusters_ranked) {
    BK_LAUNCH(cluster_bucket_to_rank, GRID1(c->n_clusters, 128), 128, 0, c->st, c->clusters.as<bkid_cluster_rec>(), (uint32_t)c->n_clusters, c->bucket_rank_of.as<int32_t>());
    c->clusters_ranked = true;
  }
  TRY(c, sync_check(c));
  *dev = c->clusters.as<bkid_cluster_rec>(); *n = c->n_clusters;
  return 0;
}

int bkid_shard_set_clusters(bkid_ctx *c, const bkid_cluster_rec *dev, int64_t n)
{
  if (!c || n < 0) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, c->clusters.ensure((size_t)(n + 1) * sizeof(bkid_cluster_rec), 0, c->st));
  if (n > 0 && dev != c->clusters.as<bkid_cluster_rec>()) CU(c, cudaMemcpyAsync(c->clusters.p, dev, (size_t)n * sizeof(bkid_cluster_rec), cudaMemcpyDeviceToDevice, c->st));
  c->n_clusters = n; c->clusters_ranked = true; c->clustered = true; c->refined = false;
  return sync_check(c);
}

int bkid_shard_sa_rows(bkid_ctx *c, const bkid_sarow **dev, int64_t *n)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, refine_build_rows(c));
  TRY(c, sync_check(c));
  *dev = (const bkid_sarow *)c->sarows.p; *n = c->n_sa;
  return 0;
}

int bkid_shard_set_sa_rows(bkid_ctx *c, const bkid_sarow *dev, int64_t n)
{
  if (!c || n < 0) return BKID_ERR_ARG;
  c->rows_ptr = dev; c->n_rows = n;
  return 0;
}

int bkid_shard_maxspan(bkid_ctx *c, int32_t *maxspan)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  int ms = 0;
  TRY(c, refine_local_maxspan(c, &ms));
  *maxspan = ms;
  return 0;
}

int bkid_shard_set_maxspan(bkid_ctx *c, int32_t maxspan) { if (!c) return BKID_ERR_ARG; c->maxspan = maxspan; return 0; }

int bkid_shard_coverage(bkid_ctx *c, double dist, uint32_t **dev_cov, int64_t *n)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, refine_coverage(c, dist));
  *dev_cov = c->cov.as<uint32_t>(); *n = 2 * c->n_clusters;
  return 0;
}

int bkid_shard_vote(bkid_ctx *c)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, refine_vote(c));
  return sync_check(c);
}

int bkid_shard_depth(bkid_ctx *c, uint32_t **dev_depth, int64_t *n)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, refine_depth(c));
  TRY(c, sync_check(c));
  *dev_depth = c->depth.as<uint32_t>(); *n = 2 * c->n_clusters;
  return 0;
}

int bkid_shard_finish(bkid_ctx *c, int64_t *n_called)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device); c->err.clear();
  TRY(c, refine_finish(c));
  c->refined = true;
  c->tm.n_called = c->n_called;
  if (n_called) *n_called = c->n_called;
  return 0;
}

int bkid_device_copy(bkid_ctx *c, void *dst, const void *src, uint64_t bytes)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  // on the context's own stream (a non-blocking stream does not order against the legacy default stream), then
  // synchronised: the copy is complete, and ordered after everything the library queued, when this returns
  if (bytes) { CU(c, cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDefault, c->st)); CU(c, cudaStreamSynchronize(c->st)); }
  return 0;
}

// row gather for the exchange routing: dst[i] = src[idx[i]], rows of row_bytes (multiple of 16), 16 bytes per thread
__global__ void gather_rows16(const uint4 *__restrict__ src, const long long *__restrict__ idx, long long n, int chunks, uint4 *__restrict__ dst)
{
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * chunks) return;
  long long r = t / chunks; int k = (int)(t - r * chunks);
  dst[t] = src[idx[r] * chunks + k];
}
int bkid_device_gather_rows(bkid_ctx *c, void *dst, const void *src, const int64_t *idx, int64_t n, int32_t row_bytes)
{
  if (!c || n < 0 || row_bytes <= 0 || (row_bytes & 15)) return c ? fail(c, BKID_ERR_ARG, "gather rows: row size must be a multiple of 16") : BKID_ERR_ARG;
  cudaSetDevice(c->device);
  if (n == 0) return 0;
  int chunks = row_bytes / 16;
  BK_LAUNCH(gather_rows16, GRID1(n * chunks, 256), 256, 0, c->st, (const uint4 *)src, (const long long *)idx, (long long)n, chunks, (uint4 *)dst);
  return sync_check(c);
}

int bkid_fetch_bucket_ranks(bkid_ctx *c, int32_t *out, int64_t cap, int64_t *nb)
{
  if (!c || !c->scanned) return c ? fail(c, BKID_ERR_ARG, "bkid_fetch_bucket_ranks before scan") : BKID_ERR_ARG;
  cudaSetDevice(c->device);
  if (nb) *nb = c->nb;
  long long k = std::min<long long>(cap, c->nb);
  if (out && k > 0) CU(c, cudaMemcpy(out, c->bucket_rank_of.p, (size_t)k * 4, cudaMemcpyDeviceToHost));
  return 0;
}

int bkid_run(bkid_ctx *c, double *mean, double *sd, double *dist, int64_t *n_called)
{
  if (!c) return BKID_ERR_ARG;
  long long l0 = g_bk_launches;
  int rc;
  cudaSetDevice(c->device);
  cudaEventRecord(c->ev_run[0], c->st);
  c->err.clear();
  // classify; then the sd pass + max span run on the side streams while the main stream does the
  // distance-independent half of the join (compaction, gather, sort by name hash, run detection)
  if ((rc = classify_impl(c)) != 0) return rc;
  if (!c->have_stats && (rc = side_launch(c)) != 0) return rc;
  double d = 0;
  int64_t ncl, ncall;
  if ((rc = scan_impl(c, &d, true)) != 0) return rc;
  if ((rc = bkid_cluster(c, d, c->prm.fast, &ncl)) != 0) return rc;
  if ((rc = bkid_refine(c, d, &ncall)) != 0) return rc;
  if (mean) *mean = c->mean;
  if (sd) *sd = c->sd;
  if (dist) *dist = d;
  if (n_called) *n_called = ncall;
  c->tm.kernel_launches = g_bk_launches - l0;
  cudaEventRecord(c->ev_run[1], c->st);
  cudaEventSynchronize(c->ev_run[1]);
  cudaEventElapsedTime(&c->tm.total, c->ev_run[0], c->ev_run[1]);          // whole step as the device saw it, host gaps included
  return 0;
}

int bkid_fetch_clusters(bkid_ctx *c, bkid_cluster_rec *out, int64_t cap, int64_t *n)
{
  if (!c || !c->refined) return c ? fail(c, BKID_ERR_ARG, "bkid_fetch_clusters before bkid_refine") : BKID_ERR_ARG;
  cudaSetDevice(c->device);
  if (n) *n = c->n_called;
  if (out && cap > 0 && c->n_called > 0) {
    long long k = std::min<long long>(cap, c->n_called);
    CU(c, cudaMemcpy(out, c->clusters_out.p, (size_t)k * sizeof(bkid_cluster_rec), cudaMemcpyDeviceToHost));
  }
  return 0;
}

__global__ void pairs_by_index(const bkid_pair *__restrict__ src, const uint32_t *__restrict__ idx, const uint32_t *__restrict__ bucket, const int32_t *__restrict__ cluster,
                               long long n, bkid_pair *__restrict__ dst)
{
  long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  bkid_pair P = src[idx[p]];
  if (bucket) P.bucket = (int32_t)bucket[p];
  if (cluster) P.cluster = cluster[p];
  dst[p] = P;
}

int bkid_fetch_pairs(bkid_ctx *c, int stage, bkid_pair *out, int64_t cap, int64_t *n)
{
  if (!c || !c->scanned) return c ? fail(c, BKID_ERR_ARG, "bkid_fetch_pairs before bkid_scan") : BKID_ERR_ARG;
  if (stage > 0 && !c->clustered) return fail(c, BKID_ERR_ARG, "stage not computed yet");
  cudaSetDevice(c->device);
  long long cnt = stage == 0 ? c->np0 : stage == 1 ? c->n1 : c->n2;
  if (n) *n = cnt;
  if (!out || cap <= 0 || cnt == 0) return 0;
  long long k = std::min<long long>(cap, cnt);
  if (stage == 0) { CU(c, cudaMemcpy(out, c->pairs0.p, (size_t)k * sizeof(bkid_pair), cudaMemcpyDeviceToHost)); return 0; }
  TRY(c, c->pairs_tmp.ensure((size_t)cnt * sizeof(bkid_pair), 0, c->st));
  if (stage == 1)
    BK_LAUNCH(pairs_by_index, GRID1(cnt, 256), 256, 0, c->st, c->pairs0.as<bkid_pair>(), c->cur1.as<uint32_t>(), c->curb1.as<uint32_t>(), (const int32_t *)nullptr, cnt, c->pairs_tmp.as<bkid_pair>());
  else
    BK_LAUNCH(pairs_by_index, GRID1(cnt, 256), 256, 0, c->st, c->pairs0.as<bkid_pair>(), c->mem_pair.as<uint32_t>(), c->mem_bucket.as<uint32_t>(), c->mem_cluster.as<int32_t>(), cnt,
              c->pairs_tmp.as<bkid_pair>());
  TRY(c, sync_check(c));
  CU(c, cudaMemcpy(out, c->pairs_tmp.p, (size_t)k * sizeof(bkid_pair), cudaMemcpyDeviceToHost));
  return 0;
}

int bkid_fetch_class(bkid_ctx *c, uint8_t *out, int64_t cap)
{
  if (!c || !c->classified) return c ? fail(c, BKID_ERR_ARG, "not classified yet") : BKID_ERR_ARG;
  cudaSetDevice(c->device);
  long long k = std::min<long long>(cap, c->n);
  if (k > 0) CU(c, cudaMemcpy(out, c->cls.p, (size_t)k, cudaMemcpyDeviceToHost));
  return 0;
}

// per-kernel device times: switch on, run, then read "name<TAB>launches<TAB>milliseconds" lines (all kernels launched
// since it was switched on, summed by name; the report resets the collection)
int bkid_profile_kernels(int on)
{
  g_bk_prof_on = on != 0;
  return 0;
}
int64_t bkid_profile_report(char *buf, int64_t cap)
{
  cudaDeviceSynchronize();
  std::map<std::string, std::pair<long long, double>> agg;
  std::vector<std::string> order;
  for (auto &r : g_prof_recs) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, r.e0, r.e1) != cudaSuccess) { cudaGetLastError(); ms = 0; }
    std::string nm = r.name;
    while (!nm.empty() && (nm.front() == '(' || nm.front() == ' ')) nm.erase(nm.begin());
    while (!nm.empty() && (nm.back() == ')' || nm.back() == ' ')) nm.pop_back();
    auto it = agg.find(nm);
    if (it == agg.end()) { order.push_back(nm); agg[nm] = {1, (double)ms}; } else { it->second.first++; it->second.second += ms; }
    g_prof_pool.push_back(r.e0); g_prof_pool.push_back(r.e1);
  }
  g_prof_recs.clear();
  std::string out;
  char line[256];
  for (auto &nm : order) { snprintf(line, sizeof line, "%s\t%lld\t%.6f\n", nm.c_str(), agg[nm].first, agg[nm].second); out += line; }
  if (buf && cap > 0) { size_t k = std::min<size_t>((size_t)cap - 1, out.size()); memcpy(buf, out.data(), k); buf[k] = 0; }
  return (int64_t)out.size() + 1;
}

int bkid_get_timings(bkid_ctx *c, bkid_timings *t)
{
  if (!c || !t) return BKID_ERR_ARG;
  *t = c->tm;
  t->kernel_launches = g_bk_launches - c->launches0;      // launches since the last bkid_reset / create
  return 0;
}

// ---- stand-alone operators ------------------------------------------------------------------
int bkid_op_sort_perm(bkid_ctx *c, int64_t n, const uint32_t *key, uint32_t *perm)
{
  if (!c || n < 0) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->err.clear();
  if (n == 0) return 0;
  cudaStream_t st = c->st;
  DBuf k, v, so;
  int rc = 0;
  if ((rc = k.ensure((size_t)n * 4 + 16, 0, st)) || (rc = v.ensure((size_t)n * 4 + 16, 0, st)) || (rc = so.ensure(16, 0, st))) return fail(c, rc, g_last_cuda_err);
  uint32_t seg[2] = {0, (uint32_t)n};
  cudaMemcpyAsync(k.p, key, (size_t)n * 4, cudaMemcpyHostToDevice, st);
  cudaMemcpyAsync(so.p, seg, 8, cudaMemcpyHostToDevice, st);
  BK_LAUNCH(iota_u32, GRID1(n, 256), 256, 0, st, v.as<uint32_t>(), (long long)n);
  rc = exact_sort_segments(c, k.as<uint32_t>(), v.as<uint32_t>(), so.as<uint32_t>(), 1, n);
  if (!rc) rc = sync_check(c);
  if (!rc) cudaMemcpy(perm, v.p, (size_t)n * 4, cudaMemcpyDeviceToHost);
  k.release(); v.release(); so.release();
  return rc;
}

static int op_setup(bkid_ctx *c, int64_t n, const uint32_t *p1, const uint32_t *p2, DBuf &x, DBuf &y, DBuf &cur, DBuf &curb, DBuf &seg)
{
  cudaStream_t st = c->st;
  size_t m = (size_t)std::max<int64_t>(n, 1) * 4 + 16;
  TRY(c, x.ensure(m, 0, st)); TRY(c, y.ensure(m, 0, st)); TRY(c, cur.ensure(m, 0, st)); TRY(c, curb.ensure(m, 0, st)); TRY(c, seg.ensure(16, 0, st));
  TRY(c, c->counters.ensure(1024, 0, st));
  uint32_t so[2] = {0, (uint32_t)n};
  if (n > 0) {
    CU(c, cudaMemcpyAsync(x.p, p1, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CU(c, cudaMemcpyAsync(y.p, p2, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    BK_LAUNCH(iota_u32, GRID1(n, 256), 256, 0, st, cur.as<uint32_t>(), (long long)n);
    CU(c, cudaMemsetAsync(curb.p, 0, (size_t)n * 4, st));
  }
  CU(c, cudaMemcpyAsync(seg.p, so, 8, cudaMemcpyHostToDevice, st));
  return sync_check(c);
}

int bkid_op_remove_isolated(bkid_ctx *c, int64_t n, const uint32_t *p1, const uint32_t *p2, double w, uint32_t *out_idx, int64_t *n_out)
{
  if (!c || n < 0) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->err.clear();
  DBuf x, y, cur, curb, seg;
  int rc = op_setup(c, n, p1, p2, x, y, cur, curb, seg);
  if (!rc) rc = remove_isolated_all(c, cur.as<uint32_t>(), curb.as<uint32_t>(), seg.as<uint32_t>(), n, 1, x.as<uint32_t>(), y.as<uint32_t>(), w);
  if (!rc) rc = sync_check(c);
  if (!rc) {
    *n_out = c->n1;
    if (c->n1 > 0) cudaMemcpy(out_idx, c->cur1.p, (size_t)c->n1 * 4, cudaMemcpyDeviceToHost);
  }
  for (DBuf *b : {&x, &y, &cur, &curb, &seg}) b->release();
  return rc;
}

int bkid_op_cluster(bkid_ctx *c, int mode, int64_t n, const uint32_t *p1, const uint32_t *p2, double thr, uint32_t *out_idx, int32_t *out_cluster, int64_t *n_out,
                    int32_t *n_roots)
{
  if (!c || n < 0) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->err.clear();
  DBuf x, y, cur, curb, seg;
  int rc = op_setup(c, n, p1, p2, x, y, cur, curb, seg);
  if (!rc) rc = mode ? cluster_fast(c, cur.as<uint32_t>(), curb.as<uint32_t>(), seg.as<uint32_t>(), n, 1, x.as<uint32_t>(), y.as<uint32_t>(), thr, n)
                     : cluster_ahc(c, cur.as<uint32_t>(), curb.as<uint32_t>(), seg.as<uint32_t>(), n, 1, x.as<uint32_t>(), y.as<uint32_t>(), thr);
  if (!rc) rc = sync_check(c);
  if (!rc) {
    *n_out = c->n2;
    if (n_roots) *n_roots = c->roots_per_bucket.empty() ? 0 : c->roots_per_bucket[0];
    if (c->n2 > 0) {
      cudaMemcpy(out_idx, c->mem_pair.p, (size_t)c->n2 * 4, cudaMemcpyDeviceToHost);
      cudaMemcpy(out_cluster, c->mem_cluster.p, (size_t)c->n2 * 4, cudaMemcpyDeviceToHost);
    }
  }
  for (DBuf *b : {&x, &y, &cur, &curb, &seg}) b->release();
  return rc;
}


// K6 on a caller-built member list: pairs of ONE chr-pair bucket with their cluster ids (grouped by cluster id, as after the
// reference's sort by cmp_enspan_id, src/BreakID.cc:141).  Leaves the summaries in the context as bkid_cluster does, so
// bkid_refine / bkid_fetch_clusters follow.  The records' `bucket` is the pairs' own.
int bkid_op_summarize(bkid_ctx *c, int64_t n, const bkid_pair *pairs, double dist, int64_t *n_clusters)
{
  if (!c || n < 0 || (n > 0 && !pairs)) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->err.clear();
  cudaStream_t st = c->st;
  size_t m = (size_t)std::max<int64_t>(n, 1);
  TRY(c, c->pairs0.ensure(m * sizeof(bkid_pair), 0, st));
  TRY(c, c->mem_pair.ensure(m * 4 + 16, 0, st)); TRY(c, c->mem_bucket.ensure(m * 4 + 16, 0, st)); TRY(c, c->mem_cluster.ensure(m * 4 + 16, 0, st));
  TRY(c, c->counters.ensure(1024, 0, st));
  std::vector<int32_t> cl((size_t)n);
  for (int64_t i = 0; i < n; ++i) {
    cl[(size_t)i] = pairs[i].cluster;
    if (i > 0 && pairs[i].cluster < pairs[i - 1].cluster) return fail(c, BKID_ERR_ARG, "bkid_op_summarize: pairs are not grouped by ascending cluster id");
  }
  c->n2 = n; c->n_clusters = 0;
  if (n > 0) {
    CU(c, cudaMemcpyAsync(c->pairs0.p, pairs, (size_t)n * sizeof(bkid_pair), cudaMemcpyHostToDevice, st));
    CU(c, cudaMemcpyAsync(c->mem_cluster.p, cl.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CU(c, cudaMemsetAsync(c->mem_bucket.p, 0, (size_t)n * 4, st));
    BK_LAUNCH(iota_u32, GRID1(n, 256), 256, 0, st, c->mem_pair.as<uint32_t>(), (long long)n);
    TRY(c, sync_check(c));                                   // `cl` and the caller's pairs are pageable: copies done before return
  }
  TRY(c, summarize_impl(c, dist));
  TRY(c, sync_check(c));
  c->clustered = true; c->clusters_ranked = true; c->refined = false;
  c->tm.n_clusters = c->n_clusters;
  if (n_clusters) *n_clusters = c->n_clusters;
  return 0;
}

// thresholds of the NEXT stage calls (qual, times, min_reads, bp_pos_error, mismatch_num, sd_mult, validate_align, fast);
// pairs and clusters derived from the old ones are dropped (and the classification, if qual changed); the records stay
int bkid_set_params(bkid_ctx *c, const bkid_params *p)
{
  if (!c || !p) return BKID_ERR_ARG;
  if (p->times < 1 || p->min_reads < 1 || p->qual < 0) return fail(c, BKID_ERR_ARG, "bad parameters");
  cudaSetDevice(c->device);
  if (p->qual != c->prm.qual) invalidate(c);               // the class bytes depend on the MAPQ threshold
  else c->scanned = c->clustered = c->refined = false;
  c->prm = *p;
  return 0;
}

}  // extern "C"
