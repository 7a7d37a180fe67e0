// bkid_sort.cuh -- bkid_sort_records: the records a context holds into coordinate order on the device.  Included by
// bkid_core.cu after bkid_api.cuh (context, fail / CU / TRY, set_ptrs, invalidate).
//
//   sort_check      one pass over tid / pos: argument errors, "already non-decreasing in (tid as uint32, pos)", max pos + 1
//   sort_keys       key = (tid as uint32, pos + 1, flag & BAM_FREVERSE) packed into the fewest bits the batch needs
//                   (tid -1 -> n_targets, the largest rank), value = push index; then ONE onesweep sort (prims.cuh), so the
//                   launch count does not depend on the number of targets
//   sort_pack       the remaining narrow fields of a record into one 8-byte row (16 bytes when a column is held wide), so
//                   the random gather reads one sector per record instead of one per column
//   sort_unpack     new record i <- row[perm[i]]; tid / pos are decoded from the sorted key
//   sparse / SA     a per-record slot map (old record -> sparse row / SA row), flags in the new order, an exclusive scan per
//                   table, rows re-emitted in ascending new record index; SA segments re-laid out one warp per row
// n >= 2^30 (the onesweep limit): targets are cut into consecutive groups of < 2^30 records, the records are stably
// partitioned by group (one flag pass + scan per group, 64-bit group offsets) and every group is sorted with the full key.
#pragma once

constexpr long long SORT_GROUP_LIMIT = 1ll << 30;

static inline int bits_for(unsigned long long x) { int b = 0; while (b < 64 && (1ull << b) <= x) ++b; return b; }

__device__ __forceinline__ uint32_t sort_tid_rank(int32_t tid, int nt) { return tid < 0 ? (uint32_t)nt : (uint32_t)tid; }

__device__ __forceinline__ uint64_t sort_key(int32_t tid, int32_t pos, uint16_t flag, int nt, int pbits)
{
  return ((uint64_t)sort_tid_rank(tid, nt) << pbits) | ((uint64_t)((uint32_t)pos + 1u) << 1) | (uint64_t)((flag >> 4) & 1u);
}

// out[0] = records with tid outside [-1, nt) or pos < -1, out[1] = descents in (tid as uint32, pos), out[2] = max (pos + 1)
__global__ void sort_check(const int32_t *__restrict__ tid, const int32_t *__restrict__ pos, long long n, int nt, unsigned long long *__restrict__ out)
{
  unsigned long long bad = 0, desc = 0, mx = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    int32_t t = tid[i], p = pos[i];
    if (t < -1 || t >= nt || p < -1) ++bad;
    unsigned long long p1 = (unsigned long long)((uint32_t)p + 1u);
    if (p >= -1 && p1 > mx) mx = p1;
    if (i > 0) {
      uint32_t ta = (uint32_t)tid[i - 1], tb = (uint32_t)t;
      if (ta > tb || (ta == tb && pos[i - 1] > p)) ++desc;
    }
  }
  bad = bk::warp_sum(bad); desc = bk::warp_sum(desc);
  for (int o = 16; o; o >>= 1) { unsigned long long u = __shfl_xor_sync(0xffffffffu, mx, o); mx = u > mx ? u : mx; }
  if (bk::lane_id() == 0) {
    if (bad) atomicAdd(&out[0], bad);
    if (desc) atomicAdd(&out[1], desc);
    if (mx) atomicMax(&out[2], mx);
  }
}

// records per target rank (tid -1 = rank nt); warp-aggregated because sorted runs hit one bin
__global__ void sort_tid_hist(const int32_t *__restrict__ tid, long long n, int nt, unsigned long long *__restrict__ h)
{
  for (long long b = (long long)blockIdx.x * blockDim.x; b < n; b += (long long)gridDim.x * blockDim.x) {
    long long i = b + threadIdx.x;
    unsigned r = i < n ? sort_tid_rank(tid[i], nt) : 0xffffffffu;
    unsigned m = __match_any_sync(0xffffffffu, r);
    if (r != 0xffffffffu && (int)bk::lane_id() == __ffs(m) - 1) atomicAdd(&h[r], (unsigned long long)__popc(m));
  }
}

// flag[i] = record i belongs to group g
__global__ void sort_group_flag(const int32_t *__restrict__ tid, long long n, int nt, const int32_t *__restrict__ group_of, int g, uint8_t *__restrict__ flag)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flag[i] = group_of[sort_tid_rank(tid[i], nt)] == g;
}

// keys and push indices; with `slot` only the records of group g, at their stable slot inside the group
__global__ void sort_keys(const int32_t *__restrict__ tid, const int32_t *__restrict__ pos, const uint16_t *__restrict__ flag, long long n, int nt, int pbits,
                          const uint8_t *__restrict__ in_group, const uint32_t *__restrict__ slot, uint64_t *__restrict__ key, uint32_t *__restrict__ val)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (in_group && !in_group[i]) return;
  long long k = slot ? (long long)slot[i] : i;
  key[k] = sort_key(tid[i], pos[i], flag[i], nt, pbits);
  val[k] = (uint32_t)i;
}

// the row of one record: flag | mapq | isize | span (8 B when both are narrow, else 16 B with the wide values)
struct SortSrc {
  const uint16_t *flag; const uint8_t *mapq; const int32_t *isize; const int16_t *isize16; const int32_t *endpos; const uint16_t *span16;
};
struct SortDst {
  uint16_t *flag; uint8_t *mapq; int32_t *tid, *pos, *isize; int16_t *isize16; int32_t *endpos; uint16_t *span16;
};

__global__ void sort_pack8(SortSrc s, long long n, uint64_t *__restrict__ row)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  row[i] = (uint64_t)s.flag[i] | ((uint64_t)s.mapq[i] << 16) | ((uint64_t)(uint16_t)s.isize16[i] << 24) | ((uint64_t)s.span16[i] << 40);
}

__global__ void sort_pack16(SortSrc s, long long n, uint4 *__restrict__ row)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint4 r;
  r.x = (uint32_t)s.flag[i] | ((uint32_t)s.mapq[i] << 16);
  r.y = s.isize ? (uint32_t)s.isize[i] : (uint32_t)(int32_t)s.isize16[i];
  r.z = s.endpos ? (uint32_t)s.endpos[i] : (uint32_t)s.span16[i];
  r.w = 0;
  row[i] = r;
}

__device__ __forceinline__ void sort_decode(uint64_t k, int nt, int pbits, int32_t &tid, int32_t &pos)
{
  uint32_t t = (uint32_t)(k >> pbits);
  tid = t == (uint32_t)nt ? -1 : (int32_t)t;
  pos = (int32_t)((uint32_t)((k >> 1) & ((1ull << (pbits - 1)) - 1)) - 1u);
}

__global__ void sort_unpack8(const uint64_t *__restrict__ key, const uint32_t *__restrict__ perm, const uint64_t *__restrict__ row, long long n, int nt, int pbits, SortDst d)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t t, p;
  sort_decode(key[i], nt, pbits, t, p);
  uint64_t r = row[perm[i]];
  d.tid[i] = t; d.pos[i] = p;
  d.flag[i] = (uint16_t)r; d.mapq[i] = (uint8_t)(r >> 16); d.isize16[i] = (int16_t)(uint16_t)(r >> 24); d.span16[i] = (uint16_t)(r >> 40);
}

__global__ void sort_unpack16(const uint64_t *__restrict__ key, const uint32_t *__restrict__ perm, const uint4 *__restrict__ row, long long n, int nt, int pbits, SortDst d)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t t, p;
  sort_decode(key[i], nt, pbits, t, p);
  uint4 r = row[perm[i]];
  d.tid[i] = t; d.pos[i] = p;
  d.flag[i] = (uint16_t)r.x; d.mapq[i] = (uint8_t)(r.x >> 16);
  if (d.isize) d.isize[i] = (int32_t)r.y; else d.isize16[i] = (int16_t)r.y;
  if (d.endpos) d.endpos[i] = (int32_t)r.z; else d.span16[i] = (uint16_t)r.z;
}

// slot map: slot[rec[j]] = j + 1
__global__ void sort_slot_scatter(const uint32_t *__restrict__ rec, long long m, uint32_t *__restrict__ slot)
{
  long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < m) slot[rec[j]] = (uint32_t)j + 1u;
}

// flags of the new record order: record perm[i] has a sparse row / an SA row
__global__ void sort_slot_flags(const uint32_t *__restrict__ perm, long long n, const uint32_t *__restrict__ slot_x, const uint32_t *__restrict__ slot_sa,
                                uint8_t *__restrict__ fx, uint8_t *__restrict__ fsa)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t o = perm[i];
  if (slot_x) fx[i] = slot_x[o] != 0;
  if (slot_sa) fsa[i] = slot_sa[o] != 0;
}

// new row k = off[i] of every flagged new record i: its new record index and the old row it comes from
__global__ void sort_emit_rows(const uint32_t *__restrict__ perm, long long n, const uint8_t *__restrict__ f, const uint32_t *__restrict__ off,
                               const uint32_t *__restrict__ slot, uint32_t *__restrict__ new_rec, uint32_t *__restrict__ src_row)
{
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !f[i]) return;
  uint32_t k = off[i];
  new_rec[k] = (uint32_t)i;
  src_row[k] = slot[perm[i]] - 1u;
}

__global__ void sort_gather_x(const uint32_t *__restrict__ src, long long m, const int32_t *__restrict__ mtid, const int32_t *__restrict__ mpos, const uint64_t *__restrict__ nh,
                              int32_t *__restrict__ o_mtid, int32_t *__restrict__ o_mpos, uint64_t *__restrict__ o_nh)
{
  long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= m) return;
  uint32_t j = src[k];
  o_mtid[k] = mtid[j]; o_mpos[k] = mpos[j];
  o_nh[2 * k] = nh[2 * (size_t)j]; o_nh[2 * k + 1] = nh[2 * (size_t)j + 1];
}

// segment lengths of SA row src[k] in the new order (entry m = 0 so that the exclusive scan ends in the total)
struct SaSegs { const uint32_t *off[4]; uint32_t *len[4]; uint32_t *noff[4]; const uint8_t *src[4]; uint8_t *dst[4]; int unit[4]; int k; };

__global__ void sort_sa_lens(const uint32_t *__restrict__ src, long long m, const int32_t *__restrict__ seq_len, int32_t *__restrict__ o_seq_len, SaSegs s)
{
  long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k > m) return;
  for (int q = 0; q < s.k; ++q) s.len[q][k] = k < m ? s.off[q][src[k] + 1] - s.off[q][src[k]] : 0u;
  if (k < m && seq_len) o_seq_len[k] = seq_len[src[k]];
}

// one warp per SA row: every segment kind of the row, copied in units of 4 bytes (cig_ops) or 1 byte
__global__ void sort_sa_copy(const uint32_t *__restrict__ src, long long m, SaSegs s)
{
  long long k = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= m) return;
  unsigned l = bk::lane_id();
  uint32_t j = src[k];
  for (int q = 0; q < s.k; ++q) {
    uint32_t a = s.off[q][j], len = s.off[q][j + 1] - a, b = s.noff[q][k];
    if (s.unit[q] == 4) {
      const uint32_t *in = (const uint32_t *)s.src[q] + a; uint32_t *out = (uint32_t *)s.dst[q] + b;
      for (uint32_t t = l; t < len; t += 32) out[t] = in[t];
    } else {
      const uint8_t *in = s.src[q] + a; uint8_t *out = s.dst[q] + b;
      for (uint32_t t = l; t < len; t += 32) out[t] = in[t];
    }
  }
}

extern "C" {

int bkid_sort_records(bkid_ctx *c, int32_t *was_sorted)
{
  if (!c) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  cudaStream_t st = c->st;
  const long long n = c->n, nx = c->n_x, ns = c->n_sa;
  const int nt = c->nt;
  if (n == 0) { invalidate(c); if (was_sorted) *was_sorted = 1; return 0; }

  // ---- 1. validate + already sorted? (nothing is written before this returns) ----
  unsigned long long *chk = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);     // scratch of the scans, free here
  unsigned long long h[3] = {0, 0, 0};
  CU(c, cudaMemsetAsync(chk, 0, 24, st));
  int grid = (int)std::min<long long>(div_up(n, 256), (long long)c->n_sm * 16);
  BK_LAUNCH(sort_check, grid, 256, 0, st, c->p_tid, c->p_pos, n, nt, chk);
  CU(c, cudaMemcpyAsync(h, chk, 24, cudaMemcpyDeviceToHost, st));
  TRY(c, sync_check(c));
  if (h[0]) return fail(c, BKID_ERR_ARG, "bkid_sort_records: a record has tid outside [-1, n_targets) or pos < -1");
  if (h[1] == 0) { invalidate(c); if (was_sorted) *was_sorted = 1; return 0; }

  const int pbits = bits_for(h[2]) + 1, kbits = bits_for((unsigned long long)nt) + pbits;
  // ---- 2. groups of targets (only when n >= 2^30) ----
  std::vector<int32_t> group_of(nt + 1, 0);
  std::vector<long long> goff(1, 0);
  if (n >= SORT_GROUP_LIMIT) {
    TRY(c, c->tmpD.ensure((size_t)(nt + 1) * 8 + 64, 0, st));
    unsigned long long *dh = c->tmpD.as<unsigned long long>();
    CU(c, cudaMemsetAsync(dh, 0, (size_t)(nt + 1) * 8, st));
    BK_LAUNCH(sort_tid_hist, grid, 256, 0, st, c->p_tid, n, nt, dh);
    std::vector<unsigned long long> cnt(nt + 1);
    CU(c, cudaMemcpyAsync(cnt.data(), dh, (size_t)(nt + 1) * 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    long long cur = 0;
    for (int t = 0; t <= nt; ++t) {
      if ((long long)cnt[t] >= SORT_GROUP_LIMIT) return fail(c, BKID_ERR_ARG, "bkid_sort_records: one target holds 2^30 records or more");
      if (cur + (long long)cnt[t] >= SORT_GROUP_LIMIT) { goff.push_back(goff.back() + cur); cur = 0; }
      cur += (long long)cnt[t];
      group_of[t] = (int32_t)goff.size() - 1;
    }
    goff.push_back(goff.back() + cur);
  } else goff.push_back(n);
  const int ngroups = (int)goff.size() - 1;
  long long gmax = 0;
  for (int g = 0; g < ngroups; ++g) gmax = std::max(gmax, goff[g + 1] - goff[g]);

  // ---- 3. every allocation before the first column is overwritten ----
  const bool row8 = c->form_isize == 2 && c->form_span == 2;
  const size_t un = (size_t)n;
  TRY(c, c->sc.keys.ensure(un * 8, 0, st)); TRY(c, c->sc.vals.ensure(un * 4, 0, st));
  TRY(c, c->sc.keys_alt.ensure((size_t)std::max<long long>(gmax, 1) * 8, 0, st)); TRY(c, c->sc.vals_alt.ensure((size_t)std::max<long long>(gmax, 1) * 4, 0, st));
  TRY(c, c->sc.hist.ensure(bk::radix_hist_elems(gmax) * 4, 0, st));
  TRY(c, c->sc.scan_tmp.ensure((bk::scan_tmp_elems(n) + 8) * 8, 0, st));
  TRY(c, c->tmpA.ensure(un * (row8 ? 8 : 16) + 64, 0, st));
  // per record: slot maps (x, sa) 8 B, flags 2 B, offsets 8 B (the group pass uses the first flag / offset arrays before)
  const bool side = nx > 0 || ns > 0;
  size_t per = side || ngroups > 1 ? un * 18 + 256 : 64;
  TRY(c, c->tmpC.ensure(per, 0, st));
  // side tables in their new order
  uint32_t tot_h[4] = {0, 0, 0, 0};               // cig ops, sa bytes, oc bytes, seq bytes
  const bool seq = c->have_seq && ns > 0;
  if (ns) {
    CU(c, cudaMemcpyAsync(&tot_h[0], c->p_cig_off + ns, 4, cudaMemcpyDeviceToHost, st));
    CU(c, cudaMemcpyAsync(&tot_h[1], c->p_sa_off + ns, 4, cudaMemcpyDeviceToHost, st));
    CU(c, cudaMemcpyAsync(&tot_h[2], c->p_oc_off + ns, 4, cudaMemcpyDeviceToHost, st));
    if (seq) CU(c, cudaMemcpyAsync(&tot_h[3], c->p_seq_off + ns, 4, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
  }
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  size_t side_b = al((size_t)nx * 4) * 4 + al((size_t)nx * 16) + al((size_t)ns * 4) * 3 + al((size_t)(ns + 1) * 4) * 8 + al((size_t)tot_h[0] * 4) +
                  al(tot_h[1]) + al(tot_h[2]) + al(tot_h[3]) + 256;
  if (side) TRY(c, c->tmpB.ensure(side_b, 0, st));
  const bool own = c->borrowed;                   // borrowed device columns: the sorted records go to owned copies
  if (own) {
    TRY(c, c->flag.ensure(un * 2 + 64, 0, st)); TRY(c, c->mapq.ensure(un + 64, 0, st));
    TRY(c, c->tid.ensure(un * 4 + 64, 0, st)); TRY(c, c->pos.ensure(un * 4 + 64, 0, st));
    if (c->form_isize == 1) TRY(c, c->isize.ensure(un * 4 + 64, 0, st)); else TRY(c, c->isize16.ensure(un * 2 + 64, 0, st));
    if (c->form_span == 1) TRY(c, c->endpos.ensure(un * 4 + 64, 0, st)); else TRY(c, c->span16.ensure(un * 2 + 64, 0, st));
    TRY(c, c->x_rec.ensure((size_t)nx * 4 + 64, 0, st)); TRY(c, c->x_mtid.ensure((size_t)nx * 4 + 64, 0, st));
    TRY(c, c->x_mpos.ensure((size_t)nx * 4 + 64, 0, st)); TRY(c, c->x_nh.ensure((size_t)nx * 16 + 64, 0, st));
    TRY(c, c->sa_rec.ensure((size_t)ns * 4 + 64, 0, st));
    TRY(c, c->cig_off.ensure((size_t)(ns + 1) * 4 + 64, 0, st)); TRY(c, c->sa_off.ensure((size_t)(ns + 1) * 4 + 64, 0, st));
    TRY(c, c->oc_off.ensure((size_t)(ns + 1) * 4 + 64, 0, st));
    TRY(c, c->cig_ops.ensure((size_t)tot_h[0] * 4 + 64, 0, st)); TRY(c, c->sa_txt.ensure((size_t)tot_h[1] + 64, 0, st));
    TRY(c, c->oc_txt.ensure((size_t)tot_h[2] + 64, 0, st));
    if (seq) {
      TRY(c, c->seq_off.ensure((size_t)(ns + 1) * 4 + 64, 0, st)); TRY(c, c->seq_len.ensure((size_t)ns * 4 + 64, 0, st));
      TRY(c, c->seq4.ensure((size_t)tot_h[3] + 64, 0, st));
    }
  }
  invalidate(c);

  // ---- 4. keys, one stable sort per group ----
  uint64_t *K = c->sc.keys.as<uint64_t>();
  uint32_t *V = c->sc.vals.as<uint32_t>();
  char *pc = (char *)c->tmpC.p;
  uint32_t *slot_x = (uint32_t *)pc, *slot_sa = slot_x + un, *off_x = slot_sa + un, *off_sa = off_x + un;
  uint8_t *fx = (uint8_t *)(off_sa + un), *fsa = fx + un;
  unsigned long long *stmp = c->sc.scan_tmp.as<unsigned long long>();
  const bk::RadixTmp rt{c->sc.keys_alt.as<uint64_t>(), c->sc.vals_alt.as<uint32_t>(), c->sc.hist.as<uint32_t>(), stmp};
  if (ngroups == 1) BK_LAUNCH(sort_keys, GRID1(n, 256), 256, 0, st, c->p_tid, c->p_pos, c->p_flag, n, nt, pbits, nullptr, nullptr, K, V);
  else {
    TRY(c, c->tmpD.ensure((size_t)(nt + 1) * 4 + 64, 0, st));
    CU(c, cudaMemcpyAsync(c->tmpD.p, group_of.data(), (size_t)(nt + 1) * 4, cudaMemcpyHostToDevice, st));
    for (int g = 0; g < ngroups; ++g) {
      BK_LAUNCH(sort_group_flag, GRID1(n, 256), 256, 0, st, c->p_tid, n, nt, c->tmpD.as<int32_t>(), g, fx);
      bk::exclusive_scan<uint8_t, uint32_t>(fx, off_x, n, stmp, nullptr, st);
      BK_LAUNCH(sort_keys, GRID1(n, 256), 256, 0, st, c->p_tid, c->p_pos, c->p_flag, n, nt, pbits, fx, off_x, K + goff[g], V + goff[g]);
    }
  }
  for (int g = 0; g < ngroups; ++g)
    if (bk::radix_sort_pairs(K + goff[g], V + goff[g], goff[g + 1] - goff[g], 0, kbits, rt, st) < 0)
      return fail(c, BKID_ERR_CUDA, "bkid_sort_records: group of 2^30 records or more");

  // ---- 5. dense columns: pack, gather ----
  SortSrc src{c->p_flag, c->p_mapq, c->p_isize, c->p_isize16, c->p_endpos, c->p_span16};
  if (row8) BK_LAUNCH(sort_pack8, GRID1(n, 256), 256, 0, st, src, n, c->tmpA.as<uint64_t>());
  else BK_LAUNCH(sort_pack16, GRID1(n, 256), 256, 0, st, src, n, c->tmpA.as<uint4>());

  // ---- 6. sparse and SA rows in the new order (reads the old x_rec / sa_rec: before any side column is written) ----
  uint32_t *xs_rec = nullptr, *xs_src = nullptr, *sa_new = nullptr, *sa_src = nullptr;
  char *pb = (char *)c->tmpB.p;
  auto take = [&](size_t b) { char *r = pb; pb += al(b); return r; };
  if (side) {
    CU(c, cudaMemsetAsync(slot_x, 0, un * 8, st));
    if (nx) BK_LAUNCH(sort_slot_scatter, GRID1(nx, 256), 256, 0, st, c->p_x_rec, nx, slot_x);
    if (ns) BK_LAUNCH(sort_slot_scatter, GRID1(ns, 256), 256, 0, st, c->p_sa_rec, ns, slot_sa);
    BK_LAUNCH(sort_slot_flags, GRID1(n, 256), 256, 0, st, V, n, nx ? slot_x : nullptr, ns ? slot_sa : nullptr, fx, fsa);
    if (nx) {
      bk::exclusive_scan<uint8_t, uint32_t>(fx, off_x, n, stmp, nullptr, st);
      xs_rec = (uint32_t *)take((size_t)nx * 4); xs_src = (uint32_t *)take((size_t)nx * 4);
      BK_LAUNCH(sort_emit_rows, GRID1(n, 256), 256, 0, st, V, n, fx, off_x, slot_x, xs_rec, xs_src);
    }
    if (ns) {
      bk::exclusive_scan<uint8_t, uint32_t>(fsa, off_sa, n, stmp, nullptr, st);
      sa_new = (uint32_t *)take((size_t)ns * 4); sa_src = (uint32_t *)take((size_t)ns * 4);
      BK_LAUNCH(sort_emit_rows, GRID1(n, 256), 256, 0, st, V, n, fsa, off_sa, slot_sa, sa_new, sa_src);
    }
  }
  int32_t *x_mtid = nullptr, *x_mpos = nullptr; uint64_t *x_nh = nullptr;
  if (nx) {
    x_mtid = (int32_t *)take((size_t)nx * 4); x_mpos = (int32_t *)take((size_t)nx * 4); x_nh = (uint64_t *)take((size_t)nx * 16);
    BK_LAUNCH(sort_gather_x, GRID1(nx, 256), 256, 0, st, xs_src, nx, c->p_x_mtid, c->p_x_mpos, c->p_x_nh, x_mtid, x_mpos, x_nh);
  }
  SaSegs sg{};
  int32_t *seq_len = nullptr;
  if (ns) {
    const uint32_t *offs[4] = {c->p_cig_off, c->p_sa_off, c->p_oc_off, c->p_seq_off};
    const uint8_t *srcs[4] = {(const uint8_t *)c->p_cig_ops, c->p_sa_txt, c->p_oc_txt, c->p_seq4};
    sg.k = seq ? 4 : 3;
    for (int q = 0; q < sg.k; ++q) {
      sg.off[q] = offs[q]; sg.src[q] = srcs[q]; sg.unit[q] = q == 0 ? 4 : 1;
      sg.len[q] = (uint32_t *)take((size_t)(ns + 1) * 4); sg.noff[q] = (uint32_t *)take((size_t)(ns + 1) * 4);
      sg.dst[q] = (uint8_t *)take((size_t)tot_h[q] * sg.unit[q]);
    }
    seq_len = (int32_t *)take((size_t)ns * 4);
    BK_LAUNCH(sort_sa_lens, GRID1(ns + 1, 256), 256, 0, st, sa_src, ns, seq ? c->p_seq_len : nullptr, seq_len, sg);
    for (int q = 0; q < sg.k; ++q) bk::exclusive_scan<uint32_t, uint32_t>(sg.len[q], sg.noff[q], ns + 1, stmp, nullptr, st);
    BK_LAUNCH(sort_sa_copy, GRID1((ns) * 32, 256), 256, 0, st, sa_src, ns, sg);
  }

  // ---- 7. write the context's columns (first write to record data) ----
  SortDst dst{c->flag.as<uint16_t>(), c->mapq.as<uint8_t>(), c->tid.as<int32_t>(), c->pos.as<int32_t>(),
              c->form_isize == 1 ? c->isize.as<int32_t>() : nullptr, c->form_isize == 2 ? c->isize16.as<int16_t>() : nullptr,
              c->form_span == 1 ? c->endpos.as<int32_t>() : nullptr, c->form_span == 2 ? c->span16.as<uint16_t>() : nullptr};
  if (row8) BK_LAUNCH(sort_unpack8, GRID1(n, 256), 256, 0, st, K, V, c->tmpA.as<uint64_t>(), n, nt, pbits, dst);
  else BK_LAUNCH(sort_unpack16, GRID1(n, 256), 256, 0, st, K, V, c->tmpA.as<uint4>(), n, nt, pbits, dst);
  if (nx) {
    CU(c, cudaMemcpyAsync(c->x_rec.p, xs_rec, (size_t)nx * 4, cudaMemcpyDeviceToDevice, st));
    CU(c, cudaMemcpyAsync(c->x_mtid.p, x_mtid, (size_t)nx * 4, cudaMemcpyDeviceToDevice, st));
    CU(c, cudaMemcpyAsync(c->x_mpos.p, x_mpos, (size_t)nx * 4, cudaMemcpyDeviceToDevice, st));
    CU(c, cudaMemcpyAsync(c->x_nh.p, x_nh, (size_t)nx * 16, cudaMemcpyDeviceToDevice, st));
  }
  if (ns) {
    CU(c, cudaMemcpyAsync(c->sa_rec.p, sa_new, (size_t)ns * 4, cudaMemcpyDeviceToDevice, st));
    DBuf *offb[4] = {&c->cig_off, &c->sa_off, &c->oc_off, &c->seq_off}, *datb[4] = {&c->cig_ops, &c->sa_txt, &c->oc_txt, &c->seq4};
    for (int q = 0; q < sg.k; ++q) {
      CU(c, cudaMemcpyAsync(offb[q]->p, sg.noff[q], (size_t)(ns + 1) * 4, cudaMemcpyDeviceToDevice, st));
      if (tot_h[q]) CU(c, cudaMemcpyAsync(datb[q]->p, sg.dst[q], (size_t)tot_h[q] * sg.unit[q], cudaMemcpyDeviceToDevice, st));
    }
    if (seq) CU(c, cudaMemcpyAsync(c->seq_len.p, seq_len, (size_t)ns * 4, cudaMemcpyDeviceToDevice, st));
  }
  if (own) {
    c->borrowed = false;
    c->n_cig = tot_h[0]; c->sa_bytes = tot_h[1]; c->oc_bytes = tot_h[2]; c->seq_bytes = tot_h[3];
    c->have_seq = seq;
    if (ns == 0) { CU(c, cudaMemsetAsync(c->cig_off.p, 0, 4, st)); CU(c, cudaMemsetAsync(c->sa_off.p, 0, 4, st)); CU(c, cudaMemsetAsync(c->oc_off.p, 0, 4, st)); }
  }
  set_ptrs(c);
  TRY(c, sync_check(c));
  if (was_sorted) *was_sorted = 0;
  return 0;
}

}  // extern "C"
