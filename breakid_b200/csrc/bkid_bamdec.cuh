// bkid_bamdec.cuh -- BGZF inflate + BAM record decode on the device (SURVEY.md 8 f-1).  Included by bkid_core.cu.
//
// Replaces, as the producer of records for the hot path, htslib's bgzf_read_block / inflate_block
// (htslib-1.3.1/bgzf.c:545-600,388-419) and bam_read1 (sam.c:407-441) driven by the samread / sam_read1 loops of
// src/BreakID.cc:1414,1929, plus bam_endpos (sam.c:344-350) and bam_aux_get (sam.c:1267-1290) for SA:Z / OC:Z.
// The host only walks the BGZF block headers (BSIZE / ISIZE) and parses the BAM header; compressed bytes go to
// the GPU as they are in the file.
//
//   bgzf_inflate      groups of 8 lanes, one BGZF block each, four groups per warp in lock step (bkid_inflate.cuh);
//                     4 warps per CTA, 2.3 KB of Huffman tables per group in shared memory
//   bam_seed          record boundaries are a serial chain (each record starts where the previous one ends); the
//                     uncompressed chunk is cut into 256 KiB segments and every segment gets a SEED: the first
//                     offset that passes a strong record-header predicate three records deep
//   bam_walk          one thread per segment follows the chain from its seed to the next seed
//   bam_stitch        a chain is accepted only if the previous segment's walk lands EXACTLY on the seed (induction
//                     from the known first record); a seed that is not hit is dropped and the walk repeated, so
//                     a false-positive seed can cost time but never correctness
//   bam_extract_cols  one thread per record: dense columns + per-record sizes of its sparse / SA table entries
//   bam_extract_side  after the scans: sparse mate/name table, SA side table (cigar ops, SA / OC text)
//
// Chunks of <= 1.5 GiB compressed / 3 GiB uncompressed (~48k BGZF blocks: several waves of the inflate grid) stream
// through double-buffered staging, so a whole-genome
// BAM (uncompressed 200+ GB) never has to be resident: only the 19 B/record columns stay.
#pragma once
#include "bkid_inflate.cuh"

namespace bamdec {

constexpr uint32_t SEG = 256u << 10;
constexpr uint32_t NONE = 0xffffffffu;
constexpr int INF_LITMAX = 4;         // literals per lane and step
constexpr int INF_STEPS = 8;          // lane steps between two rounds of block fetch / header scheduling
constexpr int INF_HBATCH = 6;         // a block header is parsed once this many lanes of the warp wait for one ...
constexpr int INF_HWAIT = 24;         // ... or a lane has waited this many rounds (the parse is a long divergent section)
constexpr int INF_CTAS_PER_SM = 5;    // 44 KB of tables per warp

struct Task { uint64_t src; uint32_t dst; uint32_t clen, ulen; };

// One warp per CTA, one BGZF block per LANE (bkid_inflate.cuh): every lane fetches its blocks from a global queue and
// runs its own decoder; the warp executes the union of the lanes' paths.  Header parses (thousands of instructions,
// once per deflate block) are batched: a lane that reaches a header waits until a few others have too.
__global__ void __launch_bounds__(32, INF_CTAS_PER_SM) bgzf_inflate(const uint8_t *__restrict__ comp, const Task *__restrict__ tasks, int ntask, uint8_t *__restrict__ unc,
                                                                    int *__restrict__ err, unsigned *__restrict__ next_task)
{
  extern __shared__ __align__(16) unsigned char inf_smem[];
  bki::Tab &T = reinterpret_cast<bki::Tab *>(inf_smem)[threadIdx.x];
  enum { FETCH = 8, IDLE = 9 };
  bki::Lane L;
  L.phase = FETCH;
  int t = -1, waited = 0;
  for (;;) {
    if (L.phase == FETCH) {
      t = (int)atomicAdd(next_task, 1u);
      if (t >= ntask) L.phase = IDLE;
      else { Task k = tasks[t]; bki::lane_init(L, comp + k.src, k.clen, unc + k.dst, k.ulen); waited = 0; }
    }
    int rc = 0;
    const bool want_h = L.phase == bki::PH_HEADER;
    const unsigned hm = __ballot_sync(0xffffffffu, want_h);
    if (hm) {
      const unsigned busy = __ballot_sync(0xffffffffu, L.phase == bki::PH_TOKENS || L.phase == bki::PH_STORED);
      if (want_h) ++waited;
      const bool go = __popc(hm) >= INF_HBATCH || busy == 0u || __any_sync(0xffffffffu, want_h && waited > INF_HWAIT);
      if (go && want_h) { rc = bki::lane_header(L, T); waited = 0; }
    }
#pragma unroll 1
    for (int r = 0; r < INF_STEPS; ++r)
      if (!rc && (L.phase == bki::PH_TOKENS || L.phase == bki::PH_STORED)) rc = bki::lane_step<INF_LITMAX>(L, T);
    bool finished = false;
    if (!rc && L.phase == bki::PH_DONE) { rc = bki::lane_finish(L); finished = true; }
    if (rc) { atomicCAS(err, 0, (t << 4) | rc); finished = true; }
    if (finished) L.phase = FETCH;
    if (__all_sync(0xffffffffu, L.phase == IDLE)) break;
  }
}

// gzip CRC32 of every inflated block against the value stored after its deflate payload (htslib bgzf.c:338,404-416):
// one warp per block, 32 contiguous slices, partials advanced over the bytes that follow and XORed together
__global__ void __launch_bounds__(256) bgzf_crc32(const uint8_t *__restrict__ comp, const Task *__restrict__ tasks, int ntask, const uint8_t *__restrict__ unc, int *__restrict__ err)
{
  __shared__ uint32_t tab[256];
  tab[threadIdx.x] = bki::crc_table_entry(threadIdx.x);
  __syncthreads();
  const unsigned lane = threadIdx.x & 31;
  for (int t = blockIdx.x * 8 + (threadIdx.x >> 5); t < ntask; t += gridDim.x * 8) {
    Task k = tasks[t];
    uint32_t per = (k.ulen + 31u) / 32u;
    uint32_t lo = min(lane * per, k.ulen), hi = min(lo + per, k.ulen);
    uint32_t c = bki::crc_run(tab, lane == 0 ? 0xffffffffu : 0u, unc + k.dst + lo, hi - lo);
    c = bki::crc_shift(c, k.ulen - hi);
    for (int o = 16; o; o >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, o);
    c ^= 0xffffffffu;
    const uint8_t *q = comp + k.src + k.clen;             // CRC32, ISIZE follow the payload
    uint32_t want = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24);
    if (lane == 0 && c != want) atomicCAS(err, 0, t + 1);
  }
}

__device__ __forceinline__ uint32_t ld32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
__device__ __forceinline__ uint32_t ld16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// does a BAM alignment record plausibly start at u[o]?  (SAM spec 4.2: block_size, refID, pos, l_read_name, mapq, bin,
// n_cigar_op, flag, l_seq, next_refID, next_pos, tlen, read_name NUL-terminated and printable)
__device__ bool looks_like_record(const uint8_t *__restrict__ u, uint32_t o, uint32_t total, int n_ref, uint32_t *next)
{
  if ((uint64_t)o + 36 > total) return false;
  uint32_t bs = ld32(u + o);
  if (bs < 34 || bs > (1u << 28)) return false;
  int32_t tid = (int32_t)ld32(u + o + 4), pos = (int32_t)ld32(u + o + 8);
  if (tid < -1 || tid >= n_ref || pos < -1) return false;
  uint32_t l_name = u[o + 12];
  if (l_name < 2) return false;
  uint32_t n_cig = ld16(u + o + 16);
  int32_t l_seq = (int32_t)ld32(u + o + 20);
  if (l_seq < 0) return false;
  int32_t mtid = (int32_t)ld32(u + o + 24), mpos = (int32_t)ld32(u + o + 28);
  if (mtid < -1 || mtid >= n_ref || mpos < -1) return false;
  uint64_t need = 32ull + l_name + 4ull * n_cig + (uint64_t)((l_seq + 1) / 2) + (uint64_t)l_seq;
  if (need > bs) return false;
  if ((uint64_t)o + 36 + l_name > total) return false;
  if (u[o + 36 + l_name - 1] != 0) return false;
  for (uint32_t k = 0; k + 1 < l_name; ++k) { uint8_t ch = u[o + 36 + k]; if (ch < 33 || ch > 126) return false; }
  *next = o + 4 + bs;                       // may wrap for absurd bs: bounded above
  return true;
}

// one warp per segment s >= first_seg (1 when the chain origin is known, 0 when a block range starts mid-stream):
// first offset in [s*SEG, (s+1)*SEG) that starts a chain of 3 plausible records
__global__ void bam_seed(const uint8_t *__restrict__ u, uint32_t total, int n_ref, uint32_t nseg, uint32_t *__restrict__ seed, uint32_t first_seg)
{
  uint32_t s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5) + first_seg;
  if (s >= nseg) return;
  uint32_t lane = threadIdx.x & 31;
  uint32_t lo = s * SEG, hi = min(total, lo + SEG);
  uint32_t found = NONE;
  for (uint32_t base = lo; base < hi; base += 32) {
    uint32_t o = base + lane;
    bool ok = false;
    if (o < hi) {
      uint32_t o1, o2, o3;
      ok = looks_like_record(u, o, total, n_ref, &o1);
      if (ok && (uint64_t)o1 + 36 <= total) ok = looks_like_record(u, o1, total, n_ref, &o2) && ((uint64_t)o2 + 36 > total || looks_like_record(u, o2, total, n_ref, &o3));
    }
    unsigned m = __ballot_sync(0xffffffffu, ok);
    if (m) { found = base + (uint32_t)__ffs(m) - 1; break; }
  }
  if (lane == 0) seed[s] = found;
}

// one thread per segment: follow the record chain from seed[s] up to the next live seed (or the end of the data)
// count pass: cnt / land / why (0 = reached the next seed, 1 = end of data or partial record, 2 = block_size < 32)
template <bool WRITE>
__global__ void bam_walk(const uint8_t *__restrict__ u, uint32_t total, uint32_t nseg, const uint32_t *__restrict__ seed, uint32_t *__restrict__ cnt, uint32_t *__restrict__ land,
                         uint32_t *__restrict__ why, const uint32_t *__restrict__ base, uint32_t *__restrict__ rec_off, int *__restrict__ err, uint32_t stop_at)
{
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  uint32_t o = seed[s];
  if (o == NONE) { if (!WRITE) { cnt[s] = 0; land[s] = NONE; why[s] = 0; } return; }
  uint32_t limit = total;
  for (uint32_t j = s + 1; j < nseg; ++j) if (seed[j] != NONE) { limit = seed[j]; break; }
  uint32_t n = 0, w = WRITE ? base[s] : 0, y = 0;
  while (o < limit && o < stop_at) {                       // records starting at or after stop_at belong to the next block range
    if ((uint64_t)o + 4 > total) { y = 1; break; }
    uint32_t bs = ld32(u + o);
    if (bs < 32) { if (WRITE) atomicCAS(err, 0, 1); y = 2; break; }
    if ((uint64_t)o + 4 + bs > total) { y = 1; break; }      // partial record at the end of the chunk: carried over
    if (WRITE) rec_off[w + n] = o;
    ++n;
    o += 4 + bs;
  }
  if (!WRITE) { cnt[s] = n; land[s] = o; why[s] = y; }
}

// accept seeds by induction from segment 0; drop the first seed the previous walk does not land on.
// A seed is tested against the chain BEFORE the range-end test: the record that straddles the end of a block range can
// jump over a false-positive seed that lies before stop_at, and such a seed must not stay live (its walk would emit
// records that do not exist).  When the range ends inside segment `prev`, every later seed is killed and the walk repeated.
__global__ void bam_stitch(uint32_t nseg, uint32_t *__restrict__ seed, const uint32_t *__restrict__ land, const uint32_t *__restrict__ why,
                           int *__restrict__ state /* [0] changed, [1] corrupt, [2] carry start */, uint32_t stop_at)
{
  if (blockIdx.x || threadIdx.x) return;
  uint32_t prev = 0;
  state[0] = 0;
  for (uint32_t s = 1; s < nseg; ++s) {
    if (seed[s] == NONE) continue;
    if (land[prev] != seed[s]) {                            // seed s is not on the true chain (or lies inside the trailing partial record)
      if (land[prev] >= stop_at) {                          // the range ends inside segment prev: nothing behind it is ours
        for (uint32_t j = s; j < nseg; ++j) seed[j] = NONE;
        state[0] = 1;
        return;
      }
      if (why[prev] == 2) state[1] = 1;                     // the true chain itself hit a corrupt block_size
      seed[s] = NONE; state[0] = 1;
      return;
    }
    if (land[prev] >= stop_at) break;                        // on the chain, but at or behind the range end: its walk emits nothing
    prev = s;
  }
  if (why[prev] == 2) state[1] = 1;
  state[2] = (int)land[prev];
}

struct Cols {
  uint16_t *flag; uint8_t *mapq; int32_t *tid, *pos, *isize, *endpos;
};
struct RecMeta { uint32_t xf, sf, ncig, salen, oclen; };     // arrays of per-record sizes (scanned in place)

// aux walk: offsets (relative to the record start) of the first SA:Z and OC:Z values, 0 = absent (bam_aux_get)
// *bad = 1 when a Z / H value has no NUL inside the record (every later length scan relies on that terminator)
__device__ void find_sa_oc(const uint8_t *__restrict__ r, uint32_t a, uint32_t end, uint32_t *sa, uint32_t *oc, int *bad)
{
  *sa = 0; *oc = 0;
  while (a + 3 <= end) {
    uint8_t t0 = r[a], t1 = r[a + 1], ty = r[a + 2];
    uint32_t v = a + 3;
    uint32_t len;
    switch (ty) {
      case 'A': case 'c': case 'C': len = 1; break;
      case 's': case 'S': len = 2; break;
      case 'i': case 'I': case 'f': len = 4; break;
      case 'd': len = 8; break;
      case 'Z': case 'H': { uint32_t k = v; while (k < end && r[k]) ++k; if (k >= end) { *bad = 1; return; } len = (k - v) + 1; break; }
      case 'B': {
        if (v + 5 > end) { len = end - v; break; }
        uint8_t st = r[v]; uint32_t cnt = ld32(r + v + 1);
        uint32_t es = (st == 'c' || st == 'C') ? 1u : (st == 's' || st == 'S') ? 2u : 4u;
        uint64_t l = 5ull + (uint64_t)es * cnt;
        len = l > (uint64_t)(end - v) ? (end - v) : (uint32_t)l; break;
      }
      default: len = end - v; break;
    }
    if (ty == 'Z') {
      if (t0 == 'S' && t1 == 'A' && !*sa) *sa = v;
      if (t0 == 'O' && t1 == 'C' && !*oc) *oc = v;
    }
    if (len > end - v) break;
    a = v + len;
  }
}

__global__ void bam_extract_cols(const uint8_t *__restrict__ u, const uint32_t *__restrict__ rec_off, uint32_t nrec, long long n0, Cols C,
                                 uint32_t *__restrict__ xf, uint32_t *__restrict__ sf, uint32_t *__restrict__ ncig, uint32_t *__restrict__ salen, uint32_t *__restrict__ oclen,
                                 uint32_t *__restrict__ sa_ptr, uint32_t *__restrict__ oc_ptr, uint32_t *__restrict__ seqb, int *__restrict__ err)
{
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nrec) return;
  uint32_t o = rec_off[i];
  const uint8_t *r = u + o;
  uint32_t bs = ld32(r);
  int32_t tid = (int32_t)ld32(r + 4), pos = (int32_t)ld32(r + 8);
  uint32_t l_name = r[12];
  uint32_t n_cig = ld16(r + 16), fl = ld16(r + 18);
  int32_t l_seq = (int32_t)ld32(r + 20);
  long long g = n0 + i;
  // bam_read1 (htslib sam.c:427-429) rejects l_qseq < 0, l_qname < 1 and fixed fields that do not fit the record:
  // everything below indexes the record by these lengths
  if (l_seq < 0 || l_name < 1 || 32ull + l_name + 4ull * n_cig + (uint64_t)((l_seq + 1) / 2) + (uint64_t)l_seq > (uint64_t)bs) {
    atomicCAS(err, 0, 3);
    C.tid[g] = tid; C.pos[g] = pos; C.mapq[g] = 0; C.flag[g] = 0; C.isize[g] = 0; C.endpos[g] = pos + 1;
    xf[i] = sf[i] = ncig[i] = salen[i] = oclen[i] = sa_ptr[i] = oc_ptr[i] = seqb[i] = 0u;
    return;
  }
  C.tid[g] = tid; C.pos[g] = pos; C.mapq[g] = r[13]; C.flag[g] = (uint16_t)fl; C.isize[g] = (int32_t)ld32(r + 32);
  uint32_t cg = 36 + l_name;
  int32_t rlen = 0;
  uint32_t end = 4 + bs;
  for (uint32_t k = 0; k < n_cig && cg + 4 * k + 4 <= end; ++k) {
    uint32_t c = ld32(r + cg + 4 * k), op = c & 0xf;
    if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rlen += (int32_t)(c >> 4);
  }
  C.endpos[g] = (!(fl & 0x4) && n_cig > 0) ? pos + rlen : pos + 1;                      // bam_endpos, sam.c:344-350
  uint64_t a64 = (uint64_t)cg + 4ull * n_cig + (uint64_t)((l_seq + 1) / 2) + (uint64_t)l_seq;
  uint32_t sa = 0, oc = 0;
  int bad = 0;
  if (a64 < end) find_sa_oc(r, (uint32_t)a64, end, &sa, &oc, &bad);
  if (bad) { atomicCAS(err, 0, 3); sa = oc = 0; }
  bool has_sa = sa && r[sa];
  uint32_t sl = 0, ol = 0;
  if (has_sa) {                                            // both values are NUL-terminated inside the record (find_sa_oc)
    while (sa + sl < end && r[sa + sl]) ++sl;
    if (oc) while (oc + ol < end && r[oc + ol]) ++ol;
  }
  xf[i] = (!(fl & 0x2) || has_sa) ? 1u : 0u;
  sf[i] = has_sa ? 1u : 0u;
  ncig[i] = has_sa ? n_cig : 0u;
  salen[i] = sl; oclen[i] = ol;
  sa_ptr[i] = has_sa ? o + sa : 0u;
  oc_ptr[i] = (has_sa && ol) ? o + oc : 0u;
  seqb[i] = has_sa ? (uint32_t)((l_seq + 1) / 2) : 0u;
}

struct Side {
  uint32_t *x_rec; int32_t *x_mtid, *x_mpos; uint64_t *x_nh;
  uint32_t *sa_rec, *cig_off, *cig_ops, *sa_off, *oc_off; uint8_t *sa_txt, *oc_txt;
  uint32_t *seq_off; uint8_t *seq4; int32_t *seq_len;
  long long x0, s0, cig0, sab0, ocb0, seqb0;   // entries already in the context
};

__global__ void bam_extract_side(const uint8_t *__restrict__ u, const uint32_t *__restrict__ rec_off, uint32_t nrec, long long n0, Side S,
                                 const uint32_t *__restrict__ xf, const uint32_t *__restrict__ xo, const uint32_t *__restrict__ sf, const uint32_t *__restrict__ so,
                                 const uint32_t *__restrict__ ncig, const uint32_t *__restrict__ cigo, const uint32_t *__restrict__ salen, const uint32_t *__restrict__ sao,
                                 const uint32_t *__restrict__ oclen, const uint32_t *__restrict__ oco, const uint32_t *__restrict__ sa_ptr, const uint32_t *__restrict__ oc_ptr,
                                 const uint32_t *__restrict__ seqb, const uint32_t *__restrict__ seqo)
{
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nrec) return;
  const uint8_t *r = u + rec_off[i];
  if (xf[i]) {
    long long x = S.x0 + xo[i];
    S.x_rec[x] = (uint32_t)(n0 + i);
    S.x_mtid[x] = (int32_t)ld32(r + 24); S.x_mpos[x] = (int32_t)ld32(r + 28);
    uint64_t a = 0xcbf29ce484222325ULL, b = 0x9E3779B97F4A7C15ULL;           // bkid_name_hash (include/breakid_b200.h)
    uint32_t l_name = r[12];
    for (uint32_t k = 0; k < l_name && r[36 + k]; ++k) {
      uint64_t c = r[36 + k];
      a = (a ^ c) * 0x100000001b3ULL;
      b = (b ^ c) * 0xff51afd7ed558ccdULL;
      b ^= b >> 32;
    }
    S.x_nh[2 * x] = a; S.x_nh[2 * x + 1] = b;
  }
  if (sf[i]) {
    long long s = S.s0 + so[i];
    S.sa_rec[s] = (uint32_t)(n0 + i);
    uint32_t nc = ncig[i], l_name = r[12];
    long long c0 = S.cig0 + cigo[i];
    for (uint32_t k = 0; k < nc; ++k) S.cig_ops[c0 + k] = ld32(r + 36 + l_name + 4 * k);
    S.cig_off[s + 1] = (uint32_t)(c0 + nc);
    long long t0 = S.sab0 + sao[i];
    const uint8_t *sp = u + sa_ptr[i];
    for (uint32_t k = 0; k < salen[i]; ++k) S.sa_txt[t0 + k] = sp[k];
    S.sa_off[s + 1] = (uint32_t)(t0 + salen[i]);
    long long q0 = S.ocb0 + oco[i];
    if (oclen[i]) { const uint8_t *op = u + oc_ptr[i]; for (uint32_t k = 0; k < oclen[i]; ++k) S.oc_txt[q0 + k] = op[k]; }
    S.oc_off[s + 1] = (uint32_t)(q0 + oclen[i]);
    long long b0 = S.seqb0 + seqo[i];
    const uint8_t *sq = r + 36 + l_name + 4 * nc;
    for (uint32_t k = 0; k < seqb[i]; ++k) S.seq4[b0 + k] = sq[k];
    S.seq_off[s + 1] = (uint32_t)(b0 + seqb[i]);
    S.seq_len[s] = (int32_t)ld32(r + 20);
  }
}

}  // namespace bamdec

struct bkid_decoder {                 // per-context streaming state, allocated on first use
  DBuf comp[2], unc, carry, tasks, seed, cnt, land, base, rec_off, meta[8], metao[6], state;
  uint8_t *h_stage[2] = {nullptr, nullptr}; size_t h_cap = 0;
  bamdec::Task *h_tasks = nullptr; size_t h_tasks_cap = 0;
  cudaStream_t st_copy = nullptr;
  cudaEvent_t ev_h2d[2], ev_free[2], ev_t[8];
  DBuf aux, nm_txt, nm_off, nm_slot;    // SAM decode (bkid_samdec.cuh): per-line fields, target-name lookup table
  uint32_t nm_mask = 0; bool names_built = false;
  bool init = false;
  bool skip_crc = false;                // BKID_BGZF_NO_CRC=1: timing experiments only
  bkid_decode_stats stats;
};

static int decoder_init(bkid_ctx *c)
{
  if (!c->dec) c->dec = new bkid_decoder();
  bkid_decoder *d = c->dec;
  if (d->init) return 0;
  CU(c, cudaStreamCreateWithFlags(&d->st_copy, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) { CU(c, cudaEventCreateWithFlags(&d->ev_h2d[i], cudaEventDisableTiming)); CU(c, cudaEventCreateWithFlags(&d->ev_free[i], cudaEventDisableTiming)); }
  for (int i = 0; i < 8; ++i) CU(c, cudaEventCreate(&d->ev_t[i]));
  CU(c, cudaFuncSetAttribute(bamdec::bgzf_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(32 * sizeof(bki::Tab))));
  d->init = true;
  return 0;
}

static void decoder_free(bkid_ctx *c)
{
  bkid_decoder *d = c->dec;
  if (!d) return;
  for (DBuf *b : {&d->comp[0], &d->comp[1], &d->unc, &d->carry, &d->tasks, &d->seed, &d->cnt, &d->land, &d->base, &d->rec_off, &d->state, &d->aux, &d->nm_txt, &d->nm_off, &d->nm_slot}) b->release();
  for (auto &b : d->meta) b.release();
  for (auto &b : d->metao) b.release();
  for (int i = 0; i < 2; ++i) if (d->h_stage[i]) cudaFreeHost(d->h_stage[i]);
  if (d->h_tasks) cudaFreeHost(d->h_tasks);
  if (d->init) {
    cudaStreamDestroy(d->st_copy);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(d->ev_h2d[i]); cudaEventDestroy(d->ev_free[i]); }
    for (int i = 0; i < 8; ++i) cudaEventDestroy(d->ev_t[i]);
  }
  delete d;
  c->dec = nullptr;
}

// Decode the records that START in the uncompressed extent of blocks [b_begin, b_end).  b_begin == 0: the chain starts at
// first_record_uoffset; otherwise the first record is found by seeding (and reported in *first_uoff so that the caller
// can verify it against where the previous range landed).  b_end < n_blocks: up to `overlap` further blocks are read
// so that the record straddling the range end completes; *land_uoff = start of the first record of the NEXT range.
static int push_bgzf_impl(bkid_ctx *c, const uint8_t *file, uint64_t file_size, const bkid_bgzf_block *blocks, int64_t n_blocks, uint64_t first_record_uoffset, int64_t b_begin, int64_t b_end,
                          int64_t *n_records, uint64_t *first_uoff, uint64_t *land_uoff)
{
  using namespace bamdec;
  if (!c || !file || !blocks || n_blocks < 0 || b_begin < 0 || b_end < b_begin || b_end > n_blocks) return c ? fail(c, BKID_ERR_ARG, "bad bgzf arguments") : BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->err.clear();
  if (c->borrowed) return fail(c, BKID_ERR_ARG, "context holds borrowed device columns; bkid_reset first");
  TRY(c, decoder_init(c));
  bkid_decoder *d = c->dec;
  cudaStream_t st = c->st;
  invalidate(c);
  TRY(c, settle_forms(c, 1, 1, 0));                           // the decoder writes the wide insert-size / end columns
  memset(&d->stats, 0, sizeof d->stats);
  d->skip_crc = getenv("BKID_BGZF_NO_CRC") != nullptr;
  size_t COMP_CAP = (size_t)1536 << 20, UNC_CAP = (size_t)3072 << 20, CARRY_CAP = (size_t)64 << 20;   // unc offsets are 32-bit: UNC_CAP + CARRY_CAP < 4 GiB
  if (const char *e = getenv("BKID_BGZF_CHUNK_KB")) {          // tests: small chunks exercise the streaming / carry logic on small files
    long kb = atol(e);
    if (kb >= 64) { UNC_CAP = (size_t)kb << 10; COMP_CAP = UNC_CAP; }
  }
  // is the file already in pinned host memory?  then H2D goes straight from it
  bool pinned = false;
  {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, file) == cudaSuccess) pinned = (pa.type == cudaMemoryTypeHost);
    cudaGetLastError();
  }
  // chunk boundaries
  std::vector<std::pair<int64_t, int64_t>> chunks;
  uint64_t total_u = 0;
  size_t max_span = 0, max_unc = 0;
  const int64_t OVERLAP = 64;                               // blocks read past the range end for the straddling record (4 MiB)
  const int64_t b_last = b_end < n_blocks ? std::min<int64_t>(n_blocks, b_end + OVERLAP) : n_blocks;
  uint64_t u_begin = 0, u_end = 0;                          // uncompressed offsets of the range in the whole stream
  for (int64_t b = 0; b < b_end; ++b) { if (b < b_begin) u_begin += blocks[b].usize; u_end += blocks[b].usize; }
  const bool open_end = b_end >= n_blocks;
  for (int64_t b0 = b_begin; b0 < b_last;) {
    size_t cb = 0, ub = 0; int64_t b1 = b0;
    uint64_t span0 = blocks[b0].payload_off;
    // (a small first chunk to fill the copy pipeline sooner was measured slower: one inflate launch costs a full
    // per-block latency of ~20 ms whatever its size, so fewer, bigger launches win)
    const size_t ccap = COMP_CAP, ucap = UNC_CAP;
    while (b1 < b_last) {
      size_t span = (size_t)(blocks[b1].payload_off + blocks[b1].payload_len + 8 - span0);
      if (b1 > b0 && (span > ccap || ub + blocks[b1].usize > ucap)) break;
      if (blocks[b1].usize > (1u << 16) || (b1 > b0 && blocks[b1].payload_off < blocks[b1 - 1].payload_off + blocks[b1 - 1].payload_len) ||
          blocks[b1].payload_off > file_size || (uint64_t)blocks[b1].payload_len + 8 > file_size - blocks[b1].payload_off)
        return fail(c, BKID_ERR_IO, "corrupt BGZF block table (a block lies outside the file or overlaps its predecessor)");
      cb = span; ub += blocks[b1].usize; ++b1;
    }
    if (cb > COMP_CAP + (1u << 17)) return fail(c, BKID_ERR_IO, "BGZF block larger than 64 KiB");
    chunks.push_back({b0, b1});
    total_u += ub;
    max_span = std::max(max_span, cb); max_unc = std::max(max_unc, ub);
    b0 = b1;
  }
  // buffers are sized by what this file needs (small files: small allocations); the carry buffer grows on demand
  size_t carry_cap = std::min<size_t>(CARRY_CAP, (size_t)4 << 20);
  TRY(c, d->unc.ensure(max_unc + CARRY_CAP + 256, 0, st));
  TRY(c, d->carry.ensure(carry_cap + 256, 0, st));
  TRY(c, d->state.ensure(256, 0, st));
  for (int i = 0; i < (chunks.size() > 1 ? 2 : 1); ++i) TRY(c, d->comp[i].ensure(max_span + 256, 0, st));
  if (!pinned && d->h_cap < max_span + 256) {
    for (int i = 0; i < 2; ++i) { if (d->h_stage[i]) cudaFreeHost(d->h_stage[i]); d->h_stage[i] = nullptr; }
    for (int i = 0; i < (chunks.size() > 1 ? 2 : 1); ++i) CU(c, cudaMallocHost((void **)&d->h_stage[i], max_span + 256));
    d->h_cap = chunks.size() > 1 ? max_span + 256 : 0;          // a single-slot allocation is not reused for multi-chunk files
  }
  size_t max_tasks = 0;
  for (auto &ch : chunks) max_tasks = std::max<size_t>(max_tasks, (size_t)(ch.second - ch.first));
  if (d->h_tasks_cap < 2 * max_tasks + 2) {
    if (d->h_tasks) cudaFreeHost(d->h_tasks);
    CU(c, cudaMallocHost((void **)&d->h_tasks, (2 * max_tasks + 2) * sizeof(Task)));
    d->h_tasks_cap = 2 * max_tasks + 2;
  }
  TRY(c, d->tasks.ensure((2 * max_tasks + 2) * sizeof(Task), 0, st));
  int *state = d->state.as<int>();           // [0] changed [1] corrupt [2] carry start [4] inflate err [5] walk err [6] crc mismatch (block + 1)
  CU(c, cudaMemsetAsync(state, 0, 64, st));
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  if (c->n_sa == 0) { TRY(c, reserve_impl(c, c->n, c->n_x, 1, 1, 1, 1)); CU(c, cudaMemsetAsync(c->cig_off.p, 0, 4, st)); CU(c, cudaMemsetAsync(c->sa_off.p, 0, 4, st)); CU(c, cudaMemsetAsync(c->oc_off.p, 0, 4, st)); }

  auto stage_chunk = [&](size_t k) -> int {            // host copy (if needed) + async H2D of chunk k into slot k&1
    int slot = (int)(k & 1);
    int64_t b0 = chunks[k].first, b1 = chunks[k].second;
    uint64_t span0 = blocks[b0].payload_off;
    size_t span = (size_t)(blocks[b1 - 1].payload_off + blocks[b1 - 1].payload_len + 8 - span0);
    CU(c, cudaStreamWaitEvent(d->st_copy, d->ev_free[slot], 0));          // the inflate that read this slot has finished
    const uint8_t *src = file + span0;
    if (!pinned) {
      CU(c, cudaEventSynchronize(d->ev_h2d[slot]));                        // previous H2D out of this staging buffer done
      memcpy(d->h_stage[slot], src, span);
      src = d->h_stage[slot];
    }
    CU(c, cudaMemcpyAsync(d->comp[slot].p, src, span, cudaMemcpyHostToDevice, d->st_copy));
    CU(c, cudaEventRecord(d->ev_h2d[slot], d->st_copy));
    d->stats.compressed_bytes += (int64_t)span;
    return 0;
  };
  for (int i = 0; i < 2; ++i) { CU(c, cudaEventRecord(d->ev_free[i], st)); CU(c, cudaEventRecord(d->ev_h2d[i], d->st_copy)); }
  cudaEventRecord(d->ev_t[0], st);
  if (!chunks.empty()) TRY(c, stage_chunk(0));
  uint32_t carry = 0;
  uint64_t skip = b_begin == 0 ? first_record_uoffset : 0;      // bytes of the uncompressed stream before the first record (BAM header)
  bool seek = b_begin > 0;                         // the first record of a mid-stream range is found by seeding
  bool range_done = false;
  uint64_t chunk_u0 = u_begin;                     // stream offset of the first NEW byte of the current chunk
  if (first_uoff) *first_uoff = first_record_uoffset;
  if (land_uoff) *land_uoff = 0;
  long long n_first = c->n;
  float ms_inf = 0, ms_bound = 0, ms_ext = 0;
  for (size_t k = 0; k < chunks.size() && !range_done; ++k) {
    int slot = (int)(k & 1);
    if (k + 1 < chunks.size()) TRY(c, stage_chunk(k + 1));
    int64_t b0 = chunks[k].first, b1 = chunks[k].second;
    uint64_t span0 = blocks[b0].payload_off;
    Task *ht = d->h_tasks + (size_t)slot * max_tasks;
    int nt = 0; uint32_t uo = carry;
    std::vector<int64_t> task_block;                          // empty blocks get no task: error messages name the real block
    for (int64_t b = b0; b < b1; ++b) {
      if (blocks[b].usize) { ht[nt++] = Task{blocks[b].payload_off - span0, uo, blocks[b].payload_len, blocks[b].usize}; task_block.push_back(b); }
      uo += blocks[b].usize;
    }
    auto block_of = [&](long long t) -> long long { return t >= 0 && t < (long long)task_block.size() ? (long long)task_block[(size_t)t] : (long long)b0 + t; };
    uint32_t total = uo;
    uint8_t *u = d->unc.as<uint8_t>();
    Task *dt = d->tasks.as<Task>() + (size_t)slot * max_tasks;
    if (carry) CU(c, cudaMemcpyAsync(u, d->carry.p, carry, cudaMemcpyDeviceToDevice, st));
    CU(c, cudaMemcpyAsync(dt, ht, (size_t)nt * sizeof(Task), cudaMemcpyHostToDevice, st));
    CU(c, cudaStreamWaitEvent(st, d->ev_h2d[slot], 0));
    cudaEventRecord(d->ev_t[1], st);
    if (nt) {
      CU(c, cudaMemsetAsync(state + 7, 0, 4, st));            // block queue head
      BK_LAUNCH(bgzf_inflate, std::min((nt + 31) / 32, 148 * INF_CTAS_PER_SM), 32, 32 * sizeof(bki::Tab), st, d->comp[slot].as<uint8_t>(), dt, nt, u, state + 4, (unsigned *)(state + 7));
    }
    if (nt && !d->skip_crc) BK_LAUNCH(bgzf_crc32, std::min((nt + 7) / 8, 148 * 8), 256, 0, st, d->comp[slot].as<uint8_t>(), dt, nt, u, state + 6);
    CU(c, cudaEventRecord(d->ev_free[slot], st));
    cudaEventRecord(d->ev_t[2], st);
    d->stats.n_blocks += nt; d->stats.uncompressed_bytes += (int64_t)(total - carry);
    // ---- record boundaries ----
    const uint64_t buf_u0 = chunk_u0 - carry;                 // stream offset of buffer position 0
    chunk_u0 += total - carry;
    const uint32_t stop_at = (!open_end && u_end - buf_u0 < (uint64_t)total) ? (uint32_t)(u_end - buf_u0) : 0xffffffffu;
    uint32_t start = 0;
    if (skip) {
      if (skip >= total) { skip -= total; carry = 0; TRY(c, sync_check(c)); continue; }
      start = (uint32_t)skip; skip = 0;
    }
    uint32_t nseg = (total + SEG - 1) / SEG;
    // segments before `start` hold header bytes only
    uint32_t seg0 = start / SEG;
    size_t sb = (size_t)(nseg + 2) * 4;
    TRY(c, d->seed.ensure(sb, 0, st)); TRY(c, d->cnt.ensure(sb, 0, st)); TRY(c, d->land.ensure(sb, 0, st)); TRY(c, d->base.ensure(sb, 0, st));
    TRY(c, c->sc.ensure((long long)nseg + 8, st));
    uint32_t *seed = d->seed.as<uint32_t>();
    CU(c, cudaMemsetAsync(seed, 0xff, sb, st));
    // the walk kernels treat segment `seg0` as the chain origin: shift the arrays so that it is index 0
    uint32_t nsg = nseg - seg0;
    uint32_t *seedv = seed + seg0;
    if (seek) {
      // mid-stream range: every segment is seeded, the first seed is the chain origin (verified by the caller against
      // the landing point of the previous range)
      BK_LAUNCH(bam_seed, GRID1(nseg + 1, 8), 256, 0, st, u, total, c->nt, nseg, seed, 0u);
      std::vector<uint32_t> hseed(nseg);
      CU(c, cudaMemcpyAsync(hseed.data(), seed, (size_t)nseg * 4, cudaMemcpyDeviceToHost, st));
      TRY(c, sync_check(c));
      uint32_t s0 = 0;
      while (s0 < nseg && hseed[s0] == NONE) ++s0;
      if (s0 == nseg) return fail(c, BKID_ERR_IO, "no BAM record start found at the beginning of the block range");
      seg0 = s0; nsg = nseg - seg0; seedv = seed + seg0; start = hseed[s0];
      if (first_uoff) *first_uoff = buf_u0 + start;
      seek = false;
    } else {
      if (nsg > 1) {
        // seeds for segments seg0+1 .. nseg-1 (kernel indexes segments from the start of the buffer)
        BK_LAUNCH(bam_seed, GRID1(nseg, 8), 256, 0, st, u, total, c->nt, nseg, seed, 1u);
      }
      CU(c, cudaMemcpyAsync(seedv, &start, 4, cudaMemcpyHostToDevice, st));   // pageable 4-byte copy: staged by the driver before return
      if (seg0) CU(c, cudaMemsetAsync(seed, 0xff, (size_t)seg0 * 4, st));
    }
    const uint32_t stop_rel = stop_at;                        // buffer coordinates (seedv / walkers use absolute buffer offsets)
    int hstate[8];
    for (int iter = 0;; ++iter) {
      BK_LAUNCH((bam_walk<false>), GRID1(nsg, 128), 128, 0, st, u, total, nsg, seedv, d->cnt.as<uint32_t>(), d->land.as<uint32_t>(), d->base.as<uint32_t>(), (const uint32_t *)nullptr, (uint32_t *)nullptr, state + 5, stop_rel);
      BK_LAUNCH(bam_stitch, 1, 32, 0, st, nsg, seedv, d->land.as<uint32_t>(), d->base.as<uint32_t>(), state, stop_rel);
      CU(c, cudaMemcpyAsync(hstate, state, 32, cudaMemcpyDeviceToHost, st));
      TRY(c, sync_check(c));
      if (hstate[4]) return fail(c, BKID_ERR_IO, "inflate failed: BGZF block " + std::to_string(block_of(hstate[4] >> 4)) + " (deflate error " + std::to_string(hstate[4] & 15) + ")");
      if (hstate[6]) return fail(c, BKID_ERR_IO, "CRC32 mismatch in BGZF block " + std::to_string(block_of(hstate[6] - 1)));
      if (hstate[1]) return fail(c, BKID_ERR_IO, "corrupt BAM record (block_size < 32)");
      if (!hstate[0]) break;
      d->stats.seed_repairs++;
      if (iter > (int)nsg + 2) return fail(c, BKID_ERR_IO, "record boundary search did not converge");
    }
    uint32_t carry_start = (uint32_t)hstate[2];
    bk::exclusive_scan<uint32_t, uint32_t>(d->cnt.as<uint32_t>(), d->base.as<uint32_t>(), nsg, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
    unsigned long long nrec64 = 0;
    CU(c, cudaMemcpyAsync(&nrec64, tot, 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    uint32_t nrec = (uint32_t)nrec64;
    cudaEventRecord(d->ev_t[3], st);
    if ((unsigned long long)(c->n + nrec) >= 0xffffffffull) return fail(c, BKID_ERR_ARG, "more than 2^32-1 records per context");
    if (nrec) {
      // capacity: after the first chunk extrapolate from records per uncompressed byte
      long long want = c->n + nrec;
      if (k == 0 && chunks.size() > 1 && total > start) want = std::max<long long>(want, c->n + (long long)((double)nrec / (double)(total - start) * (double)total_u * 1.03) + 1024);
      want = std::min<long long>(want, 0xfffffffell);
      TRY(c, reserve_impl(c, std::max<long long>(want, c->n + nrec), c->n_x, std::max<long long>(c->n_sa, 1), std::max<long long>(c->n_cig, 1), std::max<long long>(c->sa_bytes, 1), std::max<long long>(c->oc_bytes, 1)));
      TRY(c, d->rec_off.ensure((size_t)nrec * 4 + 64, 0, st));
      for (auto &m : d->meta) TRY(c, m.ensure((size_t)nrec * 4 + 64, 0, st));
      for (auto &m : d->metao) TRY(c, m.ensure((size_t)nrec * 4 + 64, 0, st));
      TRY(c, c->sc.ensure((long long)nrec + 8, st));
      BK_LAUNCH((bam_walk<true>), GRID1(nsg, 128), 128, 0, st, u, total, nsg, seedv, d->cnt.as<uint32_t>(), d->land.as<uint32_t>(), (uint32_t *)nullptr, d->base.as<uint32_t>(), d->rec_off.as<uint32_t>(), state + 5, stop_rel);
      Cols C{c->flag.as<uint16_t>(), c->mapq.as<uint8_t>(), c->tid.as<int32_t>(), c->pos.as<int32_t>(), c->isize.as<int32_t>(), c->endpos.as<int32_t>()};
      uint32_t *m[8]; for (int i = 0; i < 8; ++i) m[i] = d->meta[i].as<uint32_t>();        // [5],[6] = tag pointers, [7] = seq bytes
      uint32_t *mo[6]; for (int i = 0; i < 6; ++i) mo[i] = d->metao[i].as<uint32_t>();
      BK_LAUNCH(bam_extract_cols, GRID1(nrec, 128), 128, 0, st, u, d->rec_off.as<uint32_t>(), nrec, c->n, C, m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], state + 5);
      unsigned long long *tots = (unsigned long long *)(c->counters.as<unsigned>() + CS_DECODE);     // 6 x u64
      for (int i = 0; i < 5; ++i) bk::exclusive_scan<uint32_t, uint32_t>(m[i], mo[i], nrec, c->sc.scan_tmp.as<unsigned long long>(), tots + i, st);
      bk::exclusive_scan<uint32_t, uint32_t>(m[7], mo[5], nrec, c->sc.scan_tmp.as<unsigned long long>(), tots + 5, st);
      unsigned long long ht5[6];
      int hs5 = 0;
      CU(c, cudaMemcpyAsync(ht5, tots, 48, cudaMemcpyDeviceToHost, st));
      CU(c, cudaMemcpyAsync(&hs5, state + 5, 4, cudaMemcpyDeviceToHost, st));
      TRY(c, sync_check(c));
      if (hs5 == 3) return fail(c, BKID_ERR_IO, "corrupt BAM record (fixed fields do not fit block_size, or an unterminated tag value)");
      if (hs5) return fail(c, BKID_ERR_IO, "corrupt BAM record (block_size < 32)");
      TRY(c, reserve_impl(c, c->n + nrec, c->n_x + (long long)ht5[0], c->n_sa + (long long)ht5[1], c->n_cig + (long long)ht5[2], c->sa_bytes + (long long)ht5[3], c->oc_bytes + (long long)ht5[4]));
      {
        size_t s_new = (size_t)(c->n_sa + (long long)ht5[1]);
        TRY(c, c->seq_off.ensure((s_new + 1) * 4 + 64, (size_t)(c->n_sa + 1) * 4, st));
        TRY(c, c->seq_len.ensure(s_new * 4 + 64, (size_t)c->n_sa * 4, st));
        TRY(c, c->seq4.ensure((size_t)c->seq_bytes + (size_t)ht5[5] + 64, (size_t)c->seq_bytes, st));
        if (c->n_sa == 0) CU(c, cudaMemsetAsync(c->seq_off.p, 0, 4, st));
      }
      Side S{c->x_rec.as<uint32_t>(), c->x_mtid.as<int32_t>(), c->x_mpos.as<int32_t>(), c->x_nh.as<uint64_t>(),
             c->sa_rec.as<uint32_t>(), c->cig_off.as<uint32_t>(), c->cig_ops.as<uint32_t>(), c->sa_off.as<uint32_t>(), c->oc_off.as<uint32_t>(), c->sa_txt.as<uint8_t>(), c->oc_txt.as<uint8_t>(),
             c->seq_off.as<uint32_t>(), c->seq4.as<uint8_t>(), c->seq_len.as<int32_t>(),
             c->n_x, c->n_sa, c->n_cig, c->sa_bytes, c->oc_bytes, c->seq_bytes};
      BK_LAUNCH(bam_extract_side, GRID1(nrec, 128), 128, 0, st, u, d->rec_off.as<uint32_t>(), nrec, c->n, S, m[0], mo[0], m[1], mo[1], m[2], mo[2], m[3], mo[3], m[4], mo[4], m[5], m[6], m[7], mo[5]);
      c->n += nrec; c->n_x += (long long)ht5[0]; c->n_sa += (long long)ht5[1]; c->n_cig += (long long)ht5[2]; c->sa_bytes += (long long)ht5[3]; c->oc_bytes += (long long)ht5[4];
      c->seq_bytes += (long long)ht5[5];
    }
    if (carry_start >= stop_at) {                             // the walk reached the end of the block range: done
      if (land_uoff) *land_uoff = buf_u0 + carry_start;
      range_done = true; carry = 0;
      cudaEventRecord(d->ev_t[4], st);
      TRY(c, sync_check(c));
      continue;
    }
    // ---- carry the partial record at the end of the chunk ----
    carry = total - carry_start;
    if (carry > CARRY_CAP) return fail(c, BKID_ERR_IO, "BAM record larger than 64 MiB");
    if (carry) { TRY(c, d->carry.ensure((size_t)carry + 256, 0, st)); CU(c, cudaMemcpyAsync(d->carry.p, u + carry_start, carry, cudaMemcpyDeviceToDevice, st)); }
    cudaEventRecord(d->ev_t[4], st);
    TRY(c, sync_check(c));
    {
      int hs[8]; CU(c, cudaMemcpy(hs, state, 32, cudaMemcpyDeviceToHost));
      if (hs[5]) return fail(c, BKID_ERR_IO, "corrupt BAM record (block_size < 32)");
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, d->ev_t[1], d->ev_t[2]); ms_inf += ms;
    cudaEventElapsedTime(&ms, d->ev_t[2], d->ev_t[3]); ms_bound += ms;
    cudaEventElapsedTime(&ms, d->ev_t[3], d->ev_t[4]); ms_ext += ms;
  }
  if (!open_end && !range_done) return fail(c, BKID_ERR_IO, "the record straddling the end of the block range does not complete within the overlap");
  if (carry) return fail(c, BKID_ERR_IO, "truncated BAM record at the end of the file");
  if (open_end && land_uoff) *land_uoff = chunk_u0;
  if (skip) return fail(c, BKID_ERR_IO, "first_record_uoffset beyond the end of the uncompressed stream");
  cudaEventRecord(d->ev_t[5], st);
  TRY(c, sync_check(c));
  CU(c, cudaStreamSynchronize(d->st_copy));
  set_ptrs(c);
  cudaEventElapsedTime(&d->stats.total_ms, d->ev_t[0], d->ev_t[5]);
  d->stats.inflate_ms = ms_inf; d->stats.boundaries_ms = ms_bound; d->stats.extract_ms = ms_ext;
  d->stats.n_records = c->n - n_first;
  d->stats.n_chunks = (int64_t)chunks.size();
  c->have_seq = true;                    // the decoder always extracts the read bases of the SA records
  if (n_records) *n_records = c->n - n_first;
  return 0;
}

int bkid_push_bgzf(bkid_ctx *c, const uint8_t *file, uint64_t file_size, const bkid_bgzf_block *blocks, int64_t n_blocks, uint64_t first_record_uoffset, int64_t *n_records)
{
  return push_bgzf_impl(c, file, file_size, blocks, n_blocks, first_record_uoffset, 0, n_blocks, n_records, nullptr, nullptr);
}

int bkid_push_bgzf_range(bkid_ctx *c, const uint8_t *file, uint64_t file_size, const bkid_bgzf_block *blocks, int64_t n_blocks, uint64_t first_record_uoffset, int64_t first_block, int64_t end_block,
                         int64_t *n_records, uint64_t *first_record_uoff, uint64_t *next_record_uoff)
{
  return push_bgzf_impl(c, file, file_size, blocks, n_blocks, first_record_uoffset, first_block, end_block, n_records, first_record_uoff, next_record_uoff);
}

int bkid_get_decode_stats(bkid_ctx *c, bkid_decode_stats *s)
{
  if (!c || !s) return BKID_ERR_ARG;
  if (!c->dec) { memset(s, 0, sizeof *s); return 0; }
  *s = c->dec->stats;
  return 0;
}

// parity-test getter: copy one input column of the context to the host
int bkid_fetch_column(bkid_ctx *c, const char *name, void *out, int64_t cap_bytes, int64_t *n_bytes)
{
  if (!c || !name) return BKID_ERR_ARG;
  cudaSetDevice(c->device);
  std::string k(name);
  const void *p = nullptr; size_t nb = 0;
  size_t n = (size_t)c->n, nx = (size_t)c->n_x, ns = (size_t)c->n_sa;
  if (k == "flag") { p = c->p_flag; nb = n * 2; } else if (k == "mapq") { p = c->p_mapq; nb = n; }
  else if (k == "tid") { p = c->p_tid; nb = n * 4; } else if (k == "pos") { p = c->p_pos; nb = n * 4; }
  else if (k == "isize" || k == "endpos") {
    nb = n * 4;
    p = k == "isize" ? (const void *)c->p_isize : (const void *)c->p_endpos;
    if (!p && n) {                                         // kept narrow in HBM: the getter hands out the wide form
      TRY(c, c->tmpH.ensure(nb + 64, 0, c->st));
      if (k == "isize") BK_LAUNCH(widen_isize16, GRID1(n, 256), 256, 0, c->st, c->p_isize16, (long long)n, c->tmpH.as<int32_t>());
      else BK_LAUNCH(widen_span16, GRID1(n, 256), 256, 0, c->st, c->p_pos, c->p_span16, (long long)n, c->tmpH.as<int32_t>());
      p = c->tmpH.p;
    }
  }
  else if (k == "x_rec") { p = c->p_x_rec; nb = nx * 4; } else if (k == "x_mtid") { p = c->p_x_mtid; nb = nx * 4; }
  else if (k == "x_mpos") { p = c->p_x_mpos; nb = nx * 4; } else if (k == "x_name_hash") { p = c->p_x_nh; nb = nx * 16; }
  else if (k == "sa_rec") { p = c->p_sa_rec; nb = ns * 4; } else if (k == "cig_off") { p = c->p_cig_off; nb = (ns + 1) * 4; }
  else if (k == "cig_ops") { p = c->p_cig_ops; nb = (size_t)c->n_cig * 4; } else if (k == "sa_off") { p = c->p_sa_off; nb = (ns + 1) * 4; }
  else if (k == "sa_txt") { p = c->p_sa_txt; nb = (size_t)c->sa_bytes; } else if (k == "oc_off") { p = c->p_oc_off; nb = (ns + 1) * 4; }
  else if (k == "oc_txt") { p = c->p_oc_txt; nb = (size_t)c->oc_bytes; }
  else if (k == "seq_off") { p = c->have_seq ? c->p_seq_off : nullptr; nb = c->have_seq ? (ns + 1) * 4 : 0; }
  else if (k == "seq4") { p = c->have_seq ? c->p_seq4 : nullptr; nb = c->have_seq ? (size_t)c->seq_bytes : 0; }
  else if (k == "seq_len") { p = c->have_seq ? c->p_seq_len : nullptr; nb = c->have_seq ? ns * 4 : 0; }
  else return fail(c, BKID_ERR_ARG, "unknown column " + k);
  if (n_bytes) *n_bytes = (int64_t)nb;
  if (out && nb) {
    if ((int64_t)nb > cap_bytes) return fail(c, BKID_ERR_ARG, "column buffer too small");
    CU(c, cudaStreamSynchronize(c->st));
    CU(c, cudaMemcpy(out, p, nb, cudaMemcpyDeviceToHost));
  }
  return 0;
}
