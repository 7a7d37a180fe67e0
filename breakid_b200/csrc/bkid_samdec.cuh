// bkid_samdec.cuh -- SAM text decode on the device (bkid_push_sam).  Included by bkid_core.cu after bkid_bamdec.cuh.
//
// The result is defined by the BAM path: for every accepted SAM text, every column bkid_fetch_column returns is
// byte-identical to what bkid_push_bgzf leaves for a BAM holding the same records (SAM spec 1.4 / 4.2 field mapping),
// so every later stage, bkid_sort_records and the sharded run see no difference.
//
//   sam_nl_count / sam_nl_write  16-byte loads, newline count per 4 KiB tile, exclusive scan, line start offsets
//   sam_parse                    one warp per line: tab positions by ballot over 16-byte vectors, the fixed fields
//                                parsed by one lane each in parallel, RNAME / RNEXT through an open-addressing table of
//                                the context's target names; writes the dense columns and the per-line sizes of the
//                                sparse / SA rows (the same arrays bam_extract_cols fills, scanned by the same code)
//   sam_extract_side             one warp per line with a sparse or SA row: name hash, mate fields, CIGAR text -> ops,
//                                SA / OC bytes, SEQ -> 4-bit codes
//
// Lines are ~350 bytes: a thread per line would issue hundreds of dependent byte loads, a warp reads a line in one or
// two 512-byte rounds.  The host cuts the text at newlines into chunks of <= 1 GiB (in-chunk offsets stay 32-bit), so no
// line ever straddles two chunks; chunks go through double-buffered staging and the copy of chunk k+1 overlaps the
// parse of chunk k.
#pragma once

namespace samdec {

constexpr int NL_T = 256;                     // sam_nl_*: 16 bytes per thread, 4 KiB per block
constexpr int PW = 8;                         // sam_parse / sam_extract_side: warps (lines) per block

// per-line error codes; the lowest failing line wins (atomicMin on line << 8 | code)
enum {
  SE_FIELDS = 1, SE_EMPTY, SE_HEADER, SE_QNAME, SE_FLAG, SE_RNAME, SE_RNAME_UNKNOWN, SE_POS, SE_MAPQ, SE_CIGAR, SE_RNEXT,
  SE_RNEXT_UNKNOWN, SE_PNEXT, SE_TLEN, SE_SEQ, SE_QUAL, SE_CIGAR_SEQ, SE_OPT
};

// target-name lookup: slot[h & mask] = tid or -1 (linear probing, capacity >= 2 * n_targets), names verified in full
struct Names { const uint8_t *txt; const uint32_t *off; const int32_t *slot; uint32_t mask; };

__host__ __device__ inline uint32_t name_h32(const uint8_t *p, uint32_t n)
{
  uint32_t h = 2166136261u;
  for (uint32_t k = 0; k < n; ++k) h = (h ^ p[k]) * 16777619u;
  return h;
}

__device__ int lookup(const Names &N, const uint8_t *p, uint32_t n)
{
  for (uint32_t i = name_h32(p, n) & N.mask;; i = (i + 1) & N.mask) {
    int t = N.slot[i];
    if (t < 0) return -1;
    uint32_t a = N.off[t], b = N.off[t + 1];
    if (b - a == n) {
      uint32_t k = 0;
      while (k < n && N.txt[a + k] == p[k]) ++k;
      if (k == n) return t;
    }
  }
}

// unsigned decimal of 1..18 digits, <= mx
__device__ bool dec_u(const uint8_t *p, uint32_t n, unsigned long long mx, unsigned long long *v)
{
  if (n == 0 || n > 18) return false;
  unsigned long long x = 0;
  for (uint32_t k = 0; k < n; ++k) {
    uint32_t d = (uint32_t)p[k] - '0';
    if (d > 9) return false;
    x = x * 10 + d;
  }
  *v = x;
  return x <= mx;
}

__device__ __forceinline__ int cigar_op(uint8_t ch)
{
  switch (ch) {
    case 'M': return 0; case 'I': return 1; case 'D': return 2; case 'N': return 3; case 'S': return 4;
    case 'H': return 5; case 'P': return 6; case '=': return 7; case 'X': return 8; default: return -1;
  }
}

// BAM 4-bit base code (SAM spec 4.2.3, "=ACMGRSVTWYHKDBN"), case-insensitive; any other letter or '.' -> 15
__device__ __forceinline__ uint32_t nt16(uint8_t ch)
{
  if (ch >= 'a' && ch <= 'z') ch -= 32;
  switch (ch) {
    case '=': return 0; case 'A': return 1; case 'C': return 2; case 'M': return 3; case 'G': return 4; case 'R': return 5;
    case 'S': return 6; case 'V': return 7; case 'T': return 8; case 'W': return 9; case 'Y': return 10; case 'H': return 11;
    case 'K': return 12; case 'D': return 13; case 'B': return 14; default: return 15;
  }
}
__device__ __forceinline__ bool seq_char(uint8_t ch) { return (ch >= 'A' && ch <= 'Z') || (ch >= 'a' && ch <= 'z') || ch == '=' || ch == '.'; }
__device__ __forceinline__ bool alnum(uint8_t ch) { return (ch >= 'A' && ch <= 'Z') || (ch >= 'a' && ch <= 'z') || (ch >= '0' && ch <= '9'); }

// 16-bit mask of the bytes equal to `ch` in the 16 bytes at T + v (v 16-aligned)
__device__ __forceinline__ uint32_t eq_mask16(const uint8_t *__restrict__ T, uint32_t v, uint32_t ch4)
{
  uint4 q = *reinterpret_cast<const uint4 *>(T + v);
  uint32_t w[4] = {q.x, q.y, q.z, q.w}, m = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t e = __vcmpeq4(w[j], ch4);                       // 0xff in every equal byte
    m |= ((e & 1u) | ((e >> 7) & 2u) | ((e >> 14) & 4u) | ((e >> 21) & 8u)) << (4 * j);
  }
  return m;
}

__global__ void __launch_bounds__(NL_T) sam_nl_count(const uint8_t *__restrict__ T, uint32_t len, uint32_t *__restrict__ cnt)
{
  __shared__ uint32_t sh[33];
  uint32_t v = (blockIdx.x * NL_T + threadIdx.x) * 16u;
  uint32_t m = 0;
  if (v < len) { m = eq_mask16(T, v, 0x0a0a0a0au); if (len - v < 16) m &= (1u << (len - v)) - 1u; }
  uint32_t tot;
  bk::block_excl_scan<uint32_t>(__popc(m), sh, tot);
  if (threadIdx.x == 0) cnt[blockIdx.x] = tot;
}

// lstart[0] = 0, lstart[k + 1] = 1 + offset of the k-th newline
__global__ void __launch_bounds__(NL_T) sam_nl_write(const uint8_t *__restrict__ T, uint32_t len, const uint32_t *__restrict__ base, uint32_t *__restrict__ lstart)
{
  __shared__ uint32_t sh[33];
  uint32_t v = (blockIdx.x * NL_T + threadIdx.x) * 16u;
  uint32_t m = 0;
  if (v < len) { m = eq_mask16(T, v, 0x0a0a0a0au); if (len - v < 16) m &= (1u << (len - v)) - 1u; }
  uint32_t tot;
  uint32_t o = base[blockIdx.x] + bk::block_excl_scan<uint32_t>(__popc(m), sh, tot);
  while (m) { lstart[++o] = v + (uint32_t)__ffs(m); m &= m - 1; }
  if (blockIdx.x == 0 && threadIdx.x == 0) lstart[0] = 0;
}

struct Aux { int32_t mtid, mpos; uint32_t qlen, cig_at, seq_at, lseq; };   // what sam_extract_side needs of a parsed line

// one warp per line.  Line i is [lstart[i], lstart[i + 1] - 1), the last one of an unterminated text ends at len.
__global__ void __launch_bounds__(PW * 32) sam_parse(const uint8_t *__restrict__ T, uint32_t len, const uint32_t *__restrict__ lstart, uint32_t nnl, uint32_t nrec,
                                                     long long n0, bamdec::Cols C, Names N, uint32_t *__restrict__ xf, uint32_t *__restrict__ sf, uint32_t *__restrict__ ncig,
                                                     uint32_t *__restrict__ salen, uint32_t *__restrict__ oclen, uint32_t *__restrict__ sa_ptr, uint32_t *__restrict__ oc_ptr,
                                                     uint32_t *__restrict__ seqb, Aux *__restrict__ aux, unsigned long long *__restrict__ err)
{
  __shared__ uint32_t sh_tab[PW][11];
  __shared__ unsigned long long sh_sa[PW], sh_oc[PW];
  __shared__ int sh_bad[PW];
  const unsigned FULL = 0xffffffffu, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const uint32_t i = blockIdx.x * PW + w;
  if (i >= nrec) return;                                     // whole warps only
  const uint32_t s = lstart[i];
  uint32_t e = i < nnl ? lstart[i + 1] - 1 : len;
  if (e > s && T[e - 1] == '\r') --e;                        // CRLF: one \r before the newline is dropped
  int code = 0;
  if (e == s) code = SE_EMPTY;
  else if (T[s] == '@') code = SE_HEADER;
  if (lane == 0) { sh_sa[w] = ~0ull; sh_oc[w] = ~0ull; sh_bad[w] = 0; }
  __syncwarp();
  // ---- tab positions: lane l holds bytes [b + 16 l, b + 16 l + 16) of a 512-byte round ----
  uint32_t ntab = 0;
  for (uint32_t b = s & ~15u; !code && b < e; b += 512) {
    const uint32_t v = b + 16 * lane;
    uint32_t m = 0;
    if (v < e) {
      m = eq_mask16(T, v, 0x09090909u);
      if (v < s) m &= 0xffffu << (s - v);
      if (e - v < 16) m &= (1u << (e - v)) - 1u;
    }
    const uint32_t c = __popc(m), incl = bk::warp_incl_scan(c);
    uint32_t idx = ntab + incl - c;
    for (; m; m &= m - 1, ++idx) {
      const uint32_t p = v + (uint32_t)__ffs(m) - 1;
      if (idx < 11) sh_tab[w][idx] = p;
      if (idx >= 10) {                                       // tab idx opens optional field idx + 1: TG:T:VALUE, type one of AifZHB
        const uint32_t q = p + 1;
        bool ok = q + 5 <= e && (((T[q] | 32) >= 'a' && (T[q] | 32) <= 'z')) && alnum(T[q + 1]) && T[q + 2] == ':' && T[q + 4] == ':';
        const uint8_t ty = ok ? T[q + 3] : 0;
        ok = ok && (ty == 'A' || ty == 'i' || ty == 'f' || ty == 'Z' || ty == 'H' || ty == 'B');
        if (!ok) sh_bad[w] = 1;
        else if (ty == 'Z' && T[q] == 'S' && T[q + 1] == 'A') atomicMin(&sh_sa[w], ((unsigned long long)idx << 32) | (q + 5));   // the first SA:Z
        else if (ty == 'Z' && T[q] == 'O' && T[q + 1] == 'C') atomicMin(&sh_oc[w], ((unsigned long long)idx << 32) | (q + 5));
      }
    }
    ntab += __shfl_sync(FULL, incl, 31);
  }
  __syncwarp();
  if (!code && ntab < 10) code = SE_FIELDS;
  if (!code && sh_bad[w]) code = SE_OPT;
  // ---- fixed fields: lane k parses field k ----
  uint32_t fs = 0, fe = 0;
  if (!code && lane < 11) { fs = lane == 0 ? s : sh_tab[w][lane - 1] + 1; fe = lane < 10 ? sh_tab[w][lane] : (ntab > 10 ? sh_tab[w][10] : e); }
  const uint32_t seq_s = __shfl_sync(FULL, fs, 9), seq_e = __shfl_sync(FULL, fe, 9);
  const bool seq_star = !code && seq_e - seq_s == 1 && T[seq_s] == '*';
  const uint32_t lseq = code || seq_star ? 0u : seq_e - seq_s;
  int fcode = 0;
  unsigned long long val = 0;
  uint32_t nops = 0, rlen = 0, qlen = 0;
  const bool star = !code && lane < 11 && fe - fs == 1 && T[fs] == '*';
  if (!code && lane < 11) {
    const uint8_t *f = T + fs;
    const uint32_t n = fe - fs;
    switch (lane) {
      case 0: if (n < 1 || n > 254) fcode = SE_QNAME; break;
      case 1: if (!dec_u(f, n, 65535, &val)) fcode = SE_FLAG; break;
      case 2: case 6: {                                      // RNAME, RNEXT
        if (n == 0) { fcode = lane == 2 ? SE_RNAME : SE_RNEXT; break; }
        if (star) { val = (unsigned long long)-1; break; }
        if (lane == 6 && n == 1 && f[0] == '=') { val = 1ull << 40; break; }   // resolved against RNAME below
        int t = lookup(N, f, n);
        if (t < 0) fcode = lane == 2 ? SE_RNAME_UNKNOWN : SE_RNEXT_UNKNOWN;
        else val = (unsigned long long)(long long)t;
        break;
      }
      case 3: case 7: if (!dec_u(f, n, 0x7fffffffull, &val)) fcode = lane == 3 ? SE_POS : SE_PNEXT; break;
      case 4: if (!dec_u(f, n, 255, &val)) fcode = SE_MAPQ; break;
      case 5: {                                              // CIGAR: * or (len op)+, len 1..2^28-1, <= 65535 ops
        if (star) break;
        if (n == 0) { fcode = SE_CIGAR; break; }
        uint32_t k = 0;
        while (k < n) {
          uint32_t d0 = k;
          unsigned long long L = 0;
          while (k < n && f[k] >= '0' && f[k] <= '9' && k - d0 < 10) L = L * 10 + (f[k++] - '0');
          int op = k < n ? cigar_op(f[k]) : -1;
          if (k == d0 || op < 0 || L < 1 || L >= (1ull << 28) || nops == 65535) { fcode = SE_CIGAR; break; }
          ++k; ++nops;
          if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rlen += (uint32_t)L;
          if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) qlen += (uint32_t)L;
        }
        break;
      }
      case 8: {                                              // TLEN: int32
        uint32_t k = n && (f[0] == '-' || f[0] == '+') ? 1 : 0;
        if (!dec_u(f + k, n - k, k && f[0] == '-' ? 0x80000000ull : 0x7fffffffull, &val)) fcode = SE_TLEN;
        else val = (unsigned long long)(k && f[0] == '-' ? -(long long)val : (long long)val);
        break;
      }
      case 10: if (n == 0 || (!star && n != lseq)) fcode = SE_QUAL; break;
      default: break;
    }
  }
  // SEQ: * or [A-Za-z=.]+, every lane a stride of the bytes
  bool seq_bad = !code && !seq_star && seq_e == seq_s;
  if (!code && !seq_star) for (uint32_t p = seq_s + lane; p < seq_e; p += 32) seq_bad |= !seq_char(T[p]);
  if (__any_sync(FULL, seq_bad) && lane == 9) fcode = SE_SEQ;
  const uint32_t nops_ = __shfl_sync(FULL, nops, 5), qlen_ = __shfl_sync(FULL, qlen, 5);
  if (lane == 5 && !fcode && nops_ && !seq_star && qlen_ != lseq) fcode = SE_CIGAR_SEQ;
  const unsigned bad = __ballot_sync(FULL, fcode != 0);
  if (!code && bad) code = __shfl_sync(FULL, fcode, __ffs(bad) - 1);    // the first failing field
  // ---- SA / OC values: from the value start to the next tab or the line end ----
  uint32_t sa_at = 0, sl = 0, oc_at = 0, ol = 0;
  const bool any_sa = !code && sh_sa[w] != ~0ull, any_oc = !code && sh_oc[w] != ~0ull;
  if (any_sa) {
    sa_at = (uint32_t)sh_sa[w];
    for (uint32_t p0 = sa_at;; p0 += 32) {
      const uint32_t p = p0 + lane;
      const unsigned hit = __ballot_sync(FULL, p >= e || T[p] == '\t');
      if (hit) { sl = p0 + __ffs(hit) - 1 - sa_at; break; }
    }
  }
  const bool has_sa = sl > 0;
  if (has_sa && any_oc) {
    oc_at = (uint32_t)sh_oc[w];
    for (uint32_t p0 = oc_at;; p0 += 32) {
      const uint32_t p = p0 + lane;
      const unsigned hit = __ballot_sync(FULL, p >= e || T[p] == '\t');
      if (hit) { ol = p0 + __ffs(hit) - 1 - oc_at; break; }
    }
  }
  const long long flag = (long long)__shfl_sync(FULL, val, 1), tidv = (long long)__shfl_sync(FULL, val, 2), posv = (long long)__shfl_sync(FULL, val, 3);
  const long long mapq = (long long)__shfl_sync(FULL, val, 4), mt = (long long)__shfl_sync(FULL, val, 6), mposv = (long long)__shfl_sync(FULL, val, 7);
  const int32_t isize = (int32_t)(long long)__shfl_sync(FULL, val, 8);
  const uint32_t rlen_ = __shfl_sync(FULL, rlen, 5), cig_at = __shfl_sync(FULL, fs, 5), q_len = __shfl_sync(FULL, fe, 0) - s;
  if (lane) return;
  if (code) {
    atomicMin(err, ((unsigned long long)i << 8) | (unsigned)code);
    xf[i] = sf[i] = ncig[i] = salen[i] = oclen[i] = sa_ptr[i] = oc_ptr[i] = seqb[i] = 0u;
    return;
  }
  const long long g = n0 + i;
  const int32_t tid = (int32_t)tidv, pos = (int32_t)(posv - 1);
  C.flag[g] = (uint16_t)flag; C.mapq[g] = (uint8_t)mapq; C.tid[g] = tid; C.pos[g] = pos; C.isize[g] = isize;
  C.endpos[g] = (!(flag & 0x4) && nops_ > 0) ? (int32_t)((uint32_t)pos + rlen_) : pos + 1;      // bam_endpos, sam.c:344-350
  const bool x = !(flag & 0x2) || has_sa;
  xf[i] = x ? 1u : 0u;
  sf[i] = has_sa ? 1u : 0u;
  ncig[i] = has_sa ? nops_ : 0u;
  salen[i] = sl; oclen[i] = has_sa ? ol : 0u;
  sa_ptr[i] = has_sa ? sa_at : 0u;
  oc_ptr[i] = (has_sa && ol) ? oc_at : 0u;
  seqb[i] = has_sa ? (lseq + 1) / 2 : 0u;
  if (x || has_sa) aux[i] = Aux{mt == (1ll << 40) ? tid : (int32_t)mt, (int32_t)(mposv - 1), q_len, cig_at, seq_s, lseq};
}

__global__ void __launch_bounds__(PW * 32) sam_extract_side(const uint8_t *__restrict__ T, const uint32_t *__restrict__ lstart, uint32_t nrec, long long n0, bamdec::Side S,
                                                            const uint32_t *__restrict__ xf, const uint32_t *__restrict__ xo, const uint32_t *__restrict__ sf, const uint32_t *__restrict__ so,
                                                            const uint32_t *__restrict__ ncig, const uint32_t *__restrict__ cigo, const uint32_t *__restrict__ salen, const uint32_t *__restrict__ sao,
                                                            const uint32_t *__restrict__ oclen, const uint32_t *__restrict__ oco, const uint32_t *__restrict__ sa_ptr, const uint32_t *__restrict__ oc_ptr,
                                                            const uint32_t *__restrict__ seqb, const uint32_t *__restrict__ seqo, const Aux *__restrict__ aux)
{
  const unsigned lane = threadIdx.x & 31;
  const uint32_t i = blockIdx.x * PW + (threadIdx.x >> 5);
  if (i >= nrec || (!xf[i] && !sf[i])) return;              // whole warps only
  const Aux a = aux[i];
  if (xf[i] && lane == 0) {
    const long long x = S.x0 + xo[i];
    S.x_rec[x] = (uint32_t)(n0 + i);
    S.x_mtid[x] = a.mtid; S.x_mpos[x] = a.mpos;
    uint64_t h = 0xcbf29ce484222325ULL, h2 = 0x9E3779B97F4A7C15ULL;           // bkid_name_hash (include/breakid_b200.h)
    const uint8_t *q = T + lstart[i];
    for (uint32_t k = 0; k < a.qlen; ++k) {
      uint64_t c = q[k];
      h = (h ^ c) * 0x100000001b3ULL;
      h2 = (h2 ^ c) * 0xff51afd7ed558ccdULL;
      h2 ^= h2 >> 32;
    }
    S.x_nh[2 * x] = h; S.x_nh[2 * x + 1] = h2;
  }
  if (!sf[i]) return;
  const long long s = S.s0 + so[i];
  const uint32_t nc = ncig[i];
  const long long c0 = S.cig0 + cigo[i];
  if (lane == 0) {
    S.sa_rec[s] = (uint32_t)(n0 + i);
    const uint8_t *f = T + a.cig_at;                        // validated by sam_parse
    for (uint32_t k = 0, j = 0; k < nc; ++k) {
      uint32_t L = 0;
      while (f[j] >= '0' && f[j] <= '9') L = L * 10 + (f[j++] - '0');
      S.cig_ops[c0 + k] = (L << 4) | (uint32_t)cigar_op(f[j++]);
    }
    S.cig_off[s + 1] = (uint32_t)(c0 + nc);
  }
  const long long t0 = S.sab0 + sao[i];
  for (uint32_t k = lane; k < salen[i]; k += 32) S.sa_txt[t0 + k] = T[sa_ptr[i] + k];
  const long long q0 = S.ocb0 + oco[i];
  for (uint32_t k = lane; k < oclen[i]; k += 32) S.oc_txt[q0 + k] = T[oc_ptr[i] + k];
  const long long b0 = S.seqb0 + seqo[i];
  for (uint32_t k = lane; k < seqb[i]; k += 32) {
    const uint32_t p = a.seq_at + 2 * k;
    S.seq4[b0 + k] = (uint8_t)((nt16(T[p]) << 4) | (2 * k + 1 < a.lseq ? nt16(T[p + 1]) : 0u));
  }
  if (lane == 0) {
    S.sa_off[s + 1] = (uint32_t)(t0 + salen[i]);
    S.oc_off[s + 1] = (uint32_t)(q0 + oclen[i]);
    S.seq_off[s + 1] = (uint32_t)(b0 + seqb[i]);
    S.seq_len[s] = (int32_t)a.lseq;
  }
}

static const char *err_text(int code)
{
  switch (code) {
    case SE_FIELDS: return "fewer than 11 tab-separated fields";
    case SE_EMPTY: return "empty line";
    case SE_HEADER: return "header line among the alignment lines";
    case SE_QNAME: return "QNAME must have 1..254 characters";
    case SE_FLAG: return "FLAG is not a decimal in 0..65535";
    case SE_RNAME: return "RNAME is empty";
    case SE_RNAME_UNKNOWN: return "RNAME names no @SQ line";
    case SE_POS: return "POS is not a decimal in 0..2^31-1";
    case SE_MAPQ: return "MAPQ is not a decimal in 0..255";
    case SE_CIGAR: return "CIGAR is not * or operations MIDNSHP=X with lengths 1..2^28-1 (at most 65535)";
    case SE_RNEXT: return "RNEXT is empty";
    case SE_RNEXT_UNKNOWN: return "RNEXT names no @SQ line";
    case SE_PNEXT: return "PNEXT is not a decimal in 0..2^31-1";
    case SE_TLEN: return "TLEN is not a 32-bit integer";
    case SE_SEQ: return "SEQ is not * or letters, '=' and '.'";
    case SE_QUAL: return "QUAL is neither * nor as long as SEQ";
    case SE_CIGAR_SEQ: return "CIGAR query length differs from the SEQ length";
    case SE_OPT: return "optional field is not TG:T:VALUE with type one of AifZHB";
    default: return "malformed line";
  }
}

}  // namespace samdec

// the device lookup table of the context's target names, built on the first SAM push
static int sam_names_init(bkid_ctx *c)
{
  bkid_decoder *d = c->dec;
  if (d->names_built) return 0;
  uint32_t cap = 2;
  while (cap < 2u * (uint32_t)c->nt) cap <<= 1;
  std::vector<int32_t> slot(cap, -1);
  std::vector<uint32_t> off(1, 0);
  std::string txt;
  for (int t = 0; t < c->nt; ++t) {
    const std::string &nm = c->names[t];
    txt += nm; off.push_back((uint32_t)txt.size());
    uint32_t h = samdec::name_h32((const uint8_t *)nm.data(), (uint32_t)nm.size()) & (cap - 1);
    while (slot[h] >= 0 && c->names[slot[h]] != nm) h = (h + 1) & (cap - 1);
    if (slot[h] < 0) slot[h] = t;                            // a repeated name resolves to its first target
  }
  cudaStream_t st = c->st;
  TRY(c, d->nm_txt.ensure(txt.size() + 64, 0, st)); TRY(c, d->nm_off.ensure(off.size() * 4 + 64, 0, st)); TRY(c, d->nm_slot.ensure((size_t)cap * 4 + 64, 0, st));
  if (!txt.empty()) CU(c, cudaMemcpy(d->nm_txt.p, txt.data(), txt.size(), cudaMemcpyHostToDevice));
  CU(c, cudaMemcpy(d->nm_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice));
  CU(c, cudaMemcpy(d->nm_slot.p, slot.data(), (size_t)cap * 4, cudaMemcpyHostToDevice));
  d->nm_mask = cap - 1;
  d->names_built = true;
  return 0;
}

static int push_sam_impl(bkid_ctx *c, const uint8_t *text, uint64_t len, int64_t first_line)
{
  using namespace samdec;
  TRY(c, decoder_init(c));
  bkid_decoder *d = c->dec;
  cudaStream_t st = c->st;
  invalidate(c);
  TRY(c, settle_forms(c, 1, 1, 0));                           // wide insert-size / end columns, as the BAM decoder writes them
  memset(&d->stats, 0, sizeof d->stats);
  TRY(c, sam_names_init(c));
  size_t CAP = (size_t)1 << 30;
  if (const char *e = getenv("BKID_SAM_CHUNK_KB")) {           // tests: small chunks exercise the chunk cuts on small texts
    long kb = atol(e);
    if (kb >= 1) CAP = (size_t)kb << 10;
  }
  const uint64_t MAX_CHUNK = 0xffffffffull - 1024;            // in-chunk offsets (and lstart = offset + 1) stay 32-bit
  std::vector<std::pair<uint64_t, uint64_t>> chunks;          // [begin, end): whole lines
  size_t max_chunk = 0;
  for (uint64_t o = 0; o < len;) {
    uint64_t e = std::min<uint64_t>(len, o + CAP);
    if (e < len) {
      const void *nl = memrchr(text + o, '\n', (size_t)(e - o));
      if (nl) e = (uint64_t)((const uint8_t *)nl - text) + 1;
      else {                                                   // one line longer than the chunk size
        nl = memchr(text + e, '\n', (size_t)(len - e));
        e = nl ? (uint64_t)((const uint8_t *)nl - text) + 1 : len;
      }
    }
    if (e - o > MAX_CHUNK) return fail(c, BKID_ERR_IO, "SAM line " + std::to_string(first_line) + "+: a line longer than 4 GiB");
    chunks.push_back({o, e});
    max_chunk = std::max<size_t>(max_chunk, (size_t)(e - o));
    o = e;
  }
  bool pinned = false;
  {
    cudaPointerAttributes pa;
    if (len && cudaPointerGetAttributes(&pa, text) == cudaSuccess) pinned = (pa.type == cudaMemoryTypeHost);
    cudaGetLastError();
  }
  const int slots = chunks.size() > 1 ? 2 : 1;
  for (int k = 0; k < slots; ++k) TRY(c, d->comp[k].ensure(max_chunk + 256, 0, st));
  if (!pinned && !chunks.empty()) TRY(c, ensure_staging(c, max_chunk + 256, slots));
  TRY(c, d->state.ensure(256, 0, st));
  unsigned long long *derr = (unsigned long long *)d->state.as<int>() + 8;
  unsigned long long *tot = (unsigned long long *)(c->counters.as<unsigned>() + CS_TOTAL);
  if (c->n_sa == 0) { TRY(c, reserve_impl(c, c->n, c->n_x, 1, 1, 1, 1)); CU(c, cudaMemsetAsync(c->cig_off.p, 0, 4, st)); CU(c, cudaMemsetAsync(c->sa_off.p, 0, 4, st)); CU(c, cudaMemsetAsync(c->oc_off.p, 0, 4, st)); }

  auto stage_chunk = [&](size_t k) -> int {                   // host copy (pageable input) + async H2D of chunk k into slot k&1
    const int slot = (int)(k & 1);
    const size_t n = (size_t)(chunks[k].second - chunks[k].first);
    CU(c, cudaStreamWaitEvent(d->st_copy, d->ev_free[slot], 0));   // the parse that read this slot has finished
    const uint8_t *src = text + chunks[k].first;
    if (!pinned) {
      CU(c, cudaEventSynchronize(d->ev_h2d[slot]));                 // previous H2D out of this staging buffer done
      memcpy(d->h_stage[slot], src, n);
      src = d->h_stage[slot];
    }
    CU(c, cudaMemcpyAsync(d->comp[slot].p, src, n, cudaMemcpyHostToDevice, d->st_copy));
    CU(c, cudaEventRecord(d->ev_h2d[slot], d->st_copy));
    return 0;
  };
  for (int k = 0; k < 2; ++k) { CU(c, cudaEventRecord(d->ev_free[k], st)); CU(c, cudaEventRecord(d->ev_h2d[k], d->st_copy)); }
  cudaEventRecord(d->ev_t[0], st);
  if (!chunks.empty()) TRY(c, stage_chunk(0));
  const long long n_first = c->n;
  long long line0 = first_line;                               // file line number of the chunk's first line
  float ms_lines = 0, ms_parse = 0;
  for (size_t k = 0; k < chunks.size(); ++k) {
    const int slot = (int)(k & 1);
    const uint32_t L = (uint32_t)(chunks[k].second - chunks[k].first);
    const uint8_t *T = d->comp[slot].as<uint8_t>();
    // ---- line starts ----
    CU(c, cudaStreamWaitEvent(st, d->ev_h2d[slot], 0));
    cudaEventRecord(d->ev_t[1], st);
    const uint32_t ntile = (uint32_t)div_up(L, NL_T * 16);
    TRY(c, c->sc.ensure((long long)ntile + 8, st));
    uint32_t *cnt = c->sc.a32.as<uint32_t>(), *base = c->sc.b32.as<uint32_t>();
    BK_LAUNCH(sam_nl_count, ntile, NL_T, 0, st, T, L, cnt);
    bk::exclusive_scan<uint32_t, uint32_t>(cnt, base, ntile, c->sc.scan_tmp.as<unsigned long long>(), tot, st);
    unsigned long long nnl64 = 0;
    CU(c, cudaMemcpyAsync(&nnl64, tot, 8, cudaMemcpyDeviceToHost, st));
    TRY(c, sync_check(c));
    const uint32_t nnl = (uint32_t)nnl64;
    const uint32_t nrec = nnl + (text[chunks[k].second - 1] != '\n' ? 1u : 0u);
    if ((unsigned long long)(c->n + nrec) >= 0xffffffffull) return fail(c, BKID_ERR_ARG, "more than 2^32-1 records per context");
    TRY(c, d->rec_off.ensure((size_t)(nnl + 1) * 4 + 64, 0, st));
    uint32_t *lstart = d->rec_off.as<uint32_t>();
    BK_LAUNCH(sam_nl_write, ntile, NL_T, 0, st, T, L, base, lstart);
    cudaEventRecord(d->ev_t[2], st);
    // ---- parse ----
    {
      long long want = c->n + nrec;                           // capacity: after the first chunk extrapolate from records per byte
      if (k == 0 && chunks.size() > 1) want = std::max<long long>(want, c->n + (long long)((double)nrec / (double)L * (double)len * 1.03) + 1024);
      want = std::min<long long>(want, 0xfffffffell);
      TRY(c, reserve_impl(c, std::max<long long>(want, c->n + nrec), c->n_x, std::max<long long>(c->n_sa, 1), std::max<long long>(c->n_cig, 1), std::max<long long>(c->sa_bytes, 1), std::max<long long>(c->oc_bytes, 1)));
    }
    for (auto &m : d->meta) TRY(c, m.ensure((size_t)nrec * 4 + 64, 0, st));
    for (auto &m : d->metao) TRY(c, m.ensure((size_t)nrec * 4 + 64, 0, st));
    TRY(c, d->aux.ensure((size_t)nrec * sizeof(Aux) + 64, 0, st));
    TRY(c, c->sc.ensure((long long)nrec + 8, st));
    uint32_t *m[8]; for (int i = 0; i < 8; ++i) m[i] = d->meta[i].as<uint32_t>();        // [5],[6] = SA / OC offsets, [7] = seq bytes
    uint32_t *mo[6]; for (int i = 0; i < 6; ++i) mo[i] = d->metao[i].as<uint32_t>();
    CU(c, cudaMemsetAsync(derr, 0xff, 8, st));
    bamdec::Cols C{c->flag.as<uint16_t>(), c->mapq.as<uint8_t>(), c->tid.as<int32_t>(), c->pos.as<int32_t>(), c->isize.as<int32_t>(), c->endpos.as<int32_t>()};
    Names N{d->nm_txt.as<uint8_t>(), d->nm_off.as<uint32_t>(), d->nm_slot.as<int32_t>(), d->nm_mask};
    Aux *aux = d->aux.as<Aux>();
    if (nrec) BK_LAUNCH(sam_parse, GRID1(nrec, PW), PW * 32, 0, st, T, L, lstart, nnl, nrec, c->n, C, N, m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7], aux, derr);
    unsigned long long *tots = (unsigned long long *)(c->counters.as<unsigned>() + CS_DECODE);     // 6 x u64
    for (int i = 0; i < 5; ++i) bk::exclusive_scan<uint32_t, uint32_t>(m[i], mo[i], nrec, c->sc.scan_tmp.as<unsigned long long>(), tots + i, st);
    bk::exclusive_scan<uint32_t, uint32_t>(m[7], mo[5], nrec, c->sc.scan_tmp.as<unsigned long long>(), tots + 5, st);
    unsigned long long ht[7];
    CU(c, cudaMemcpyAsync(ht, tots, 48, cudaMemcpyDeviceToHost, st));
    CU(c, cudaMemcpyAsync(ht + 6, derr, 8, cudaMemcpyDeviceToHost, st));
    if (k + 1 < chunks.size()) TRY(c, stage_chunk(k + 1));    // the host copy of the next chunk overlaps this parse
    TRY(c, sync_check(c));
    if (ht[6] != ~0ull)
      return fail(c, BKID_ERR_IO, "SAM line " + std::to_string(line0 + (long long)(ht[6] >> 8)) + ": " + err_text((int)(ht[6] & 0xff)));
    TRY(c, reserve_impl(c, c->n + nrec, c->n_x + (long long)ht[0], c->n_sa + (long long)ht[1], c->n_cig + (long long)ht[2], c->sa_bytes + (long long)ht[3], c->oc_bytes + (long long)ht[4]));
    {
      size_t s_new = (size_t)(c->n_sa + (long long)ht[1]);
      TRY(c, c->seq_off.ensure((s_new + 1) * 4 + 64, (size_t)(c->n_sa + 1) * 4, st));
      TRY(c, c->seq_len.ensure(s_new * 4 + 64, (size_t)c->n_sa * 4, st));
      TRY(c, c->seq4.ensure((size_t)c->seq_bytes + (size_t)ht[5] + 64, (size_t)c->seq_bytes, st));
      if (c->n_sa == 0) CU(c, cudaMemsetAsync(c->seq_off.p, 0, 4, st));
    }
    bamdec::Side S{c->x_rec.as<uint32_t>(), c->x_mtid.as<int32_t>(), c->x_mpos.as<int32_t>(), c->x_nh.as<uint64_t>(),
                   c->sa_rec.as<uint32_t>(), c->cig_off.as<uint32_t>(), c->cig_ops.as<uint32_t>(), c->sa_off.as<uint32_t>(), c->oc_off.as<uint32_t>(), c->sa_txt.as<uint8_t>(), c->oc_txt.as<uint8_t>(),
                   c->seq_off.as<uint32_t>(), c->seq4.as<uint8_t>(), c->seq_len.as<int32_t>(),
                   c->n_x, c->n_sa, c->n_cig, c->sa_bytes, c->oc_bytes, c->seq_bytes};
    if (ht[0] || ht[1])
      BK_LAUNCH(sam_extract_side, GRID1(nrec, PW), PW * 32, 0, st, T, lstart, nrec, c->n, S, m[0], mo[0], m[1], mo[1], m[2], mo[2], m[3], mo[3], m[4], mo[4], m[5], m[6], m[7], mo[5], aux);
    CU(c, cudaEventRecord(d->ev_free[slot], st));
    cudaEventRecord(d->ev_t[3], st);
    c->n += nrec; c->n_x += (long long)ht[0]; c->n_sa += (long long)ht[1]; c->n_cig += (long long)ht[2]; c->sa_bytes += (long long)ht[3]; c->oc_bytes += (long long)ht[4];
    c->seq_bytes += (long long)ht[5];
    line0 += nrec;
    TRY(c, sync_check(c));
    float ms = 0;
    cudaEventElapsedTime(&ms, d->ev_t[1], d->ev_t[2]); ms_lines += ms;
    cudaEventElapsedTime(&ms, d->ev_t[2], d->ev_t[3]); ms_parse += ms;
  }
  cudaEventRecord(d->ev_t[5], st);
  TRY(c, sync_check(c));
  CU(c, cudaStreamSynchronize(d->st_copy));
  cudaEventElapsedTime(&d->stats.total_ms, d->ev_t[0], d->ev_t[5]);
  d->stats.boundaries_ms = ms_lines; d->stats.extract_ms = ms_parse;
  d->stats.uncompressed_bytes = (int64_t)len;
  d->stats.n_records = c->n - n_first;
  d->stats.n_chunks = (int64_t)chunks.size();
  c->have_seq = true;                    // like the BAM decoder: the read bases of the SA records are extracted
  return 0;
}

int bkid_push_sam(bkid_ctx *c, const uint8_t *text, uint64_t len, int64_t first_line, int64_t *n_records)
{
  if (!c || (!text && len)) return c ? fail(c, BKID_ERR_ARG, "bad SAM text arguments") : BKID_ERR_ARG;
  cudaSetDevice(c->device);
  c->err.clear();
  if (c->borrowed) return fail(c, BKID_ERR_ARG, "context holds borrowed device columns; bkid_reset first");
  NO_STREAM(c);
  // records are only ever appended: a failed call restores the counts and leaves every column as it was
  const long long n = c->n, n_x = c->n_x, n_sa = c->n_sa, n_cig = c->n_cig, sa_b = c->sa_bytes, oc_b = c->oc_bytes, seq_b = c->seq_bytes;
  int rc = push_sam_impl(c, text, len, first_line);
  if (rc) {
    cudaStreamSynchronize(c->st);
    if (c->dec && c->dec->init) cudaStreamSynchronize(c->dec->st_copy);
    c->n = n; c->n_x = n_x; c->n_sa = n_sa; c->n_cig = n_cig; c->sa_bytes = sa_b; c->oc_bytes = oc_b; c->seq_bytes = seq_b;
  }
  set_ptrs(c);
  if (n_records) *n_records = rc ? 0 : c->n - n;
  return rc;
}
