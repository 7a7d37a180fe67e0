// bam_reader.cc -- host-side BAM decode into the struct-of-arrays batch of include/breakid_b200.h.
//
// Role in the reference: htslib's bgzf inflate + bam_read1 (thirdparty/.../htslib-1.3.1/sam.c:407-441)
// driven by the samread / sam_read1 loops of src/BreakID.cc:1414,1929.  BASELINE.json keeps decode on
// the host; this is a from-scratch multi-threaded BGZF/BAM reader (zlib only) that extracts exactly
// the columns the hot path consumes: the bam1_core_t fields, bam_endpos (sam.c:344-350), a 128-bit
// read-name hash, and for SA-tagged records the raw cigar ops and SA / OC tag text.
//
// BGZF blocks are located by walking the BSIZE fields, inflated in parallel, and record boundaries
// are then walked once; column extraction is parallel over records.
#include "bam_reader.h"

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

namespace {

struct Block { size_t coff; uint32_t csize, usize; size_t uoff; };

inline uint32_t rd32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline uint16_t rd16(const uint8_t *p) { uint16_t v; memcpy(&v, p, 2); return v; }

bool inflate_block(const uint8_t *src, uint32_t csize, uint8_t *dst, uint32_t usize)
{
  // BGZF: 12-byte gzip header + XLEN extra, deflate payload, CRC32, ISIZE
  uint16_t xlen = rd16(src + 10);
  const uint8_t *payload = src + 12 + xlen;
  uint32_t plen = csize - 12 - xlen - 8;
  z_stream zs;
  memset(&zs, 0, sizeof zs);
  if (inflateInit2(&zs, -15) != Z_OK) return false;
  zs.next_in = const_cast<uint8_t *>(payload); zs.avail_in = plen;
  zs.next_out = dst; zs.avail_out = usize;
  int r = inflate(&zs, Z_FINISH);
  inflateEnd(&zs);
  return r == Z_STREAM_END && zs.total_out == usize;
}

template <class F>
void parallel_for(int threads, size_t n, F f)
{
  if (threads <= 1 || n < 2) { f(0, n); return; }
  std::vector<std::thread> th;
  size_t chunk = (n + threads - 1) / threads;
  for (int t = 0; t < threads; ++t) {
    size_t b = t * chunk, e = b + chunk < n ? b + chunk : n;
    if (b >= e) break;
    th.emplace_back([=] { f(b, e); });
  }
  for (auto &x : th) x.join();
}

}  // namespace

struct bkid_host_bam {
  std::vector<uint32_t> target_len;
  std::vector<std::string> names;
  std::vector<const char *> name_ptrs;
  bkid_header hdr;
  std::vector<uint16_t> flag;
  std::vector<uint8_t> mapq;
  std::vector<int32_t> tid, pos, isize, endpos;
  std::vector<uint32_t> x_rec;
  std::vector<int32_t> x_mtid, x_mpos;
  std::vector<uint64_t> x_name_hash;
  std::vector<uint32_t> sa_rec, cig_off, cig_ops, sa_off, oc_off;
  std::vector<uint8_t> sa_txt, oc_txt;
  std::vector<uint32_t> seq_off; std::vector<uint8_t> seq4; std::vector<int32_t> seq_len;      // read bases of the SA records
  int32_t first_l_qseq = 0;
  bkid_batch batch;
  // narrow encodings (include/breakid_b200.h), filled when the whole batch fits them
  std::vector<int16_t> isize16; std::vector<uint16_t> span16; std::vector<uint32_t> run_start; std::vector<int32_t> run_tid;
  bkid_batch batch_narrow;
  double t_inflate = 0, t_parse = 0;
};

static void set_err(char *err, int errlen, const std::string &s)
{
  if (err && errlen > 0) { snprintf(err, errlen, "%s", s.c_str()); }
}

extern "C" bkid_host_bam *bkid_host_read_bam(const char *path, int threads, char *err, int errlen)
{
  if (threads < 1) threads = 1;
  int fd = open(path, O_RDONLY);
  if (fd < 0) { set_err(err, errlen, std::string("cannot open ") + path); return nullptr; }
  struct stat st;
  if (fstat(fd, &st) != 0 || st.st_size <= 0) { close(fd); set_err(err, errlen, std::string("cannot stat ") + path); return nullptr; }
  size_t fsz = (size_t)st.st_size;
  const uint8_t *file = (const uint8_t *)mmap(nullptr, fsz, PROT_READ, MAP_PRIVATE, fd, 0);
  close(fd);
  if (file == MAP_FAILED) { set_err(err, errlen, "mmap failed"); return nullptr; }

  // 1. locate BGZF blocks
  std::vector<Block> blocks;
  size_t off = 0, utotal = 0;
  while (off + 18 <= fsz) {
    const uint8_t *p = file + off;
    if (p[0] != 0x1f || p[1] != 0x8b) { munmap((void *)file, fsz); set_err(err, errlen, "not a BGZF file"); return nullptr; }
    uint16_t xlen = rd16(p + 10);
    uint32_t bsize = 0;
    if (off + 12 + xlen > fsz) { munmap((void *)file, fsz); set_err(err, errlen, "corrupt BGZF block"); return nullptr; }
    for (uint32_t x = 0; x + 4 <= xlen;) {        // find the BC subfield (every subfield must lie inside XLEN)
      const uint8_t *q = p + 12 + x;
      uint16_t slen = rd16(q + 2);
      if (x + 4 + (uint32_t)slen > xlen) break;
      if (q[0] == 'B' && q[1] == 'C' && slen == 2) bsize = (uint32_t)rd16(q + 4) + 1;
      x += 4 + slen;
    }
    if (!bsize || off + bsize > fsz || bsize < 12u + xlen + 8u) { munmap((void *)file, fsz); set_err(err, errlen, "corrupt BGZF block"); return nullptr; }
    uint32_t usize = rd32(p + bsize - 4);
    blocks.push_back(Block{off, bsize, usize, utotal});
    utotal += usize;
    off += bsize;
  }
  // 2. inflate in parallel
  std::vector<uint8_t> u(utotal + 8);
  std::atomic<bool> ok{true};
  std::atomic<size_t> next{0};
  {
    std::vector<std::thread> th;
    for (int t = 0; t < threads; ++t)
      th.emplace_back([&] {
        for (;;) {
          size_t i = next.fetch_add(16);
          if (i >= blocks.size()) break;
          size_t e = i + 16 < blocks.size() ? i + 16 : blocks.size();
          for (; i < e; ++i) {
            const Block &b = blocks[i];
            if (b.usize && !inflate_block(file + b.coff, b.csize, u.data() + b.uoff, b.usize)) ok = false;
          }
        }
      });
    for (auto &x : th) x.join();
  }
  munmap((void *)file, fsz);
  if (!ok) { set_err(err, errlen, "inflate failed"); return nullptr; }

  // 3. header
  bkid_host_bam *h = new bkid_host_bam();
  const uint8_t *p = u.data();
  if (utotal < 12 || memcmp(p, "BAM\1", 4) != 0) { delete h; set_err(err, errlen, "not a BAM file"); return nullptr; }
  size_t o = 4;
  uint32_t l_text = rd32(p + o); o += 4 + l_text;
  uint32_t n_ref = rd32(p + o); o += 4;
  for (uint32_t i = 0; i < n_ref; ++i) {
    uint32_t l_name = rd32(p + o); o += 4;
    h->names.emplace_back((const char *)(p + o)); o += l_name;
    h->target_len.push_back(rd32(p + o)); o += 4;
  }
  // 4. record boundaries
  std::vector<size_t> rec;
  while (o + 4 <= utotal) {
    uint32_t bs = rd32(p + o);
    if (o + 4 + bs > utotal) { delete h; set_err(err, errlen, "truncated BAM record"); return nullptr; }
    rec.push_back(o);
    o += 4 + bs;
  }
  size_t n = rec.size();
  h->flag.resize(n); h->mapq.resize(n);
  h->tid.resize(n); h->pos.resize(n); h->isize.resize(n); h->endpos.resize(n);
  // 5. columns (parallel) + per-thread SA side tables (merged in order afterwards)
  struct Side { std::vector<uint32_t> rec, ncig, cig, salen, oclen; std::vector<uint8_t> sa, oc, seq; std::vector<int32_t> lseq;
                std::vector<uint32_t> xrec; std::vector<int32_t> xmtid, xmpos; std::vector<uint64_t> xhash; };
  int T = threads;
  std::vector<Side> sides(T);
  std::atomic<bool> bad_record{false};
  size_t chunk = (n + T - 1) / (T ? T : 1);
  parallel_for(T, (size_t)T, [&](size_t tb, size_t te) {
    for (size_t t = tb; t < te; ++t) {
      Side &S = sides[t];
      size_t b = t * chunk, e = b + chunk < n ? b + chunk : n;
      for (size_t i = b; i < e; ++i) {
        const uint8_t *r = p + rec[i];
        uint32_t bs = rd32(r);
        int32_t tid = (int32_t)rd32(r + 4), pos = (int32_t)rd32(r + 8);
        uint8_t l_name = r[12], mq = r[13];
        uint16_t n_cig = rd16(r + 16), fl = rd16(r + 18);
        int32_t l_seq = (int32_t)rd32(r + 20);
        // bam_read1 (sam.c:427-429) rejects l_qseq < 0, l_qname < 1 and fixed fields that do not fit the record
        if (l_seq < 0 || l_name < 1 || 32ull + l_name + 4ull * n_cig + (uint64_t)((l_seq + 1) / 2) + (uint64_t)l_seq > bs) { bad_record = true; continue; }
        h->tid[i] = tid; h->pos[i] = pos; h->mapq[i] = mq; h->flag[i] = fl;
        h->isize[i] = (int32_t)rd32(r + 32);
        const char *qn = (const char *)(r + 36);
        const uint8_t *cg = r + 36 + l_name;
        int32_t rlen = 0;
        for (uint32_t k = 0; k < n_cig; ++k) {
          uint32_t c = rd32(cg + 4 * k), op = c & 0xf;
          if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rlen += (int32_t)(c >> 4);
        }
        h->endpos[i] = (!(fl & 0x4) && n_cig > 0) ? pos + rlen : pos + 1;   // bam_endpos, sam.c:344-350
        // aux scan for SA:Z / OC:Z (first occurrence, like bam_aux_get)
        const uint8_t *a = cg + 4 * (size_t)n_cig + (size_t)((l_seq + 1) / 2) + (size_t)l_seq;
        const uint8_t *end = r + 4 + bs;
        const uint8_t *sa = nullptr, *oc = nullptr;
        while (a + 3 <= end) {
          uint8_t t0 = a[0], t1 = a[1], ty = a[2];
          const uint8_t *v = a + 3;
          size_t len;
          switch (ty) {
            case 'A': case 'c': case 'C': len = 1; break;
            case 's': case 'S': len = 2; break;
            case 'i': case 'I': case 'f': len = 4; break;
            case 'd': len = 8; break;
            case 'Z': case 'H': len = strnlen((const char *)v, end - v) + 1; break;
            case 'B': {
              if (v + 5 > end) { len = (size_t)(end - v); break; }
              uint8_t st = v[0]; uint32_t cnt = rd32(v + 1);
              size_t es = (st == 'c' || st == 'C') ? 1 : (st == 's' || st == 'S') ? 2 : 4;
              len = 5 + es * cnt; break;
            }
            default: len = (size_t)(end - v); break;
          }
          if (ty == 'Z') {
            if (t0 == 'S' && t1 == 'A' && !sa) sa = v;
            if (t0 == 'O' && t1 == 'C' && !oc) oc = v;
          }
          if (len > (size_t)(end - v)) break;
          a = v + len;
        }
        // an unterminated Z value (no NUL inside the record) is corrupt
        if ((sa && strnlen((const char *)sa, end - sa) == (size_t)(end - sa)) || (oc && strnlen((const char *)oc, end - oc) == (size_t)(end - oc))) { bad_record = true; continue; }
        bool has_sa = sa && sa[0];
        if (!(fl & 0x2) || has_sa) {             // sparse table: mate fields + name hash only where they can ever be read
          uint64_t lo, hi;
          {                                    // bkid_name_hash over at most l_name bytes (a name without NUL cannot run past its field)
            uint64_t a = 0xcbf29ce484222325ULL, b = 0x9E3779B97F4A7C15ULL;
            for (uint32_t k = 0; k < l_name && qn[k]; ++k) { uint64_t ch = (unsigned char)qn[k]; a = (a ^ ch) * 0x100000001b3ULL; b = (b ^ ch) * 0xff51afd7ed558ccdULL; b ^= b >> 32; }
            lo = a; hi = b;
          }
          S.xrec.push_back((uint32_t)i); S.xmtid.push_back((int32_t)rd32(r + 24)); S.xmpos.push_back((int32_t)rd32(r + 28));
          S.xhash.push_back(lo); S.xhash.push_back(hi);
        }
        if (has_sa) {                            // saTag() != "" (src/BreakID.cc:896-898)
          S.rec.push_back((uint32_t)i);
          S.ncig.push_back(n_cig);
          for (uint32_t k = 0; k < n_cig; ++k) S.cig.push_back(rd32(cg + 4 * k));
          size_t sl = strlen((const char *)sa);
          S.salen.push_back((uint32_t)sl);
          S.sa.insert(S.sa.end(), sa, sa + sl);
          size_t ol = oc ? strlen((const char *)oc) : 0;
          S.oclen.push_back((uint32_t)ol);
          if (ol) S.oc.insert(S.oc.end(), oc, oc + ol);
          const uint8_t *sq = cg + 4 * (size_t)n_cig;
          S.lseq.push_back(l_seq);
          S.seq.insert(S.seq.end(), sq, sq + (size_t)((l_seq + 1) / 2));
        }
        if (i == 0) h->first_l_qseq = l_seq;
      }
    }
  });
  if (bad_record) { delete h; set_err(err, errlen, "corrupt BAM record (fields do not fit block_size or unterminated tag)"); return nullptr; }
  h->cig_off.push_back(0); h->sa_off.push_back(0); h->oc_off.push_back(0); h->seq_off.push_back(0);
  for (Side &S : sides) {
    size_t ci = 0;
    for (size_t k = 0; k < S.rec.size(); ++k) {
      h->sa_rec.push_back(S.rec[k]);
      for (uint32_t c = 0; c < S.ncig[k]; ++c) h->cig_ops.push_back(S.cig[ci++]);
      h->cig_off.push_back((uint32_t)h->cig_ops.size());
      h->sa_off.push_back(h->sa_off.back() + S.salen[k]);
      h->oc_off.push_back(h->oc_off.back() + S.oclen[k]);
      h->seq_len.push_back(S.lseq[k]);
      h->seq_off.push_back(h->seq_off.back() + (uint32_t)((S.lseq[k] + 1) / 2));
    }
    h->seq4.insert(h->seq4.end(), S.seq.begin(), S.seq.end());
    h->sa_txt.insert(h->sa_txt.end(), S.sa.begin(), S.sa.end());
    h->oc_txt.insert(h->oc_txt.end(), S.oc.begin(), S.oc.end());
    h->x_rec.insert(h->x_rec.end(), S.xrec.begin(), S.xrec.end());
    h->x_mtid.insert(h->x_mtid.end(), S.xmtid.begin(), S.xmtid.end());
    h->x_mpos.insert(h->x_mpos.end(), S.xmpos.begin(), S.xmpos.end());
    h->x_name_hash.insert(h->x_name_hash.end(), S.xhash.begin(), S.xhash.end());
  }
  for (auto &s : h->names) h->name_ptrs.push_back(s.c_str());
  h->hdr.n_targets = (int32_t)h->names.size();
  h->hdr.target_len = h->target_len.data();
  h->hdr.target_name = h->name_ptrs.data();
  bkid_batch &B = h->batch;
  B.n = (int64_t)n;
  B.flag = h->flag.data(); B.mapq = h->mapq.data();
  B.tid = h->tid.data(); B.pos = h->pos.data();
  B.isize = h->isize.data(); B.endpos = h->endpos.data();
  B.n_x = (int64_t)h->x_rec.size();
  B.x_rec = h->x_rec.data(); B.x_mtid = h->x_mtid.data(); B.x_mpos = h->x_mpos.data(); B.x_name_hash = h->x_name_hash.data();
  B.n_sa = (int64_t)h->sa_rec.size();
  B.sa_rec = h->sa_rec.data(); B.cig_off = h->cig_off.data(); B.cig_ops = h->cig_ops.data();
  B.sa_off = h->sa_off.data(); B.sa_txt = h->sa_txt.data();
  B.oc_off = h->oc_off.data(); B.oc_txt = h->oc_txt.data();
  B.isize16 = nullptr; B.span16 = nullptr; B.n_tid_runs = 0; B.tid_run_start = nullptr; B.tid_run_tid = nullptr;
  B.seq_off = h->seq_off.data(); B.seq4 = h->seq4.data(); B.seq_len = h->seq_len.data();
  // narrow forms: 19 -> 11 B/record over PCIe when every value fits
  h->batch_narrow = B;
  {
    bool span_ok = true, isz_ok = true;
    for (size_t i = 0; i < n && (span_ok || isz_ok); ++i) {
      int64_t sp = (int64_t)h->endpos[i] - (int64_t)h->pos[i];
      if (sp < 0 || sp > 65535) span_ok = false;
      uint16_t fl = h->flag[i];
      bool read_isize = (fl & 0x1) && (fl & 0x2) && !(fl & (0x4 | 0x100 | 0x200 | 0x400));       // src/BreakID.cc:1932
      if (read_isize && (h->isize[i] < -32768 || h->isize[i] > 32767)) isz_ok = false;
    }
    if (span_ok && n) { h->span16.resize(n); for (size_t i = 0; i < n; ++i) h->span16[i] = (uint16_t)(h->endpos[i] - h->pos[i]); h->batch_narrow.span16 = h->span16.data(); h->batch_narrow.endpos = nullptr; }
    if (isz_ok && n) {
      h->isize16.resize(n);
      for (size_t i = 0; i < n; ++i) { int32_t v = h->isize[i]; h->isize16[i] = (int16_t)(v < -32768 ? -32768 : v > 32767 ? 32767 : v); }
      h->batch_narrow.isize16 = h->isize16.data(); h->batch_narrow.isize = nullptr;
    }
    for (size_t i = 0; i < n; ++i)
      if (i == 0 || h->tid[i] != h->tid[i - 1]) { h->run_start.push_back((uint32_t)i); h->run_tid.push_back(h->tid[i]); }
    if (n && h->run_start.size() <= 65536) {
      h->batch_narrow.n_tid_runs = (int64_t)h->run_start.size(); h->batch_narrow.tid_run_start = h->run_start.data(); h->batch_narrow.tid_run_tid = h->run_tid.data();
      h->batch_narrow.tid = nullptr;
    }
  }
  return h;
}

extern "C" const bkid_header *bkid_host_bam_header(const bkid_host_bam *h) { return &h->hdr; }
extern "C" const bkid_batch *bkid_host_bam_batch(const bkid_host_bam *h) { return &h->batch; }
extern "C" const bkid_batch *bkid_host_bam_batch_narrow(const bkid_host_bam *h) { return &h->batch_narrow; }
extern "C" void bkid_host_bam_free(bkid_host_bam *h) { delete h; }

// ---- host half of the device decode path ----------------------------------------------------------------
struct bkid_host_bgzf {
  const uint8_t *file = nullptr; size_t fsz = 0;
  bool mapped = false;
  std::vector<bkid_bgzf_block> blocks;
  std::vector<uint32_t> target_len;
  std::vector<std::string> names;
  std::vector<const char *> name_ptrs;
  bkid_header hdr;
  uint64_t first_record = 0, usize = 0;
  int32_t first_l_qseq = -1;
};

// the one BGZF block walker (SAM spec 4.1): the whole blocks at the front of buf[0, len) are appended to `out` with
// payload_off relative to buf; returns the bytes they span (an incomplete trailing block is not consumed), or -1 with
// `msg` when a block header is not BGZF (magic, FEXTRA, BC subfield, BSIZE)
static int64_t bgzf_walk(const uint8_t *buf, uint64_t len, std::vector<bkid_bgzf_block> &out, std::string &msg)
{
  uint64_t off = 0;
  while (off + 18 <= len) {
    const uint8_t *p = buf + off;
    if (p[0] != 0x1f || p[1] != 0x8b) { msg = "not a BGZF file"; return -1; }
    if (!(p[3] & 4)) { msg = "corrupt BGZF block (no extra field: plain gzip is not BGZF)"; return -1; }
    uint16_t xlen = rd16(p + 10);
    if (off + 12 + xlen > len) break;
    uint32_t bsize = 0;
    for (uint32_t x = 0; x + 4 <= xlen;) {        // find the BC subfield (every subfield must lie inside XLEN)
      const uint8_t *q = p + 12 + x;
      uint16_t slen = rd16(q + 2);
      if (x + 4 + (uint32_t)slen > xlen) break;
      if (q[0] == 'B' && q[1] == 'C' && slen == 2) bsize = (uint32_t)rd16(q + 4) + 1;
      x += 4 + slen;
    }
    if (!bsize || bsize < 12u + xlen + 8u) { msg = "corrupt BGZF block (no BC subfield or BSIZE too small)"; return -1; }
    if (off + bsize > len) break;
    bkid_bgzf_block b;
    b.payload_off = off + 12 + xlen; b.payload_len = bsize - 12 - xlen - 8; b.usize = rd32(p + bsize - 4);
    out.push_back(b);
    off += bsize;
  }
  return (int64_t)off;
}

// BAM header (SAM spec 4.2) from the leading blocks: zlib on just enough of them.  1 = parsed, 0 = the blocks end
// before the header does (need more bytes; `complete` = they are the whole stream: an error instead), -1 = error in msg
static int bam_header_parse(bkid_host_bgzf *h, const uint8_t *buf, const bkid_bgzf_block *blocks, int64_t n_blocks, bool complete, std::string &msg)
{
  std::vector<uint8_t> u;
  int64_t nb = 0;
  bool bad = false;
  auto need = [&](size_t bytes) -> bool {
    while (u.size() < bytes && nb < n_blocks && !bad) {
      const bkid_bgzf_block &b = blocks[nb++];
      size_t o = u.size();
      u.resize(o + b.usize);
      if (b.usize) {
        z_stream zs; memset(&zs, 0, sizeof zs);
        if (inflateInit2(&zs, -15) != Z_OK) { bad = true; break; }
        zs.next_in = const_cast<uint8_t *>(buf + b.payload_off); zs.avail_in = b.payload_len;
        zs.next_out = u.data() + o; zs.avail_out = b.usize;
        int r = inflate(&zs, Z_FINISH);
        inflateEnd(&zs);
        if (r != Z_STREAM_END || zs.total_out != b.usize) bad = true;
      }
    }
    return !bad && u.size() >= bytes;
  };
  auto short_of = [&](const char *what) -> int {             // the data ran out (or did not inflate) before `bytes`
    if (bad || complete) { msg = what; return -1; }
    return 0;
  };
  h->names.clear(); h->target_len.clear(); h->name_ptrs.clear();
  if (!need(12)) return short_of("not a BAM file");
  if (memcmp(u.data(), "BAM\1", 4) != 0) { msg = "not a BAM file"; return -1; }
  size_t o = 4;
  uint32_t l_text = rd32(u.data() + o); o += 4;
  if (!need(o + l_text + 4)) return short_of("truncated BAM header");
  o += l_text;
  uint32_t n_ref = rd32(u.data() + o); o += 4;
  for (uint32_t i = 0; i < n_ref; ++i) {
    if (!need(o + 4)) return short_of("truncated BAM header");
    uint32_t l_name = rd32(u.data() + o); o += 4;
    if (!need(o + l_name + 4)) return short_of("truncated BAM header");
    h->names.emplace_back((const char *)(u.data() + o)); o += l_name;
    h->target_len.push_back(rd32(u.data() + o)); o += 4;
  }
  h->first_record = o;
  if (need(o + 36)) h->first_l_qseq = (int32_t)rd32(u.data() + o + 20);
  for (auto &s : h->names) h->name_ptrs.push_back(s.c_str());
  h->hdr.n_targets = (int32_t)h->names.size();
  h->hdr.target_len = h->target_len.data();
  h->hdr.target_name = h->name_ptrs.data();
  return 1;
}

extern "C" int64_t bkid_host_bgzf_walk(const uint8_t *buf, uint64_t len, bkid_bgzf_block *out, int64_t cap, int64_t *n_blocks, char *err, int errlen)
{
  std::vector<bkid_bgzf_block> v;
  std::string msg;
  int64_t used = bgzf_walk(buf, len, v, msg);
  if (used < 0) { set_err(err, errlen, msg); if (n_blocks) *n_blocks = 0; return -1; }
  if ((int64_t)v.size() > cap) {                             // a table that does not fit: consume only the blocks it holds
    v.resize((size_t)std::max<int64_t>(cap, 0));
    used = v.empty() ? 0 : (int64_t)(v.back().payload_off + v.back().payload_len + 8);
  }
  if (!v.empty()) memcpy(out, v.data(), v.size() * sizeof(bkid_bgzf_block));
  if (n_blocks) *n_blocks = (int64_t)v.size();
  return used;
}

extern "C" bkid_host_bgzf *bkid_host_bgzf_parse(const uint8_t *buf, const bkid_bgzf_block *blocks, int64_t n_blocks, int *need_more, char *err, int errlen)
{
  bkid_host_bgzf *h = new bkid_host_bgzf();
  std::string msg;
  int r = bam_header_parse(h, buf, blocks, n_blocks, false, msg);
  if (need_more) *need_more = r == 0;
  if (r != 1) { if (r < 0) set_err(err, errlen, msg); delete h; return nullptr; }
  return h;
}

extern "C" bkid_host_bgzf *bkid_host_bgzf_open(const char *path, char *err, int errlen)
{
  int fd = open(path, O_RDONLY);
  if (fd < 0) { set_err(err, errlen, std::string("cannot open ") + path); return nullptr; }
  struct stat st;
  if (fstat(fd, &st) != 0 || st.st_size <= 0) { close(fd); set_err(err, errlen, std::string("cannot stat ") + path); return nullptr; }
  size_t fsz = (size_t)st.st_size;
  const uint8_t *file = (const uint8_t *)mmap(nullptr, fsz, PROT_READ, MAP_PRIVATE, fd, 0);
  close(fd);
  if (file == MAP_FAILED) { set_err(err, errlen, "mmap failed"); return nullptr; }
  bkid_host_bgzf *h = new bkid_host_bgzf();
  h->file = file; h->fsz = fsz; h->mapped = true;
  auto bail = [&](const std::string &msg) -> bkid_host_bgzf * { set_err(err, errlen, msg); munmap((void *)file, fsz); delete h; return nullptr; };
  std::string msg;
  int64_t used = bgzf_walk(file, fsz, h->blocks, msg);
  if (used < 0) return bail(msg);
  if ((uint64_t)used != fsz) return bail(fsz - (uint64_t)used < 18 ? "trailing bytes after the last BGZF block" : "corrupt BGZF block");
  for (const bkid_bgzf_block &b : h->blocks) h->usize += b.usize;
  if (bam_header_parse(h, file, h->blocks.data(), (int64_t)h->blocks.size(), true, msg) != 1) return bail(msg);
  return h;
}
extern "C" const bkid_header *bkid_host_bgzf_header(const bkid_host_bgzf *h) { return &h->hdr; }
extern "C" const uint8_t *bkid_host_bgzf_data(const bkid_host_bgzf *h) { return h->file; }
extern "C" uint64_t bkid_host_bgzf_size(const bkid_host_bgzf *h) { return h->fsz; }
extern "C" const bkid_bgzf_block *bkid_host_bgzf_blocks(const bkid_host_bgzf *h) { return h->blocks.data(); }
extern "C" int64_t bkid_host_bgzf_n_blocks(const bkid_host_bgzf *h) { return (int64_t)h->blocks.size(); }
extern "C" uint64_t bkid_host_bgzf_first_record(const bkid_host_bgzf *h) { return h->first_record; }
extern "C" uint64_t bkid_host_bgzf_usize(const bkid_host_bgzf *h) { return h->usize; }
extern "C" int32_t bkid_host_bgzf_first_l_qseq(const bkid_host_bgzf *h) { return h->first_l_qseq; }
extern "C" void bkid_host_bgzf_close(bkid_host_bgzf *h)
{
  if (!h) return;
  if (h->mapped) munmap((void *)h->file, h->fsz);
  delete h;
}

// ---- host half of the SAM path (bkid_push_sam): the @SQ lines of the header become the target table ----------
struct bkid_host_sam {
  const uint8_t *data = nullptr; size_t size = 0;
  bool mapped = false;
  std::vector<uint32_t> target_len;
  std::vector<std::string> names;
  std::vector<const char *> name_ptrs;
  bkid_header hdr;
  uint64_t first_record = 0;
  int64_t first_line = 1;
};

static bool sam_parse_header(bkid_host_sam *h, std::string &msg)
{
  const char *p = (const char *)h->data, *end = p + h->size;
  int64_t line = 1;
  std::vector<std::string> seen;
  while (p < end && *p == '@') {
    const char *nl = (const char *)memchr(p, '\n', (size_t)(end - p));
    const char *le = nl ? nl : end;
    std::string ln(p, (size_t)(le - p));
    if (!ln.empty() && ln.back() == '\r') ln.pop_back();
    if (ln.compare(0, 4, "@SQ\t") == 0) {
      std::string sn, lnv;
      bool have_sn = false, have_ln = false;
      for (size_t a = 4; a <= ln.size();) {
        size_t b = ln.find('\t', a);
        if (b == std::string::npos) b = ln.size();
        std::string f = ln.substr(a, b - a);
        if (f.compare(0, 3, "SN:") == 0 && !have_sn) { sn = f.substr(3); have_sn = true; }
        if (f.compare(0, 3, "LN:") == 0 && !have_ln) { lnv = f.substr(3); have_ln = true; }
        a = b + 1;
      }
      const std::string where = "header line " + std::to_string(line) + ": ";
      if (!have_sn || sn.empty()) { msg = where + "@SQ without SN"; return false; }
      if (!have_ln) { msg = where + "@SQ " + sn + " without LN"; return false; }
      unsigned long long v = 0;
      bool ok = !lnv.empty() && lnv.size() <= 10;
      for (char ch : lnv) { ok = ok && ch >= '0' && ch <= '9'; v = v * 10 + (unsigned)(ch - '0'); }
      if (!ok || v > 0x7fffffffull) { msg = where + "LN of " + sn + " is not a number in 0..2^31-1"; return false; }
      for (const std::string &s : h->names)
        if (s == sn) { msg = where + "duplicate @SQ SN " + sn; return false; }
      h->names.push_back(sn);
      h->target_len.push_back((uint32_t)v);
    }
    ++line;
    p = nl ? nl + 1 : end;
  }
  h->first_record = (uint64_t)(p - (const char *)h->data);
  h->first_line = line;
  for (auto &s : h->names) h->name_ptrs.push_back(s.c_str());
  h->hdr.n_targets = (int32_t)h->names.size();
  h->hdr.target_len = h->target_len.data();
  h->hdr.target_name = h->name_ptrs.data();
  return true;
}

extern "C" bkid_host_sam *bkid_host_sam_open(const char *path, char *err, int errlen)
{
  int fd = open(path, O_RDONLY);
  if (fd < 0) { set_err(err, errlen, std::string("cannot open ") + path); return nullptr; }
  struct stat st;
  if (fstat(fd, &st) != 0 || st.st_size <= 0) { close(fd); set_err(err, errlen, std::string("cannot stat ") + path + " (or it is empty)"); return nullptr; }
  size_t fsz = (size_t)st.st_size;
  const uint8_t *file = (const uint8_t *)mmap(nullptr, fsz, PROT_READ, MAP_PRIVATE, fd, 0);
  close(fd);
  if (file == MAP_FAILED) { set_err(err, errlen, "mmap failed"); return nullptr; }
  bkid_host_sam *h = new bkid_host_sam();
  h->data = file; h->size = fsz; h->mapped = true;
  std::string msg;
  if (!sam_parse_header(h, msg)) { set_err(err, errlen, msg.c_str()); munmap((void *)file, fsz); delete h; return nullptr; }
  return h;
}

extern "C" bkid_host_sam *bkid_host_sam_parse(const uint8_t *buf, uint64_t len, char *err, int errlen)
{
  bkid_host_sam *h = new bkid_host_sam();
  h->data = buf; h->size = (size_t)len;
  std::string msg;
  if (!sam_parse_header(h, msg)) { set_err(err, errlen, msg.c_str()); delete h; return nullptr; }
  return h;
}

extern "C" const bkid_header *bkid_host_sam_header(const bkid_host_sam *h) { return &h->hdr; }
extern "C" const uint8_t *bkid_host_sam_data(const bkid_host_sam *h) { return h->data; }
extern "C" uint64_t bkid_host_sam_size(const bkid_host_sam *h) { return h->size; }
extern "C" uint64_t bkid_host_sam_first_record(const bkid_host_sam *h) { return h->first_record; }
extern "C" int64_t bkid_host_sam_first_line(const bkid_host_sam *h) { return h->first_line; }
extern "C" void bkid_host_sam_close(bkid_host_sam *h)
{
  if (!h) return;
  if (h->mapped) munmap((void *)h->data, h->size);
  delete h;
}
