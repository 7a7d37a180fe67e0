/* breakid_b200.h -- C ABI of the B200 implementation of BreakID's data-parallel core.
 *
 * The reference (SinOncology/BreakID) has no library target, plugin or FFI ("We don't make a
 * library at the moment", reference src/CMakeLists.txt:5): its hot path is a set of C++ free
 * functions called from main() (reference src/BreakID.cc:93-170).  This header is the boundary a
 * maintainer binds instead: each entry point names the reference function(s) it replaces.
 * Plain pointers and sizes only; no C++ or torch types.  One context per GPU; a context is not
 * thread-safe, different contexts are independent.  Every function returns 0 on success and a
 * negative bkid_status on failure (bkid_last_error() gives the message); nothing throws.
 * There is NO CPU fallback: without a usable CUDA device bkid_create() fails.
 *
 * Stage order (mirrors reference main(), src/BreakID.cc:98-170):
 *   bkid_create -> [bkid_reserve] -> bkid_push_batch* -> bkid_insert_stats -> bkid_scan
 *   -> bkid_cluster -> [bkid_set_nib*] -> bkid_refine -> bkid_fetch_clusters -> bkid_destroy
 * or the single call bkid_run() which does insert_stats..refine with dist from the reference's
 * own formula (src/BreakID.cc:103).
 */
#ifndef BREAKID_B200_H
#define BREAKID_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BKID_ABI_VERSION 3

typedef enum {
  BKID_OK = 0,
  BKID_ERR_CUDA = -1,       /* CUDA runtime / no device */
  BKID_ERR_ARG = -2,        /* bad argument or call order */
  BKID_ERR_NOMEM = -3,      /* device memory exhausted (e.g. AHC component too large) */
  BKID_ERR_CIGAR = -4,      /* the reference's fatal "error cigar" path, src/BreakID.cc:954-968 */
  BKID_ERR_HASH = -5,       /* > 4096 records share the 64-bit name hash of different read names (names with equal 64-bit hashes
                               are otherwise told apart by the other 64 bits of the 128-bit hash) */
  BKID_ERR_IO = -6
} bkid_status;

typedef struct bkid_ctx bkid_ctx;

/* BAM header facts the path needs (reference: bam_header_t target_len / target_name as used by
 * src/util_bam.cc:57-68 combine_genome_chr_pos and src/BreakID.cc:1500-1512 bucket naming). */
typedef struct {
  int32_t n_targets;
  const uint32_t *target_len;       /* [n_targets] */
  const char *const *target_name;   /* [n_targets] NUL-terminated */
} bkid_header;

/* Reference command-line parameters (src/BreakID.cc:27-39) plus the constants it hard-codes. */
typedef struct {
  int32_t qual;            /* -q   [20]  src/BreakID.cc:29,1419 */
  int32_t times;           /* -t   [2]   src/BreakID.cc:30,103 */
  int32_t fast;            /* -fast [0]  src/BreakID.cc:35,129 */
  int32_t min_reads;       /* 2          src/BreakID.cc:34 */
  int32_t bp_pos_error;    /* 2          src/BreakID.cc:444-445 */
  int32_t mismatch_num;    /* 10         src/BreakID.cc:891 */
  int32_t sd_mult;         /* 3          the literal in src/BreakID.cc:103 (north_star's -s) */
  int32_t validate_align;  /* 0          extension (north_star kernel 4, not in the reference): 1 = a split alignment only counts as
                              evidence if the soft-clipped bases of the read align to the reference at the position its SA
                              tag claims (banded edit distance, band 8, at most len/10 + 2 edits); needs seq4 + nib */
} bkid_params;

/* One struct-of-arrays batch of decoded alignment records, in BAM file order.  All pointers are
 * borrowed for the duration of the call.  Dense per-record columns (19 B/record) are the bam1_core_t
 * fields every record needs (htslib sam.h:148-157) + bam_endpos (htslib sam.c:344-350).
 * The mate fields and the 128-bit read-name hash (bkid_name_hash; it replaces std::string equality in
 * the mate join, src/BreakID.cc:1424, and the split-read name match, src/BreakID.cc:605) are only ever
 * read for records that can become discordant candidates or split-read evidence, so they travel in a
 * SPARSE table: the host lists every record that is not a proper pair (flag & 0x2 clear -- a superset of
 * the candidate predicate src/BreakID.cc:1419-1420) or carries an SA tag, ~1 % of a normal BAM.  The
 * device re-derives the candidate predicate itself and fails with BKID_ERR_ARG if a candidate is missing
 * from the table.
 * Records carrying an SA:Z tag additionally appear in the SA side table with their raw BAM cigar ops
 * and the raw SA / OC tag text; all CIGAR / SA arithmetic happens on the device. */
typedef struct {
  int64_t n;
  const uint16_t *flag;
  const uint8_t *mapq;
  const int32_t *tid, *pos, *isize, *endpos;
  int64_t n_x;                      /* sparse table of improper / SA-tagged records */
  const uint32_t *x_rec;            /* [n_x] ascending batch-local record index */
  const int32_t *x_mtid, *x_mpos;   /* [n_x] */
  const uint64_t *x_name_hash;      /* [2 n_x]: lo, hi */
  int64_t n_sa;
  const uint32_t *sa_rec;           /* [n_sa] ascending batch-local record index */
  const uint32_t *cig_off;          /* [n_sa+1] into cig_ops */
  const uint32_t *cig_ops;          /* BAM encoding len<<4|op */
  const uint32_t *sa_off;           /* [n_sa+1] into sa_txt */
  const uint8_t *sa_txt;            /* SA:Z value bytes, no terminator */
  const uint32_t *oc_off;           /* [n_sa+1] into oc_txt (all equal when no OC tags) */
  const uint8_t *oc_txt;
  /* Optional narrow encodings of three dense columns for host batches (bkid_push_batch): a non-NULL narrow column
   * REPLACES its wide column (pass that one as NULL); the device widens it after the copy.  19 -> 11 B/record
   * over PCIe.  A decoder uses a narrow form only when the whole batch fits it and sends the wide column otherwise.
   * A context whose batches all carry a column in its narrow form KEEPS it narrow in HBM (the classify kernel then reads
   * 8 B/record including the span maximum the region queries need); bkid_push_batch_device adopts resident isize16 /
   * span16 columns in place (tid must be resident in its wide form). */
  const int16_t *isize16;           /* [n] replaces isize: every isize of a record passing the insert-statistics predicate
                                       (src/BreakID.cc:1932, the only reader of isize) fits int16; other records: any value */
  const uint16_t *span16;           /* [n] replaces endpos: endpos - pos */
  int64_t n_tid_runs;               /* run-length form of tid (records are coordinate sorted: one run per target) */
  const uint32_t *tid_run_start;    /* [n_tid_runs] ascending first record index of each run, [0] = 0 */
  const int32_t *tid_run_tid;       /* [n_tid_runs] */
  /* Optional: read bases of the SA-tagged records, exactly as the BAM record stores them (4-bit codes "=ACMGRSVTWYHKDBN",
   * two per byte, high nibble first), for the banded-alignment evidence validator (bkid_params.validate_align).
   * All three NULL = not provided (the validator then leaves every evidence row as it is). */
  const uint32_t *seq_off;          /* [n_sa+1] byte offsets into seq4 */
  const uint8_t *seq4;
  const int32_t *seq_len;           /* [n_sa] l_seq */
} bkid_batch;

/* A discordant pair (reference struct discordant_pair, src/BreakID.h:39-58) as kept on the device. */
typedef struct {
  uint64_t name_lo, name_hi;
  int32_t p1_tid, p2_tid;
  uint32_t p1_pos, p2_pos;          /* 1-based */
  uint32_t p1_chr_pos, p2_chr_pos;  /* genome-wide, uint32 wrap */
  uint16_t p1_flag, p2_flag;
  uint8_t p1_mapq, p2_mapq;
  uint8_t p1_strand, p2_strand;     /* '+' '-' */
  int32_t bucket;                   /* dense rank of "chrA_chrB" in std::map<string> order */
  int32_t cluster;
  uint32_t orig;                    /* index in scan output order */
  uint32_t _pad;
} bkid_pair;

/* One discordant-scan candidate record (passes src/BreakID.cc:1419-1420), the unit the mate join works on and
 * the unit ranks exchange in the multi-GPU path.  gidx = position in the global coordinate-sorted stream. */
typedef struct {
  uint64_t name_lo, name_hi;
  int32_t tid, pos, mtid, mpos;
  uint64_t gidx;
  uint16_t flag;
  uint8_t mapq;
  uint8_t _pad[5];
} bkid_cand;

/* One called cluster (reference struct cluster_info, src/BreakID.h:60-113), numeric part.  The
 * host driver adds gene annotation (src/BreakID.cc:492-567) and writes the call file. */
typedef struct {
  int32_t bucket;
  int32_t id;
  int32_t p1_tid, p2_tid;
  uint64_t p1_mean_pos, p2_mean_pos;
  uint32_t p1_min_pos, p1_max_pos, p2_min_pos, p2_max_pos;
  uint32_t p1_exact_pos;
  int32_t p2_exact_pos;
  int64_t n_split_read, n_discordant_pair;
  double p1_bp_depth, p2_bp_depth;
  float p1_alle_freq, p2_alle_freq;
  int32_t fusion_type;              /* 0 Unknown 1 Translocation 2 Inversion 3 Duplication 4 Deletion */
  int32_t is_rpt;
  char p1_rpt[44], p2_rpt[44];      /* 41-mer neighbour sequences, NUL padded */
} bkid_cluster_rec;

/* per-stage device timings of the last run, milliseconds (CUDA events) */
typedef struct {
  float h2d, insert_stats, classify, join, bucket_sort, mask, cluster, summarize, evidence, refine, total;
  int64_t n_records, n_candidates, n_pairs, n_masked, n_clustered, n_clusters, n_sa, n_evidence, n_called;
  int64_t kernel_launches;
} bkid_timings;

/* 128-bit read-name hash (FNV-1a 64 + an independent multiply-xorshift 64). */
static inline void bkid_name_hash(const char *s, uint64_t *lo, uint64_t *hi)
{
  uint64_t a = 0xcbf29ce484222325ULL, b = 0x9E3779B97F4A7C15ULL;
  for (; *s; ++s) {
    uint64_t c = (unsigned char)*s;
    a = (a ^ c) * 0x100000001b3ULL;
    b = (b ^ c) * 0xff51afd7ed558ccdULL;
    b ^= b >> 32;
  }
  *lo = a; *hi = b;
}

int bkid_abi_version(void);
const char *bkid_last_error(const bkid_ctx *ctx);       /* ctx may be NULL: last create error */
void bkid_default_params(bkid_params *p);

/* replaces: process start-up in reference main() (src/BreakID.cc:93-112).  The context holds the rank of every
 * "<name>_<name>" bucket string over the header's targets and "*", (n_targets + 1)^2 entries indexed as int32: a header
 * with more than BKID_MAX_TARGETS targets, or one whose table does not fit in host memory, makes it return NULL with
 * the reason in bkid_last_error(NULL).  Equal bucket strings (e.g. "scaf" + "1_2" and "scaf_1" + "2") get one rank,
 * as they are one bucket of the reference's std::map. */
#define BKID_MAX_TARGETS 46339
bkid_ctx *bkid_create(int device, const bkid_header *hdr, const bkid_params *params);
void bkid_destroy(bkid_ctx *ctx);

/* optional capacity hint so pushes never reallocate */
int bkid_reserve(bkid_ctx *ctx, int64_t n_records, int64_t n_x, int64_t n_sa, int64_t n_cig_ops, int64_t sa_bytes, int64_t oc_bytes);
/* replaces: the samread / sam_read1 loops (src/BreakID.cc:1414,1929) as the producer of records.
 * Host pointers; the host->device copy happens inside (pinned staging, async). */
int bkid_push_batch(bkid_ctx *ctx, const bkid_batch *batch);
/* same, but every pointer in `batch` is a DEVICE pointer (already-resident input) */
int bkid_push_batch_device(bkid_ctx *ctx, const bkid_batch *batch);
/* ---- device BGZF / BAM decode (SURVEY.md 8 f-1) ----------------------------------------------------------
 * replaces, as the producer of records: bgzf_read_block + inflate_block (htslib-1.3.1/bgzf.c:545-600,388-419) and
 * bam_read1 (htslib-1.3.1/sam.c:407-441) under the samread / sam_read1 loops of src/BreakID.cc:1414,1929, together
 * with bam_endpos (sam.c:344-350) and bam_aux_get (sam.c:1267-1290) for the SA:Z / OC:Z tags.
 * `file` is the whole BAM file in host memory (mmap or a pinned buffer; pinned memory is copied from directly) and
 * `file_size` its length: every block of the table must lie inside it (payload + CRC32 + ISIZE), else BKID_ERR_IO;
 * `blocks` its BGZF block table in file order (the host only walks the BSIZE / ISIZE fields, see
 * breakid_b200/host/bam_reader.h: bkid_host_bgzf_open), `first_record_uoffset` the offset of the first alignment
 * record in the uncompressed stream (= size of the BAM header).  Compressed bytes are streamed to the device in
 * chunks; inflate, record-boundary search and column extraction run there and append to the context exactly
 * what bkid_push_batch would have been given by a host decoder.  Deflate stream errors, a wrong ISIZE, a CRC32
 * mismatch (checked per block like htslib bgzf.c:404-416), corrupt record sizes and a truncated last record
 * return BKID_ERR_IO. */
typedef struct {
  uint64_t payload_off;             /* file offset of the raw deflate payload (block start + 12 + XLEN) */
  uint32_t payload_len;             /* BSIZE + 1 - 12 - XLEN - 8 */
  uint32_t usize;                   /* ISIZE (<= 65536) */
} bkid_bgzf_block;
typedef struct {
  int64_t n_chunks, n_blocks, compressed_bytes, uncompressed_bytes, n_records;
  float total_ms, inflate_ms, boundaries_ms, extract_ms;
  int32_t seed_repairs, reserved;
} bkid_decode_stats;
int bkid_push_bgzf(bkid_ctx *ctx, const uint8_t *file, uint64_t file_size, const bkid_bgzf_block *blocks, int64_t n_blocks,
                   uint64_t first_record_uoffset, int64_t *n_records);
/* Same for one rank of a multi-GPU job: decode only the records that START inside the uncompressed extent of BGZF blocks
 * [first_block, end_block) (genomic-bin sharding of the file itself, SURVEY.md 8e).  A range that begins mid-stream finds
 * its first record by seeding and reports its stream offset in *first_record_uoff; *next_record_uoff is the offset of
 * the first record of the following range (the walk reads up to 64 blocks past end_block to complete the straddling
 * record).  The caller verifies next_record_uoff[r] == first_record_uoff[r+1] across ranks: with that check the union
 * of the ranges is exactly the record sequence of the whole file. */
int bkid_push_bgzf_range(bkid_ctx *ctx, const uint8_t *file, uint64_t file_size, const bkid_bgzf_block *blocks, int64_t n_blocks,
                         uint64_t first_record_uoffset, int64_t first_block, int64_t end_block, int64_t *n_records,
                         uint64_t *first_record_uoff, uint64_t *next_record_uoff);
int bkid_get_decode_stats(bkid_ctx *ctx, bkid_decode_stats *stats);
/* Extension (the reference reads BAM only): append the records of SAM alignment text, parsed on the device.
 * `text` holds alignment lines only (no header), in host memory (pinned memory is copied from directly, pageable memory
 * through the library's pinned staging); it ends at a line end or at the end of a complete last line.  Every column
 * bkid_fetch_column returns is byte-identical to what bkid_push_bgzf leaves for a BAM holding the same records (SAM spec
 * 1.4 / 4.2): RNAME / RNEXT resolve against the context's target names in header order ("*" -> -1, RNEXT "=" -> the
 * record's own tid), POS / PNEXT are 1-based, SEQ letters become BAM 4-bit codes, the first SA:Z / OC:Z fields give the
 * SA / OC text.  Each line needs at least 11 tab-separated fields; a \r before the newline is dropped.  Anything else
 * (empty or '@' lines, numbers out of range, unknown reference names, bad CIGAR, SEQ / QUAL / CIGAR lengths that
 * disagree, optional fields that are not TG:T:VALUE of type AifZHB) returns BKID_ERR_IO with a message naming the file
 * line (`first_line` = 1-based line number of text[0]) and the field; the context then holds exactly what it held
 * before the call.  bkid_get_decode_stats: uncompressed_bytes = text bytes, boundaries_ms = line split, extract_ms =
 * parse; inflate_ms and compressed_bytes are 0. */
int bkid_push_sam(bkid_ctx *ctx, const uint8_t *text, uint64_t len, int64_t first_line, int64_t *n_records);
/* Extension (the reference requires a coordinate-sorted, indexed BAM): put the records the context holds (every batch
 * pushed so far) into coordinate order on the device.
 * *was_sorted = 1: they already were non-decreasing in (tid as uint32, so tid -1 is last; pos).  Nothing moves: a file
 *   sorted by any tool, with any tie order, runs exactly as it does without the call.
 * Otherwise: stable sort (ties keep push order) by the lexicographic key (tid as uint32, pos + 1, flag & BAM_FREVERSE).
 *   That is the order samtools 1.3.1 `sort` writes (the version the reference vendors): its key is
 *   (uint64_t)tid << 32 | (pos + 1) << 1 | bam_is_rev under a stable merge sort, and the two keys agree for
 *   pos + 1 < 2^30, which covers every human contig.
 * Every dense column is permuted in the form the context holds it (narrow isize16 / span16 stay narrow), x_rec / sa_rec
 * are renumbered, the sparse table and the SA side table (with cig_ops, sa_txt, oc_txt, seq4) are re-emitted in
 * ascending new record index.  Like a push, the call invalidates every stage result; a push after it appends in push
 * order (sort again).  A context holding borrowed device columns (bkid_push_batch_device) gets owned copies; the
 * caller's memory is never written.
 * Errors: a tid outside [-1, n_targets) or pos < -1 -> BKID_ERR_ARG; with 2^30 records or more, one target holding
 * 2^30 records or more -> BKID_ERR_ARG.  All scratch is allocated before the first column is overwritten, so
 * BKID_ERR_ARG and BKID_ERR_NOMEM leave the context exactly as it was.
 * Device scratch (kept by the context for the next call), bytes per record: 24 (keys + push index, sort buffers)
 * + 8 (packed row; 16 when a column is held wide) + 18 (slot maps, flags, offsets; only with sparse / SA rows or
 * 2^30 records or more), plus about 2x the sparse and SA tables; a borrowed context adds its owned columns. */
int bkid_sort_records(bkid_ctx *ctx, int32_t *was_sorted);
/* parity-test getter: one input column of the context by name ("flag", "pos", "x_name_hash", "sa_txt", ...) */
int bkid_fetch_column(bkid_ctx *ctx, const char *name, void *out, int64_t cap_bytes, int64_t *n_bytes);
/* forget all records (keeps allocations) */
int bkid_reset(bkid_ctx *ctx);

/* Extension (BASELINE.json north_star / configs[2]: exclude-BED; the reference has no such filter, SURVEY.md section 0):
 * records whose leftmost coordinate (tid, 0-based pos) lies in one of the half-open intervals [beg, end) are
 * invisible to every stage -- the result is exactly what the reference computes on a BAM from which those records
 * were removed.  Intervals may overlap and come in any order; n_intervals = 0 clears the filter.  Requires the
 * coordinate-sorted record order BreakID needs anyway.  Call before bkid_insert_stats / bkid_run. */
int bkid_set_exclude(bkid_ctx *ctx, int64_t n_intervals, const int32_t *tid, const int32_t *beg, const int32_t *end);
/* replaces get_mean_insert_size (src/BreakID.cc:1909-1954) */
int bkid_insert_stats(bkid_ctx *ctx, double *mean, double *sd);
/* replaces scan_discordant_pairs (src/BreakID.cc:1362-1515): classify, mate join, p1/p2 order, bucket */
int bkid_scan(bkid_ctx *ctx, double w, int64_t *n_pairs);
/* replaces, per bucket, remove_isolated_pairs + find_cluster_pairs_enspan_{ahc,fast} + the summary
 * half of findClusterBreakPointInfoSaTag (src/BreakID.cc:119-144,201-352); mode 0 = AHC, 1 = -fast */
int bkid_cluster(bkid_ctx *ctx, double dist, int mode, int64_t *n_clusters);
/* replaces nib::open/getBase (src/nibtools.cc:7-64): packed 4-bit payload (file bytes after the 8-byte header) */
int bkid_set_nib(bkid_ctx *ctx, int32_t tid, const uint8_t *packed, uint64_t n_bases);
/* replaces findEncompassingReadsAndBreakPointInfo (src/BreakID.cc:390-490: find_sa_reads, find_bp_pair,
 * cal_single_base_depth, AF, fusion type) and the 41-mer / homopolymer part of annotate (:554-561) */
int bkid_refine(bkid_ctx *ctx, double dist, int64_t *n_called);
/* everything from insert stats to refine; dist = times*sqrt(times)*(mean+sd_mult*sd) (src/BreakID.cc:103) */
int bkid_run(bkid_ctx *ctx, double *mean, double *sd, double *dist, int64_t *n_called);

/* results, in the order reference main() appends them (bucket order, then cluster id; src/BreakID.cc:154-161) */
int bkid_fetch_clusters(bkid_ctx *ctx, bkid_cluster_rec *out, int64_t cap, int64_t *n);
/* stage outputs for parity tests: stage 0 = after scan, 1 = after isolated-pair removal, 2 = after clustering */
int bkid_fetch_pairs(bkid_ctx *ctx, int stage, bkid_pair *out, int64_t cap, int64_t *n);
int bkid_fetch_class(bkid_ctx *ctx, uint8_t *out, int64_t cap);   /* per-record class mask of the classify kernel */
int bkid_get_timings(bkid_ctx *ctx, bkid_timings *t);
/* Measurement aid: with profiling on, every kernel the library launches is bracketed by two CUDA events on its own stream.
 * bkid_profile_report writes one "kernel<TAB>launches<TAB>milliseconds" line per kernel name (summed since switched on; the
 * report resets the collection) into buf and returns the size needed.  Process-wide; off by default. */
int bkid_profile_kernels(int on);
int64_t bkid_profile_report(char *buf, int64_t cap);

/* ---- multi-GPU shard entry points -----------------------------------------------------------------
 * One context per rank holds a contiguous slice of the coordinate-sorted record stream (genomic bins).
 * The caller (breakid_b200/dist.py over torch.distributed / NCCL) performs the exchanges named in
 * SURVEY.md 8(e) between these calls; every handed-out pointer is a DEVICE pointer owned by the context
 * and valid until the next call.  Single-GPU bkid_scan / bkid_refine are compositions of the same pieces. */
typedef struct { uint64_t q[11]; } bkid_sarow;        /* opaque 88-byte split-read evidence row (self-contained) */
/* insert statistics of the local records (src/BreakID.cc:1932-1941): sum |isize|, count, sum isize^2 -> all-reduce (sum);
 * max |isize| -> all-reduce (max) */
int bkid_shard_insert_partial(bkid_ctx *ctx, int64_t *sum_abs, int64_t *count, uint64_t *sum_sq, uint64_t *max_abs);
/* upper bound of the binade the truncating sd accumulator (src/BreakID.cc:1913,1944) can reach, from the GLOBAL sums */
int bkid_sd_upper_binade(uint64_t sum_abs, uint64_t count, uint64_t sum_sq, uint64_t max_abs);
/* one streaming pass per rank, all ranks at once, asynchronous: sum floor((|isize| - mean)^2) and the number of records whose
 * rounding could ever add 1 below that binade.  All-reduce (sum) both: when the second sum is 0 -- the normal case -- the
 * accumulator equals the first sum EXACTLY, independent of the record order, and there is no rank-to-rank chain. */
int bkid_shard_sd_fast(bkid_ctx *ctx, double mean, int32_t upper_binade);
int bkid_shard_sd_fast_collect(bkid_ctx *ctx, uint64_t *sum_floor, uint64_t *n_correctable);
/* otherwise: the exact order-dependent replay, block tables on all ranks at once, then chained rank to rank */
int bkid_shard_sd_prepare(bkid_ctx *ctx, double mean);
int bkid_shard_sd_partial(bkid_ctx *ctx, double mean, int64_t t_in, int64_t *t_out);
int bkid_shard_set_stats(bkid_ctx *ctx, double mean, double sd);
int bkid_shard_candidates(bkid_ctx *ctx, uint64_t index_offset, const bkid_cand **dev, int64_t *n);   /* -> all-to-all by name hash */
int bkid_shard_join(bkid_ctx *ctx, const bkid_cand *dev_cand, int64_t n, double w, const bkid_pair **dev_pairs, int64_t *n_pairs);  /* -> all-to-all by bucket owner */
int bkid_shard_set_pairs(bkid_ctx *ctx, const bkid_pair *dev_pairs, int64_t n);                  /* then bkid_cluster() on the owned buckets */
int bkid_shard_clusters(bkid_ctx *ctx, const bkid_cluster_rec **dev, int64_t *n);                /* bucket = GLOBAL name rank -> all-gather */
int bkid_shard_set_clusters(bkid_ctx *ctx, const bkid_cluster_rec *dev, int64_t n);              /* all clusters in global order */
int bkid_shard_sa_rows(bkid_ctx *ctx, const bkid_sarow **dev, int64_t *n);                       /* -> all-gather (coordinate order = rank order) */
int bkid_shard_set_sa_rows(bkid_ctx *ctx, const bkid_sarow *dev, int64_t n);
int bkid_shard_maxspan(bkid_ctx *ctx, int32_t *maxspan);                                         /* -> all-reduce (max) */
int bkid_shard_set_maxspan(bkid_ctx *ctx, int32_t maxspan);
int bkid_shard_coverage(bkid_ctx *ctx, double dist, uint32_t **dev_cov, int64_t *n);             /* partial counts -> all-reduce (sum) in place */
int bkid_shard_vote(bkid_ctx *ctx);
int bkid_shard_depth(bkid_ctx *ctx, uint32_t **dev_depth, int64_t *n);                           /* partial counts -> all-reduce (sum) in place */
int bkid_shard_finish(bkid_ctx *ctx, int64_t *n_called);
int bkid_fetch_bucket_ranks(bkid_ctx *ctx, int32_t *out, int64_t cap, int64_t *nb);
/* plain device/host memcpy on the context's device (lets a caller move shard buffers into its own allocations) */
int bkid_device_copy(bkid_ctx *ctx, void *dst, const void *src, uint64_t bytes);
/* dst[i] = src[idx[i]] for rows of row_bytes (multiple of 16) on the context's device: the send-side permutation of the all-to-all routing */
int bkid_device_gather_rows(bkid_ctx *ctx, void *dst, const void *src, const int64_t *idx, int64_t n, int32_t row_bytes);

/* ---- the sharded path with the exchanges inside the library ------------------------------------------------------------
 * One rank per GPU; rank r holds the r-th genomic bin of the coordinate-sorted record stream (pushed with bkid_push_batch /
 * bkid_push_bgzf_range as usual).  bkid_dist_run is COLLECTIVE: every rank calls it with its own context and communicator
 * and gets the same calls (bkid_fetch_clusters), identical to a single-context run over the whole stream.  The exchanges
 * (all-reduce of the insert sums, all-to-all of candidate records by name-hash owner and of pairs by bucket owner,
 * all-gather of cluster summaries / evidence rows, all-reduce of coverage / depth counts) are NCCL calls on the context's
 * stream: ncclAllReduce and grouped ncclSend / ncclRecv.  libnccl.so.2 is loaded on first use.
 *   one rank per process:  rank 0 calls bkid_comm_nccl_unique_id and hands the 128 bytes to the others (any channel:
 *                          MPI, torch.distributed, a file), then every rank calls bkid_comm_nccl_init;
 *   one process, one host thread per GPU:  bkid_comm_nccl_init_all(devices, world, comms), then bkid_dist_run from the
 *                          rank's own thread, or bkid_dist_run_threads which starts the threads itself;
 *   bkid_comm_local_create: ranks as threads of one process whose contexts may share ONE device -- exchanges are device
 *                          copies behind a barrier.  For tests on a one-GPU box; same code path otherwise. */
typedef struct bkid_comm bkid_comm;
int bkid_comm_nccl_unique_id(uint8_t *id128);
bkid_comm *bkid_comm_nccl_init(const uint8_t *id128, int rank, int world, int device);
int bkid_comm_nccl_init_all(const int *devices, int world, bkid_comm **out);
int bkid_comm_local_create(int world, bkid_comm **out);
void bkid_comm_destroy(bkid_comm *comm);
/* stage_ms (optional, 9 floats): insert statistics, candidates, candidate all-to-all, join, pair all-to-all, mask + cluster,
 * gathers, refinement, total -- host wall clock of this rank */
int bkid_dist_run(bkid_ctx *ctx, bkid_comm *comm, int mode, double *mean, double *sd, double *dist, int64_t *n_called, float *stage_ms);
/* The bucket -> rank table of the pair exchange: longest-processing-time-first on the GLOBAL pairs-per-bucket histogram
 * (index = bucket name rank), cost model m * (1 + log2(m + 1) / 16).  Pure host code, identical on every rank. */
int bkid_lpt_owner_table(const uint64_t *hist, int n_buckets, int world, uint8_t *owner);
int bkid_dist_run_threads(bkid_ctx **ctxs, bkid_comm **comms, int world, int mode, double *mean, double *sd, double *dist, int64_t *n_called);

/* Stand-alone operator entry points (device work on caller host arrays) used by the parity tests:
 * util_cluster / std::sort replay / isolated-pair mask on one bucket. */
int bkid_op_sort_perm(bkid_ctx *ctx, int64_t n, const uint32_t *key, uint32_t *perm);
int bkid_op_remove_isolated(bkid_ctx *ctx, int64_t n, const uint32_t *p1, const uint32_t *p2, double w,
                            uint32_t *out_idx, int64_t *n_out);
int bkid_op_cluster(bkid_ctx *ctx, int mode, int64_t n, const uint32_t *p1, const uint32_t *p2, double thr,
                    uint32_t *out_idx, int32_t *out_cluster, int64_t *n_out, int32_t *n_roots);

/* K6 + the per-bucket call of src/BreakID.cc:146 (findClusterBreakPointInfoSaTag) for a caller that drives the stages
 * bucket by bucket like the reference's main(): `pairs` = the pairs of ONE chr-pair bucket with their cluster ids, grouped
 * by ascending cluster id (src/BreakID.cc:141 sorts by cmp_enspan_id).  Leaves the cluster summaries in the context exactly
 * as bkid_cluster does; bkid_refine + bkid_fetch_clusters then return the bucket's cluster_info records.  Used by
 * include/compat/BreakID_stages.h. */
int bkid_op_summarize(bkid_ctx *ctx, int64_t n, const bkid_pair *pairs, double dist, int64_t *n_clusters);
/* Replace the thresholds used by the next stage calls (the context keeps its records).  src/BreakID.cc passes qual / w /
 * min_reads to every stage function separately; the stage-wise compat layer forwards them through this call. */
int bkid_set_params(bkid_ctx *ctx, const bkid_params *params);

/* Extension (BASELINE.json north_star kernel 4; the reference has no sequence alignment, SURVEY.md 8 f-3): banded
 * unit-cost edit distance of n query strings (e.g. the soft-clipped part of a split read) against their own reference
 * windows, ASCII bases, 'N' never matches.  q / r are the concatenated strings, q_off / r_off their [n+1] offsets,
 * w (<= 15) the band half-width |j - i| <= w.  out[i] = distance, -1 when the length difference exceeds w, -2 when a
 * string is longer than 512.  One warp per pair, anti-diagonal wavefront with warp shuffles.  bkid_refine uses the same
 * kernel as a default-off evidence validator (bkid_params.validate_align + the seq_* table of the batch). */
int bkid_op_banded_align(bkid_ctx *ctx, int64_t n, const uint8_t *q, const uint32_t *q_off, const uint8_t *r, const uint32_t *r_off,
                         int32_t w, int32_t *out);

#ifdef __cplusplus
}
#endif
#endif /* BREAKID_B200_H */
