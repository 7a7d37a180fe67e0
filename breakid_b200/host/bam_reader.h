// bam_reader.h -- host BAM decode -> bkid_batch (see bam_reader.cc)
#pragma once
#include "../../include/breakid_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bkid_host_bam bkid_host_bam;

/* Decode a whole BAM into one record batch.  Returns NULL and fills `err` on failure. */
bkid_host_bam *bkid_host_read_bam(const char *path, int threads, char *err, int errlen);
const bkid_header *bkid_host_bam_header(const bkid_host_bam *h);
const bkid_batch *bkid_host_bam_batch(const bkid_host_bam *h);            /* wide columns */
const bkid_batch *bkid_host_bam_batch_narrow(const bkid_host_bam *h);     /* same batch, narrow encodings where the data fits (11 B/record) */
void bkid_host_bam_free(bkid_host_bam *h);


/* Host half of the device decode path (bkid_push_bgzf): mmap the file, walk the BGZF block headers (BSIZE / ISIZE)
 * into a block table and inflate just enough leading blocks (zlib) to parse the BAM header.  Nothing else is
 * decompressed on the host. */
typedef struct bkid_host_bgzf bkid_host_bgzf;
bkid_host_bgzf *bkid_host_bgzf_open(const char *path, char *err, int errlen);
const bkid_header *bkid_host_bgzf_header(const bkid_host_bgzf *h);
const uint8_t *bkid_host_bgzf_data(const bkid_host_bgzf *h);            /* the mapped file */
uint64_t bkid_host_bgzf_size(const bkid_host_bgzf *h);
const bkid_bgzf_block *bkid_host_bgzf_blocks(const bkid_host_bgzf *h);
int64_t bkid_host_bgzf_n_blocks(const bkid_host_bgzf *h);
uint64_t bkid_host_bgzf_first_record(const bkid_host_bgzf *h);          /* uncompressed offset of the first record */
uint64_t bkid_host_bgzf_usize(const bkid_host_bgzf *h);                 /* total uncompressed size */
int32_t bkid_host_bgzf_first_l_qseq(const bkid_host_bgzf *h);           /* read length of the first record (driver's _params.txt), -1 if none */
void bkid_host_bgzf_close(bkid_host_bgzf *h);

/* Host half of the SAM path (bkid_push_sam): the header's @SQ SN:/LN: lines become the target table in @SQ order
 * (other header lines are ignored; a duplicate SN, an @SQ without SN, or a missing or non-numeric LN is an error).
 * The alignment lines start at first_record, on file line first_line (1-based).  A file without header lines is valid
 * (it has no targets: every RNAME must be *).  bkid_host_sam_open maps a file; bkid_host_sam_parse reads the header
 * lines at the start of a caller-owned buffer (e.g. what was read from stdin) and keeps pointing into it. */
typedef struct bkid_host_sam bkid_host_sam;
bkid_host_sam *bkid_host_sam_open(const char *path, char *err, int errlen);
bkid_host_sam *bkid_host_sam_parse(const uint8_t *buf, uint64_t len, char *err, int errlen);
const bkid_header *bkid_host_sam_header(const bkid_host_sam *h);
const uint8_t *bkid_host_sam_data(const bkid_host_sam *h);              /* the mapped file / the buffer */
uint64_t bkid_host_sam_size(const bkid_host_sam *h);
uint64_t bkid_host_sam_first_record(const bkid_host_sam *h);            /* offset of the first alignment line */
int64_t bkid_host_sam_first_line(const bkid_host_sam *h);               /* its 1-based line number */
void bkid_host_sam_close(bkid_host_sam *h);

#ifdef __cplusplus
}
#endif
