/*
 * smc_bamio.h -- C ABI of libsmc_bamio.so: BAM (BGZF) -> the flat read buffers of smc_reads_soa (include/smc_b200.h).
 *
 * Host-side input decoding for the calling path: replaces what the reference obtains from pysam per pileup read
 * (pysam.AlignmentFile(bamFile) + pileup(), smCounter.py:275,316-349: qname, flag, mapq, cigar, query_sequence,
 * query_qualities, tags) with ONE decode per BAM record.  Read identity follows smCounter.py:319-325
 * (BC = qname.split(':')[-2], readid = ':'.join(parts[:-2])), NM follows :329-334 (first NM tag, else 0).
 * Unmapped records are dropped (htslib never piles them up); nothing else is filtered (stepper='nofilter').
 *
 * BGZF blocks are inflated by `threads` host threads (zlib) and every pass of the record decode runs on the same number of
 * threads (record boundaries per byte range with a verified speculative start, fields + identity hashes, fragment numbering by
 * hash partition, prefix sums, payload copy); results are identical for any thread count.
 *
 * Two ways in.  smc_bam_open reads and inflates the whole file.  smc_bam_open_indexed takes the file's BAM index (.bai, SAMv1
 * section 5.2) as well and inflates only the blocks of the header; smc_bam_decode then works out from the index which chunks its
 * target intervals need (the standard bin + linear-index query), reads only their compressed byte ranges and inflates only
 * their blocks, so time and memory follow the reads used rather than the file size.  Both give identical arrays.
 *
 * All returned pointers stay valid until smc_bam_close().  Functions return 0 or a negative code; message via
 * smc_bam_last_error().  -3: the index is malformed or does not fit the BAM (the message names the index file).
 */
#ifndef SMC_BAMIO_H
#define SMC_BAMIO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct smc_bam smc_bam;

/* The decoded buffers: field for field the arrays of smc_reads_soa, in BAM order. */
typedef struct smc_bam_reads {
    int64_t         n_reads;
    const int32_t  *ref_id;
    const int32_t  *pos;
    const uint16_t *flag;
    const uint8_t  *mapq;
    const int32_t  *nm;
    const int32_t  *l_seq;
    const int64_t  *seq_off;
    const int64_t  *qual_off;
    const int64_t  *cigar_off;
    const uint16_t *n_cigar;
    const uint64_t *umi;        /* 2-bit pack with a leading 1 when the barcode is <= 31 nt of ACGT, else (1<<63 | dictionary id) */
    const uint32_t *frag_id;    /* (barcode, readid) numbered by first appearance among the kept reads */
    const uint8_t  *seq;
    int64_t         seq_bytes;
    const uint8_t  *qual;
    int64_t         qual_bytes;
    const uint32_t *cigar;
    int64_t         n_cigar_words;
    int64_t         n_dict_umis; /* barcodes that needed the dictionary (see smc_bam_dict_umi) */
    const int32_t  *store_lo;   /* trim mode (smc_bam_set_trim): the stored window of smc_reads_soa, else NULL */
    const int32_t  *store_len;
    const uint64_t *qual_hist;  /* 256 counts: how often every phred value occurs in qual[] (decides the upload codebook) */
} smc_bam_reads;

int         smc_bam_open(const char *path, int threads, smc_bam **out);   /* read + inflate + parse the header */
/* Inflate the header blocks only and parse the index (magic, n_ref == the header's reference count, bins with their chunks,
 * linear index, optional n_no_coor).  smc_bam_decode with n_intervals > 0 reads the chunks the intervals need; with
 * n_intervals == 0 it reads the whole file. */
int         smc_bam_open_indexed(const char *path, const char *index_path, int threads, smc_bam **out);
void        smc_bam_close(smc_bam *h);
/* trim != 0: smc_bam_decode keeps, for every read that is one plain aligned run, only the query bases between its first and
 * its last target position (store_lo / store_len of include/smc_b200.h); needs n_intervals > 0.  Default off. */
void        smc_bam_set_trim(smc_bam *h, int trim);
const char *smc_bam_last_error(smc_bam *h);                               /* h may be NULL: error of smc_bam_open */
int         smc_bam_n_refs(smc_bam *h);
const char *smc_bam_ref_name(smc_bam *h, int i);
int64_t     smc_bam_ref_length(smc_bam *h, int i);

/* Walk the records.  n_intervals > 0: keep only reads whose reference span touches one of the target intervals
 * (iv_ref = index into the BAM's reference list, 0-based half-open [iv_start, iv_end)); n_intervals == 0: keep all mapped. */
int         smc_bam_decode(smc_bam *h, int64_t n_intervals, const int32_t *iv_ref, const int32_t *iv_start, const int32_t *iv_end,
                           smc_bam_reads *out);
const char *smc_bam_dict_umi(smc_bam *h, int64_t i);                      /* barcode string of dictionary id i */

/* The decoder's own raw-DEFLATE routine (csrc/smc_inflate.h), exposed for tests: inflates one stream of exactly out_len bytes;
 * `in` must be readable up to in + in_len + 64.  0, or -1 when the stream is malformed / of another size (the BAM decoder then
 * hands the block to zlib). */
int         smc_bam_inflate_raw(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len);

/* ---- The compressed blocks of a decode, for a decoder elsewhere (the GPU decoder of include/smc_b200.h: smc_decode_bam).
 * Plan, then read: smc_bam_plan works out which compressed byte ranges the decode needs (with intervals and an index, the
 * index chunks exactly as smc_bam_decode chooses them; otherwise the whole file) and their total size; the caller allocates
 * comp_bytes + 64 bytes and smc_bam_read_blocks reads the ranges into it
 * (threaded pread, the 64 bytes of slack zeroed) and lists their BGZF blocks.  Inflating block i and storing its bytes
 * [lo, hi) at uoff of the stream gives, for every i, exactly the stream smc_bam_decode walks; its first record is at
 * first_record (the header's length for a whole file, 0 for index chunks).  Index errors are -3 with smc_bam_decode's
 * messages.  Both need a handle opened header-only; the block table stays valid until smc_bam_close(). */
typedef struct smc_bgzf_block {
    int64_t  coff;      /* deflate payload at buf + coff ... */
    int64_t  clen;      /* ... of clen bytes */
    int64_t  uoff;      /* where [lo, hi) of the inflated block goes in the stream */
    uint32_t isize;     /* inflated size of the block */
    uint32_t lo, hi;
    uint32_t reserved;
} smc_bgzf_block;

typedef struct smc_bgzf_plan {
    int64_t               n_blocks;
    const smc_bgzf_block *blocks;
    int64_t               comp_bytes;
    int64_t               raw_bytes;     /* length of the inflated stream */
    int64_t               first_record;
} smc_bgzf_plan;

/* header-only open without an index (smc_bam_open_indexed is header-only already); smc_bam_decode on it reads the whole file */
int         smc_bam_open_header(const char *path, int threads, smc_bam **out);
int         smc_bam_plan(smc_bam *h, int64_t n_intervals, const int32_t *iv_ref, const int32_t *iv_start, const int32_t *iv_end,
                         int64_t *comp_bytes);
int         smc_bam_read_blocks(smc_bam *h, uint8_t *buf, smc_bgzf_plan *out);

#ifdef __cplusplus
}
#endif
#endif
