/*
 * smc_b200.h -- C ABI of libsmc_b200.so: smCounter's per-locus calling hot path on one B200.
 *
 * This library replaces the body of the reference's per-locus worker
 *     vc(bamFile, chrom, pos, minBQ, minMQ, mtDepth, rpb, hpLen, mismatchThr, mtDrop, maxMT, primerDist, refGenome)
 *         (reference smCounter.py:274-600, fanned out one locus at a time by
 *          multiprocessing.Pool.apply_async(vc_wrapper, ...) at smCounter.py:683-685)
 * with ONE batched call per GPU: all target loci of a shard and all reads overlapping them go in as flat
 * structure-of-arrays buffers, all per-locus integer tallies, prediction indices, Fisher statistics and
 * filter bits come out as flat arrays.  String work (row formatting smCounter.py:575-600, HP/LowC
 * smCounter.py:122-177, repeat filters :699-785, writers :787-901) stays on the host.
 *
 * Conventions
 *   - plain C, no C++/torch types; every pointer is HOST memory owned by the caller (pinned memory makes the
 *     copies faster but is not required); the library owns all device memory and grows it lazily.
 *   - every function returns 0 on success or a negative SMC_E_* code; the message is in smc_last_error().
 *     Nothing throws or exits across the ABI (the reference's vc_wrapper turns exceptions into a string,
 *     smCounter.py:605-611; the Python binding raises RuntimeError naming the locus range instead).
 *   - one smc_ctx per GPU; a ctx is not thread-safe, different ctxs may be driven from different host threads.
 *   - there is no CPU fallback: without a CUDA device smc_ctx_create fails with SMC_E_CUDA.
 */
#ifndef SMC_B200_H
#define SMC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMC_ABI_VERSION 3

/* error codes */
#define SMC_OK            0
#define SMC_E_CUDA       -1   /* CUDA runtime error / no device */
#define SMC_E_ARG        -2   /* bad argument */
#define SMC_E_LIMIT      -3   /* input exceeds a documented batch limit (split the batch) */
#define SMC_E_OVERFLOW   -4   /* an internal table overflowed even after regrowth */
#define SMC_E_STATE      -5   /* call order violated (e.g. run before upload) */

/* Parameters of vc() that reach the device (reference smCounter.py:274, CLI :619-633). */
typedef struct smc_params {
    int32_t minBQ;        /* --minBQ       (smCounter.py:626) */
    int32_t minMQ;        /* --minMQ       (:627) */
    int32_t mtDepth;      /* --mtDepth     (:623)  ds = maxMT or round(2*mtDepth), :486 */
    int32_t mtDrop;       /* --mtDrop      (:630) */
    int32_t maxMT;        /* --maxMT       (:631) */
    int32_t primerDist;   /* --primerDist  (:632) */
    double  rpb;          /* --rpb         (:624)  strong-MT bar 2/3/4, :303-308 */
    double  mismatchThr;  /* --mismatchThr (:629) */
    int32_t fisherLegacy; /* which scipy.stats.fisher_exact the run is to match (smCounter.py:215,238,248,260; scipy is unpinned in the
                             reference): 0 = scipy >= 1.7 (two-sided p sums every outcome with pmf <= pmf(observed) * (1 + 1e-7 ... 1e-14);
                             the installed scipy the oracle calls), 1 = the scipy of the reference's day (<= 1.6: epsilon = 1 - 1e-4, i.e.
                             p = 1 when pmf(observed) is within 1e-4 of the mode's, outcomes up to pmf(observed) / (1 - 1e-4) are summed) */
    int32_t reserved0;
} smc_params;

/*
 * Reads, one entry per BAM record, in BAM (coordinate) order: the index of a read is its pileup order
 * (fragment merge at smCounter.py:467-479 is order dependent).  Replaces what the reference pulls out of
 * pysam per pileup read at smCounter.py:319-365, 372-375, 424-425.
 */
typedef struct smc_reads_soa {
    int64_t         n_reads;    /* <= 2^30 per batch */
    const int32_t  *ref_id;     /* contig index */
    const int32_t  *pos;        /* 0-based leftmost reference position */
    const uint16_t *flag;       /* BAM flag: 0x4 unmapped (skipped), 0x10 reverse, 0x40 read1, 0x80 read2 */
    const uint8_t  *mapq;
    const int32_t  *nm;         /* NM tag, 0 when absent (smCounter.py:329-334) */
    const int32_t  *l_seq;      /* query length incl. soft clips (<= 65535) */
    const int64_t  *seq_off;    /* byte offset of the read's bases in seq[]           } each may be NULL = "packed": the payloads */
    const int64_t  *qual_off;   /* byte offset of the read's qualities in qual[]      } lie back to back in read order (what a BAM  */
    const int64_t  *cigar_off;  /* index of the read's first word in cigar[]          } decode produces); the offsets are then      */
                                /* derived on the device from l_seq / n_cigar and 24 B per read never cross PCIe                  */
    const uint16_t *n_cigar;
    const uint64_t *umi;        /* injective 64-bit code of the barcode string  (BC, smCounter.py:323) */
    const uint32_t *frag_id;    /* id of (BC, readid) (smCounter.py:321), numbered by first appearance in BAM order:
                                   ascending frag_id is the canonical fragment order inside a barcode; ids are dense
                                   (every id < n_reads, checked: SMC_E_ARG otherwise) */
    const uint8_t  *seq;        /* BAM 4-bit bases, high nibble first, every read byte aligned */
    int64_t         seq_bytes;  /* < 4 GiB per batch */
    const uint8_t  *qual;       /* phred */
    int64_t         qual_bytes; /* < 4 GiB per batch */
    const uint32_t *cigar;      /* BAM cigar words: len<<4 | op (M0 I1 D2 N3 S4 H5 P6 =7 X8) */
    int64_t         n_cigar_words; /* < 2^32 per batch */
    /* Optional stored window (both NULL = every read is stored whole).  A pileup over the target loci never looks at the
     * bases of a read that hang off the target intervals, so a decoder may store only query bases
     * [store_lo, store_lo + store_len) of a read in seq[] / qual[]: (store_len+1)/2 bytes and store_len bytes.  store_lo must
     * be even; reads that are not one plain aligned run (indels, hard clips, several M runs) must be stored whole; every
     * target base of the read must be inside the window (all checked on the device: SMC_E_ARG).  l_seq, nm, the CIGAR
     * and all other scalars keep describing the whole read.  On amplicon panels this halves the bytes that cross PCIe. */
    const int32_t  *store_lo;
    const int32_t  *store_len;
    /* Optional compact encodings (ABI v3): fewer bytes over PCIe, expanded on the device in one pass.  All zero / NULL = off.
     *   scalar_bits 16 / 8: l_seq, nm, store_lo and store_len point to uint16 / uint8 arrays (every value < 65536 / < 256:
     *     reads of up to 255 bases) instead of int32.
     *   qual_bits 4 or 2: qual[] holds one qual_bits-wide code per stored base, low bits first, every read starting on a byte
     *     boundary ((stored bases * qual_bits + 7) / 8 bytes per read, qual_bytes = their sum); the phred value of code c is
     *     qual_lut[c] (16 or 4 entries).  Sequencers that bin qualities (4 - 8 distinct values) fit 2 or 4 bits.  Requires the
     *     packed layout (qual_off == NULL). */
    int32_t         scalar_bits;
    int32_t         qual_bits;
    const uint8_t  *qual_lut;
    /*   seq_bits 2: seq[] holds 2-bit base codes A0 C1 G2 T3, four bases per byte, low bits first, every read starting on a byte
     *     boundary ((stored bases + 3) / 4 bytes per read, seq_bytes = their sum).  A base that is not A/C/G/T carries code 0 and
     *     is listed in the exception arrays (ascending read index; position = index of the base inside the read's stored
     *     window; its BAM nibble).  Requires the packed layout (seq_off == NULL).  0 or 4 = BAM nibbles as above. */
    int32_t         seq_bits;
    int32_t         ref_id_bits;    /* 8: ref_id points to a uint8 array (every reference index < 256); 0 or 32: int32 */
    int64_t         n_seq_exc;
    const uint32_t *seq_exc_read;
    const uint32_t *seq_exc_pos;
    const uint8_t  *seq_exc_nib;
    int32_t         umi_bits;       /* 32: umi points to a uint32 array (every barcode code < 2^32: barcodes of <= 15 nt); 0 or 64: uint64 */
    int32_t         reserved2;
} smc_reads_soa;

/* Target loci: unique, sorted by (ref_id, pos0).  At most 4 194 302 per batch. */
typedef struct smc_loci {
    int64_t         n_loci;
    const int32_t  *ref_id;
    const int32_t  *pos0;       /* 0-based position (reference's pos is 1-based: pos0 = int(pos) - 1) */
    const uint8_t  *ref_base;   /* upper-case ASCII reference base (origRef, smCounter.py:311-313) */
} smc_loci;

/*
 * Optional down-sampling mask (smCounter.py:496-500): for the listed loci only the listed barcodes are used.
 * The selection itself (random.seed(pos); random.sample(bcDict.keys(), ds)) depends on CPython-2 dict order and
 * is made on the host; the device only applies it.
 */
typedef struct smc_umi_keep {
    int64_t         n_loci;     /* number of masked loci */
    const int64_t  *locus;      /* ascending indices into smc_loci */
    const int64_t  *off;        /* n_loci + 1 offsets into umi[] */
    const uint64_t *umi;        /* kept barcode codes, ascending inside each locus */
} smc_umi_keep;

/* ---- outputs -------------------------------------------------------------------------------------------- */

/* Fixed allele slots (index a of the per-allele arrays), in the library's canonical allele order. */
#define SMC_A_A    0
#define SMC_A_C    1
#define SMC_A_DEL  2   /* locus lies inside a deletion ('DEL', smCounter.py:416-421) */
#define SMC_A_T    3
#define SMC_A_G    4
#define SMC_NFIXED 5
/* Allele references in smc_out (alt/max/second): 0..4 = fixed slot, 5 + j = row j of the dyn_* arrays, -1 none. */

/* per-allele counters (index c) */
#define SMC_C_ALLELE   0   /* alleleCnt        :379,401,459 */
#define SMC_C_FWD      1   /* forwardCnt       :389,411,457 */
#define SMC_C_REV      2   /* reverseCnt       :387,409,455 */
#define SMC_C_LOWQ     3   /* lowQReads        :429 */
#define SMC_C_R1LE     4   /* #r1BcEndPos <= 20      :234-237 */
#define SMC_C_R1TOT    5   /* len(r1BcEndPos)        */
#define SMC_C_R2LE     6   /* #r2BcEndPos <= 20      :244-247 */
#define SMC_C_R2TOT    7   /* len(r2BcEndPos) == len(r2PrimerEndPos) */
#define SMC_C_R2PLE    8   /* #r2PrimerEndPos <= primerDist :256-259 */
#define SMC_C_CONCORD  9   /* concordPairCnt   :476 */
#define SMC_C_DISCORD 10   /* discordPairCnt   :479 */
#define SMC_C_MT      11   /* MTCnt            :517,523 */
#define SMC_C_STRONG  12   /* strongMTCnt      :519 */
#define SMC_NCNT      13

/* per-locus scalars (index k) */
#define SMC_L_CVG      0   /* cvg       :368 */
#define SMC_L_ALLFRAG  1   /* allFrag   :483 */
#define SMC_L_ALLMT    2   /* allMT     :482 */
#define SMC_L_USEDFRAG 3   /* usedFrag  :501 */
#define SMC_L_NBC      4   /* len(bcDict) before down-sampling */
#define SMC_L_USEDMT   5   /* barcodes actually used (== min(ds, len(bcDict)) when the mask is right) */
#define SMC_L_MT3      6
#define SMC_L_MT5      7
#define SMC_L_MT7      8
#define SMC_L_MT10     9
#define SMC_L_KEYMASK 10   /* bit a set: fixed allele a is a key of finalDict (:512) */
#define SMC_L_STATUS  11   /* SMC_ST_* bits */
#define SMC_NLOC      12

#define SMC_ST_ZERO_COVERAGE   1u   /* usedMT == 0 (:492-494) */
#define SMC_ST_NEED_DOWNSAMPLE 2u   /* len(bcDict) > ds and no mask given: tallies cover ALL barcodes; re-run with a mask */
#define SMC_ST_UMI_OVERFLOW    4u   /* a barcode showed > 6 distinct non-ACGT/DEL alleles at this locus (unsupported) */
#define SMC_ST_BAD_MASK        8u   /* mask given but kept count != ds */

/* dynamic allele kinds (dyn_kind) */
#define SMC_K_BASE 0   /* single non-ACGT base (N or IUPAC): dyn_site = BAM nibble */
#define SMC_K_INS  1   /* 'INS|s|s+inserted'  (:371-375): dyn_site = nibble of s, dyn_len = inserted length */
#define SMC_K_DEL  2   /* 'DEL|s+deleted|s'   (:392-396): dyn_site = nibble of s (the READ's base), dyn_len = deleted length */

/* filter bits (fl1 / fl2): the device-evaluated part of filterVariants(), smCounter.py:182-269 */
#define SMC_F_LM        (1u << 0)
#define SMC_F_LSM       (1u << 1)
#define SMC_F_DP        (1u << 2)
#define SMC_F_SB        (1u << 3)
#define SMC_F_LOWQ      (1u << 4)
#define SMC_F_R1CP      (1u << 5)
#define SMC_F_R2CP      (1u << 6)
#define SMC_F_PRIMERCP  (1u << 7)
#define SMC_F_HPGATE    (1u << 16)  /* MTCnt[alt]/usedMT < 0.99: HP / LowC apply if the host finds the region (:198,202) */
#define SMC_F_EVALUATED (1u << 17)  /* filterVariants() was entered for this candidate (:549 / :563) */

/* Fisher tests per candidate (index t) */
#define SMC_T_SB     0
#define SMC_T_R1     1
#define SMC_T_R2     2
#define SMC_T_PRIMER 3

/*
 * All arrays are caller-allocated.  Per-locus arrays use the layout [field][locus] so that the device writes
 * them coalesced:  loc[k * n_loci + i],  cnt[(a * SMC_NCNT + c) * n_loci + i],  pi[a * n_loci + i],
 * fisher_p[((cand * 4) + t) * n_loci + i].
 */
typedef struct smc_out {
    int64_t   n_loci;        /* capacity of the per-locus arrays (must equal smc_loci.n_loci) */
    int32_t  *loc;           /* [SMC_NLOC][n_loci] */
    int32_t  *cnt;           /* [SMC_NFIXED][SMC_NCNT][n_loci] */
    double   *pi;            /* [SMC_NFIXED][n_loci]  finalDict: exactly rounded sum of per-barcode terms (:512) */
    /* call-level results (smCounter.py:534-573) */
    int32_t  *max_allele;    /* [n_loci] maxBase        (allele reference) */
    int32_t  *second_allele; /* [n_loci] secondMaxBase */
    int32_t  *alt_allele;    /* [n_loci] origAlt before the bi-allelic step (:541) */
    double   *alt_pi;        /* [n_loci] altPI (unrounded) */
    double   *second_pi;     /* [n_loci] secondMaxPI */
    uint32_t *fl1;           /* [n_loci] filter bits of candidate 1 = origAlt */
    uint32_t *fl2;           /* [n_loci] filter bits of candidate 2 = secondMaxBase when the bi-allelic test (:555) holds */
    uint8_t  *biallelic;     /* [n_loci] 1 when the condition at :555 holds */
    double   *fisher_p;      /* [2][4][n_loci]  NaN when the test was not evaluated */
    double   *fisher_or;     /* [2][4][n_loci] */
    /* dynamic alleles (anything that is not A/C/G/T/'DEL'), sorted by (locus, kind, site, len, bases) */
    int64_t   dyn_capacity;  /* rows available in the dyn_* arrays */
    int64_t   n_dyn;         /* OUT: rows written (if > dyn_capacity the call fails with SMC_E_LIMIT) */
    int32_t  *dyn_locus;     /* [dyn_capacity] */
    uint8_t  *dyn_kind;      /* SMC_K_* */
    uint8_t  *dyn_site;
    int32_t  *dyn_len;
    uint32_t *dyn_rep_read;  /* a read (index into smc_reads_soa) that carries the allele ... */
    int32_t  *dyn_rep_qpos;  /* ... and the query position of its site base: inserted bases are seq[qpos+1 .. qpos+len] */
    uint8_t  *dyn_iskey;     /* 1 when the allele is a key of finalDict */
    int32_t  *dyn_cnt;       /* [dyn_capacity][SMC_NCNT] (row major) */
    double   *dyn_pi;        /* [dyn_capacity] */
    int64_t  *dyn_first;     /* [n_loci + 1] rows of locus i are dyn_first[i] .. dyn_first[i+1]-1 */
} smc_out;

/* CUDA-event timings and work counts of the last smc_run_resident() / smc_call_batch(). */
typedef struct smc_timings {
    float   ms_h2d, ms_prep, ms_sort, ms_pileup, ms_stats, ms_d2h, ms_total_device;
    float   ms_k_pileup;   /* k_gather + k_merge (the pileup stage without its memsets) */
    int64_t n_reads, n_loci, n_tile_events, n_pileup_events /* sum of cvg */, n_umi_groups, n_dyn, n_fisher;
    int64_t bytes_h2d, bytes_d2h;
    int32_t kernel_launches;
    float   ms_k_gather;   /* K3a alone: base/quality gather, read tallies, fragment merge (the HBM-facing kernel) */
    float   ms_k_merge;    /* K3b alone: per-barcode posterior, prediction index, consensus (FP64) */
    int32_t code_mult;     /* fragment-code slots per tile event in the last run: 1, or 3 after a unit overflowed (worst-case layout) */
    int32_t dyn_capacity;  /* capacity of the dynamic-allele table in the last run (grows x4 on overflow) */
    int32_t pipe_chunks;   /* smc_call_batch: chunks the bases / qualities were uploaded in (1 = no overlap, small batch) */
    int32_t pipe_launches; /* smc_call_batch: (k_gather, k_merge) launch pairs issued as the chunks arrived */
    /* ABI v3: CUDA-event times of the kernels north_star names besides the pileup pair, and what they move */
    float   ms_read_sort;  /* the radix passes over the reads on (barcode slot, fragment id): histogram + scan + scatter per pass */
    float   ms_k_read_prep;/* k_read_prep alone */
    float   ms_event_sort; /* (read x tile) events: k_expand_scan + the radix pass by tile */
    int32_t read_sort_passes;
    int64_t read_prep_bytes; /* read SoA bytes in + the two per-read records out */
} smc_timings;

typedef struct smc_ctx smc_ctx;

int         smc_version(void);
int         smc_ctx_create(int device, const smc_params *params, smc_ctx **out);
void        smc_ctx_destroy(smc_ctx *ctx);
const char *smc_last_error(smc_ctx *ctx);            /* ctx may be NULL: last error of smc_ctx_create */

/* One call = host buffers in, host buffers out (H2D, all kernels, D2H).  For batches with >= 96 MiB of bases + qualities
 * the upload is pipelined: the per-read scalars, CIGARs and loci go first; the read sort, read prep and tile sort run while
 * the bases / qualities follow in chunks of consecutive reads on a second stream, and the pileup kernels are launched per
 * chunk for the units whose reads have arrived.  Results are identical to smc_upload + smc_run_resident + smc_download. */
int smc_call_batch(smc_ctx *ctx, const smc_reads_soa *reads, const smc_loci *loci, const smc_umi_keep *keep /* nullable */,
                   smc_out *out);

/* The same three phases separately, so that the kernels can be timed with inputs resident in HBM. */
/* When smc_upload returns an error, no copy from the caller's buffers is still in flight. */
int smc_upload(smc_ctx *ctx, const smc_reads_soa *reads, const smc_loci *loci, const smc_umi_keep *keep /* nullable */);
int smc_run_resident(smc_ctx *ctx);
int smc_download(smc_ctx *ctx, smc_out *out);

int smc_get_timings(smc_ctx *ctx, smc_timings *t);

/* For loci flagged SMC_ST_NEED_DOWNSAMPLE (after smc_run_resident / smc_call_batch): list the barcodes of bcDict (those
 * with >= 1 read passing incCond, smCounter.py:467) so that the host can draw the reference's sample (:496-500).
 * locus[n] ascending; off_out[n+1] receives the offsets (off_out[k+1]-off_out[k] == loc[SMC_L_NBC] of locus k); umi_out /
 * first_read_out receive, per locus in unspecified order, the barcode codes and the index (into smc_reads_soa) of the
 * barcode's first passing read at that locus (ascending first_read = the insertion order of bcDict).  Returns
 * SMC_E_LIMIT with off_out filled when umi_capacity < off_out[n].  The listing pass invalidates the batch results: run
 * the batch again (with the mask) before smc_download. */
int smc_list_barcodes(smc_ctx *ctx, int64_t n, const int64_t *locus, int64_t *off_out, uint64_t *umi_out,
                      uint32_t *first_read_out, int64_t umi_capacity);

/*
 * isHPorLowComp() (smCounter.py:122-177) for a batch of candidates in one launch: is the candidate inside / next to a
 * homopolymer of >= hpLen bases, or a 2*hpLen window whose two most frequent nucleotides make up >= 99 %?  Replaces the six
 * FastaFile.fetch() round trips per candidate of the reference (:127-129, :143-145).  For candidate k the caller passes
 *   - one upper-case reference window  bases[win_off[k] .. +win_len[k])  =  reference[w0, w1)  with
 *       w0 = max(0, pos0 - 2*hpLen),  w1 = min(contig length, pos0 + max(len(ref), len(alt)) + 2*hpLen),
 *     and win_pos[k] = pos0 - w0 (the candidate's position inside the window);
 *   - the VCF-style REF and ALT strings of convertToVcf() (:103-117) at ref_off/ref_len and alt_off/alt_len of bases[].
 * flags_out[k]: bit 0 = homopolymer, bit 1 = low complexity.  Independent of any uploaded batch.
 */
typedef struct smc_hp_batch {
    int64_t         n;          /* candidates */
    int32_t         hpLen;      /* --hpLen (smCounter.py:628) */
    const uint8_t  *bases;      /* windows and allele strings, concatenated */
    int64_t         n_bases;
    const int64_t  *win_off;
    const int32_t  *win_len;
    const int32_t  *win_pos;
    const int64_t  *ref_off;
    const int32_t  *ref_len;
    const int64_t  *alt_off;
    const int32_t  *alt_len;
} smc_hp_batch;
#define SMC_HP_HOMOPOLYMER 1u
#define SMC_HP_LOWCOMP     2u

int smc_hp_lowcomp(smc_ctx *ctx, const smc_hp_batch *batch, uint8_t *flags_out);

/*
 * The Fisher exact test kernel on caller-supplied 2x2 tables (what filterVariants() asks scipy for at smCounter.py:215, 238,
 * 248, 260): tables[4*i .. 4*i+3] = a, b, c, d of [[a, b], [c, d]]; p_out[i] = two-sided p, or_out[i] = sample odds ratio
 * (inf / nan as scipy returns them).  Uses the context's fisherLegacy setting.  A utility for validating the device
 * arithmetic against scipy on tables of the caller's choosing; smc_call_batch does not need it.
 */
int smc_fisher_exact(smc_ctx *ctx, int64_t n, const int32_t *tables, double *p_out, double *or_out);

/* Page-locked host memory for the buffers of smc_reads_soa / smc_out: copies from / to it run as one DMA and overlap the
 * kernels (pageable memory is staged by the driver at a fraction of the link rate).  Not tied to a context. */
int  smc_host_alloc(int64_t bytes, void **out);
void smc_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* SMC_B200_H */
