/*
 * npore_b200.h -- C ABI of libnpore_b200.so: nPoRe's realignment hot path on one NVIDIA B200 (sm_100a).
 *
 * Drop-in boundary (SURVEY.md section 8(b)).  Each entry point names the reference interface it replaces
 * (paths relative to the TimD1/nPoRe tree):
 *
 *   npore_ctx_create      <- the per-process state every align() call reads: score tables passed as
 *                            arguments (src/aln.pyx:379-382), cfg.args.max_n / max_l read at call time
 *                            (src/aln.pyx:207-208, 436-437), and align()'s keyword defaults
 *                            indel_start=5, indel_extend=1, max_b_rows=20000, r=30 (src/aln.pyx:381-382).
 *   npore_align_batch     <- src/aln.pyx:379-787 align() for a batch of independent items, optionally
 *                            followed by the CIGAR standardisation of src/bam.pyx:65-78 (== :105-118;
 *                            src/cig.pyx:102-192) and the run-length collapse of src/cig.pyx:13-38.
 *                            One call replaces one multiprocessing.Pool fan-out
 *                            (src/realign.py:110-114, src/standardize_vcf.py:30-31).
 *   npore_upload / npore_run / npore_download
 *                         <- the same work split into its three phases (host->device staging, kernels,
 *                            device->host) so callers can time / overlap them; npore_align_batch is
 *                            exactly upload + run + download.
 *   npore_get_np_info     <- src/aln.pyx:179-251 get_np_info() (device implementation, for tests and
 *                            for callers such as src/bed.py:56-76).
 *   npore_confusion_batch <- src/bam.pyx:351-510 calc_confusion_matrices() for a batch of get_ranges() windows
 *                            (src/bam.pyx:149-164), computed from the alignments themselves instead of the text of
 *                            `samtools mpileup | cut -f5` (src/bam.pyx:300-314); the sum over the ranges is what
 *                            src/bam.pyx:184-192 get_confusion_matrices() reduces to.
 *   npore_bgzf_*          <- the BGZF compression of `samtools view -b` (SAM spec section 4.1) that users ran on the
 *                            reference's SAM output: the realigned records are written as BAM, deflated on the device.
 *   npore_last_stats      <- the wall-clock prints of src/realign.py:109,115 (per-phase device times,
 *                            cell-update counts).
 *
 * Conventions: every function returns NPORE_OK (0) or a negative error code; nothing aborts the process.
 * All pointers are HOST pointers owned by the caller (pinned memory makes the copies asynchronous but is
 * not required).  The library owns all device memory.  A context is bound to one CUDA device and is not
 * re-entrant; use one context per GPU (and per host thread).
 *
 * Base codes: N=0 A=1 C=2 G=3 T=4 (src/cig.pyx:212-229).  CIGAR input: BAM-style run-length words
 * (len << 4 | op) with op in M=0 I=1 D=2 ==7 X=8 (src/cfg.py:28-32); S/H/N/P must already be stripped
 * (src/bam.pyx:59).  The CIGAR must consume exactly ref_len reference and seq_len read bases; the reference
 * has undefined behaviour otherwise (boundscheck off), this library reports item status NPORE_ST_BAD_CIGAR.
 */
#ifndef NPORE_B200_H
#define NPORE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct npore_ctx npore_ctx;

/* error codes */
#define NPORE_OK               0
#define NPORE_ERR_BAD_ARG     -1
#define NPORE_ERR_CUDA        -2
#define NPORE_ERR_OOM         -3
#define NPORE_ERR_NO_DEVICE   -4
#define NPORE_ERR_STATE       -5
#define NPORE_ERR_CAPACITY    -6

/* per-item status (the conditions of src/aln.pyx:689-716, 737-739; the CIGAR is then partial, as there) */
#define NPORE_ST_OK            0
#define NPORE_ST_ROW_NEG       1
#define NPORE_ST_COL_NEG       2
#define NPORE_ST_RUN_ZERO      3
#define NPORE_ST_BAD_TYPE      4
#define NPORE_ST_RUN_OVERFLOW  8    /* n-polymer (LEN/SHR) runs >= 2047 ops are handled by a transparent second pass (wide kernels);
                                       this status remains only if more than 65,536 such records occur in one batch: CIGAR partial */
#define NPORE_ST_BAD_CIGAR     16   /* input CIGAR inconsistent with ref_len / seq_len: item skipped, empty output */

/* output selection flags for npore_run / npore_align_batch */
#define NPORE_OUT_STANDARDIZE  1u   /* apply src/bam.pyx:65-78: ops over {M,I,D} instead of align()'s {=,X,I,D} */
#define NPORE_OUT_RLE          2u   /* additionally produce run-length words (len<<4|op), i.e. collapse_cigar */
#define NPORE_OUT_NO_EXPANDED  4u   /* do not copy the one-byte-per-op array back (only with NPORE_OUT_RLE) */

typedef struct npore_batch {
    int32_t        n_items;
    const uint8_t *ref_codes;    /* concatenated / shared reference codes                                   */
    const int64_t *ref_start;    /* [n] item i uses ref_codes[ref_start[i] .. +ref_len[i]) (may overlap)     */
    const int32_t *ref_len;      /* [n]                                                                      */
    int64_t        ref_total;    /* bytes in ref_codes                                                       */
    const uint8_t *seq_codes;    /* concatenated read codes                                                  */
    const int64_t *seq_start;    /* [n]                                                                      */
    const int32_t *seq_len;      /* [n]                                                                      */
    int64_t        seq_total;
    const uint32_t *cigar_rle;   /* concatenated BAM-style words                                             */
    const int64_t *cigar_off;    /* [n+1] word offsets                                                       */
    /* Optional PACKED read bases in BAM's own encoding (SAM spec 4.2.3: 4 bits per base, "=ACMGRSVTWYHKDBN", first base in
     * the high nibble).  When seq_nib is not NULL, seq_codes / seq_start / seq_total are ignored and item i's read is the
     * seq_len[i] nibbles starting at nibble seq_nib_start[i] of seq_nib (nibble k lives in byte k/2, high half for even k).
     * Half the host->device bytes of seq_codes, and the bases of a BAM record go in as they lie in the file: the device
     * decodes them (replaces the per-character src/cig.pyx:212-229 bases_to_int; A,C,G,T -> 1..4, every other code -> 0 = N,
     * which is what bases_to_int yields for the IUPAC letters).  Leave all three zero for unpacked input. */
    const uint8_t *seq_nib;
    const int64_t *seq_nib_start; /* [n] nibble offsets                                                        */
    int64_t        seq_nib_bytes; /* bytes in seq_nib                                                          */
} npore_batch;

typedef struct npore_result {
    /* expanded ops, one ASCII char per op.  Capacity needed: sum(ref_len+seq_len).  May be NULL with NO_EXPANDED. */
    uint8_t  *ops;
    int64_t   ops_capacity;
    int64_t  *ops_off;           /* [n+1] written: item i's ops are ops[ops_off[i] .. ops_off[i+1])          */
    /* run-length words (len<<4|op; op codes as above), only with NPORE_OUT_RLE.  Capacity: as ops.          */
    uint32_t *rle;
    int64_t   rle_capacity;
    int64_t  *rle_off;           /* [n+1]                                                                    */
    /* DP score of every chunk = MAT value at the chunk's end cell (src/aln.pyx:683 at the first traceback
     * step).  Item i's chunks are chunk_scores[score_off[i] .. score_off[i+1]).  Capacity: npore_count_chunks. */
    float    *chunk_scores;
    int64_t   score_capacity;
    int64_t  *score_off;         /* [n+1]                                                                    */
    int32_t  *status;            /* [n]                                                                      */
} npore_result;

typedef struct npore_stats {
    int64_t n_items, n_chunks;
    int64_t n_cu;                /* cell updates = sum over chunks of b_rows * (2r+1)   (SURVEY.md 8(d))     */
    int64_t h2d_bytes, d2h_bytes;
    int64_t tb_bytes;            /* traceback records written to HBM by the forward kernel                   */
    float   ms_plan, ms_annotate, ms_forward, ms_traceback, ms_finish, ms_kernels_total;
    float   ms_h2d, ms_d2h;
    int32_t launches;            /* kernel launches of the last npore_run                                    */
    int32_t n_sub_batches;
    int32_t fwd_warps_per_sm;    /* resident forward-kernel warps per SM of the last run (occupancy achieved) */
    int32_t sm_count;
} npore_stats;

int  npore_ctx_create(npore_ctx **out, int device,
                      const float *sub_scores /* [5][5], indexed [seq_base][ref_base] (src/aln.pyx:575) */,
                      const float *np_scores  /* [np_n][np_dim][np_dim] (src/aln.pyx:274)               */,
                      int np_n, int np_dim, int max_n, int max_l,
                      float indel_start, float indel_extend, int max_b_rows, int r);
void npore_ctx_destroy(npore_ctx *ctx);

/* run all copies and kernels of this context on the caller's CUDA stream (a cudaStream_t, e.g. torch's current
 * stream) instead of the context's own; the caller keeps ownership of the stream */
int  npore_set_stream(npore_ctx *ctx, void *cuda_stream);

/* number of chunks align() will cut the batch into (src/aln.pyx:344-358): capacity for chunk_scores */
int64_t npore_count_chunks(const npore_ctx *ctx, int32_t n_items, const int32_t *ref_len, const int32_t *seq_len);

int  npore_upload(npore_ctx *ctx, const npore_batch *batch);
int  npore_run(npore_ctx *ctx, uint32_t flags);
int  npore_download(npore_ctx *ctx, npore_result *result);
int  npore_align_batch(npore_ctx *ctx, const npore_batch *batch, uint32_t flags, npore_result *result);

/* src/aln.pyx:179-251 on device: out is int32 [len][2][max_n] (L plane, L_IDX plane), like the reference's array */
int  npore_get_np_info(npore_ctx *ctx, const uint8_t *codes, int32_t len, int32_t *out);
/* the same for n_seqs sequences codes[off[i] .. off[i+1]) (off[0] == 0), one CTA each: src/bed.py:56-76 calls get_np_info
 * once per chunk_width window of the reference; out is the concatenation of the per-sequence arrays */
int  npore_get_np_info_batch(npore_ctx *ctx, int32_t n_seqs, const uint8_t *codes, const int64_t *off, int32_t *out);

/* Basecaller confusion matrices (src/bam.pyx:351-510).  One range = one (ctg, start, end) tuple of get_ranges().
 * The caller has already dropped the reads samtools mpileup drops by default (flag & (UNMAP|SECONDARY|QCFAIL|DUP));
 * reads are alignments as stored in the BAM (soft clips included in seq and CIGAR), coordinate sorted. */
typedef struct npore_pileup_batch {
    int32_t        n_ranges;
    const int64_t *range_start;      /* [R] 0-based, contig coordinates                                          */
    const int64_t *range_end;        /* [R] half-open                                                            */
    const uint8_t *ref_ascii;        /* raw contig bytes, range r owns [ref_off[r], ref_off[r+1]) =              */
    const int64_t *ref_off;          /* [R+1]  contig[start : min(contig_len, end + 1 + max_n)]                  */
    int32_t        n_reads;
    const int64_t *read_pos;         /* [n] 0-based leftmost reference position                                  */
    const uint8_t *seq_ascii;        /* concatenated read bases (ASCII, any case)                                */
    const uint8_t *qual;             /* concatenated base qualities (phred, not +33), same offsets; NULL = all pass */
    const int64_t *seq_off;          /* [n+1]                                                                    */
    const uint32_t *cigar_rle;       /* concatenated BAM words len<<4|op, op in M I D N S H = X (P, B: error)    */
    const int64_t *cigar_off;        /* [n+1]                                                                    */
    const int32_t *range_reads;      /* per range: indices of the reads overlapping it, ascending position       */
    const int64_t *range_reads_off;  /* [R+1]                                                                    */
    int32_t        min_base_q;       /* samtools mpileup -Q (default 13)                                         */
    /* Optional: the reads in BAM's own packing, as npore_bam_gather_nib / npore_bam_gather write them, so that the host does
     * no per-base work.  When seq_nib is not NULL, seq_ascii is ignored: read i's bases are the seq_off[i+1] - seq_off[i]
     * nibbles starting at nibble seq_nib_start[i] of seq_nib (same layout as npore_batch.seq_nib), decoded through
     * "=ACMGRSVTWYHKDBN" into the letter the ASCII form would hold (so N is base 0 and =, IUPAC codes drop the rest of the
     * line, as in the ASCII form).  qual then holds phred+33 bytes (npore_bam_gather's qual_ascii) at seq_off, and has_qual
     * [n] is required with it: a read with has_qual[i] == 0 (QUAL 0xFF in the file) passes every base, as qual == NULL does
     * for all reads.  Leave all four zero for the ASCII form. */
    const uint8_t *seq_nib;
    const int64_t *seq_nib_start;    /* [n] nibble offsets                                                        */
    int64_t        seq_nib_bytes;    /* bytes in seq_nib                                                          */
    const int32_t *has_qual;         /* [n] nibble form only                                                      */
} npore_pileup_batch;
/* outputs (int64, overwritten with the totals of this call): subs[5][5] indexed [ref][call], nps[max_n][max_l+1][max_l+1]
 * indexed [n-1][ref copies][called copies], inss[max_l+1], dels[max_l+1] */
int  npore_confusion_batch(npore_ctx *ctx, const npore_pileup_batch *batch, int64_t *subs, int64_t *nps, int64_t *inss, int64_t *dels);

/* BGZF compression on the device (SAM spec section 4.1).  The input is cut into members of at most 65,280 bytes; each member is
 * a gzip member with the BC extra field, one final deflate block (dynamic Huffman codes with LZ77 matches, or stored when that
 * is not larger) and CRC32 / ISIZE.  The output depends only on the input bytes.  No EOF block is appended.
 * A handle has its own stream and device buffers (grown on demand); it is not a context and may live beside them.  The
 * pointers are host pointers; the call returns when out holds *out_len bytes.  n == 0 writes nothing.  device_ms (may be
 * NULL) receives the kernel time. */
typedef struct npore_bgzf npore_bgzf;
int     npore_bgzf_create(npore_bgzf **out, int device);
void    npore_bgzf_destroy(npore_bgzf *z);
int64_t npore_bgzf_bound(int64_t n);   /* worst case: every member stored */
int     npore_bgzf_compress(npore_bgzf *z, const uint8_t *in, int64_t n, uint8_t *out, int64_t out_capacity,
                            int64_t *out_len, float *device_ms /* may be NULL */);

/* The BAM index (SAM spec section 5.2) contribution of the records compressed by the handle's last npore_bgzf_compress call,
 * computed on the device from the input and member sizes still there.  rec_off[n_rec+1]: offset of every record's block_size
 * field in that input, rec_off[n_rec] = its length (npore_bam_format_offsets).  base: file offset of the first member.
 * Virtual offsets are (file offset of the member << 16 | offset inside it); the end of the input takes the form
 * (base + compressed length) << 16, where the next member starts.  Records must be in (ref_id, pos) order and placed.
 * Results, in host memory owned by the handle and valid until its next call, as rows of uint64:
 *   chunks [n_chunks][4]   (ref_id, bin, vbeg, vend): one per run of consecutive records with the same (ref_id, bin),
 *                          in (ref_id, bin, vbeg) order, chunks of one bin merged when the first ends in the BGZF member
 *                          where the second begins (htslib's rule);
 *   refs [n_refs][7]       (ref_id, first vbeg, last vend, mapped records, unmapped records, first 16 kb window, windows);
 *   windows [n_windows]    the refs' windows in turn: the smallest vbeg of a mapped record overlapping it, ~0 where none does.
 * Returns NPORE_ERR_BAD_ARG with error_bits set (1 unsorted, 2 inconsistent record bytes, 4 unplaced record) when the records
 * cannot be indexed.  device_ms (may be NULL) receives the time of the index kernels. */
typedef struct {
    const uint64_t *chunks; int64_t n_chunks;
    const uint64_t *refs; int64_t n_refs;
    const uint64_t *windows; int64_t n_windows;
    uint64_t error_bits;
} npore_bai_lists;
int     npore_bgzf_index(npore_bgzf *z, const int64_t *rec_off, int64_t n_rec, uint64_t base, npore_bai_lists *out,
                         float *device_ms /* may be NULL */);

int  npore_last_stats(const npore_ctx *ctx, npore_stats *stats);
const char *npore_strerror(int code);
const char *npore_last_error(const npore_ctx *ctx);   /* detail of the last failure (e.g. the CUDA error string) */
const char *npore_version(void);

#ifdef __cplusplus
}
#endif
#endif /* NPORE_B200_H */
