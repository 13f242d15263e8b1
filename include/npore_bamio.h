/*
 * npore_bamio.h -- native BAM ingest and SAM record output for the realignment path (part of libnpore_b200.so).
 *
 * These entry points replace, for this path only, what the reference gets from pysam / htslib (a compiled
 * third-party dependency, not part of the TimD1/nPoRe tree):
 *
 *   npore_bam_open / _advance / _columns / _gather
 *                                        <- pysam.AlignmentFile(bam).fetch(...) and the per-read attribute reads of
 *                                           src/bam.pyx:18-47 get_read_data(): flag, reference_start, reference_length,
 *                                           mapping_quality, cigar, query_alignment_sequence / _qualities (soft clips
 *                                           removed), HP tag.  BGZF members are inflated on n_threads host threads.
 *   npore_sam_format / npore_sam_format_fd <- the record print of src/bam.pyx:81-84 realign_read():
 *                                           name flag rname start+1 mapq CIGAR * 0 (stop-start) seq quals HP:i:hap
 *                                           for a whole batch, in input order, from the run-length words the GPU returns.
 *   npore_bam_format                     <- the same records as BAM (what `samtools view -b` makes of that SAM text).
 *
 * Plain C ABI; all pointers are caller-owned host memory.  Functions return 0 or a negative code; the text of the last
 * error of the calling thread is npore_io_last_error().  No CUDA involved.
 */
#ifndef NPORE_BAMIO_H
#define NPORE_BAMIO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct npore_bam npore_bam;

#define NPORE_IO_OK         0
#define NPORE_IO_ERR_OPEN  -1   /* file missing / unreadable                      */
#define NPORE_IO_ERR_FORMAT -2  /* not BGZF / not BAM / truncated / CRC mismatch  */
#define NPORE_IO_ERR_ARG   -3

const char *npore_io_last_error(void);

/* open the file and read the BAM header (text + reference list); n_threads (<= 0: all cores) inflate BGZF members */
int      npore_bam_open(const char *path, int n_threads, npore_bam **out);
/* load the next window of records: members are inflated until at least max_bytes of record data are available
 * (<= 0: the rest of the file); records straddling the window end are carried over.  Returns the number of records in
 * the window (0 at end of file, negative on error).  _n_records / _columns / _gather refer to the current window. */
int64_t  npore_bam_advance(npore_bam *b, int64_t max_bytes);
void     npore_bam_close(npore_bam *b);
int64_t  npore_bam_header_text(const npore_bam *b, const char **text);          /* returns the text length */
int32_t  npore_bam_n_refs(const npore_bam *b);
int      npore_bam_ref(const npore_bam *b, int32_t i, const char **name, int64_t *length);
/* optional: inflate and index the window after the current one on a background thread (the current window stays valid for
 * npore_bam_columns / npore_bam_gather); the next npore_bam_advance then only swaps it in.  max_bytes as for npore_bam_advance. */
int      npore_bam_prefetch(npore_bam *b, int64_t max_bytes);
int64_t  npore_bam_n_records(const npore_bam *b);
/* Read only through a BAM index: after this call (before the first npore_bam_advance, once) windows hold only the records whose
 * start virtual offset lies in one of the n chunks [vbeg, vend) (sorted, disjoint; bamio.read_bai(...).query gives them).  The
 * reader seeks to vbeg >> 16, skips vbeg & 0xffff inflated bytes and inflates members until the last record that starts before
 * vend is complete; members between chunks are not read.  n == 0: no record. */
int      npore_bam_restrict(npore_bam *b, int64_t n, const uint64_t *vbeg, const uint64_t *vend);
/* virtual offset of every record of the current window (file offset of its member << 16 | offset inside the member) */
int      npore_bam_voffsets(const npore_bam *b, uint64_t *out);
/* BGZF member bytes read from the file so far (the header's included) */
int64_t  npore_bam_bytes_read(const npore_bam *b);

/* one value per record of the current window, file order.  end = pos + reference span of the CIGAR (M D N = X); aln_len = SEQ length without
 * the soft-clipped ends (pysam query_alignment_sequence); n_cigar = CIGAR words once S and H are dropped (bam.pyx:59);
 * hp = value of the HP tag or 0 (bam.pyx:46); has_qual = 0 when QUAL is stored as 0xff.  Any pointer may be NULL. */
int      npore_bam_columns(const npore_bam *b, int32_t *ref_id, int32_t *pos, int32_t *end, int32_t *flag, int32_t *mapq,
                           int32_t *aln_len, int32_t *n_cigar, int32_t *name_len, int32_t *hp, int32_t *has_qual);

/* copy the selected records (indices into file order) into flat arrays.  The three offset arrays [n_sel+1] are the
 * caller's exclusive prefix sums of aln_len / n_cigar / name_len over the selection.  seq_ascii is upper-cased;
 * seq_codes uses N A C G T = 0..4 (anything else 0, src/cig.pyx:212-229); qual_ascii is phred+33 (unspecified bytes when
 * has_qual == 0); cigar words keep BAM op codes.  Any output pointer may be NULL. */
int      npore_bam_gather(const npore_bam *b, int64_t n_sel, const int64_t *sel, int n_threads,
                          uint8_t *seq_ascii, uint8_t *seq_codes, uint8_t *qual_ascii, const int64_t *seq_off,
                          uint32_t *cigar, const int64_t *cig_off, uint8_t *names, const int64_t *name_off);

/* the selected records' aligned bases in BAM's own 4-bit packing, for npore_batch.seq_nib (include/npore_b200.h): whole bytes are
 * copied out of the records (soft-clipped ends skipped at byte granularity), nib_start[k] is the nibble offset of record k's first
 * aligned base inside `nib`.  Two calls: nib == NULL fills byte_off[n_sel+1] (exclusive prefix sum of the bytes per record) so that
 * the caller can size `nib`; the second call copies.  Replaces the per-base decode of npore_bam_gather's seq_codes on the upload path. */
int      npore_bam_gather_nib(const npore_bam *b, int64_t n_sel, const int64_t *sel, int n_threads, int64_t *byte_off, uint8_t *nib,
                              int64_t *nib_start);

/* src/bam.pyx:83 for n records.  ref_names / ref_name_off: concatenated contig names; rle / rle_off: the collapsed CIGAR of
 * every record as (len<<4|op) words (npore_result.rle).  has_qual[i] == 0 or an empty sequence prints '*' for QUAL; a ref_id outside
 * [0, n_refs) prints '*' for RNAME.
 * Returns the number of bytes written to out (each record ends in '\n'), or a negative code; out_capacity must be at
 * least npore_sam_bound(...). */
int64_t  npore_sam_bound(int64_t n, const int64_t *name_off, const int64_t *seq_off, const int64_t *rle_off, int64_t max_ref_name);
int64_t  npore_sam_format(int64_t n, int n_threads,
                          const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                          const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                          const int32_t *pos, const int32_t *end, const int32_t *mapq,
                          const uint32_t *rle, const int64_t *rle_off,
                          const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                          const int32_t *hp, uint8_t *out, int64_t out_capacity);
/* npore_sam_format + the append to the output file (the `print(..., file=fh)` of src/bam.pyx:81-84) in one pass: every formatter
 * thread pwrite()s its finished slice of records to `fd` at file_offset + (its offset inside the block) while the others still
 * format -- the copy into the page cache runs on all threads and overlaps the formatting.  `scratch` (>= npore_sam_bound bytes)
 * holds the text meanwhile.  Returns the number of bytes appended; the caller advances its end-of-file offset by it.  `fd` must
 * not be in O_APPEND mode (Linux then ignores the offset of pwrite). */
int64_t  npore_sam_format_fd(int64_t n, int n_threads,
                             const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                             const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                             const int32_t *pos, const int32_t *end, const int32_t *mapq,
                             const uint32_t *rle, const int64_t *rle_off,
                             const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                             const int32_t *hp, uint8_t *scratch, int64_t scratch_capacity, int fd, int64_t file_offset);

/* The records of npore_sam_format as binary BAM records (SAM spec 4.2, each with its block_size), same arguments, same order.
 * The fields are encoded as htslib's SAM -> BAM conversion encodes that SAM line: refID -1 where RNAME is '*', next_refID and
 * next_pos -1, tlen = end - pos, bin = reg2bin(pos, pos + reference span of the CIGAR, 1 if 0), SEQ in 4 bits, QUAL phred or
 * 0xFF * l_seq without qualities, HP as the smallest integer type holding the value (C/S/I, c/s/i when negative).
 * Returns the bytes written; out_capacity must be at least npore_bam_bound(...).  A read name longer than 254 bytes or a CIGAR
 * of more than 65535 operations is an error. */
int64_t  npore_bam_bound(int64_t n, const int64_t *name_off, const int64_t *seq_off, const int64_t *rle_off);
int64_t  npore_bam_format(int64_t n, int n_threads,
                          const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                          const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                          const int32_t *pos, const int32_t *end, const int32_t *mapq,
                          const uint32_t *rle, const int64_t *rle_off,
                          const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                          const int32_t *hp, uint8_t *out, int64_t out_capacity);
/* npore_bam_format that also fills rec_off[n+1]: the offset of record k's block_size field inside `out`, and the bytes written
 * at [n].  These are the positions a BAM index needs (npore_bgzf_index, include/npore_b200.h). */
int64_t  npore_bam_format_offsets(int64_t n, int n_threads,
                                  const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                                  const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                                  const int32_t *pos, const int32_t *end, const int32_t *mapq,
                                  const uint32_t *rle, const int64_t *rle_off,
                                  const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                                  const int32_t *hp, uint8_t *out, int64_t out_capacity, int64_t *rec_off);

#ifdef __cplusplus
}
#endif
#endif /* NPORE_BAMIO_H */
