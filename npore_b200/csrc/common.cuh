// common.cuh -- shared device/host types of libnpore_b200 (sm_100a).
//
// Vocabulary follows the reference (TimD1/nPoRe, src/aln.pyx): an *item* is one align() call (a read or a
// haplotype), cut into *chunks* of at most max_b_rows anti-diagonals (aln.pyx:344-358, 445-454); a chunk is a
// band of W = 2r+1 cells per anti-diagonal ("b_row" x "b_col", aln.pyx:315-338) around the input alignment path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define NP_MAXN 6          // compile-time ceiling for cfg.args.max_n (realign.py:47-49 default 6)
#define NP_RING 8          // anti-diagonals of history kept for the LEN/SHR gathers (needs >= max_n + 1)
// packed traceback record (uint16): [15] INS state extended (aln.pyx:536)  [14] DEL state extended (val2 < val1, aln.pyx:558)
// [13:11] TYP  [10:0] RUN of a MAT / LEN / SHR record.  INS/DEL run lengths are not stored: they are the number of consecutive
// 'extended' bits walked by the traceback (equal to the reference's RUN by its recurrence aln.pyx:537-543).  The flags sit on
// top because the forward kernel gets them as float sign bits (forward.cuh).
#define NP_RUN_SAT 2047
#define NP_REC_TYP 11
#define NP_REC_IE 0x8000u
#define NP_REC_DE 0x4000u
#define NP_PAD 96          // zero records after every colrec/rowrec slice (band prefetch runs ahead)
#define NP_TABQ 2048       // q = trunc(run/n) entries of the re-laid score tables (run saturates at NP_RUN_SAT < NP_TABQ; forward.cuh)

enum { T_MAT = 0, T_INS = 1, T_LEN = 2, T_DEL = 3, T_SHR = 4 };   // aln.pyx:411-416

// One item of the batch (device copy of the host arguments + planner outputs).
struct ItemDesc {
    int64_t ref_start, seq_start;   // into ref_codes / seq_codes
    int64_t cig_off;                // first RLE word
    int64_t bit_word_off;           // first word of this item's op bit-string (1 = 'I', 0 = 'D'; M/=/X -> D,I)
    int64_t out_off;                // first byte of this item's region in the op scratch / final arrays (prefix of Lr+Ls)
    int32_t ref_len, seq_len;
    int32_t cig_n;                  // RLE words
    int32_t n_chunks;
    int32_t chunk_first;            // index of the item's first chunk
    int32_t total_ops;              // Lr + Ls  (= length of the D/I string of a consistent CIGAR)
    int32_t status;                 // written by the planner (BAD_CIGAR) and the traceback
    int32_t pad;
};

// One chunk (written by the plan kernel; offsets into per-sub-batch scratch are assigned on the host).
struct ChunkDesc {
    int32_t item;
    int32_t brk;        // first global anti-diagonal (index into the item's D/I string)
    int32_t B;          // anti-diagonals in the chunk: next_brk - brk + 1
    int32_t r0, c0;     // inss[brk], dels[brk]: A-space origin of the chunk
    int32_t imax, jmax; // inss[next_brk]-r0, dels[next_brk]-c0
    int32_t rlen, slen; // lengths of the np_info slices ref[c0:c1+1], seq[r0:r1+1] (clipped; aln.pyx:453-454)
    int32_t valid;
    int32_t pad[2];
};

// Scratch placement of one chunk inside the current sub-batch (assigned on the host from size upper bounds).
struct ChunkSlot {
    int64_t col_off;    // first colrec entry (32 B each); the raw scratch of the ref slice uses the same offsets
    int64_t row_off;    // first rowrec entry (4 B each); likewise for the read slice
    int64_t tb_off;     // first traceback row; row stride = 32*TBS uint16
    int32_t col_cap, row_cap;   // entries reserved (>= slice length + NP_PAD)
};

struct ChunkOut {
    float   score;      // MAT value at the chunk's end cell
    int32_t status;
    int32_t start;      // offset (within the item's op region) of the first emitted op of this chunk
    int32_t len;        // emitted ops
};

struct AlignParams {
    int r, W, max_n, max_l, max_b_rows;
    int np_dim, np_clamp;       // table side (101) and the index clamp max_l-1 (aln.pyx:269-272 as called at :615)
    int np_rows;                // max_n * (max_l+1): rows of each re-laid table; row np_rows is all +INF ("no candidate")
    float gap_open, gap_ext;
};

#define NP_FULL 0xffffffffu

static __host__ __device__ __forceinline__ int np_tbs(int cpl) { return cpl <= 1 ? 1 : cpl <= 2 ? 2 : cpl <= 4 ? 4 : 8; }

// [lo, hi) of slice `part` of n elements cut into `parts` slices of ceil(n / parts) (per-item kernels on a grid (items, parts))
__device__ __forceinline__ void np_slice(int n, int parts, int part, int &lo, int &hi)
{
    const int per = (n + parts - 1) / parts;
    lo = min(n, part * per); hi = min(n, lo + per);
}
