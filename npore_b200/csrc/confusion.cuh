// confusion.cuh -- calc_confusion_matrices (reference: src/bam.pyx:351-510) straight from the alignments.
//
// The reference shells out to `samtools mpileup | cut -f5` (bam.pyx:300-314) and walks the text of every pileup
// line with a character state machine.  Here no text exists: one warp owns one reference position of a range,
// its lanes take the reads spanning that position in BAM order, each lane locates the position inside its read's
// CIGAR by binary search over per-group prefix offsets and derives what mpileup would have printed for it
// (base / '*' / '>' ; the '+len seq' or '-len' announcement on the last position before an I / D op; the -Q 13
// base-quality filter), and the order-dependent part of the state machine (was_ins / was_del, bam.pyx:388, 409-420,
// 491-501) is resolved with ballots.  Semantics of the text this replaces: oracle/pileup_oracle.py.
//
//   per pileup LINE k (k counts printed lines = positions somebody spans; the reference indexes the reference base and
//   np_info by k, bam.pyx:386-390, 502 -- restated as is), entries e in BAM order:
//     base entry   : subs[ref_base][b]++ ; close the previous window ; open a new one            bam.pyx:404-420
//     '-' len      : window.del = 1 ; per period n with a tract starting at k+1: nps[n][l][l - len/n]++ if it is a
//                    whole number of units and fits, else nps[n][l][l]++ ; dels[min(max_l,len)]++ if no n explained it
//     '+' len seq  : window.ins = 1 ; likewise with seq == unit * (len/n) (unit = RAW reference bytes)   bam.pyx:450-484
//     '*'          : nothing (its '+' still marks the open window)
//     anything else: the rest of the line is dropped                                                bam.pyx:486-489
//     closing a window: inss[0] += !ins ; dels[0] += !del ; nps[n][l][l]++ for tract starts if neither; the window
//     open before the first base entry is never counted (flags start true).
#pragma once
#include "common.cuh"
#include "annotate.cuh"

#define CM_THREADS 256

struct ConfusionArgs {
    int n_ranges, n_reads;
    const int64_t *range_start, *range_end;      // [R]
    const uint8_t *ref_ascii; const int64_t *ref_off;   // [R+1] raw bytes contig[start : min(len, end+1+max_n)]
    uint8_t *ref_codes;                           // same layout, N A C G T - -> 0..5 (cig.pyx:212-229)
    uint8_t *raw;                                 // np_info bytes, 8 per reference byte (annotate.cuh)
    uint32_t *ebits;
    const int64_t *read_pos; const uint8_t *seq; const uint8_t *qual; const int64_t *seq_off;
    const uint32_t *rle; const int64_t *cig_off;
    int32_t *g_roff, *g_qoff;                     // per CIGAR word: reference / query offset at its start
    int64_t *read_end;                            // [n]
    const int32_t *range_reads; const int64_t *range_reads_off;   // per-range read lists (ascending position)
    int64_t *list_maxend;                         // per list entry: max read_end over the entries up to it
    int32_t *line_of; const int64_t *pos_off;     // per range position: pileup line index or -1; [R+1] prefix of range lengths
    int32_t *diff;                                // coverage difference array, pos_off layout + one per range
    unsigned long long *subs, *nps, *inss, *dels; // outputs
    int *bad;                                     // set when an unsupported CIGAR op (P, B) is seen
    int max_n, max_l, min_bq;
    // nibble form (CmNibRead): seq holds BAM's 4-bit bases, read rd's base i is nibble seq_nib_start[rd] + i; qual is phred+33
    // and only read for reads with has_qual[rd] != 0.  Last in the struct so that the ASCII form's parameter offsets stay put.
    const int64_t *seq_nib_start; const int32_t *has_qual;
};

// How cm_pileup_kernel reads a read's bases and qualities.  load() runs once per (position, read); base() returns the letter
// the ASCII form would hold at query offset off + i (upper case for the nibble form), qual() the phred value at query offset i.
struct CmAsciiRead {
    __device__ __forceinline__ void load(const ConfusionArgs &, int) {}
    __device__ __forceinline__ uint8_t base(const ConfusionArgs &a, int64_t sb, int64_t off, int i) const { return a.seq[sb + off + i]; }
    __device__ __forceinline__ int qual(const ConfusionArgs &a, int64_t sb, int i) const { return a.qual ? (int)a.qual[sb + i] : 255; }
};

// BAM's base table "=ACMGRSVTWYHKDBN" (SAM spec 4.2.3), eight letters per 64-bit immediate (byte k = letter k): the decode
// reads no memory, and no __constant__ table shifts the constant-bank layout of the other kernels of the module
constexpr uint64_t cm_pack8(const char *s) { uint64_t v = 0; for (int k = 7; k >= 0; k--) v = v << 8 | (uint8_t)s[k]; return v; }
constexpr uint64_t kCmNt16Lo = cm_pack8("=ACMGRSV"), kCmNt16Hi = cm_pack8("TWYHKDBN");
__device__ __forceinline__ uint8_t cm_nt16(uint32_t nib) { return (uint8_t)(((nib & 8u) ? kCmNt16Hi : kCmNt16Lo) >> (8 * (nib & 7u))); }

struct CmNibRead {
    int64_t nb = 0; bool hq = false;
    __device__ __forceinline__ void load(const ConfusionArgs &a, int rd) { nb = a.seq_nib_start[rd]; hq = a.qual && a.has_qual[rd]; }
    __device__ __forceinline__ uint8_t base(const ConfusionArgs &a, int64_t, int64_t off, int i) const {
        const int64_t k = nb + off + i;
        const uint8_t v = a.seq[k >> 1];
        return cm_nt16((k & 1) ? (v & 15u) : (v >> 4u));      // SAM spec 4.2.3: first base in the high nibble
    }
    __device__ __forceinline__ int qual(const ConfusionArgs &a, int64_t sb, int i) const { return hq ? (int)(uint8_t)(a.qual[sb + i] - 33) : 255; }
};

__global__ void cm_codes_kernel(const uint8_t *ascii, uint8_t *codes, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint8_t c = ascii[i];
        codes[i] = c == 'A' ? 1 : c == 'C' ? 2 : c == 'G' ? 3 : c == 'T' ? 4 : c == '-' ? 5 : 0;
    }
}

// get_np_info(bases_to_int(refs[ctg][start:end+1])) (bam.pyx:381), one CTA per range
__global__ void __launch_bounds__(ANN_THREADS) cm_np_kernel(const ConfusionArgs a)
{
    const int r = blockIdx.x;
    const int64_t b = a.ref_off[r];
    const int64_t have = a.ref_off[r + 1] - b, want = a.range_end[r] + 1 - a.range_start[r];
    const int len = (int)(have < want ? have : want);
    annotate_slice(a.ref_codes + b, len, a.max_n, a.max_l, a.raw + b * 8, nullptr,
                   len > ANN_MAX_WORDS * 32 ? a.ebits + (b >> 5) + 2 * r : nullptr);
}

// per read: reference / query offset of every CIGAR word, and the read's end.  One warp per read.
__global__ void __launch_bounds__(CM_THREADS) cm_read_kernel(const ConfusionArgs a)
{
    const int lane = threadIdx.x & 31;
    const int rd = blockIdx.x * (CM_THREADS / 32) + (threadIdx.x >> 5);
    if (rd >= a.n_reads) return;
    const int64_t c0 = a.cig_off[rd], c1 = a.cig_off[rd + 1];
    int rsum = 0, qsum = 0;
    for (int64_t base = c0; base < c1; base += 32) {
        const int64_t g = base + lane;
        int rl = 0, ql = 0;
        if (g < c1) {
            const uint32_t w = a.rle[g];
            const int op = (int)(w & 15u), n = (int)(w >> 4);
            // M I D N S H P = X : consumes reference M D N = X ; consumes query M I S = X
            if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rl = n;
            if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) ql = n;
            if (op == 6 || op > 8) *a.bad = 1;
        }
        int xr = rl, xq = ql;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int yr = __shfl_up_sync(NP_FULL, xr, o), yq = __shfl_up_sync(NP_FULL, xq, o);
            if (lane >= o) { xr += yr; xq += yq; }
        }
        if (g < c1) { a.g_roff[g] = rsum + xr - rl; a.g_qoff[g] = qsum + xq - ql; }
        rsum += __shfl_sync(NP_FULL, xr, 31); qsum += __shfl_sync(NP_FULL, xq, 31);
    }
    if (lane == 0) a.read_end[rd] = a.read_pos[rd] + rsum;
}

// per range: running maximum of read ends along its read list (bounds the candidate search of a position from below),
// which positions print a pileup line (somebody spans them) and the index of that line.  One CTA per range.
__global__ void __launch_bounds__(CM_THREADS) cm_range_kernel(const ConfusionArgs a)
{
    __shared__ long long s_w[CM_THREADS / 32];
    __shared__ int s_i[CM_THREADS / 32][2];
    __shared__ long long s_carry; __shared__ int s_c[2];
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int64_t start = a.range_start[r], end = a.range_end[r];
    const int64_t l0 = a.range_reads_off[r], l1 = a.range_reads_off[r + 1];
    int32_t *diff = a.diff + a.pos_off[r] + r;
    if (tid == 0) s_carry = INT64_MIN;
    __syncthreads();
    for (int64_t base = l0; base < l1; base += CM_THREADS) {
        const int64_t k = base + tid;
        long long v = INT64_MIN;
        if (k < l1) {
            const int rd = a.range_reads[k];
            v = a.read_end[rd];
            const int64_t lo = max(a.read_pos[rd], start), hi = min((int64_t)v, end);
            if (lo < hi) { atomicAdd(diff + (lo - start), 1); atomicAdd(diff + (hi - start), -1); }
        }
        long long x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(NP_FULL, x, o); if (lane >= o) x = max(x, y); }
        if (lane == 31) s_w[wid] = x;
        __syncthreads();
        long long p = s_carry;
        for (int q = 0; q < wid; q++) p = max(p, s_w[q]);
        x = max(x, p);
        if (k < l1) a.list_maxend[k] = x;
        __syncthreads();
        if (tid == CM_THREADS - 1) s_carry = x;
        __syncthreads();
    }
    // depth = prefix sum of diff; line index = number of spanned positions before this one
    if (tid == 0) { s_c[0] = 0; s_c[1] = 0; }
    __syncthreads();
    const int len = (int)(end - start);
    int32_t *line_of = a.line_of + a.pos_off[r];
    for (int base = 0; base < len; base += CM_THREADS) {
        const int p = base + tid;
        const int v = p < len ? diff[p] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(NP_FULL, x, o); if (lane >= o) x += y; }
        if (lane == 31) s_i[wid][0] = x;
        __syncthreads();
        int pre = s_c[0];
        for (int q = 0; q < wid; q++) pre += s_i[q][0];
        const int depth = pre + x;
        const int f = (p < len && depth > 0) ? 1 : 0;
        int y = f;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int z = __shfl_up_sync(NP_FULL, y, o); if (lane >= o) y += z; }
        if (lane == 31) s_i[wid][1] = y;
        __syncthreads();
        int pre2 = s_c[1];
        for (int q = 0; q < wid; q++) pre2 += s_i[q][1];
        if (p < len) line_of[p] = f ? pre2 + y - 1 : -1;
        __syncthreads();
        if (tid == CM_THREADS - 1) { s_c[0] = depth; s_c[1] = pre2 + y; }
        __syncthreads();
    }
}

__device__ __forceinline__ uint32_t cm_below(int k) { return k >= 32 ? 0xffffffffu : ((1u << k) - 1u); }

// one warp per reference position; CTA-local histograms for the hot counters.  Rd: CmAsciiRead or CmNibRead.
template <typename Rd>
__global__ void __launch_bounds__(CM_THREADS) cm_pileup_kernel(const ConfusionArgs a)
{
    __shared__ unsigned int s_subs[25];
    __shared__ unsigned int s_inss[128], s_dels[128];
    const int tid = threadIdx.x, lane = tid & 31;
    for (int t = tid; t < 128; t += CM_THREADS) { s_inss[t] = 0u; s_dels[t] = 0u; if (t < 25) s_subs[t] = 0u; }
    __syncthreads();
    const int64_t total = a.pos_off[a.n_ranges];
    const int max_n = a.max_n, max_l = a.max_l, T = max_l + 1;
    for (int64_t gp = (int64_t)blockIdx.x * (CM_THREADS / 32) + (tid >> 5); gp < total; gp += (int64_t)gridDim.x * (CM_THREADS / 32)) {
        // range of this position
        int lo_r = 0, hi_r = a.n_ranges - 1;
        while (lo_r < hi_r) { const int m = (lo_r + hi_r + 1) >> 1; if (a.pos_off[m] <= gp) lo_r = m; else hi_r = m - 1; }
        const int r = lo_r;
        const int x = (int)(gp - a.pos_off[r]);
        const int line = a.line_of[gp];
        if (line < 0) continue;
        const int64_t start = a.range_start[r], p = start + x;
        const int64_t rb0 = a.ref_off[r], have = a.ref_off[r + 1] - rb0;
        const int64_t want = a.range_end[r] + 1 - start;
        const int np_len = (int)(have < want ? have : want);
        const uint8_t *refa = a.ref_ascii + rb0;
        const int rbase = a.ref_codes[rb0 + line] > 4 ? 0 : a.ref_codes[rb0 + line];
        // tracts starting at line+1 (bam.pyx:413-419): bit n-1 of tmask, copies in my_l of lane n-1
        int my_l = 0;
        if (lane < max_n && line + 1 < np_len) {
            const uint8_t b = a.raw[(rb0 + line + 1) * 8 + lane];
            if ((b & 0x80u) && (b & 0x7fu)) my_l = b & 0x7f;
        }
        const uint32_t tmask = __ballot_sync(NP_FULL, my_l != 0);
        // candidate reads: list entries [lo, hi)
        const int64_t l0 = a.range_reads_off[r], l1 = a.range_reads_off[r + 1];
        int64_t lo = l0, hi = l1;
        {   // hi = first entry whose read starts after p
            int64_t u = l0, v = l1;
            while (u < v) { const int64_t m = (u + v) >> 1; if (a.read_pos[a.range_reads[m]] <= p) u = m + 1; else v = m; }
            hi = u;
            u = l0; v = hi;   // lo = first entry with running max end > p
            while (u < v) { const int64_t m = (u + v) >> 1; if (a.list_maxend[m] > p) v = m; else u = m + 1; }
            lo = u;
        }
        bool c_ins = true, c_del = true;          // flags of the open window (bam.pyx:388)
        int n_noins = 0, n_nodel = 0, n_neither = 0;
        for (int64_t k0 = lo; k0 < hi; k0 += 32) {
            const int64_t k = k0 + lane;
            bool entry = false, err = false, isbase = false;
            int code = 0, indel = 0;
            int64_t q0 = 0, sb = 0; int lq = 0;
            Rd rdr;
            if (k < hi) {
                const int rd = a.range_reads[k];
                if (p < a.read_end[rd]) {
                    const int xr = (int)(p - a.read_pos[rd]);
                    const int64_t c0 = a.cig_off[rd], c1 = a.cig_off[rd + 1];
                    int64_t u = c0, v = c1;       // last word with g_roff <= xr
                    while (v - u > 1) { const int64_t m = (u + v) >> 1; if (a.g_roff[m] <= xr) u = m; else v = m; }
                    const uint32_t w = a.rle[u];
                    const int op = (int)(w & 15u), n = (int)(w >> 4), t = xr - a.g_roff[u];
                    const bool is_del = (op == 2 || op == 3);
                    const int qoff = a.g_qoff[u];
                    const int qpos = is_del ? qoff : qoff + t;
                    sb = a.seq_off[rd]; lq = (int)(a.seq_off[rd + 1] - sb);
                    rdr.load(a, rd);
                    if (t == n - 1 && u + 1 < c1) {        // announcement of the next op (htslib resolve_cigar2)
                        const int op2 = (int)(a.rle[u + 1] & 15u);
                        if (op2 == 2 && op != 2) { for (int64_t g = u + 1; g < c1 && (a.rle[g] & 15u) == 2u; g++) indel -= (int)(a.rle[g] >> 4); }
                        else if (op2 == 1) { for (int64_t g = u + 1; g < c1 && (a.rle[g] & 15u) == 1u; g++) indel += (int)(a.rle[g] >> 4); }
                    }
                    const int q = qpos < lq ? rdr.qual(a, sb, qpos) : 0;
                    entry = q >= a.min_bq;
                    if (is_del) err = (op == 3);
                    else {
                        uint8_t ch = qpos < lq ? rdr.base(a, sb, qpos, 0) : (uint8_t)'N';
                        if (ch >= 'a' && ch <= 'z') ch -= 32;
                        code = ch == 'N' ? 0 : ch == 'A' ? 1 : ch == 'C' ? 2 : ch == 'G' ? 3 : ch == 'T' ? 4 : -1;
                        err = code < 0; isbase = !err;
                    }
                    q0 = is_del ? qoff : qoff + n;
                }
            }
            const uint32_t E = __ballot_sync(NP_FULL, entry);
            const uint32_t ERR = __ballot_sync(NP_FULL, entry && err);
            const uint32_t V = E & (ERR ? cm_below(__ffs(ERR) - 1) : 0xffffffffu);
            const bool live = (V >> lane) & 1u;
            const uint32_t Bm = __ballot_sync(NP_FULL, live && isbase);
            const uint32_t Im = __ballot_sync(NP_FULL, live && indel > 0);
            const uint32_t Dm = __ballot_sync(NP_FULL, live && indel < 0);
            // substitutions (bam.pyx:404-406)
#pragma unroll
            for (int v = 0; v < 5; v++) {
                const uint32_t m = __ballot_sync(NP_FULL, live && isbase && code == v);
                if (lane == v && m) atomicAdd(&s_subs[rbase * 5 + v], (unsigned)__popc(m));
            }
            // windows closed by this chunk's base entries
            bool wi = true, wd = true;
            if (live && isbase) {
                const uint32_t prev = Bm & cm_below(lane);
                if (prev) {
                    const uint32_t m = cm_below(lane) & ~cm_below(31 - __clz(prev));
                    wi = (Im & m) != 0u; wd = (Dm & m) != 0u;
                } else {
                    const uint32_t m = cm_below(lane);
                    wi = c_ins || (Im & m) != 0u; wd = c_del || (Dm & m) != 0u;
                }
            }
            n_noins += __popc(__ballot_sync(NP_FULL, !wi));
            n_nodel += __popc(__ballot_sync(NP_FULL, !wd));
            n_neither += __popc(__ballot_sync(NP_FULL, !wi && !wd));
            if (Bm) {
                const uint32_t m = ~cm_below(31 - __clz(Bm));
                c_ins = (Im & m) != 0u; c_del = (Dm & m) != 0u;
            } else { c_ins = c_ins || Im != 0u; c_del = c_del || Dm != 0u; }
            // the indel announcements themselves (bam.pyx:422-484)
            if (live && indel != 0) {
                const int len = indel < 0 ? -indel : indel;
                bool explained = false;
                for (int n = 1; n <= max_n; n++) {
                    if (!((tmask >> (n - 1)) & 1u)) continue;
                    // (my_l of lane n-1; fetched without a shuffle because this code is divergent)
                    const int l = a.raw[(rb0 + line + 1) * 8 + n - 1] & 0x7f;
                    bool cnv = (len % n) == 0;
                    int call = l;
                    if (cnv && indel < 0) { cnv = len <= l * n; call = l - len / n; }
                    else if (cnv) {
                        if ((int64_t)line + 1 + n > have) cnv = false;       // unit clipped at the contig end never matches
                        for (int i = 0; cnv && i < len; i++) {
                            uint8_t ch = (q0 + i) < lq ? rdr.base(a, sb, q0, i) : (uint8_t)0;
                            if (ch >= 'a' && ch <= 'z') ch -= 32;
                            cnv = ch == refa[line + 1 + (i % n)];
                        }
                        call = min(max_l, l + len / n);
                    }
                    if (cnv) { explained = true; atomicAdd(a.nps + ((size_t)(n - 1) * T + l) * T + call, 1ull); }
                    else atomicAdd(a.nps + ((size_t)(n - 1) * T + l) * T + l, 1ull);
                }
                if (!explained) atomicAdd(indel < 0 ? &s_dels[min(max_l, len)] : &s_inss[min(max_l, len)], 1u);
            }
            if (ERR) break;                       // bam.pyx:486-489: the rest of the line is not read
        }
        // end of line: the last window (bam.pyx:491-501)
        if (!c_ins) n_noins++;
        if (!c_del) n_nodel++;
        if (!c_ins && !c_del) n_neither++;
        if (lane == 0) { if (n_noins) atomicAdd(&s_inss[0], (unsigned)n_noins); if (n_nodel) atomicAdd(&s_dels[0], (unsigned)n_nodel); }
        if (n_neither && lane < max_n && my_l) atomicAdd(a.nps + ((size_t)lane * T + my_l) * T + my_l, (unsigned long long)n_neither);
    }
    __syncthreads();
    for (int t = tid; t < 128; t += CM_THREADS) {
        if (t < 25 && s_subs[t]) atomicAdd(a.subs + t, (unsigned long long)s_subs[t]);
        if (t <= max_l && s_inss[t]) atomicAdd(a.inss + t, (unsigned long long)s_inss[t]);
        if (t <= max_l && s_dels[t]) atomicAdd(a.dels + t, (unsigned long long)s_dels[t]);
    }
}
