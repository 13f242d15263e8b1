// finish.cuh -- per-item epilogue on device:
//   item_len / gather    concatenate the chunks' op strings (aln.pyx:742 `full_aln += aln[::-1]`), one CTA per chunk
//   rle_* kernels        src/cig.pyx:13-38 collapse_cigar as BAM-style words (len<<4 | op); with `to_m` set X and = are
//                        first mapped to M (bam.pyx:65)
//   standardize_kernel   src/bam.pyx:65-78 in the RUN-LENGTH domain: push_indels_left(D, ref); push_inss_thru_dels;
//                        push_indels_left(I, seq); push_inss_thru_dels (src/cig.pyx:102-192; the reference's `while True`
//                        body runs exactly once because old_cig aliases int_cig); 'ID' -> 'M'.  Each pass is one
//                        sequential sweep over the item's groups with a stack-like output (O(#groups), ~1000 per 10 kb
//                        read, instead of the reference's 4 sweeps over every op), one warp (lane 0) per item.
//   expand_* kernels     run-length words -> one char per op (the expanded 'MID' string realign_hap returns)
//   scan / pack kernels  exclusive prefix of the per-item output sizes and a dense copy, so that the D2H transfer moves
//                        exactly the bytes the caller gets.
#pragma once
#include "common.cuh"

#define FIN_THREADS 128
#define FIN_WIDE 256             // threads of the part-parallel kernels
#define FIN_MAX_PARTS 64

// Items differ in size by four orders of magnitude (a 10 kb read has 2e4 ops, a whole-contig haplotype 1e8): every
// per-item kernel below runs on a grid (items, parts) and a CTA handles the part-th slice of its item; `parts` is chosen
// on the host from the largest item (1 for read batches).  Slices that need a running count across the item (group
// indices, output offsets) get it from a small counting pass (part_cnt) summed over the preceding parts.
struct FinishArgs {
    const ItemDesc *items; int n_items;
    const ChunkDesc *chunks; int n_chunks;
    const ChunkOut *chunk_out;
    int32_t *chunk_dst;           // per chunk: offset of its piece inside the item's op string
    const uint8_t *scratch;       // right-aligned chunk pieces
    uint8_t *ops;                 // per-item op strings (item region at out_off)
    int32_t *item_len;            // ops per item
    int32_t *item_status;
    const uint8_t *ref_codes, *seq_codes;
    uint32_t *rleA, *rleB;        // per-item group buffers (item region at out_off), ping-pong
    int32_t *rle_len;
    int32_t *rle_which;           // 0: result in rleA, 1: in rleB
    int to_m;
    int parts; int32_t *part_cnt; // [n_items * parts]
    // packing
    int64_t *ops_off, *rle_off;   // [n+1] exclusive prefixes (device)
    uint8_t *pack_ops; uint32_t *pack_rle;
};

// block-wide inclusive scan of one int per thread; returns the inclusive value, `total` = sum over the block.
// s_w: shared int[blockDim/32].  Ends with a barrier, so s_w can be reused by the next call.
template <int THREADS>
__device__ __forceinline__ int fin_block_scan(int v, int *s_w, int &total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(NP_FULL, x, o); if (lane >= o) x += y; }
    if (lane == 31) s_w[wid] = x;
    __syncthreads();
    int pre = 0, tot = 0;
#pragma unroll
    for (int q = 0; q < THREADS / 32; q++) { const int t = s_w[q]; if (q < wid) pre += t; tot += t; }
    __syncthreads();
    total = tot;
    return pre + x;
}

// where each chunk's op string goes inside its item (aln.pyx:742 `full_aln += aln[::-1]`), the item's length and status
__global__ void __launch_bounds__(FIN_THREADS) item_len_kernel(const FinishArgs a)
{
    __shared__ int s_w[FIN_THREADS / 32];
    __shared__ int s_first;
    const int it = blockIdx.x;
    const ItemDesc &I = a.items[it];
    if (threadIdx.x == 0) s_first = 0x7fffffff;
    __syncthreads();
    int carry = 0;
    for (int base = 0; base < I.n_chunks; base += FIN_THREADS) {
        const int k = base + threadIdx.x;
        int len = 0;
        if (k < I.n_chunks) {
            const ChunkOut co = a.chunk_out[I.chunk_first + k];
            len = co.len;
            if (co.status) atomicMin(&s_first, k);
        }
        int tot;
        const int x = fin_block_scan<FIN_THREADS>(len, s_w, tot);
        if (k < I.n_chunks) a.chunk_dst[I.chunk_first + k] = carry + x - len;
        carry += tot;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        a.item_len[it] = carry;
        a.item_status[it] = I.status ? I.status : (s_first != 0x7fffffff ? a.chunk_out[I.chunk_first + s_first].status : 0);
    }
}

// one CTA per chunk: copy the chunk's op string to its place
__global__ void __launch_bounds__(FIN_THREADS) gather_kernel(const FinishArgs a)
{
    const int c = blockIdx.x;
    const ItemDesc &I = a.items[a.chunks[c].item];
    const ChunkOut co = a.chunk_out[c];
    uint8_t *dst = a.ops + I.out_off + a.chunk_dst[c];
    const uint8_t *src = a.scratch + I.out_off + co.start;
    for (int t = threadIdx.x; t < co.len; t += FIN_THREADS) dst[t] = src[t];
}

__device__ __forceinline__ uint32_t op_code(uint8_t ch, int to_m)
{
    if (ch == 'I') return 1u;
    if (ch == 'D') return 2u;
    if (to_m || ch == 'M') return 0u;
    return ch == '=' ? 7u : 8u;                                   // cfg.py:28-32
}

// ---- expanded chars -> run-length words (cig.pyx:13-38) in three part-parallel steps
// (1) group starts per slice
__global__ void __launch_bounds__(FIN_WIDE) rle_count_kernel(const FinishArgs a)
{
    __shared__ int s_w[FIN_WIDE / 32];
    const int it = blockIdx.x, part = blockIdx.y;
    const uint8_t *c = a.ops + a.items[it].out_off;
    int lo, hi;
    np_slice(a.item_len[it], a.parts, part, lo, hi);
    int cnt = 0;
    for (int k = lo + threadIdx.x; k < hi; k += FIN_WIDE) cnt += (k == 0) || (op_code(c[k], a.to_m) != op_code(c[k - 1], a.to_m));
    int tot;
    fin_block_scan<FIN_WIDE>(cnt, s_w, tot);
    if (threadIdx.x == 0) a.part_cnt[it * a.parts + part] = tot;
}

// (2) start position of every group -> rleB (scratch); 4 consecutive ops per thread
__global__ void __launch_bounds__(FIN_WIDE) rle_start_kernel(const FinishArgs a)
{
    __shared__ int s_w[FIN_WIDE / 32];
    const int it = blockIdx.x, part = blockIdx.y;
    const ItemDesc &I = a.items[it];
    const uint8_t *c = a.ops + I.out_off;
    uint32_t *startp = a.rleB + I.out_off;
    int lo, hi;
    np_slice(a.item_len[it], a.parts, part, lo, hi);
    int carry = 0;
    if (a.parts > 1) for (int q = 0; q < part; q++) carry += a.part_cnt[it * a.parts + q];
    for (int base = lo; base < hi; base += FIN_WIDE * 4) {
        const int k0 = base + threadIdx.x * 4;
        uint32_t prev = (k0 > 0 && k0 < hi) ? op_code(c[k0 - 1], a.to_m) : 0xffu;
        uint32_t fl = 0u;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (k0 + j < hi) {
                const uint32_t o = op_code(c[k0 + j], a.to_m);
                if (o != prev) fl |= 1u << j;
                prev = o;
            }
        }
        int tot;
        int at = carry + fin_block_scan<FIN_WIDE>(__popc(fl), s_w, tot) - __popc(fl);
#pragma unroll
        for (int j = 0; j < 4; j++) if ((fl >> j) & 1u) startp[at++] = (uint32_t)(k0 + j);
        carry += tot;
    }
    if (part == a.parts - 1 && threadIdx.x == 0) { a.rle_len[it] = carry; a.rle_which[it] = 0; }
}

// (3) words from consecutive starts
__global__ void __launch_bounds__(FIN_WIDE) rle_word_kernel(const FinishArgs a)
{
    const int it = blockIdx.x;
    const ItemDesc &I = a.items[it];
    const uint8_t *c = a.ops + I.out_off;
    uint32_t *w = a.rleA + I.out_off;
    const uint32_t *startp = a.rleB + I.out_off;
    const int n = a.item_len[it], m = a.rle_len[it];
    int lo, hi;
    np_slice(m, a.parts, blockIdx.y, lo, hi);
    for (int g = lo + threadIdx.x; g < hi; g += FIN_WIDE) {
        const uint32_t st = startp[g], en = (g + 1 < m) ? startp[g + 1] : (uint32_t)n;
        w[g] = ((en - st) << 4) | op_code(c[st], a.to_m);
    }
}

// ---- stack-like output list of run-length groups (merges equal neighbours, drops empty groups).  The top group lives in
// a register, so a sweep's loop-carried dependency never goes through memory (a store followed by a load of the same
// word costs an L1/L2 round trip per group; the sweeps are latency-bound).
struct GroupStack {
    uint32_t *g; int m; uint32_t top;              // groups 0..m-2 are in g[], group m-1 is `top`
    __device__ __forceinline__ void push(uint32_t op, uint32_t len)
    {
        if (!len) return;
        if (m > 0 && (top & 15u) == op) top += len << 4;
        else { if (m > 0) g[m - 1] = top; top = (len << 4) | op; m++; }
    }
    __device__ __forceinline__ bool top_is(uint32_t op) const { return m > 0 && (top & 15u) == op; }
    __device__ __forceinline__ uint32_t top_len() const { return top >> 4; }
    __device__ __forceinline__ void pop() { m--; if (m > 0) top = g[m - 1]; }
    __device__ __forceinline__ void shrink(uint32_t k) { top -= k << 4; if ((top >> 4) == 0u) pop(); }
    __device__ __forceinline__ int finish() { if (m > 0) g[m - 1] = top; return m; }
};

// cig.pyx:102-159 on groups.  sp counts M ops and push_op runs passed (= position in `seq`, which is the reference for
// push_op == D and the read for push_op == I).  A run of push_op of length L preceded by an M group moves left over k of
// those M's, k = number of consecutive t with seq[sp-t-1] == seq[sp-t-1+L].
__device__ __forceinline__ int rle_push_indels_left(const uint32_t *in, int m, uint32_t *out, const uint8_t *__restrict__ seq, uint32_t push_op,
                                                    const int32_t *eq_run = nullptr)
{
    GroupStack st{out, 0, 0u};
    int sp = 0;
    for (int g = 0; g < m; g++) {
        const uint32_t op = in[g] & 15u, len = in[g] >> 4;
        if (op != push_op) { st.push(op, len); if (op == 0u) sp += (int)len; continue; }
        int k = 0;
        if (st.top_is(0u)) {
            const int lim = min((int)st.top_len(), sp);
            if (eq_run) k = min(eq_run[g], lim);
            else while (k < lim && seq[sp - k - 1] == seq[sp - k - 1 + (int)len]) k++;
            if (k) st.shrink((uint32_t)k);
        }
        st.push(push_op, len);
        st.push(0u, (uint32_t)k);
        sp += (int)len;
    }
    return st.finish();
}

// The base comparisons of rle_push_indels_left do not depend on the stack: for the run of push_op at group g,
// eq_run[g] = number of consecutive t with seq[sp-t-1] == seq[sp-t-1+len], sp = ops of kind M / push_op before g.
// The whole warp computes them (a scan for sp, one lane per run), so the cold byte loads of all runs overlap instead of
// sitting one after the other inside the sequential sweep.
__device__ __forceinline__ void rle_eq_runs(const uint32_t *in, int m, const uint8_t *__restrict__ seq, uint32_t push_op, int32_t *eq_run)
{
    const int lane = threadIdx.x & 31;
    int carry = 0;
    for (int base = 0; base < m; base += 32) {
        const int g = base + lane;
        const uint32_t w = g < m ? in[g] : 0u, op = w & 15u;
        const int len = (int)(w >> 4);
        const int adv = (g < m && (op == 0u || op == push_op)) ? len : 0;
        int x = adv;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(NP_FULL, x, o); if (lane >= o) x += y; }
        const int sp = carry + x - adv;
        if (g < m && op == push_op) {
            int k = 0;
            while (k < sp && seq[sp - k - 1] == seq[sp - k - 1 + len]) k++;
            eq_run[g] = k;
        }
        carry += __shfl_sync(NP_FULL, x, 31);
    }
    __syncwarp();
}

// cig.pyx:164-192 on groups: an I run that follows a D run is moved in front of it
__device__ __forceinline__ int rle_push_inss_thru_dels(const uint32_t *in, int m, uint32_t *out)
{
    GroupStack st{out, 0, 0u};
    for (int g = 0; g < m; g++) {
        const uint32_t op = in[g] & 15u, len = in[g] >> 4;
        if (op == 1u && st.top_is(2u)) {
            const uint32_t d = st.top_len();
            st.pop();
            st.push(1u, len);
            st.push(2u, d);
        } else st.push(op, len);
    }
    return st.finish();
}

// bam.pyx:78  .replace('ID','M') on groups: the last I of a run and the first D of the run that follows become one M
__device__ __forceinline__ int rle_id_to_m(const uint32_t *in, int m, uint32_t *out)
{
    GroupStack st{out, 0, 0u};
    for (int g = 0; g < m; g++) {
        const uint32_t op = in[g] & 15u, len = in[g] >> 4;
        if (op == 2u && st.top_is(1u)) {
            st.shrink(1u);
            st.push(0u, 1u);
            st.push(2u, len - 1u);
        } else st.push(op, len);
    }
    return st.finish();
}

// one item per WARP: lane 0 does the sweeps (32 different sequential sweeps inside one warp would serialise), all lanes
// prepare the base comparisons of the two push_indels_left sweeps.  The comparison results go to the upper half of the
// input buffer's item region (capacity Lref+Lseq words, of which the groups use the first m).
__global__ void __launch_bounds__(FIN_THREADS) standardize_kernel(const FinishArgs a)
{
    const int it = blockIdx.x * (FIN_THREADS / 32) + (threadIdx.x >> 5);
    if (it >= a.n_items) return;
    if (a.rle_which[it] != 0) return;                             // already standardised by standardize_long_kernel (launched first)
    const bool lead = (threadIdx.x & 31) == 0;
    const ItemDesc &I = a.items[it];
    uint32_t *A = a.rleA + I.out_off, *B = a.rleB + I.out_off;
    const uint8_t *ref = a.ref_codes + I.ref_start, *seq = a.seq_codes + I.seq_start;
    const int cap = I.total_ops;
    int32_t *E = reinterpret_cast<int32_t *>(A + cap / 2);
    int m = a.rle_len[it];
    bool pre = 2 * m <= cap;
    if (pre) rle_eq_runs(A, m, ref, 2u, E);
    if (lead) {
        m = rle_push_indels_left(A, m, B, ref, 2u, pre ? E : nullptr);
        m = rle_push_inss_thru_dels(B, m, A);
    }
    m = __shfl_sync(NP_FULL, m, 0);
    __threadfence_block();
    __syncwarp();
    pre = 2 * m <= cap;
    if (pre) rle_eq_runs(A, m, seq, 1u, E);
    if (!lead) return;
    m = rle_push_indels_left(A, m, B, seq, 1u, pre ? E : nullptr);
    m = rle_push_inss_thru_dels(B, m, A);
    m = rle_id_to_m(A, m, B);
    int tot = 0;
    for (int g = 0; g < m; g++) tot += (int)(B[g] >> 4);
    a.rle_len[it] = m; a.rle_which[it] = 1; a.item_len[it] = tot;
}

// ---- the same five sweeps for LONG items (whole-contig haplotypes: 1e4..1e6 groups), one CTA per item.
// A single lane needs ~150 ns per group and sweep; here the group list is cut into segments at M groups that no shift
// can consume (for the push sweeps: the equality run of the next indel is shorter than the M group; for the other sweeps:
// any M group), every thread runs the SAME sequential routine on its own segment, and the segment outputs are
// concatenated and equal neighbours merged.  Anything that does not fit the scratch layout falls back to one thread.
#define STDL_BLOCK 48

__device__ __forceinline__ bool stdl_safe_cut(const uint32_t *X, int m, int g, int kind, uint32_t push_op, const int32_t *E)
{
    if (g == 0) return true;
    if ((X[g] & 15u) != 0u) return false;
    if (kind != 0) return true;                                   // thru_dels / id_to_m: every M group separates
    return g + 1 >= m || (X[g + 1] & 15u) != push_op || E[g + 1] < (int)(X[g] >> 4);
}

// one sweep: dense X[0,m) -> dense Y[0,m'); kind 0 = push_indels_left(push_op, seq), 1 = push_inss_thru_dels, 2 = id_to_m
__device__ int stdl_sweep(int kind, uint32_t push_op, const uint8_t *__restrict__ seq, uint32_t *X, int m, uint32_t *Y, int cap, int *s_w)
{
    __shared__ int s_m;
    const int tid = threadIdx.x;
    const int nblk = (m + STDL_BLOCK - 1) / STDL_BLOCK;
    const bool fits = m > 0 && (long long)4 * m + 3ll * (nblk + 2) + 64 <= cap;
    if (!fits) {                                                  // sequential fallback (also m == 0)
        if (tid == 0)
            s_m = kind == 0 ? rle_push_indels_left(X, m, Y, seq, push_op) : kind == 1 ? rle_push_inss_thru_dels(X, m, Y) : rle_id_to_m(X, m, Y);
        __syncthreads();
        const int r = s_m;
        __syncthreads();
        return r;
    }
    int32_t *E = reinterpret_cast<int32_t *>(X + cap / 2);         // [m]   equality runs (push sweeps)
    int32_t *S = reinterpret_cast<int32_t *>(Y + cap) - (nblk + 2);   // [nblk+1] segment starts
    int32_t *Cn = S - (nblk + 2), *O = Cn - (nblk + 2);           // [nblk+1] output counts, offsets
    if (kind == 0) {                                              // CTA-wide rle_eq_runs
        int carry = 0;
        for (int base = 0; base < m; base += FIN_WIDE) {
            const int g = base + tid;
            const uint32_t w = g < m ? X[g] : 0u, op = w & 15u;
            const int len = (int)(w >> 4);
            const int adv = (g < m && (op == 0u || op == push_op)) ? len : 0;
            int tot;
            const int sp = carry + fin_block_scan<FIN_WIDE>(adv, s_w, tot) - adv;
            if (g < m && op == push_op) {
                int k = 0;
                while (k < sp && seq[sp - k - 1] == seq[sp - k - 1 + len]) k++;
                E[g] = k;
            }
            carry += tot;
        }
        __syncthreads();
    }
    for (int b = tid; b <= nblk; b += FIN_WIDE) {                 // segment b = [S[b], S[b+1])
        int g = min(b * STDL_BLOCK, m);
        while (g < m && !stdl_safe_cut(X, m, g, kind, push_op, E)) g++;
        S[b] = g;
    }
    __syncthreads();
    for (int b = tid; b < nblk; b += FIN_WIDE) {
        const int g0 = S[b], n = S[b + 1] - g0;
        int c = 0;
        if (n > 0) {
            uint32_t *out = Y + 2 * g0;
            c = kind == 0 ? rle_push_indels_left(X + g0, n, out, seq, push_op, E + g0)
              : kind == 1 ? rle_push_inss_thru_dels(X + g0, n, out) : rle_id_to_m(X + g0, n, out);
        }
        Cn[b] = c;
    }
    __syncthreads();
    int carry = 0;
    for (int base = 0; base < nblk; base += FIN_WIDE) {
        const int b = base + tid;
        const int c = b < nblk ? Cn[b] : 0;
        int tot;
        const int x = fin_block_scan<FIN_WIDE>(c, s_w, tot);
        if (b < nblk) O[b] = carry + x - c;
        carry += tot;
    }
    const int md = carry;                                         // groups before merging
    __syncthreads();
    for (int b = tid; b < nblk; b += FIN_WIDE) {                  // dense concatenation into X (its old contents are dead)
        const uint32_t *src = Y + 2 * S[b];
        uint32_t *dst = X + O[b];
        for (int j = 0, c = Cn[b]; j < c; j++) dst[j] = src[j];
    }
    __syncthreads();
    carry = 0;                                                    // merge equal neighbours: X[0,md) -> Y[0,m')
    for (int base = 0; base < md; base += FIN_WIDE) {
        const int j = base + tid;
        const uint32_t w = j < md ? X[j] : 0u;
        const int head = (j < md && (j == 0 || (X[j - 1] & 15u) != (w & 15u))) ? 1 : 0;
        int tot;
        const int x = fin_block_scan<FIN_WIDE>(head, s_w, tot);
        if (head) {
            uint32_t acc = w;
            for (int t = j + 1; t < md && (X[t] & 15u) == (w & 15u); t++) acc += X[t] & ~15u;
            Y[carry + x - 1] = acc;
        }
        carry += tot;
    }
    __syncthreads();
    return carry;
}

__global__ void __launch_bounds__(FIN_WIDE) standardize_long_kernel(const FinishArgs a, int min_groups)
{
    __shared__ int s_w[FIN_WIDE / 32];
    const int it = blockIdx.x;
    int m = a.rle_len[it];
    if (m < min_groups) return;                                   // (short items: standardize_kernel)
    const ItemDesc &I = a.items[it];
    uint32_t *A = a.rleA + I.out_off, *B = a.rleB + I.out_off;
    const uint8_t *ref = a.ref_codes + I.ref_start, *seq = a.seq_codes + I.seq_start;
    const int cap = I.total_ops;
    m = stdl_sweep(0, 2u, ref, A, m, B, cap, s_w);
    m = stdl_sweep(1, 0u, nullptr, B, m, A, cap, s_w);
    m = stdl_sweep(0, 1u, seq, A, m, B, cap, s_w);
    m = stdl_sweep(1, 0u, nullptr, B, m, A, cap, s_w);
    m = stdl_sweep(2, 0u, nullptr, A, m, B, cap, s_w);
    int part = 0;
    for (int g = threadIdx.x; g < m; g += FIN_WIDE) part += (int)(B[g] >> 4);
    int tot;
    fin_block_scan<FIN_WIDE>(part, s_w, tot);
    if (threadIdx.x == 0) { a.rle_len[it] = m; a.rle_which[it] = 1; a.item_len[it] = tot; }
}

// ---- run-length words -> chars (the expanded 'MID' string realign_hap returns), two part-parallel steps
__global__ void __launch_bounds__(FIN_WIDE) expand_count_kernel(const FinishArgs a)
{
    __shared__ int s_w[FIN_WIDE / 32];
    const int it = blockIdx.x, part = blockIdx.y;
    const uint32_t *w = (a.rle_which[it] ? a.rleB : a.rleA) + a.items[it].out_off;
    int lo, hi;
    np_slice(a.rle_len[it], a.parts, part, lo, hi);
    int cnt = 0;
    for (int g = lo + threadIdx.x; g < hi; g += FIN_WIDE) cnt += (int)(w[g] >> 4);
    int tot;
    fin_block_scan<FIN_WIDE>(cnt, s_w, tot);
    if (threadIdx.x == 0) a.part_cnt[it * a.parts + part] = tot;
}

// short groups are written by their own thread, long ones (haplotype-sized M runs) by a whole warp
__global__ void __launch_bounds__(FIN_WIDE) expand_fill_kernel(const FinishArgs a)
{
    __shared__ int s_w[FIN_WIDE / 32];
    __shared__ int s_long[FIN_WIDE][2];
    __shared__ int s_nlong;
    const int it = blockIdx.x, part = blockIdx.y;
    const ItemDesc &I = a.items[it];
    const uint32_t *w = (a.rle_which[it] ? a.rleB : a.rleA) + I.out_off;
    uint8_t *c = a.ops + I.out_off;
    int lo, hi;
    np_slice(a.rle_len[it], a.parts, part, lo, hi);
    int carry = 0;
    if (a.parts > 1) for (int q = 0; q < part; q++) carry += a.part_cnt[it * a.parts + q];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int base = lo; base < hi; base += FIN_WIDE) {
        const int g = base + threadIdx.x;
        const uint32_t word = g < hi ? w[g] : 0u;
        const int len = (int)(word >> 4);
        if (threadIdx.x == 0) s_nlong = 0;
        int tot;
        const int start = carry + fin_block_scan<FIN_WIDE>(len, s_w, tot) - len;      // (barrier inside: s_nlong visible)
        if (len > 16) { const int q = atomicAdd(&s_nlong, 1); s_long[q][0] = start; s_long[q][1] = (int)word; }
        else { const uint8_t ch = "MIDNSHP=XB"[word & 15u]; for (int t = 0; t < len; t++) c[start + t] = ch; }
        __syncthreads();
        for (int q = wid; q < s_nlong; q += FIN_WIDE / 32) {
            const int st = s_long[q][0], ln = s_long[q][1] >> 4;
            const uint8_t ch = "MIDNSHP=XB"[s_long[q][1] & 15];
            for (int t = lane; t < ln; t += 32) c[st + t] = ch;
        }
        __syncthreads();
        carry += tot;
    }
}

// exclusive prefix sums of item_len / rle_len over items (single CTA; n is small next to the DP)
__global__ void __launch_bounds__(1024) scan_kernel(const FinishArgs a)
{
    __shared__ long long s_w[32][2];
    __shared__ long long s_carry[2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_carry[0] = s_carry[1] = 0; }
    __syncthreads();
    for (int base = 0; base < a.n_items; base += 1024) {
        const int it = base + threadIdx.x;
        long long v0 = it < a.n_items ? a.item_len[it] : 0, v1 = it < a.n_items ? a.rle_len[it] : 0;
        long long x0 = v0, x1 = v1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y0 = __shfl_up_sync(NP_FULL, x0, o), y1 = __shfl_up_sync(NP_FULL, x1, o);
            if (lane >= o) { x0 += y0; x1 += y1; }
        }
        if (lane == 31) { s_w[wid][0] = x0; s_w[wid][1] = x1; }
        __syncthreads();
        long long p0 = s_carry[0], p1 = s_carry[1];
        for (int q = 0; q < wid; q++) { p0 += s_w[q][0]; p1 += s_w[q][1]; }
        if (it < a.n_items) { a.ops_off[it] = p0 + x0 - v0; a.rle_off[it] = p1 + x1 - v1; }
        __syncthreads();
        if (threadIdx.x == 1023) { s_carry[0] = p0 + x0; s_carry[1] = p1 + x1; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { a.ops_off[a.n_items] = s_carry[0]; a.rle_off[a.n_items] = s_carry[1]; }
}

__global__ void __launch_bounds__(FIN_WIDE) pack_kernel(const FinishArgs a, int want_ops, int want_rle)
{
    const int it = blockIdx.x;
    const ItemDesc &I = a.items[it];
    int lo, hi;
    if (want_ops) {
        const uint8_t *src = a.ops + I.out_off; uint8_t *dst = a.pack_ops + a.ops_off[it];
        np_slice(a.item_len[it], a.parts, blockIdx.y, lo, hi);
        for (int t = lo + threadIdx.x; t < hi; t += FIN_WIDE) dst[t] = src[t];
    }
    if (want_rle) {
        const uint32_t *src = (a.rle_which[it] ? a.rleB : a.rleA) + I.out_off; uint32_t *dst = a.pack_rle + a.rle_off[it];
        np_slice(a.rle_len[it], a.parts, blockIdx.y, lo, hi);
        for (int t = lo + threadIdx.x; t < hi; t += FIN_WIDE) dst[t] = src[t];
    }
}
