// plan.cuh -- align() prologue on device (reference: src/aln.pyx:386-392).
//
//   * CIGAR -> D/I op string (aln.pyx:386: every X,=,M becomes "DI"), stored as ONE BIT per op (1 = 'I').
//     inss[g] (aln.pyx:279-292) is then a rank query: cumI[g>>5] + popc(low bits); dels[g] = g - inss[g]
//     (aln.pyx:296-311), so the two int32[P+1] prefix arrays of the reference are never materialised.
//   * get_breaks (aln.pyx:344-358) -> one ChunkDesc per chunk, including the "don't split a DI pair" shift.
// Block-wide scans over the item's RLE words / bit words (kernels at the end of this file).
#pragma once
#include "common.cuh"

#define PLAN_THREADS 256

__device__ __forceinline__ int plan_block_exscan(int v, int *s_warp, int &total)
{
    // exclusive scan of one int per thread across the CTA; returns this thread's prefix, total = CTA sum
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(NP_FULL, x, o); if (lane >= o) x += y; }
    if (lane == 31) s_warp[wid] = x;
    __syncthreads();
    if (wid == 0) {
        int w = lane < (PLAN_THREADS / 32) ? s_warp[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(NP_FULL, w, o); if (lane >= o) w += y; }
        if (lane < (PLAN_THREADS / 32)) s_warp[lane] = w;      // inclusive per-warp sums
    }
    __syncthreads();
    const int base = wid ? s_warp[wid - 1] : 0;
    total = s_warp[PLAN_THREADS / 32 - 1];
    __syncthreads();
    return base + x - v;
}

__device__ __forceinline__ uint32_t plan_rank(const uint32_t *bits, const uint32_t *cum, int g)
{
    const uint32_t w = bits[g >> 5];
    return cum[g >> 5] + __popc(w & ((1u << (g & 31)) - 1u));
}

// The prologue runs as four kernels so that an item of any length (a 64 Mb haplotype has 4e6 bit words) is not one
// CTA's job: groups (1 CTA / item), bit words + popcount partial sums (items x parts), popcount prefix (items x parts),
// chunk descriptors (items x parts).  `parts` comes from the largest item of the batch (1 for read batches).
struct PlanArgs {
    ItemDesc *items; int n_items;
    const uint32_t *rle; int32_t *grp_off;
    uint32_t *bits, *cum;
    ChunkDesc *chunks;
    int max_b_rows;
    int parts; int32_t *part_cnt;        // [n_items * parts] popcount of the part's words
};

// phase A: bit offset of every RLE group; consistency with ref_len / seq_len (status 16 and invalid chunks otherwise)
__global__ void __launch_bounds__(PLAN_THREADS) plan_groups_kernel(const PlanArgs a)
{
    __shared__ int s_warp[PLAN_THREADS / 32];
    __shared__ int s_bad;
    const int it = blockIdx.x;
    const ItemDesc I = a.items[it];
    const uint32_t *g_rle = a.rle + I.cig_off;
    int32_t *g_off = a.grp_off + I.cig_off + it;         // cig_n + 1 entries per item
    const int P = I.total_ops;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    int carry = 0, nD = 0, nI = 0;
    for (int base = 0; base < I.cig_n; base += PLAN_THREADS) {
        const int g = base + threadIdx.x;
        int nb = 0;
        if (g < I.cig_n) {
            const uint32_t w = g_rle[g]; const int len = (int)(w >> 4), op = (int)(w & 15);
            if (op == 0 || op == 7 || op == 8) { nb = 2 * len; nD += len; nI += len; }
            else if (op == 1) { nb = len; nI += len; }
            else if (op == 2) { nb = len; nD += len; }
            else s_bad = 1;
        }
        int tot;
        const int ex = plan_block_exscan(nb, s_warp, tot);
        if (g < I.cig_n) g_off[g] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) g_off[I.cig_n] = carry;
    int tD, tI;
    plan_block_exscan(nD, s_warp, tD);
    plan_block_exscan(nI, s_warp, tI);
    __syncthreads();
    const bool bad = s_bad || tD != I.ref_len || tI != I.seq_len || carry != P;
    if (bad) {
        if (threadIdx.x == 0) a.items[it].status = 16;    // NPORE_ST_BAD_CIGAR
        for (int k = threadIdx.x; k < I.n_chunks; k += PLAN_THREADS) {
            ChunkDesc c = {}; c.item = it; c.valid = 0; c.B = 0;
            a.chunks[I.chunk_first + k] = c;
        }
    }
}

// phase B: the bit words of one slice of the item + their popcount
__global__ void __launch_bounds__(PLAN_THREADS) plan_bits_kernel(const PlanArgs a)
{
    __shared__ int s_warp[PLAN_THREADS / 32];
    const int it = blockIdx.x, part = blockIdx.y;
    const ItemDesc I = a.items[it];
    if (I.status) { if (threadIdx.x == 0) a.part_cnt[it * a.parts + part] = 0; return; }
    const uint32_t *g_rle = a.rle + I.cig_off;
    const int32_t *g_off = a.grp_off + I.cig_off + it;
    uint32_t *g_bits = a.bits + I.bit_word_off;
    const int P = I.total_ops;
    const int nwords = (P >> 5) + 1;
    int wlo, whi;
    np_slice(nwords, a.parts, part, wlo, whi);
    int cnt = 0;
    for (int w = wlo + threadIdx.x; w < whi; w += PLAN_THREADS) {
        uint32_t word = 0;
        const int lo = w << 5, hi = min(lo + 32, P);
        if (lo < hi) {
            int x = 0, y = I.cig_n;                        // last group with g_off <= lo
            while (y - x > 1) { const int m = (x + y) >> 1; if (g_off[m] <= lo) x = m; else y = m; }
            int g = x, pos = lo;
            while (pos < hi) {
                const int gs = g_off[g], ge = g_off[g + 1];
                const int e = min(ge, hi);
                if (e > pos) {
                    const int op = (int)(g_rle[g] & 15);
                    const int n = e - pos, sh = pos - lo;
                    const uint32_t span = (n >= 32 ? 0xffffffffu : ((1u << n) - 1u)) << sh;
                    if (op == 1) word |= span;
                    else if (op != 2) {
                        // D,I,D,I,... starting at gs: odd offsets from gs are 'I'
                        const uint32_t alt = ((gs - lo) & 1) ? 0x55555555u : 0xaaaaaaaau;
                        word |= span & alt;
                    }
                    pos = e;
                }
                g++;
            }
        }
        g_bits[w] = word;
        cnt += __popc(word);
    }
    int tot;
    plan_block_exscan(cnt, s_warp, tot);
    if (threadIdx.x == 0) {
        a.part_cnt[it * a.parts + part] = tot;
        if (part == a.parts - 1) g_bits[nwords] = 0;
    }
}

// phase C: exclusive prefix of the popcounts (rank array)
__global__ void __launch_bounds__(PLAN_THREADS) plan_cum_kernel(const PlanArgs a)
{
    __shared__ int s_warp[PLAN_THREADS / 32];
    const int it = blockIdx.x, part = blockIdx.y;
    const ItemDesc I = a.items[it];
    if (I.status) return;
    const uint32_t *g_bits = a.bits + I.bit_word_off;
    uint32_t *g_cum = a.cum + I.bit_word_off;
    const int nwords = (I.total_ops >> 5) + 1;
    int wlo, whi;
    np_slice(nwords, a.parts, part, wlo, whi);
    int carry = 0;
    for (int q = 0; q < part; q++) carry += a.part_cnt[it * a.parts + q];
    for (int base = wlo; base < whi; base += PLAN_THREADS) {
        const int w = base + threadIdx.x;
        const int c = w < whi ? __popc(g_bits[w]) : 0;
        int tot;
        const int ex = plan_block_exscan(c, s_warp, tot);
        if (w < whi) g_cum[w] = (uint32_t)(carry + ex);
        carry += tot;
    }
    if (part == a.parts - 1 && threadIdx.x == 0) g_cum[nwords] = (uint32_t)carry;
}

// phase D: chunk descriptors (get_breaks)
__global__ void __launch_bounds__(PLAN_THREADS) plan_chunks_kernel(const PlanArgs a)
{
    const int it = blockIdx.x;
    const ItemDesc I = a.items[it];
    if (I.status) return;
    const uint32_t *g_bits = a.bits + I.bit_word_off, *g_cum = a.cum + I.bit_word_off;
    const int P = I.total_ops;
    const int step = a.max_b_rows - 1;
    int klo, khi;
    np_slice(I.n_chunks, a.parts, blockIdx.y, klo, khi);
    for (int k = klo + threadIdx.x; k < khi; k += PLAN_THREADS) {
        int brk = k * step, nxt = (k + 1 < I.n_chunks) ? (k + 1) * step : P;
        if (k > 0 && ((g_bits[brk >> 5] >> (brk & 31)) & 1u) && !((g_bits[(brk - 1) >> 5] >> ((brk - 1) & 31)) & 1u)) brk--;
        if (k + 1 < I.n_chunks && ((g_bits[nxt >> 5] >> (nxt & 31)) & 1u) && !((g_bits[(nxt - 1) >> 5] >> ((nxt - 1) & 31)) & 1u)) nxt--;
        ChunkDesc c;
        c.item = it; c.brk = brk; c.B = nxt - brk + 1;
        c.r0 = (int)plan_rank(g_bits, g_cum, brk); c.c0 = brk - c.r0;
        const int r1 = (int)plan_rank(g_bits, g_cum, nxt), c1 = nxt - r1;
        c.imax = r1 - c.r0; c.jmax = c1 - c.c0;
        c.rlen = max(0, min(c1 + 1, I.ref_len) - c.c0);
        c.slen = max(0, min(r1 + 1, I.seq_len) - c.r0);
        c.valid = 1; c.pad[0] = c.pad[1] = 0;
        a.chunks[I.chunk_first + k] = c;
    }
}
