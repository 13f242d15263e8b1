// bai.cuh -- the BAM index (SAM spec section 5.2) contribution of one batch of BAM records, computed on the device from the
// records and BGZF member sizes that npore_bgzf_compress (bgzf.cuh) leaves there.  Four kernels:
//   bai_member_kernel  file offset of every member: base + exclusive scan of the member sizes (one CTA)
//   bai_record_kernel  one thread per record: ref_id, pos, flag and the CIGAR's reference span from the record bytes; end
//                      (htslib's bam_endpos: pos + span, pos + 1 when unmapped or the span is 0), bin = reg2bin(pos, end),
//                      and the virtual offsets of the record's first byte and of the byte after it
//   bai_chunk_kernel   one CTA over the records in file order: a chunk per run of records with the same (ref_id, bin), one
//                      segment per reference; the chunks put in (ref_id, bin, vbeg) order; chunks of one bin merged when the
//                      previous one ends in the BGZF block where the next starts (htslib's compress_binning); per reference the
//                      first / last voffset, the mapped / unmapped counts and the range of 16 kb windows its mapped records cover
//   bai_linear_kernel  one thread per mapped record: atomic min of its vbeg over every window it overlaps
// Sorting needs no general sort: within one reference the records are in position order, so the bins of one level
// (0, 1-8, 9-72, 73-584, 585-4680, 4681-37448) are non-decreasing in file order, and (bin, vbeg) order is the stable
// partition of the chunks by level.
//
// Voffsets.  A member holds BGZF_BLOCK input bytes, so input byte u lies in member u / BGZF_BLOCK at offset u % BGZF_BLOCK.
// The end of the batch is a member boundary (the next batch starts a new member); it takes the canonical "next member, offset
// 0" form that htslib's bgzf_tell gives there: (base + all member bytes) << 16.
#pragma once
#include <cstdint>

#include "bgzf.cuh"

#define BAI_THREADS 512
#define BAI_ERR_UNSORTED 1ull     // records out of (ref_id, pos) order
#define BAI_ERR_RECORD 2ull       // record offsets or a record's fields inconsistent with the bytes
#define BAI_ERR_UNPLACED 4ull     // ref_id < 0 or pos < 0: not indexable here

namespace bai {

struct Rec { int32_t ref, bin, pos, wlast, seg, pad; uint64_t vbeg, vend; };       // wlast < 0: unmapped
struct Chunk { int32_t ref, bin, seg, rank; uint64_t beg, end; };                   // rank: level-wise exclusive count
struct Seg {
    int32_t ref, c0, wfirst, wlast;
    uint64_t beg, end;
    unsigned long long n_mapped, n_unmapped;
    int32_t lev0[6], lev1[6];                     // per bin level: exclusive count at the segment's first chunk / inclusive at its last
    int64_t woff;                                 // first window of the segment in the window array
};

__device__ __forceinline__ uint32_t ld32(const uint8_t *p) { return p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

__device__ __forceinline__ int reg2bin(int64_t beg, int64_t end)       // hts_reg2bin for the half-open [beg, end), 14 / 5 levels
{
    --end;
    if (beg >> 14 == end >> 14) return (int)(4681 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(585 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(73 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(9 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(1 + (beg >> 26));
    return 0;
}

__device__ __forceinline__ int bin_level(int bin) { return bin >= 4681 ? 5 : bin >= 585 ? 4 : bin >= 73 ? 3 : bin >= 9 ? 2 : bin >= 1 ? 1 : 0; }

// inclusive scan over the CTA; *total receives the CTA's sum.  Every thread of the CTA calls it.
__device__ __forceinline__ uint64_t block_scan(uint64_t v, uint64_t *warp_sum, uint64_t *total)
{
    constexpr int NW = BAI_THREADS / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    if (lane == 31) warp_sum[warp] = v;
    __syncthreads();
    if (warp == 0) {
        uint64_t w = lane < NW ? warp_sum[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        if (lane < NW) warp_sum[lane] = w;
    }
    __syncthreads();
    if (warp > 0) v += warp_sum[warp - 1];
    *total = warp_sum[NW - 1];
    __syncthreads();                               // warp_sum is free again
    return v;
}

__device__ __forceinline__ uint64_t voff(const uint64_t *moff, int64_t u, int64_t n_in, int64_t members)
{
    if (u >= n_in) return moff[members] << 16;
    return moff[u / BGZF_BLOCK] << 16 | (uint64_t)(u % BGZF_BLOCK);
}

// moff[k] = base + sizes[0] + ... + sizes[k-1], k = 0..members
__global__ void __launch_bounds__(BAI_THREADS)
bai_member_kernel(const int32_t *__restrict__ sizes, int64_t members, uint64_t base, uint64_t *__restrict__ moff)
{
    __shared__ uint64_t warp_sum[BAI_THREADS / 32];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = base;
    __syncthreads();
    for (int64_t t0 = 0; t0 < members; t0 += BAI_THREADS) {
        const int64_t k = t0 + threadIdx.x;
        const uint64_t v = k < members ? (uint64_t)sizes[k] : 0;
        uint64_t total;
        const uint64_t incl = block_scan(v, warp_sum, &total);
        if (k < members) moff[k] = carry + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) moff[members] = carry;
}

__global__ void __launch_bounds__(256)
bai_record_kernel(const uint8_t *__restrict__ in, int64_t n_in, int64_t members, const int64_t *__restrict__ rec_off, int64_t n,
                  const uint64_t *__restrict__ moff, Rec *__restrict__ recs, unsigned long long *__restrict__ err)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t a = rec_off[i], b = rec_off[i + 1];
    Rec r{};
    r.ref = -1; r.wlast = -1;
    bool bad = a < 0 || b > n_in || b - a < 36;
    if (!bad) {
        const uint8_t *p = in + a;
        const uint32_t l_name = p[12], n_cig = p[16] | (uint32_t)p[17] << 8, flag = p[18] | (uint32_t)p[19] << 8;
        bad = (int64_t)ld32(p) + 4 != b - a || 36 + (int64_t)l_name + 4 * (int64_t)n_cig > b - a;
        if (!bad) {
            r.ref = (int32_t)ld32(p + 4);
            r.pos = (int32_t)ld32(p + 8);
            int64_t span = 0;
            const uint8_t *cg = p + 36 + l_name;
            for (uint32_t c = 0; c < n_cig; c++) {
                const uint32_t w = ld32(cg + 4 * c), op = w & 15u;
                if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += w >> 4;
            }
            const bool mapped = !(flag & 4u);
            const int64_t end = (int64_t)r.pos + (mapped && span ? span : 1);
            if (r.ref < 0 || r.pos < 0) atomicOr(err, BAI_ERR_UNPLACED);
            else {
                r.bin = reg2bin(r.pos, end);
                r.wlast = mapped ? (int32_t)((end - 1) >> 14) : -1;
            }
        }
    }
    if (bad) atomicOr(err, BAI_ERR_RECORD);
    else {
        r.vbeg = voff(moff, a, n_in, members);
        r.vend = voff(moff, b, n_in, members);
    }
    recs[i] = r;
}

// One CTA.  counts: [0] merged chunks, [1] segments, [2] windows, [3] error bits (zeroed by the caller).
// out_chunk: rows (ref_id, bin, vbeg, vend); out_ref: rows (ref_id, vbeg, vend, n_mapped, n_unmapped, first window, windows).
__global__ void __launch_bounds__(BAI_THREADS, 1)
bai_chunk_kernel(Rec *__restrict__ recs, int64_t n, Chunk *__restrict__ ch, Chunk *__restrict__ sorted, Seg *__restrict__ seg,
                 uint64_t *__restrict__ out_chunk, uint64_t *__restrict__ out_ref, unsigned long long *__restrict__ counts)
{
    __shared__ uint64_t warp_sum[BAI_THREADS / 32];
    __shared__ uint64_t carry[6];
    const int tid = threadIdx.x;
    if (tid < 6) carry[tid] = 0;
    __syncthreads();
    // ---- A. runs of (ref_id, bin) -> chunks; runs of ref_id -> segments
    for (int64_t t0 = 0; t0 < n; t0 += BAI_THREADS) {
        const int64_t i = t0 + tid;
        const bool ok = i < n;
        Rec r{};
        bool run0 = false, seg0 = false, run1 = false, seg1 = false;
        if (ok) {
            r = recs[i];
            if (i == 0) run0 = seg0 = true;
            else {
                const Rec &q = recs[i - 1];
                seg0 = q.ref != r.ref;
                run0 = seg0 || q.bin != r.bin;
                if (r.ref < q.ref || (r.ref == q.ref && r.pos < q.pos)) atomicOr(&counts[3], BAI_ERR_UNSORTED);
            }
            if (i == n - 1) run1 = seg1 = true;
            else {
                const Rec &q = recs[i + 1];
                seg1 = q.ref != r.ref;
                run1 = seg1 || q.bin != r.bin;
            }
        }
        uint64_t total;
        const uint64_t incl = block_scan((uint64_t)run0 | (uint64_t)seg0 << 32, warp_sum, &total);
        const int64_t ci = (int64_t)carry[0] + (int64_t)(incl & 0xffffffffu) - 1, si = (int64_t)carry[1] + (int64_t)(incl >> 32) - 1;
        if (ok) {
            recs[i].seg = (int32_t)si;
            if (run0) { ch[ci].ref = r.ref; ch[ci].bin = r.bin; ch[ci].seg = (int32_t)si; ch[ci].beg = r.vbeg; }
            if (run1) ch[ci].end = r.vend;
            if (seg0) {
                Seg &s = seg[si];
                s.ref = r.ref; s.c0 = (int32_t)ci; s.wfirst = 0x7fffffff; s.wlast = -1; s.beg = r.vbeg; s.n_mapped = s.n_unmapped = 0;
            }
        }
        __syncthreads();                          // the segment heads above are written before the atomics below
        if (ok) {
            Seg &s = seg[si];
            if (r.wlast >= 0) {
                atomicAdd(&s.n_mapped, 1ull);
                atomicMin(&s.wfirst, r.pos >> 14);
                atomicMax(&s.wlast, r.wlast);
            } else atomicAdd(&s.n_unmapped, 1ull);
            if (seg1) s.end = r.vend;
        }
        if (tid == 0) { carry[0] += total & 0xffffffffu; carry[1] += total >> 32; }
        __syncthreads();
    }
    const int64_t n_ch = (int64_t)carry[0], n_seg = (int64_t)carry[1];
    __syncthreads();
    if (tid < 6) carry[tid] = 0;
    __syncthreads();
    // ---- B1. level-wise ranks: six 10-bit counters in one scan (a tile adds at most BAI_THREADS = 512 to each)
    for (int64_t t0 = 0; t0 < n_ch; t0 += BAI_THREADS) {
        const int64_t c = t0 + tid;
        const bool ok = c < n_ch;
        const int lv = ok ? bin_level(ch[c].bin) : 0;
        uint64_t total;
        const uint64_t incl = block_scan(ok ? 1ull << (10 * lv) : 0, warp_sum, &total);
        if (ok) {
            const Chunk k = ch[c];
            ch[c].rank = (int32_t)(carry[lv] + ((incl >> (10 * lv)) & 1023) - 1);
            Seg &s = seg[k.seg];
            if (s.c0 == c) {
#pragma unroll
                for (int l = 0; l < 6; l++) s.lev0[l] = (int32_t)(carry[l] + ((incl >> (10 * l)) & 1023) - (l == lv));
            }
            if (c == n_ch - 1 || ch[c + 1].seg != k.seg) {
#pragma unroll
                for (int l = 0; l < 6; l++) s.lev1[l] = (int32_t)(carry[l] + ((incl >> (10 * l)) & 1023));
            }
        }
        __syncthreads();
        if (tid < 6) carry[tid] += (total >> (10 * tid)) & 1023;
        __syncthreads();
    }
    // ---- B2. stable partition by (segment, level): (ref_id, bin, vbeg) order
    for (int64_t c = tid; c < n_ch; c += BAI_THREADS) {
        const Chunk k = ch[c];
        const Seg &s = seg[k.seg];
        const int lv = bin_level(k.bin);
        int64_t dst = s.c0 + (k.rank - s.lev0[lv]);
#pragma unroll
        for (int l = 0; l < 6; l++)
            if (l < lv) dst += s.lev1[l] - s.lev0[l];
        sorted[dst] = k;
    }
    __syncthreads();
    // ---- C. same-block merge within a bin
    if (tid == 0) carry[0] = 0;
    __syncthreads();
    auto starts = [&](int64_t c) {
        if (c == 0) return true;
        const Chunk &p = sorted[c - 1], &k = sorted[c];
        return p.ref != k.ref || p.bin != k.bin || (p.end >> 16) < (k.beg >> 16);
    };
    for (int64_t t0 = 0; t0 < n_ch; t0 += BAI_THREADS) {
        const int64_t c = t0 + tid;
        const bool ok = c < n_ch, st = ok && starts(c);
        uint64_t total;
        const int64_t mi = (int64_t)carry[0] + (int64_t)block_scan(st ? 1 : 0, warp_sum, &total) - 1;
        if (ok) {
            const Chunk k = sorted[c];
            uint64_t *o = out_chunk + 4 * mi;
            if (st) { o[0] = (uint64_t)k.ref; o[1] = (uint64_t)k.bin; o[2] = k.beg; }
            if (c == n_ch - 1 || starts(c + 1)) o[3] = k.end;
        }
        __syncthreads();
        if (tid == 0) carry[0] += total;
        __syncthreads();
    }
    const int64_t n_merged = (int64_t)carry[0];
    __syncthreads();
    // ---- D. per reference: the window range and its place in the window array
    if (tid == 0) carry[0] = 0;
    __syncthreads();
    for (int64_t t0 = 0; t0 < n_seg; t0 += BAI_THREADS) {
        const int64_t g = t0 + tid;
        const bool ok = g < n_seg;
        Seg s{};
        if (ok) s = seg[g];
        const uint64_t nw = ok && s.wlast >= 0 ? (uint64_t)(s.wlast - s.wfirst + 1) : 0;
        uint64_t total;
        const uint64_t woff = carry[0] + block_scan(nw, warp_sum, &total) - nw;
        if (ok) {
            seg[g].woff = (int64_t)woff;
            uint64_t *o = out_ref + 7 * g;
            o[0] = (uint64_t)s.ref; o[1] = s.beg; o[2] = s.end; o[3] = s.n_mapped; o[4] = s.n_unmapped;
            o[5] = nw ? (uint64_t)s.wfirst : 0; o[6] = nw;
        }
        __syncthreads();
        if (tid == 0) carry[0] += total;
        __syncthreads();
    }
    if (tid == 0) { counts[0] = n_merged; counts[1] = n_seg; counts[2] = carry[0]; }
}

// win: the segments' windows, set to ~0 by the caller; a window no record overlaps stays ~0 (the host fills it)
__global__ void __launch_bounds__(256)
bai_linear_kernel(const Rec *__restrict__ recs, int64_t n, const Seg *__restrict__ seg, unsigned long long *__restrict__ win)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Rec r = recs[i];
    if (r.wlast < 0 || r.ref < 0) return;
    const Seg &s = seg[r.seg];
    for (int w = r.pos >> 14; w <= r.wlast; w++) atomicMin(&win[s.woff + (w - s.wfirst)], (unsigned long long)r.vbeg);
}

}  // namespace bai
