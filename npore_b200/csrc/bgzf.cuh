// bgzf.cuh -- BGZF compression on the device (SAM spec section 4.1): the input stream is cut into members of at most
// BGZF_BLOCK bytes, and every member is one gzip member with the BC extra field, one final deflate block (RFC 1951) and the
// CRC32 / ISIZE trailer.  One CTA compresses one member:
//   1. stage the member in shared memory; every thread hashes its positions (3 bytes -> BGZF_HASH_BITS)
//   2. warp 0 links every position to the previous one of the same hash (prev[], exact, in position order) while the
//      other warps compute the CRC32 of their segments
//   3. every thread parses its own segment greedily (zlib level 1 is a greedy parse too): matches reach back through the
//      chains into earlier segments (distance <= 32768) but end at the segment's end; tokens go to global scratch and
//      their symbols into block-wide histograms (integer atomics: the counts do not depend on the order)
//   4. warp 0 builds the length-limited Huffman codes (litlen / distance <= 15 bits, code-length code <= 7 bits)
//   5. an exclusive scan of the per-thread bit counts places every thread's tokens; the bits are OR-ed into a zeroed
//      shared buffer (disjoint ranges: the result does not depend on the order either)
//   6. if the coded block is not smaller than a stored one, the member is stored (BTYPE 00)
// The member is written to its own 64 KiB slot; bgzf_gather_kernel packs the slots into one contiguous stream.
#pragma once
#include <cstdint>

#define BGZF_BLOCK 65280          // input bytes per member (htslib's BGZF_BLOCK_SIZE)
#define BGZF_SLOT 65536           // the largest member
#define BGZF_THREADS 256
#define BGZF_HASH_BITS 13
#define BGZF_NONE 0xFFFFu         // no earlier position (positions are < BGZF_BLOCK < 0xFFFF)
#define BGZF_CHAIN 16             // candidates tried per position
#define BGZF_NICE 128             // a match this long ends the search
#define BGZF_MEMBER_OVERHEAD 26   // 18 header bytes + CRC32 + ISIZE

namespace bgzf {

constexpr int kInBytes = 65536;                               // staged input, zero padded for the 3-byte hash
constexpr int kPrevBytes = BGZF_BLOCK * 2;                    // prev[]; afterwards the output bit buffer (>= 65536 + 8)
constexpr int kHeadBytes = (1 << BGZF_HASH_BITS) * 2;
constexpr int kDynSmem = kInBytes + kPrevBytes + kHeadBytes;

__constant__ uint16_t kLenBase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t kLenExtra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint8_t kHeader[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};   // BSIZE follows
__constant__ uint8_t kClOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

__device__ __forceinline__ int len_code(int len)              // 3..258 -> 0..28 (symbol 257 + code)
{
    if (len == 258) return 28;
    const int l = len - 3;
    if (l < 8) return l;
    const int b = 31 - __clz(l), e = b - 2;
    return 4 * (b - 1) + ((l >> e) & 3);
}

__device__ __forceinline__ int dist_code(int dist)            // 1..32768 -> 0..29
{
    const int d = dist - 1;
    if (d < 4) return d;
    const int b = 31 - __clz(d);
    return 2 * b + ((d >> (b - 1)) & 1);
}

__device__ __forceinline__ int dist_extra_bits(int code) { return code < 4 ? 0 : (code >> 1) - 1; }
__device__ __forceinline__ int dist_base(int code) { return code < 4 ? code + 1 : ((2 | (code & 1)) << dist_extra_bits(code)) + 1; }

// zlib's GF(2) product modulo the CRC-32 polynomial (reflected): crc32_combine without its tables
__device__ __forceinline__ uint32_t multmodp(uint32_t a, uint32_t b)
{
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}

__device__ __forceinline__ uint32_t x8nmodp(uint32_t n, const uint32_t *x2n)   // x^(8n) mod p; x2n[k] = x^(2^k)
{
    uint32_t p = 1u << 31;
    for (int k = 3; n; n >>= 1, k++)
        if (n & 1) p = multmodp(x2n[k & 31], p);
    return p;
}

__device__ __forceinline__ uint32_t bitrev(uint32_t code, int len) { return __brev(code) >> (32 - len); }

__device__ __forceinline__ void put_bits(uint32_t *w, uint32_t pos, uint32_t v, int nb)
{
    if (!nb) return;
    const uint32_t sh = pos & 31;
    atomicOr(&w[pos >> 5], v << sh);
    if (sh + nb > 32) atomicOr(&w[(pos >> 5) + 1], v >> (32 - sh));
}

struct Small {                                      // the static shared state of one member
    uint32_t crc_tab[256], x2n[32];
    uint32_t seg_crc[BGZF_THREADS], seg_len[BGZF_THREADS], seg_bits[BGZF_THREADS];
    uint32_t hist_ll[288], hist_d[32], hist_cl[19];
    uint8_t len_ll[288], len_d[32], len_cl[19];
    uint16_t code_ll[288], code_d[32], code_cl[19];
    uint32_t key[288]; uint16_t sym[288];           // tree build: used symbols sorted by (frequency, symbol)
    uint32_t num[33], next[16];
    uint16_t cl_tok[320];                           // run-length coded code lengths: symbol | extra << 5
    int n_cl_tok, hlit, hdist, hclen;
    uint32_t header_bits;
};

// Length-limited Huffman code lengths for freq[0..n) (called by one warp).  Fewer than two used symbols get symbols 0 / 1
// added, so that every code is complete.  Lengths: the in-place minimum-redundancy algorithm of Moffat and Katajainen on
// the sorted frequencies, then the Kraft repair that moves codes deeper than max_bits up (as miniz does).
__device__ void build_lengths(Small &s, uint32_t *freq, int n, int max_bits, uint8_t *len, uint16_t *code, int lane)
{
    for (int i = lane; i < n; i += 32) len[i] = 0;
    if (lane == 0) {
        int used = 0;
        for (int i = 0; i < n; i++) used += freq[i] != 0;
        for (int i = 0; i < 2 && used < 2; i++)
            if (!freq[i]) { freq[i] = 1; used++; }
    }
    __syncwarp();
    for (int i = lane; i < n; i += 32) {
        const uint32_t f = freq[i];
        if (!f) continue;
        int r = 0;
        for (int j = 0; j < n; j++) r += freq[j] && (freq[j] < f || (freq[j] == f && j < i));
        s.key[r] = f; s.sym[r] = (uint16_t)i;
    }
    __syncwarp();
    if (lane == 0) {
        int m = 0;
        for (int i = 0; i < n; i++) m += freq[i] != 0;
        uint32_t *A = s.key;
        A[0] += A[1];
        int root = 0, leaf = 2;
        for (int nx = 1; nx < m - 1; nx++) {
            if (leaf >= m || A[root] < A[leaf]) { A[nx] = A[root]; A[root++] = (uint32_t)nx; }
            else A[nx] = A[leaf++];
            if (leaf >= m || (root < nx && A[root] < A[leaf])) { A[nx] += A[root]; A[root++] = (uint32_t)nx; }
            else A[nx] += A[leaf++];
        }
        A[m - 2] = 0;
        for (int nx = m - 3; nx >= 0; nx--) A[nx] = A[A[nx]] + 1;
        int avbl = 1, used = 0, dpth = 0;
        root = m - 2;
        int nx = m - 1;
        while (avbl > 0) {
            while (root >= 0 && (int)A[root] == dpth) { used++; root--; }
            while (avbl > used) { A[nx--] = (uint32_t)dpth; avbl--; }
            avbl = 2 * used; dpth++; used = 0;
        }
        for (int i = 0; i <= 32; i++) s.num[i] = 0;
        for (int i = 0; i < m; i++) s.num[min(A[i], 32u)]++;
        for (int i = max_bits + 1; i <= 32; i++) { s.num[max_bits] += s.num[i]; s.num[i] = 0; }
        uint32_t total = 0;
        for (int i = max_bits; i > 0; i--) total += s.num[i] << (max_bits - i);
        while (total != (1u << max_bits)) {
            s.num[max_bits]--;
            for (int i = max_bits - 1; i > 0; i--)
                if (s.num[i]) { s.num[i]--; s.num[i + 1] += 2; break; }
            total--;
        }
        for (int i = 1, j = m; i <= max_bits; i++)
            for (uint32_t k = s.num[i]; k > 0; k--) len[s.sym[--j]] = (uint8_t)i;
        // canonical codes (RFC 1951 3.2.2), bit-reversed: deflate sends Huffman codes from their top bit
        s.next[0] = 0;
        for (int b = 1; b <= max_bits; b++) s.next[b] = (s.next[b - 1] + s.num[b - 1]) << 1;
        for (int i = 0; i < n; i++)
            code[i] = len[i] ? (uint16_t)bitrev(s.next[len[i]]++, len[i]) : 0;
    }
    __syncwarp();
}

// One member per CTA.  tok: BGZF_BLOCK uint32 of scratch per member; slots: BGZF_SLOT bytes per member; sizes: member bytes.
__global__ void __launch_bounds__(BGZF_THREADS, 1)
bgzf_deflate_kernel(const uint8_t *__restrict__ in, int64_t n_total, uint32_t *__restrict__ tok, uint8_t *__restrict__ slots,
                    int32_t *__restrict__ sizes)
{
    extern __shared__ __align__(16) uint8_t dyn[];
    __shared__ Small s;
    uint8_t *buf = dyn;
    uint16_t *prev = reinterpret_cast<uint16_t *>(dyn + kInBytes);
    uint16_t *head = reinterpret_cast<uint16_t *>(dyn + kInBytes + kPrevBytes);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t m = blockIdx.x;
    const int64_t at = m * BGZF_BLOCK;
    const int n = (int)min((int64_t)BGZF_BLOCK, n_total - at);
    uint32_t *mtok = tok + m * BGZF_BLOCK;

    // ---- 1. stage, tables
    for (int i = tid; i < kInBytes; i += BGZF_THREADS) buf[i] = i < n ? in[at + i] : 0;
    for (int i = tid; i < (1 << BGZF_HASH_BITS); i += BGZF_THREADS) head[i] = BGZF_NONE;
    {
        uint32_t c = (uint32_t)tid;
        for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
        s.crc_tab[tid] = c;
    }
    for (int i = tid; i < 288; i += BGZF_THREADS) s.hist_ll[i] = 0;
    if (tid < 32) s.hist_d[tid] = 0;
    if (tid < 19) s.hist_cl[tid] = 0;
    if (tid == 0) {
        uint32_t p = 1u << 30;                       // x^1
        s.x2n[0] = p;
        for (int k = 1; k < 32; k++) s.x2n[k] = p = multmodp(p, p);
    }
    __syncthreads();
    for (int i = tid; i < n; i += BGZF_THREADS)
        prev[i] = (uint16_t)((((uint32_t)buf[i] << 16 | (uint32_t)buf[i + 1] << 8 | buf[i + 2]) * 2654435761u) >> (32 - BGZF_HASH_BITS));
    __syncthreads();

    const int seg = (n + BGZF_THREADS - 1) / BGZF_THREADS;
    const int lo = min(n, tid * seg), hi = min(n, lo + seg);
    // ---- 2. hash chains (warp 0, 32 positions a step, in order) beside the segment CRCs (all other threads, then warp 0)
    if (warp == 0) {
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            const bool ok = i + 2 < n;
            const uint32_t h = ok ? prev[i] : 0x10000u + lane;
            const uint32_t same = __match_any_sync(0xffffffffu, h);
            const uint32_t lower = same & ((1u << lane) - 1);
            uint32_t cand = BGZF_NONE;
            if (ok) cand = lower ? (uint32_t)(base + 31 - __clz(lower)) : head[h];
            __syncwarp();
            if (i < n) prev[i] = (uint16_t)cand;
            if (ok && lane == 31 - __clz(same)) head[h] = (uint16_t)i;
            __syncwarp();
        }
    }
    {
        uint32_t c = 0xFFFFFFFFu;
        for (int i = lo; i < hi; i++) c = s.crc_tab[(c ^ buf[i]) & 0xFF] ^ (c >> 8);
        s.seg_crc[tid] = ~c;
        s.seg_len[tid] = (uint32_t)(hi - lo);
    }
    __syncthreads();
    // combine the segment CRCs pairwise: crc(A B) = crc(A) * x^(8|B|) + crc(B)
    for (int stride = 1; stride < BGZF_THREADS; stride <<= 1) {
        if ((tid & (2 * stride - 1)) == 0) {
            const uint32_t rl = s.seg_len[tid + stride];
            if (rl) s.seg_crc[tid] = multmodp(x8nmodp(rl, s.x2n), s.seg_crc[tid]) ^ s.seg_crc[tid + stride];
            s.seg_len[tid] += rl;
        }
        __syncthreads();
    }

    // ---- 3. greedy parse of this thread's segment
    int nt = 0;
    for (int p = lo; p < hi;) {
        const int maxl = min(258, hi - p);
        int best = 0, bdist = 0;
        if (maxl >= 3) {
            uint32_t c = prev[p];
            for (int steps = 0; steps < BGZF_CHAIN && c != BGZF_NONE && p - (int)c <= 32768; steps++) {
                if (buf[c + best] == buf[p + best] || best == 0) {
                    int l = 0;
                    while (l < maxl && buf[c + l] == buf[p + l]) l++;
                    if (l > best) { best = l; bdist = p - (int)c; if (l >= BGZF_NICE || l == maxl) break; }
                }
                c = prev[c];
            }
        }
        if (best == 3 && bdist > 4096) best = 0;          // a far 3-byte match costs more than its literals (zlib's TOO_FAR)
        if (best >= 3) {
            mtok[lo + nt++] = 0x80000000u | (uint32_t)best << 16 | (uint32_t)bdist;
            atomicAdd(&s.hist_ll[257 + len_code(best)], 1u);
            atomicAdd(&s.hist_d[dist_code(bdist)], 1u);
            p += best;
        } else {
            mtok[lo + nt++] = buf[p];
            atomicAdd(&s.hist_ll[buf[p]], 1u);
            p++;
        }
    }
    if (tid == 0) s.hist_ll[256] = 1;                      // end of block
    __syncthreads();

    // ---- 4. codes
    if (warp == 0) {
        build_lengths(s, s.hist_ll, 286, 15, s.len_ll, s.code_ll, lane);
        build_lengths(s, s.hist_d, 30, 15, s.len_d, s.code_d, lane);
        if (lane == 0) {
            int hlit = 286, hdist = 30;
            while (hlit > 257 && !s.len_ll[hlit - 1]) hlit--;
            while (hdist > 1 && !s.len_d[hdist - 1]) hdist--;
            s.hlit = hlit; s.hdist = hdist;
            const int total = hlit + hdist;
            int k = 0;
            auto L = [&](int i) { return i < hlit ? s.len_ll[i] : s.len_d[i - hlit]; };
            for (int i = 0; i < total;) {
                const int v = L(i);
                int run = 1;
                while (i + run < total && L(i + run) == v) run++;
                i += run;
                if (v == 0) {
                    while (run >= 11) { const int r = min(run, 138); s.cl_tok[k++] = (uint16_t)(18 | (r - 11) << 5); run -= r; }
                    if (run >= 3) { s.cl_tok[k++] = (uint16_t)(17 | (run - 3) << 5); run = 0; }
                    while (run-- > 0) s.cl_tok[k++] = 0;
                } else {
                    s.cl_tok[k++] = (uint16_t)v;
                    run--;
                    while (run >= 3) { const int r = min(run, 6); s.cl_tok[k++] = (uint16_t)(16 | (r - 3) << 5); run -= r; }
                    while (run-- > 0) s.cl_tok[k++] = (uint16_t)v;
                }
            }
            s.n_cl_tok = k;
            for (int j = 0; j < k; j++) s.hist_cl[s.cl_tok[j] & 31]++;
        }
        __syncwarp();
        build_lengths(s, s.hist_cl, 19, 7, s.len_cl, s.code_cl, lane);
        if (lane == 0) {
            int hclen = 19;
            while (hclen > 4 && !s.len_cl[kClOrder[hclen - 1]]) hclen--;
            s.hclen = hclen;
            uint32_t bits = 3 + 5 + 5 + 4 + 3 * hclen;
            for (int j = 0; j < s.n_cl_tok; j++) {
                const int sy = s.cl_tok[j] & 31;
                bits += s.len_cl[sy] + (sy == 16 ? 2 : sy == 17 ? 3 : sy == 18 ? 7 : 0);
            }
            s.header_bits = bits;
        }
    }
    __syncthreads();

    // ---- 5. bit counts, placement
    uint32_t my_bits = 0;
    for (int k = 0; k < nt; k++) {
        const uint32_t t = mtok[lo + k];
        if (t & 0x80000000u) {
            const int len = (t >> 16) & 0x1FF, dist = t & 0xFFFF, lc = len_code(len), dc = dist_code(dist);
            my_bits += s.len_ll[257 + lc] + kLenExtra[lc] + s.len_d[dc] + dist_extra_bits(dc);
        } else {
            my_bits += s.len_ll[t];
        }
    }
    s.seg_bits[tid] = my_bits;
    __syncthreads();
    for (int stride = 1; stride < BGZF_THREADS; stride <<= 1) {   // inclusive scan (Hillis-Steele)
        const uint32_t v = tid >= stride ? s.seg_bits[tid - stride] : 0;
        __syncthreads();
        s.seg_bits[tid] += v;
        __syncthreads();
    }
    const uint32_t data_end = s.header_bits + s.seg_bits[BGZF_THREADS - 1];
    const uint32_t coded_bytes = (data_end + s.len_ll[256] + 7) / 8;
    const bool stored = coded_bytes >= (uint32_t)n + 5;
    const uint32_t dbytes = stored ? (uint32_t)n + 5 : coded_bytes;
    uint8_t *out = slots + m * BGZF_SLOT;
    uint32_t *wbuf = reinterpret_cast<uint32_t *>(prev);     // prev[] is not read any more
    if (!stored) {
        const int words = (int)(dbytes + 3) / 4 + 1;
        for (int i = tid; i < words; i += BGZF_THREADS) wbuf[i] = 0;
        __syncthreads();
        if (tid == 0) {
            uint32_t pos = 0;
            put_bits(wbuf, pos, 5, 3); pos += 3;                 // BFINAL = 1, BTYPE = 10
            put_bits(wbuf, pos, (uint32_t)(s.hlit - 257), 5); pos += 5;
            put_bits(wbuf, pos, (uint32_t)(s.hdist - 1), 5); pos += 5;
            put_bits(wbuf, pos, (uint32_t)(s.hclen - 4), 4); pos += 4;
            for (int j = 0; j < s.hclen; j++) { put_bits(wbuf, pos, s.len_cl[kClOrder[j]], 3); pos += 3; }
            for (int j = 0; j < s.n_cl_tok; j++) {
                const int sy = s.cl_tok[j] & 31, ex = s.cl_tok[j] >> 5;
                put_bits(wbuf, pos, s.code_cl[sy], s.len_cl[sy]); pos += s.len_cl[sy];
                const int eb = sy == 16 ? 2 : sy == 17 ? 3 : sy == 18 ? 7 : 0;
                put_bits(wbuf, pos, (uint32_t)ex, eb); pos += eb;
            }
            put_bits(wbuf, data_end, s.code_ll[256], s.len_ll[256]);
        }
        uint32_t pos = s.header_bits + s.seg_bits[tid] - my_bits;
        for (int k = 0; k < nt; k++) {
            const uint32_t t = mtok[lo + k];
            if (t & 0x80000000u) {
                const int len = (t >> 16) & 0x1FF, dist = t & 0xFFFF, lc = len_code(len), dc = dist_code(dist);
                put_bits(wbuf, pos, s.code_ll[257 + lc], s.len_ll[257 + lc]); pos += s.len_ll[257 + lc];
                put_bits(wbuf, pos, (uint32_t)(len - kLenBase[lc]), kLenExtra[lc]); pos += kLenExtra[lc];
                put_bits(wbuf, pos, s.code_d[dc], s.len_d[dc]); pos += s.len_d[dc];
                put_bits(wbuf, pos, (uint32_t)(dist - dist_base(dc)), dist_extra_bits(dc)); pos += dist_extra_bits(dc);
            } else {
                put_bits(wbuf, pos, s.code_ll[t], s.len_ll[t]); pos += s.len_ll[t];
            }
        }
        __syncthreads();
    }
    // ---- 6. the member: header, deflate data, CRC32, ISIZE
    const uint32_t size = 18 + dbytes + 8;
    if (tid < 18) out[tid] = tid < 16 ? kHeader[tid] : (uint8_t)((size - 1) >> (8 * (tid - 16)));
    if (tid < 8) {
        const uint32_t v = tid < 4 ? s.seg_crc[0] : (uint32_t)n;
        out[18 + dbytes + tid] = (uint8_t)(v >> (8 * (tid & 3)));
    }
    if (stored) {
        if (tid < 5)                                     // BFINAL = 1, BTYPE = 00; LEN, NLEN
            out[18 + tid] = tid == 0 ? 1 : (uint8_t)((tid < 3 ? n : ~n) >> (8 * ((tid - 1) & 1)));
        for (int i = tid; i < n; i += BGZF_THREADS) out[23 + i] = buf[i];
    } else {
        const uint8_t *bytes = reinterpret_cast<const uint8_t *>(wbuf);
        for (uint32_t i = tid; i < dbytes; i += BGZF_THREADS) out[18 + i] = bytes[i];
    }
    if (tid == 0) sizes[m] = (int32_t)size;
}

// Packs the member slots into one stream: CTA m adds the sizes of members 0..m-1 and copies its member there; the last
// CTA writes the total.
__global__ void __launch_bounds__(BGZF_THREADS)
bgzf_gather_kernel(const uint8_t *__restrict__ slots, const int32_t *__restrict__ sizes, int n_members, uint8_t *__restrict__ out,
                   int64_t *__restrict__ total)
{
    __shared__ long long part[BGZF_THREADS / 32];
    const int m = blockIdx.x, tid = threadIdx.x;
    long long acc = 0;
    for (int i = tid; i < m; i += BGZF_THREADS) acc += sizes[i];
    for (int o = 16; o; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if ((tid & 31) == 0) part[tid >> 5] = acc;
    __syncthreads();
    long long off = 0;
    for (int w = 0; w < BGZF_THREADS / 32; w++) off += part[w];
    const int sz = sizes[m];
    const uint8_t *src = slots + (int64_t)m * BGZF_SLOT;
    for (int i = tid; i < sz; i += BGZF_THREADS) out[off + i] = src[i];
    if (m == n_members - 1 && tid == 0) *total = off + sz;
}

}  // namespace bgzf
