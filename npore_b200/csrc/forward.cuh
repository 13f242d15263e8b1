// forward.cuh -- the align() recurrence (reference: src/aln.pyx:465-667) as an anti-diagonal wavefront.  Round-2 form.
//
// One warp (or team of warps, below) owns one chunk at a time (persistent warps, round-robin run queue).  Lane layout is COLUMN-STATIONARY: physical
// slot s = (column index j) mod NC, NC = 32*CPL >= W = 2r+1, lane l holds slots l*CPL .. l*CPL+CPL-1 in registers (CPL = 2
// at the default r = 30).  The band of anti-diagonal d is the window of columns [jlo, jlo+NC), jlo = (#D ops so far) - r;
// b_col = j - jlo.  Consequences:
//   * a cell's row advances by one every anti-diagonal, so the reference's coordinate transforms (aln.pyx:485-492) become
//     FIXED neighbour relations: top (i-1,j) = the slot's own previous value, left (i,j-1) = the previous value of slot s-1,
//     diag (i-1,j-1) = the `left` value fetched one step earlier: 4 warp shuffles per anti-diagonal, no op-dependent paths.
//   * everything that depends on the reference column (np-info of aln.pyx:510-515, pre-decoded by annotate.cuh into SHR / LEN
//     candidate descriptors, the base, a 2-bit 6-mer) stays put in 8 registers per slot while the column is in the band; a 'D'
//     op retires the column at b_col == 0 and the slot loads the record of column j+NC in place.
//   * read-side context (aln.pyx:516-521; 4 bytes per row) moves one slot per step; an 'I' op inserts the next row at b_col 0.
//   * LEN / SHR (aln.pyx:596-667, scatter form) in GATHER form, period n descending with strict '<' (= the reference's
//     processing order; larger n wins ties).  The source cell n anti-diagonals back is read from an 8-deep shared-memory
//     ring, 16 bytes per slot: {MAT.VAL, LEN run-start value, SHR run-start value, LEN.RUN | SHR.RUN << 16}.  Carrying the
//     value at the start of the run replaces the look-back of aln.pyx:623-629, 657-663.
//   * "INF ring": every slot of every anti-diagonal writes the ring -- interior cells their values, everything else (EDGE
//     cells aln.pyx:502-507, cells outside the chunk aln.pyx:497-499, slots beyond the band) +INF -- and a state no candidate
//     set carries run-start value +INF.  A candidate whose source is not a live interior cell is then +INF and can never
//     beat the state's initial 100*d, so the steady-state code evaluates candidates WITHOUT the reference's source tests
//     (aln.pyx:609-612, 620-622, 645-647, 655-656).  One exception: when NC - W < 4, NC-W+3 equal ops among the last n <= max_n
//     make slot (j-n) mod NC alias a live cell of another column; 32-step blocks that contain such a window (six equal ops
//     in a row at r = 30) run the checked variant.  The form is validated on the CPU by oracle/pull_model.c:pm2_align.
//   * score tables re-laid per (n, L), q-major: tabS[q][row] = np_score(n, L, -(q+1)), tabL[q][row] = np_score(n, L, q+1)
//     (aln.pyx:257-274 incl. its clamps and its "ref_l + indel < 0 -> 100"), q = trunc(run/n) < NP_TABQ = 2048 = the saturated
//     run, so no clamp instruction; row np_rows is all +INF ("no candidate").  run/n is one IMAD.HI with the 17-bit reciprocal
//     held in the descriptor (exact for runs below 2^16).
//   * MAT's packed 16-bit record (TYP, RUN, two INDEL 'extended' bits; common.cuh) -- all that traceback reads
//     (aln.pyx:683-685) -- is streamed to HBM, one coalesced 64*CPL-byte row per anti-diagonal, in slot order.
//   * the anti-diagonals of a chunk are walked in blocks of <= 32 (one word of the D/I bit string).  A block is STEADY when
//     every cell 1 <= b_col <= 2r-1 of every step is an interior cell with i, j >= 2 and no aliasing window occurs; steady
//     blocks run a lean step (constant bounds, no first-row/column code, no source tests), the others the checked step.
//   * forward_kernel<CPL, T>: T = 1 as above; T = 2 / 4 splits the band's NC = 32*CPL*T slots across the warps of a TEAM (team
//     ring, 16-byte mailbox for the neighbour across the warp border, one named barrier per anti-diagonal) -- for launches that
//     cannot fill the warp slots and for bands wider than 64 cells (api.cu: forward_team).  Teams are time-sliced like warps.
//   * flags that stay live across the warp votes of a step are kept as data words (lwm[], gN), not bools: ptxas keeps live
//     predicates by packing them bit by bit into a register, which cost 12 instructions per anti-diagonal.
// Arithmetic: fp32 add / subtract and strict compare only, tie-break order of aln.pyx:585-592; compiled with --fmad=false.
#pragma once
#include "common.cuh"
#include <type_traits>

#ifndef FWD_WARPS
#define FWD_WARPS 4
#endif
#ifndef FWD_WARPS_WIDE
#define FWD_WARPS_WIDE 6   // wide bands (CPL >= 4): a ring is 16-32 KB per warp
#endif
// warps per CTA of forward_kernel<CPL, T>: T = warps that share one chunk (a "team": the band is split across them)
static __host__ __device__ constexpr int fwd_warps(int cpl, int t = 1) { return t == 1 ? (cpl >= 4 ? FWD_WARPS_WIDE : FWD_WARPS) : (cpl >= 4 ? 6 * t : 2 * t); }

struct ForwardArgs {
    const ChunkDesc *chunks;
    const ChunkSlot *slots;       // indexed like `order`
    const int32_t *order;
    int n;
    const ItemDesc *items;
    const uint32_t *bits;
    const uint8_t *ref_codes, *seq_codes;
    const uint4 *colrec;          // two uint4 per reference-slice position (annotate.cuh)
    const uint2 *relaid;
    const uint32_t *rowrec;
    uint16_t *tb;
    const float *tab;             // tabS [NP_TABQ][np_rows+1] (q-major), then tabL likewise
    const float *sub_tab;         // [5][5]  indexed [seq_base][ref_base]
    ChunkOut *out;                // indexed by chunk id
    // round-robin time slicing: run queue + per-chunk saved state
    int *rr_q; int rr_mask; int *rr_ctl;      // ctl[0] head, ctl[1] tail, ctl[2] finished chunks
    int *err;                                 // raised if the shared-memory window does not hold the rings (host bug)
    uint4 *ovf; int ovf_cap; int *ovf_cnt;    // WIDE runs only: {chunk id, anti-diagonal, slot, run} of records whose LEN/SHR run does not fit 11 bits
    uint32_t *rr_state; int rr_slice;
    AlignParams P;
};

#ifndef FWD_SPIN_NS
#define FWD_SPIN_NS 256
#endif
// words of saved per-lane state per cell: Mv1 Iv1 Dv1 dgv Mr1 dgr cc(8) rw
#define FWD_IE_BIT 31      // NP_REC_IE / NP_REC_DE in the upper half word of a record: IE is the sign bit of the INS difference as it
#define FWD_DE_BIT 30      // stands, DE the sign bit of the DEL difference moved down by one
#define FWD_TYP_SH (NP_REC_TYP + 16)
static_assert((NP_REC_IE << 16) == (1u << FWD_IE_BIT) && (NP_REC_DE << 16) == (1u << FWD_DE_BIT), "record flag bits");
static_assert(((7u << FWD_TYP_SH) | ((uint32_t)NP_RUN_SAT << 16)) < (1u << FWD_DE_BIT), "TYP and RUN below the flag bits");
#define FWD_RR_WORDS 15
#define FWD_RR_HDR 32      // uint32 words: d, Id, Dd
static __host__ __device__ inline size_t fwd_rr_state_words(int cpl) { return (size_t)FWD_RR_HDR + (size_t)FWD_RR_WORDS * cpl * 32 + (size_t)32 * cpl * 32; }

__global__ void rr_init_kernel(int *q, int cap, int n, int *ctl)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) q[i] = i < n ? i : -1;
    if (blockIdx.x == 0 && threadIdx.x == 0) { ctl[0] = 0; ctl[1] = n; ctl[2] = 0; }
}

// Run-queue words and the saved chunk state are read with gpu-scope STRONG loads served by L2 (ld.relaxed.gpu) and published
// with __threadfence() + a strong store.  An acquire load would be the textbook consumer side, but ptxas implements it as
// LDG.STRONG + CCTL.IVALL, i.e. every poll would throw away the SM's L1 (the score-table lines of all resident warps;
// measured in round 1 with system-scope loads: one spinning warp made a lone chunk 3x slower).  Nothing read after a pop
// can be stale in L1: the state is only ever read through L2.
__device__ __forceinline__ int ld_cg_poll(const int *p)
{ int v; asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ uint32_t ld_state(const uint32_t *p)
{ uint32_t v; asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ uint4 ld_state4(const uint4 *p)
{ uint4 v; asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory"); return v; }

// ---- explicit shared-memory access by 32-bit byte address
__device__ __forceinline__ float lds_f(uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
template <int OFF> __device__ __forceinline__ float lds_f_off(uint32_t a)
{ float v; asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(a), "n"(OFF)); return v; }
template <int OFF> __device__ __forceinline__ uint32_t lds_u_off(uint32_t a)
{ uint32_t v; asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF)); return v; }
__device__ __forceinline__ void lds_pair(uint32_t a, float &v, uint32_t &w)
{ asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];" : "=f"(v), "=r"(w) : "r"(a)); }
__device__ __forceinline__ void sts_slot(uint32_t a, float w0, float w1, float w2, uint32_t w3)
{ asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" :: "r"(a), "f"(w0), "f"(w1), "f"(w2), "r"(w3) : "memory"); }

// 16 bytes global -> shared without a register round trip (LDGSTS), L2 only
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src)
{ asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst), "l"(src) : "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ uint4 lds128(uint32_t a)
{ uint4 v; asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)); return v; }

// a ? b : c per bit (one LOP3)
__device__ __forceinline__ uint32_t bitsel(uint32_t m, uint32_t x, uint32_t y) { return (x & m) | (y & ~m); }
__device__ __forceinline__ float bitsel_f(uint32_t m, float x, float y) { return __uint_as_float((__float_as_uint(x) & m) | (__float_as_uint(y) & ~m)); }
// a | (b & M) as one LOP3 (left to itself, ptxas ORs two such masked words together first: one LOP3 more)
template <uint32_t M> __device__ __forceinline__ uint32_t or_masked(uint32_t a, uint32_t b)
{ uint32_t d; asm("lop3.b32 %0, %1, %2, %3, 0xf8;" : "=r"(d) : "r"(a), "r"(b), "n"(M)); return d; }

#define FWD_INF_BITS 0x7f800000u
#define FWD_SAT16 ((uint32_t)NP_RUN_SAT << 16)

// Ring of one warp: [NP_RING rows][NC positions] x 16 B {W0 MAT value or +INF, W1 LEN run-start value, W2 SHR run-start
// value, W3 = LEN.RUN | SHR.RUN << 16}; NC*128 bytes, aligned to its size.  Slot s sits at position (s % CPL)*32 + s / CPL
// of its row, so that the 32 lanes' 16-byte stores of one cell index are contiguous.
//
// One SHR candidate (aln.pyx:642-667 in gather form) from a pre-decoded descriptor {A, B, C} (annotate.cuh):
//   A [31:16] byte offset of the source pair inside the ring, row = (-n) mod 8: {W0,W1} if the source column starts the tract
//             (L_IDX == 0: run 0, value MAT.VAL), {W2,W3} otherwise; its low 3 bits hold n     [15:0] table row (n, L)
//   B ceil(65536 / n)        C 0 (start) or 0xffff0000 (continue: SHR.RUN << 16 of the source)
// An empty descriptor addresses the +INF table row.  `ok` is the checked variant's source test (always true when lean).
template <int NC, uint32_t SAT16 = FWD_SAT16>
__device__ __forceinline__ void shr_eval(uint32_t A, uint32_t B, uint32_t C, uint32_t dsh, uint32_t wbase, const float *__restrict__ tabS, uint32_t trows,
                                         bool ok, float &Sv, float &Sb, uint32_t &Sr)
{
    const uint32_t ad = (((A >> 16) + dsh) & (uint32_t)(NC * 128 - 8)) | wbase;
    float base; uint32_t w;
    lds_pair(ad, base, w);
    const uint32_t xs = w & C;                                        // SHR.RUN << 16 of the source, 0 at a tract start
    uint32_t q = __umulhi(xs, B);                                     // trunc(run / n) <= NP_RUN_SAT < NP_TABQ
    if (SAT16 != FWD_SAT16) q = min(q, (uint32_t)(NP_TABQ - 1));      // (WIDE: runs up to 65535; the tables are constant beyond q = 127)
#if FWD_TAB_PROBE      // timing probe only (results are wrong): every lookup hits one cache line = the bound on what staging the table could buy
    const float cand = base + __ldg(tabS + ((q * trows + (A & 0xffffu)) & 7u));
#else
    const float cand = base + __ldg(tabS + (q * trows + (A & 0xffffu)));
#endif
    const bool better = ok && cand < Sv;
    const uint32_t nr = __viaddmin_u32(xs, A & 0x70000u, SAT16);
    Sv = better ? cand : Sv; Sb = better ? base : Sb; Sr = better ? nr : Sr;
}

__device__ __forceinline__ float fmin3(float a, float b, float c)
{ float d; asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c)); return d; }

#ifndef FWD_TAB_PROBE
#define FWD_TAB_PROBE 0
#endif
#ifndef FWD_MINB
#define FWD_MINB 4      // min resident CTAs of the narrow-band instantiations: caps ptxas at 128 registers (4 CTAs x 4 warps per SM);
                        // with a hint of 1 it takes 164 and only 3 CTAs fit (measured: 29.0 instead of 26.7 ms per C2 step)
#endif
// T > 1: a TEAM of T warps shares one chunk -- the band's NC = 32*CPL*T slots are split across the warps (warp w of the team owns slots
// [w*32*CPL, (w+1)*32*CPL)), the history ring is the team's, the left neighbour of a warp's first cell comes from the previous warp
// through a double-buffered mailbox, and one named barrier per anti-diagonal orders ring / mailbox writes against the next step's
// reads.  Used where one chunk per warp is the wrong granularity: launches with fewer chunks than warp slots (latency bound) and
// bands wider than 128 cells (<4,2> instead of <8,1>: 168 registers and twice the warps instead of 255 registers).  Teams are not
// time-sliced (every chunk runs to its end).
// WIDE: the fallback for items whose traceback met a saturated n-polymer run (status 8 of the normal kernel): runs are carried
// unsaturated (16 bits, max_b_rows <= 65000), a record whose LEN/SHR run does not fit the 11-bit field stores 2047 and its true run
// goes to an overflow list the traceback consults.  Same arithmetic otherwise; api.cu re-runs a batch with WIDE only when needed.
template <int CPL, int T, bool WIDE = false>
__global__ void __launch_bounds__(fwd_warps(CPL, T) * 32, T == 4 ? 2 : CPL <= 2 ? FWD_MINB : (CPL == 4 && T == 1) ? 2 : 1) forward_kernel(const ForwardArgs a)
{
    constexpr uint32_t SAT16 = WIDE ? 0xffff0000u : FWD_SAT16;        // saturation of the carried LEN / SHR runs (<< 16)
    constexpr int NC = 32 * CPL * T;
    constexpr int WARPS = fwd_warps(CPL, T), TEAMS = WARPS / T;
    constexpr uint32_t ROWB = NC * 16, RING_BYTES = NC * 128;        // bytes per ring row / per team
    constexpr int SH = NC == 32 ? 27 : NC == 64 ? 26 : NC == 128 ? 25 : 24;      // 32 - log2(NC)
    extern __shared__ float smem[];
    __shared__ float s_sub[64];
    __shared__ uint32_t s_m16[8];
    __shared__ uint4 s_mail[2][T > 1 ? WARPS : 1];      // {MAT, DEL value, match run, row record} of every warp's last cell, by step parity
    __shared__ int s_pop[T > 1 ? TEAMS : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int team = warp / T, wt = warp % T;            // team of this warp, index inside the team
    auto team_sync = [&]() {
        if (T > 1) asm volatile("bar.sync %0, %1;" :: "r"(team + 1), "n"(T * 32) : "memory"); else __syncwarp();
    };
    for (int t = threadIdx.x; t < 64; t += WARPS * 32) {
        const int sb = t >> 3, rb = t & 7;
        s_sub[t] = (sb < 5 && rb < 5) ? a.sub_tab[sb * 5 + rb] : 0.f;
    }
    if (threadIdx.x < 8) s_m16[threadIdx.x] = threadIdx.x ? (65536u + threadIdx.x - 1u) / threadIdx.x : 0u;
    __syncthreads();
    const uint32_t smem_raw = (uint32_t)__cvta_generic_to_shared(smem);
    const uint32_t smem_base = (smem_raw + RING_BYTES - 1u) & ~(RING_BYTES - 1u);
    {   // the host sizes the dynamic window from the kernel's static size (launch_forward); never run past it
        uint32_t dyn; asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
        const uint32_t front = smem_base - smem_raw;
        const uint32_t need = front + (uint32_t)TEAMS * RING_BYTES + (front >= (uint32_t)WARPS * 1024u ? 0u : (uint32_t)WARPS * 1024u);
        if (need > dyn) {
            if (threadIdx.x == 0) atomicExch(a.err, 1);
            return;
        }
    }
    const uint32_t wbase = smem_base + (uint32_t)team * RING_BYTES;
    // column-record FIFO of the warp (32 records x 32 B, filled by cp.async 16 records ahead of use): in the alignment slack
    // in front of the rings when it is large enough, else behind them (launch_forward sizes the window the same way)
    constexpr uint32_t STAGE_BYTES = 32u * 32u;
    const bool stage_front = smem_base - smem_raw >= (uint32_t)WARPS * STAGE_BYTES;
    const uint32_t stbase = (stage_front ? smem_raw : smem_base + (uint32_t)TEAMS * RING_BYTES) + (uint32_t)warp * STAGE_BYTES;
    const uint32_t mailbase = (uint32_t)__cvta_generic_to_shared(&s_mail[0][0]);
    const uint32_t subbase = (uint32_t)__cvta_generic_to_shared(s_sub);
    const uint32_t m16base = (uint32_t)__cvta_generic_to_shared(s_m16);

    const int r = a.P.r;
    const float gopen = a.P.gap_open, gext = a.P.gap_ext;
    const float *__restrict__ tabS = a.tab;
    const float *__restrict__ tabL = a.tab + (size_t)(a.P.np_rows + 1) * NP_TABQ;
    const uint32_t trows = (uint32_t)a.P.np_rows + 1u;          // row stride of the q-major score tables
    const uint32_t empty_A = (((uint32_t)(NP_RING - 1) * ROWB) << 16) | (uint32_t)a.P.np_rows;      // annotate.cuh: "no candidate" -> the +INF table row
    const int src_lane = (lane + 31) & 31;
    const int spare = NC - (2 * r + 1);
    // aliasing windows (header): none possible when spare >= 4 or max_n < spare + 3; a run of 6 equal ops when spare == 3 and
    // max_n == 6; otherwise (band widths nobody uses: W = NC-1, NC-2, NC) every block runs the checked variant
    const int risk_mode = (spare >= 4 || a.P.max_n < spare + 3) ? 0 : (spare == 3 ? 1 : 2);
    const uint32_t in_lim = (uint32_t)(2 * r - 2) << SH;        // es <= in_lim  <=>  1 <= b_col <= 2r-1
    uint32_t mypos[CPL];                                         // byte offset of the lane's slots inside a ring row
#pragma unroll
    for (int k = 0; k < CPL; k++) mypos[k] = (uint32_t)(k * 32 * T + wt * 32 + lane) * 16u;

    for (;;) {
        int idx = 0;
        {   // pop the next runnable chunk (FIFO).  An empty queue stays empty -- a chunk is handed back only while another one
            // waits (tail - head > 0 at its slice boundary), and a finished chunk takes one out -- so a warp (team) that finds
            // nothing queued is done and leaves: idle pollers would take issue slots from the warps still working on the tail.
            // Only a warp that saw an entry and lost the race for it waits (for a hand-back, or for the end of the launch).
            if (lane == 0 && wt == 0) {
                int v = -2;
                if (ld_cg_poll(a.rr_ctl + 1) - ld_cg_poll(a.rr_ctl) > 0) {
                    const int pos = atomicAdd(a.rr_ctl, 1);
                    int *qp = a.rr_q + (pos & a.rr_mask);
                    unsigned ns = FWD_SPIN_NS;
                    while ((v = ld_cg_poll(qp)) < 0) {
                        if (ld_cg_poll(a.rr_ctl + 2) >= a.n) { v = -2; break; }
                        __nanosleep(ns);
                        if (ns < 4096u) ns <<= 1;
                    }
                    if (v >= 0) __stcg(qp, -1);
                }
                idx = v;
            }
            if (T > 1) {      // the team's first warp popped: hand the index to the others
                if (lane == 0 && wt == 0) s_pop[team] = idx;
                team_sync();
                idx = s_pop[team];
                team_sync();
            } else idx = __shfl_sync(NP_FULL, idx, 0);
            if (idx < 0) break;
        }
        const int cid = a.order[idx];
        const ChunkDesc c = a.chunks[cid];
        if (!c.valid) {
            if (lane == 0 && wt == 0) { a.out[cid].score = 0.f; atomicAdd(a.rr_ctl + 2, 1); }
            continue;
        }
        const ChunkSlot sl = a.slots[idx];
        const ItemDesc &I = a.items[c.item];
        const uint32_t *__restrict__ bits = a.bits + I.bit_word_off;
        const uint4 *__restrict__ col = a.colrec + 2 * sl.col_off;
        const uint2 *__restrict__ rel = a.relaid + sl.col_off;
        const uint32_t *__restrict__ row = a.rowrec + sl.row_off;
        const uint8_t *__restrict__ refs = a.ref_codes + I.ref_start + min(c.c0, I.ref_len);
        const uint8_t *__restrict__ seqs = a.seq_codes + I.seq_start + min(c.r0, I.seq_len);
        uint16_t *tbp = a.tb + (size_t)sl.tb_off * NC + (wt * 32 + lane) * CPL;
        const int B = c.B, imax = c.imax, jmax = c.jmax;

        // ---- per-slot state.  At d = 0: jlo = -r, slot s holds column j = -r + ((s + r) mod NC), row i = -j.
        float Mv1[CPL], Iv1[CPL], Dv1[CPL], dgv[CPL];   // previous anti-diagonal: MAT/INS/DEL values; diag MAT value
        uint32_t Mr1[CPL], dgr[CPL];                      // match run << 16 (RUN if TYP==MAT else 0) of the cell; of the diag cell
        uint4 ca[CPL], cb[CPL];                           // column record: ca = {S0.A, S0.B, S0.C, S1.A}, cb = {S1.B, S1.C, Z, LEN}
        uint32_t rw[CPL], es[CPL];                        // row record; ((b_col - 1) mod NC) << SH
        int d0 = 0, Id = 0, Dd = 0;
        uint32_t *st = a.rr_state + (size_t)idx * fwd_rr_state_words(NC / 32);
        d0 = (int)ld_state(st);
        if (d0 > 0) {     // resume: scalars, per-lane registers, history ring
            Id = (int)ld_state(st + 1); Dd = (int)ld_state(st + 2);
            constexpr int LT = 32 * T;                          // lanes of the team: the stride of one saved register word
            const uint32_t *sp = st + FWD_RR_HDR + wt * 32 + lane;
#pragma unroll
            for (int k = 0; k < CPL; k++) {
                const uint32_t *q = sp + (size_t)k * FWD_RR_WORDS * LT;
                Mv1[k] = __uint_as_float(ld_state(q)); Iv1[k] = __uint_as_float(ld_state(q + LT)); Dv1[k] = __uint_as_float(ld_state(q + 2 * LT));
                dgv[k] = __uint_as_float(ld_state(q + 3 * LT)); Mr1[k] = ld_state(q + 4 * LT); dgr[k] = ld_state(q + 5 * LT);
                ca[k] = make_uint4(ld_state(q + 6 * LT), ld_state(q + 7 * LT), ld_state(q + 8 * LT), ld_state(q + 9 * LT));
                cb[k] = make_uint4(ld_state(q + 10 * LT), ld_state(q + 11 * LT), ld_state(q + 12 * LT), ld_state(q + 13 * LT));
                rw[k] = ld_state(q + 14 * LT);
                es[k] = (uint32_t)((wt * 32 + lane) * CPL + k + r - Dd - 1) << SH;
            }
            const uint4 *rp = reinterpret_cast<const uint4 *>(st + FWD_RR_HDR + (size_t)FWD_RR_WORDS * CPL * LT);
#pragma unroll
            for (int t = wt; t < NC / 4; t += T) {
                const uint4 v = ld_state4(rp + t * 32 + lane);
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(wbase + (uint32_t)(t * 32 + lane) * 16u), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
            }
            // the mailbox entry the next step reads (par = 0 reads half 1): the warp's last cell as the previous step left it
            if (T > 1 && lane == 31)
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(mailbase + ((uint32_t)WARPS + (uint32_t)warp) * 16u),
                             "r"(__float_as_uint(Mv1[CPL - 1])), "r"(__float_as_uint(Dv1[CPL - 1])), "r"(Mr1[CPL - 1]), "r"(rw[CPL - 1]) : "memory");
        } else {
            const uint4 e0 = make_uint4(empty_A, 0u, 0u, empty_A), e1 = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
            for (int k = 0; k < CPL; k++) {
                Mv1[k] = Iv1[k] = Dv1[k] = dgv[k] = 0.f; Mr1[k] = dgr[k] = 0u;
                const int s = (wt * 32 + lane) * CPL + k;
                const int bc = (s + r) & (NC - 1);
                es[k] = (uint32_t)(bc - 1) << SH;
                const int j0 = bc - r;
                rw[k] = (j0 <= 0) ? row[-j0] : 0u;
                const int jc = j0 >= 0 ? j0 : (j0 == -r ? NC - r : -1);
                ca[k] = jc >= 0 ? col[2 * jc] : e0;
                cb[k] = jc >= 0 ? col[2 * jc + 1] : e1;
            }
            // the ring starts all-INF: sources before the chunk's first anti-diagonal are no candidates (aln.pyx:497-499)
#pragma unroll
            for (int t = wt; t < NC / 4; t += T)
                asm volatile("st.shared.v4.u32 [%0], {%1,%1,%1,%2};" :: "r"(wbase + (uint32_t)(t * 32 + lane) * 16u), "r"(FWD_INF_BITS), "r"(0u) : "memory");
        }
        {   // prime the column-record FIFO: records [cn, (cn & ~15) + 32), cn = the next column to enter the band.  The previous
            // chunk's last refill may still be in flight (nothing waited for it if the chunk ended or was handed back first) and
            // would land on top of the new records: drain it before the slots are written again (racecheck found this WAW)
#ifndef FWD_NO_PRIME_DRAIN      // (A/B switch)
            cp_async_wait_all();
            __syncwarp();
#endif
            const int cn = Dd - r + NC + 1, lim = (cn & ~15) + 32;
#pragma unroll
            for (int t = 0; t < 2; t++) {
                const int cf = cn + t * 16 + (lane >> 1);
                if (cf < lim) cp_async16(stbase + ((uint32_t)cf & 31u) * 32u + (uint32_t)(lane & 1) * 16u, col + 2 * cf + (lane & 1));
            }
            cp_async_wait_all();
        }
        team_sync();
        float infd = (float)(100 * (d0 > 0 ? d0 - 1 : 0));   // 100*d, exact in fp32 (d < 2^16); advanced at the top of a step
        uint32_t dsh = (uint32_t)d0 * ROWB;                    // d * ROWB (ring row of this anti-diagonal, before masking)
        uint16_t *rowp = tbp + (size_t)d0 * NC;
        uint32_t hist = 0;                                     // op history (bit t = op t+1 steps back), checked variant only
        int dEnd = min(B, d0 + a.rr_slice);
        int d = d0;
        uint32_t par = 0u;                                      // step parity: which mailbox half this step writes

        // ------------------------------------------------------------------------------------------------ one step
        auto step = [&](auto steady_tag, const uint32_t o, const bool first, uint32_t &nrow_buf, int &nrow_i) {
            constexpr bool STEADY = decltype(steady_tag)::value;
            // steady block: edge and spare slots compute like interior ones and are overridden where read (ring store below).  Not at
            // CPL 8: that form already runs at 255 registers, and the second ring store's extra live values cost it more spills
            constexpr bool LEAN_EDGE = STEADY && CPL <= 4;
            float lMv[CPL], lDv[CPL]; uint32_t lMr[CPL];
            if (STEADY || !first) {
                infd += 100.f;
                const float a0s = __shfl_sync(NP_FULL, Mv1[CPL - 1], src_lane);
                const float a1s = __shfl_sync(NP_FULL, Dv1[CPL - 1], src_lane);
                const uint32_t a2s = __shfl_sync(NP_FULL, Mr1[CPL - 1], src_lane);
                uint32_t a3 = __shfl_sync(NP_FULL, rw[CPL - 1], src_lane);
                float a0 = a0s, a1 = a1s; uint32_t a2 = a2s;
                if (T > 1 && lane == 0) {      // the left neighbour of the warp's first cell is the previous warp's last cell
                    const uint4 m = lds128(mailbase + ((par ^ 1u) * (uint32_t)WARPS + (uint32_t)(team * T + (wt + T - 1) % T)) * 16u);
                    a0 = __uint_as_float(m.x); a1 = __uint_as_float(m.y); a2 = m.z; a3 = m.w;
                }
#pragma unroll
                for (int k = CPL - 1; k >= 0; k--) {
                    lMv[k] = k ? Mv1[k > 0 ? k - 1 : 0] : a0;
                    lDv[k] = k ? Dv1[k > 0 ? k - 1 : 0] : a1;
                    lMr[k] = k ? Mr1[k > 0 ? k - 1 : 0] : a2;
                    rw[k] = k ? rw[k > 0 ? k - 1 : 0] : a3;
                }
                if (o) {      // 'I': the next row enters at b_col == 0
                    Id++;
                    const uint32_t nrow = __shfl_sync(NP_FULL, nrow_buf, nrow_i);
                    nrow_i++;
#pragma unroll
                    for (int k = 0; k < CPL; k++) if (es[k] == (0xffffffffu << SH)) rw[k] = nrow;
                } else {      // 'D': every column moves down one b_col; the one reaching 0 is dead, its slot takes column j+NC
                    Dd++;
                    const int cnew = Dd - r + NC;                 // the column that takes over the retired slot
#pragma unroll
                    for (int k = 0; k < CPL; k++) {
                        es[k] -= 1u << SH;
                        if (es[k] == (0xffffffffu << SH)) {
                            const uint32_t sa = stbase + ((uint32_t)cnew & 31u) * 32u;
                            ca[k] = lds128(sa); cb[k] = lds128(sa + 16u);
                        }
                    }
                    if ((cnew & 15) == 15) {      // an aligned batch of 16 records is consumed: refill its FIFO slots, 16 D ops ahead of use
                        cp_async_wait_all();      // (the batch requested 16 D ops ago, about to be consumed)
                        __syncwarp();
                        const int cf = cnew + 17 + (lane >> 1);
                        cp_async16(stbase + ((uint32_t)cf & 31u) * 32u + (uint32_t)(lane & 1) * 16u, col + 2 * cf + (lane & 1));
                    }
                }
                if (!STEADY) hist = ((hist << 1) | o) & 0x3fu;
            } else {
#pragma unroll
                for (int k = 0; k < CPL; k++) { lMv[k] = lDv[k] = 0.f; lMr[k] = 0u; }
            }
            const float edgev = infd + 100.f;

            bool in[CPL];
            int bc[CPL];                                  // numeric b_col (checked variant only)
            if (STEADY) {
#pragma unroll
                for (int k = 0; k < CPL; k++) in[k] = es[k] <= in_lim;
            } else {      // interior-cell bounds on b_col for this anti-diagonal (aln.pyx:497-507)
                int lo = max(1, max(Id + r - imax, r - Dd)), hi = min(2 * r - 1, min(Id + r, jmax + r - Dd));
                if (hi < lo) { lo = 1; hi = 0; }
#pragma unroll
                for (int k = 0; k < CPL; k++) {
                    bc[k] = (int)(((es[k] >> SH) + 1u) & (uint32_t)(NC - 1));
                    in[k] = (unsigned)(bc[k] - lo) <= (unsigned)(hi - lo) && hi >= lo;
                }
            }
            // #I among the last n ops, n = 1..6, 4 bits each at nibble n (checked variant: source tests)
            uint32_t sip = 0;
            if (!STEADY) {
#pragma unroll
                for (int n = 1; n <= 6; n++) sip |= (uint32_t)__popc(hist & ((1u << n) - 1u)) << (4 * n);
            }

            float Sv[CPL], Sb[CPL], Lv[CPL], Lb[CPL]; uint32_t Sr[CPL], Lr[CPL];     // runs << 16
            uint32_t any1 = 0u, anyl = 0u, anyg = 0u, gN = 0u;
            uint32_t lwm[CPL];      // LEN eligibility as data words, not predicates: they stay live across the votes below, and ptxas
                                    // packs live predicates into a register bit by bit (that was 12 instructions per anti-diagonal)
#pragma unroll
            for (int k = 0; k < CPL; k++) {
                Sv[k] = infd; Lv[k] = infd; Sb[k] = __uint_as_float(FWD_INF_BITS); Lb[k] = __uint_as_float(FWD_INF_BITS); Sr[k] = 0u; Lr[k] = 0u;
                // one-hot LEN period vs the row's "tract present" bits, interior cells only -- except in a steady block, where the
                // other slots (b_col 0, b_col 2r, spares) may evaluate a LEN candidate: their value is replaced by the edge value,
                // their record by 0, their match run by 0, and their ring slot by the all-INF one below, so it is never read
                lwm[k] = (LEAN_EDGE || in[k]) ? (rw[k] & cb[k].w & 0x03f00000u) : 0u;
                any1 |= ca[k].w ^ empty_A; anyl |= lwm[k]; anyg |= cb[k].z;      // (votes on the unmasked words: slightly conservative)
            }
            // ---- SHR gather: descriptor 0 (largest period), then descriptor 1 if any lane has one
#pragma unroll
            for (int k = 0; k < CPL; k++) {
                bool ok = true;
                if (!STEADY) { const uint32_t n = (ca[k].x >> 16) & 7u; ok = in[k] && bc[k] > (int)((sip >> (4 * n)) & 7u); }
                shr_eval<NC, SAT16>(ca[k].x, ca[k].y, ca[k].z, dsh, wbase, tabS, trows, ok, Sv[k], Sb[k], Sr[k]);
            }
            if (__any_sync(NP_FULL, any1 != 0u)) {
#pragma unroll
                for (int k = 0; k < CPL; k++) {
                    bool ok = true;
                    if (!STEADY) { const uint32_t n = (ca[k].w >> 16) & 7u; ok = in[k] && bc[k] > (int)((sip >> (4 * n)) & 7u); }
                    shr_eval<NC, SAT16>(ca[k].w, cb[k].x, cb[k].y, dsh, wbase, tabS, trows, ok, Sv[k], Sb[k], Sr[k]);
                }
            }
            // ---- LEN gather (aln.pyx:602-633): single eligible period, 2-bit k-mer unit compare in registers
            if (__any_sync(NP_FULL, anyl != 0u)) {
#pragma unroll
                for (int k = 0; k < CPL; k++) {
                    if (lwm[k] != 0u) {
                        const uint32_t D = cb[k].w;
                        if ((cb[k].z | rw[k]) & 2u) {
                            gN |= 1u << k; anyg |= 1u;             // an N inside a k-mer: byte-wise compare on the generic path
                        } else {
                            const uint32_t n = D & 7u;
                            // match() of aln.pyx:606-607: seq[i-n .. i) against ref[j .. j+n).  The row record carries the 6-mer
                            // that ENDS at seq[i-1] (its last n codes = the top 2n bits of the field are the read-side unit), the
                            // column record ref[j .. j+n) already moved to those bits, and their mask 12 bits higher (annotate.cuh)
                            bool ok = ((rw[k] ^ cb[k].z) & (cb[k].z >> 12) & 0xfff00u) == 0u;
                            if (!STEADY) ok = ok && (bc[k] + (int)n - (int)((sip >> (4 * n)) & 7u) <= 2 * r - 1);
                            const bool start = (rw[k] & (lwm[k] << 6)) != 0u;                      // "tract start" bit 25+n = the eligible "present" bit 19+n << 6
                            const uint32_t ad = ((dsh - n * ROWB + mypos[k]) & (RING_BYTES - 16u)) | wbase;
                            const float base = lds_f(ad + (start ? 0u : 4u));                       // MAT.VAL or the carried LEN run-start value
                            const uint32_t run0 = start ? 0u : (lds_u_off<12>(ad) & 0xffffu);
                            uint32_t q = __umulhi(run0 << 16, lds_u_off<0>(m16base + n * 4u));
                            if (WIDE) q = min(q, (uint32_t)(NP_TABQ - 1));
                            const float cand = base + __ldg(tabL + (q * trows + ((D >> 3) & 0x3ffu)));
                            if (ok && cand < Lv[k]) { Lv[k] = cand; Lr[k] = min(run0 + n, SAT16 >> 16) << 16; Lb[k] = base; }
                        }
                    }
                }
            }
            // ---- generic path (rare): all periods from the relaid byte record in global memory
            if (__any_sync(NP_FULL, (anyg & 1u) != 0u)) {
#pragma unroll
                for (int k = 0; k < CPL; k++) {
                    if (in[k] && ((cb[k].z | (gN >> k)) & 1u) != 0u) {
                        const int bcn = (int)(((es[k] >> SH) + 1u) & (uint32_t)(NC - 1));
                        const int i = Id + r - bcn, j = Dd - r + bcn;
                        const uint2 rb = rel[j];
                        const uint32_t h6 = STEADY ? 0u : hist;       // (steady blocks need no source tests)
                        if (cb[k].z & 1u) {
                            for (int n = a.P.max_n; n >= 1; n--) {      // SHR, every period
                                const uint32_t byte = ((n <= 4 ? rb.x : rb.y) >> ((8 * (n - 1)) & 31)) & 0xffu;
                                const uint32_t L = byte & 0x7fu;
                                if (!L) continue;
                                if (!STEADY && bcn <= __popc(h6 & ((1u << n) - 1u))) continue;
                                const uint32_t sslot = (uint32_t)(j - n) & (uint32_t)(NC - 1);
                                const uint32_t off = (uint32_t)((-n) & (NP_RING - 1)) * ROWB + ((sslot % CPL) * (uint32_t)(32 * T) + sslot / CPL) * 16u + ((byte & 0x80u) ? 0u : 8u);
                                const uint32_t A = ((off | (uint32_t)n) << 16) | (uint32_t)((n - 1) * (a.P.max_l + 1) + (int)L);
                                shr_eval<NC, SAT16>(A, lds_u_off<0>(m16base + n * 4u), (byte & 0x80u) ? 0u : 0xffff0000u, dsh, wbase, tabS, trows, true, Sv[k], Sb[k], Sr[k]);
                            }
                        }
                        uint32_t lm = (rb.y >> 22) & (rw[k] >> 20) & 0x3fu;   // LEN, every eligible period
                        while (lm) {
                            const int n = 32 - __clz(lm);
                            lm &= ~(1u << (n - 1));
                            if (!STEADY && bcn + n - __popc(h6 & ((1u << n) - 1u)) > 2 * r - 1) continue;
                            const int si = i - n;
                            bool eq = true;
                            for (int t = 0; t < n; t++) eq = eq && (seqs[si + t] == refs[j + t]);
                            if (!eq) continue;
                            const uint2 cjn = rel[j + n];
                            const int L = (int)(((n <= 4 ? cjn.x : cjn.y) >> ((8 * (n - 1)) & 31)) & 0x7fu);
                            const bool start = ((rw[k] >> (25 + n)) & 1u) != 0u;
                            const uint32_t ad = ((dsh - (uint32_t)n * ROWB + mypos[k]) & (RING_BYTES - 16u)) | wbase;
                            const float base = lds_f(ad + (start ? 0u : 4u));
                            const uint32_t run0 = start ? 0u : (lds_u_off<12>(ad) & 0xffffu);
                            uint32_t q = __umulhi(run0 << 16, lds_u_off<0>(m16base + n * 4u));
                            if (WIDE) q = min(q, (uint32_t)(NP_TABQ - 1));
                            const float cand = base + __ldg(tabL + (q * trows + (uint32_t)((n - 1) * (a.P.max_l + 1) + L)));
                            if (cand < Lv[k]) { Lv[k] = cand; Lr[k] = min(run0 + (uint32_t)n, SAT16 >> 16) << 16; Lb[k] = base; }
                        }
                    }
                }
            }

            // ---- INS / DEL / MAT (aln.pyx:525-592); records are assembled in the upper half word
            uint32_t pk[CPL];
            float Mv[CPL], Iv[CPL], Dv[CPL];
            const uint32_t rowad = (dsh & (RING_BYTES - 1u)) | wbase;
#pragma unroll
            for (int k = 0; k < CPL; k++) {
                // INS from top = own previous value; DEL from left.  Only the "extended" bits are kept (see common.cuh)
                const float iv1 = Mv1[k] + gopen, iv2 = Iv1[k] + gext;
                // "extended" (aln.pyx:536, 558) = strict '<' = the sign bit of the difference: the operands are finite (MAT / INS / DEL values
                // are never the ring's +INF), a difference of distinct floats never rounds to zero, and x - x = +0
                uint32_t iext = __float_as_uint(iv2 - iv1);
                Iv[k] = fminf(iv1, iv2);
                const float dv1 = lMv[k] + gopen, dv2 = lDv[k] + gext;
                uint32_t dext = __float_as_uint(dv2 - dv1);
                Dv[k] = fminf(dv1, dv2);
                uint32_t pm = __viaddmin_u32(dgr[k], 0x10000u, FWD_SAT16);           // typ MAT = 0
                float dg = dgv[k] + lds_f(subbase + ((rw[k] | cb[k].z) & 0xfcu));    // sub_scores[seq[i-1]][ref[j-1]] (aln.pyx:575)
                if (!STEADY) {
                    const int i = Id + r - bc[k], j = Dd - r + bc[k];
                    if (i <= 1) iext = 0u;                                           // aln.pyx:537-538 (run restarts), :525-528
                    if (j <= 1) dext = 0u;                                           // aln.pyx:559-560, :547-550
                    if (i == 0) Iv[k] = (float)(100 * (j + 1));
                    if (j == 0) Dv[k] = (float)(100 * (i + 1));
                    if (!(i > 0 && j > 0)) { dg = Dv[k] + 100.f; pm = 0u; }
                }
                // MAT = the first minimum in the order diag, INS, LEN, DEL, SHR (strict '<' chain of aln.pyx:585-592)
                const float best = fmin3(fmin3(dg, Iv[k], Lv[k]), Dv[k], Sv[k]);
                uint32_t p = ((uint32_t)T_SHR << FWD_TYP_SH) | (WIDE ? min(Sr[k], FWD_SAT16) : Sr[k]);
                if (Dv[k] == best) p = (uint32_t)T_DEL << FWD_TYP_SH;
                if (Lv[k] == best) p = ((uint32_t)T_LEN << FWD_TYP_SH) | (WIDE ? min(Lr[k], FWD_SAT16) : Lr[k]);
                if (Iv[k] == best) p = (uint32_t)T_INS << FWD_TYP_SH;
                if (dg == best) p = pm;
                // the flags are sign bits: IE stays where it is, DE moves down one bit, dext >> 1 written as the high word of
                // dext * 2^31 so that it is an IMAD.HI on the FMA pipe, not a SHF on the busy ALU pipe.  Two LOP3s are left.
                p = or_masked<1u << FWD_DE_BIT>(or_masked<1u << FWD_IE_BIT>(p, iext), __umulhi(dext, 1u << (FWD_DE_BIT + 1)));
                if (!in[k]) p = 0u;
                if (WIDE) {      // a LEN / SHR record whose run does not fit the field: the true run goes to the overflow list
                    const uint32_t t3 = (p >> FWD_TYP_SH) & 7u, full = t3 == (uint32_t)T_LEN ? Lr[k] : Sr[k];
                    if ((t3 == (uint32_t)T_LEN || t3 == (uint32_t)T_SHR) && full >= FWD_SAT16) {
                        const int e = atomicAdd(a.ovf_cnt, 1);
                        if (e < a.ovf_cap) a.ovf[e] = make_uint4((uint32_t)cid, dsh / ROWB, (uint32_t)((wt * 32 + lane) * CPL + k), full >> 16);
                    }
                }
                Mr1[k] = dg == best && in[k] ? pm : 0u;                              // match run of this cell (0 unless TYP == MAT)
                pk[k] = p;
                // history ring: every slot writes; +INF unless the cell is interior.  The lean step stores every slot as computed and
                // lets the few non-interior slots store again, all three values +INF (same lane, program order: the second store
                // wins): one predicated STS instead of two FSELs per cell.  Their run word is then never used (a source whose
                // values are +INF yields a +INF candidate whatever its run).
                if (LEAN_EDGE) {
                    sts_slot(rowad + mypos[k], best, Lb[k], Sb[k], __byte_perm(Lr[k], Sr[k], 0x7632));
                    if (!in[k]) sts_slot(rowad + mypos[k], __uint_as_float(FWD_INF_BITS), __uint_as_float(FWD_INF_BITS), __uint_as_float(FWD_INF_BITS), 0u);
                } else {
                    sts_slot(rowad + mypos[k], in[k] ? best : __uint_as_float(FWD_INF_BITS), Lb[k], in[k] ? Sb[k] : __uint_as_float(FWD_INF_BITS),
                             __byte_perm(Lr[k], Sr[k], 0x7632));
                }
                // EDGE (b_col 0 / 2r): every state INF*(b_row+1), TYP MAT, RUN 0 (aln.pyx:502-507).  Cells outside the chunk
                // (aln.pyx:497-499) are never read by interior cells; they get the same harmless value.
                Mv[k] = in[k] ? best : edgev;
                Iv[k] = in[k] ? Iv[k] : edgev;
                Dv[k] = in[k] ? Dv[k] : edgev;
            }
            // ---- traceback row (slot order), streamed once, read once by the traceback
            if (CPL == 1) __stcs(reinterpret_cast<unsigned short *>(rowp), (unsigned short)(pk[0] >> 16));
            else {
#pragma unroll
                for (int k = 0; k < CPL; k += 2)
                    __stcs(reinterpret_cast<unsigned int *>(rowp) + (k >> 1), __byte_perm(pk[k], pk[k + 1 < CPL ? k + 1 : k], 0x7632));
            }
            if (T > 1 && lane == 31)
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(mailbase + (par * (uint32_t)WARPS + (uint32_t)warp) * 16u),
                             "r"(__float_as_uint(Mv[CPL - 1])), "r"(__float_as_uint(Dv[CPL - 1])), "r"(Mr1[CPL - 1]), "r"(rw[CPL - 1]) : "memory");
            team_sync();
            par ^= 1u;
#pragma unroll
            for (int k = 0; k < CPL; k++) {
                dgv[k] = lMv[k]; dgr[k] = lMr[k];                 // next step's diagonal neighbour = this step's left
                Mv1[k] = Mv[k]; Iv1[k] = Iv[k]; Dv1[k] = Dv[k];
            }
            dsh += ROWB;
            rowp += NC;
        };   // step

        // ------------------------------------------------------------------------------------------------ block loop
        uint32_t cw_prev = 0u; int have_prev = -1;        // previous bit word (for the aliasing-window test) and its index
        for (;;) {
            if (d >= dEnd) {
                if (dEnd >= B) break;
                // slice over: hand the chunk back only if another chunk is waiting for a warp (tail - head > 0)
                int queued = 0;
                if (lane == 0 && wt == 0) queued = ld_cg_poll(a.rr_ctl + 1) - ld_cg_poll(a.rr_ctl);
                if (T > 1) {      // one decision per team
                    if (lane == 0 && wt == 0) s_pop[team] = queued;
                    team_sync();
                    queued = s_pop[team];
                    team_sync();
                } else queued = __shfl_sync(NP_FULL, queued, 0);
                if (queued > 0) break;
                dEnd = min(B, dEnd + a.rr_slice);
            }
            uint32_t nrow_buf = row[Id + r + 1 + lane];       // the next 32 rows to enter the band (at b_col == 0)
            int nrow_i = 0;
            if (d == 0) {
                step(std::false_type{}, 0u, true, nrow_buf, nrow_i);
                d = 1;
                continue;
            }
            const int g = c.brk + d - 1;                       // op that leads to anti-diagonal d
            const int wi = g >> 5, b0 = g & 31;
            const uint32_t cw = bits[wi];
            if (have_prev != wi - 1) { cw_prev = wi > 0 ? bits[wi - 1] : 0u; }
            const int nst = min(32 - b0, dEnd - d);
            uint32_t ops = cw >> b0;
            const uint32_t opm = nst >= 32 ? 0xffffffffu : ((1u << nst) - 1u);
            const int nI = __popc(ops & opm), nD = nst - nI;
            // steady block: every cell 1 <= b_col <= 2r-1 of every step is interior with i, j >= 2
            bool steady = Id >= r + 1 && Dd >= r + 1 && Id + nI <= imax - r + 1 && Dd + nD <= jmax - r + 1;
            const uint64_t win = ((uint64_t)cw << 32) | cw_prev;      // op g' at bit 32 + (g' - 32*wi)
            if (risk_mode == 2) steady = false;
            else if (risk_mode == 1 && steady) {
                // six equal ops ending at one of this block's ops: run of ones / zeros of length 6 whose last bit is in
                // [32 + b0, 32 + b0 + nst)
                const uint64_t x1 = win, x0 = ~win;
                uint64_t y1 = x1 & (x1 >> 1); y1 = y1 & (y1 >> 2) & (y1 >> 4);      // bit p: ops p .. p+5 all 'I'
                uint64_t y0 = x0 & (x0 >> 1); y0 = y0 & (y0 >> 2) & (y0 >> 4);
                const uint64_t endm = (nst >= 32 ? 0xffffffffull : ((1ull << nst) - 1ull)) << (32 + b0 - 5);
                if ((y1 | y0) & endm) steady = false;
            }
            if (steady) {
#pragma unroll 1
                for (int t = 0; t < nst; t++) { step(std::true_type{}, ops & 1u, false, nrow_buf, nrow_i); ops >>= 1; }
            } else {
                hist = (uint32_t)(__brevll(win >> (32 + b0 - 6)) >> 58) & 0x3fu;       // ops g-1 .. g-6 at bits 0 .. 5
#pragma unroll 1
                for (int t = 0; t < nst; t++) { step(std::false_type{}, ops & 1u, false, nrow_buf, nrow_i); ops >>= 1; }
            }
            d += nst;
            cw_prev = cw; have_prev = wi;
        }

        if (dEnd < B) {     // slice over: save the chunk's state and hand it back to the run queue
            constexpr int LT = 32 * T;
            uint32_t *sp = st + FWD_RR_HDR + wt * 32 + lane;
#pragma unroll
            for (int k = 0; k < CPL; k++) {
                uint32_t *q = sp + (size_t)k * FWD_RR_WORDS * LT;
                __stcg(q, __float_as_uint(Mv1[k])); __stcg(q + LT, __float_as_uint(Iv1[k])); __stcg(q + 2 * LT, __float_as_uint(Dv1[k]));
                __stcg(q + 3 * LT, __float_as_uint(dgv[k])); __stcg(q + 4 * LT, Mr1[k]); __stcg(q + 5 * LT, dgr[k]);
                __stcg(q + 6 * LT, ca[k].x); __stcg(q + 7 * LT, ca[k].y); __stcg(q + 8 * LT, ca[k].z); __stcg(q + 9 * LT, ca[k].w);
                __stcg(q + 10 * LT, cb[k].x); __stcg(q + 11 * LT, cb[k].y); __stcg(q + 12 * LT, cb[k].z); __stcg(q + 13 * LT, cb[k].w);
                __stcg(q + 14 * LT, rw[k]);
            }
            uint4 *rp = reinterpret_cast<uint4 *>(st + FWD_RR_HDR + (size_t)FWD_RR_WORDS * CPL * LT);
#pragma unroll
            for (int t = wt; t < NC / 4; t += T) {
                uint4 v;
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(wbase + (uint32_t)(t * 32 + lane) * 16u));
                __stcg(rp + t * 32 + lane, v);
            }
            if (lane == 0 && wt == 0) { __stcg(st, (uint32_t)dEnd); __stcg(st + 1, (uint32_t)Id); __stcg(st + 2, (uint32_t)Dd); }
            __threadfence();
            team_sync();      // every warp's part of the state is out (and fenced) before the chunk becomes runnable again
            if (lane == 0 && wt == 0) {
                __threadfence();
                const int p2 = atomicAdd(a.rr_ctl + 1, 1);
                __stcg(a.rr_q + (p2 & a.rr_mask), idx);
            }
            continue;
        }
        // chunk score = MAT value of the end cell (b_col == r on the last anti-diagonal)
#pragma unroll
        for (int k = 0; k < CPL; k++)
            if (es[k] == ((uint32_t)(r - 1) << SH)) a.out[cid].score = Mv1[k];
        team_sync();
        if (lane == 0 && wt == 0) { __threadfence(); atomicAdd(a.rr_ctl + 2, 1); }
    }
}
