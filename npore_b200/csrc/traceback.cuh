// traceback.cuh -- align() traceback (reference: src/aln.pyx:671-742) over the packed 16-bit records (common.cuh)
// the forward kernel streamed to HBM.  Separate kernel, one walker thread per chunk: pointer chasing that
// jumps RUN cells at a time (MAT-typed runs are diagonal steps re-evaluated as '='/'X' by base compare,
// aln.pyx:727-736).  Ops are emitted right-aligned into the chunk's slice of the item's op scratch
// (a chunk covering anti-diagonals [brk, nxt] emits at most nxt-brk ops) and compacted by finish.cuh.
// Anomalies map to the reference's three checks + unknown type (aln.pyx:689-716, 737-739) as status 1..4;
// the partial op string is kept, as there.
#pragma once
#include "common.cuh"

#define TB_THREADS 128          // 4 warps, one chunk per warp

struct TracebackArgs {
    const ChunkDesc *chunks;
    const ChunkSlot *slots;
    const int32_t *order;
    int n;
    const ItemDesc *items;
    const uint32_t *bits, *cum;
    const uint8_t *ref_codes, *seq_codes;
    const uint16_t *tb;
    uint8_t *ops;                 // op scratch, item regions at ItemDesc::out_off
    ChunkOut *out;
    int r, W, cpl, tbs;           // cpl: cells per lane of the forward instantiation; tbs * 32 = NC = records per anti-diagonal row
    const uint4 *ovf; const int *ovf_cnt; int ovf_cap;    // overflow list of a WIDE forward run (forward.cuh), else null
    int *n_sat;                   // incremented for every chunk that ends in status 8 (api.cu re-runs the batch WIDE)
};

// One warp per chunk: the walk itself is a chain of dependent record loads (every lane reads the same record, a
// broadcast), but each step emits a whole run, which the 32 lanes write (and, for MAT runs, compare) in parallel.
__global__ void __launch_bounds__(TB_THREADS) traceback_kernel(const TracebackArgs a)
{
    const int lane = threadIdx.x & 31;
    const int idx = blockIdx.x * (TB_THREADS / 32) + (threadIdx.x >> 5);
    if (idx >= a.n) return;
    const int cid = a.order[idx];
    const ChunkDesc c = a.chunks[cid];
    if (!c.valid) { if (lane == 0) { ChunkOut o; o.score = 0.f; o.status = 0; o.start = 0; o.len = 0; a.out[cid] = o; } return; }
    const ChunkSlot sl = a.slots[idx];
    const ItemDesc &I = a.items[c.item];
    const uint8_t *__restrict__ refs = a.ref_codes + I.ref_start + min(c.c0, I.ref_len);
    const uint8_t *__restrict__ seqs = a.seq_codes + I.seq_start + min(c.r0, I.seq_len);
    const uint16_t *__restrict__ tb = a.tb + (size_t)sl.tb_off * (32 * a.tbs);
    uint8_t *region = a.ops + I.out_off + c.brk;
    const int cap = c.B - 1, ncm = 32 * a.tbs - 1;
    int pos = cap, i = c.imax, j = c.jmax, status = 0;
    const size_t rs = (size_t)32 * a.tbs;
#define TB_REC(dd, jj) ((dd) >= 0 && (dd) < c.B ? (uint32_t)tb[(size_t)(dd) * rs + ((jj) & ncm)] : 0u)
    while (i > 0 || j > 0) {
        if (i < 0) { status = 1; break; }
        if (j < 0) { status = 2; break; }
        // records are stored per anti-diagonal in slot order: slot = column index mod NC (forward.cuh)
        const int d = i + j;
        const uint32_t rec = TB_REC(d, j);
        const int typ = (int)((rec >> NP_REC_TYP) & 7u);
        int run = (int)(rec & (uint32_t)NP_RUN_SAT);
        if (typ == T_INS) {             // RUN = number of consecutive extensions up the column + 1 (aln.pyx:537-543)
            run = 1;
            uint32_t q = rec; int ii = i;
            while ((q & NP_REC_IE) && ii > 0) { run++; ii--; q = TB_REC(ii + j, j); }
        } else if (typ == T_DEL) {      // likewise along the row (aln.pyx:559-565)
            run = 1;
            uint32_t q = rec; int jj = j;
            while ((q & NP_REC_DE) && jj > 0) { run++; jj--; q = TB_REC(i + jj, jj); }
        } else if ((typ == T_LEN || typ == T_SHR) && run == NP_RUN_SAT) {
            // run field saturated: a WIDE forward run left the true run in the overflow list ({chunk, anti-diagonal, slot, run})
            int found = 0;
            if (a.ovf) {
                const int cnt = min(*a.ovf_cnt, a.ovf_cap);
                for (int e = lane; e < cnt && !found; e += 32) {
                    const uint4 v = a.ovf[e];
                    if (v.x == (uint32_t)cid && v.y == (uint32_t)d && v.z == (uint32_t)(j & ncm)) found = (int)v.w;
                }
                for (int o = 16; o; o >>= 1) found = max(found, __shfl_xor_sync(NP_FULL, found, o));
            }
            if (!found) { status = 8; break; }
            run = found;
        }
        if (run < 1) { status = 3; break; }
        if (typ == T_INS || typ == T_LEN || typ == T_DEL || typ == T_SHR) {
            const uint8_t ch = (typ == T_INS || typ == T_LEN) ? 'I' : 'D';
            const int w = min(run, pos);
            for (int t = lane; t < w; t += 32) region[pos - 1 - t] = ch;
            pos -= w;
            if (ch == 'I') i -= run; else j -= run;
        } else if (typ == T_MAT) {
            const int steps = min(run, min(i, j));                 // cells that exist; a longer run leaves the matrix
            const int w = min(steps, pos);
            for (int t = lane; t < w; t += 32) region[pos - 1 - t] = (refs[j - 1 - t] == seqs[i - 1 - t]) ? '=' : 'X';
            pos -= w;
            if (steps < run) { i -= steps + 1; j -= steps + 1; } else { i -= run; j -= run; }
        } else { status = 4; break; }
    }
#undef TB_REC
    __syncwarp();
    if (lane == 0) {
        ChunkOut o;
        o.score = a.out[cid].score;
        o.status = status; o.start = c.brk + pos; o.len = cap - pos;
        a.out[cid] = o;
        if (status == 8 && a.n_sat) atomicAdd(a.n_sat, 1);
    }
}
