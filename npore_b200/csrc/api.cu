// api.cu -- C ABI of libnpore_b200.so (include/npore_b200.h) and the host side of the GPU batch scheduler that
// replaces the reference's multiprocessing.Pool fan-out (src/realign.py:110-114, src/standardize_vcf.py:30-31).
//
// Pipeline of one batch (all on one stream of one B200):
//   upload   : items / base codes / RLE CIGARs -> HBM
//   run      : plan_* kernels   (aln.pyx:386-392  D/I bit string, rank arrays, chunk descriptors)
//              per sub-batch of chunks, largest first (scratch bounded by the memory budget):
//                annotate_kernel  (aln.pyx:179-251  np-info records of both slices of every chunk)
//                forward_kernel   (aln.pyx:465-667  the recurrence; persistent warps, one chunk per warp)
//                traceback_kernel (aln.pyx:671-742)
//              gather / standardize / rle kernels (aln.pyx:742, bam.pyx:65-78, cig.pyx:13-38)
//   download : per-item op strings, run-length words, chunk scores, status -> host
// The BGZF compressor (npore_bgzf_*, bgzf.cuh) is a separate handle with its own stream: it is not a context, so it does not
// count among the device's live contexts that share the scratch budget.
// There is no CPU fallback: every entry point fails with NPORE_ERR_NO_DEVICE / NPORE_ERR_CUDA without a GPU.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/npore_b200.h"
#include "common.cuh"
#include "plan.cuh"
#include "annotate.cuh"
#include "forward.cuh"
#include "traceback.cuh"
#include "finish.cuh"
#include "confusion.cuh"
#include "bgzf.cuh"
#include "bai.cuh"

namespace {

struct DevBuf {       // device memory owned by its context: freed when the context is deleted
    void *p = nullptr; size_t cap = 0;
    DevBuf &operator=(DevBuf &&) = delete;     // and with it both copies: a block has one owner
    ~DevBuf() { release(); }
    // grow-only; contents are NOT preserved.  The new block is allocated before the old one is released, so a failed growth
    // leaves the buffer usable at its old size; only if both do not fit is the old block given up first.
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        void *q = nullptr;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&q, want);
        if (e != cudaSuccess) { cudaGetLastError(); want = bytes; e = cudaMalloc(&q, want); }
        if (e != cudaSuccess && p) {
            cudaGetLastError();
            cudaFree(p); p = nullptr; cap = 0;
            e = cudaMalloc(&q, want);
        }
        if (e != cudaSuccess) { cudaGetLastError(); return e; }
        if (p) cudaFree(p);
        p = q; cap = want;
        return cudaSuccess;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct HostBuf {      // pinned staging owned by the library (download path)
    void *p = nullptr; size_t cap = 0;
    HostBuf &operator=(HostBuf &&) = delete;   // and with it both copies
    ~HostBuf() { if (p) cudaFreeHost(p); }
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMallocHost(&p, bytes + bytes / 8 + 256);
        if (e == cudaSuccess) cap = bytes + bytes / 8 + 256;
        return e;
    }
};

// pinned block npore_run fills for npore_download: per-item lengths, status, run-length counts; chunk results; counters at the end
struct SmallBlock {
    static size_t bytes(int n, int64_t n_chunks) { return (size_t)n * 12 + (size_t)n_chunks * sizeof(ChunkOut) + 64; }
    int32_t *len, *status, *rle_len; ChunkOut *chunk_out; int *counters;
    SmallBlock(void *base, int n, int64_t n_chunks)
        : len(static_cast<int32_t *>(base)), status(len + n), rle_len(status + n), chunk_out(reinterpret_cast<ChunkOut *>(rle_len + n + (n & 1))),
          counters(reinterpret_cast<int *>(static_cast<char *>(base) + bytes(n, n_chunks) - 16)) {}
};

struct SubBatch { int first, count; };
enum { EV_COPY_BEGIN, EV_COPY_END, EV_PLAN_BEGIN, EV_PLAN_END, EV_FINISH_BEGIN, EV_FINISH_END, N_EVENTS };   // ctx->ev

std::atomic<long long> g_par_inflight[64];  // effective parallelism (forward_team) of the forward launches in flight per device, all contexts
std::atomic<int> g_ctx_on_device[64];      // live contexts per device: they share the scratch budget (PipelinedRealigner)

}  // namespace

struct npore_ctx {
    int device = 0, sm_count = 0;
    std::atomic<int> *on_device = nullptr;           // the device's entries in g_ctx_on_device and g_par_inflight, set
    std::atomic<long long> *par_inflight = nullptr;  // once the context is counted (devices 0-63)
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    AlignParams P{};
    int cpl = 2, tbs = 2;
    size_t scratch_budget = 0;
    DevBuf d_sub, d_np;
    // batch-resident
    DevBuf d_nib, d_nib_start, d_ovf;
    DevBuf d_items, d_ref, d_seq, d_rle, d_grp, d_bits, d_cum, d_chunks, d_chunk_out, d_scratch_ops, d_ops,
        d_item_len, d_item_status, d_rleA, d_rleB, d_rle_len, d_rle_which, d_ops_off, d_rle_off, d_pack_ops, d_pack_rle, d_order, d_slots, d_counter;
    // per sub-batch scratch
    DevBuf d_colrec, d_relaid, d_rowrec, d_raw_ref, d_raw_seq, d_tb, d_rr_q, d_rr_ctl, d_rr_state;
    int rr_slice = 512;
    DevBuf d_chunk_dst, d_part_cnt;
    // npore_confusion_batch staging (kept between calls); npore_get_np_info_batch shares ref_codes, ref_off, raw, ebits and out
    struct {
        DevBuf range_start, range_end, ref_ascii, ref_off, ref_codes, raw, ebits;
        DevBuf read_pos, seq, qual, seq_off, rle, cig_off, g_roff, g_qoff, read_end;
        DevBuf nib_start, has_qual;    // the nibble form's extra arrays (seq then holds the packed bases)
        DevBuf range_reads, range_reads_off, list_maxend, line_of, pos_off;
        DevBuf out;                    // zeroed: the counts, the error flag, the coverage difference array
    } pileup;
    HostBuf h_small;
    std::vector<ItemDesc> items;
    std::vector<int32_t> order, chunk_bmax;
    std::vector<ChunkSlot> slots;
    std::vector<SubBatch> subs;
    int64_t n_chunks = 0, total_ops = 0, total_rle = 0;
    bool uploaded = false, ran = false, budget_fixed = false;
    uint32_t run_flags = 0;
    npore_stats stats{};
    cudaEvent_t ev[N_EVENTS]{};
    std::vector<cudaEvent_t> sub_ev;     // 4 per sub-batch
    std::string err;
};

struct npore_bgzf {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[2]{};
    DevBuf d_in, d_tok, d_slots, d_sizes, d_out, d_total;
    int64_t last_n = 0;                  // input bytes of the last npore_bgzf_compress (still in d_in, its member sizes in d_sizes)
    // npore_bgzf_index
    DevBuf d_rec_off, d_moff, d_recs, d_chunks, d_sorted, d_segs, d_out_chunks, d_out_refs, d_win, d_counts;
    HostBuf h_counts, h_lists;
    ~npore_bgzf()
    {
        for (auto &e : ev) if (e) cudaEventDestroy(e);
        if (stream) cudaStreamDestroy(stream);
    }
};

namespace {

int fail(npore_ctx *c, int code, const char *what, cudaError_t e = cudaSuccess)
{
    if (c) {
        c->err = what;
        if (e != cudaSuccess) { c->err += ": "; c->err += cudaGetErrorString(e); }
    }
    cudaGetLastError();
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? NPORE_ERR_OOM : NPORE_ERR_CUDA, #call, e_); \
    } while (0)

inline int chunks_of(int total, int max_b_rows)
{
    const int step = max_b_rows - 1;
    return total > 0 ? (total + step - 1) / step : 0;
}

template <int CPL, int T, bool WIDE>
int launch_forward(npore_ctx *ctx, const ForwardArgs &fa, int n_sub)
{
    constexpr int WARPS = fwd_warps(CPL, T), TEAMS = WARPS / T;
    // rings (one per team of T warps) are aligned to their size inside the CTA's shared window (cell address = offset | base).
    // The dynamic window starts after the per-CTA reservation and the kernel's static arrays, so the slack needed is known
    // exactly; the kernel re-derives it from the real addresses and raises the error flag instead of running past the window.
    constexpr size_t RING = (size_t)NP_RING * 32 * CPL * T * 16;
    cudaFuncAttributes fattr;
    CU(cudaFuncGetAttributes(&fattr, forward_kernel<CPL, T, WIDE>));
    int reserved = 1024;
    cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, ctx->device);
    const size_t start = (size_t)reserved + fattr.sharedSizeBytes;
    const size_t slack = (RING - start % RING) % RING;
    // + the per-warp column-record FIFOs (1 KB each): inside the slack when it is large enough, else behind the rings
    const size_t smem = (size_t)TEAMS * RING + slack + (slack >= (size_t)WARPS * 1024 ? 0 : (size_t)WARPS * 1024);
    CU(cudaFuncSetAttribute(forward_kernel<CPL, T, WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, forward_kernel<CPL, T, WIDE>, WARPS * 32, smem));
    if (per_sm < 1) per_sm = 1;
    {   // ask for the smallest shared-memory carve-out that holds the resident CTAs: the rest of the 256 KB is L1 for the
        // score-table lookups (the default picked 196 KB where 164 KB is enough, leaving 56 instead of 92 KB of L1)
        const size_t need = (size_t)per_sm * (smem + fattr.sharedSizeBytes + reserved);
        int pct = (int)((need * 100 + 233472 - 1) / 233472);
        if (pct > 100) pct = 100;
        CU(cudaFuncSetAttribute(forward_kernel<CPL, T, WIDE>, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    }
    ctx->stats.fwd_warps_per_sm = per_sm * WARPS;
    if (getenv("NPORE_DEBUG"))
        fprintf(stderr, "[npore] forward_kernel<%d,%d>: %d warps/CTA, %zu B dynamic + %zu B static shared, %d regs, %d CTAs/SM, %d chunks\n", CPL, T, WARPS, smem,
                (size_t)fattr.sharedSizeBytes, fattr.numRegs, per_sm, n_sub);
    int grid = std::min((n_sub + TEAMS - 1) / TEAMS, ctx->sm_count * per_sm);
    if (grid < 1) grid = 1;
    forward_kernel<CPL, T, WIDE><<<grid, WARPS * 32, smem, ctx->stream>>>(fa);
    CU(cudaGetLastError());
    return NPORE_OK;
}

// Which instantiation runs a sub-batch at band slots NC = 32 * nc32: one chunk per warp, or a team of warps per chunk
// (forward.cuh).  Measured on C4 (profiles/r02_ab_experiments.md): NC = 256 runs fastest as four-warp teams <2,4> (126 registers,
// 16 warps/SM; <8,1> needs 255), NC = 128 as two-warp teams <2,2>.  NC = 64: one warp per chunk unless the launch cannot fill the
// warp slots.  A launch whose chunks never wait for a warp takes (longest chunk) x (time per anti-diagonal at that occupancy); one
// whose chunks queue takes (sum of chunk lengths) x (time per anti-diagonal at full occupancy) / slots.  Both forms are estimated
// from the measured per-anti-diagonal times below (profiles/r02_batch_size_sweep.md: us per anti-diagonal of a chunk vs the share
// of the warp slots in use) with par = (sum of chunk lengths) / (longest chunk), and the faster one is taken: teams for C1, for
// batches below ~900 reads, for 50 k-row windows (1,801 chunks of very different lengths); one warp for C5's 1,600 equal chunks.
// Beside other contexts (live on the device, or `others` = the par of their launches in flight: PipelinedRealigner, the file
// pipeline) the one-warp form is the better neighbour -- a 1,000-read batch leaves 60% of the warp slots to the next batch
// instead of 20% -- so teams only while everything in flight together is below a quarter of the slots.
// NPORE_TEAM=1/2/4 forces the choice (tests, A/B).
inline double lerp_tab(const double (*tab)[2], int n, double x)
{
    if (x <= tab[0][0]) return tab[0][1];
    for (int i = 1; i < n; i++)
        if (x <= tab[i][0]) return tab[i - 1][1] + (tab[i][1] - tab[i - 1][1]) * (x - tab[i - 1][0]) / (tab[i][0] - tab[i - 1][0]);
    return tab[n - 1][1];
}

inline int forward_team(const npore_ctx *ctx, int nc32, int n_chunks, double par, double others)
{
    if (nc32 == 1) return 1;
    if (const char *e = getenv("NPORE_TEAM")) { const int t = atoi(e); if (t == 1 || t == 2) return t; if (t == 4) return nc32 == 8 ? 4 : 2; }
    if (nc32 == 8) return 4;
    if (nc32 == 4) return 2;
    const double slots = ctx->sm_count * 16.0;          // resident one-warp chunks of <2,1>
    const bool siblings = ctx->on_device && ctx->on_device->load() > 1;      // a pipeline: the next batch is on its way
    if (others > 0.0 || siblings) return 4.0 * (par + others) <= slots ? 2 : 1;
    // us per anti-diagonal of one chunk (r = 30, 10 kb reads) against the share of the warp slots the launch occupies
    static const double S1[][2] = {{0.04, 0.536}, {0.10, 0.559}, {0.21, 0.582}, {0.32, 0.635}, {0.42, 0.652}, {0.63, 0.750}, {0.84, 0.897}, {1.0, 0.93}};
    static const double S2[][2] = {{0.08, 0.458}, {0.21, 0.476}, {0.42, 0.537}, {0.63, 0.588}, {0.84, 0.663}, {1.0, 0.80}};
    const double t1 = std::max(lerp_tab(S1, 8, std::min(1.0, n_chunks / slots)), par * 0.93 / slots);
    const double t2 = std::max(lerp_tab(S2, 6, std::min(1.0, 2.0 * n_chunks / slots)), par * 0.60 / (0.5 * slots));
    return t2 < t1 ? 2 : 1;
}

// BAM 4-bit bases -> base codes (cig.pyx:212-229 on the device): grid (items, parts)
__global__ void unpack_nib_kernel(const ItemDesc *items, const uint8_t *nib, const int64_t *nib_start, uint8_t *codes, int parts)
{
    const ItemDesc &I = items[blockIdx.x];
    int lo, hi;
    np_slice(I.seq_len, parts, blockIdx.y, lo, hi);
    const int64_t ns = nib_start[blockIdx.x];
    uint8_t *out = codes + I.seq_start;
    for (int t = lo + threadIdx.x; t < hi; t += blockDim.x) {
        const int64_t k = ns + t;
        const uint32_t b = nib[k >> 1];
        const uint32_t v = (k & 1) ? (b & 15u) : (b >> 4);
        out[t] = v == 1u ? 1 : v == 2u ? 2 : v == 4u ? 3 : v == 8u ? 4 : 0;      // "=ACMGRSVTWYHKDBN": A=1 C=2 G=4 T=8
    }
}

struct InFlight {    // this pass's entry in par_inflight: set per sub-batch, withdrawn when the pass has synchronised (or failed)
    std::atomic<long long> *g; long long mine = 0;
    long long set(long long par) { const long long before = g ? g->fetch_add(par - mine) : mine; const long long o = before - mine; mine = par; return o > 0 ? o : 0; }
    ~InFlight() { if (g && mine) g->fetch_sub(mine); }
};

// Sub-batches: greedy over `order` under the scratch budget (sizes from the host-side upper bounds).  The budget is this
// context's share of the device (contexts on one device run side by side: PipelinedRealigner); if the scratch still does not
// fit (other tenants of the device), the batch is re-cut with half the budget instead of failing.  *rr_cap: run-queue capacity.
int cut_sub_batches(npore_ctx *ctx, int *rr_cap)
{
    const int64_t nchunks = ctx->n_chunks;
    size_t budget = ctx->scratch_budget;
    if (!ctx->budget_fixed && ctx->on_device) budget /= (size_t)std::max(1, ctx->on_device->load());
    for (int attempt = 0;; attempt++) {
        ctx->slots.assign(nchunks, ChunkSlot{});
        ctx->subs.clear();
        size_t max_col = 0, max_row = 0, max_tb = 0;
        const size_t per_entry = 32 + 8 + 8 + 4 + 8;   // colrec, relaid, raw_ref, rowrec, raw_seq
        size_t col = 0, row = 0, tb = 0; int first = 0;
        for (int64_t k = 0; k < nchunks; k++) {
            const int bm = ctx->chunk_bmax[ctx->order[k]];
            const size_t ent = (size_t)((bm + 32 * ctx->cpl + 128 + 31) & ~31);
            const size_t need = (col + ent) * per_entry + (tb + bm) * (size_t)(64 * ctx->tbs);
            if (k > first && need > budget) {
                ctx->subs.push_back({first, (int)(k - first)});
                max_col = std::max(max_col, col); max_row = std::max(max_row, row); max_tb = std::max(max_tb, tb);
                col = row = tb = 0; first = (int)k;
            }
            ChunkSlot &sl = ctx->slots[k];
            sl.col_off = (int64_t)col; sl.row_off = (int64_t)row; sl.tb_off = (int64_t)tb;
            sl.col_cap = sl.row_cap = (int32_t)ent;
            col += ent; row += ent; tb += bm;
        }
        if (nchunks > first) {
            ctx->subs.push_back({first, (int)(nchunks - first)});
            max_col = std::max(max_col, col); max_row = std::max(max_row, row); max_tb = std::max(max_tb, tb);
        }
        cudaError_t e = ctx->d_colrec.ensure(max_col * 32 + 64);
        if (e == cudaSuccess) e = ctx->d_relaid.ensure(max_col * 8 + 64);
        if (e == cudaSuccess) e = ctx->d_raw_ref.ensure(max_col * 8 + 64);
        if (e == cudaSuccess) e = ctx->d_rowrec.ensure(max_row * 4 + 64);
        if (e == cudaSuccess) e = ctx->d_raw_seq.ensure(max_row * 8 + 64);
        if (e == cudaSuccess) e = ctx->d_tb.ensure(max_tb * (size_t)(64 * ctx->tbs) + 256);
        if (e == cudaSuccess) break;
        cudaGetLastError();
        if (e != cudaErrorMemoryAllocation || attempt >= 4 || ctx->subs.size() >= (size_t)std::max<int64_t>(nchunks, 1))
            return fail(ctx, e == cudaErrorMemoryAllocation ? NPORE_ERR_OOM : NPORE_ERR_CUDA, "scratch allocation", e);
        ctx->d_tb.release(); ctx->d_colrec.release();          // give back what the failed attempt may have grabbed
        budget /= 2;
    }
    int max_sub = 1;
    for (const SubBatch &sb : ctx->subs) max_sub = std::max(max_sub, sb.count);
    *rr_cap = 1;
    while (*rr_cap < 2 * max_sub + 16384) *rr_cap <<= 1;
    CU(ctx->d_rr_q.ensure(sizeof(int) * (size_t)*rr_cap));
    CU(ctx->d_rr_ctl.ensure(64));
    CU(ctx->d_rr_state.ensure(sizeof(uint32_t) * fwd_rr_state_words(ctx->cpl) * (size_t)max_sub));
    while (ctx->sub_ev.size() < 4 * ctx->subs.size()) {
        cudaEvent_t e; CU(cudaEventCreate(&e)); ctx->sub_ev.push_back(e);
    }
    if (nchunks) CU(cudaMemcpyAsync(ctx->d_slots.p, ctx->slots.data(), sizeof(ChunkSlot) * (size_t)nchunks, cudaMemcpyHostToDevice, ctx->stream));
    return NPORE_OK;
}

int launch_forward_for(npore_ctx *ctx, int team, bool wide, const ForwardArgs &fa, int n)
{
    switch (ctx->cpl * 100 + team * 10 + (wide ? 1 : 0)) {      // digits: cpl, team, WIDE (the second pass: forward.cuh)
    case 110: return launch_forward<1, 1, false>(ctx, fa, n);
    case 210: return launch_forward<2, 1, false>(ctx, fa, n);
    case 220: return launch_forward<1, 2, false>(ctx, fa, n);
    case 410: return launch_forward<4, 1, false>(ctx, fa, n);
    case 420: return launch_forward<2, 2, false>(ctx, fa, n);
    case 810: return launch_forward<8, 1, false>(ctx, fa, n);
    case 820: return launch_forward<4, 2, false>(ctx, fa, n);
    case 840: return launch_forward<2, 4, false>(ctx, fa, n);
    case 111: return launch_forward<1, 1, true>(ctx, fa, n);
    case 211: return launch_forward<2, 1, true>(ctx, fa, n);
    case 221: return launch_forward<1, 2, true>(ctx, fa, n);
    case 411: return launch_forward<4, 1, true>(ctx, fa, n);
    case 421: return launch_forward<2, 2, true>(ctx, fa, n);
    case 821: return launch_forward<4, 2, true>(ctx, fa, n);
    case 811:                                      // <8, 1, true> is not instantiated: W > 128 runs as teams of four
    case 841:                                      // forward_team yields no other pair: the last case takes the rest
    default: return launch_forward<2, 4, true>(ctx, fa, n);
    }
}

int run_sub_batch(npore_ctx *ctx, size_t si, bool wide, int rr_cap, InFlight &inflight)
{
    const SubBatch &sb = ctx->subs[si];
    cudaEvent_t *ev = &ctx->sub_ev[4 * si];          // annotate, forward and traceback each run between two of them
    AnnotateArgs aa{};
    aa.chunks = ctx->d_chunks.as<ChunkDesc>(); aa.slots = ctx->d_slots.as<ChunkSlot>() + sb.first;
    aa.order = ctx->d_order.as<int32_t>() + sb.first; aa.n = sb.count; aa.items = ctx->d_items.as<ItemDesc>();
    aa.ref_codes = ctx->d_ref.as<uint8_t>(); aa.seq_codes = ctx->d_seq.as<uint8_t>();
    aa.raw_ref = ctx->d_raw_ref.as<uint8_t>(); aa.raw_seq = ctx->d_raw_seq.as<uint8_t>();
    aa.colrec = ctx->d_colrec.as<uint4>(); aa.relaid = ctx->d_relaid.as<uint2>(); aa.rowrec = ctx->d_rowrec.as<uint32_t>();
    aa.max_n = ctx->P.max_n; aa.max_l = ctx->P.max_l; aa.nc = 32 * ctx->cpl; aa.inf_row = ctx->P.np_rows;
    int bm = 1;
    double bsum = 0.0;
    for (int k = 0; k < sb.count; k++) { const int b = ctx->chunk_bmax[ctx->order[sb.first + k]]; bm = std::max(bm, b); bsum += b; }
    const long long par = (long long)(bsum / bm) + 1;
    const long long others = inflight.set(par);                  // the other contexts' launches on this device
    const int team = forward_team(ctx, ctx->cpl, sb.count, (double)par, (double)others);      // warps per chunk of this sub-batch's forward launch
    aa.cpl = ctx->cpl / team;
    CU(cudaEventRecord(ev[0], ctx->stream));
    {   // equality words of all periods in dynamic shared memory: 6 planes of (longest slice / 32 + 2) words
        aa.e6_stride = (bm + 1 + 31) / 32 + 2;
        const size_t dyn = (size_t)NP_MAXN * aa.e6_stride * sizeof(uint32_t);
        if (dyn > 48 * 1024) CU(cudaFuncSetAttribute(annotate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        annotate_kernel<<<2 * sb.count, ANN_THREADS, dyn, ctx->stream>>>(aa);
    }
    CU(cudaGetLastError()); ctx->stats.launches++;
    CU(cudaEventRecord(ev[1], ctx->stream));

    ForwardArgs fa{};
    fa.chunks = aa.chunks; fa.slots = aa.slots; fa.order = aa.order; fa.n = sb.count;
    fa.items = aa.items; fa.bits = ctx->d_bits.as<uint32_t>(); fa.err = ctx->d_counter.as<int>();
    fa.ovf = wide ? ctx->d_ovf.as<uint4>() : nullptr; fa.ovf_cap = 65536; fa.ovf_cnt = ctx->d_counter.as<int>() + 1;
    fa.ref_codes = aa.ref_codes; fa.seq_codes = aa.seq_codes; fa.colrec = aa.colrec; fa.relaid = aa.relaid; fa.rowrec = aa.rowrec;
    fa.tb = ctx->d_tb.as<uint16_t>(); fa.tab = ctx->d_np.as<float>(); fa.sub_tab = ctx->d_sub.as<float>();
    fa.out = ctx->d_chunk_out.as<ChunkOut>();
    fa.P = ctx->P;
    fa.rr_q = ctx->d_rr_q.as<int>(); fa.rr_mask = rr_cap - 1; fa.rr_ctl = ctx->d_rr_ctl.as<int>();
    fa.rr_state = ctx->d_rr_state.as<uint32_t>(); fa.rr_slice = ctx->rr_slice;
    CU(cudaMemsetAsync(ctx->d_rr_state.p, 0, sizeof(uint32_t) * fwd_rr_state_words(ctx->cpl) * (size_t)sb.count, ctx->stream));
    rr_init_kernel<<<64, 256, 0, ctx->stream>>>(fa.rr_q, rr_cap, sb.count, fa.rr_ctl);
    CU(cudaGetLastError()); ctx->stats.launches++;
    if (int rc = launch_forward_for(ctx, team, wide, fa, sb.count); rc != NPORE_OK) return rc;
    ctx->stats.launches++;
    CU(cudaEventRecord(ev[2], ctx->stream));

    TracebackArgs ta{};
    ta.chunks = aa.chunks; ta.slots = aa.slots; ta.order = aa.order; ta.n = sb.count; ta.items = aa.items;
    ta.bits = fa.bits; ta.cum = ctx->d_cum.as<uint32_t>(); ta.ref_codes = aa.ref_codes; ta.seq_codes = aa.seq_codes;
    ta.tb = fa.tb; ta.ops = ctx->d_scratch_ops.as<uint8_t>(); ta.out = fa.out;
    ta.r = ctx->P.r; ta.W = ctx->P.W; ta.cpl = ctx->cpl; ta.tbs = ctx->tbs;
    ta.ovf = fa.ovf; ta.ovf_cnt = fa.ovf_cnt; ta.ovf_cap = fa.ovf_cap; ta.n_sat = ctx->d_counter.as<int>() + 2;
    traceback_kernel<<<(sb.count + TB_THREADS / 32 - 1) / (TB_THREADS / 32), TB_THREADS, 0, ctx->stream>>>(ta);
    CU(cudaGetLastError()); ctx->stats.launches++;
    CU(cudaEventRecord(ev[3], ctx->stream));
    for (int k = 0; k < sb.count; k++) ctx->stats.tb_bytes += (int64_t)ctx->chunk_bmax[ctx->order[sb.first + k]] * 64 * ctx->tbs;
    return NPORE_OK;
}

// the finish kernels; per-item sizes / status / chunk results and the counters travel with the run (npore_download knows exact sizes)
int launch_finish(npore_ctx *ctx, uint32_t flags, int parts, int max_ops)
{
    const int n = (int)ctx->items.size();
    npore_stats &S = ctx->stats;
    const bool want_ops = !(flags & NPORE_OUT_NO_EXPANDED), want_rle = (flags & NPORE_OUT_RLE) != 0;
    CU(cudaEventRecord(ctx->ev[EV_FINISH_BEGIN], ctx->stream));
    CU(ctx->h_small.ensure(SmallBlock::bytes(n, ctx->n_chunks)));
    const SmallBlock hs(ctx->h_small.p, n, ctx->n_chunks);
    if (n) {
        FinishArgs fa{};
        fa.items = ctx->d_items.as<ItemDesc>(); fa.n_items = n; fa.chunk_out = ctx->d_chunk_out.as<ChunkOut>();
        fa.scratch = ctx->d_scratch_ops.as<uint8_t>(); fa.ops = ctx->d_ops.as<uint8_t>();
        fa.item_len = ctx->d_item_len.as<int32_t>(); fa.item_status = ctx->d_item_status.as<int32_t>();
        fa.ref_codes = ctx->d_ref.as<uint8_t>(); fa.seq_codes = ctx->d_seq.as<uint8_t>();
        fa.rleA = ctx->d_rleA.as<uint32_t>(); fa.rleB = ctx->d_rleB.as<uint32_t>();
        fa.rle_len = ctx->d_rle_len.as<int32_t>(); fa.rle_which = ctx->d_rle_which.as<int32_t>();
        fa.to_m = (flags & NPORE_OUT_STANDARDIZE) ? 1 : 0;
        fa.ops_off = ctx->d_ops_off.as<int64_t>(); fa.rle_off = ctx->d_rle_off.as<int64_t>();
        fa.pack_ops = ctx->d_pack_ops.as<uint8_t>(); fa.pack_rle = ctx->d_pack_rle.as<uint32_t>();
        CU(ctx->d_chunk_dst.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(ctx->n_chunks, 1)));
        fa.chunks = ctx->d_chunks.as<ChunkDesc>(); fa.n_chunks = (int)ctx->n_chunks;
        fa.chunk_dst = ctx->d_chunk_dst.as<int32_t>(); fa.parts = parts; fa.part_cnt = ctx->d_part_cnt.as<int32_t>();
        const dim3 grid_np(n, parts);
        item_len_kernel<<<n, FIN_THREADS, 0, ctx->stream>>>(fa);
        CU(cudaGetLastError()); S.launches++;
        if (ctx->n_chunks) {
            gather_kernel<<<(unsigned)ctx->n_chunks, FIN_THREADS, 0, ctx->stream>>>(fa);
            CU(cudaGetLastError()); S.launches++;
        }
        if (flags & (NPORE_OUT_RLE | NPORE_OUT_STANDARDIZE)) {
            if (parts > 1) { rle_count_kernel<<<grid_np, FIN_WIDE, 0, ctx->stream>>>(fa); S.launches++; }
            rle_start_kernel<<<grid_np, FIN_WIDE, 0, ctx->stream>>>(fa);
            rle_word_kernel<<<grid_np, FIN_WIDE, 0, ctx->stream>>>(fa);
            CU(cudaGetLastError()); S.launches += 2;
        } else CU(cudaMemsetAsync(ctx->d_rle_len.p, 0, sizeof(int32_t) * (size_t)n, ctx->stream));
        if (flags & NPORE_OUT_STANDARDIZE) {
            // items with many run-length groups (haplotypes) get a whole CTA each; NPORE_STD_LONG_MIN overrides the split (tests)
            int long_min = 4096;
            if (const char *e = getenv("NPORE_STD_LONG_MIN")) long_min = std::max(1, atoi(e));
            const bool any_long = max_ops >= long_min;              // an item cannot have more groups than ops
            // the long-item kernel goes first and marks its items (rle_which = 1); the per-warp kernel takes what is left.
            // (Both look at the group count BEFORE standardisation: the sweeps change it.)
            if (any_long) {
                standardize_long_kernel<<<n, FIN_WIDE, 0, ctx->stream>>>(fa, long_min);
                CU(cudaGetLastError()); S.launches++;
            }
            standardize_kernel<<<(n + FIN_THREADS / 32 - 1) / (FIN_THREADS / 32), FIN_THREADS, 0, ctx->stream>>>(fa);
            CU(cudaGetLastError()); S.launches++;
            if (want_ops) {
                if (parts > 1) { expand_count_kernel<<<grid_np, FIN_WIDE, 0, ctx->stream>>>(fa); S.launches++; }
                expand_fill_kernel<<<grid_np, FIN_WIDE, 0, ctx->stream>>>(fa);
                CU(cudaGetLastError()); S.launches++;
            }
        }
        scan_kernel<<<1, 1024, 0, ctx->stream>>>(fa);
        CU(cudaGetLastError()); S.launches++;
        if (want_ops || want_rle) {
            pack_kernel<<<grid_np, FIN_WIDE, 0, ctx->stream>>>(fa, want_ops ? 1 : 0, want_rle ? 1 : 0);
            CU(cudaGetLastError()); S.launches++;
        }
        CU(cudaMemcpyAsync(hs.len, ctx->d_item_len.p, 4 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(hs.status, ctx->d_item_status.p, 4 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(hs.rle_len, ctx->d_rle_len.p, 4 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
        if (ctx->n_chunks) CU(cudaMemcpyAsync(hs.chunk_out, ctx->d_chunk_out.p, sizeof(ChunkOut) * (size_t)ctx->n_chunks, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaMemcpyAsync(hs.counters, ctx->d_counter.p, 12, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaEventRecord(ctx->ev[EV_FINISH_END], ctx->stream));
    return NPORE_OK;
}

int run_pass(npore_ctx *ctx, uint32_t flags, bool wide, int *n_sat)
{
    CU(cudaSetDevice(ctx->device));
    ctx->ran = false;
    InFlight inflight{ctx->par_inflight};
    const int n = (int)ctx->items.size();
    npore_stats &S = ctx->stats;
    S.launches = 0; S.tb_bytes = 0;
    ctx->run_flags = flags;
    if (flags & (NPORE_OUT_RLE | NPORE_OUT_STANDARDIZE))
        for (DevBuf *d : {&ctx->d_rleA, &ctx->d_rleB}) CU(d->ensure(sizeof(uint32_t) * (size_t)(ctx->total_ops + 64)));
    if (!(flags & NPORE_OUT_NO_EXPANDED)) CU(ctx->d_pack_ops.ensure((size_t)ctx->total_ops + 64));
    if (flags & NPORE_OUT_RLE) CU(ctx->d_pack_rle.ensure(sizeof(uint32_t) * (size_t)(ctx->total_ops + 64)));
    int rr_cap = 1, rc = cut_sub_batches(ctx, &rr_cap);
    if (rc != NPORE_OK) return rc;
    CU(cudaMemsetAsync(ctx->d_counter.p, 0, 16, ctx->stream));     // [0] forward-kernel error flag  [1] overflow records  [2] saturated chunks
    if (wide) CU(ctx->d_ovf.ensure(sizeof(uint4) * 65536));
    CU(cudaEventRecord(ctx->ev[EV_PLAN_BEGIN], ctx->stream));
    int max_ops = 1;
    for (const ItemDesc &I : ctx->items) max_ops = std::max(max_ops, I.total_ops);
    const int parts = std::min(FIN_MAX_PARTS, (max_ops + 32767) / 32768);     // slices per item for the per-item kernels
    if (n) {
        CU(ctx->d_part_cnt.ensure(sizeof(int32_t) * (size_t)n * parts));
        PlanArgs pa{};
        pa.items = ctx->d_items.as<ItemDesc>(); pa.n_items = n; pa.rle = ctx->d_rle.as<uint32_t>(); pa.grp_off = ctx->d_grp.as<int32_t>();
        pa.bits = ctx->d_bits.as<uint32_t>(); pa.cum = ctx->d_cum.as<uint32_t>(); pa.chunks = ctx->d_chunks.as<ChunkDesc>();
        pa.max_b_rows = ctx->P.max_b_rows; pa.parts = parts; pa.part_cnt = ctx->d_part_cnt.as<int32_t>();
        const dim3 grid_np(n, parts);
        plan_groups_kernel<<<n, PLAN_THREADS, 0, ctx->stream>>>(pa);
        plan_bits_kernel<<<grid_np, PLAN_THREADS, 0, ctx->stream>>>(pa);
        plan_cum_kernel<<<grid_np, PLAN_THREADS, 0, ctx->stream>>>(pa);
        plan_chunks_kernel<<<grid_np, PLAN_THREADS, 0, ctx->stream>>>(pa);
        CU(cudaGetLastError()); S.launches += 4;
    }
    CU(cudaEventRecord(ctx->ev[EV_PLAN_END], ctx->stream));
    for (size_t si = 0; si < ctx->subs.size(); si++)
        if ((rc = run_sub_batch(ctx, si, wide, rr_cap, inflight)) != NPORE_OK) return rc;
    if ((rc = launch_finish(ctx, flags, parts, max_ops)) != NPORE_OK) return rc;
    CU(cudaStreamSynchronize(ctx->stream));
    const int *counters = SmallBlock(ctx->h_small.p, n, ctx->n_chunks).counters;
    if (counters[0]) return fail(ctx, NPORE_ERR_CUDA, "forward kernel: shared-memory window smaller than the history rings");
    *n_sat = counters[2];
    float ms[3] = {0, 0, 0}, t;                       // annotate, forward, traceback
    for (size_t si = 0; si < ctx->subs.size(); si++)
        for (int k = 0; k < 3; k++) { cudaEventElapsedTime(&t, ctx->sub_ev[4 * si + k], ctx->sub_ev[4 * si + k + 1]); ms[k] += t; }
    cudaEventElapsedTime(&S.ms_plan, ctx->ev[EV_PLAN_BEGIN], ctx->ev[EV_PLAN_END]);
    cudaEventElapsedTime(&S.ms_finish, ctx->ev[EV_FINISH_BEGIN], ctx->ev[EV_FINISH_END]);
    cudaEventElapsedTime(&S.ms_kernels_total, ctx->ev[EV_PLAN_BEGIN], ctx->ev[EV_FINISH_END]);
    S.ms_annotate = ms[0]; S.ms_forward = ms[1]; S.ms_traceback = ms[2];
    S.n_sub_batches = (int)ctx->subs.size();
    ctx->ran = true;
    return NPORE_OK;
}

}  // namespace

extern "C" {

const char *npore_version(void) { return "npore_b200 0.1.0 (sm_100a)"; }

const char *npore_strerror(int code)
{
    switch (code) {
    case NPORE_OK: return "ok";
    case NPORE_ERR_BAD_ARG: return "bad argument";
    case NPORE_ERR_CUDA: return "CUDA error";
    case NPORE_ERR_OOM: return "out of device memory";
    case NPORE_ERR_NO_DEVICE: return "no CUDA device";
    case NPORE_ERR_STATE: return "call out of order (upload -> run -> download)";
    case NPORE_ERR_CAPACITY: return "caller buffer too small";
    default: return "unknown error";
    }
}

const char *npore_last_error(const npore_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int npore_ctx_create(npore_ctx **out, int device, const float *sub_scores, const float *np_scores, int np_n,
                     int np_dim, int max_n, int max_l, float indel_start, float indel_extend, int max_b_rows, int r)
{
    if (!out) return NPORE_ERR_BAD_ARG;
    *out = nullptr;
    if (!sub_scores || !np_scores) return NPORE_ERR_BAD_ARG;
    if (max_n < 0 || max_n > NP_MAXN || max_n > np_n) return NPORE_ERR_BAD_ARG;
    if (max_l < 1 || max_l > 127 || np_dim < max_l) return NPORE_ERR_BAD_ARG;   // L must fit 7 bits; index clamp is max_l-1
    if (max_b_rows < 2 || max_b_rows > 65000) return NPORE_ERR_BAD_ARG;          // runs are carried in 16 bits
    if (r < 1 || 2 * r + 1 > 32 * 8) return NPORE_ERR_BAD_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return NPORE_ERR_NO_DEVICE; }
    if (device < 0 || device >= ndev) return NPORE_ERR_BAD_ARG;
    npore_ctx *ctx = new npore_ctx();
    ctx->device = device;
    auto bail = [&](int code) { npore_ctx_destroy(ctx); return code; };
    if (cudaSetDevice(device) != cudaSuccess) return bail(NPORE_ERR_CUDA);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(NPORE_ERR_CUDA);
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(NPORE_ERR_CUDA);
    for (auto &e : ctx->ev) if (cudaEventCreate(&e) != cudaSuccess) return bail(NPORE_ERR_CUDA);
    ctx->P.r = r; ctx->P.W = 2 * r + 1; ctx->P.max_n = max_n; ctx->P.max_l = max_l; ctx->P.max_b_rows = max_b_rows;
    ctx->P.np_dim = np_dim; ctx->P.np_clamp = max_l - 1; ctx->P.np_rows = max_n * (max_l + 1);
    ctx->P.gap_open = indel_start; ctx->P.gap_ext = indel_extend;
    const int W = 2 * r + 1;
    ctx->cpl = W <= 32 ? 1 : W <= 64 ? 2 : W <= 128 ? 4 : 8;
    ctx->tbs = np_tbs(ctx->cpl);
    if (ctx->d_sub.ensure(25 * sizeof(float)) != cudaSuccess) return bail(NPORE_ERR_OOM);
    // score tables re-laid per (period n, tract length L) so that a candidate is one load (forward.cuh): row (n-1)*(max_l+1)+L,
    //   tabS[row][q] = np_score(n, L, -(q+1))   (SHR after q = trunc(run/n) units already removed)
    //   tabL[row][q] = np_score(n, L, +(q+1))   (LEN likewise)
    // (q up to the saturated run NP_RUN_SAT < NP_TABQ, so the kernel never clamps it) with np_score exactly as the reference CALLS it (aln.pyx:257-274 with max_l in the max_n slot, :615): 100.0 if
    // L + indel < 0, else np_scores[n-1][min(L, max_l-1)][min(L + indel, max_l-1)].  Row `rows` is all +INF ("no candidate").
    {
        const int rows = max_n * (max_l + 1), clampv = max_l - 1;
        std::vector<float> tab((size_t)2 * (rows + 1) * NP_TABQ, __builtin_inff());
        for (int sgn = 0; sgn < 2; sgn++)
            for (int n = 1; n <= max_n; n++)
                for (int L = 0; L <= max_l; L++)
                    for (int q = 0; q < NP_TABQ; q++) {
                        const int call = sgn ? L + q + 1 : L - q - 1;
                        float v = 100.0f;
                        if (call >= 0) v = np_scores[((size_t)(n - 1) * np_dim + std::min(L, clampv)) * np_dim + std::min(call, clampv)];
                        tab[((size_t)sgn * NP_TABQ + q) * (rows + 1) + (size_t)(n - 1) * (max_l + 1) + L] = v;      // q-major: the hot q = 0, 1, 2 of ALL rows share a few cache lines
                    }
        if (ctx->d_np.ensure(tab.size() * sizeof(float)) != cudaSuccess) return bail(NPORE_ERR_OOM);
        if (cudaMemcpy(ctx->d_np.p, tab.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) return bail(NPORE_ERR_CUDA);
    }
    if (cudaMemcpy(ctx->d_sub.p, sub_scores, 25 * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) return bail(NPORE_ERR_CUDA);
    if (ctx->d_counter.ensure(64) != cudaSuccess) return bail(NPORE_ERR_OOM);
    size_t fr = 0, tot = 0;
    cudaMemGetInfo(&fr, &tot);
    if (cudaGetLastError() != cudaSuccess) return bail(NPORE_ERR_CUDA);
    ctx->scratch_budget = (size_t)((double)fr * 0.55);          // divided by the device's live contexts at run time
    if (device < 64) { ctx->on_device = &g_ctx_on_device[device]; ctx->par_inflight = &g_par_inflight[device]; }
    if (ctx->on_device) (*ctx->on_device)++;
    if (const char *s = getenv("NPORE_SCRATCH_MB")) { ctx->scratch_budget = (size_t)atoll(s) << 20; ctx->budget_fixed = true; }
    if (const char *s = getenv("NPORE_RR_SLICE")) ctx->rr_slice = std::max(8, atoi(s));
    *out = ctx;
    return NPORE_OK;
}

void npore_ctx_destroy(npore_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->on_device) (*ctx->on_device)--;
    for (auto &e : ctx->ev) if (e) cudaEventDestroy(e);
    for (auto &e : ctx->sub_ev) cudaEventDestroy(e);
    if (ctx->stream && ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;                          // frees the buffers, on the device set above
}

int npore_set_stream(npore_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return NPORE_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->stream && ctx->own_stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    return NPORE_OK;
}

int64_t npore_count_chunks(const npore_ctx *ctx, int32_t n_items, const int32_t *ref_len, const int32_t *seq_len)
{
    if (!ctx || n_items < 0 || (n_items && (!ref_len || !seq_len))) return NPORE_ERR_BAD_ARG;
    int64_t n = 0;
    for (int i = 0; i < n_items; i++) n += chunks_of(ref_len[i] + seq_len[i], ctx->P.max_b_rows);
    return n;
}

int npore_upload(npore_ctx *ctx, const npore_batch *b)
{
    if (!ctx || !b || b->n_items < 0) return NPORE_ERR_BAD_ARG;
    const int n = b->n_items;
    const bool packed_seq = b->seq_nib != nullptr;
    if (n && (!b->ref_start || !b->ref_len || !b->seq_len || !b->cigar_off || (packed_seq ? !b->seq_nib_start : !b->seq_start)))
        return fail(ctx, NPORE_ERR_BAD_ARG, "null batch array");
    CU(cudaSetDevice(ctx->device));
    ctx->uploaded = ctx->ran = false;
    ctx->items.assign(n, ItemDesc{});
    int64_t out_off = 0, words = 0, nchunks = 0, n_cu = 0, seq_run = 0, max_seq = 1;
    for (int i = 0; i < n; i++) {
        ItemDesc &I = ctx->items[i];
        const int64_t rl = b->ref_len[i], sl = b->seq_len[i];
        if (rl < 0 || sl < 0 || rl + sl >= (1ll << 28)) return fail(ctx, NPORE_ERR_BAD_ARG, "item too long (ref_len + seq_len must be < 2^28)");
        if (b->ref_start[i] < 0 || b->ref_start[i] + rl > b->ref_total) return fail(ctx, NPORE_ERR_BAD_ARG, "sequence range outside buffer");
        if (packed_seq) {
            if (b->seq_nib_start[i] < 0 || b->seq_nib_start[i] + sl > 2 * b->seq_nib_bytes) return fail(ctx, NPORE_ERR_BAD_ARG, "packed read outside buffer");
        } else if (b->seq_start[i] < 0 || b->seq_start[i] + sl > b->seq_total) return fail(ctx, NPORE_ERR_BAD_ARG, "sequence range outside buffer");
        const int64_t cn = b->cigar_off[i + 1] - b->cigar_off[i];
        if (cn < 0 || cn > 0x7ffffff0ll) return fail(ctx, NPORE_ERR_BAD_ARG, "bad cigar_off");
        I.ref_start = b->ref_start[i]; I.seq_start = packed_seq ? seq_run : b->seq_start[i];
        seq_run += sl;
        I.ref_len = (int32_t)rl; I.seq_len = (int32_t)sl;
        I.cig_off = b->cigar_off[i] - b->cigar_off[0]; I.cig_n = (int32_t)cn;
        I.total_ops = (int32_t)(rl + sl);
        max_seq = std::max<int64_t>(max_seq, sl);
        I.bit_word_off = words; words += (I.total_ops >> 5) + 2;
        I.out_off = out_off; out_off += (I.total_ops + 3) & ~3;      // keep item regions 4-byte aligned
        I.n_chunks = chunks_of(I.total_ops, ctx->P.max_b_rows);
        if (nchunks + I.n_chunks > 0x7ffffff0ll) return fail(ctx, NPORE_ERR_BAD_ARG, "too many chunks");
        I.chunk_first = (int32_t)nchunks; nchunks += I.n_chunks;
        n_cu += ((int64_t)I.total_ops + I.n_chunks) * ctx->P.W;
        I.status = 0;
    }
    ctx->n_chunks = nchunks; ctx->total_ops = out_off;
    ctx->total_rle = n ? b->cigar_off[n] - b->cigar_off[0] : 0;

    // chunk size upper bounds (exact B needs the break shift computed on device) and processing order
    const int step = ctx->P.max_b_rows - 1;
    ctx->chunk_bmax.resize(nchunks);
    ctx->order.resize(nchunks);
    std::vector<int32_t> partial;
    int64_t w = 0;
    for (int i = 0; i < n; i++) {
        const ItemDesc &I = ctx->items[i];
        for (int k = 0; k < I.n_chunks; k++) {
            const int cid = I.chunk_first + k;
            const bool last = (k + 1 == I.n_chunks);
            ctx->chunk_bmax[cid] = last ? (I.total_ops - k * step + 2) : (step + 2);
            if (!last) ctx->order[w++] = cid; else partial.push_back(cid);
        }
    }
    std::sort(partial.begin(), partial.end(), [&](int32_t x, int32_t y) {
        return ctx->chunk_bmax[x] != ctx->chunk_bmax[y] ? ctx->chunk_bmax[x] > ctx->chunk_bmax[y] : x < y; });
    // full chunks first unless some final chunk is longer than a full one (never: bmax(last) <= step + 2)
    for (int32_t cid : partial) ctx->order[w++] = cid;

    // device buffers
    CU(ctx->d_items.ensure(sizeof(ItemDesc) * (size_t)std::max(n, 1)));
    CU(ctx->d_ref.ensure((size_t)b->ref_total + 64));
    const int64_t seq_total = packed_seq ? seq_run : b->seq_total;
    CU(ctx->d_seq.ensure((size_t)seq_total + 64));
    if (packed_seq) {
        CU(ctx->d_nib.ensure((size_t)b->seq_nib_bytes + 64));
        CU(ctx->d_nib_start.ensure(sizeof(int64_t) * (size_t)std::max(n, 1)));
    }
    CU(ctx->d_rle.ensure(sizeof(uint32_t) * (size_t)(ctx->total_rle + 1)));
    CU(ctx->d_grp.ensure(sizeof(int32_t) * (size_t)(ctx->total_rle + n + 1)));
    for (DevBuf *d : {&ctx->d_bits, &ctx->d_cum}) CU(d->ensure(sizeof(uint32_t) * (size_t)(words + 128)));
    CU(ctx->d_chunks.ensure(sizeof(ChunkDesc) * (size_t)std::max<int64_t>(nchunks, 1)));
    CU(ctx->d_chunk_out.ensure(sizeof(ChunkOut) * (size_t)std::max<int64_t>(nchunks, 1)));
    CU(ctx->d_order.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(nchunks, 1)));
    CU(ctx->d_slots.ensure(sizeof(ChunkSlot) * (size_t)std::max<int64_t>(nchunks, 1)));
    for (DevBuf *d : {&ctx->d_scratch_ops, &ctx->d_ops}) CU(d->ensure((size_t)out_off + 64));
    for (DevBuf *d : {&ctx->d_item_len, &ctx->d_item_status, &ctx->d_rle_len, &ctx->d_rle_which}) CU(d->ensure(sizeof(int32_t) * (size_t)std::max(n, 1)));
    for (DevBuf *d : {&ctx->d_ops_off, &ctx->d_rle_off}) CU(d->ensure(sizeof(int64_t) * (size_t)(n + 1)));

    CU(cudaMemsetAsync(ctx->d_bits.p, 0, sizeof(uint32_t) * (size_t)(words + 128), ctx->stream));   // incl. the read-ahead padding
    CU(cudaEventRecord(ctx->ev[EV_COPY_BEGIN], ctx->stream));
    if (n) CU(cudaMemcpyAsync(ctx->d_items.p, ctx->items.data(), sizeof(ItemDesc) * n, cudaMemcpyHostToDevice, ctx->stream));
    if (b->ref_total) CU(cudaMemcpyAsync(ctx->d_ref.p, b->ref_codes, (size_t)b->ref_total, cudaMemcpyHostToDevice, ctx->stream));
    if (packed_seq) {
        if (b->seq_nib_bytes) CU(cudaMemcpyAsync(ctx->d_nib.p, b->seq_nib, (size_t)b->seq_nib_bytes, cudaMemcpyHostToDevice, ctx->stream));
        if (n) {
            CU(cudaMemcpyAsync(ctx->d_nib_start.p, b->seq_nib_start, sizeof(int64_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
            const int parts = (int)std::min<int64_t>(64, (max_seq + 65535) / 65536);
            unpack_nib_kernel<<<dim3(n, parts), 256, 0, ctx->stream>>>(ctx->d_items.as<ItemDesc>(), ctx->d_nib.as<uint8_t>(), ctx->d_nib_start.as<int64_t>(),
                                                                      ctx->d_seq.as<uint8_t>(), parts);
            CU(cudaGetLastError());
        }
    } else if (b->seq_total) CU(cudaMemcpyAsync(ctx->d_seq.p, b->seq_codes, (size_t)b->seq_total, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->total_rle)
        CU(cudaMemcpyAsync(ctx->d_rle.p, b->cigar_rle + b->cigar_off[0], sizeof(uint32_t) * (size_t)ctx->total_rle, cudaMemcpyHostToDevice, ctx->stream));
    if (nchunks) CU(cudaMemcpyAsync(ctx->d_order.p, ctx->order.data(), sizeof(int32_t) * (size_t)nchunks, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaEventRecord(ctx->ev[EV_COPY_END], ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    npore_stats &S = ctx->stats;
    S = npore_stats{};
    S.n_items = n; S.n_chunks = nchunks; S.n_cu = n_cu; S.sm_count = ctx->sm_count;
    S.h2d_bytes = (int64_t)sizeof(ItemDesc) * n + b->ref_total + (packed_seq ? b->seq_nib_bytes + 8 * (int64_t)n : b->seq_total) + 4 * ctx->total_rle + 4 * nchunks;
    cudaEventElapsedTime(&S.ms_h2d, ctx->ev[EV_COPY_BEGIN], ctx->ev[EV_COPY_END]);
    ctx->uploaded = true;
    return NPORE_OK;
}

int npore_run(npore_ctx *ctx, uint32_t flags)
{
    if (!ctx) return NPORE_ERR_BAD_ARG;
    if (!ctx->uploaded) return fail(ctx, NPORE_ERR_STATE, "npore_run before npore_upload");
    if ((flags & NPORE_OUT_NO_EXPANDED) && !(flags & NPORE_OUT_RLE)) return fail(ctx, NPORE_ERR_BAD_ARG, "NO_EXPANDED needs RLE");
    int n_sat = 0;
    int rc = run_pass(ctx, flags, false, &n_sat);
    // A traceback met an n-polymer (LEN/SHR) run that saturated the 11-bit record field (>= 2047 ops; the reference has no such
    // limit): the batch is redone with the WIDE forward kernels, which carry runs unsaturated and keep the true run of such records
    // in an overflow list.  Costs a second pass for that batch only; status 8 remains only if that list overflows (65,536 records).
    if (rc == NPORE_OK && n_sat > 0) rc = run_pass(ctx, flags, true, &n_sat);
    // drain what an error left queued: the context stays reusable, and npore_download reports NPORE_ERR_STATE (ran is false)
    if (rc != NPORE_OK) { cudaStreamSynchronize(ctx->stream); cudaGetLastError(); }
    return rc;
}

int npore_download(npore_ctx *ctx, npore_result *res)
{
    if (!ctx || !res) return NPORE_ERR_BAD_ARG;
    if (!ctx->ran) return fail(ctx, NPORE_ERR_STATE, "npore_download before npore_run");
    CU(cudaSetDevice(ctx->device));
    const int n = (int)ctx->items.size();
    const uint32_t flags = ctx->run_flags;
    const bool want_ops = !(flags & NPORE_OUT_NO_EXPANDED) && res->ops && res->ops_off;
    const bool want_rle = (flags & NPORE_OUT_RLE) && res->rle && res->rle_off;
    npore_stats &S = ctx->stats;
    const SmallBlock hs(ctx->h_small.p, n, ctx->n_chunks);
    // offsets first (sizes arrived with npore_run), then one exact-size copy per output straight into the caller's buffers
    int64_t o = 0, ro = 0, so = 0;
    for (int i = 0; i < n; i++) {
        if (res->status) res->status[i] = hs.status[i];
        if (want_ops) { res->ops_off[i] = o; o += hs.len[i]; }
        if (want_rle) { res->rle_off[i] = ro; ro += hs.rle_len[i]; }
        if (res->chunk_scores && res->score_off) {
            const ItemDesc &I = ctx->items[i];
            res->score_off[i] = so;
            if (so + I.n_chunks > res->score_capacity) return fail(ctx, NPORE_ERR_CAPACITY, "score buffer too small");
            for (int k = 0; k < I.n_chunks; k++) res->chunk_scores[so + k] = hs.chunk_out[I.chunk_first + k].score;
            so += I.n_chunks;
        }
    }
    if (want_ops) { res->ops_off[n] = o; if (o > res->ops_capacity) return fail(ctx, NPORE_ERR_CAPACITY, "ops buffer too small"); }
    if (want_rle) { res->rle_off[n] = ro; if (ro > res->rle_capacity) return fail(ctx, NPORE_ERR_CAPACITY, "rle buffer too small"); }
    if (res->chunk_scores && res->score_off) res->score_off[n] = so;
    S.d2h_bytes = (int64_t)n * 12 + (int64_t)ctx->n_chunks * sizeof(ChunkOut);
    CU(cudaEventRecord(ctx->ev[EV_COPY_BEGIN], ctx->stream));
    if (want_ops && o) { CU(cudaMemcpyAsync(res->ops, ctx->d_pack_ops.p, (size_t)o, cudaMemcpyDeviceToHost, ctx->stream)); S.d2h_bytes += o; }
    if (want_rle && ro) { CU(cudaMemcpyAsync(res->rle, ctx->d_pack_rle.p, 4 * (size_t)ro, cudaMemcpyDeviceToHost, ctx->stream)); S.d2h_bytes += 4 * ro; }
    CU(cudaEventRecord(ctx->ev[EV_COPY_END], ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&S.ms_d2h, ctx->ev[EV_COPY_BEGIN], ctx->ev[EV_COPY_END]);
    return NPORE_OK;
}

int npore_align_batch(npore_ctx *ctx, const npore_batch *batch, uint32_t flags, npore_result *result)
{
    int rc = npore_upload(ctx, batch);
    if (rc != NPORE_OK) return rc;
    rc = npore_run(ctx, flags);
    if (rc != NPORE_OK) return rc;
    return npore_download(ctx, result);
}

int npore_get_np_info_batch(npore_ctx *ctx, int32_t n_seqs, const uint8_t *codes, const int64_t *off, int32_t *out)
{
    if (!ctx || n_seqs < 0 || (n_seqs && (!codes || !off || !out))) return NPORE_ERR_BAD_ARG;
    if (n_seqs == 0) return NPORE_OK;
    const int64_t total = off[n_seqs] - off[0];
    if (off[0] != 0 || total < 0) return fail(ctx, NPORE_ERR_BAD_ARG, "offsets must start at 0 and increase");
    for (int i = 0; i < n_seqs; i++)
        if (off[i + 1] < off[i] || off[i + 1] - off[i] > 0x7ffffff0ll) return fail(ctx, NPORE_ERR_BAD_ARG, "bad sequence offsets");
    if (total == 0) return NPORE_OK;
    CU(cudaSetDevice(ctx->device));
    // staging lives in the context (grow-only, shared with npore_confusion_batch): no cudaMalloc / cudaFree per call
    auto &d = ctx->pileup;
    const size_t ob = (size_t)total * 2 * ctx->P.max_n * sizeof(int32_t);
    int rc = NPORE_OK;
    if (d.ref_codes.ensure((size_t)total) != cudaSuccess || d.ref_off.ensure(sizeof(int64_t) * (size_t)(n_seqs + 1)) != cudaSuccess ||
        d.raw.ensure((size_t)total * 8) != cudaSuccess || d.out.ensure(std::max<size_t>(ob, 4)) != cudaSuccess ||
        d.ebits.ensure(sizeof(uint32_t) * (size_t)(total / 32 + 2 * (size_t)n_seqs + 8)) != cudaSuccess)
        rc = fail(ctx, NPORE_ERR_OOM, "np_info scratch");
    if (rc == NPORE_OK) {
        cudaError_t e = cudaMemcpyAsync(d.ref_codes.p, codes, (size_t)total, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d.ref_off.p, off, sizeof(int64_t) * (size_t)(n_seqs + 1), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) {
            np_info_kernel<<<n_seqs, ANN_THREADS, 0, ctx->stream>>>(d.ref_codes.as<uint8_t>(), d.ref_off.as<int64_t>(), ctx->P.max_n, ctx->P.max_l,
                                                                    d.raw.as<uint8_t>(), d.out.as<int32_t>(), d.ebits.as<uint32_t>());
            e = cudaGetLastError();
        }
        if (e == cudaSuccess && ob) e = cudaMemcpyAsync(out, d.out.p, ob, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, NPORE_ERR_CUDA, "np_info", e);
    }
    return rc;
}

int npore_get_np_info(npore_ctx *ctx, const uint8_t *codes, int32_t len, int32_t *out)
{
    if (!ctx || len < 0 || (len && (!codes || !out))) return NPORE_ERR_BAD_ARG;
    if (len == 0) return NPORE_OK;
    const int64_t off[2] = {0, len};
    return npore_get_np_info_batch(ctx, 1, codes, off, out);
}

int npore_confusion_batch(npore_ctx *ctx, const npore_pileup_batch *b, int64_t *subs, int64_t *nps, int64_t *inss, int64_t *dels)
{
    if (!ctx || !b || !subs || !nps || !inss || !dels || b->n_ranges < 0 || b->n_reads < 0) return NPORE_ERR_BAD_ARG;
    const int R = b->n_ranges, n = b->n_reads, T = ctx->P.max_l + 1;
    const bool nib = b->seq_nib != nullptr;     // BAM's 4-bit bases and phred+33 qualities instead of ASCII and phred
    const size_t n_out = 25 + (size_t)ctx->P.max_n * T * T + 2 * (size_t)T;
    std::memset(subs, 0, 25 * sizeof(int64_t)); std::memset(nps, 0, (size_t)ctx->P.max_n * T * T * sizeof(int64_t));
    std::memset(inss, 0, T * sizeof(int64_t)); std::memset(dels, 0, T * sizeof(int64_t));
    if (R == 0) return NPORE_OK;
    if (!b->range_start || !b->range_end || !b->ref_ascii || !b->ref_off || !b->range_reads_off ||
        (n && (!b->read_pos || (nib ? !b->seq_nib_start : !b->seq_ascii) || !b->seq_off || !b->cigar_rle || !b->cigar_off)))
        return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: null array");
    if (nib && n && b->qual && !b->has_qual) return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: has_qual is required with packed bases and qualities");
    if (nib && b->seq_nib_bytes < 0) return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: negative seq_nib_bytes");
    if (b->ref_off[0] != 0 || b->range_reads_off[0] != 0 || (n && (b->seq_off[0] != 0 || b->cigar_off[0] != 0)))
        return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: offsets must start at 0");
    std::vector<int64_t> pos_off((size_t)R + 1, 0);
    for (int r = 0; r < R; r++) {
        const int64_t len = b->range_end[r] - b->range_start[r], have = b->ref_off[r + 1] - b->ref_off[r];
        if (len <= 0 || len > 0x7ffffff0ll || b->range_start[r] < 0 || have < len || have > 0x7ffffff0ll ||
            b->range_reads_off[r + 1] < b->range_reads_off[r])
            return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: bad range (need end > start and the reference bytes of the whole range)");
        pos_off[r + 1] = pos_off[r] + len;
    }
    const int64_t n_list = b->range_reads_off[R], total_pos = pos_off[R], total_ref = b->ref_off[R];
    if (n_list && !b->range_reads) return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: null read list");
    for (int r = 0; r < R; r++)
        for (int64_t k = b->range_reads_off[r]; k < b->range_reads_off[r + 1]; k++) {
            const int32_t rd = b->range_reads[k];
            if (rd < 0 || rd >= n) return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: read index out of range");
            if (k > b->range_reads_off[r] && b->read_pos[rd] < b->read_pos[b->range_reads[k - 1]])
                return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: a range's reads must be in coordinate order");
        }
    for (int i = 0; i < n; i++)
        if (b->seq_off[i + 1] < b->seq_off[i] || b->cigar_off[i + 1] < b->cigar_off[i] || b->seq_off[i + 1] - b->seq_off[i] > 0x7ffffff0ll)
            return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: bad read offsets");
    if (nib)
        for (int i = 0; i < n; i++)
            if (b->seq_nib_start[i] < 0 || b->seq_nib_start[i] + (b->seq_off[i + 1] - b->seq_off[i]) > 2 * b->seq_nib_bytes)
                return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: packed read outside seq_nib");
    const int64_t seq_total = n ? b->seq_off[n] : 0, n_words = n ? b->cigar_off[n] : 0;
    CU(cudaSetDevice(ctx->device));
    auto &d = ctx->pileup;
    auto put = [&](DevBuf &buf, const void *src, size_t bytes) -> cudaError_t {
        cudaError_t e = buf.ensure(std::max<size_t>(bytes, 16));
        if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
        return e;
    };
    cudaError_t e = cudaSuccess;
    int rc = NPORE_OK;
    const bool have_q = b->qual != nullptr;
#define CM_TRY(x) do { if (e == cudaSuccess) e = (x); } while (0)
    CM_TRY(put(d.range_start, b->range_start, sizeof(int64_t) * R));
    CM_TRY(put(d.range_end, b->range_end, sizeof(int64_t) * R));
    CM_TRY(put(d.ref_ascii, b->ref_ascii, (size_t)total_ref));
    CM_TRY(put(d.ref_off, b->ref_off, sizeof(int64_t) * (R + 1)));
    CM_TRY(d.ref_codes.ensure(std::max<size_t>((size_t)total_ref, 16)));
    CM_TRY(d.raw.ensure(std::max<size_t>((size_t)total_ref * 8, 16)));
    CM_TRY(d.ebits.ensure(sizeof(uint32_t) * (size_t)(total_ref / 32 + 2 * (size_t)R + 8)));
    CM_TRY(put(d.read_pos, b->read_pos, sizeof(int64_t) * n));
    if (nib) {
        CM_TRY(put(d.seq, b->seq_nib, (size_t)b->seq_nib_bytes));
        CM_TRY(put(d.nib_start, b->seq_nib_start, sizeof(int64_t) * n));
        if (have_q) CM_TRY(put(d.has_qual, b->has_qual, sizeof(int32_t) * n));
    } else CM_TRY(put(d.seq, b->seq_ascii, (size_t)seq_total));
    if (have_q) CM_TRY(put(d.qual, b->qual, (size_t)seq_total));
    CM_TRY(put(d.seq_off, b->seq_off, sizeof(int64_t) * (n + 1)));
    CM_TRY(put(d.rle, b->cigar_rle, sizeof(uint32_t) * (size_t)n_words));
    CM_TRY(put(d.cig_off, b->cigar_off, sizeof(int64_t) * (n + 1)));
    for (DevBuf *g : {&d.g_roff, &d.g_qoff}) CM_TRY(g->ensure(std::max<size_t>(sizeof(int32_t) * (size_t)n_words, 16)));
    CM_TRY(d.read_end.ensure(std::max<size_t>(sizeof(int64_t) * (size_t)n, 16)));
    CM_TRY(put(d.range_reads, b->range_reads, sizeof(int32_t) * (size_t)n_list));
    CM_TRY(put(d.range_reads_off, b->range_reads_off, sizeof(int64_t) * (R + 1)));
    CM_TRY(d.list_maxend.ensure(std::max<size_t>(sizeof(int64_t) * (size_t)n_list, 16)));
    CM_TRY(d.line_of.ensure(std::max<size_t>(sizeof(int32_t) * (size_t)total_pos, 16)));
    CM_TRY(put(d.pos_off, pos_off.data(), sizeof(int64_t) * (R + 1)));
    const size_t out_bytes = sizeof(int32_t) * (size_t)(total_pos + R) + sizeof(unsigned long long) * n_out + 16;
    CM_TRY(d.out.ensure(out_bytes));
    CM_TRY(cudaMemsetAsync(d.out.p, 0, out_bytes, ctx->stream));
    if (e != cudaSuccess) rc = fail(ctx, e == cudaErrorMemoryAllocation ? NPORE_ERR_OOM : NPORE_ERR_CUDA, "confusion staging", e);
    std::vector<unsigned long long> h_out(n_out + 2);
    if (rc == NPORE_OK) {
        ConfusionArgs a;
        a.n_ranges = R; a.n_reads = n;
        a.range_start = d.range_start.as<int64_t>(); a.range_end = d.range_end.as<int64_t>();
        a.ref_ascii = d.ref_ascii.as<uint8_t>(); a.ref_off = d.ref_off.as<int64_t>(); a.ref_codes = d.ref_codes.as<uint8_t>();
        a.raw = d.raw.as<uint8_t>(); a.ebits = d.ebits.as<uint32_t>();
        a.read_pos = d.read_pos.as<int64_t>(); a.seq = d.seq.as<uint8_t>(); a.qual = have_q ? d.qual.as<uint8_t>() : nullptr;
        a.seq_off = d.seq_off.as<int64_t>(); a.rle = d.rle.as<uint32_t>(); a.cig_off = d.cig_off.as<int64_t>();
        a.g_roff = d.g_roff.as<int32_t>(); a.g_qoff = d.g_qoff.as<int32_t>(); a.read_end = d.read_end.as<int64_t>();
        a.range_reads = d.range_reads.as<int32_t>(); a.range_reads_off = d.range_reads_off.as<int64_t>(); a.list_maxend = d.list_maxend.as<int64_t>();
        a.line_of = d.line_of.as<int32_t>(); a.pos_off = d.pos_off.as<int64_t>();
        // zeroed block: outputs first (8-byte aligned), then the coverage difference array
        unsigned long long *o = d.out.as<unsigned long long>();
        a.subs = o; a.nps = o + 25; a.inss = a.nps + (size_t)ctx->P.max_n * T * T; a.dels = a.inss + T;
        a.bad = reinterpret_cast<int *>(o + n_out);
        a.diff = reinterpret_cast<int32_t *>(o + n_out + 2);
        a.max_n = ctx->P.max_n; a.max_l = ctx->P.max_l; a.min_bq = b->min_base_q;
        a.seq_nib_start = nib ? d.nib_start.as<int64_t>() : nullptr; a.has_qual = nib && have_q ? d.has_qual.as<int32_t>() : nullptr;
        const int sm = ctx->stats.sm_count > 0 ? ctx->stats.sm_count : 148;
        cm_codes_kernel<<<sm * 4, 256, 0, ctx->stream>>>(a.ref_ascii, a.ref_codes, total_ref);
        cm_np_kernel<<<R, ANN_THREADS, 0, ctx->stream>>>(a);
        if (n) cm_read_kernel<<<(n + CM_THREADS / 32 - 1) / (CM_THREADS / 32), CM_THREADS, 0, ctx->stream>>>(a);
        cm_range_kernel<<<R, CM_THREADS, 0, ctx->stream>>>(a);
        const int64_t want = (total_pos + CM_THREADS / 32 - 1) / (CM_THREADS / 32);
        const int grid = (int)std::min<int64_t>(want, (int64_t)sm * 8);
        if (nib) cm_pileup_kernel<CmNibRead><<<grid, CM_THREADS, 0, ctx->stream>>>(a);
        else cm_pileup_kernel<CmAsciiRead><<<grid, CM_THREADS, 0, ctx->stream>>>(a);
        e = cudaGetLastError();
        CM_TRY(cudaMemcpyAsync(h_out.data(), o, sizeof(unsigned long long) * (n_out + 2), cudaMemcpyDeviceToHost, ctx->stream));
        CM_TRY(cudaStreamSynchronize(ctx->stream));
        if (e != cudaSuccess) rc = fail(ctx, NPORE_ERR_CUDA, "confusion kernels", e);
    }
#undef CM_TRY

    if (rc != NPORE_OK) return rc;
    if (*reinterpret_cast<int *>(&h_out[n_out])) return fail(ctx, NPORE_ERR_BAD_ARG, "confusion: CIGAR op P or B is not supported");
    std::memcpy(subs, h_out.data(), 25 * sizeof(int64_t));
    std::memcpy(nps, h_out.data() + 25, (size_t)ctx->P.max_n * T * T * sizeof(int64_t));
    std::memcpy(inss, h_out.data() + 25 + (size_t)ctx->P.max_n * T * T, T * sizeof(int64_t));
    std::memcpy(dels, h_out.data() + 25 + (size_t)ctx->P.max_n * T * T + T, T * sizeof(int64_t));
    return NPORE_OK;
}

int npore_bgzf_create(npore_bgzf **out, int device)
{
    if (!out) return NPORE_ERR_BAD_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return NPORE_ERR_NO_DEVICE; }
    if (device < 0 || device >= ndev) return NPORE_ERR_BAD_ARG;
    npore_bgzf *z = new npore_bgzf();
    z->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&z->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&z->ev[0]) != cudaSuccess || cudaEventCreate(&z->ev[1]) != cudaSuccess ||
        cudaFuncSetAttribute(bgzf::bgzf_deflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bgzf::kDynSmem) != cudaSuccess ||
        z->d_total.ensure(sizeof(int64_t)) != cudaSuccess) {
        cudaGetLastError();
        npore_bgzf_destroy(z);
        return NPORE_ERR_CUDA;
    }
    *out = z;
    return NPORE_OK;
}

void npore_bgzf_destroy(npore_bgzf *z)
{
    if (!z) return;
    cudaSetDevice(z->device);
    delete z;                            // frees the buffers, on the device set above
}

int64_t npore_bgzf_bound(int64_t n)
{
    if (n <= 0) return 0;
    return (n + BGZF_BLOCK - 1) / BGZF_BLOCK * (BGZF_MEMBER_OVERHEAD + 5) + n;
}

int npore_bgzf_compress(npore_bgzf *z, const uint8_t *in, int64_t n, uint8_t *out, int64_t out_capacity, int64_t *out_len,
                        float *device_ms)
{
    if (!z || n < 0 || !out_len || (n && (!in || !out))) return NPORE_ERR_BAD_ARG;
    *out_len = 0;
    z->last_n = 0;
    if (device_ms) *device_ms = 0.0f;
    if (!n) return NPORE_OK;
    const int64_t members = (n + BGZF_BLOCK - 1) / BGZF_BLOCK;
    if (members > (1 << 30)) return NPORE_ERR_BAD_ARG;
    auto check = [&](cudaError_t e) {
        if (e == cudaSuccess) return NPORE_OK;
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? NPORE_ERR_OOM : NPORE_ERR_CUDA;
    };
    int rc;
    if ((rc = check(cudaSetDevice(z->device))) ||
        (rc = check(z->d_in.ensure((size_t)n))) ||
        (rc = check(z->d_tok.ensure((size_t)members * BGZF_BLOCK * sizeof(uint32_t)))) ||
        (rc = check(z->d_slots.ensure((size_t)members * BGZF_SLOT))) ||
        (rc = check(z->d_sizes.ensure((size_t)members * sizeof(int32_t)))) ||
        (rc = check(z->d_out.ensure((size_t)npore_bgzf_bound(n)))))
        return rc;
    int64_t total = 0;
    if ((rc = check(cudaMemcpyAsync(z->d_in.p, in, (size_t)n, cudaMemcpyHostToDevice, z->stream))) ||
        (rc = check(cudaEventRecord(z->ev[0], z->stream))))
        return rc;
    bgzf::bgzf_deflate_kernel<<<(unsigned)members, BGZF_THREADS, bgzf::kDynSmem, z->stream>>>(
        z->d_in.as<uint8_t>(), n, z->d_tok.as<uint32_t>(), z->d_slots.as<uint8_t>(), z->d_sizes.as<int32_t>());
    bgzf::bgzf_gather_kernel<<<(unsigned)members, BGZF_THREADS, 0, z->stream>>>(
        z->d_slots.as<uint8_t>(), z->d_sizes.as<int32_t>(), (int)members, z->d_out.as<uint8_t>(), z->d_total.as<int64_t>());
    if ((rc = check(cudaGetLastError())) ||
        (rc = check(cudaEventRecord(z->ev[1], z->stream))) ||
        (rc = check(cudaMemcpyAsync(&total, z->d_total.p, sizeof(total), cudaMemcpyDeviceToHost, z->stream))) ||
        (rc = check(cudaStreamSynchronize(z->stream))))
        return rc;
    if (total > out_capacity) return NPORE_ERR_CAPACITY;
    if ((rc = check(cudaMemcpyAsync(out, z->d_out.p, (size_t)total, cudaMemcpyDeviceToHost, z->stream))) ||
        (rc = check(cudaStreamSynchronize(z->stream))))
        return rc;
    if (device_ms && (rc = check(cudaEventElapsedTime(device_ms, z->ev[0], z->ev[1])))) return rc;
    *out_len = total;
    z->last_n = n;
    return NPORE_OK;
}

int npore_bgzf_index(npore_bgzf *z, const int64_t *rec_off, int64_t n_rec, uint64_t base, npore_bai_lists *out, float *device_ms)
{
    if (!z || !out || n_rec < 0 || (n_rec && !rec_off)) return NPORE_ERR_BAD_ARG;
    std::memset(out, 0, sizeof(*out));
    if (device_ms) *device_ms = 0.0f;
    if (!n_rec) return NPORE_OK;
    const int64_t n_in = z->last_n, members = (n_in + BGZF_BLOCK - 1) / BGZF_BLOCK;
    if (rec_off[0] != 0 || rec_off[n_rec] != n_in) return NPORE_ERR_BAD_ARG;      // not the records of the last compressed input
    auto check = [&](cudaError_t e) {
        if (e == cudaSuccess) return NPORE_OK;
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? NPORE_ERR_OOM : NPORE_ERR_CUDA;
    };
    int rc;
    if ((rc = check(cudaSetDevice(z->device))) ||
        (rc = check(z->d_rec_off.ensure((size_t)(n_rec + 1) * sizeof(int64_t)))) ||
        (rc = check(z->d_moff.ensure((size_t)(members + 1) * sizeof(uint64_t)))) ||
        (rc = check(z->d_recs.ensure((size_t)n_rec * sizeof(bai::Rec)))) ||
        (rc = check(z->d_chunks.ensure((size_t)n_rec * sizeof(bai::Chunk)))) ||
        (rc = check(z->d_sorted.ensure((size_t)n_rec * sizeof(bai::Chunk)))) ||
        (rc = check(z->d_segs.ensure((size_t)n_rec * sizeof(bai::Seg)))) ||
        (rc = check(z->d_out_chunks.ensure((size_t)n_rec * 4 * sizeof(uint64_t)))) ||
        (rc = check(z->d_out_refs.ensure((size_t)n_rec * 7 * sizeof(uint64_t)))) ||
        (rc = check(z->d_counts.ensure(4 * sizeof(uint64_t)))) ||
        (rc = check(z->h_counts.ensure(4 * sizeof(uint64_t)))))
        return rc;
    unsigned long long *counts = z->d_counts.as<unsigned long long>();
    if ((rc = check(cudaMemcpyAsync(z->d_rec_off.p, rec_off, (size_t)(n_rec + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, z->stream))) ||
        (rc = check(cudaMemsetAsync(counts, 0, 4 * sizeof(uint64_t), z->stream))) ||
        (rc = check(cudaEventRecord(z->ev[0], z->stream))))
        return rc;
    bai::bai_member_kernel<<<1, BAI_THREADS, 0, z->stream>>>(z->d_sizes.as<int32_t>(), members, base, z->d_moff.as<uint64_t>());
    bai::bai_record_kernel<<<(unsigned)((n_rec + 255) / 256), 256, 0, z->stream>>>(
        z->d_in.as<uint8_t>(), n_in, members, z->d_rec_off.as<int64_t>(), n_rec, z->d_moff.as<uint64_t>(), z->d_recs.as<bai::Rec>(), counts + 3);
    bai::bai_chunk_kernel<<<1, BAI_THREADS, 0, z->stream>>>(z->d_recs.as<bai::Rec>(), n_rec, z->d_chunks.as<bai::Chunk>(),
        z->d_sorted.as<bai::Chunk>(), z->d_segs.as<bai::Seg>(), z->d_out_chunks.as<uint64_t>(), z->d_out_refs.as<uint64_t>(), counts);
    uint64_t *hc = static_cast<uint64_t *>(z->h_counts.p);
    if ((rc = check(cudaGetLastError())) ||
        (rc = check(cudaMemcpyAsync(hc, counts, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, z->stream))) ||
        (rc = check(cudaStreamSynchronize(z->stream))))
        return rc;
    out->error_bits = hc[3];
    if (hc[3]) return NPORE_ERR_BAD_ARG;
    const int64_t n_ch = (int64_t)hc[0], n_seg = (int64_t)hc[1], n_win = (int64_t)hc[2];
    const size_t b_ch = (size_t)n_ch * 4 * sizeof(uint64_t), b_seg = (size_t)n_seg * 7 * sizeof(uint64_t), b_win = (size_t)n_win * sizeof(uint64_t);
    if ((rc = check(z->d_win.ensure(std::max<size_t>(b_win, 8)))) || (rc = check(z->h_lists.ensure(b_ch + b_seg + b_win))))
        return rc;
    if (n_win) {
        if ((rc = check(cudaMemsetAsync(z->d_win.p, 0xFF, b_win, z->stream)))) return rc;
        bai::bai_linear_kernel<<<(unsigned)((n_rec + 255) / 256), 256, 0, z->stream>>>(z->d_recs.as<bai::Rec>(), n_rec, z->d_segs.as<bai::Seg>(),
                                                                                       z->d_win.as<unsigned long long>());
    }
    uint8_t *h = static_cast<uint8_t *>(z->h_lists.p);
    if ((rc = check(cudaGetLastError())) ||
        (rc = check(cudaEventRecord(z->ev[1], z->stream))) ||
        (rc = check(cudaMemcpyAsync(h, z->d_out_chunks.p, b_ch, cudaMemcpyDeviceToHost, z->stream))) ||
        (rc = check(cudaMemcpyAsync(h + b_ch, z->d_out_refs.p, b_seg, cudaMemcpyDeviceToHost, z->stream))) ||
        (n_win && (rc = check(cudaMemcpyAsync(h + b_ch + b_seg, z->d_win.p, b_win, cudaMemcpyDeviceToHost, z->stream)))) ||
        (rc = check(cudaStreamSynchronize(z->stream))))
        return rc;
    if (device_ms && (rc = check(cudaEventElapsedTime(device_ms, z->ev[0], z->ev[1])))) return rc;
    out->chunks = reinterpret_cast<const uint64_t *>(h);
    out->n_chunks = n_ch;
    out->refs = reinterpret_cast<const uint64_t *>(h + b_ch);
    out->n_refs = n_seg;
    out->windows = reinterpret_cast<const uint64_t *>(h + b_ch + b_seg);
    out->n_windows = n_win;
    return NPORE_OK;
}

int npore_last_stats(const npore_ctx *ctx, npore_stats *stats)
{
    if (!ctx || !stats) return NPORE_ERR_BAD_ARG;
    *stats = ctx->stats;
    return NPORE_OK;
}

}  // extern "C"
