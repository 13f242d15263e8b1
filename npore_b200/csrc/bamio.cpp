// bamio.cpp -- native BAM ingest (BGZF inflate + record decode) and SAM record formatting; include/npore_bamio.h.
// Replaces, for the realignment path, what the reference reads through pysam (src/bam.pyx:18-47) and prints per read
// (src/bam.pyx:81-84).  Formats follow the SAM/BAM specification (section 4: BGZF members with a BC extra field;
// records `block_size, refID, pos, l_read_name, mapq, bin, n_cigar_op, flag, l_seq, next_refID, next_pos, tlen,
// read_name, cigar, seq (4-bit =ACMGRSVTWYHKDBN), qual, aux`).
#include <sys/resource.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <cerrno>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/npore_bamio.h"

namespace {

thread_local std::string g_err;

int io_fail(int code, const std::string &what) { g_err = what; return code; }

// Background work (the prefetch of the next window) runs at nice +10: it soaks up idle cores, but the short foreground jobs of the
// pipeline -- the gathers in front of an upload, the SAM formatter -- pre-empt it instead of queueing behind 16 inflate threads
// (measured: the 0.5 ms nibble gather took 4-8 ms beside an unprioritised prefetch).
thread_local bool g_background = false;

void enter_background()
{
    g_background = true;
    setpriority(PRIO_PROCESS, (id_t)syscall(SYS_gettid), 10);       // Linux: per-thread; raising niceness needs no privilege
}

template <class F>
void parallel_for(int64_t n, int n_threads, F &&body)        // body(begin, end) on contiguous slices
{
    int t = n_threads > 0 ? n_threads : (int)std::thread::hardware_concurrency();
    t = (int)std::max<int64_t>(1, std::min<int64_t>(t, n));
    if (t == 1) { body((int64_t)0, n); return; }
    const bool bg = g_background;
    std::vector<std::thread> pool;
    for (int k = 0; k < t; k++) pool.emplace_back([=, &body] { if (bg) enter_background(); body(n * k / t, n * (k + 1) / t); });
    for (auto &th : pool) th.join();
}

// Byte buffer without value-initialisation (std::vector::resize memsets: 60 MB of zeroing + fresh page faults per file were a third of
// the serial part of a window load); capacity is kept across windows.
struct Bytes {
    uint8_t *p = nullptr; size_t n = 0, cap = 0;
    Bytes() = default;
    Bytes(const Bytes &) = delete;
    Bytes &operator=(const Bytes &) = delete;
    ~Bytes() { std::free(p); }
    size_t size() const { return n; }
    uint8_t *data() { return p; }
    const uint8_t *data() const { return p; }
    uint8_t &operator[](size_t i) { return p[i]; }
    const uint8_t &operator[](size_t i) const { return p[i]; }
    void resize(size_t m)
    {
        if (m > cap) {
            const size_t c = std::max(m, cap + cap / 2 + 4096);
            uint8_t *q = (uint8_t *)std::realloc(p, c);
            if (!q) throw std::bad_alloc();
            p = q; cap = c;
        }
        n = m;
    }
    void erase_front(size_t k) { if (k) { std::memmove(p, p + k, n - k); n -= k; } }
    void assign(const uint8_t *b, const uint8_t *e) { resize((size_t)(e - b)); if (e > b) std::memcpy(p, b, (size_t)(e - b)); }
    void swap(Bytes &o) { std::swap(p, o.p); std::swap(n, o.n); std::swap(cap, o.cap); }
};

inline uint32_t rd32(const uint8_t *p) { uint32_t v; std::memcpy(&v, p, 4); return v; }
inline uint16_t rd16(const uint8_t *p) { uint16_t v; std::memcpy(&v, p, 2); return v; }

struct Rec {                // decoded once at open
    int64_t off;            // offset of the record's refID field in `data`
    uint64_t voff;          // virtual offset of the record's block_size field (file offset of its member << 16 | offset inside)
    int32_t ref_id, pos, end, l_seq, n_cigar, n_cigar_kept, lead, trail, hp, name_len;
    uint16_t flag; uint8_t mapq, has_qual;
};

struct MSeg { size_t pos, len; uint64_t coff; size_t moff; };   // data[pos, pos + len): bytes moff.. of the member at file offset coff

// virtual offset of data[i]; a position at the end of a member belongs to the next one ("next member, offset 0")
uint64_t voff_at(const std::vector<MSeg> &segs, size_t i)
{
    size_t lo = 0, hi = segs.size();
    while (lo < hi) { const size_t m = (lo + hi) / 2; if (segs[m].pos + segs[m].len <= i) lo = m + 1; else hi = m; }
    return lo < segs.size() && segs[lo].pos <= i ? segs[lo].coff << 16 | (uint64_t)(segs[lo].moff + i - segs[lo].pos) : UINT64_MAX;
}

// data position of virtual offset v if its member is loaded, else SIZE_MAX
size_t pos_of(const std::vector<MSeg> &segs, uint64_t v)
{
    for (const MSeg &g : segs)
        if (g.coff == v >> 16 && (v & 0xffff) >= g.moff && (v & 0xffff) <= g.moff + g.len) return g.pos + (size_t)(v & 0xffff) - g.moff;
    return SIZE_MAX;
}

// the segments of data[from, ...), shifted to start at 0
std::vector<MSeg> segs_from(const std::vector<MSeg> &segs, size_t from)
{
    std::vector<MSeg> out;
    for (const MSeg &g : segs)
        if (g.pos + g.len > from) {
            MSeg h = g;
            if (h.pos < from) { h.moff += from - h.pos; h.len -= from - h.pos; h.pos = 0; }
            else h.pos -= from;
            out.push_back(h);
        }
    return out;
}

}  // namespace

struct npore_bam {
    FILE *fh = nullptr;
    bool eof = false;
    int n_threads = 0;
    int64_t file_size = 0, c_in = 0, c_out = 0;   // bytes in the file; compressed bytes consumed / inflated bytes produced so far
    int64_t coff = 0, c_read = 0;         // file offset of the next member to read; member bytes read from the file
    Bytes data;                           // inflated BAM stream of the current window (starts with the bytes carried over)
    std::vector<MSeg> segs, nsegs;        // the members in data / ndata
    // npore_bam_restrict: only records whose start lies in one of these chunks of virtual offsets (sorted, disjoint)
    bool restricted = false;
    std::vector<uint64_t> rbeg, rend;
    size_t rk = 0;                        // the chunk being read
    size_t head = 0;                      // first byte of `data` not yet consumed (header / complete records before it)
    std::string text;
    std::vector<std::string> ref_names;
    std::vector<int64_t> ref_lens;
    std::vector<Rec> recs;                // records of the current window
    // the NEXT window, inflated and indexed by a background thread while the caller gathers from the current one (npore_bam_prefetch)
    Bytes ndata; size_t nhead = 0; std::vector<Rec> nrecs;
    std::thread pf; int64_t pf_rc = 0; std::string pf_err;
    ~npore_bam() { if (pf.joinable()) pf.join(); if (fh) std::fclose(fh); }
};

namespace {

// value of an integer-typed HP aux tag, 0 if absent (bam.pyx:46)
int32_t find_hp(const uint8_t *p, const uint8_t *e)
{
    while (p + 3 <= e) {
        const bool hp = p[0] == 'H' && p[1] == 'P';
        const char t = (char)p[2];
        p += 3;
        switch (t) {
        case 'A': case 'c': case 'C': if (hp && t != 'A' && p < e) return t == 'c' ? (int8_t)p[0] : p[0]; p += 1; break;
        case 's': case 'S': if (hp && p + 2 <= e) return t == 's' ? (int16_t)rd16(p) : rd16(p); p += 2; break;
        case 'i': case 'I': if (hp && p + 4 <= e) return (int32_t)rd32(p); p += 4; break;
        case 'f': p += 4; break;
        case 'Z': case 'H': while (p < e && *p) p++; p++; break;
        case 'B': {
            if (p + 5 > e) return 0;
            const char st = (char)p[0]; const uint32_t cnt = rd32(p + 1);
            const int sz = (st == 'c' || st == 'C') ? 1 : (st == 's' || st == 'S') ? 2 : 4;
            p += 5 + (size_t)cnt * sz; break;
        }
        default: return 0;
        }
    }
    return 0;
}

const uint8_t kNt16[17] = "=ACMGRSVTWYHKDBN";

}  // namespace

extern "C" {

const char *npore_io_last_error(void) { return g_err.c_str(); }

// Append the next BGZF members of the file to b->data until at least `want` more inflated bytes are there (or EOF).
// Member layout: 12 fixed bytes, XLEN extra (subfield 'B','C' holds BSIZE = member size - 1), deflate data, CRC32, ISIZE.
// limit_coff >= 0 (a restriction): members starting after that file offset are read only while nothing has been added yet, i.e.
// when the caller needs more bytes to complete a record.  Every member's file offset goes to segs.
static int load_blocks(npore_bam *b, Bytes &data, std::vector<MSeg> &segs, size_t want, int64_t limit_coff = -1)
{
    struct Blk { size_t coff, clen, uoff, ulen; uint32_t crc; };
    Bytes cbuf;
    std::vector<Blk> blks;
    size_t added = 0;
    const size_t base = data.size();
    while (!b->eof && added < want && (limit_coff < 0 || b->coff <= limit_coff || blks.empty())) {
        uint8_t hd[12];
        const size_t got = std::fread(hd, 1, 12, b->fh);
        if (got == 0) { b->eof = true; break; }
        if (got != 12 || hd[0] != 0x1f || hd[1] != 0x8b || hd[2] != 8 || !(hd[3] & 4))
            return io_fail(NPORE_IO_ERR_FORMAT, "not a BGZF file (bad member header)");
        const size_t xlen = rd16(hd + 10);
        const size_t at = cbuf.size();
        cbuf.resize(at + xlen);
        if (xlen && std::fread(&cbuf[at], 1, xlen, b->fh) != xlen) return io_fail(NPORE_IO_ERR_FORMAT, "truncated BGZF header");
        size_t bsize = 0;
        for (size_t q = at; q + 4 <= at + xlen;) {
            const size_t sl = rd16(&cbuf[q + 2]);
            if (cbuf[q] == 'B' && cbuf[q + 1] == 'C' && sl == 2 && q + 6 <= at + xlen) bsize = (size_t)rd16(&cbuf[q + 4]) + 1;
            q += 4 + sl;
        }
        if (bsize < xlen + 20) return io_fail(NPORE_IO_ERR_FORMAT, "truncated BGZF member");
        const size_t rest = bsize - 12 - xlen;                 // deflate data + CRC32 + ISIZE
        cbuf.resize(at + rest);                                // the extra field is not needed any more: overwrite it
        if (std::fread(&cbuf[at], 1, rest, b->fh) != rest) return io_fail(NPORE_IO_ERR_FORMAT, "truncated BGZF member");
        Blk k;
        k.coff = at; k.clen = rest - 8; k.crc = rd32(&cbuf[at + rest - 8]); k.ulen = rd32(&cbuf[at + rest - 4]); k.uoff = base + added;
        if (k.ulen > 65536) return io_fail(NPORE_IO_ERR_FORMAT, "BGZF member claims more than 64 KiB of data (SAM spec 4.1: ISIZE <= 65536)");
        if (k.ulen) segs.push_back({k.uoff, k.ulen, (uint64_t)b->coff, 0});
        b->coff += (int64_t)bsize; b->c_read += (int64_t)bsize;
        added += k.ulen;
        blks.push_back(k);
    }
    data.resize(base + added);
    b->c_in += (int64_t)cbuf.size(); b->c_out += (int64_t)added;
    std::atomic<int> bad{0};
    // members are handed out one at a time (an atomic cursor: their inflate cost varies), one z_stream per thread, reset per member
    std::atomic<int64_t> next{0};
    const int64_t nblk = (int64_t)blks.size();
    parallel_for(std::min<int64_t>(nblk, 64), b->n_threads, [&](int64_t, int64_t) {
        z_stream zs;
        std::memset(&zs, 0, sizeof(zs));
        if (inflateInit2(&zs, -15) != Z_OK) { bad = 1; return; }
        for (int64_t k; (k = next.fetch_add(1)) < nblk && !bad;) {
            const Blk &m = blks[(size_t)k];
            if (!m.ulen) continue;
            inflateReset(&zs);
            zs.next_in = const_cast<Bytef *>(&cbuf[m.coff]); zs.avail_in = (uInt)m.clen;
            zs.next_out = &data[m.uoff]; zs.avail_out = (uInt)m.ulen;
            const int rc = inflate(&zs, Z_FINISH);
            if (rc != Z_STREAM_END || zs.avail_out != 0 || crc32(crc32(0L, Z_NULL, 0), &data[m.uoff], (uInt)m.ulen) != m.crc) bad = 1;
        }
        inflateEnd(&zs);
    });
    if (bad) return io_fail(NPORE_IO_ERR_FORMAT, "BGZF member failed to inflate (corrupt data or CRC mismatch)");
    return NPORE_IO_OK;
}

int npore_bam_open(const char *path, int n_threads, npore_bam **out)
{
    if (!path || !out) return io_fail(NPORE_IO_ERR_ARG, "null argument");
    *out = nullptr;
    FILE *fh = std::fopen(path, "rb");
    if (!fh) return io_fail(NPORE_IO_ERR_OPEN, std::string("cannot open ") + path);
    npore_bam *bam = new npore_bam();
    bam->fh = fh; bam->n_threads = n_threads;
    if (std::fseek(fh, 0, SEEK_END) == 0) { bam->file_size = (int64_t)std::ftell(fh); std::fseek(fh, 0, SEEK_SET); }      // (0 for a pipe: no tail merge)
    std::setvbuf(fh, nullptr, _IOFBF, 1 << 20);          // the member headers are read 12 + 6 bytes at a time
    // ---- BAM header: magic, l_text, text, n_ref, (l_name, name, l_ref)*; members are loaded until it is complete
    auto have = [&](size_t n) -> int {        // 1: n bytes available, 0: file ended first, <0: error
        while (bam->data.size() < n) {
            if (bam->eof) return 0;
            const int rc = load_blocks(bam, bam->data, bam->segs, std::max<size_t>(n - bam->data.size(), 1));
            if (rc) return rc;
        }
        return 1;
    };
    auto bail = [&](int code, const char *what) { delete bam; return io_fail(code, what); };
    int rc = have(12);
    if (rc < 0) { delete bam; return rc; }
    if (!rc || std::memcmp(bam->data.data(), "BAM\1", 4) != 0) return bail(NPORE_IO_ERR_FORMAT, "not a BAM file");
    size_t at = 4;
    const size_t l_text = rd32(&bam->data[at]); at += 4;
    if ((rc = have(at + l_text + 4)) <= 0) { if (rc < 0) { delete bam; return rc; } return bail(NPORE_IO_ERR_FORMAT, "truncated BAM header"); }
    bam->text.assign((const char *)&bam->data[at], l_text);
    bam->text = bam->text.c_str();                    // drop NUL padding
    at += l_text;
    const size_t n_ref = rd32(&bam->data[at]); at += 4;
    for (size_t i = 0; i < n_ref; i++) {
        if ((rc = have(at + 4)) <= 0) { if (rc < 0) { delete bam; return rc; } return bail(NPORE_IO_ERR_FORMAT, "truncated BAM reference list"); }
        const size_t l_name = rd32(&bam->data[at]); at += 4;
        if (!l_name || (rc = have(at + l_name + 4)) <= 0) { if (rc < 0) { delete bam; return rc; } return bail(NPORE_IO_ERR_FORMAT, "truncated BAM reference list"); }
        bam->ref_names.emplace_back((const char *)&bam->data[at], l_name - 1); at += l_name;
        bam->ref_lens.push_back((int64_t)rd32(&bam->data[at])); at += 4;
    }
    bam->head = at;
    *out = bam;
    return NPORE_IO_OK;
}

// Next window of records: drops the previous window, inflates members until at least max_bytes of record data are
// available (<= 0: the rest of the file) and indexes the complete records.  Returns their number; 0 at end of file.
static int64_t fill_window(npore_bam *bam, Bytes &data, std::vector<MSeg> &segs, std::vector<Rec> &recs, size_t &head, int64_t max_bytes)
{
    size_t want = max_bytes > 0 ? (size_t)max_bytes : (size_t)-1;
    if (max_bytes > 0 && bam->file_size > 0) {
        // a short last window is a short last batch, and a short batch costs a full chunk latency on the GPU (12 ms for 74 reads
        // of the C2 file): when what is left of the file would inflate to less than 1.4 windows, this window takes all of it.
        // Under a restriction, what is left is the compressed bytes of the chunks not read yet.
        double left = (double)(bam->file_size - bam->coff);
        if (bam->restricted) {
            left = 0;
            for (size_t k = bam->rk; k < bam->rbeg.size(); k++)
                left += (double)(bam->rend[k] >> 16) - (double)std::max<int64_t>((int64_t)(bam->rbeg[k] >> 16), bam->coff) + 65536.0;
        }
        const double ratio = bam->c_in > (1 << 16) ? (double)bam->c_out / (double)bam->c_in : 3.0;
        if ((double)data.size() + std::max(left, 0.0) * ratio < 1.4 * (double)max_bytes) want = (size_t)-1;
    }
    std::vector<int64_t> offs;
    size_t at = 0, skip = 0;
    for (;;) {
        // index the complete records present
        bool chunks_done = false, seek = false;
        for (;;) {
            if (bam->restricted) {
                // the next record starts at `at` (or in the next member of the file, at offset 0)
                const uint64_t va = at < data.size() ? voff_at(segs, at) : (uint64_t)bam->coff << 16;
                while (bam->rk < bam->rbeg.size() && va >= bam->rend[bam->rk]) bam->rk++;
                if (bam->rk == bam->rbeg.size()) { chunks_done = true; break; }
                if (va < bam->rbeg[bam->rk]) {                // before the chunk: skip to its start, in the data or by a seek
                    const size_t p = pos_of(segs, bam->rbeg[bam->rk]);
                    if (p != SIZE_MAX && p >= at) { at = p; continue; }
                    seek = true;
                    break;
                }
            }
            if (!(at + 4 <= data.size() && !(at >= want && !offs.empty()))) break;
            const size_t bs = rd32(&data[at]);
            if (bs < 32) return io_fail(NPORE_IO_ERR_FORMAT, "corrupt BAM record (block_size < 32)");
            if (at + 4 + bs > data.size()) break;
            offs.push_back((int64_t)at + 4);
            at += 4 + bs;
        }
        if (chunks_done) {                              // every chunk read: nothing after this record counts
            data.resize(at);
            while (!segs.empty() && segs.back().pos >= at) segs.pop_back();
            bam->eof = true;
            break;
        }
        if (seek) {
            const uint64_t v = bam->rbeg[bam->rk];
            data.resize(at);
            while (!segs.empty() && segs.back().pos >= at) segs.pop_back();
            if (!segs.empty() && segs.back().pos + segs.back().len > at) segs.back().len = at - segs.back().pos;
            if (std::fseek(bam->fh, (long)(v >> 16), SEEK_SET) != 0) return io_fail(NPORE_IO_ERR_FORMAT, "seek to an indexed chunk failed");
            bam->coff = (int64_t)(v >> 16); bam->eof = false;
            skip = (size_t)(v & 0xffff);
        }
        if (!seek && ((at >= want && !offs.empty()) || (bam->eof && (at + 4 > data.size() || at + 4 + rd32(&data[at]) > data.size())))) break;
        const size_t need = std::max<size_t>(want > at ? std::min<size_t>(want - at, (size_t)1 << 30) : 1, 1);
        const size_t before = data.size();
        const int64_t limit = bam->restricted && bam->rk < bam->rend.size() ? (int64_t)(bam->rend[bam->rk] >> 16) : -1;
        const int rc = load_blocks(bam, data, segs, need, limit);
        if (rc) return rc;
        if (skip) {                                     // the chunk starts inside the member just loaded
            if (data.size() == before || before + skip > data.size()) return io_fail(NPORE_IO_ERR_FORMAT, "indexed chunk starts past its BGZF member");
            at = before + skip;
            skip = 0;
        }
    }
    if (bam->eof && offs.empty() && at != data.size())
        return io_fail(NPORE_IO_ERR_FORMAT, "truncated BAM record at end of file");
    head = at;
    const Bytes &d = data;
    const int n_threads = bam->n_threads;
    recs.resize(offs.size());
    parallel_for((int64_t)offs.size(), n_threads, [&](int64_t lo, int64_t hi) {
        for (int64_t k = lo; k < hi; k++) {
            const uint8_t *r = &d[(size_t)offs[(size_t)k]];
            const size_t bs = rd32(r - 4);
            Rec &o = recs[(size_t)k];
            o.off = offs[(size_t)k];
            o.voff = voff_at(segs, (size_t)offs[(size_t)k] - 4);
            o.ref_id = (int32_t)rd32(r); o.pos = (int32_t)rd32(r + 4);
            o.name_len = r[8] ? r[8] - 1 : 0; o.mapq = r[9];
            o.n_cigar = rd16(r + 12); o.flag = rd16(r + 14); o.l_seq = (int32_t)rd32(r + 16);
            const uint8_t *cg = r + 32 + r[8];
            const uint8_t *end = r + bs;
            // malformed record (negative l_seq, or fields running past block_size): treated as empty -- checked BEFORE any pointer is formed
            if (o.l_seq < 0 || 32 + (size_t)r[8] + 4 * (size_t)o.n_cigar + ((size_t)o.l_seq + 1) / 2 + (size_t)o.l_seq > bs) { o.n_cigar = 0; o.l_seq = 0; }
            const uint8_t *sq = cg + 4 * (size_t)o.n_cigar;
            const uint8_t *ql = sq + ((size_t)o.l_seq + 1) / 2;
            const uint8_t *aux = ql + o.l_seq;
            if (aux > end) aux = end;
            int64_t span = 0; int kept = 0;
            for (int c = 0; c < o.n_cigar; c++) {
                const uint32_t w = rd32(cg + 4 * c), op = w & 15u;
                if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += w >> 4;
                if (op != 4 && op != 5) kept++;
            }
            o.end = o.pos + (int32_t)span; o.n_cigar_kept = kept;
            auto opat = [&](int c) { return rd32(cg + 4 * c) & 15u; };
            auto lnat = [&](int c) { return (int32_t)(rd32(cg + 4 * c) >> 4); };
            const int nc = o.n_cigar;
            o.lead = nc && opat(0) == 4 ? lnat(0) : (nc > 1 && opat(0) == 5 && opat(1) == 4 ? lnat(1) : 0);
            o.trail = nc && opat(nc - 1) == 4 ? lnat(nc - 1) : (nc > 1 && opat(nc - 1) == 5 && opat(nc - 2) == 4 ? lnat(nc - 2) : 0);
            if (o.lead + o.trail > o.l_seq) { o.lead = std::min(o.lead, o.l_seq); o.trail = o.l_seq - o.lead; }
            o.has_qual = (o.l_seq > 0 && ql[0] != 0xff) ? 1 : 0;
            o.hp = find_hp(aux, end);
        }
    });
    return (int64_t)recs.size();
}

int64_t npore_bam_advance(npore_bam *bam, int64_t max_bytes)
{
    if (!bam) return io_fail(NPORE_IO_ERR_ARG, "null handle");
    if (bam->pf.joinable()) {             // the next window was prefetched: swap it in
        bam->pf.join();
        if (bam->pf_rc < 0) return io_fail((int)bam->pf_rc, bam->pf_err);
        bam->data.swap(bam->ndata); std::swap(bam->recs, bam->nrecs); std::swap(bam->segs, bam->nsegs); bam->head = bam->nhead;
        return bam->pf_rc;
    }
    bam->recs.clear();
    if (bam->head) { bam->segs = segs_from(bam->segs, bam->head); bam->data.erase_front(bam->head); bam->head = 0; }
    return fill_window(bam, bam->data, bam->segs, bam->recs, bam->head, max_bytes);
}

// Start inflating + indexing the window AFTER the current one on a background thread; the current window stays valid for
// npore_bam_columns / _gather until the next npore_bam_advance, which then only swaps.  Overlaps BGZF inflate with the caller's gathers.
int npore_bam_prefetch(npore_bam *bam, int64_t max_bytes)
{
    if (!bam) return io_fail(NPORE_IO_ERR_ARG, "null handle");
    if (bam->pf.joinable()) return NPORE_IO_OK;
    bam->ndata.assign(bam->data.data() + bam->head, bam->data.data() + bam->data.size());      // the bytes carried over (a partial record)
    bam->nsegs = segs_from(bam->segs, bam->head);
    bam->nrecs.clear(); bam->nhead = 0; bam->pf_rc = 0;
    bam->pf = std::thread([bam, max_bytes]() {
        enter_background();
        bam->pf_rc = fill_window(bam, bam->ndata, bam->nsegs, bam->nrecs, bam->nhead, max_bytes);
        if (bam->pf_rc < 0) bam->pf_err = g_err;
    });
    return NPORE_IO_OK;
}

void npore_bam_close(npore_bam *b) { delete b; }

int npore_bam_restrict(npore_bam *b, int64_t n, const uint64_t *vbeg, const uint64_t *vend)
{
    if (!b || n < 0 || (n && (!vbeg || !vend))) return io_fail(NPORE_IO_ERR_ARG, "null argument");
    if (b->pf.joinable() || !b->recs.empty() || b->restricted) return io_fail(NPORE_IO_ERR_ARG, "restrict before the first window, once");
    for (int64_t k = 0; k < n; k++)
        if (vbeg[k] >= vend[k] || (k && vbeg[k] < vend[k - 1])) return io_fail(NPORE_IO_ERR_ARG, "chunks must be sorted, disjoint and non-empty");
    b->rbeg.assign(vbeg, vbeg + n); b->rend.assign(vend, vend + n);
    b->rk = 0; b->restricted = true;
    return NPORE_IO_OK;
}

int npore_bam_voffsets(const npore_bam *b, uint64_t *out)
{
    if (!b || !out) return io_fail(NPORE_IO_ERR_ARG, "null argument");
    for (size_t k = 0; k < b->recs.size(); k++) out[k] = b->recs[k].voff;
    return NPORE_IO_OK;
}

int64_t npore_bam_bytes_read(const npore_bam *b) { return b ? b->c_read : NPORE_IO_ERR_ARG; }

int64_t npore_bam_header_text(const npore_bam *b, const char **text)
{
    if (!b) return NPORE_IO_ERR_ARG;
    if (text) *text = b->text.c_str();
    return (int64_t)b->text.size();
}

int32_t npore_bam_n_refs(const npore_bam *b) { return b ? (int32_t)b->ref_names.size() : NPORE_IO_ERR_ARG; }

int npore_bam_ref(const npore_bam *b, int32_t i, const char **name, int64_t *length)
{
    if (!b || i < 0 || (size_t)i >= b->ref_names.size()) return io_fail(NPORE_IO_ERR_ARG, "reference index out of range");
    if (name) *name = b->ref_names[(size_t)i].c_str();
    if (length) *length = b->ref_lens[(size_t)i];
    return NPORE_IO_OK;
}

int64_t npore_bam_n_records(const npore_bam *b) { return b ? (int64_t)b->recs.size() : NPORE_IO_ERR_ARG; }

int npore_bam_columns(const npore_bam *b, int32_t *ref_id, int32_t *pos, int32_t *end, int32_t *flag, int32_t *mapq,
                      int32_t *aln_len, int32_t *n_cigar, int32_t *name_len, int32_t *hp, int32_t *has_qual)
{
    if (!b) return io_fail(NPORE_IO_ERR_ARG, "null handle");
    for (size_t k = 0; k < b->recs.size(); k++) {
        const Rec &r = b->recs[k];
        if (ref_id) ref_id[k] = r.ref_id;
        if (pos) pos[k] = r.pos;
        if (end) end[k] = r.end;
        if (flag) flag[k] = r.flag;
        if (mapq) mapq[k] = r.mapq;
        if (aln_len) aln_len[k] = r.l_seq - r.lead - r.trail;
        if (n_cigar) n_cigar[k] = r.n_cigar_kept;
        if (name_len) name_len[k] = r.name_len;
        if (hp) hp[k] = r.hp;
        if (has_qual) has_qual[k] = r.has_qual;
    }
    return NPORE_IO_OK;
}

int npore_bam_gather(const npore_bam *b, int64_t n_sel, const int64_t *sel, int n_threads,
                     uint8_t *seq_ascii, uint8_t *seq_codes, uint8_t *qual_ascii, const int64_t *seq_off,
                     uint32_t *cigar, const int64_t *cig_off, uint8_t *names, const int64_t *name_off)
{
    if (!b || n_sel < 0 || (n_sel && !sel)) return io_fail(NPORE_IO_ERR_ARG, "null argument");
    if (((seq_ascii || seq_codes || qual_ascii) && !seq_off) || (cigar && !cig_off) || (names && !name_off))
        return io_fail(NPORE_IO_ERR_ARG, "offsets missing");
    for (int64_t k = 0; k < n_sel; k++)
        if (sel[k] < 0 || (size_t)sel[k] >= b->recs.size()) return io_fail(NPORE_IO_ERR_ARG, "record index out of range");
    uint8_t code_of[16];
    for (int c = 0; c < 16; c++) code_of[c] = kNt16[c] == 'A' ? 1 : kNt16[c] == 'C' ? 2 : kNt16[c] == 'G' ? 3 : kNt16[c] == 'T' ? 4 : 0;
    uint16_t pair_of[256];               // packed byte -> its two letters in memory order (first base = high nibble)
    for (int v = 0; v < 256; v++) { const uint8_t two[2] = {(uint8_t)kNt16[v >> 4], (uint8_t)kNt16[v & 15]}; std::memcpy(&pair_of[v], two, 2); }
    std::atomic<int> bad{0};
    parallel_for(n_sel, n_threads, [&](int64_t lo, int64_t hi) {
        for (int64_t k = lo; k < hi; k++) {
            const Rec &r = b->recs[(size_t)sel[k]];
            const uint8_t *rec = &b->data[(size_t)r.off];
            const uint8_t *cg = rec + 32 + rec[8];
            const uint8_t *sq = cg + 4 * (size_t)r.n_cigar;
            const uint8_t *ql = sq + ((size_t)r.l_seq + 1) / 2;
            const int n = r.l_seq - r.lead - r.trail;
            if (seq_off && seq_off[k + 1] - seq_off[k] != n) { bad = 1; continue; }
            if (cig_off && cig_off[k + 1] - cig_off[k] != r.n_cigar_kept) { bad = 1; continue; }
            if (name_off && name_off[k + 1] - name_off[k] != r.name_len) { bad = 1; continue; }
            if (seq_ascii && !seq_codes) {      // the SAM-text gather: two letters per packed byte from a 256-entry table
                uint8_t *a = seq_ascii + seq_off[k];
                int t = 0, q = r.lead;
                if (n > 0 && (q & 1)) { a[t++] = kNt16[sq[q >> 1] & 15]; q++; }
                for (; t + 1 < n; t += 2, q += 2) std::memcpy(a + t, &pair_of[sq[q >> 1]], 2);
                if (t < n) a[t] = kNt16[sq[q >> 1] >> 4];
            } else if (seq_ascii || seq_codes) {
                uint8_t *a = seq_ascii ? seq_ascii + seq_off[k] : nullptr, *c = seq_codes ? seq_codes + seq_off[k] : nullptr;
                for (int t = 0; t < n; t++) {
                    const int q = r.lead + t;
                    const int nib = (q & 1) ? (sq[q >> 1] & 15) : (sq[q >> 1] >> 4);
                    if (a) a[t] = kNt16[nib];
                    if (c) c[t] = code_of[nib];
                }
            }
            if (qual_ascii && r.has_qual) {
                uint8_t *o = qual_ascii + seq_off[k];
                for (int t = 0; t < n; t++) o[t] = (uint8_t)(ql[r.lead + t] + 33);
            }
            if (cigar) {
                uint32_t *o = cigar + cig_off[k];
                for (int c = 0; c < r.n_cigar; c++) {
                    const uint32_t w = rd32(cg + 4 * c), op = w & 15u;
                    if (op != 4 && op != 5) *o++ = w;
                }
            }
            if (names) std::memcpy(names + name_off[k], rec + 32, (size_t)r.name_len);
        }
    });
    if (bad) return io_fail(NPORE_IO_ERR_ARG, "offset arrays do not match the selected records");
    return NPORE_IO_OK;
}

int npore_bam_gather_nib(const npore_bam *b, int64_t n_sel, const int64_t *sel, int n_threads, int64_t *byte_off, uint8_t *nib, int64_t *nib_start)
{
    if (!b || n_sel < 0 || (n_sel && !sel) || !byte_off) return io_fail(NPORE_IO_ERR_ARG, "null argument");
    for (int64_t k = 0; k < n_sel; k++)
        if (sel[k] < 0 || (size_t)sel[k] >= b->recs.size()) return io_fail(NPORE_IO_ERR_ARG, "record index out of range");
    if (!nib) {         // pass 1: bytes needed per record (whole bytes of the record's SEQ that hold an aligned base)
        byte_off[0] = 0;
        for (int64_t k = 0; k < n_sel; k++) {
            const Rec &r = b->recs[(size_t)sel[k]];
            const int n = r.l_seq - r.lead - r.trail;
            byte_off[k + 1] = byte_off[k] + (n > 0 ? ((r.lead & 1) + n + 1) / 2 : 0);
        }
        return NPORE_IO_OK;
    }
    if (!nib_start) return io_fail(NPORE_IO_ERR_ARG, "null argument");
    parallel_for(n_sel, n_threads, [&](int64_t lo, int64_t hi) {
        for (int64_t k = lo; k < hi; k++) {
            const Rec &r = b->recs[(size_t)sel[k]];
            const uint8_t *rec = &b->data[(size_t)r.off];
            const uint8_t *sq = rec + 32 + rec[8] + 4 * (size_t)r.n_cigar;
            const int64_t nb = byte_off[k + 1] - byte_off[k];
            if (nb > 0) std::memcpy(nib + byte_off[k], sq + (r.lead >> 1), (size_t)nb);      // the bases as they lie in the file
            nib_start[k] = 2 * byte_off[k] + (r.lead & 1);
        }
    });
    return NPORE_IO_OK;
}

static inline int dec_len(uint32_t v) { int n = 1; while (v >= 10) { v /= 10; n++; } return n; }
static inline uint8_t *put_dec(uint8_t *o, int64_t v)
{
    if (v < 0) { *o++ = '-'; v = -v; }
    char tmp[24]; int n = 0;
    do { tmp[n++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (n) *o++ = (uint8_t)tmp[--n];
    return o;
}

int64_t npore_sam_bound(int64_t n, const int64_t *name_off, const int64_t *seq_off, const int64_t *rle_off, int64_t max_ref_name)
{
    if (n < 0 || (n && (!name_off || !seq_off || !rle_off))) return NPORE_IO_ERR_ARG;
    if (!n) return 0;
    // per record: 11 tabs + newline + numeric fields (flag 5, pos 11, mapq 3, tlen 11, hp 11) + "*", "0", "HP:i:" + slack
    return (name_off[n] - name_off[0]) + 2 * (seq_off[n] - seq_off[0]) + 10 * (rle_off[n] - rle_off[0]) + n * (72 + max_ref_name);
}

static int64_t sam_format_impl(int64_t n, int n_threads,
                         const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                         const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                         const int32_t *pos, const int32_t *end, const int32_t *mapq,
                         const uint32_t *rle, const int64_t *rle_off,
                         const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                         const int32_t *hp, uint8_t *out, int64_t out_capacity, int fd, int64_t file_off)
{
    if (n < 0) return io_fail(NPORE_IO_ERR_ARG, "negative count");
    if (!n) return 0;
    if (!names || !name_off || !flag || !ref_id || !ref_names || !ref_name_off || !pos || !end || !mapq || !rle_off || !seq_off ||
        !has_qual || !hp || !out)
        return io_fail(NPORE_IO_ERR_ARG, "null argument");
    static const char kOps[] = "MIDNSHP=XB??????";
    std::vector<int64_t> at((size_t)n + 1, 0);
    // pass 1: exact record lengths
    parallel_for(n, n_threads, [&](int64_t lo, int64_t hi) {
        uint8_t tmp[32];
        for (int64_t k = lo; k < hi; k++) {
            int64_t len = 12;                                         // 11 tabs + '\n'
            len += name_off[k + 1] - name_off[k];
            len += put_dec(tmp, flag[k]) - tmp;
            const bool rok = ref_id[k] >= 0 && ref_id[k] < n_refs;        // a record without a (valid) reference prints RNAME '*'
            len += rok ? ref_name_off[ref_id[k] + 1] - ref_name_off[ref_id[k]] : 1;
            len += put_dec(tmp, (int64_t)pos[k] + 1) - tmp;
            len += put_dec(tmp, mapq[k]) - tmp;
            for (int64_t g = rle_off[k]; g < rle_off[k + 1]; g++) len += dec_len(rle[g] >> 4) + 1;
            len += 2;                                                 // "*" and "0"
            len += put_dec(tmp, (int64_t)end[k] - pos[k]) - tmp;
            const int64_t sl = seq_off[k + 1] - seq_off[k];
            len += sl + ((has_qual[k] && sl) ? sl : 1);
            len += 5 + (put_dec(tmp, hp[k]) - tmp);
            at[(size_t)k + 1] = len;
        }
    });
    for (int64_t k = 0; k < n; k++) at[(size_t)k + 1] += at[(size_t)k];
    if (at[(size_t)n] > out_capacity) return io_fail(NPORE_IO_ERR_ARG, "output buffer too small (use npore_sam_bound)");
    // pass 2: write
    std::atomic<int> wr_err{0};
    parallel_for(n, n_threads, [&](int64_t lo, int64_t hi) {
        for (int64_t k = lo; k < hi; k++) {
            uint8_t *o = out + at[(size_t)k];
            const int64_t nl = name_off[k + 1] - name_off[k];
            std::memcpy(o, names + name_off[k], (size_t)nl); o += nl; *o++ = '\t';
            o = put_dec(o, flag[k]); *o++ = '\t';
            if (ref_id[k] >= 0 && ref_id[k] < n_refs) {
                const int64_t rl = ref_name_off[ref_id[k] + 1] - ref_name_off[ref_id[k]];
                std::memcpy(o, ref_names + ref_name_off[ref_id[k]], (size_t)rl); o += rl;
            } else *o++ = '*';
            *o++ = '\t';
            o = put_dec(o, (int64_t)pos[k] + 1); *o++ = '\t';
            o = put_dec(o, mapq[k]); *o++ = '\t';
            for (int64_t g = rle_off[k]; g < rle_off[k + 1]; g++) { o = put_dec(o, rle[g] >> 4); *o++ = (uint8_t)kOps[rle[g] & 15u]; }
            *o++ = '\t'; *o++ = '*'; *o++ = '\t'; *o++ = '0'; *o++ = '\t';
            o = put_dec(o, (int64_t)end[k] - pos[k]); *o++ = '\t';
            const int64_t sl = seq_off[k + 1] - seq_off[k];
            std::memcpy(o, seq_ascii + seq_off[k], (size_t)sl); o += sl; *o++ = '\t';
            if (has_qual[k] && sl) { std::memcpy(o, qual_ascii + seq_off[k], (size_t)sl); o += sl; } else *o++ = '*';
            *o++ = '\t';
            std::memcpy(o, "HP:i:", 5); o += 5;
            o = put_dec(o, hp[k]); *o++ = '\n';
        }
        if (fd >= 0) {      // the slice is complete: straight into the file, beside the other threads' formatting and writes
            const uint8_t *p = out + at[(size_t)lo];
            int64_t left = at[(size_t)hi] - at[(size_t)lo], off = file_off + at[(size_t)lo];
            while (left > 0) {
                const ssize_t w = pwrite(fd, p, (size_t)left, (off_t)off);
                if (w < 0) { if (errno == EINTR) continue; wr_err = errno ? errno : EIO; break; }
                p += w; left -= w; off += w;
            }
        }
    });
    if (wr_err) return io_fail(NPORE_IO_ERR_OPEN, std::string("pwrite failed: ") + std::strerror(wr_err));
    return at[(size_t)n];
}

int64_t npore_sam_format(int64_t n, int n_threads,
                         const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                         const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                         const int32_t *pos, const int32_t *end, const int32_t *mapq,
                         const uint32_t *rle, const int64_t *rle_off,
                         const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                         const int32_t *hp, uint8_t *out, int64_t out_capacity)
{
    return sam_format_impl(n, n_threads, names, name_off, flag, ref_id, ref_names, ref_name_off, n_refs, pos, end, mapq, rle, rle_off,
                           seq_ascii, qual_ascii, seq_off, has_qual, hp, out, out_capacity, -1, 0);
}

int64_t npore_sam_format_fd(int64_t n, int n_threads,
                            const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                            const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                            const int32_t *pos, const int32_t *end, const int32_t *mapq,
                            const uint32_t *rle, const int64_t *rle_off,
                            const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                            const int32_t *hp, uint8_t *scratch, int64_t scratch_capacity, int fd, int64_t file_offset)
{
    if (fd < 0 || file_offset < 0) return io_fail(NPORE_IO_ERR_ARG, "bad file descriptor / offset");
    return sam_format_impl(n, n_threads, names, name_off, flag, ref_id, ref_names, ref_name_off, n_refs, pos, end, mapq, rle, rle_off,
                           seq_ascii, qual_ascii, seq_off, has_qual, hp, scratch, scratch_capacity, fd, file_offset);
}

int64_t npore_bam_bound(int64_t n, const int64_t *name_off, const int64_t *seq_off, const int64_t *rle_off)
{
    if (n < 0 || (n && (!name_off || !seq_off || !rle_off))) return NPORE_IO_ERR_ARG;
    if (!n) return 0;
    // per record: block_size + 32 fixed bytes + the name's NUL + the HP tag (at most 7 bytes); SEQ + QUAL <= 2 bytes per base
    return (name_off[n] - name_off[0]) + 2 * (seq_off[n] - seq_off[0]) + 4 * (rle_off[n] - rle_off[0]) + n * 48;
}

static int64_t bam_format_impl(int64_t n, int n_threads,
                         const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id, int32_t n_refs,
                         const int32_t *pos, const int32_t *end, const int32_t *mapq,
                         const uint32_t *rle, const int64_t *rle_off,
                         const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                         const int32_t *hp, uint8_t *out, int64_t out_capacity, int64_t *rec_off)
{
    if (n < 0) return io_fail(NPORE_IO_ERR_ARG, "negative count");
    if (!n) return 0;
    if (!names || !name_off || !flag || !ref_id || !pos || !end || !mapq || !rle_off || !seq_off || !has_qual || !hp || !out)
        return io_fail(NPORE_IO_ERR_ARG, "null argument");
    uint8_t nt16[256];
    for (int c = 0; c < 256; c++) nt16[c] = 15;
    for (int i = 0; i < 16; i++) { nt16[kNt16[i]] = (uint8_t)i; nt16[std::tolower(kNt16[i])] = (uint8_t)i; }
    auto hp_bytes = [](int32_t v) { return v < 0 ? (v >= -128 ? 1 : v >= -32768 ? 2 : 4) : (v <= 255 ? 1 : v <= 65535 ? 2 : 4); };
    std::vector<int64_t> at((size_t)n + 1, 0);
    std::atomic<int> bad{0};
    // pass 1: exact record lengths
    parallel_for(n, n_threads, [&](int64_t lo, int64_t hi) {
        for (int64_t k = lo; k < hi; k++) {
            const int64_t nl = name_off[k + 1] - name_off[k], nc = rle_off[k + 1] - rle_off[k], sl = seq_off[k + 1] - seq_off[k];
            if (nl > 254 || nc > 65535 || sl > INT32_MAX) { bad = 1; continue; }
            at[(size_t)k + 1] = 4 + 32 + nl + 1 + 4 * nc + (sl + 1) / 2 + sl + 3 + hp_bytes(hp[k]);
        }
    });
    if (bad) return io_fail(NPORE_IO_ERR_ARG, "record not representable in BAM (read name > 254 bytes or CIGAR > 65535 operations)");
    for (int64_t k = 0; k < n; k++) at[(size_t)k + 1] += at[(size_t)k];
    if (at[(size_t)n] > out_capacity) return io_fail(NPORE_IO_ERR_ARG, "output buffer too small (use npore_bam_bound)");
    // pass 2: write (SAM spec 4.2; the fields of the SAM line of npore_sam_format, encoded as htslib's SAM -> BAM conversion does)
    parallel_for(n, n_threads, [&](int64_t lo, int64_t hi) {
        for (int64_t k = lo; k < hi; k++) {
            uint8_t *o = out + at[(size_t)k];
            const int64_t nl = name_off[k + 1] - name_off[k], nc = rle_off[k + 1] - rle_off[k], sl = seq_off[k + 1] - seq_off[k];
            int64_t span = 0;
            for (int64_t g = rle_off[k]; g < rle_off[k + 1]; g++) {
                const uint32_t op = rle[g] & 15u;
                if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += rle[g] >> 4;
            }
            const int32_t p = pos[k];
            const int32_t rid = ref_id[k] >= 0 && ref_id[k] < n_refs ? ref_id[k] : -1;
            const int64_t e = (int64_t)p + (span ? span : 1) - 1;       // hts_reg2bin(beg, end) of the 0-based half-open span
            const int bin = (p >> 14 == e >> 14) ? 4681 + (p >> 14) : (p >> 17 == e >> 17) ? 585 + (p >> 17) :
                            (p >> 20 == e >> 20) ? 73 + (p >> 20) : (p >> 23 == e >> 23) ? 9 + (p >> 23) :
                            (p >> 26 == e >> 26) ? 1 + (p >> 26) : 0;
            const int32_t fixed[9] = {(int32_t)(at[(size_t)k + 1] - at[(size_t)k] - 4), rid, p, 0, 0, (int32_t)sl, -1, -1, end[k] - p};
            std::memcpy(o, fixed, 12);
            o[12] = (uint8_t)(nl + 1); o[13] = (uint8_t)mapq[k];
            const uint16_t bn = (uint16_t)bin, ncig = (uint16_t)nc, fl = (uint16_t)flag[k];
            std::memcpy(o + 14, &bn, 2); std::memcpy(o + 16, &ncig, 2); std::memcpy(o + 18, &fl, 2);
            std::memcpy(o + 20, fixed + 5, 16);
            o += 36;
            std::memcpy(o, names + name_off[k], (size_t)nl); o += nl; *o++ = 0;
            if (nc) std::memcpy(o, rle + rle_off[k], (size_t)nc * 4);
            o += 4 * nc;
            const uint8_t *sq = seq_ascii + seq_off[k];
            for (int64_t i = 0; i + 1 < sl; i += 2) *o++ = (uint8_t)(nt16[sq[i]] << 4 | nt16[sq[i + 1]]);
            if (sl & 1) *o++ = (uint8_t)(nt16[sq[sl - 1]] << 4);
            if (has_qual[k] && sl) {
                const uint8_t *q = qual_ascii + seq_off[k];
                for (int64_t i = 0; i < sl; i++) o[i] = (uint8_t)(q[i] - 33);
            } else std::memset(o, 0xFF, (size_t)sl);
            o += sl;
            const int32_t v = hp[k];
            const int nb = hp_bytes(v);
            o[0] = 'H'; o[1] = 'P'; o[2] = (uint8_t)(v < 0 ? (nb == 1 ? 'c' : nb == 2 ? 's' : 'i') : (nb == 1 ? 'C' : nb == 2 ? 'S' : 'I'));
            std::memcpy(o + 3, &v, (size_t)nb);          // little-endian: the low bytes of the value
        }
    });
    if (rec_off) std::memcpy(rec_off, at.data(), ((size_t)n + 1) * sizeof(int64_t));
    return at[(size_t)n];
}

int64_t npore_bam_format(int64_t n, int n_threads,
                         const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                         const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                         const int32_t *pos, const int32_t *end, const int32_t *mapq,
                         const uint32_t *rle, const int64_t *rle_off,
                         const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                         const int32_t *hp, uint8_t *out, int64_t out_capacity)
{
    (void)ref_names; (void)ref_name_off;
    return bam_format_impl(n, n_threads, names, name_off, flag, ref_id, n_refs, pos, end, mapq, rle, rle_off, seq_ascii, qual_ascii,
                           seq_off, has_qual, hp, out, out_capacity, nullptr);
}

int64_t npore_bam_format_offsets(int64_t n, int n_threads,
                                 const uint8_t *names, const int64_t *name_off, const int32_t *flag, const int32_t *ref_id,
                                 const uint8_t *ref_names, const int64_t *ref_name_off, int32_t n_refs,
                                 const int32_t *pos, const int32_t *end, const int32_t *mapq,
                                 const uint32_t *rle, const int64_t *rle_off,
                                 const uint8_t *seq_ascii, const uint8_t *qual_ascii, const int64_t *seq_off, const int32_t *has_qual,
                                 const int32_t *hp, uint8_t *out, int64_t out_capacity, int64_t *rec_off)
{
    (void)ref_names; (void)ref_name_off;
    if (n > 0 && !rec_off) return io_fail(NPORE_IO_ERR_ARG, "null argument");
    return bam_format_impl(n, n_threads, names, name_off, flag, ref_id, n_refs, pos, end, mapq, rle, rle_off, seq_ascii, qual_ascii,
                           seq_off, has_qual, hp, out, out_capacity, rec_off);
}

}  // extern "C"
