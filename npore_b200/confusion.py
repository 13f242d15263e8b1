"""Basecaller confusion matrices on the GPU -- host side of npore_confusion_batch (include/npore_b200.h).

Mirrors /root/reference/src/bam.pyx: get_ranges (149-164), calc_confusion_matrices (351-510) and
get_confusion_matrices (168-205).  The reference counts from the text of `samtools mpileup`; this path feeds the
alignments (position, CIGAR, bases, qualities) to the device, which derives the same events (npore_b200/csrc/confusion.cuh).

Two host paths: calc_confusion_matrices_batch packs given reads (load_alignments decodes a whole BAM file in Python, for small
files and tests); count_bam streams a BAM file of any size through the native reader, in BAM's own 4-bit packing.
"""
import os

import numpy as np

from . import cfg
from .aln import _engine

SKIP_FLAGS = 0x4 | 0x100 | 0x200 | 0x400      # samtools mpileup --ff default: UNMAP, SECONDARY, QCFAIL, DUP
_REF_OPS = np.zeros(16, dtype=bool)
_REF_OPS[[0, 2, 3, 7, 8]] = True


class AlignedReads:
    """The reads of one contig as flat arrays, coordinate sorted (stable, i.e. BAM order for equal positions)."""

    def __init__(self, records):
        """records: iterable of (pos, cigar, seq, qual, flag) with cigar = uint32 BAM words or [(len, op char)],
        seq = str, qual = uint8 array / bytes / None (stored without qualities)."""
        recs = [r for r in records if not (r[4] & SKIP_FLAGS)]
        recs.sort(key=lambda r: r[0])
        n = len(recs)
        words = []
        for r in recs:
            c = r[1]
            if not isinstance(c, np.ndarray):
                c = np.array([(int(k) << 4) | cfg.cigar_dict[op] for k, op in c], dtype=np.uint32)
            words.append(c.astype(np.uint32, copy=False))
        self.pos = np.array([r[0] for r in recs], dtype=np.int64)
        self.cigar_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum([len(w) for w in words], out=self.cigar_off[1:])
        self.cigar_rle = np.concatenate(words) if n and self.cigar_off[-1] else np.zeros(0, np.uint32)
        self.seq_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum([len(r[2]) for r in recs], out=self.seq_off[1:])
        self.seq_ascii = np.frombuffer("".join(r[2] for r in recs).encode("latin-1"), dtype=np.uint8)
        q = [np.full(len(r[2]), 255, np.uint8) if r[3] is None else np.frombuffer(bytes(r[3]), dtype=np.uint8) for r in recs]
        self.qual = np.concatenate(q) if n and self.seq_off[-1] else np.zeros(0, np.uint8)
        span = np.where(_REF_OPS[self.cigar_rle & 15], self.cigar_rle >> 4, 0).astype(np.int64)
        csum = np.concatenate(([0], np.cumsum(span)))
        self.end = self.pos + (csum[self.cigar_off[1:]] - csum[self.cigar_off[:-1]])
        self.maxend = np.maximum.accumulate(self.end) if n else self.end

    def __len__(self):
        return len(self.pos)

    def overlapping(self, start, end):
        """Indices (ascending) of the reads with pos < end and end > start."""
        hi = int(np.searchsorted(self.pos, end, "left"))
        lo = int(np.searchsorted(self.maxend[:hi], start, "right"))
        return lo + np.flatnonzero(self.end[lo:hi] > start)


class PileupPack:
    """The arrays of one npore_pileup_batch."""

    def __init__(self, ranges, refs, reads, max_n, min_base_q=13):
        """ranges: [(ctg, start, end)]; refs: {ctg: str}; reads: {ctg: AlignedReads}."""
        ctgs = sorted({c for c, _, _ in ranges})
        base, off = {}, 0
        for c in ctgs:
            base[c] = off
            off += len(reads[c]) if c in reads else 0
        have = [reads[c] for c in ctgs if c in reads and len(reads[c])]
        cat = lambda xs, dt: np.concatenate(xs) if xs else np.zeros(0, dt)   # noqa: E731
        self.read_pos = cat([a.pos for a in have], np.int64)
        self.seq_ascii = cat([a.seq_ascii for a in have], np.uint8)
        self.qual = cat([a.qual for a in have], np.uint8)
        self.cigar_rle = cat([a.cigar_rle for a in have], np.uint32)
        self.seq_off = np.zeros(len(self.read_pos) + 1, np.int64)
        self.cigar_off = np.zeros(len(self.read_pos) + 1, np.int64)
        k = so = co = 0
        for a in have:
            self.seq_off[k + 1:k + 1 + len(a)] = a.seq_off[1:] + so
            self.cigar_off[k + 1:k + 1 + len(a)] = a.cigar_off[1:] + co
            k += len(a); so += int(a.seq_off[-1]); co += int(a.cigar_off[-1])
        self.range_start = np.array([s for _, s, _ in ranges], dtype=np.int64)
        self.range_end = np.array([e for _, _, e in ranges], dtype=np.int64)
        chunks, lists = [], []
        for c, s, e in ranges:
            contig = refs[c]
            if not (0 <= s < e <= len(contig)):
                raise ValueError(f"range {c}:{s}-{e} outside the contig (length {len(contig)})")
            chunks.append(contig[s:min(len(contig), e + 1 + max_n)])
            lists.append((reads[c].overlapping(s, e) + base[c]).astype(np.int32) if c in reads and len(reads[c]) else np.zeros(0, np.int32))
        self.ref_off = np.zeros(len(ranges) + 1, np.int64)
        np.cumsum([len(x) for x in chunks], out=self.ref_off[1:])
        self.ref_ascii = np.frombuffer("".join(chunks).encode("latin-1"), dtype=np.uint8)
        self.range_reads_off = np.zeros(len(ranges) + 1, np.int64)
        np.cumsum([len(x) for x in lists], out=self.range_reads_off[1:])
        self.range_reads = cat(lists, np.int32)
        self.min_base_q = min_base_q


def get_ranges(regions):
    """bam.pyx:149-164: cut every (contig, start, stop) into chunk_width windows."""
    w = int(cfg.args.chunk_width)
    return [(ctg, s, min(stop, s + w)) for ctg, start, stop in regions for s in range(start, stop, w)]


def _np_engine():
    z = np.zeros((int(cfg.args.max_n), int(cfg.args.max_l) + 1, int(cfg.args.max_l) + 1), np.float32)
    return _engine(np.zeros((5, 5), np.float32), z, 5, 1, 20000, 30)


def load_alignments(bam_fn):
    """{contig: AlignedReads} from a BAM file (npore_b200/bamio.py reader; no pysam / samtools)."""
    from .bamio import read_bam
    _, refs, recs = read_bam(bam_fn)
    per = {}
    for r in recs:
        if r["ref_id"] >= 0:
            per.setdefault(refs[r["ref_id"]][0], []).append((r["pos"], r["cigar"], r["seq"], r["qual"], r["flag"]))
    return {c: AlignedReads(v) for c, v in per.items()}


def calc_confusion_matrices_batch(ranges, refs=None, reads=None, min_base_q=13):
    """Sum of calc_confusion_matrices over `ranges` in one device call: (subs, nps, inss, dels), int64."""
    refs = cfg.args.refs if refs is None else refs
    if reads is None:
        reads = getattr(cfg.args, "_alignments", None)
        if reads is None:
            reads = cfg.args._alignments = load_alignments(cfg.args.bam)
    return _np_engine().confusion_batch(PileupPack(list(ranges), refs, reads, int(cfg.args.max_n), min_base_q))


def _take(buf, off, sel):
    """Segments sel (ascending) of a buffer whose segment i is buf[off[i]:off[i+1]]: (concatenation, its offsets).  One slice
    per run of consecutive indices, so a batch or carry that is mostly contiguous costs a few memcpys, and a single run (a
    batch whose reads follow each other in the carry, the usual case) is a view: the carry's buffers are never written in place."""
    lens = off[sel + 1] - off[sel]
    new_off = np.zeros(len(sel) + 1, np.int64)
    np.cumsum(lens, out=new_off[1:])
    if not len(sel):
        return buf[:0].copy(), new_off
    cut = np.flatnonzero(np.diff(sel) != 1) + 1
    first, last = sel[np.concatenate(([0], cut))], sel[np.concatenate((cut - 1, [len(sel) - 1]))]
    parts = [buf[a:b] for a, b in zip(off[first].tolist(), off[last + 1].tolist())]
    return (parts[0] if len(parts) == 1 else np.concatenate(parts)), new_off


class _Carry:
    """Kept records of count_bam that a pending range still overlaps, in stream order: columns plus three variable-length
    buffers -- 4-bit bases (whole bytes per record, `nib_par` = the first base is a low nibble), phred+33 qualities and
    CIGAR words without S / H -- each with [n+1] offsets."""
    COLS = ("tid", "pos", "end", "has_qual", "nib_par")
    BUFS = (("nib", np.uint8), ("qual", np.uint8), ("cig", np.uint32))

    def __init__(self):
        for k in self.COLS:
            setattr(self, k, np.zeros(0, np.int64))
        for k, dt in self.BUFS:
            setattr(self, k, np.zeros(0, dt))
            setattr(self, k + "_off", np.zeros(1, np.int64))

    def __len__(self):
        return len(self.pos)

    def append(self, cols, bufs):
        """cols: {COLS: arrays}; bufs: {name: (buffer, offsets)} of the new records (after the present ones in the stream)."""
        for k in self.COLS:
            setattr(self, k, np.concatenate((getattr(self, k), cols[k])))
        for k, _ in self.BUFS:
            buf, off = getattr(self, k), getattr(self, k + "_off")
            nb, no = bufs[k]
            setattr(self, k, np.concatenate((buf, nb[:int(no[-1])])))
            setattr(self, k + "_off", np.concatenate((off, no[1:] + off[-1])))

    def take(self, sel):
        """(columns, {name: (buffer, offsets)}) of records sel (ascending)."""
        return ({k: getattr(self, k)[sel] for k in self.COLS},
                {k: _take(getattr(self, k), getattr(self, k + "_off"), sel) for k, _ in self.BUFS})

    def keep(self, sel):
        cols, bufs = self.take(sel)
        for k in self.COLS:
            setattr(self, k, cols[k])
        for k, _ in self.BUFS:
            setattr(self, k, bufs[k][0])
            setattr(self, k + "_off", bufs[k][1])


def _overlaps_any(tid, pos, end, r_tid, r_start, r_end):
    """Per read: does any of the ranges overlap it (pos < range end and end > range start, as AlignedReads.overlapping)?"""
    if not len(r_tid) or not len(tid):
        return np.zeros(len(tid), bool)
    o = np.lexsort((r_start, r_tid))
    k_start = (r_tid[o] << 32) | r_start[o]
    k_end = np.maximum.accumulate((r_tid[o] << 32) | r_end[o])      # ranges of earlier contigs sort below every read key
    i = np.searchsorted(k_start, (tid << 32) | end, "left")           # ranges with start < end on the read's contig (or before)
    return (i > 0) & (k_end[np.maximum(i - 1, 0)] > ((tid << 32) | pos))


class _StreamPack:
    """One npore_pileup_batch in the nibble form (PileupPack's attributes plus seq_nib, seq_nib_start, has_qual)."""

    def __init__(self, range_start, range_end, ref_chunks, lists, cols, bufs, min_base_q):
        self.range_start = np.asarray(range_start, np.int64)
        self.range_end = np.asarray(range_end, np.int64)
        self.ref_off = np.zeros(len(ref_chunks) + 1, np.int64)
        np.cumsum([len(x) for x in ref_chunks], out=self.ref_off[1:])
        self.ref_ascii = np.frombuffer(b"".join(ref_chunks), dtype=np.uint8)
        self.read_pos = cols["pos"]
        self.seq_ascii = None
        self.seq_nib, nib_off = bufs["nib"]
        self.seq_nib_start = 2 * nib_off[:-1] + cols["nib_par"]
        self.qual, self.seq_off = bufs["qual"]
        self.has_qual = cols["has_qual"].astype(np.int32)
        self.cigar_rle, self.cigar_off = bufs["cig"]
        self.range_reads_off = np.zeros(len(lists) + 1, np.int64)
        np.cumsum([len(x) for x in lists], out=self.range_reads_off[1:])
        self.range_reads = np.concatenate(lists).astype(np.int32) if lists else np.zeros(0, np.int32)
        self.min_base_q = min_base_q


def count_bam(bam_fn, refs, regions=None, min_base_q=13, window_bytes=16 << 20, max_batch_bases=256 << 20, n_threads=0,
              timings=None):
    """calc_confusion_matrices_batch(get_ranges(regions), refs, load_alignments(bam_fn), min_base_q) in one streamed pass over a
    coordinate-sorted BAM file: (subs, nps, inss, dels), int64.  Host memory stays bounded by the window and by the reads of the
    ranges in flight, not by the file.

    refs: {contig: sequence} or a FASTA path.  regions: [(contig, start, stop)]; None = every contig of the BAM header, whole.
    The file is read in windows of ~window_bytes inflated bytes (NativeBam, inflated ahead in the background).  From each window
    only the kept records (mapped, not flag & SKIP_FLAGS) that overlap a range not yet counted are gathered, in BAM's own
    packing (4-bit bases, phred+33 qualities, CIGAR without clips: the pileup of the clipped ends is empty either way), into a
    carry.  A range is complete once the stream has passed its end; complete ranges are counted on the device in batches of
    at most max_batch_bases read bases (a range with more goes alone), on a worker thread while the next window is gathered.
    Raises ValueError if the file is not coordinate sorted (checked across the whole stream) or a range lies outside its
    contig.  timings (dict) receives host seconds `open` (waits for inflate), `gather`, `pack`, `device_wait` and the counts
    `batches`, `reads`, `bases`."""
    import queue
    import threading
    import time
    from .bamio import NativeBam, read_fasta

    fa = read_fasta(refs) if isinstance(refs, str) else refs
    max_n = int(cfg.args.max_n)
    tm = {"open": 0.0, "gather": 0.0, "pack": 0.0, "device_wait": 0.0, "batches": 0, "reads": 0, "bases": 0}
    t = time.perf_counter()
    bam = NativeBam(bam_fn, n_threads, window_bytes)
    tm["open"] += time.perf_counter() - t
    try:
        names = {nm: i for i, (nm, _) in enumerate(bam.refs)}
        ranges = get_ranges(regions if regions is not None else [(nm, 0, ln) for nm, ln in bam.refs])
        for c, s, e in ranges:
            if c not in fa:
                raise ValueError(f"range {c}:{s}-{e}: contig not in the reference")
            if not (0 <= s < e <= len(fa[c])):
                raise ValueError(f"range {c}:{s}-{e} outside the contig (length {len(fa[c])})")
        # ranges on contigs the BAM does not name have no reads: nothing to count
        keep = [k for k, (c, _, _) in enumerate(ranges) if c in names]
        p_tid = np.array([names[ranges[k][0]] for k in keep], np.int64)
        p_start = np.array([ranges[k][1] for k in keep], np.int64)
        p_end = np.array([ranges[k][2] for k in keep], np.int64)
        p_ctg = [ranges[k][0] for k in keep]
        pending = np.ones(len(keep), bool)
        refb = {}

        T = int(cfg.args.max_l) + 1
        tot = [np.zeros((5, 5), np.int64), np.zeros((max_n, T, T), np.int64), np.zeros(T, np.int64), np.zeros(T, np.int64)]
        jobs, failed = queue.Queue(maxsize=1), []

        def worker():
            eng = None
            while True:
                pk = jobs.get()
                if pk is None:
                    return
                if failed:
                    continue
                try:
                    eng = eng or _np_engine()
                    for acc, m in zip(tot, eng.confusion_batch(pk)):
                        acc += m
                except BaseException as ex:          # noqa: BLE001 -- re-raised on the main thread
                    failed.append(ex)

        def submit(pk):
            t = time.perf_counter()
            jobs.put(pk)
            tm["device_wait"] += time.perf_counter() - t
            if failed:
                raise failed[0]

        def ref_chunk(c, s, e):
            b = refb.get(c)
            if b is None:
                b = refb[c] = fa[c].encode("latin-1")
            return b[s:min(len(b), e + 1 + max_n)]

        def flush(carry, done):
            """Count the complete ranges `done` (indices into the pending arrays) from the carry."""
            if not len(done) or not len(carry):
                return
            t = time.perf_counter()
            ckey = (carry.tid << 32) | carry.pos
            cmax = np.maximum.accumulate((carry.tid << 32) | carry.end)
            rt, rs, re_ = p_tid[done], p_start[done], p_end[done]
            hi = np.searchsorted(ckey, (rt << 32) | re_, "left")                   # reads starting before the range end
            lo = np.minimum(np.searchsorted(cmax, (rt << 32) | rs, "right"), hi)    # ... whose running-max end passes its start
            n_c = hi - lo
            c_off = np.concatenate(([0], np.cumsum(n_c)))
            cand = np.repeat(lo - c_off[:-1], n_c) + np.arange(c_off[-1])
            owner = np.repeat(np.arange(len(done)), n_c)
            hit = carry.end[cand] > rs[owner]
            cand, owner = cand[hit], owner[hit]
            cnt = np.bincount(owner, minlength=len(done))
            slen = carry.qual_off[cand + 1] - carry.qual_off[cand]
            rbases = np.bincount(owner, weights=slen, minlength=len(done)).astype(np.int64)
            l_off = np.concatenate(([0], np.cumsum(cnt)))
            with_reads = np.flatnonzero(cnt)
            tm["pack"] += time.perf_counter() - t
            b0 = 0
            while b0 < len(with_reads):
                b1, acc = b0 + 1, rbases[with_reads[b0]]
                while b1 < len(with_reads) and acc + rbases[with_reads[b1]] <= max_batch_bases:
                    acc += rbases[with_reads[b1]]
                    b1 += 1
                t = time.perf_counter()
                sel = with_reads[b0:b1]
                lists = [cand[l_off[r]:l_off[r + 1]] for r in sel]
                rd = np.unique(np.concatenate(lists))
                cols, bufs = carry.take(rd)
                pk = _StreamPack(rs[sel], re_[sel], [ref_chunk(p_ctg[done[r]], int(rs[r]), int(re_[r])) for r in sel],
                                 [np.searchsorted(rd, x) for x in lists], cols, bufs, min_base_q)
                tm["batches"] += 1
                tm["reads"] += len(rd)
                tm["bases"] += int(pk.seq_off[-1])
                tm["pack"] += time.perf_counter() - t
                submit(pk)
                b0 = b1

        th = threading.Thread(target=worker, name="count_bam-device", daemon=True)
        th.start()
        carry = _Carry()
        last = -1                                    # (tid << 32 | pos) of the last record seen; unmapped (ref_id -1) sort last
        n_refs = len(bam.refs)
        try:
            t = time.perf_counter()
            n = bam.n if not bam.window_bytes else bam.advance()
            tm["open"] += time.perf_counter() - t
            while True:
                if n:
                    t = time.perf_counter()
                    rid = bam.ref_id.astype(np.int64)
                    tid = np.where(rid < 0, n_refs, rid)
                    key = (tid << 32) | np.where(rid < 0, 0, bam.pos.astype(np.int64) + (1 << 31))
                    if key[0] < last or (n > 1 and np.any(key[1:] < key[:-1])):
                        raise ValueError(f"{bam_fn}: records are not coordinate-sorted")
                    last = int(key[-1])
                    ok = (rid >= 0) & ((bam.flag & SKIP_FLAGS) == 0)
                    pos, end = bam.pos.astype(np.int64), bam.end.astype(np.int64)
                    live = np.flatnonzero(pending)
                    ok &= _overlaps_any(tid, pos, end, p_tid[live], p_start[live], p_end[live])
                    sel = np.flatnonzero(ok)
                    if len(sel):
                        nib, nib_start = bam.gather_nib(sel, n_threads)
                        g = bam.gather(sel, n_threads, want_names=False, want_codes=False, want_seq=False)
                        nib_off = np.concatenate((nib_start >> 1, [len(nib)]))
                        carry.append({"tid": tid[sel], "pos": pos[sel], "end": end[sel], "has_qual": bam.has_qual[sel].astype(np.int64),
                                      "nib_par": (nib_start & 1) * (bam.aln_len[sel] > 0)},   # an empty read starts on a byte
                                     {"nib": (nib, nib_off), "qual": (g["qual_ascii"], g["seq_off"]), "cig": (g["cigar"], g["cig_off"])})
                    tm["gather"] += time.perf_counter() - t
                    # complete: the stream has passed the range's end (a later contig, or a record at or after its end)
                    l_tid, l_pos = last >> 32, (last & 0xffffffff) - (1 << 31)
                    done = np.flatnonzero(pending & ((p_tid < l_tid) | ((p_tid == l_tid) & (p_end <= l_pos))))
                else:
                    done = np.flatnonzero(pending)
                flush(carry, done)
                pending[done] = False
                if len(done) and len(carry):
                    t = time.perf_counter()
                    live = np.flatnonzero(pending)
                    carry.keep(np.flatnonzero(_overlaps_any(carry.tid, carry.pos, carry.end, p_tid[live], p_start[live], p_end[live])))
                    tm["pack"] += time.perf_counter() - t
                if not n:
                    break
                t = time.perf_counter()
                n = bam.advance()
                tm["open"] += time.perf_counter() - t
        finally:
            t = time.perf_counter()
            jobs.put(None)
            th.join()
            tm["device_wait"] += time.perf_counter() - t
        if failed:
            raise failed[0]
    finally:
        bam.close()
        if timings is not None:
            timings.update(tm)
    return tuple(tot)


def calc_confusion_matrices(range_tuple):
    """bam.pyx:351-510, same argument and return value (one (ctg, start, end) window)."""
    out = calc_confusion_matrices_batch([range_tuple])
    with cfg.counter.get_lock():
        cfg.counter.value += 1
    return out


def get_confusion_matrices():
    """bam.pyx:168-205: load the cached matrices from stats_dir, or count them from cfg.args.bam over
    get_ranges(cfg.args.regions) (count_bam: one streamed pass over the file instead of a process pool) and cache them."""
    d = cfg.args.stats_dir
    if not getattr(cfg.args, "recalc_cms", False):
        print("> loading confusion matrices")
        return tuple(np.load(os.path.join(d, f"{k}_cm.npy")) for k in ("subs", "nps", "inss", "dels"))
    print("> calculating confusion matrices")
    out = count_bam(cfg.args.bam, cfg.args.refs, cfg.args.regions)
    os.makedirs(d, exist_ok=True)
    for k, m in zip(("subs", "nps", "inss", "dels"), out):
        np.save(os.path.join(d, f"{k}_cm"), m)
    return out
