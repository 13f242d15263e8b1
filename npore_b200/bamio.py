"""BAM / FASTA / SAM I/O without pysam -- the callers either side of the hot path (SURVEY.md 8(f) rows N1, N2).

  read_bam(path)                 BGZF inflate + BAM record decode (SAM spec section 4: `<iiBBHHHiiii` core, 4-bit
                                 `=ACMGRSVTWYHKDBN` bases, `MIDNSHP=XB` op codes)
  get_read_data(bam, fasta, ..)  generator of the 11-tuples of /root/reference/src/bam.pyx:18-47 (same filters: no
                                 secondary / supplementary / unmapped; soft clips stripped from SEQ/QUAL like pysam's
                                 query_alignment_sequence; reference slice = fasta[start:stop].upper(), which is what
                                 get_reference_sequence().upper() yields)
  create_header(...)             bam.pyx:127-145: @HD VN:1.6 SO:coordinate, @SQ per contig, @PG realigner (header_text)
  write_bam(path, ...)           minimal BGZF/BAM writer (fixtures for the tests; records in input order)
  realign_bam(...)               ingest -> GPU batches -> ordered SAM: what realign.py:75-115 does end to end.  Uses the
                                 native reader / writer of libnpore_b200.so (include/npore_bamio.h: multi-threaded BGZF
                                 inflate, record decode into flat arrays, batch SAM formatting) and never builds
                                 per-read Python objects; the pure-Python functions above remain as the tuple API.
                                 out_format="bam" writes the same records as BAM: batch BAM encoding on the host, BGZF
                                 compression on the device (engine.BgzfCompressor); index=True adds the .bai index,
                                 computed on the device batch by batch (BgzfCompressor.index, BaiBuilder).
  read_bai(path).query(..)       a BAM index and the chunks hts_itr_query would read for a region
                                 One batch pipeline (_realign_segments) serves both forms: the streamed windows of one
                                 device, and with devices=[...] one region shard per device (_realign_sharded).
The GPU path is entered through npore_b200.engine (realign_bam) or npore_b200.bam.realign_reads (tuples).
"""
import contextlib
import ctypes as C
import gzip
import io
import os
import queue
import struct
import sys
import threading
import time
import zlib

import numpy as np

from . import cfg

_SEQ16 = "=ACMGRSVTWYHKDBN"
_OPS = "MIDNSHP=XB"
_SEQ_PAIR = np.frombuffer("".join(a + b for a in _SEQ16 for b in _SEQ16).encode(), dtype=np.uint8).reshape(256, 2)
_PIPES = {}                     # _pipeline's cache
_BGZF = {}                      # _compressor's cache
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")   # SAM spec 4.1.2
_PIPE_LOCK = threading.Lock()   # contexts of different devices are created one after the other
_MALLOC_TUNED = False           # _keep_freed_buffers_mapped has run


def read_fasta(path):
    """{contig: sequence} (plain or gzip FASTA)."""
    opener = gzip.open if path.endswith(".gz") else open
    out, name, parts = {}, None, []
    with opener(path, "rt") as fh:
        for line in fh:
            if line.startswith(">"):
                if name is not None:
                    out[name] = "".join(parts)
                name, parts = line[1:].split()[0], []
            else:
                parts.append(line.strip())
    if name is not None:
        out[name] = "".join(parts)
    return out


def _parse_tags(buf):
    tags, p, n = {}, 0, len(buf)
    sizes = {"A": 1, "c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}
    fmts = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I", "f": "<f"}
    while p + 3 <= n:
        tag, typ = buf[p:p + 2].decode(), chr(buf[p + 2])
        p += 3
        if typ == "A":
            tags[tag] = chr(buf[p]); p += 1
        elif typ in fmts:
            tags[tag] = struct.unpack_from(fmts[typ], buf, p)[0]; p += sizes[typ]
        elif typ in "ZH":
            e = buf.index(b"\0", p)
            tags[tag] = buf[p:e].decode(); p = e + 1
        elif typ == "B":
            sub = chr(buf[p]); cnt = struct.unpack_from("<i", buf, p + 1)[0]
            p += 5
            tags[tag] = list(struct.unpack_from("<" + str(cnt) + fmts[sub][1], buf, p)); p += cnt * sizes[sub]
        else:
            break
    return tags


def read_bam(path):
    """Returns (header_text, [(name, length)], iterator of record dicts).  Whole-file inflate (gzip concatenates the
    BGZF members); fine for the batch sizes realign handles per call."""
    with gzip.open(path, "rb") as fh:
        data = fh.read()
    if data[:4] != b"BAM\1":
        raise ValueError(f"{path}: not a BAM file")
    l_text = struct.unpack_from("<i", data, 4)[0]
    text = data[8:8 + l_text].split(b"\0")[0].decode()
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", data, p)[0]; p += 4
    refs = []
    for _ in range(n_ref):
        l_name = struct.unpack_from("<i", data, p)[0]; p += 4
        name = data[p:p + l_name - 1].decode(); p += l_name
        refs.append((name, struct.unpack_from("<i", data, p)[0])); p += 4

    def records(p=p):
        n = len(data)
        while p + 4 <= n:
            block_size = struct.unpack_from("<i", data, p)[0]; p += 4
            ref_id, pos, l_read_name, mapq, _bin, n_cigar, flag, l_seq, _nref, _npos, _tlen = struct.unpack_from("<iiBBHHHiiii", data, p)
            q = p + 32
            name = data[q:q + l_read_name - 1].decode(); q += l_read_name
            cig = np.frombuffer(data, dtype="<u4", count=n_cigar, offset=q); q += 4 * n_cigar
            packed = np.frombuffer(data, dtype=np.uint8, count=(l_seq + 1) // 2, offset=q); q += (l_seq + 1) // 2
            seq = _SEQ_PAIR[packed].tobytes()[:l_seq].decode("latin-1")
            qual = np.frombuffer(data, dtype=np.uint8, count=l_seq, offset=q); q += l_seq
            tags = _parse_tags(data[q:p + block_size])
            yield {"name": name, "flag": flag, "ref_id": ref_id, "pos": pos, "mapq": mapq, "cigar": cig, "seq": seq,
                   "qual": None if (l_seq and qual[0] == 0xFF) else qual, "tags": tags}
            p += block_size
    return text, refs, records()


def _cigar_string(words):
    return "".join(f"{int(w) >> 4}{_OPS[int(w) & 15]}" for w in words)


def get_read_data(bam_fn, fasta, regions=None, max_reads=0):
    """bam.pyx:18-47.  fasta: path or {contig: seq}.  regions: [(contig, start, stop)] or None for everything (a read
    overlapping two regions is yielded once per region, as pysam's fetch does)."""
    if not os.path.exists(bam_fn):
        print(f"\nERROR: BAM file '{bam_fn}' not found.")
        sys.exit(1)
    fa = read_fasta(fasta) if isinstance(fasta, str) else fasta
    _, refs, recs = read_bam(bam_fn)
    recs = list(recs)
    kept = 0
    for ctg, start, stop in (regions or [(None, 0, 1 << 62)]):
        for r in recs:
            if max_reads and kept >= max_reads:
                return
            if r["flag"] & (0x4 | 0x100 | 0x800) or r["ref_id"] < 0:
                continue
            rname = refs[r["ref_id"]][0]
            ops, lens = r["cigar"] & 15, r["cigar"] >> 4
            ref_span = int(lens[np.isin(ops, (0, 2, 3, 7, 8))].sum())
            rstart, rstop = r["pos"], r["pos"] + ref_span
            if ctg is not None and (rname != ctg or rstop <= start or rstart >= stop):
                continue
            # query_alignment_sequence / qualities: soft-clipped ends removed (hard clips are not in SEQ)
            lead = int(lens[0]) if len(ops) and ops[0] == 4 else (int(lens[1]) if len(ops) > 1 and ops[0] == 5 and ops[1] == 4 else 0)
            trail = int(lens[-1]) if len(ops) and ops[-1] == 4 else (int(lens[-2]) if len(ops) > 1 and ops[-1] == 5 and ops[-2] == 4 else 0)
            seq = r["seq"][lead:len(r["seq"]) - trail]
            quals = "*" if r["qual"] is None else (r["qual"][lead:len(r["qual"]) - trail] + np.uint8(33)).tobytes().decode("latin-1")
            if not quals:
                quals = "*"                                             # bam.pyx:42: an empty quality array is falsy
            hp = r["tags"].get("HP")
            kept += 1
            yield (r["name"], r["flag"], rname, rstart, r["mapq"], _cigar_string(r["cigar"]), rstop, seq.upper(), quals,
                   fa[rname][rstart:rstop].upper(), 0 if hp is None else int(hp))


def header_text(refs, argv=None):
    """bam.pyx:127-145: the @HD / @SQ / @PG lines of the output.  refs: [(name, length)]."""
    lines = ["@HD\tVN:1.6\tSO:coordinate\n"] + [f"@SQ\tSN:{name}\tLN:{length}\n" for name, length in refs]
    lines.append(f"@PG\tID:realigner\tPN:realigner\tVN:{cfg.__version__}\tCL:{' '.join(argv if argv is not None else sys.argv)}\n")
    return "".join(lines)


def create_header(outfile, refs, argv=None):
    """bam.pyx:127-145: (re)creates the SAM with @HD / @SQ / @PG lines.  refs: [(name, length)]."""
    if os.path.dirname(outfile):
        os.makedirs(os.path.dirname(outfile), exist_ok=True)
    with open(outfile, "w") as fh:
        fh.write(header_text(refs, argv))


def bam_header(refs, argv=None):
    """The uncompressed BAM header (SAM spec 4.2): magic, the text of header_text, the reference list."""
    text = header_text(refs, argv).encode()
    out = [b"BAM\1", struct.pack("<i", len(text)), text, struct.pack("<i", len(refs))]
    for name, length in refs:
        out.append(struct.pack("<i", len(name.encode()) + 1) + name.encode() + b"\0" + struct.pack("<i", length))
    return b"".join(out)


class NativeBam:
    """A BAM file opened through libnpore_b200.so (include/npore_bamio.h): header, per-record columns, flat gathers."""

    COLUMNS = ("ref_id", "pos", "end", "flag", "mapq", "aln_len", "n_cigar", "name_len", "hp", "has_qual")

    def __init__(self, path, n_threads=0, window_bytes=0, regions=None):
        """window_bytes == 0: the whole file is loaded now.  window_bytes > 0: nothing is loaded yet; every advance() call
        loads the next ~window_bytes of (inflated) records, so files larger than memory stream through.
        regions: [(contig, start, stop)]; when the file has a BAM index ({path}.bai, else {path without .bam}.bai, as htslib
        looks them up), only the index chunks of the regions are read (npore_bam_restrict): the records are those whose start
        lies in a chunk, a superset of the records overlapping the regions, in file order.  An index older than the BAM is not
        used (the whole file is read then); a malformed one raises ValueError.  self.index: the index file used, or None;
        self.bytes_read: compressed bytes read so far."""
        from ._lib import lib
        self._L = lib()
        h = C.c_void_p()
        rc = self._L.npore_bam_open(os.fsencode(path), n_threads, C.byref(h))
        if rc:
            raise (FileNotFoundError if rc == -1 else ValueError)(f"{path}: {self._L.npore_io_last_error().decode()}")
        self._h = h
        t = C.c_char_p()
        self._L.npore_bam_header_text(h, C.byref(t))
        self.text = (t.value or b"").decode()
        self.refs = []
        for i in range(self._L.npore_bam_n_refs(h)):
            name, length = C.c_char_p(), C.c_int64()
            self._L.npore_bam_ref(h, i, C.byref(name), C.byref(length))
            self.refs.append((name.value.decode(), int(length.value)))
        self.window_bytes = int(window_bytes)
        self.n = 0
        for k in self.COLUMNS:
            setattr(self, k, np.zeros(0, np.int32))
        self.index = find_index(path) if regions else None
        if self.index is not None:
            ch = region_chunks(read_bai(self.index), self.refs, regions)
            beg, end = np.ascontiguousarray(ch[:, 0]), np.ascontiguousarray(ch[:, 1])
            if self._L.npore_bam_restrict(h, len(ch), beg.ctypes.data, end.ctypes.data):
                raise ValueError(f"{self.index}: {self._L.npore_io_last_error().decode()}")
        if not self.window_bytes:
            self.advance()

    @property
    def bytes_read(self):
        """BGZF member bytes read from the file so far."""
        return int(self._L.npore_bam_bytes_read(self._h))

    def voffsets(self):
        """Virtual offset of every record of the current window (uint64)."""
        out = np.zeros(max(self.n, 1), np.uint64)
        self._L.npore_bam_voffsets(self._h, out.ctypes.data)
        return out[:self.n]

    def advance(self):
        """Load the next window; returns the number of records in it (0 at end of file)."""
        n = int(self._L.npore_bam_advance(self._h, self.window_bytes))
        if n < 0:
            raise ValueError(self._L.npore_io_last_error().decode())
        self.n = n
        cols = {k: np.zeros(max(n, 1), np.int32) for k in self.COLUMNS}
        self._L.npore_bam_columns(self._h, *[cols[k].ctypes.data for k in self.COLUMNS])
        for k, v in cols.items():
            setattr(self, k, v[:n])
        if n and self.window_bytes:          # streaming: the next window inflates in the background while this one is gathered
            self._L.npore_bam_prefetch(self._h, self.window_bytes)
        return n

    def close(self):
        if getattr(self, "_h", None):
            self._L.npore_bam_close(self._h)
            self._h = None

    __del__ = close

    def gather_nib(self, sel, n_threads=0):
        """The selected records' aligned bases as they lie in the file (4 bits per base): (nib uint8, nib_start int64[n]) for
        PackedBatch.from_flat_shared_nib -- no per-base work on the host."""
        sel = np.ascontiguousarray(sel, dtype=np.int64)
        boff = np.zeros(len(sel) + 1, np.int64)
        ps = sel.ctypes.data if len(sel) else None
        if self._L.npore_bam_gather_nib(self._h, len(sel), ps, n_threads, boff.ctypes.data, None, None):
            raise RuntimeError(self._L.npore_io_last_error().decode())
        nib = np.empty(max(int(boff[-1]), 1), np.uint8)
        start = np.zeros(max(len(sel), 1), np.int64)
        if self._L.npore_bam_gather_nib(self._h, len(sel), ps, n_threads, boff.ctypes.data, nib.ctypes.data, start.ctypes.data):
            raise RuntimeError(self._L.npore_io_last_error().decode())
        return nib[:int(boff[-1])], start[:len(sel)]

    def gather_cigar(self, sel, n_threads=0):
        """Only the CIGAR words of the selected records (S / H dropped): (words uint32, offsets int64[n+1])."""
        sel = np.ascontiguousarray(sel, dtype=np.int64)
        off = np.concatenate(([0], np.cumsum(self.n_cigar[sel], dtype=np.int64)))
        cig = np.empty(max(int(off[-1]), 1), np.uint32)
        rc = self._L.npore_bam_gather(self._h, len(sel), sel.ctypes.data if len(sel) else None, n_threads, None, None, None, None,
                                      cig.ctypes.data, off.ctypes.data, None, None)
        if rc:
            raise RuntimeError(self._L.npore_io_last_error().decode())
        return cig[:int(off[-1])], off

    def gather(self, sel, n_threads=0, want_qual=True, want_names=True, want_codes=True, want_cigar=True, want_seq=True):
        """Flat arrays of the selected records: dict with seq_ascii, seq_codes, qual_ascii, seq_off, cigar, cig_off, names,
        name_off (soft clips removed, S/H dropped from the CIGAR; bam.pyx:41-44, 59).  want_seq=False: no seq_ascii (None),
        so that e.g. a qualities-only gather does no per-base decode.  qual_ascii of a record without qualities (has_qual 0)
        is left unwritten."""
        sel = np.ascontiguousarray(sel, dtype=np.int64)
        off = lambda col: np.concatenate(([0], np.cumsum(col[sel], dtype=np.int64)))   # noqa: E731
        o = {"seq_off": off(self.aln_len), "cig_off": off(self.n_cigar), "name_off": off(self.name_len)}
        o["seq_ascii"] = np.empty(max(int(o["seq_off"][-1]), 1), np.uint8) if want_seq else None
        o["seq_codes"] = np.empty(max(int(o["seq_off"][-1]), 1), np.uint8) if want_codes else None
        o["qual_ascii"] = np.empty(max(int(o["seq_off"][-1]), 1), np.uint8) if want_qual else None
        o["cigar"] = np.empty(max(int(o["cig_off"][-1]), 1), np.uint32) if want_cigar else None
        o["names"] = np.empty(max(int(o["name_off"][-1]), 1), np.uint8) if want_names else None
        ptr = lambda a: None if a is None else a.ctypes.data   # noqa: E731
        rc = self._L.npore_bam_gather(self._h, len(sel), ptr(sel) if len(sel) else None, n_threads, ptr(o["seq_ascii"]), ptr(o["seq_codes"]),
                                      ptr(o["qual_ascii"]), ptr(o["seq_off"]), ptr(o["cigar"]), ptr(o["cig_off"]), ptr(o["names"]), ptr(o["name_off"]))
        if rc:
            raise RuntimeError(self._L.npore_io_last_error().decode())
        return o


def format_sam(bam, sel, g, rle, rle_off, n_threads=0, cols=None, fd=None, offset=0, binary=False, offsets=False):
    """bam.pyx:83 for the selected records as one bytes-like block (npore_sam_format).  cols: the records' column values
    taken earlier (dict of int32 arrays: flag ref_id pos end mapq has_qual hp) when the reader has moved on since.
    fd: also append the block to that file descriptor at `offset` while formatting (npore_sam_format_fd).
    binary: the same records as uncompressed BAM records instead (npore_bam_format; fd must be None).
    offsets (with binary): returns (block, rec_off) with every record's offset in the block and the block length at the end
    (npore_bam_format_offsets)."""
    L = bam._L
    names = "".join(n for n, _ in bam.refs).encode()
    rn_off = np.concatenate(([0], np.cumsum([len(n.encode()) for n, _ in bam.refs], dtype=np.int64)))
    rn = np.frombuffer(names, dtype=np.uint8) if names else np.zeros(1, np.uint8)
    rle = np.ascontiguousarray(rle, dtype=np.uint32)
    rle_off = np.ascontiguousarray(rle_off, dtype=np.int64)
    if cols is None:
        cols = take_columns(bam, sel)
    n = len(cols["flag"])
    if binary:
        cap = int(L.npore_bam_bound(n, g["name_off"].ctypes.data, g["seq_off"].ctypes.data, rle_off.ctypes.data))
    else:
        cap = int(L.npore_sam_bound(n, g["name_off"].ctypes.data, g["seq_off"].ctypes.data, rle_off.ctypes.data, max([len(x) for x, _ in bam.refs] + [1])))
    out = np.empty(max(cap, 1), np.uint8)
    flag, ref_id, pos, end, mapq, hq, hp = (cols[k] for k in ("flag", "ref_id", "pos", "end", "mapq", "has_qual", "hp"))
    qual = g["qual_ascii"] if g["qual_ascii"] is not None else g["seq_ascii"]
    if g["qual_ascii"] is None:
        hq = np.zeros_like(hq)
    args = (n, n_threads, g["names"].ctypes.data, g["name_off"].ctypes.data, flag.ctypes.data, ref_id.ctypes.data,
            rn.ctypes.data, rn_off.ctypes.data, len(bam.refs), pos.ctypes.data, end.ctypes.data, mapq.ctypes.data,
            rle.ctypes.data if len(rle) else None, rle_off.ctypes.data, g["seq_ascii"].ctypes.data, qual.ctypes.data,
            g["seq_off"].ctypes.data, hq.ctypes.data, hp.ctypes.data, out.ctypes.data, cap)
    rec_off = None
    if binary and offsets:
        rec_off = np.zeros(n + 1, np.int64)
        got = L.npore_bam_format_offsets(*args, rec_off.ctypes.data)
    elif binary:
        got = L.npore_bam_format(*args)
    else:
        got = L.npore_sam_format(*args) if fd is None else L.npore_sam_format_fd(*args, int(fd), int(offset))
    if got < 0:
        raise RuntimeError(L.npore_io_last_error().decode())
    return (out[:got], rec_off) if rec_off is not None else out[:got]


def take_columns(bam, sel):
    return {k: np.ascontiguousarray(getattr(bam, k)[sel], dtype=np.int32) for k in ("flag", "ref_id", "pos", "end", "mapq", "has_qual", "hp")}


def find_index(path):
    """The BAM index of path that htslib would use ({path}.bai, then {path without .bam}.bai), if it is not older than the BAM."""
    cands = [f"{path}.bai"] + ([f"{path[:-4]}.bai"] if path.endswith(".bam") else [])
    for c in cands:
        if os.path.exists(c):
            return c if os.path.getmtime(c) >= os.path.getmtime(path) else None
    return None


def region_chunks(bai, refs, regions):
    """The union of the index chunks of every region, sorted and merged: uint64 array (k, 2)."""
    names = {n: k for k, (n, _) in enumerate(refs)}
    got = [bai.query(names[c], int(a), int(b)) for c, a, b in regions if c in names]
    c = np.concatenate(got) if got else np.zeros((0, 2), np.uint64)
    c = c[np.argsort(c[:, 0], kind="stable")]
    out = []
    for b, e in c.tolist():
        if out and b <= out[-1][1]:
            out[-1][1] = max(out[-1][1], e)
        else:
            out.append([b, e])
    return np.array(out, np.uint64).reshape(-1, 2)


def _in_coordinate_order(bam, segments):
    """segments, checked to select records in (ref_id, pos) order: an index needs a sorted file.  A read overlapping two regions
    is selected once per region (bam.pyx:27-28), and its second copy would follow reads that start after it."""
    last = (-1, -1)
    for ctg, sel in segments:
        pos = bam.pos[sel]
        first = (int(bam.ref_id[sel[0]]), int(pos[0]))
        if first < last or (len(pos) > 1 and bool((pos[1:] < pos[:-1]).any())):
            raise ValueError(f"index=True: the records selected in {ctg} are not in coordinate order after the earlier ones (a read "
                             "overlapping two regions is written once per region, or the input is not sorted); the output cannot be indexed")
        last = (first[0], int(pos[-1]))
        yield ctg, sel


def select_reads(bam, regions=None, max_reads=0):
    """Record indices per region like bam.pyx:26-32: fetch(ctg, start, stop) order, no secondary / supplementary /
    unmapped reads, at most max_reads in total.  Yields (contig, indices)."""
    ok = ((bam.flag & (0x4 | 0x100 | 0x800)) == 0) & (bam.ref_id >= 0)
    names = [n for n, _ in bam.refs]
    kept = 0
    for ctg, start, stop in (regions or [(n, 0, l) for n, l in bam.refs]):
        if ctg not in names:
            continue
        sel = np.flatnonzero(ok & (bam.ref_id == names.index(ctg)) & (bam.pos < stop) & (bam.end > start))
        if max_reads:
            sel = sel[:max(0, max_reads - kept)]
        kept += len(sel)
        if len(sel):
            yield ctg, sel


# ------------------------------------------------------------------------------------------------ BAM index (SAM spec 5.2)
BAI_MAX_REF = (1 << 29) - 1             # the BAI binning scheme covers positions below 2^29
_PSEUDO_BIN = 37450
_UNSET = np.uint64(0xFFFFFFFFFFFFFFFF)


def reg2bins(beg, end):
    """Bins that may hold records overlapping [beg, end) (hts_reg2bins, 14-bit windows, 5 levels)."""
    beg, end = max(int(beg), 0), min(int(end), 1 << 29)
    if end <= beg:
        return []
    end -= 1
    out = []
    for off, shift in ((0, 29), (1, 26), (9, 23), (73, 20), (585, 17), (4681, 14)):
        out.extend(range(off + (beg >> shift), off + (end >> shift) + 1))
    return out


class BaiBuilder:
    """Folds the index lists of BgzfCompressor.index (one per written batch, in file order) into a .bai file.  Lists are kept
    as they arrive (they are small: a chunk per run of records with one bin, a few windows per batch) and folded once in
    to_bytes(): the chunks of one bin are appended in file order and merged when the previous one ends in the BGZF member
    where the next begins; the first value set in a 16 kb window wins; windows no record overlaps take the reference's first
    offset before its first record and the previous window's offset after it (htslib's update_loff).  Bins are written in
    ascending order, the pseudo-bin 37450 (first / last offset, mapped / unmapped counts) last."""

    def __init__(self, n_refs):
        self.n_refs = int(n_refs)
        self.batches = []                 # (lists, shift): offsets are lists' + shift << 16

    def add(self, lists, shift=0):
        self.batches.append((lists, int(shift)))

    def extend(self, other, shift):
        """Appends another builder's lists (e.g. a shard's, relative to its part file) whose file starts at byte `shift`."""
        self.batches.extend((lists, sh + int(shift)) for lists, sh in other.batches)

    def to_bytes(self):
        chunks, refs, wins = [], [], []
        for lists, shift in self.batches:
            sh = np.uint64(shift << 16)
            c = lists["chunks"].astype(np.uint64, copy=True)
            c[:, 2:] += sh
            r = lists["refs"].astype(np.uint64, copy=True)
            r[:, 1:3] += sh
            w = lists["windows"].astype(np.uint64, copy=True)
            w[w != _UNSET] += sh
            at = 0
            for ref, _, _, _, _, wf, nw in r.tolist():        # a batch's windows, reference by reference
                if nw:
                    wins.append((ref, wf, w[at:at + nw]))
                at += nw
            chunks.append(c); refs.append(r)
        c = np.concatenate(chunks) if chunks else np.zeros((0, 4), np.uint64)
        r = np.concatenate(refs) if refs else np.zeros((0, 7), np.uint64)
        c = c[np.lexsort((c[:, 1], c[:, 0]))]                 # stable: file order within (ref_id, bin)
        start = np.ones(len(c), bool)
        start[1:] = (c[1:, 0] != c[:-1, 0]) | (c[1:, 1] != c[:-1, 1]) | ((c[:-1, 3] >> np.uint64(16)) < (c[1:, 2] >> np.uint64(16)))
        first = np.flatnonzero(start)
        last = np.r_[first[1:] - 1, len(c) - 1].astype(np.int64)
        merged = np.stack([c[first, 0], c[first, 1], c[first, 2], c[last, 3]], axis=1) if len(c) else np.zeros((0, 4), np.uint64)
        lin = {}
        for ref, wf, vals in wins:
            cur = lin.setdefault(ref, np.zeros(0, np.uint64))
            need = wf + len(vals)
            if len(cur) < need:
                cur = lin[ref] = np.concatenate([cur, np.full(need - len(cur), _UNSET, np.uint64)])
            seg = cur[wf:need]
            fill = (seg == _UNSET) & (vals != _UNSET)                 # the first value set wins
            seg[fill] = vals[fill]
        out = [b"BAI\1", struct.pack("<i", self.n_refs)]
        bounds = np.searchsorted(merged[:, 0], np.arange(self.n_refs + 1, dtype=np.uint64)) if len(merged) else np.zeros(self.n_refs + 1, np.int64)
        for ref in range(self.n_refs):
            rows = r[r[:, 0] == ref]
            if not len(rows):
                out.append(struct.pack("<ii", 0, 0))
                continue
            m = merged[bounds[ref]:bounds[ref + 1]]
            bins, at, cnt = np.unique(m[:, 1], return_index=True, return_counts=True)
            out.append(struct.pack("<i", len(bins) + 1))
            for b, a, k in zip(bins.tolist(), at.tolist(), cnt.tolist()):
                out.append(struct.pack("<Ii", b, k) + np.ascontiguousarray(m[a:a + k, 2:4]).astype("<u8").tobytes())
            beg, end = int(rows[0, 1]), int(rows[-1, 2])
            out.append(struct.pack("<IiQQQQ", _PSEUDO_BIN, 2, beg, end, int(rows[:, 3].sum()), int(rows[:, 4].sum())))
            li = lin.get(ref, np.zeros(0, np.uint64)).copy()
            prev = np.uint64(beg)
            for k in range(len(li)):                                   # update_loff
                if li[k] == _UNSET:
                    li[k] = prev
                prev = li[k]
            out.append(struct.pack("<i", len(li)) + li.astype("<u8").tobytes())
        out.append(struct.pack("<Q", 0))                               # n_no_coor: every record written has a reference
        return b"".join(out)

    def write(self, path):
        """Writes the index atomically (a temporary file renamed over `path`)."""
        tmp = f"{path}.tmp{os.getpid()}"
        try:
            with open(tmp, "wb") as fh:
                fh.write(self.to_bytes())
            os.replace(tmp, path)
        finally:
            with contextlib.suppress(FileNotFoundError):
                os.remove(tmp)


class Bai:
    """A parsed .bai file (read_bai): refs[i] = (bins {bin: uint64 array (k, 2) of (vbeg, vend)}, linear uint64 array,
    meta (first vbeg, last vend, mapped, unmapped) or None)."""

    def __init__(self, refs, n_no_coor):
        self.refs, self.n_no_coor = refs, n_no_coor

    def query(self, ref_id, beg, end):
        """Chunks (uint64 array (k, 2) of vbeg, vend; sorted, overlapping ones merged) that hold every record of reference
        ref_id overlapping [beg, end) -- what htslib's hts_itr_query reads: the chunks of reg2bins(beg, end), less those ending
        before the linear-index offset of window beg >> 14."""
        if not 0 <= ref_id < len(self.refs):
            return np.zeros((0, 2), np.uint64)
        bins, lin, _ = self.refs[ref_id]
        got = [bins[b] for b in reg2bins(beg, end) if b in bins]
        if not got:
            return np.zeros((0, 2), np.uint64)
        c = np.concatenate(got)
        w = max(int(beg), 0) >> 14
        min_off = lin[min(w, len(lin) - 1)] if len(lin) else np.uint64(0)
        c = c[c[:, 1] > min_off]
        c = c[np.argsort(c[:, 0], kind="stable")]
        out = []
        for b, e in c.tolist():
            if out and b <= out[-1][1]:
                out[-1][1] = max(out[-1][1], e)
            else:
                out.append([b, e])
        return np.array(out, np.uint64).reshape(-1, 2)


def read_bai(path):
    """Parses a BAM index (SAM spec 5.2) into a Bai.  A malformed file raises ValueError naming it."""
    data = open(path, "rb").read()
    p = 0

    def take(fmt):
        nonlocal p
        n = struct.calcsize(fmt)
        if p + n > len(data):
            raise ValueError(f"{path}: truncated BAM index")
        v = struct.unpack_from(fmt, data, p)
        p += n
        return v

    if data[:4] != b"BAI\1":
        raise ValueError(f"{path}: not a BAM index (bad magic)")
    p = 4
    (n_ref,) = take("<i")
    if n_ref < 0:
        raise ValueError(f"{path}: negative reference count")
    refs = []
    for _ in range(n_ref):
        (n_bin,) = take("<i")
        if n_bin < 0:
            raise ValueError(f"{path}: negative bin count")
        bins, meta = {}, None
        for _ in range(n_bin):
            b, n_chunk = take("<Ii")
            if n_chunk < 0 or p + 16 * n_chunk > len(data):
                raise ValueError(f"{path}: truncated BAM index")
            c = np.frombuffer(data, "<u8", 2 * n_chunk, p).reshape(-1, 2).astype(np.uint64)
            p += 16 * n_chunk
            if b == _PSEUDO_BIN:
                if n_chunk != 2:
                    raise ValueError(f"{path}: pseudo-bin {_PSEUDO_BIN} without two chunks")
                meta = tuple(int(x) for x in c.reshape(-1))
            elif b > _PSEUDO_BIN:
                raise ValueError(f"{path}: bin {b} out of range")
            else:
                bins[b] = c
        (n_intv,) = take("<i")
        if n_intv < 0 or p + 8 * n_intv > len(data):
            raise ValueError(f"{path}: truncated BAM index")
        lin = np.frombuffer(data, "<u8", n_intv, p).astype(np.uint64)
        p += 8 * n_intv
        refs.append((bins, lin, meta))
    n_no_coor = take("<Q")[0] if p + 8 <= len(data) else None
    if p != len(data):
        raise ValueError(f"{path}: trailing bytes after the BAM index")
    return Bai(refs, n_no_coor)


def _check_indexable(refs, regions):
    """index=True: the references must fit the BAI binning, and regions must be in header order without overlaps (a read that
    still overlaps two of them is caught later, by _in_coordinate_order)."""
    for name, length in refs:
        if length > BAI_MAX_REF:
            raise ValueError(f"index=True: contig {name} is {length} bp; a BAI index covers at most {BAI_MAX_REF} bp (CSI is not supported)")
    order = {name: k for k, (name, _) in enumerate(refs)}
    prev = None
    for ctg, start, stop in regions or []:
        if ctg not in order:
            continue
        key = (order[ctg], int(start), int(stop))
        if prev is not None and (key[0] < prev[0] or (key[0] == prev[0] and key[1] < prev[2])):
            raise ValueError(f"index=True: regions must be in header contig order and must not overlap ({ctg}:{start}-{stop} follows "
                             f"{refs[prev[0]][0]}:{prev[1]}-{prev[2]}); the output would not be sorted")
        prev = key


def _pipeline(sub, npt, n_inflight, device=None):
    """Cached PipelinedRealigner per (tables, cfg, device) (same idea as aln._engine)."""
    from .engine import PipelinedRealigner
    dev = int(getattr(cfg.args, "device", 0) or 0) if device is None else int(device)
    key = (np.asarray(sub, np.float32).tobytes(), hash(np.asarray(npt, np.float32).tobytes()), int(cfg.args.max_n), int(cfg.args.max_l), n_inflight)
    for old in [k for k in _PIPES if k[0] != key]:          # tables / cfg changed: drop every cached pipeline
        _PIPES.pop(old).close()
    p = _PIPES.get((key, dev))
    if p is None:
        p = _PIPES[(key, dev)] = PipelinedRealigner(sub, npt, n_inflight=n_inflight, max_n=int(cfg.args.max_n), max_l=int(cfg.args.max_l), device=dev)
    return p


def _compressor(device, slot):
    """Cached BgzfCompressor per (device, writer slot): the writer threads that run at the same time use different slots."""
    from .engine import BgzfCompressor
    dev = int(getattr(cfg.args, "device", 0) or 0) if device is None else int(device)
    with _PIPE_LOCK:
        z = _BGZF.get((dev, slot))
        if z is None:
            z = _BGZF[(dev, slot)] = BgzfCompressor(dev)
    return z


def _write_all(fd, data, offset):
    view = memoryview(data).cast("B")
    while len(view):
        n = os.pwrite(fd, view, offset)
        view, offset = view[n:], offset + n
    return offset


def _record_ops(bam, sel):
    """D/I ops of each selected record (reference span + aligned read length), from the record columns alone."""
    return (bam.end[sel] - bam.pos[sel]).astype(np.int64) + bam.aln_len[sel]


def _read_loads(bam, sel, max_b_rows=20000, r=30):
    """Cell updates per selected record (SURVEY.md 8(d)): (Lref + Lseq + n_chunks) * (2r+1)."""
    ops = _record_ops(bam, sel)
    return (ops + -(-ops // (max_b_rows - 1))) * (2 * r + 1)


def _realign_segments(bam, segments, fa, pipe, open_out, tm, n_threads, nt_text, max_batch_ops, n_inflight, mark, t0, compressor=None,
                      bai=None):
    """The three-stage pipeline over (contig, record indices) segments, which may be produced lazily: gather batch k+1 while
    batch k is on the GPU and a writer thread formats batch k-1 and appends it to the file descriptor that open_out() returns.
    The writer calls open_out(z) before its first batch and writes from the descriptor's current size on.  compressor: None
    writes SAM text (z is None); otherwise a callable that returns the writer's BgzfCompressor z, and every batch is written as
    BAM records compressed into BGZF members (tm["compress"]: seconds in the compressor).  The descriptor must
    not be in append mode: Linux ignores the offset of a pwrite on an append-mode descriptor, and the formatter threads place
    their slices by offset.  bai (with a compressor): a BaiBuilder that receives every batch's index lists, computed on the
    device right after the batch is written (z.index, tm["index"]: seconds, tm["index_device_ms"]: its kernel milliseconds); the
    records must then be selected in coordinate order (ValueError otherwise).  Records are written in segment order and counted into cfg.counter batch by batch.  n_threads:
    threads of the nibble / CIGAR gathers and of formatting; nt_text: threads of the SAM-text gather that runs beside the
    GPU.  tm receives seconds per phase, mark(event) a trace event per step (GPU times in them count from perf_counter() = t0).
    Returns the records written."""
    from .aln import _report
    from .cig import bases_to_int
    from .engine import NPORE_OUT_NO_EXPANDED, NPORE_OUT_RLE, NPORE_OUT_STANDARDIZE, PackedBatch
    flags = NPORE_OUT_STANDARDIZE | NPORE_OUT_RLE | NPORE_OUT_NO_EXPANDED
    pending = queue.Queue(maxsize=n_inflight + 1)
    state = {"written": 0, "error": None}

    def retire_loop():
        fd = -1
        try:
            z = compressor() if compressor is not None else None
            fd = open_out(z)
            end = os.fstat(fd).st_size
        except Exception as e:                        # noqa: BLE001
            state["error"] = e
        while True:
            item = pending.get()
            if item is None:
                break
            if state["error"] is not None:
                continue                              # keep draining so that the producer never blocks
            try:
                fut, cols, g, n = item
                t1 = time.perf_counter()
                res, st_ = fut.result()
                t2 = time.perf_counter()
                mark(f"gpu done n={n} kernels_ms={st_['ms_kernels_total']:.1f} h2d_ms={st_['ms_h2d']:.1f} plan_ms={st_['ms_plan']:.1f} d2h_ms={st_['ms_d2h']:.1f} "
                     f"warps/SM={st_['fwd_warps_per_sm']} context from {1e3 * (st_['wall'][0] - t0):.1f} ms, buffers {1e3 * (st_['wall'][1] - t0):.1f}, "
                     f"to {1e3 * (st_['wall'][2] - t0):.1f} ms")
                _report(res.status[:n], "realign_read")
                if z is None:
                    end += len(format_sam(bam, None, g, res.rle, res.rle_off[:n + 1], n_threads, cols=cols, fd=fd, offset=end))
                    t3 = time.perf_counter()
                    mark("formatted + written")
                    tm["gpu_wait"] += t2 - t1; tm["format"] += t3 - t2; tm["write"] += time.perf_counter() - t3
                else:
                    raw = format_sam(bam, None, g, res.rle, res.rle_off[:n + 1], n_threads, cols=cols, binary=True, offsets=bai is not None)
                    raw, rec_off = raw if bai is not None else (raw, None)
                    t3 = time.perf_counter()
                    blob = z.compress(raw)
                    t4 = time.perf_counter()
                    start, end = end, _write_all(fd, blob, end)
                    t5 = time.perf_counter()
                    if bai is not None:
                        bai.add(z.index(rec_off, start))
                        tm["index"] += time.perf_counter() - t5
                        tm["index_device_ms"] += getattr(z, "last_index_ms", 0.0)
                    mark("formatted + written")
                    tm["gpu_wait"] += t2 - t1; tm["format"] += t3 - t2; tm["compress"] += t4 - t3; tm["write"] += t5 - t4
                state["written"] += n
                with cfg.counter.get_lock():
                    cfg.counter.value += n
            except Exception as e:                    # noqa: BLE001
                state["error"] = e
        if fd >= 0:
            os.close(fd)

    if compressor is not None:
        tm.setdefault("compress", 0.0)
    if bai is not None:
        tm.setdefault("index", 0.0)
        tm.setdefault("index_device_ms", 0.0)
    retire = threading.Thread(target=retire_loop, daemon=True)
    retire.start()
    if bai is not None:
        segments = _in_coordinate_order(bam, segments)
    try:
        for ctg, sel in segments:
            contig = fa[ctg]
            ops = np.cumsum(_record_ops(bam, sel))
            cut = 0
            while cut < len(sel) and state["error"] is None:
                stop = max(cut + 1, int(np.searchsorted(ops, (ops[cut - 1] if cut else 0) + max_batch_ops, "right")))
                part = sel[cut:stop]
                t1 = time.perf_counter()
                nib, nib_start = bam.gather_nib(part, n_threads)          # the upload: BAM's own 4-bit bases + CIGAR words
                mark("nib gathered")
                cig_words, cig_off = bam.gather_cigar(part, n_threads)
                mark("cigar gathered")
                lo, hi = int(bam.pos[part].min()), int(bam.end[part].max())
                # base codes of the batch's reference span only (not the contig: 250 Mb of chr1 for a window that covers 1 Mb)
                packed = PackedBatch.from_flat_shared_nib(bases_to_int(contig[lo:hi].upper()), bam.pos[part].astype(np.int64) - lo, bam.end[part] - bam.pos[part],
                                                          nib, nib_start, bam.aln_len[part], cig_words, cig_off)
                fut = pipe.submit(packed, flags)                          # the GPU starts; the SAM-text gather runs beside it
                mark(f"submitted n={len(part)}")
                g = bam.gather(part, nt_text, want_codes=False, want_cigar=False)    # ASCII bases / qualities / names
                mark("text gathered")
                item = (fut, take_columns(bam, part), g, len(part))
                tm["gather"] += time.perf_counter() - t1
                pending.put(item)                                        # blocks while n_inflight + 1 batches are unfinished
                cut = stop
            if state["error"] is not None:
                break
    finally:
        pending.put(None)
        retire.join()
    if state["error"] is not None:
        raise state["error"]
    return state["written"]


def _realign_sharded(bam, fa, pipes, devices, open_out, regions, max_reads, max_batch_ops, n_threads, n_inflight, tm, mark, t0, ext="sam",
                     bai=None):
    """realign.py:75-115 on several GPUs of one host (SURVEY.md 8(e)): the coordinate-sorted reads are cut into len(devices)
    contiguous genomic regions of equal cell-update load (the reference's own unit of distribution is the region,
    util.py:44-93 / bam.pyx:27-28); every region is an independent ingest -> GPU -> SAM-text pipeline on its own device (no
    data-path collective) and host threads; the host gathers the per-region SAM bodies in region order into ONE file,
    byte-identical to the single-GPU output.  Region 0 writes into the output itself (open_out), the others into part files,
    which are removed whether the call succeeds or fails.  ext "bam": every shard compresses its records on its own device and
    the part files hold BGZF members only (no header, no EOF block), so their concatenation is valid BGZF.  tm: per phase, summed over the shards, plus
    'shards': [{device, reads, cell_updates, seconds}] and 'concat' seconds.  bai: a BaiBuilder; every shard indexes its records
    with offsets in its own file, and shard g's lists join bai shifted by the offset its part file is copied to."""
    from .scheduler import cut_balanced
    tm.setdefault("concat", 0.0)
    t1 = time.perf_counter()
    G = len(devices)
    segs = list(select_reads(bam, regions, max_reads))
    if bai is not None:
        segs = list(_in_coordinate_order(bam, segs))
    loads = [_read_loads(bam, sel) for _, sel in segs]
    total = float(sum(int(x.sum()) for x in loads))
    # contiguous cuts of the (contig, start)-ordered read list at equal cumulative load
    shard_segs = [[] for _ in range(G)]
    shard_load = [0] * G
    done = 0.0
    for (ctg, sel), ld in zip(segs, loads):
        owner = cut_balanced(ld, G, done, total)                   # by the read's load midpoint
        for gidx in np.unique(owner):
            m = owner == gidx
            shard_segs[int(gidx)].append((ctg, sel[m]))
            shard_load[int(gidx)] += int(ld[m].sum())
        done += float(ld.sum())
    tm["open"] += time.perf_counter() - t1
    out = f"{cfg.args.out_prefix}.{ext}"
    parts = [f"{cfg.args.out_prefix}.part{g}.{ext}" for g in range(G)]
    opens = [open_out] + [lambda z, p=p: os.open(p, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644) for p in parts[1:]]
    nt = max(1, (n_threads or os.cpu_count() or 1) // G)
    results = [None] * G
    phases = ("gather", "gpu_wait", "format", "write") + (("compress",) if ext == "bam" else ()) + (("index", "index_device_ms") if bai is not None else ())
    shard_tm = [{k: 0.0 for k in phases} for _ in range(G)]
    shard_bai = [BaiBuilder(len(bam.refs)) if bai is not None else None for _ in range(G)]

    def shard_main(g):
        t2 = time.perf_counter()
        try:
            comp = (lambda: _compressor(devices[g], g)) if ext == "bam" else None
            n = _realign_segments(bam, shard_segs[g], fa, pipes[g], opens[g], shard_tm[g], nt, nt, max_batch_ops, n_inflight, mark, t0,
                                  compressor=comp, bai=shard_bai[g])
            results[g] = (n, time.perf_counter() - t2, None)
        except Exception as e:      # noqa: BLE001
            results[g] = (0, time.perf_counter() - t2, e)

    threads = [threading.Thread(target=shard_main, args=(g,)) for g in range(G)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    try:
        for _, _, err in results:
            if err is not None:
                raise err
        t2 = time.perf_counter()
        dst = os.open(out, os.O_WRONLY)                             # host gather: region order = coordinate order
        try:
            end = os.fstat(dst).st_size
            if bai is not None:
                bai.extend(shard_bai[0], 0)                         # shard 0 wrote after the header: absolute offsets already
            for g, part in enumerate(parts[1:], 1):
                if bai is not None:
                    bai.extend(shard_bai[g], end)
                with open(part, "rb") as src:
                    left = os.fstat(src.fileno()).st_size
                    try:                                            # in-kernel copy (no bounce through user space)
                        while left > 0:
                            n = os.copy_file_range(src.fileno(), dst, left, None, end)
                            if n <= 0:
                                break
                            left -= n; end += n
                    except (AttributeError, OSError):
                        pass
                    while left > 0:                                 # not supported here (or stopped early): plain copy of the rest
                        buf = os.pread(src.fileno(), min(left, 16 << 20), os.fstat(src.fileno()).st_size - left)
                        if not buf:
                            raise OSError(f"short read while gathering {part}")
                        os.pwrite(dst, buf, end)
                        left -= len(buf); end += len(buf)
        finally:
            os.close(dst)
        tm["concat"] += time.perf_counter() - t2
    finally:
        for part in parts[1:]:
            with contextlib.suppress(FileNotFoundError):
                os.remove(part)
    for k in phases:
        tm[k] = tm.get(k, 0.0) + sum(x[k] for x in shard_tm)
    tm["shards"] = [{"device": int(devices[g]), "reads": int(results[g][0]), "cell_updates": int(shard_load[g]), "seconds": round(results[g][1], 4)}
                    for g in range(G)]
    return sum(n for n, _, _ in results)


def _keep_freed_buffers_mapped():
    """Once per process: raise glibc's mmap / trim thresholds (mallopt) so that the pipeline's per-window buffers -- nibble and
    CIGAR gathers, SAM text columns, result arrays, the 20 MB SAM blob -- are recycled from the heap instead of being mmap'ed,
    page-faulted by 16 threads at once and munmap'ed again for every window.  Measured on the C2 file (16 host cores): the
    gathers in front of the second and third upload took 8-12 ms instead of 1 ms (page faults + address-space lock beside the
    inflating prefetch threads); with it the host is through all windows of the 3,000-read file after 27 ms and the GPU, not
    the host, limits the call (profiles/r02_ab_experiments.md).  NPORE_NO_MALLOPT=1 leaves the allocator alone."""
    global _MALLOC_TUNED
    if _MALLOC_TUNED or os.environ.get("NPORE_NO_MALLOPT"):
        return
    _MALLOC_TUNED = True
    try:
        import ctypes
        libc = ctypes.CDLL("libc.so.6")
        libc.mallopt(-3, 32 << 20)            # M_MMAP_THRESHOLD: its maximum (blocks up to 32 MB come from the heap)
        libc.mallopt(-1, 1 << 30)             # M_TRIM_THRESHOLD: keep up to 1 GB of freed heap
    except (OSError, AttributeError):         # not glibc
        pass


def realign_bam(bam_fn, fasta, out_prefix=None, regions=None, max_reads=0, argv=None, max_batch_ops=64_000_000, n_threads=0,
                timings=None, window_bytes=16 << 20, n_inflight=3, devices=None, out_format="sam", index=False):
    """realign.py:75-115 without pysam / Pool: header, ingest, GPU realignment, records appended in input order
    (= coordinate order for a sorted BAM, which is what the header claims).  Returns the number of records written.
    Flat arrays all the way, as a pipeline: the reader streams the file in windows of ~window_bytes of inflated records
    (native, multi-threaded) and gathers batch k+1 while batch k is on the GPU (n_inflight contexts) and a third thread
    formats (native) and writes batch k-1.  One shared reference slice is uploaded per batch.
    timings: optional dict that receives host seconds per phase (open, gather, gpu_wait, format = formatting + the append to the
    file, write = 0 since the formatter threads write themselves); timings["trace"] = [] collects (seconds, event) of every step.
    devices: CUDA device indices; more than one: one region-shard pipeline per device, gathered in order into one file
    (_realign_sharded; the whole file is loaded, no streaming).
    out_format: "sam" writes {out_prefix}.sam; "bam" writes the same header and records to {out_prefix}.bam as BAM, each batch
    encoded on the host and compressed into BGZF members on the batch's device, with one BGZF EOF block at the end; timings then
    also has "compress", the seconds spent in the compressor.  An index of an earlier run beside the BAM output is removed.
    index=True (BAM only): also writes the BAM index {out_prefix}.bam.bai, computed on the device batch by batch
    (BgzfCompressor.index) and written once the BAM is complete; timings then has "index", the seconds spent on it, and
    "index_device_ms", its kernel time.  Regions must then be in header contig order without overlaps, and no contig may be
    longer than 2^29 - 1 bp (ValueError before any work); a read selected by two regions makes the output unsorted and raises
    ValueError when it is met.  A call that fails leaves no index.
    regions and an index of the input (NativeBam): only the index chunks of the regions are read and inflated; the output is the
    same as without the index."""
    if out_format not in ("sam", "bam"):
        raise ValueError(f"out_format must be 'sam' or 'bam', not {out_format!r}")
    if index and out_format != "bam":
        raise ValueError("index=True needs out_format='bam'")
    from .bam import _tables
    tm = timings if timings is not None else {}
    for k in ("open", "gather", "gpu_wait", "format", "write"):
        tm.setdefault(k, 0.0)
    _keep_freed_buffers_mapped()
    t0 = time.perf_counter()
    trace = tm.get("trace")                       # optional list: (seconds since the call, event) of every pipeline step
    mark = (lambda ev: trace.append((round(time.perf_counter() - t0, 5), ev))) if trace is not None else (lambda ev: None)
    if out_prefix is not None:
        cfg.args.out_prefix = out_prefix
    if not os.path.exists(bam_fn):
        print(f"\nERROR: BAM file '{bam_fn}' not found.")
        sys.exit(1)
    fa = read_fasta(fasta) if isinstance(fasta, str) else fasta
    devices = list(devices or [None])
    # several regions are served region by region (bam.pyx:27-28), and region shards are cut from every record's span: both
    # need the whole file at hand
    streaming = len(devices) == 1 and not (regions and len(regions) > 1)
    bam = NativeBam(bam_fn, n_threads, window_bytes=window_bytes if streaming else 0, regions=regions)
    mark("bam open")
    out = f"{cfg.args.out_prefix}.{out_format}"
    bai = None
    if index:
        try:
            _check_indexable(bam.refs, regions)
        except ValueError:
            bam.close()
            raise
        bai = BaiBuilder(len(bam.refs))

    def open_out(z):
        # called by the writer thread: the header (and the truncation of a previous output: ~2 ms for a 60 MB file) is written
        # beside the first window's inflate
        if z is None:
            create_header(out, bam.refs, argv)
        else:
            if os.path.dirname(out):
                os.makedirs(os.path.dirname(out), exist_ok=True)
            with contextlib.suppress(FileNotFoundError):
                os.remove(f"{out}.bai")                 # an earlier run's index does not describe this file
            with open(out, "wb") as fh:
                fh.write(z.compress(bam_header(bam.refs, argv)))
        mark("header written")
        return os.open(out, os.O_WRONLY)

    try:
        sub, npt = _tables()
        with _PIPE_LOCK:
            pipes = [_pipeline(sub, npt, n_inflight, d) for d in devices]
        tm["open"] += time.perf_counter() - t0
        mark("opened")
        if len(devices) > 1:
            written = _realign_sharded(bam, fa, pipes, devices, open_out, regions, max_reads, max_batch_ops, n_threads, n_inflight,
                                       tm, mark, t0, ext=out_format, bai=bai)
        else:
            def segments():
                kept = 0
                while True:
                    if bam.window_bytes:
                        t1 = time.perf_counter()
                        more = bam.advance()
                        tm["open"] += time.perf_counter() - t1
                        mark(f"window of {more} records")
                        if not more:
                            return
                    for ctg, sel in select_reads(bam, regions, (max_reads - kept) if max_reads else 0):
                        kept += len(sel)
                        yield ctg, sel
                    if not bam.window_bytes or (max_reads and kept >= max_reads):
                        return

            # the text gather runs right after a submit: leave cores to the GPU worker thread that has just been woken (on 16
            # cores a 16-thread gather delayed the start of the upload by 2 ms) and to the writer
            nt_text = max(1, (n_threads or os.cpu_count() or 1) - int(os.environ.get("NPORE_SPARE_CORES", "3")))
            comp = (lambda: _compressor(devices[0], 0)) if out_format == "bam" else None
            written = _realign_segments(bam, segments(), fa, pipes[0], open_out, tm, n_threads, nt_text, max_batch_ops, n_inflight, mark, t0,
                                        compressor=comp, bai=bai)
        if out_format == "bam":
            fd = os.open(out, os.O_WRONLY)
            try:
                _write_all(fd, BGZF_EOF, os.fstat(fd).st_size)
            finally:
                os.close(fd)
        if bai is not None:
            t1 = time.perf_counter()
            bai.write(f"{out}.bai")
            tm["index"] += time.perf_counter() - t1
            mark("index written")
    finally:
        bam.close()
    mark("closed")
    return written


# ------------------------------------------------------------------------------------------------ minimal BAM writer
def _bgzf_block(payload: bytes, level: int = 6) -> bytes:
    comp = zlib.compressobj(level, zlib.DEFLATED, -15)
    cdata = comp.compress(payload) + comp.flush()
    bsize = len(cdata) + 25
    return (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", bsize) + cdata +
            struct.pack("<II", zlib.crc32(payload) & 0xffffffff, len(payload)))


def _reg2bin(beg, end):
    end -= 1
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return off + (beg >> shift)
    return 0


def write_bam(path, header_text, refs, records, level=6):
    """records: dicts with name, flag, ref_id, pos, mapq, cigar (list of (len, op_char)), seq, qual (bytes/None), tags
    ({'HP': int} supported).  level: zlib level of the BGZF members."""
    lut = np.full(256, 15, np.uint8)
    for i, c in enumerate(_SEQ16):
        lut[ord(c)] = i
    out = io.BytesIO()
    text = header_text.encode()
    out.write(b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs)))
    for name, length in refs:
        out.write(struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", length))
    for r in records:
        cig = [(n << 4) | _OPS.index(op) for n, op in r["cigar"]]
        seq = r["seq"]
        codes = np.zeros(len(seq) + (len(seq) & 1), np.uint8)
        codes[:len(seq)] = lut[np.frombuffer(seq.encode("latin-1"), np.uint8)]
        packed = ((codes[0::2] << 4) | codes[1::2]).tobytes()
        qual = bytes([0xFF] * len(seq)) if r.get("qual") is None else bytes(r["qual"])
        tags = b"".join(b"HPi" + struct.pack("<i", v) if k == "HP" else b"" for k, v in r.get("tags", {}).items())
        span = sum(n for n, op in r["cigar"] if op in "MDN=X") or 1
        name = r["name"].encode() + b"\0"
        body = struct.pack("<iiBBHHHiiii", r["ref_id"], r["pos"], len(name), r["mapq"], _reg2bin(r["pos"], r["pos"] + span),
                           len(cig), r["flag"], len(seq), -1, -1, 0)
        body += name + struct.pack(f"<{len(cig)}I", *cig) + packed + qual + tags
        out.write(struct.pack("<i", len(body)) + body)
    raw = out.getvalue()
    with open(path, "wb") as fh:
        for i in range(0, len(raw), 60000):
            fh.write(_bgzf_block(raw[i:i + 60000], level))
        fh.write(_bgzf_block(b""))
