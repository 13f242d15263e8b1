"""Host side of the GPU batch scheduler: packs items into the flat buffers of the C ABI and drives
libnpore_b200.so.  Replaces the reference's Pool fan-out (/root/reference/src/realign.py:110-114,
standardize_vcf.py:30-31): one `Realigner.run()` call = one batch on one B200.

PyTorch is used only to allocate pinned host buffers (and to pick the CUDA device); all compute is in the
CUDA library.  There is no CPU path: constructing a Realigner without a GPU raises.
"""
import ctypes as C
import re

import numpy as np

from . import _lib
from ._lib import NPORE_OUT_NO_EXPANDED, NPORE_OUT_RLE, NPORE_OUT_STANDARDIZE  # noqa: F401

_RLE = re.compile(rb"(\d+)([MIDNSHP=XB])")
_OPCODE = np.full(256, 255, dtype=np.uint8)
for _k, _c in enumerate("MIDNSHP=XB"):            # cfg.py:27-32
    _OPCODE[ord(_c)] = _k
_OPCHAR = np.frombuffer(b"MIDNSHP=XB", dtype=np.uint8)


_CODE_TABLE = bytes(({78: 0, 65: 1, 67: 2, 71: 3, 84: 4, 45: 5}).get(i, 0) for i in range(256))     # cig.pyx:212-229


class NporeError(RuntimeError):
    pass


MAX_ITEM_OPS = (1 << 28) - 1      # include/npore_b200.h: ref_len + seq_len of one item (bit offsets / run-length fields are 28 bits wide)


def check_item_sizes(ref_len, seq_len, what="item"):
    """Raise a per-item error BEFORE a batch is sent: one oversize item would otherwise fail the whole npore_upload with
    NPORE_ERR_BAD_ARG, valid items included (the reference has no such limit; a 134 Mb haplotype is ours)."""
    tot = np.asarray(ref_len, dtype=np.int64) + np.asarray(seq_len, dtype=np.int64)
    bad = np.flatnonzero(tot > MAX_ITEM_OPS)
    if len(bad):
        k = int(bad[0])
        raise NporeError(f"{what} {k}: ref_len + seq_len = {int(tot[k])} exceeds the library limit of {MAX_ITEM_OPS} "
                         f"(2^28 - 1; a haplotype of ~134 Mb).  Realign this {what} by contig halves or raise the limit in csrc/.")


def _pinned(n, dtype):
    """Pinned host array (numpy view of a torch pinned tensor); falls back to pageable if torch has no CUDA."""
    import torch
    n = max(int(n), 1)
    if torch.cuda.is_available():
        t = torch.empty(n, dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True)
        return t.numpy(), t          # the numpy view keeps the pinned storage alive
    return np.empty(n, dtype=dtype), None


def cigar_to_rle(cigar: str) -> np.ndarray:
    """CIGAR text -> BAM-style words (len<<4|op).  Accepts run-length text ('3=2D') or expanded text ('===DD').
    S and H groups are dropped (bam.pyx:59)."""
    b = cigar.encode("latin-1")
    if not b:
        return np.zeros(0, np.uint32)
    if b[0] in b"0123456789":
        m = _RLE.findall(b)
        lens = np.array([int(x) for x, _ in m], dtype=np.uint32)
        ops = _OPCODE[np.frombuffer(b"".join(o for _, o in m), dtype=np.uint8)].astype(np.uint32)
    else:
        a = np.frombuffer(b, dtype=np.uint8)
        cut = np.flatnonzero(a[1:] != a[:-1]) + 1
        starts = np.concatenate(([0], cut))
        lens = np.diff(np.concatenate((starts, [len(a)]))).astype(np.uint32)
        ops = _OPCODE[a[starts]].astype(np.uint32)
    keep = (ops != 4) & (ops != 5)
    return ((lens[keep] << 4) | ops[keep]).astype(np.uint32)


def rle_to_text(words: np.ndarray) -> str:
    """words (len<<4|op) -> '12M1I...' (cig.pyx:13-38 collapse_cigar output)."""
    if len(words) == 0:
        return ""
    lens = (words >> 4).tolist()
    ops = _OPCHAR[words & 15].tobytes().decode()
    return "".join(f"{n}{o}" for n, o in zip(lens, ops))


def cigars_to_rle_batch(cigars):
    """Many CIGAR texts -> (words uint32, off int64[n+1]) in one vectorised pass (no per-character Python).
    All texts must be of one kind: run-length ('3=2D...') or expanded ('===DD...').  S/H groups are dropped."""
    n = len(cigars)
    off = np.zeros(n + 1, dtype=np.int64)
    if n == 0:
        return np.zeros(0, np.uint32), off
    big = "\n".join(cigars).encode("latin-1") + b"\n"
    a = np.frombuffer(big, dtype=np.uint8)
    first = next((c for c in cigars if c), "")
    if first[:1].isdigit():
        isd = (a >= 48) & (a <= 57)
        op_idx = np.flatnonzero(~isd)                          # op letters and the '\n' item separators
        dpos = np.flatnonzero(isd)
        gid = np.cumsum(~isd)[dpos]                            # group (next non-digit) of every digit
        w = np.power(10, op_idx[gid] - dpos - 1, dtype=np.int64)
        lens = np.bincount(gid, weights=(a[dpos] - 48).astype(np.int64) * w, minlength=len(op_idx)).astype(np.int64)
        ops = _OPCODE[a[op_idx]]
    else:
        cut = np.flatnonzero((a[1:] != a[:-1]) | (a[1:] == 10)) + 1         # every separator is its own run
        starts = np.concatenate(([0], cut))
        lens = np.diff(np.concatenate((starts, [len(a)]))).astype(np.int64)
        ops = _OPCODE[a[starts]]
        op_idx = starts
    sep = a[op_idx] == 10
    item = np.cumsum(sep) - sep                                # item index of every group
    keep = ~sep & (ops != 4) & (ops != 5)
    if (ops[keep] == 255).any():
        raise ValueError("unsupported CIGAR operation")
    words = ((lens[keep] << 4) | ops[keep]).astype(np.uint32)
    np.cumsum(np.bincount(item[keep], minlength=n)[:n], out=off[1:])
    return words, off


def rle_to_text_batch(words, off):
    """Run-length words of many items -> list of CIGAR texts (collapse_cigar output), vectorised digit formatting."""
    n = len(off) - 1
    if n <= 0:
        return []
    words = np.asarray(words[:off[-1]], dtype=np.uint32)
    lens = (words >> 4).astype(np.int64)
    nd = np.ones(len(lens), dtype=np.int64)
    for t in (10, 100, 1000, 10_000, 100_000, 1_000_000, 10_000_000, 100_000_000):
        nd += lens >= t
    width = nd + 1
    end = np.cumsum(width)
    pos = end - width
    out = np.empty(int(end[-1]) if len(end) else 0, dtype=np.uint8)
    for p in range(int(nd.max()) if len(nd) else 0):
        m = nd > p
        out[pos[m] + p] = 48 + (lens[m] // np.power(10, nd[m] - 1 - p)) % 10
    out[pos + nd] = _OPCHAR[words & 15]
    bstart = np.concatenate(([0], end))[np.asarray(off, dtype=np.int64)]
    buf = out.tobytes()
    return [buf[bstart[i]:bstart[i + 1]].decode("latin-1") for i in range(n)]


def bases_to_int_batch(seqs):
    """Many base strings -> (codes uint8 concatenated, lengths int32) with one table lookup (cig.pyx:212-229)."""
    lens = np.fromiter((len(x) for x in seqs), dtype=np.int32, count=len(seqs))
    joined = "".join(seqs).encode("latin-1")
    codes = np.frombuffer(joined.translate(_CODE_TABLE), dtype=np.uint8) if joined else np.zeros(0, np.uint8)
    return codes, lens


class PackedBatch:
    """Flat host buffers in the layout of `npore_batch` (include/npore_b200.h)."""

    def __init__(self, refs, seqs, cigars, shared_ref=None, ref_ranges=None, pinned=True):
        """refs/seqs: lists of uint8 code arrays; cigars: list of RLE word arrays.
        shared_ref + ref_ranges[(start, stop)]: items index one shared reference (region sharding, SURVEY 8(e))."""
        n = len(seqs)
        self.n = n
        alloc = (lambda m, dt: _pinned(m, dt)[0]) if pinned else (lambda m, dt: np.empty(max(int(m), 1), dtype=dt))
        self.seq_len = np.array([len(s) for s in seqs], dtype=np.int32)
        self.seq_start = np.zeros(n, dtype=np.int64)
        if n:
            np.cumsum(self.seq_len[:-1], out=self.seq_start[1:])
        self.seq_total = int(self.seq_len.sum())
        self.seq_codes = alloc(self.seq_total, np.uint8)
        if self.seq_total:
            np.concatenate(seqs, out=self.seq_codes[:self.seq_total])
        if shared_ref is not None:
            self.ref_total = int(len(shared_ref))
            self.ref_codes = alloc(self.ref_total, np.uint8)
            self.ref_codes[:self.ref_total] = shared_ref
            self.ref_start = np.array([a for a, _ in ref_ranges], dtype=np.int64)
            self.ref_len = np.array([b - a for a, b in ref_ranges], dtype=np.int32)
        else:
            self.ref_len = np.array([len(s) for s in refs], dtype=np.int32)
            self.ref_start = np.zeros(n, dtype=np.int64)
            if n:
                np.cumsum(self.ref_len[:-1], out=self.ref_start[1:])
            self.ref_total = int(self.ref_len.sum())
            self.ref_codes = alloc(self.ref_total, np.uint8)
            if self.ref_total:
                np.concatenate(refs, out=self.ref_codes[:self.ref_total])
        self.cigar_off = np.zeros(n + 1, dtype=np.int64)
        if n:
            np.cumsum([len(c) for c in cigars], out=self.cigar_off[1:])
        self.cigar_rle = alloc(int(self.cigar_off[-1]), np.uint32)
        if int(self.cigar_off[-1]):
            np.concatenate(cigars, out=self.cigar_rle[:int(self.cigar_off[-1])])
        self.total_ops = int(self.ref_len.astype(np.int64).sum() + self.seq_len.astype(np.int64).sum())

    @classmethod
    def from_flat(cls, ref_codes, ref_len, seq_codes, seq_len, cigar_rle, cigar_off):
        """Wrap already concatenated arrays (vectorised packers above) without copying item by item."""
        self = cls.__new__(cls)
        self.n = len(seq_len)
        self.ref_codes = np.ascontiguousarray(ref_codes, dtype=np.uint8) if len(ref_codes) else np.zeros(1, np.uint8)
        self.seq_codes = np.ascontiguousarray(seq_codes, dtype=np.uint8) if len(seq_codes) else np.zeros(1, np.uint8)
        self.ref_len = np.ascontiguousarray(ref_len, dtype=np.int32)
        self.seq_len = np.ascontiguousarray(seq_len, dtype=np.int32)
        self.ref_start = np.zeros(self.n, dtype=np.int64)
        self.seq_start = np.zeros(self.n, dtype=np.int64)
        if self.n:
            np.cumsum(self.ref_len[:-1], out=self.ref_start[1:])
            np.cumsum(self.seq_len[:-1], out=self.seq_start[1:])
        self.ref_total = int(self.ref_len.astype(np.int64).sum())
        self.seq_total = int(self.seq_len.astype(np.int64).sum())
        self.cigar_off = np.ascontiguousarray(cigar_off, dtype=np.int64)
        self.cigar_rle = np.ascontiguousarray(cigar_rle, dtype=np.uint32) if len(cigar_rle) else np.zeros(1, np.uint32)
        self.total_ops = self.ref_total + self.seq_total
        return self

    @classmethod
    def from_flat_shared(cls, ref_codes, ref_start, ref_len, seq_codes, seq_len, cigar_rle, cigar_off):
        """Like from_flat, but every item addresses a window (ref_start, ref_len) of ONE shared reference buffer (a contig
        slice uploaded once instead of one copy per read; SURVEY 8(e))."""
        self = cls.from_flat(np.zeros(0, np.uint8), ref_len, seq_codes, seq_len, cigar_rle, cigar_off)
        self.ref_codes = np.ascontiguousarray(ref_codes, dtype=np.uint8) if len(ref_codes) else np.zeros(1, np.uint8)
        self.ref_start = np.ascontiguousarray(ref_start, dtype=np.int64)
        self.ref_total = int(len(ref_codes))
        self.total_ops = int(self.ref_len.astype(np.int64).sum()) + self.seq_total
        return self

    @classmethod
    def from_strings(cls, refs, seqs, cigars):
        """refs / seqs: base strings; cigars: CIGAR texts (all run-length or all expanded)."""
        rc, rl = bases_to_int_batch(refs)
        sc, sl = bases_to_int_batch(seqs)
        words, off = cigars_to_rle_batch(cigars)
        return cls.from_flat(rc, rl, sc, sl, words, off)

    seq_nib = None          # packed reads (BAM 4-bit nibbles) instead of seq_codes: set by from_flat_shared_nib

    @classmethod
    def from_flat_shared_nib(cls, ref_codes, ref_start, ref_len, seq_nib, seq_nib_start, seq_len, cigar_rle, cigar_off):
        """Like from_flat_shared, with the reads in BAM's own 4-bit packing (npore_batch.seq_nib): item i's read is the seq_len[i]
        nibbles from nibble seq_nib_start[i] of seq_nib.  Half the upload bytes; the device decodes (cig.pyx:212-229)."""
        self = cls.from_flat_shared(ref_codes, ref_start, ref_len, np.zeros(0, np.uint8), seq_len, cigar_rle, cigar_off)
        self.seq_nib = np.ascontiguousarray(seq_nib, dtype=np.uint8) if len(seq_nib) else np.zeros(1, np.uint8)
        self.seq_nib_start = np.ascontiguousarray(seq_nib_start, dtype=np.int64)
        self.seq_nib_bytes = int(len(seq_nib))
        self.seq_total = int(self.seq_len.astype(np.int64).sum())
        self.total_ops = int(self.ref_len.astype(np.int64).sum()) + self.seq_total
        return self

    def c_struct(self):
        p = lambda a: a.ctypes.data  # noqa: E731
        if self.seq_nib is not None:
            return _lib.Batch(self.n, p(self.ref_codes), p(self.ref_start), p(self.ref_len), self.ref_total,
                              None, None, p(self.seq_len), 0, p(self.cigar_rle), p(self.cigar_off),
                              p(self.seq_nib), p(self.seq_nib_start), self.seq_nib_bytes)
        return _lib.Batch(self.n, p(self.ref_codes), p(self.ref_start), p(self.ref_len), self.ref_total,
                          p(self.seq_codes), p(self.seq_start), p(self.seq_len), self.seq_total,
                          p(self.cigar_rle), p(self.cigar_off), None, None, 0)

    def h2d_bytes(self):
        seq = self.seq_nib_bytes + 8 * self.n if self.seq_nib is not None else self.seq_total
        return self.ref_total + seq + 4 * int(self.cigar_off[-1])


class BatchResult:
    """Host buffers in the layout of `npore_result`.  want_ops=False leaves out the expanded-ops buffer (NPORE_OUT_NO_EXPANDED);
    rle_buf / rle_off_buf: caller-owned arrays (uint32 / int64[n+1]) the run-length words and offsets are written into -- e.g.
    slices of a buffer shared between the per-GPU processes, so that the device-to-host copy IS the gather."""

    def __init__(self, n, total_ops, n_chunks, want_rle, pinned=True, want_ops=True, rle_buf=None, rle_off_buf=None):
        alloc = (lambda m, dt: _pinned(m, dt)[0]) if pinned else (lambda m, dt: np.empty(max(int(m), 1), dtype=dt))
        self.n = n
        self.ops = alloc(total_ops, np.uint8) if want_ops else None
        self.ops_off = np.zeros(n + 1, dtype=np.int64)
        if rle_buf is not None:
            assert rle_buf.dtype == np.uint32 and rle_buf.flags.c_contiguous
            self.rle = rle_buf
        else:
            self.rle = alloc(total_ops if want_rle else 1, np.uint32)
        if rle_off_buf is not None:
            assert rle_off_buf.dtype == np.int64 and len(rle_off_buf) >= n + 1 and rle_off_buf.flags.c_contiguous
            self.rle_off = rle_off_buf
        else:
            self.rle_off = np.zeros(n + 1, dtype=np.int64)
        self.chunk_scores = np.zeros(max(n_chunks, 1), dtype=np.float32)
        self.score_off = np.zeros(n + 1, dtype=np.int64)
        self.status = np.zeros(max(n, 1), dtype=np.int32)
        self.want_rle = want_rle

    def c_struct(self):
        p = lambda a: a.ctypes.data  # noqa: E731
        return _lib.Result(p(self.ops) if self.ops is not None else None, len(self.ops) if self.ops is not None else 0,
                           p(self.ops_off) if self.ops is not None else None,
                           p(self.rle) if self.want_rle else None, len(self.rle), p(self.rle_off) if self.want_rle else None,
                           p(self.chunk_scores), len(self.chunk_scores), p(self.score_off), p(self.status))

    def ops_str(self, i) -> str:
        return self.ops[self.ops_off[i]:self.ops_off[i + 1]].tobytes().decode()

    def rle_words(self, i) -> np.ndarray:
        return self.rle[self.rle_off[i]:self.rle_off[i + 1]]

    def cigar_text(self, i) -> str:
        return rle_to_text(self.rle_words(i))

    def cigar_texts(self):
        """All collapsed CIGAR texts of the batch at once."""
        return rle_to_text_batch(self.rle, self.rle_off)

    def scores(self, i) -> np.ndarray:
        return self.chunk_scores[self.score_off[i]:self.score_off[i + 1]]


class Realigner:
    """One GPU context (npore_ctx).  Parameters mirror align()'s (aln.pyx:379-382) and cfg.args.max_n/max_l."""

    def __init__(self, sub_scores, np_scores, max_n=6, max_l=100, indel_start=5.0, indel_extend=1.0,
                 max_b_rows=20000, r=30, device=0):
        self._ctx = C.c_void_p()
        self._L = _lib.lib()
        sub = np.ascontiguousarray(sub_scores, dtype=np.float32)
        npt = np.ascontiguousarray(np_scores, dtype=np.float32)
        if sub.shape != (5, 5) or npt.ndim != 3 or npt.shape[1] != npt.shape[2]:
            raise ValueError("sub_scores must be [5,5], np_scores [n, l, l]")
        self.params = dict(max_n=max_n, max_l=max_l, indel_start=indel_start, indel_extend=indel_extend,
                           max_b_rows=max_b_rows, r=r, device=device)
        rc = self._L.npore_ctx_create(C.byref(self._ctx), device, sub.ctypes.data, npt.ctypes.data, npt.shape[0], npt.shape[1],
                                      max_n, max_l, indel_start, indel_extend, max_b_rows, r)
        if rc != 0:
            self._ctx = C.c_void_p()
            raise NporeError(f"npore_ctx_create failed: {self._L.npore_strerror(rc).decode()} "
                             "(npore_b200 needs a CUDA device; there is no CPU fallback)")

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._L.npore_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    __del__ = close

    def _check(self, rc, what):
        if rc != 0:
            raise NporeError(f"{what}: {self._L.npore_strerror(rc).decode()} [{self._L.npore_last_error(self._ctx).decode()}]")

    def set_stream(self, cuda_stream: int):
        """Run on the caller's CUDA stream (e.g. torch.cuda.current_stream().cuda_stream)."""
        self._check(self._L.npore_set_stream(self._ctx, C.c_void_p(cuda_stream)), "npore_set_stream")

    def count_chunks(self, packed: PackedBatch) -> int:
        return int(self._L.npore_count_chunks(self._ctx, packed.n, packed.ref_len.ctypes.data, packed.seq_len.ctypes.data))

    def new_result(self, packed: PackedBatch, flags: int, pinned=True) -> BatchResult:
        return BatchResult(packed.n, packed.total_ops, self.count_chunks(packed), bool(flags & NPORE_OUT_RLE), pinned,
                           want_ops=not (flags & NPORE_OUT_NO_EXPANDED))

    # three-phase API (npore_upload / npore_run / npore_download)
    def upload(self, packed: PackedBatch):
        check_item_sizes(packed.ref_len, packed.seq_len)
        b = packed.c_struct()
        self._check(self._L.npore_upload(self._ctx, C.byref(b)), "npore_upload")

    def run(self, flags: int = 0):
        self._check(self._L.npore_run(self._ctx, flags), "npore_run")

    def download(self, result: BatchResult):
        r = result.c_struct()
        self._check(self._L.npore_download(self._ctx, C.byref(r)), "npore_download")
        return result

    def align_packed(self, packed: PackedBatch, flags: int = 0, result: BatchResult = None) -> BatchResult:
        """npore_align_batch: host buffers in, host buffers out."""
        check_item_sizes(packed.ref_len, packed.seq_len)
        result = result or self.new_result(packed, flags)
        b, r = packed.c_struct(), result.c_struct()
        self._check(self._L.npore_align_batch(self._ctx, C.byref(b), flags, C.byref(r)), "npore_align_batch")
        return result

    def stats(self) -> dict:
        s = _lib.Stats()
        self._check(self._L.npore_last_stats(self._ctx, C.byref(s)), "npore_last_stats")
        return s.as_dict()

    def get_np_info(self, codes: np.ndarray) -> np.ndarray:
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        out = np.zeros((max(len(codes), 1), 2, self.params["max_n"]), dtype=np.int32)
        self._check(self._L.npore_get_np_info(self._ctx, codes.ctypes.data if len(codes) else None, len(codes), out.ctypes.data), "npore_get_np_info")
        return out[:len(codes)]

    def get_np_info_batch(self, seqs):
        """get_np_info for many code arrays in one launch (one CTA each); returns a list of int32 [len, 2, max_n]."""
        seqs = [np.ascontiguousarray(s, dtype=np.uint8) for s in seqs]
        off = np.zeros(len(seqs) + 1, dtype=np.int64)
        np.cumsum([len(s) for s in seqs], out=off[1:])
        if off[-1] == 0:
            return [np.zeros((0, 2, self.params["max_n"]), np.int32) for _ in seqs]
        codes = np.concatenate(seqs)
        out = np.zeros((int(off[-1]), 2, self.params["max_n"]), dtype=np.int32)
        self._check(self._L.npore_get_np_info_batch(self._ctx, len(seqs), codes.ctypes.data, off.ctypes.data, out.ctypes.data), "npore_get_np_info_batch")
        return [out[off[i]:off[i + 1]] for i in range(len(seqs))]

    def confusion_batch(self, pb):
        """calc_confusion_matrices (bam.pyx:351-510) for the ranges of a confusion.PileupPack; returns int64
        subs[5,5], nps[max_n,max_l+1,max_l+1], inss[max_l+1], dels[max_l+1] summed over the ranges.
        A pack with a `seq_nib` attribute (not None) is in the nibble form of npore_pileup_batch: bases in BAM's 4-bit packing
        (seq_nib, seq_nib_start), phred+33 qualities and has_qual; its seq_ascii is ignored."""
        from ._lib import PileupBatch
        T = self.params["max_l"] + 1
        subs = np.zeros((5, 5), np.int64); nps = np.zeros((self.params["max_n"], T, T), np.int64)
        inss = np.zeros(T, np.int64); dels = np.zeros(T, np.int64)
        ptr = lambda a: a.ctypes.data if a is not None and a.size else None   # noqa: E731
        b = PileupBatch(len(pb.range_start), ptr(pb.range_start), ptr(pb.range_end), ptr(pb.ref_ascii), pb.ref_off.ctypes.data,
                        len(pb.read_pos), ptr(pb.read_pos), ptr(pb.seq_ascii), ptr(pb.qual), pb.seq_off.ctypes.data,
                        ptr(pb.cigar_rle), pb.cigar_off.ctypes.data, ptr(pb.range_reads), pb.range_reads_off.ctypes.data,
                        int(pb.min_base_q))
        nib = getattr(pb, "seq_nib", None)
        if nib is not None:                  # the pointer must be set even when every read is empty
            b.seq_nib, b.seq_nib_start, b.seq_nib_bytes = nib.ctypes.data, ptr(pb.seq_nib_start), len(nib)
            b.has_qual = ptr(pb.has_qual)
        self._check(self._L.npore_confusion_batch(self._ctx, C.byref(b), subs.ctypes.data, nps.ctypes.data, inss.ctypes.data,
                                                  dels.ctypes.data), "npore_confusion_batch")
        return subs, nps, inss, dels

    # convenience: python objects in, python objects out
    def align_many(self, refs, seqs, cigars, standardize=False, collapse=False):
        """refs/seqs: lists of uint8 code arrays; cigars: CIGAR texts (run-length or expanded).
        Returns (list of CIGAR strings, list of per-chunk score arrays, status array)."""
        rles = [cigar_to_rle(c) for c in cigars]
        packed = PackedBatch([np.ascontiguousarray(r, dtype=np.uint8) for r in refs],
                             [np.ascontiguousarray(s, dtype=np.uint8) for s in seqs], rles, pinned=False)
        flags = (NPORE_OUT_STANDARDIZE if standardize else 0) | (NPORE_OUT_RLE if collapse else 0)
        res = self.align_packed(packed, flags, self.new_result(packed, flags, pinned=False))
        if collapse:
            outs = [res.cigar_text(i) for i in range(packed.n)]
        else:
            outs = [res.ops_str(i) for i in range(packed.n)]
        return outs, [res.scores(i).copy() for i in range(packed.n)], res.status[:packed.n].copy()


class BgzfCompressor:
    """BGZF compression on one device (npore_bgzf_*): compress(buf) returns the BGZF members of buf (no EOF block) as a
    view of a pinned buffer that the next call reuses.  last_device_ms: kernel time of the last call."""

    def __init__(self, device=0):
        self._L = _lib.lib()
        self._z = C.c_void_p()
        self.device = int(device)
        rc = self._L.npore_bgzf_create(C.byref(self._z), self.device)
        if rc != 0:
            self._z = C.c_void_p()
            raise NporeError(f"npore_bgzf_create failed: {self._L.npore_strerror(rc).decode()} "
                             "(npore_b200 needs a CUDA device; there is no CPU fallback)")
        self._in = self._out = None
        self.last_device_ms = self.last_index_ms = 0.0

    def compress(self, buf):
        src = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf.reshape(-1).view(np.uint8)
        n = len(src)
        if self._in is None or len(self._in[0]) < n:
            self._in = _pinned(n + n // 4, np.uint8)
        cap = int(self._L.npore_bgzf_bound(n))
        if self._out is None or len(self._out[0]) < cap:
            self._out = _pinned(cap + cap // 4, np.uint8)
        pin_in, pin_out = self._in[0], self._out[0]
        pin_in[:n] = src
        got, ms = C.c_int64(), C.c_float()
        rc = self._L.npore_bgzf_compress(self._z, pin_in.ctypes.data, n, pin_out.ctypes.data, len(pin_out), C.byref(got), C.byref(ms))
        if rc != 0:
            raise NporeError(f"npore_bgzf_compress: {self._L.npore_strerror(rc).decode()}")
        self.last_device_ms = float(ms.value)
        return pin_out[:got.value]

    def index(self, rec_off, base):
        """BAM index lists of the records of the last compress() call (npore_bgzf_index): rec_off[n+1] are the records' offsets
        in its input, base the file offset its first member is written at.  Returns {"chunks": (n, 4), "refs": (m, 7),
        "windows": (w,)} uint64 arrays (copies); ValueError when the records cannot be indexed.  last_index_ms: kernel time."""
        rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
        lists, ms = _lib.BaiLists(), C.c_float()
        rc = self._L.npore_bgzf_index(self._z, rec_off.ctypes.data, len(rec_off) - 1, int(base), C.byref(lists), C.byref(ms))
        if rc != 0:
            if lists.error_bits:
                why = [w for b, w in ((1, "records out of coordinate order"), (2, "inconsistent record bytes"),
                                      (4, "records without a reference or position")) if lists.error_bits & b]
                raise ValueError(f"cannot index the BAM output: {', '.join(why)}")
            raise NporeError(f"npore_bgzf_index: {self._L.npore_strerror(rc).decode()}")
        self.last_index_ms = float(ms.value)

        def rows(ptr, n, width):
            if not n:
                return np.zeros((0, width) if width > 1 else 0, np.uint64)
            a = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint64)), shape=(n * width,)).copy()
            return a.reshape(n, width) if width > 1 else a
        return {"chunks": rows(lists.chunks, lists.n_chunks, 4), "refs": rows(lists.refs, lists.n_refs, 7),
                "windows": rows(lists.windows, lists.n_windows, 1)}

    def close(self):
        if getattr(self, "_z", None) and self._z.value:
            self._L.npore_bgzf_destroy(self._z)
            self._z = C.c_void_p()

    __del__ = close


class PipelinedRealigner:
    """Several batches in flight on one GPU: `n_inflight` independent contexts, each with its own CUDA stream and host
    thread.  While one batch is in its kernels, the next one's host->device copies and the previous one's device->host
    copies proceed, and the tail of one forward kernel (SMs going idle) is filled by the head of the next.  Batches are
    independent (bam.pyx:51), so nothing is shared between the contexts; results come back as futures, in submit order
    if the caller keeps the futures in order."""

    def __init__(self, sub_scores, np_scores, n_inflight=2, **kw):
        import queue
        from concurrent.futures import ThreadPoolExecutor
        self.engines = [Realigner(sub_scores, np_scores, **kw) for _ in range(max(1, n_inflight))]
        self._free = queue.SimpleQueue()
        for e in self.engines:
            self._free.put(e)
        self._pool = ThreadPoolExecutor(len(self.engines))

    def submit(self, packed: PackedBatch, flags: int = 0, result: BatchResult = None, pinned_result=False):
        """Future of (BatchResult, stats dict) for npore_align_batch on the next free context."""
        def work():
            import time
            eng = self._free.get()
            try:
                t0 = time.perf_counter()
                out = result or eng.new_result(packed, flags, pinned=pinned_result)
                t1 = time.perf_counter()
                res = eng.align_packed(packed, flags, out)
                st = eng.stats()
                st["wall"] = (t0, t1, time.perf_counter())      # context acquired, result buffers ready, batch done (perf_counter)
                return res, st
            finally:
                self._free.put(eng)
        return self._pool.submit(work)

    def close(self):
        self._pool.shutdown(wait=True)
        for e in self.engines:
            e.close()
