"""BAM index (SAM spec 5.2) written beside realign_bam's BAM output, and read back by bamio.read_bai.

The reference indexer here is written from the spec and htslib's indexing rules (hts_idx_push, compress_binning without the
parent-bin move, update_loff): it walks a BGZF file member by member with zlib, maps each record to its virtual offset (a
position on a member boundary takes the "next member, offset 0" form) and builds the expected .bai bytes record by record.
  - CPU: the pipeline with the echo engine and a zlib stand-in compressor whose index() is the reference indexer applied to
    one batch; query completeness of read_bai(...).query; refusals.
  - GPU: npore_bgzf_index against the reference indexer batch by batch, and realign_bam(index=True) end to end."""
import gzip
import os
import re
import struct
import zlib

import numpy as np
import pytest

from npore_b200 import bamio, cfg, synth

HERE = os.path.dirname(os.path.abspath(__file__))
BLOCK = 65280
UNSET = (1 << 64) - 1


# ------------------------------------------------------------------------------------------------ reference indexer
def reg2bin(beg, end):
    end -= 1
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return off + (beg >> shift)
    return 0


def record_fields(data, at):
    """(ref_id, pos, end, bin, mapped, record length) of the record whose block_size field is at data[at]."""
    bs, ref, pos, l_name, _mapq, _bin, n_cig, flag = struct.unpack_from("<iiiBBHHH", data, at)
    cig = struct.unpack_from(f"<{n_cig}I", data, at + 36 + l_name)
    span = sum(w >> 4 for w in cig if (w & 15) in (0, 2, 3, 7, 8))
    mapped = not flag & 4
    end = pos + (span if mapped and span else 1)
    return ref, pos, end, reg2bin(pos, end), mapped, bs + 4


def walk_members(data):
    """[(file offset, inflated offset, inflated size)] of every member, and the inflated stream."""
    out, raw, p, u = [], [], 0, 0
    while p < len(data):
        bsize = struct.unpack_from("<H", data, p + 16)[0] + 1
        d = zlib.decompressobj(-15)
        payload = d.decompress(data[p + 18:p + bsize - 8]) + d.flush()
        out.append((p, u, len(payload)))
        raw.append(payload)
        p += bsize
        u += len(payload)
    return out, b"".join(raw)


def voffset_map(members, end_offset):
    """u -> voffset; a position at the end of a member maps to the start of the next one."""
    starts = np.array([u for _, u, n in members if n], np.int64)
    offs = [c for c, _, n in members if n]
    sizes = [n for _, _, n in members if n]

    def v(u):
        k = int(np.searchsorted(starts, u, "right")) - 1
        if k < 0 or u >= starts[k] + sizes[k]:
            nxt = [c for c, s, _ in members if s >= u]          # the next member, the EOF block included
            return (nxt[0] if nxt else end_offset) << 16
        return offs[k] << 16 | (u - int(starts[k]))
    return v


class RefIndex:
    """htslib's index build, one record at a time (records in file order)."""

    def __init__(self, n_refs):
        self.bins = [dict() for _ in range(n_refs)]
        self.lin = [dict() for _ in range(n_refs)]
        self.meta = [None] * n_refs
        self.last = None                    # (ref, bin) of the open chunk
        self.n_refs = n_refs

    def push(self, ref, pos, end, bin_, mapped, vbeg, vend):
        if self.last != (ref, bin_):
            self.bins[ref].setdefault(bin_, []).append([vbeg, vend])
            self.last = (ref, bin_)
        else:
            self.bins[ref][bin_][-1][1] = vend
        m = self.meta[ref] or [vbeg, vend, 0, 0]
        m[1] = vend
        m[2 if mapped else 3] += 1
        self.meta[ref] = m
        if mapped:
            for w in range(pos >> 14, ((end - 1) >> 14) + 1):
                self.lin[ref].setdefault(w, vbeg)

    def merged_bins(self, ref):
        out = {}
        for b, lst in sorted(self.bins[ref].items()):
            m = [list(lst[0])]
            for beg, end in lst[1:]:
                if m[-1][1] >> 16 >= beg >> 16:
                    m[-1][1] = max(m[-1][1], end)
                else:
                    m.append([beg, end])
            out[b] = m
        return out

    def to_bytes(self):
        out = [b"BAI\1", struct.pack("<i", self.n_refs)]
        for ref in range(self.n_refs):
            if self.meta[ref] is None:
                out.append(struct.pack("<ii", 0, 0))
                continue
            bins = self.merged_bins(ref)
            out.append(struct.pack("<i", len(bins) + 1))
            for b, lst in bins.items():
                out.append(struct.pack("<Ii", b, len(lst)) + b"".join(struct.pack("<QQ", *c) for c in lst))
            out.append(struct.pack("<IiQQQQ", 37450, 2, *self.meta[ref]))
            lin = self.lin[ref]
            n = max(lin) + 1 if lin else 0
            vals, prev = [], self.meta[ref][0]
            for w in range(n):
                prev = lin.get(w, prev)
                vals.append(prev)
            out.append(struct.pack("<i", n) + b"".join(struct.pack("<Q", v) for v in vals))
        out.append(struct.pack("<Q", 0))
        return b"".join(out)


def header_end(u):
    l_text = struct.unpack_from("<i", u, 4)[0]
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", u, p)[0]
    p += 4
    for _ in range(n_ref):
        p += 4 + struct.unpack_from("<i", u, p)[0] + 4
    return p, n_ref


def file_records(path):
    """[(ref, pos, end, bin, mapped, vbeg, vend, record index)] of a BGZF BAM file, and its reference count."""
    data = open(path, "rb").read()
    members, u = walk_members(data)
    v = voffset_map(members, len(data))
    p, n_ref = header_end(u)
    out, k = [], 0
    while p < len(u):
        ref, pos, end, b, mapped, ln = record_fields(u, p)
        out.append((ref, pos, end, b, mapped, v(p), v(p + ln), k))
        p += ln
        k += 1
    return out, n_ref


def ref_bai(path):
    recs, n_ref = file_records(path)
    ix = RefIndex(n_ref)
    for ref, pos, end, b, mapped, vb, ve, _ in recs:
        ix.push(ref, pos, end, b, mapped, vb, ve)
    return ix.to_bytes()


def ref_batch_lists(payload, sizes, rec_off, base):
    """The reference indexer on one batch: the lists npore_bgzf_index returns for these records."""
    moff = np.concatenate(([0], np.cumsum(sizes))).astype(np.int64) + base
    n_in = len(payload)

    def v(u):
        return int(moff[-1]) << 16 if u >= n_in else int(moff[u // BLOCK]) << 16 | (u % BLOCK)
    recs = [record_fields(payload, int(a))[:5] + (v(int(a)), v(int(b))) for a, b in zip(rec_off[:-1], rec_off[1:])]
    refs = sorted({r[0] for r in recs})
    ix = RefIndex(max(refs) + 1)
    for r in recs:
        ix.push(*r)
    chunks, rows, wins = [], [], []
    for ref in refs:
        for b, lst in ix.merged_bins(ref).items():
            chunks += [(ref, b, beg, end) for beg, end in lst]
        lin = ix.lin[ref]
        wf = min(lin) if lin else 0
        nw = max(lin) - wf + 1 if lin else 0
        wins += [lin.get(w, UNSET) for w in range(wf, wf + nw)]
        rows.append((ref, *ix.meta[ref], wf, nw))
    return {"chunks": np.array(chunks, np.uint64).reshape(-1, 4), "refs": np.array(rows, np.uint64).reshape(-1, 7),
            "windows": np.array(wins, np.uint64)}


# ------------------------------------------------------------------------------------------------ stand-ins
class _EchoEngine:
    """The "realigned" CIGAR of every record is its input CIGAR; submit number fail_at (1-based) fails."""

    def __init__(self, fail_at=0):
        self.fail_at, self.submitted = fail_at, 0

    def submit(self, packed, flags=0):
        import concurrent.futures
        import time
        import types
        self.submitted += 1
        fut = concurrent.futures.Future()
        if self.submitted == self.fail_at:
            fut.set_exception(RuntimeError("stand-in batch failure"))
            return fut
        t = time.perf_counter()
        res = types.SimpleNamespace(rle=packed.cigar_rle, rle_off=packed.cigar_off, status=np.zeros(max(packed.n, 1), np.int32))
        fut.set_result((res, {"ms_kernels_total": 0.0, "ms_h2d": 0.0, "ms_plan": 0.0, "ms_d2h": 0.0, "fwd_warps_per_sm": 0, "wall": (t, t, t)}))
        return fut


class _ZlibCompressor:
    """BGZF members from zlib; index() is the reference indexer applied to the last compressed batch."""

    def compress(self, buf):
        self.last = bytes(buf)
        blocks = [bamio._bgzf_block(self.last[i:i + BLOCK], 1) for i in range(0, len(self.last), BLOCK)]
        self.sizes = [len(b) for b in blocks]
        return b"".join(blocks)

    def index(self, rec_off, base):
        return ref_batch_lists(self.last, self.sizes, rec_off, base)


@pytest.fixture(scope="module")
def fixture_bam(tmp_path_factory, tables):
    """Two contigs of 1 kb reads with and without qualities (the fixture of test_bam_output.py)."""
    S, NP = tables
    rng = np.random.default_rng(99)
    cm = synth.call_length_model(NP)
    contigs, recs = [], []
    for ci, (name, length, n_reads) in enumerate((("chrA", 24_000, 50), ("chrB", 15_000, 30))):
        ref, tr = synth.make_reference_with_tracts(length, rng)
        contigs.append((name, ref))
        for k, rd in enumerate(synth.make_reads(ref, n_reads, 1000, rng, cm, tracts=tr)):
            recs.append({"name": f"{name}_{rd[0]}", "flag": 0, "ref_id": ci, "pos": rd[3], "mapq": 60, "seq": rd[7],
                         "qual": None if k % 4 == 1 else bytes(rng.integers(0, 40, len(rd[7])).astype(np.uint8)),
                         "cigar": [(int(a), b) for a, b in re.findall(r"(\d+)(\D)", rd[5])], "tags": {"HP": k % 3}})
    path = str(tmp_path_factory.mktemp("bai") / "in.bam")
    bamio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n", [(n, len(s)) for n, s in contigs], recs)
    return path, dict(contigs), S, NP


@pytest.fixture
def stand_ins(fixture_bam, monkeypatch):
    _, _, S, NP = fixture_bam
    monkeypatch.setattr(cfg.args, "sub_scores", S)
    monkeypatch.setattr(cfg.args, "np_scores", NP)
    monkeypatch.setattr(cfg.args, "out_prefix", cfg.args.out_prefix)
    made = []

    def install(fail_at=0):
        eng = _EchoEngine(fail_at)
        monkeypatch.setattr(bamio, "_pipeline", lambda sub, npt, n_inflight, device=None: eng)
        monkeypatch.setattr(bamio, "_compressor", lambda device, slot: made.append((device, slot)) or _ZlibCompressor())
        return made
    return install


def _records_in_chunks(recs, chunks):
    return {r[7] for r in recs if any(b <= r[5] < e for b, e in chunks.tolist())}


def _brute(recs, ref, beg, end):
    return {r[7] for r in recs if r[0] == ref and r[1] < end and r[2] > beg}


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("kw", [{}, {"window_bytes": 20_000, "max_batch_ops": 5_000}, {"window_bytes": 0, "n_inflight": 1},
                                {"devices": [0, 0], "max_batch_ops": 5_000}, {"devices": [0, 0, 0], "max_batch_ops": 5_000}])
def test_index_matches_the_reference_indexer(fixture_bam, stand_ins, tmp_path, kw):
    bam, fa, _, _ = fixture_bam
    stand_ins()
    tm = {}
    n = bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "x"), argv=["t"], timings=tm, out_format="bam", index=True, **kw)
    assert n == 80 and "index" in tm
    path = str(tmp_path / "x.bam")
    assert open(path + ".bai", "rb").read() == ref_bai(path)
    assert sorted(os.listdir(tmp_path)) == ["x.bam", "x.bam.bai"]


def test_no_index_by_default_and_a_stale_index_is_removed(fixture_bam, stand_ins, tmp_path):
    bam, fa, _, _ = fixture_bam
    stand_ins()
    tm = {}
    bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "x"), argv=["t"], out_format="bam", index=True)
    bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "x"), argv=["t"], out_format="bam", timings=tm)
    assert os.listdir(tmp_path) == ["x.bam"] and "index" not in tm


def _long_read_bam(path, seed=5, n_reads=600):
    """Sorted reads on two contigs, 300 bp to 40 kb of reference (D operations), many starting or ending on 16 kb / 128 kb
    window edges; BGZF members of 9,000 bytes, so that records straddle members."""
    rng = np.random.default_rng(seed)
    recs = []
    for ci, length in enumerate((1_300_000, 400_000)):
        edges = [e for k in (14, 17, 20) for e in range(1 << k, length, 1 << k)]
        pos = np.sort(np.concatenate([rng.integers(0, length - 50_000, n_reads // 2), rng.choice(edges, 60) - rng.integers(-2, 3, 60)]))
        for k, p in enumerate(pos.tolist()):
            span = int(rng.choice([300, 2_000, 17_000, 40_000]))
            m = 150
            cig = [(m, "M"), (span - 2 * m, "D"), (m, "M")] if span > 2 * m else [(span, "M")]
            seq = "".join(rng.choice(list("ACGT"), sum(n for n, op in cig if op == "M")))
            recs.append({"name": f"r{ci}_{k}", "flag": 4 if k % 37 == 5 else 0, "ref_id": ci, "pos": max(int(p), 0), "mapq": 60,
                         "seq": seq, "qual": None, "cigar": cig, "tags": {"HP": 0}})
    refs = [("c1", 1_300_000), ("c2", 400_000)]
    bamio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n", refs, recs)
    data = open(path, "rb").read()
    raw = gzip.decompress(data)
    with open(path, "wb") as fh:                           # re-cut into 9,000-byte members
        for i in range(0, len(raw), 9000):
            fh.write(bamio._bgzf_block(raw[i:i + 9000], 1))
        fh.write(bamio.BGZF_EOF)
    return refs


def test_query_returns_every_overlapping_record(tmp_path):
    path = str(tmp_path / "long.bam")
    refs = _long_read_bam(path)
    with open(path + ".bai", "wb") as fh:
        fh.write(ref_bai(path))
    recs, _ = file_records(path)
    assert any(r[2] - r[1] > 16_384 for r in recs)
    ix = bamio.read_bai(path + ".bai")
    rng = np.random.default_rng(1)
    cases = []
    for ref, (_, length) in enumerate(refs):
        for e in (1 << 14, 1 << 17, 1 << 20):
            cases += [(ref, b, b + w) for b in range(e, length, e)[:3] for w in (1, 1000, 20_000)]
        cases += [(ref, int(b), int(b) + int(w)) for b, w in zip(rng.integers(0, length, 90), rng.integers(1, 200_000, 90))]
    assert len(cases) >= 200
    for ref, beg, end in cases:
        got = _records_in_chunks(recs, ix.query(ref, beg, end))
        want = _brute(recs, ref, beg, end)
        assert want <= got, (ref, beg, end, sorted(want - got)[:5])
        # and no record overlapping the region is missed by the chunks' own overlap filter
        assert {k for k in got if recs[k][2] > beg and recs[k][1] < end} == want


def test_read_bai_refuses_malformed_files(tmp_path):
    path = str(tmp_path / "long.bam")
    _long_read_bam(path, n_reads=50)
    good = ref_bai(path)
    for name, data in (("magic", b"BAX\1" + good[4:]), ("short", good[:len(good) // 2]), ("empty", b"")):
        p = tmp_path / f"{name}.bai"
        p.write_bytes(data)
        with pytest.raises(ValueError, match=str(p)):
            bamio.read_bai(str(p))
    p = tmp_path / "ok.bai"
    p.write_bytes(good)
    assert len(bamio.read_bai(str(p)).refs) == 2


def test_index_refusals_before_any_file(fixture_bam, stand_ins, tmp_path):
    bam, fa, _, _ = fixture_bam
    made = stand_ins()
    for kw in ({"out_format": "sam"},
               {"out_format": "bam", "regions": [("chrB", 0, 5_000), ("chrA", 0, 5_000)]},
               {"out_format": "bam", "regions": [("chrA", 0, 5_000), ("chrA", 4_000, 9_000)]},
               {"out_format": "bam", "regions": [("chrA", 6_000, 9_000), ("chrA", 0, 5_000)]}):
        with pytest.raises(ValueError):
            bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "out"), argv=["t"], index=True, **kw)
    assert os.listdir(tmp_path) == [] and made == []
    big = str(tmp_path.parent / "big_contig.bam")
    bamio.write_bam(big, "@HD\tVN:1.6\tSO:coordinate\n", [("huge", 1 << 29)], [])
    with pytest.raises(ValueError, match="2\\^29|536870911"):
        bamio.realign_bam(big, {"huge": ""}, out_prefix=str(tmp_path / "out"), argv=["t"], out_format="bam", index=True)
    assert os.listdir(tmp_path) == []
    # sorted regions that no read spans are fine
    n = bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "ok"), argv=["t"], out_format="bam", index=True,
                          regions=[("chrA", 0, 5_000), ("chrA", 12_000, 20_000), ("chrB", 0, 4_000)], max_batch_ops=5_000)
    assert n > 0 and open(tmp_path / "ok.bam.bai", "rb").read() == ref_bai(str(tmp_path / "ok.bam"))


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_a_read_selected_by_two_regions_is_not_indexed(fixture_bam, stand_ins, tmp_path, devices):
    """Touching regions select the reads across their edge twice, so the output is not sorted: no index is written."""
    bam, fa, _, _ = fixture_bam
    stand_ins()
    with pytest.raises(ValueError, match="coordinate order"):
        bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "t"), argv=["t"], out_format="bam", index=True, devices=devices,
                          regions=[("chrA", 0, 5_000), ("chrA", 5_000, 9_000)], max_batch_ops=5_000)
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".bai") or ".part" in f]


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_failed_batch_leaves_no_index(fixture_bam, stand_ins, tmp_path, devices):
    bam, fa, _, _ = fixture_bam
    stand_ins(fail_at=3)
    with pytest.raises(RuntimeError, match="stand-in batch failure"):
        bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "out"), argv=["t"], window_bytes=20_000, max_batch_ops=5_000,
                          devices=devices, out_format="bam", index=True)
    assert not [f for f in os.listdir(tmp_path) if ".part" in f or f.endswith(".bai") or ".tmp" in f]


# ------------------------------------------------------------------------------------------------ reading through an index
@pytest.fixture(scope="module")
def long_bam(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("long") / "long.bam")
    refs = _long_read_bam(path)
    with open(path + ".bai", "wb") as fh:
        fh.write(ref_bai(path))
    recs, _ = file_records(path)
    return path, refs, recs


REGIONS = [[("c1", 500_000, 510_000)], [("c2", 390_000, 400_000)], [("c1", 100_000, 300_000), ("c2", 0, 50_000)],
           [("c1", 0, 10)], [("c1", (1 << 20) - 5, (1 << 20) + 5)], [("nope", 0, 5)]]


@pytest.mark.parametrize("window_bytes", [0, 20_000])
def test_restricted_reader_yields_the_chunk_records(long_bam, window_bytes):
    path, refs, recs = long_bam
    ix = bamio.read_bai(path + ".bai")
    names = [n for n, _ in refs]
    for regions in REGIONS:
        nb = bamio.NativeBam(path, window_bytes=window_bytes, regions=regions)
        assert nb.index == path + ".bai"
        vo, pos, ref, end = [], [], [], []
        while True:
            if window_bytes and not nb.advance():
                break
            vo += nb.voffsets().tolist(); pos += nb.pos.tolist(); ref += nb.ref_id.tolist(); end += nb.end.tolist()
            if not window_bytes:
                break
        chunks = bamio.region_chunks(ix, refs, regions)
        want = [r for r in recs if any(b <= r[5] < e for b, e in chunks.tolist())]
        assert vo == [r[5] for r in want], regions                  # the voffsets of the reference walk, in file order
        assert (ref, pos) == ([r[0] for r in want], [r[1] for r in want])
        for ctg, beg, stop in regions:                              # every record overlapping a region is there
            if ctg in names:
                got = {v for v, q, p, e in zip(vo, ref, pos, end) if q == names.index(ctg) and p < stop and e > beg}
                assert got == {r[5] for r in recs if r[0] == names.index(ctg) and r[1] < stop and r[2] > beg}
        nb.close()


def test_restricted_reader_reads_little_of_the_file(long_bam):
    path, _, _ = long_bam
    size = os.path.getsize(path)
    whole = bamio.NativeBam(path)
    assert whole.bytes_read == size
    for regions in ([("c1", 500_000, 510_000)], [("c2", 390_000, 400_000)]):
        nb = bamio.NativeBam(path, regions=regions)
        assert 0 < nb.n and nb.bytes_read < 0.25 * size, (regions, nb.bytes_read, size)


def test_stale_or_malformed_index(long_bam, tmp_path):
    path, _, recs = long_bam
    import shutil
    mine = str(tmp_path / "x.bam")
    shutil.copy(path, mine)
    shutil.copy(path + ".bai", str(tmp_path / "x.bai"))            # the {path without .bam}.bai form
    nb = bamio.NativeBam(mine, regions=[("c2", 390_000, 400_000)])
    assert nb.index == str(tmp_path / "x.bai") and nb.n < len(recs)
    st = os.stat(mine)
    os.utime(str(tmp_path / "x.bai"), (st.st_atime, st.st_mtime - 100))         # older than the BAM: not used
    nb = bamio.NativeBam(mine, regions=[("c2", 390_000, 400_000)])
    assert nb.index is None and nb.n == len(recs) and nb.bytes_read == os.path.getsize(mine)
    good = open(path + ".bai", "rb").read()
    for bad in (b"BAX\1" + good[4:], good[:len(good) // 3]):
        with open(mine + ".bai", "wb") as fh:
            fh.write(bad)
        with pytest.raises(ValueError, match="x.bam.bai"):
            bamio.NativeBam(mine, regions=[("c1", 0, 1000)])


@pytest.mark.parametrize("fmt", ["sam", "bam"])
def test_realign_regions_through_the_index_is_byte_identical(fixture_bam, stand_ins, tmp_path, fmt):
    bam, fa, _, _ = fixture_bam
    stand_ins()
    plain, indexed = str(tmp_path / "plain.bam"), str(tmp_path / "indexed.bam")
    raw = gzip.decompress(open(bam, "rb").read())
    for p in (plain, indexed):                                      # 20,000-byte members: several per region
        with open(p, "wb") as fh:
            for i in range(0, len(raw), 20_000):
                fh.write(bamio._bgzf_block(raw[i:i + 20_000], 1))
            fh.write(bamio.BGZF_EOF)
    with open(indexed + ".bai", "wb") as fh:
        fh.write(ref_bai(indexed))
    for k, kw in enumerate(({"regions": [("chrB", 3_000, 9_000)]},
                            {"regions": [("chrB", 3_000, 9_000)], "window_bytes": 20_000, "max_batch_ops": 5_000},
                            {"regions": [("chrA", 0, 5_000), ("chrB", 0, 4_000)], "max_batch_ops": 5_000},
                            {"regions": [("chrA", 2_000, 20_000), ("chrA", 10_000, 12_000)], "max_reads": 17},
                            {"regions": [("chrA", 15_000, 16_000)], "max_reads": 3, "window_bytes": 20_000})):
        outs = []
        for src in (plain, indexed):
            pre = str(tmp_path / f"o{k}_{os.path.basename(src)[:-4]}")
            n = bamio.realign_bam(src, fa, out_prefix=pre, argv=["t"], out_format=fmt, **kw)
            outs.append((n, open(f"{pre}.{fmt}", "rb").read()))
        assert outs[0][0] > 0 and outs[0][0] == outs[1][0], kw
        if fmt == "bam" and kw.get("window_bytes"):
            # streamed windows: the region's records are cut into batches per window, and a restricted window holds other records
            # than a full one, so the BGZF member boundaries (one member run per batch) may differ; the BAM stream may not
            assert gzip.decompress(outs[0][1]) == gzip.decompress(outs[1][1]), kw
        else:
            assert outs[0][1] == outs[1][1], kw
    nb = bamio.NativeBam(indexed, regions=[("chrB", 3_000, 9_000)])
    assert nb.index == indexed + ".bai" and nb.bytes_read < bamio.NativeBam(plain, regions=[("chrB", 3_000, 9_000)]).bytes_read


def test_index_kernels_do_not_spill():
    """-Xptxas -v for sm_100a: the bai.cuh kernels use no stack frame and spill nothing."""
    import shutil
    import subprocess
    import tempfile
    nvcc = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
    if nvcc is None:
        pytest.skip("nvcc not available")
    src = os.path.join(os.path.dirname(HERE), "npore_b200", "csrc", "bai.cuh")
    with tempfile.TemporaryDirectory() as d:
        unit = os.path.join(d, "k.cu")
        with open(unit, "w") as fh:
            fh.write(f'#include "{src}"\n')
        r = subprocess.run([nvcc, "-cubin", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v",
                            "-o", os.path.join(d, "k.cubin"), unit], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    report = r.stderr.split("Compiling entry function")[1:]
    kernels = [blk for blk in report if "bai_" in blk.split("\n")[0]]
    assert len(kernels) == 4, r.stderr
    for blk in kernels:
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in blk, blk


# ------------------------------------------------------------------------------------------------ GPU
def _raw_record(ref, pos, span, name, flag=0, pad=0):
    cig = [(span, 0)] if span <= 150 else [(100, 0), (span - 150, 2), (50, 0)]
    n_seq = sum(n for n, op in cig if op == 0)
    nm = name.encode() + b"\0"
    tags = b"XZZ" + b"x" * pad + b"\0" if pad else b""
    body = struct.pack("<iiBBHHHiiii", ref, pos, len(nm), 60, reg2bin(pos, pos + span), len(cig), flag, n_seq, -1, -1, 0)
    body += nm + b"".join(struct.pack("<I", n << 4 | op) for n, op in cig) + bytes((n_seq + 1) // 2) + b"\xff" * n_seq + tags
    return struct.pack("<i", len(body)) + body


def synthetic_batch(rng, min_bytes=3 << 20):
    """Sorted records on two contigs, at least min_bytes of them, crossing 16 kb / 128 kb / 1 Mb edges, one record starting exactly on a
    member boundary (65,280 x 3) and many straddling members."""
    out, offs, at = [], [0], 0
    plan = []
    for ref, length in ((0, 3_000_000), (1, 2_500_000)):
        pos = np.sort(np.concatenate([rng.integers(0, length - 60_000, 6_500),
                                      np.repeat([(1 << 14) * 7, (1 << 17) * 3, 1 << 20, 2 << 20], 5) - rng.integers(0, 3_000, 20)]))
        plan += [(ref, int(p)) for p in pos]
    target = 3 * BLOCK
    for k, (ref, p) in enumerate(plan):
        span = int(rng.choice([80, 2_000, 20_000, 150_000]))
        rec = _raw_record(ref, p, span, f"q{k}", flag=4 if k % 53 == 7 else 0)
        if at < target < at + len(rec) + 400:               # a filler record that ends exactly on the boundary (gap >= 400)
            small = _raw_record(ref, p, 80, f"f{k}")
            fill = _raw_record(ref, p, 80, f"f{k}", pad=target - at - len(small) - 4)
            out.append(fill)
            at += len(fill)
            offs.append(at)
        out.append(rec)
        at += len(rec)
        offs.append(at)
    assert target in offs and at >= min_bytes
    return b"".join(out), np.array(offs, np.int64)


@pytest.fixture(scope="module")
def compressor(have_gpu):
    if not have_gpu:
        pytest.skip("needs a CUDA device")
    from npore_b200.engine import BgzfCompressor
    z = BgzfCompressor(0)
    yield z
    z.close()


def _check_batch(z, payload, rec_off, base):
    blob = bytes(z.compress(payload))
    sizes = [len(m) for m in _split_members(blob)]
    got = z.index(rec_off, base)
    want = ref_batch_lists(payload, sizes, rec_off, base)
    for k in ("chunks", "refs", "windows"):
        assert np.array_equal(got[k], want[k]), (k, got[k][:5], want[k][:5])
    return got


def _split_members(data):
    out, p = [], 0
    while p < len(data):
        bsize = struct.unpack_from("<H", data, p + 16)[0] + 1
        out.append(data[p:p + bsize])
        p += bsize
    return out


@pytest.mark.gpu
def test_device_index_matches_reference_on_a_synthetic_batch(compressor):
    payload, rec_off = synthetic_batch(np.random.default_rng(4))
    assert len(payload) >= 3 << 20
    got = _check_batch(compressor, payload, rec_off, 12_345)
    assert len(got["refs"]) == 2 and compressor.last_index_ms > 0
    assert any((int(c[1]) < 4681) for c in got["chunks"])          # records in larger bins than the 16 kb level
    # a record starting on the member boundary maps to (member 3, offset 0)
    _check_batch(compressor, payload[:3 * BLOCK], rec_off[rec_off <= 3 * BLOCK], 0)


@pytest.mark.gpu
def test_device_index_matches_reference_on_the_fixture_batches(fixture_bam, compressor):
    bam, _, _, _ = fixture_bam
    nb = bamio.NativeBam(bam)
    sel = np.arange(nb.n)
    g = nb.gather(sel, want_codes=False, want_cigar=False)
    cig, off = nb.gather_cigar(sel)
    raw, rec_off = bamio.format_sam(nb, sel, g, cig, off, binary=True, offsets=True)
    assert rec_off[-1] == len(raw)
    for lo, hi in ((0, nb.n), (0, 17), (30, 79)):
        part = np.ascontiguousarray(raw[rec_off[lo]:rec_off[hi]])
        _check_batch(compressor, part, rec_off[lo:hi + 1] - rec_off[lo], 999)
    nb.close()


@pytest.fixture
def device_tables(fixture_bam, monkeypatch, have_gpu):
    if not have_gpu:
        pytest.skip("needs a CUDA device")
    _, _, S, NP = fixture_bam
    monkeypatch.setattr(cfg.args, "sub_scores", S)
    monkeypatch.setattr(cfg.args, "np_scores", NP)
    monkeypatch.setattr(cfg.args, "out_prefix", cfg.args.out_prefix)
    monkeypatch.setattr(cfg.args, "max_n", 6)
    monkeypatch.setattr(cfg.args, "max_l", 100)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [{}, {"window_bytes": 20_000, "max_batch_ops": 20_000}, {"regions": [("chrA", 2_000, 9_000), ("chrB", 0, 9_000)]}])
def test_realign_bam_index_on_device(fixture_bam, device_tables, tmp_path, kw):
    bam, fa, _, _ = fixture_bam
    tm = {}
    n = bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "e2e"), argv=["t"], out_format="bam", index=True, timings=tm, **kw)
    path = str(tmp_path / "e2e.bam")
    assert n > 0 and tm["index"] > 0
    assert open(path + ".bai", "rb").read() == ref_bai(path)
    recs, _ = file_records(path)
    ix = bamio.read_bai(path + ".bai")
    rng = np.random.default_rng(2)
    for ref, length in ((0, 24_000), (1, 15_000)):
        for beg, w in zip(rng.integers(0, length, 20).tolist(), rng.integers(1, 8_000, 20).tolist()):
            assert _brute(recs, ref, beg, beg + w) <= _records_in_chunks(recs, ix.query(ref, beg, beg + w))
            nb = bamio.NativeBam(path, regions=[(("chrA", "chrB")[ref], beg, beg + w)])          # the restricted reader
            assert nb.index == path + ".bai"
            got = {v for v, q, p, e in zip(nb.voffsets().tolist(), nb.ref_id, nb.pos, nb.end) if q == ref and p < beg + w and e > beg}
            assert got == {recs[k][5] for k in _brute(recs, ref, beg, beg + w)}


@pytest.mark.gpu
def test_sharded_index_on_devices(fixture_bam, device_tables, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two CUDA devices")
    bam, fa, _, _ = fixture_bam
    bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "many"), argv=["t"], max_batch_ops=20_000, devices=[0, 1], out_format="bam",
                      index=True)
    path = str(tmp_path / "many.bam")
    assert open(path + ".bai", "rb").read() == ref_bai(path)
