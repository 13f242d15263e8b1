"""confusion.count_bam: confusion matrices from a whole BAM file in one streamed pass, and the nibble form of
npore_confusion_batch it feeds.

CPU tests: the device is replaced by a stand-in that decodes each batch (4-bit bases, phred+33 qualities, CIGARs without
clips) and runs oracle/pileup_oracle.py per range; the sum must equal the oracle over the file's reads with their full
CIGARs (soft clips in), and every batch must hold exactly the kept reads that overlap its ranges.  GPU tests (-m gpu):
count_bam == calc_confusion_matrices_batch(load_alignments(...)) bit for bit, the golden windows through a BAM file, the
nibble form == the ASCII form, and argument checks of the nibble form.  Counts are integers: everything is exact."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle
import pileup_oracle as po
from npore_b200 import bamio, cfg, confusion, synth

SEQ16 = "=ACMGRSVTWYHKDBN"
OPS = "MIDNSHP=XB"


@pytest.fixture
def small_cfg(monkeypatch):
    monkeypatch.setattr(cfg.args, "max_n", 6)
    monkeypatch.setattr(cfg.args, "max_l", 100)
    monkeypatch.setattr(cfg.args, "chunk_width", 100000)


def _rec(k, ref_id, r):
    return {"name": f"r{k}", "flag": r[4], "ref_id": ref_id, "pos": r[0], "mapq": r[5], "cigar": r[1], "seq": r[2], "qual": r[3]}


def _special_reads(contig, rng):
    """Reads the generator does not make: a leading S followed by I, hard clips on both ends, '=' and IUPAC bases, an empty
    SEQ, and the flags mpileup drops (unmapped-but-placed, secondary, QC-fail, duplicate)."""
    L = len(contig)
    out = []
    for k in range(12):
        p = int(rng.integers(0, L - 200))
        body = contig[p:p + 150].upper()
        kind = k % 6
        if kind == 0:
            out.append((p, [(3, "S"), (2, "I"), (150, "M"), (4, "S")], "GTA" + "CC" + body + "ACGT", bytes(rng.integers(3, 41, 159).astype(np.uint8)), 0, 60))
        elif kind == 1:
            out.append((p, [(5, "H"), (2, "S"), (150, "M"), (3, "S"), (7, "H")], "TT" + body + "GGG", None, 16, 30))
        elif kind == 2:
            s = "=" + body[1:20] + "M" + body[21:80] + "=" + body[81:]
            out.append((p, [(150, "M")], s, bytes(rng.integers(3, 41, 150).astype(np.uint8)), 0, 60))
        elif kind == 3:
            out.append((p, [(150, "M")], "", None, 0, 60))
        else:
            flag = [0x4, 0x100, 0x200, 0x400][k % 4]
            out.append((p, [(150, "M")], body, None, flag, 60))
    return out


def _make_bam(path, seed, n_reads=(40, 25), read_len=400, unmapped_tail=3):
    """Two contigs with reads, one contig without, unmapped reads at the end.  Returns ({contig: seq}, records)."""
    rng = np.random.default_rng(seed)
    ctgs = {"a": synth.make_reference(int(rng.integers(2500, 4000)), rng, p_np=0.4),
            "b": synth.make_reference(int(rng.integers(1500, 3000)), rng, p_np=0.4),
            "e": synth.make_reference(800, rng)}
    recs = []
    for ref_id, (c, n) in enumerate(zip(("a", "b"), n_reads)):
        reads = synth.make_aligned_reads(ctgs[c], n, read_len, rng) + _special_reads(ctgs[c], rng)
        reads.sort(key=lambda r: r[0])
        recs += [_rec(len(recs) + k, ref_id, r) for k, r in enumerate(reads)]
    for k in range(unmapped_tail):
        recs.append({"name": f"u{k}", "flag": 4, "ref_id": -1, "pos": -1, "mapq": 0, "cigar": [], "seq": "ACGTN" * 20, "qual": None})
    bamio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n", [(c, len(s)) for c, s in ctgs.items()], recs)
    return ctgs, recs


def _read_id(pos, cigar, seq):
    """What identifies a read in a batch: position, CIGAR without S / H, aligned bases."""
    return (pos, tuple((n, op) for n, op in cigar if op not in "SH"), seq)


def _file_reads(path):
    """{contig: [(po.Read with the full CIGAR, read id)]} in file order, every record with a reference."""
    _, refs, recs = bamio.read_bam(path)
    out = {}
    for r in recs:
        if r["ref_id"] < 0:
            continue
        cig = [(int(w) >> 4, OPS[int(w) & 15]) for w in r["cigar"]]
        ops = [op for _, op in cig]
        lead = cig[0][0] if ops[:1] == ["S"] else (cig[1][0] if ops[:2] == ["H", "S"] else 0)
        trail = cig[-1][0] if ops[-1:] == ["S"] else (cig[-2][0] if ops[-2:] == ["S", "H"] else 0)
        seq = r["seq"][lead:len(r["seq"]) - trail]
        out.setdefault(refs[r["ref_id"]][0], []).append(
            (po.Read(r["pos"], cig, r["seq"], None if r["qual"] is None else bytes(r["qual"]), r["flag"]), _read_id(r["pos"], cig, seq)))
    return out


class StandIn:
    """Device stand-in: decodes each nibble-form batch and counts it with the oracle, range by range."""

    def __init__(self):
        self.batches = []

    def confusion_batch(self, pk):
        assert pk.seq_ascii is None and pk.seq_nib is not None
        n = len(pk.read_pos)
        reads, ids = [], []
        for i in range(n):
            a, b = int(pk.seq_off[i]), int(pk.seq_off[i + 1])
            k = int(pk.seq_nib_start[i]) + np.arange(b - a)
            v = pk.seq_nib[k >> 1]
            seq = "".join(SEQ16[x] for x in np.where(k & 1, v & 15, v >> 4))
            qual = (pk.qual[a:b] - 33).astype(np.uint8).tobytes() if pk.has_qual[i] else None
            cig = [(int(w) >> 4, OPS[int(w) & 15]) for w in pk.cigar_rle[pk.cigar_off[i]:pk.cigar_off[i + 1]]]
            reads.append(po.Read(int(pk.read_pos[i]), cig, seq, qual))
            ids.append(_read_id(int(pk.read_pos[i]), cig, seq))
        T = int(cfg.args.max_l) + 1
        tot = [np.zeros((5, 5), np.int64), np.zeros((int(cfg.args.max_n), T, T), np.int64), np.zeros(T, np.int64), np.zeros(T, np.int64)]
        used = set()
        ranges = []
        for r in range(len(pk.range_start)):
            s, e = int(pk.range_start[r]), int(pk.range_end[r])
            chunk = pk.ref_ascii[pk.ref_off[r]:pk.ref_off[r + 1]].tobytes().decode("latin-1")
            ref = " " * s + chunk                  # the oracle reads contig[start : end + 1 + max_n], as the chunk holds
            lst = pk.range_reads[pk.range_reads_off[r]:pk.range_reads_off[r + 1]].tolist()
            assert lst == sorted(lst)
            used.update(lst)
            for acc, m in zip(tot, po.confusion([reads[i] for i in lst], ref, s, e, oracle.get_np_info, oracle.bases_to_int,
                                                int(cfg.args.max_n), int(cfg.args.max_l), int(pk.min_base_q))):
                acc += m
            ranges.append((s, e, sorted(ids[i] for i in lst)))
        assert used == set(range(n)), "a batch holds a read none of its ranges uses"
        self.batches.append({"ranges": ranges, "bases": int(pk.seq_off[-1]), "n_reads": n})
        return tuple(tot)


@pytest.fixture
def stand_in(monkeypatch):
    s = StandIn()
    monkeypatch.setattr(confusion, "_np_engine", lambda: s)
    return s


def _oracle_sum(file_reads, ctgs, ranges):
    T = int(cfg.args.max_l) + 1
    tot = [np.zeros((5, 5), np.int64), np.zeros((int(cfg.args.max_n), T, T), np.int64), np.zeros(T, np.int64), np.zeros(T, np.int64)]
    want = []
    for c, s, e in ranges:
        rs = file_reads.get(c, [])
        for acc, m in zip(tot, po.confusion([r for r, _ in rs], ctgs[c], s, e, oracle.get_np_info, oracle.bases_to_int)):
            acc += m
        kept = sorted(i for r, i in rs if not (r.flag & confusion.SKIP_FLAGS) and r.pos < e and r.end > s)
        if kept:
            want.append((c, s, e, kept))
    return tot, want


def _check_batches(stand_in, want, max_batch_bases):
    """Each range with reads is counted once, with exactly its kept overlapping reads; ranges without reads never go."""
    got = sorted((s, e, ids) for b in stand_in.batches for s, e, ids in b["ranges"])
    assert got == sorted((s, e, ids) for _, s, e, ids in want)
    for b in stand_in.batches:
        assert b["bases"] <= max_batch_bases or len(b["ranges"]) == 1


CASES = [  # (seed, regions, chunk_width, window_bytes, max_batch_bases)
    (1, None, 100000, 16 << 20, 256 << 20),
    (2, None, 97, 3000, 256 << 20),                       # reads carried across many windows
    (3, None, 1000, 600, 256 << 20),                      # windows smaller than one record
    (4, [("b", 200, 1400), ("a", 0, 900), ("a", 500, 2100), ("e", 0, 800), ("a", 2000, 2001)], 300, 2000, 256 << 20),
    (5, None, 700, 5000, 500),                            # max_batch_bases below one range's bases
    (6, [("a", 100, 2400), ("b", 0, 1000)], 450, 0, 4000),  # whole file in one window
]


@pytest.mark.parametrize("seed,regions,chunk_width,window_bytes,max_batch_bases", CASES)
def test_count_bam_matches_oracle(tmp_path, small_cfg, stand_in, monkeypatch, seed, regions, chunk_width, window_bytes, max_batch_bases):
    monkeypatch.setattr(cfg.args, "chunk_width", chunk_width)
    path = str(tmp_path / "s.bam")
    ctgs, _ = _make_bam(path, seed)
    fr = _file_reads(path)
    ranges = confusion.get_ranges(regions if regions is not None else [(c, 0, len(s)) for c, s in ctgs.items()])
    tm = {}
    got = confusion.count_bam(path, ctgs, regions, window_bytes=window_bytes, max_batch_bases=max_batch_bases, timings=tm)
    want, per_range = _oracle_sum(fr, ctgs, ranges)
    for nm, a, b in zip(("subs", "nps", "inss", "dels"), want, got):
        assert a.dtype == b.dtype == np.int64 and np.array_equal(a, b), f"{nm} differs"
    assert int(got[0].sum()) > 0
    _check_batches(stand_in, per_range, max_batch_bases)
    assert tm["batches"] == len(stand_in.batches) and tm["reads"] == sum(b["n_reads"] for b in stand_in.batches)
    assert set(tm) >= {"open", "gather", "pack", "device_wait", "bases"}
    if max_batch_bases < 1000:
        assert any(len(b["ranges"]) == 1 and b["bases"] > max_batch_bases for b in stand_in.batches)


def test_count_bam_fasta_path_and_carry_bound(tmp_path, small_cfg, stand_in, monkeypatch):
    """refs as a FASTA path; the carry never keeps a read that no pending range overlaps."""
    monkeypatch.setattr(cfg.args, "chunk_width", 200)
    path = str(tmp_path / "s.bam")
    ctgs, _ = _make_bam(path, 11)
    fa = tmp_path / "ref.fa"
    fa.write_text("".join(f">{c}\n{s}\n" for c, s in ctgs.items()))
    seen = []
    orig = confusion._Carry.keep

    def keep(self, sel):
        orig(self, sel)
        seen.append((len(self), int(self.qual_off[-1])))
    monkeypatch.setattr(confusion._Carry, "keep", keep)
    got = confusion.count_bam(path, str(fa), None, window_bytes=4000)
    want, _ = _oracle_sum(_file_reads(path), ctgs, confusion.get_ranges([(c, 0, len(s)) for c, s in ctgs.items()]))
    assert all(np.array_equal(a, b) for a, b in zip(want, got))
    # with 200-base ranges and reads of at most ~500 bases, the carry holds a few reads' worth, never the file
    assert seen and max(n for n, _ in seen) < 40 and seen[-1][0] == 0


def test_count_bam_rejects_unsorted_and_bad_ranges(tmp_path, small_cfg, stand_in, monkeypatch):
    path = str(tmp_path / "s.bam")
    ctgs, recs = _make_bam(path, 21, unmapped_tail=0)
    with pytest.raises(ValueError, match="outside the contig"):
        confusion.count_bam(path, ctgs, [("a", 0, len(ctgs["a"]) + 1)])
    # records of contig a after those of contig b, positions sorted within each: unsorted across a window boundary
    swapped = [r for r in recs if r["ref_id"] == 1] + [r for r in recs if r["ref_id"] == 0]
    bad = str(tmp_path / "unsorted.bam")
    bamio.write_bam(bad, "@HD\tVN:1.6\n", [(c, len(s)) for c, s in ctgs.items()], swapped)
    for wb in (2000, 0):
        with pytest.raises(ValueError, match="not coordinate-sorted"):
            confusion.count_bam(bad, ctgs, None, window_bytes=wb)
    saved = {k: getattr(cfg.args, k, None) for k in ("bam", "refs", "regions", "stats_dir", "recalc_cms")}
    try:
        cfg.args.bam, cfg.args.refs, cfg.args.regions = bad, ctgs, None
        cfg.args.stats_dir, cfg.args.recalc_cms = str(tmp_path / "stats"), True
        with pytest.raises(ValueError, match="not coordinate-sorted"):
            confusion.get_confusion_matrices()
        assert not os.path.exists(tmp_path / "stats") or not any(f.endswith(".npy") for f in os.listdir(tmp_path / "stats"))
        # the sorted file goes through the same path and is cached
        cfg.args.bam = path
        out = confusion.get_confusion_matrices()
        assert os.path.exists(tmp_path / "stats" / "subs_cm.npy") and int(out[0].sum()) > 0
    finally:
        for k, v in saved.items():
            setattr(cfg.args, k, v)


def test_gather_without_bases(tmp_path):
    """NativeBam.gather(want_seq=False): qualities and CIGARs, no bases."""
    path = str(tmp_path / "s.bam")
    _make_bam(path, 31)
    bam = bamio.NativeBam(path)
    try:
        sel = np.flatnonzero(bam.has_qual)[:10]
        g = bam.gather(sel, want_seq=False, want_codes=False, want_names=False)
        full = bam.gather(sel)
        assert g["seq_ascii"] is None and g["names"] is None
        n = int(g["seq_off"][-1])
        assert np.array_equal(g["qual_ascii"][:n], full["qual_ascii"][:n])
        assert np.array_equal(g["cigar"][:int(g["cig_off"][-1])], full["cigar"][:int(full["cig_off"][-1])])
    finally:
        bam.close()


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("seed", [41, 42, 43])
def test_gpu_count_bam_equals_batch_path(tmp_path, small_cfg, monkeypatch, seed):
    """count_bam == calc_confusion_matrices_batch(get_ranges(regions), refs, load_alignments(bam)) bit for bit."""
    path = str(tmp_path / "s.bam")
    ctgs, _ = _make_bam(path, seed, n_reads=(120, 80), read_len=600)
    reads = confusion.load_alignments(path)
    La, Lb = len(ctgs["a"]), len(ctgs["b"])
    for chunk_width, regions in ((100000, None), (333, [("b", 100, Lb - 300), ("a", 0, 1500), ("a", 700, La), ("e", 10, 700)])):
        monkeypatch.setattr(cfg.args, "chunk_width", chunk_width)
        rg = regions if regions is not None else [(c, 0, len(s)) for c, s in ctgs.items()]
        want = confusion.calc_confusion_matrices_batch(confusion.get_ranges(rg), ctgs, reads)
        for window_bytes in (64 << 10, 8 << 10, 0):
            for max_batch_bases in (2000, 256 << 20):
                got = confusion.count_bam(path, ctgs, regions, window_bytes=window_bytes, max_batch_bases=max_batch_bases)
                for nm, a, b in zip(("subs", "nps", "inss", "dels"), want, got):
                    assert np.array_equal(a, b), f"{nm} differs (chunk {chunk_width}, window {window_bytes}, batch {max_batch_bases})"
        assert int(want[0].sum()) > 0


def _case_reads(c):
    return [(r[0], [(n, op) for n, op in r[1]], r[2], None if r[3] is None else bytes(ord(ch) - 33 for ch in r[3]), r[4], r[5])
            for r in c["reads"]]


@pytest.mark.gpu
def test_gpu_count_bam_golden(tmp_path, small_cfg, monkeypatch, golden):
    """Every golden window (the compiled reference's counts), written to a BAM file, through count_bam."""
    for c in golden("confusion_kats.json.gz"):
        monkeypatch.setattr(cfg.args, "chunk_width", c["end"] - c["start"])
        # stable: BAM order for equal positions; BAM stores no case (the device upper-cases read bases either way)
        reads = [(r[0], r[1], r[2].upper()) + r[3:] for r in sorted(_case_reads(c), key=lambda r: r[0])]
        path = str(tmp_path / "g.bam")
        bamio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n", [("c", len(c["contig"]))], [_rec(k, 0, r) for k, r in enumerate(reads)])
        got = confusion.count_bam(path, {"c": c["contig"]}, [("c", c["start"], c["end"])], window_bytes=4096)
        nps = np.zeros((6, 101, 101), np.int64)
        for a, b, d, v in c["nps"]:
            nps[a, b, d] = v
        want = (np.array(c["subs"], np.int64), nps, np.array(c["inss"], np.int64), np.array(c["dels"], np.int64))
        for nm, a, b in zip(("subs", "nps", "inss", "dels"), want, got):
            assert np.array_equal(a, b), f"seed {c['seed']}: {nm} differs"


def _nibble_pack(pk, reads, rng):
    """The nibble form of an ASCII PileupPack built from `reads` (AlignedReads order): every read at a random nibble parity."""
    kept = sorted((r for r in reads if not (r[4] & confusion.SKIP_FLAGS)), key=lambda r: r[0])
    lut = np.full(256, 15, np.uint8)
    for i, ch in enumerate(SEQ16):
        lut[ord(ch)] = i
    nib, starts, at = [], [], 0
    for r in kept:
        codes = lut[np.frombuffer(r[2].upper().encode(), np.uint8)]
        par = int(rng.integers(0, 2))
        full = np.concatenate(([0] * par, codes, [0] * ((par + len(codes)) & 1))).astype(np.uint8)
        nib.append((full[0::2] << 4) | full[1::2])
        starts.append(2 * at + par)
        at += len(full) // 2
    has_qual = np.array([r[3] is not None for r in kept], np.int32)
    nb = type("NibPack", (), {})()
    nb.__dict__.update(pk.__dict__)
    nb.seq_ascii = None
    nb.seq_nib = np.concatenate(nib).astype(np.uint8) if nib else np.zeros(0, np.uint8)
    nb.seq_nib_start = np.array(starts, np.int64)
    nb.qual = (pk.qual + 33).astype(np.uint8)     # phred+33; the bytes of reads without qualities are not read
    nb.has_qual = has_qual
    return nb


@pytest.mark.gpu
def test_gpu_nibble_form_equals_ascii_form(small_cfg):
    """Realigner.confusion_batch: the nibble form == the ASCII form on the seeded windows of test_gpu_confusion_fuzz_vs_oracle,
    plus reads with N, IUPAC letters and '=', with and without qualities, and with an empty SEQ."""
    eng = confusion._np_engine()
    for seed in range(40):
        rng = np.random.default_rng(9100 + seed)
        L = int(rng.integers(300, 3000))
        contig = synth.make_reference(L, rng, p_np=0.4)
        if seed % 4 == 1:
            contig = contig[:L // 2] + contig[L // 2:].lower()
        reads = synth.make_aligned_reads(contig, int(rng.integers(1, 60)) if seed % 5 else 250, int(rng.integers(50, 900)), rng)
        start, end = (0, L) if seed % 3 == 0 else sorted(int(x) for x in rng.choice(L + 1, size=2, replace=False))
        cuts = sorted({start, end, *(int(x) for x in rng.integers(start, end + 1, size=int(rng.integers(0, 4))))})
        ranges = [("c", a, b) for a, b in zip(cuts[:-1], cuts[1:])]
        extra = []
        for k in range(6):
            p = int(rng.integers(0, max(1, L - 120)))
            body = contig[p:p + 100]
            s = "".join(ch if rng.random() > 0.08 else str(rng.choice(list("N=RYKMSWBDHV"))) for ch in body)
            qual = None if k % 2 else bytes(rng.integers(3, 41, len(s)).astype(np.uint8))
            extra.append((p, [(len(body), "M")], "" if k == 5 else s, qual if k != 5 else None, 0, 60))
        reads = sorted(reads + extra, key=lambda r: r[0])
        ar = confusion.AlignedReads([r[:5] for r in reads])
        pk = confusion.PileupPack(ranges, {"c": contig}, {"c": ar}, 6)
        want = eng.confusion_batch(pk)
        got = eng.confusion_batch(_nibble_pack(pk, reads, rng))
        for nm, a, b in zip(("subs", "nps", "inss", "dels"), want, got):
            assert np.array_equal(a, b), f"seed {seed}: {nm} differs"


@pytest.mark.gpu
def test_gpu_nibble_form_argument_checks(small_cfg):
    """Nibbles outside seq_nib, a negative nibble offset and a missing has_qual are NPORE_ERR_BAD_ARG, not a fault."""
    from npore_b200._lib import PileupBatch
    eng = confusion._np_engine()
    rs, re_ = np.array([0], np.int64), np.array([8], np.int64)
    ref = np.frombuffer(b"ACGTACGTACGTACGT", np.uint8)
    ref_off = np.array([0, 16], np.int64)
    pos = np.array([0], np.int64)
    seq_off = np.array([0, 8], np.int64)
    cig = np.array([8 << 4], np.uint32)
    cig_off = np.array([0, 1], np.int64)
    lst, lst_off = np.array([0], np.int32), np.array([0, 1], np.int64)
    nib = np.array([0x12, 0x48, 0x12, 0x48], np.uint8)
    qual = np.full(8, 40 + 33, np.uint8)
    hq = np.array([1], np.int32)
    T = 101
    out = [np.zeros(25, np.int64), np.zeros(6 * T * T, np.int64), np.zeros(T, np.int64), np.zeros(T, np.int64)]

    def call(nib_start, nib_bytes, has_qual):
        b = PileupBatch(1, rs.ctypes.data, re_.ctypes.data, ref.ctypes.data, ref_off.ctypes.data, 1, pos.ctypes.data, None,
                        qual.ctypes.data, seq_off.ctypes.data, cig.ctypes.data, cig_off.ctypes.data, lst.ctypes.data, lst_off.ctypes.data, 13,
                        nib.ctypes.data, np.array([nib_start], np.int64).ctypes.data, nib_bytes, has_qual)
        start = np.array([nib_start], np.int64)
        b.seq_nib_start = start.ctypes.data
        return eng._L.npore_confusion_batch(eng._ctx, C.byref(b), *[o.ctypes.data for o in out])

    assert call(0, 4, hq.ctypes.data) == 0 and out[0].reshape(5, 5).trace() == 8
    assert call(1, 4, hq.ctypes.data) == -1          # last nibble past seq_nib
    assert call(0, 3, hq.ctypes.data) == -1
    assert call(-1, 4, hq.ctypes.data) == -1
    assert call(0, 4, None) == -1                    # qualities in the nibble form need has_qual
    assert call(0, 4, hq.ctypes.data) == 0           # the context is still usable
