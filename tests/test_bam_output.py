"""BAM output of bamio.realign_bam (out_format="bam"), layer by layer:
  - the native record encoder (npore_bam_format) against a reference encoder written here from the SAM text and the field
    rules of htslib's SAM -> BAM conversion;
  - the file pipeline with a stand-in engine and a zlib stand-in compressor (CPU);
  - the GPU BGZF compressor (npore_bgzf_compress), member by member against zlib, its size against zlib level 1, and the
    end-to-end output against the SAM path on the device."""
import gzip
import os
import re
import struct
import zlib

import numpy as np
import pytest

from npore_b200 import bamio, cfg, synth

HERE = os.path.dirname(os.path.abspath(__file__))
_SEQ16 = "=ACMGRSVTWYHKDBN"
_NT16 = {c: i for i, c in enumerate(_SEQ16)}
_OPS = "MIDNSHP=XB"
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


# ------------------------------------------------------------------------------------------------ reference encoder
def _reg2bin(beg, end):
    end -= 1
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return off + (beg >> shift)
    return 0


def _hp_tag(v):
    if v < 0:
        typ, fmt = ("c", "<b") if v >= -128 else ("s", "<h") if v >= -32768 else ("i", "<i")
    else:
        typ, fmt = ("C", "<B") if v <= 255 else ("S", "<H") if v <= 65535 else ("I", "<I")
    return b"HP" + typ.encode() + struct.pack(fmt, v)


def ref_record(line, refs):
    """One SAM line of bam.sam_record -> its BAM record (block_size included), with the field encodings htslib chooses."""
    f = line.rstrip("\n").split("\t")
    name, flag, rname, pos1, mapq, cigar, _rnext, _pnext, tlen, seq, qual = f[:11]
    names = [n for n, _ in refs]
    ref_id = names.index(rname) if rname in names else -1
    pos = int(pos1) - 1
    ops = [(int(a), b) for a, b in re.findall(r"(\d+)([MIDNSHP=XB])", cigar)]
    span = sum(n for n, op in ops if op in "MDN=X")
    cig = b"".join(struct.pack("<I", n << 4 | _OPS.index(op)) for n, op in ops)
    codes = [_NT16.get(c.upper(), 15) for c in seq] + [0]
    packed = bytes((codes[i] << 4) | (codes[i + 1] if i + 1 < len(seq) else 0) for i in range(0, len(seq), 2))
    qb = bytes([0xFF] * len(seq)) if qual == "*" else bytes(ord(c) - 33 for c in qual)
    assert f[11].startswith("HP:i:")
    tags = _hp_tag(int(f[11][5:]))
    nm = name.encode() + b"\0"
    body = struct.pack("<iiBBHHHiiii", ref_id, pos, len(nm), int(mapq), _reg2bin(pos, pos + (span or 1)), len(ops), int(flag),
                       len(seq), -1, -1, int(tlen)) + nm + cig + packed + qb + tags
    return struct.pack("<i", len(body)) + body


def ref_bam_stream(sam_text, refs):
    """The uncompressed BAM stream (header + records) of a SAM file written by realign_bam."""
    lines = sam_text.splitlines(keepends=True)
    text = "".join(ln for ln in lines if ln.startswith("@")).encode()
    out = [b"BAM\1", struct.pack("<i", len(text)), text, struct.pack("<i", len(refs))]
    for name, length in refs:
        out.append(struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", length))
    out += [ref_record(ln, refs) for ln in lines if not ln.startswith("@")]
    return b"".join(out)


def members(data):
    """Splits a BGZF file into its members, checking every header and trailer field."""
    out, p = [], 0
    while p < len(data):
        assert data[p:p + 16] == bytes.fromhex("1f8b08040000000000ff060042430200"), p
        bsize = struct.unpack_from("<H", data, p + 16)[0] + 1
        assert bsize <= 65536
        out.append(data[p:p + bsize])
        p += bsize
    assert p == len(data)
    return out


def check_members(data, payload):
    """Every member: header, BSIZE, size, ISIZE, CRC, and raw inflate of its slice; the whole: gzip.decompress."""
    at = 0
    for mb in members(data):
        crc, isize = struct.unpack_from("<II", mb, len(mb) - 8)
        assert 0 < isize <= 65280
        d = zlib.decompressobj(-15)
        got = d.decompress(mb[18:-8]) + d.flush()
        assert d.eof and not d.unused_data
        assert got == payload[at:at + isize] and crc == zlib.crc32(got)
        at += isize
    assert at == len(payload)
    assert gzip.decompress(bytes(data)) == bytes(payload)


# ------------------------------------------------------------------------------------------------ streams
def _read_stream(n_reads, with_quals, seed=7):
    """BAM records of synthetic 10 kb reads (the recipe of the size figures in DESIGN.md section 5)."""
    rng = np.random.default_rng(seed)
    ref, tracts = synth.make_reference_with_tracts(300_000, rng)
    reads = synth.make_reads(ref, n_reads, 10_000, rng, None, tracts=tracts)

    def quals(n):
        m = np.convolve(rng.normal(18, 6, n + 50), np.ones(50) / 50, "valid")[:n]
        return np.clip(m + rng.normal(0, 5, n), 2, 50).astype(np.uint8).tobytes()
    recs = [{"name": r[0], "flag": 0, "ref_id": 0, "pos": r[3], "mapq": 60, "seq": r[7], "qual": quals(len(r[7])) if with_quals else None,
             "cigar": [(int(a), b) for a, b in re.findall(r"(\d+)(\D)", r[5])], "tags": {"HP": r[10]}} for r in reads]
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"npore_bgzf_stream_{os.getpid()}.bam")
    try:
        bamio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n", [("chr1", len(ref))], recs, level=0)
        return gzip.open(path).read()
    finally:
        os.remove(path)


def _zlib1_size(payload):
    total = 0
    for i in range(0, len(payload), 65280):
        c = zlib.compressobj(1, zlib.DEFLATED, -15)
        total += len(c.compress(payload[i:i + 65280]) + c.flush()) + 26
    return total


def _contents(n, kind, rng):
    if kind == "zeros":
        return bytes(n)
    if kind == "random":
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    if kind == "text_quals":
        unit = b"@SQ\tSN:chr1\tLN:248956422\n@PG\tID:realigner\tPN:realigner\n" + bytes(np.clip(rng.normal(20, 6, 300), 2, 50).astype(np.uint8) + 33)
        return (unit * (n // len(unit) + 1))[:n]
    if kind == "far_repeats":            # a random block repeated at distance exactly 32768 and 32769
        blk = rng.integers(0, 256, 32768, dtype=np.uint8).tobytes()
        s = blk + blk + b"x" + blk
        return (s * (n // len(s) + 1))[:n]
    if kind == "fibonacci":              # byte frequencies 1, 1, 2, 3, 5, ...: unlimited Huffman codes would be deeper than 15
        fib, a, b = [], 1, 1
        while len(fib) < 24:
            fib.append(a); a, b = b, a + b
        sym = np.repeat(np.arange(len(fib), dtype=np.uint8), fib)
        return rng.permutation(np.resize(sym, n)).astype(np.uint8).tobytes()
    raise ValueError(kind)


SIZES = [0, 1, 258, 259, 32_768, 32_769, 65_279, 65_280, 65_281, 10 * 65_280 + 17]
KINDS = ["zeros", "random", "text_quals", "far_repeats", "fibonacci"]


@pytest.fixture(scope="module")
def compressor(have_gpu):
    if not have_gpu:
        pytest.skip("needs a CUDA device")
    from npore_b200.engine import BgzfCompressor
    z = BgzfCompressor(0)
    yield z
    z.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_compressor_members_conform(compressor, kind):
    rng = np.random.default_rng(11)
    for n in SIZES:
        payload = _contents(n, kind, rng)
        out = bytes(compressor.compress(payload))
        if n == 0:
            assert out == b""
            continue
        check_members(out, payload)
        if kind == "random":             # incompressible: every member is stored (BTYPE 00, BFINAL 1)
            assert all(mb[18] == 1 for mb in members(out)), n
        if kind in ("zeros", "fibonacci") and n >= 32_769:
            assert len(out) < n // 2, (kind, n)
        if kind == "far_repeats" and n >= 65_279:       # copies 32768 bytes back in the same member are matched, as zlib does
            assert len(out) <= 1.05 * _zlib1_size(payload), (kind, n)


@pytest.mark.gpu
def test_compressor_matches_reach_32768_back(compressor):
    """A random 32 KiB block repeated at distance 32768 compresses to little more than one copy."""
    blk = np.random.default_rng(3).integers(0, 256, 32768, dtype=np.uint8).tobytes()
    out = bytes(compressor.compress(blk + blk[:32000]))
    check_members(out, blk + blk[:32000])
    assert len(out) < 32768 + 3000


@pytest.mark.gpu
@pytest.mark.parametrize("with_quals", [False, True])
def test_compressor_size_is_within_5_percent_of_zlib_level_1(compressor, with_quals):
    payload = _read_stream(200, with_quals)
    out = bytes(compressor.compress(payload))
    check_members(out, payload)
    assert len(out) <= 1.05 * _zlib1_size(payload), (len(out), _zlib1_size(payload), len(payload))


@pytest.mark.gpu
def test_compressor_is_deterministic(compressor):
    payload = _read_stream(40, True, seed=5)
    a = bytes(compressor.compress(payload))
    b = bytes(compressor.compress(payload))
    assert a == b


# ------------------------------------------------------------------------------------------------ fixture BAM, stand-ins
IUPAC = "RYKMSWBDHVN"
HPS = [0, 255, 256, 70_000, -1, -200, 40_000]


@pytest.fixture(scope="module")
def fixture_bam(tmp_path_factory, tables):
    """Two contigs; reads with and without qualities, IUPAC bases, HP values 0 / 255 / 256 / 70000 and negative ones."""
    S, NP = tables
    rng = np.random.default_rng(99)
    cm = synth.call_length_model(NP)
    contigs, recs = [], []
    for ci, (name, length, n_reads) in enumerate((("chrA", 24_000, 50), ("chrB", 15_000, 30))):
        ref, tr = synth.make_reference_with_tracts(length, rng)
        contigs.append((name, ref))
        for k, rd in enumerate(synth.make_reads(ref, n_reads, 1000, rng, cm, tracts=tr)):
            seq = list(rd[7])
            if k % 3 == 0:
                for at in rng.choice(len(seq), 4, replace=False):
                    seq[at] = IUPAC[int(at) % len(IUPAC)]
            recs.append({"name": f"{name}_{rd[0]}", "flag": 0, "ref_id": ci, "pos": rd[3], "mapq": 60, "seq": "".join(seq),
                         "qual": None if k % 4 == 1 else bytes(rng.integers(0, 40, len(seq)).astype(np.uint8)),
                         "cigar": [(int(a), b) for a, b in re.findall(r"(\d+)(\D)", rd[5])], "tags": {"HP": HPS[k % len(HPS)]}})
    path = str(tmp_path_factory.mktemp("bamout") / "in.bam")
    bamio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n", [(n, len(s)) for n, s in contigs], recs)
    return path, dict(contigs), S, NP


class _EchoEngine:
    """Engine stand-in: the "realigned" CIGAR of every record is its input CIGAR; submit number fail_at (1-based) fails."""

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
    """Compressor stand-in for CPU runs: BGZF members from zlib (the product has no CPU compressor)."""

    def compress(self, buf):
        buf = bytes(buf)
        return b"".join(bamio._bgzf_block(buf[i:i + 65280], 1) for i in range(0, len(buf), 65280))


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


def _sam_and_bam(bam, fa, tmp_path, name, **kw):
    tm_s, tm_b = {}, {"trace": []}
    n_s = bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / f"{name}_s"), argv=["t"], timings=tm_s, **kw)
    n_b = bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / f"{name}_b"), argv=["t"], timings=tm_b, out_format="bam", **kw)
    assert n_s == n_b
    sam = open(tmp_path / f"{name}_s.sam").read()
    data = open(tmp_path / f"{name}_b.bam", "rb").read()
    return n_b, sam, data, tm_s, tm_b


def _check_bam_file(path, data, sam, refs, n):
    """The file decompresses to the reference encoding of the SAM-mode file, ends in exactly one EOF block, and both readers
    read it back."""
    assert data.endswith(BGZF_EOF)
    ms = members(data)
    assert [struct.unpack_from("<I", mb, len(mb) - 4)[0] for mb in ms].count(0) == 1
    assert gzip.decompress(data) == ref_bam_stream(sam, refs)
    text, got_refs, recs = bamio.read_bam(path)
    assert got_refs == refs and text == "".join(ln for ln in sam.splitlines(keepends=True) if ln.startswith("@"))
    assert len(list(recs)) == n
    nb = bamio.NativeBam(path)
    assert nb.n == n and nb.refs == refs
    nb.close()


# ------------------------------------------------------------------------------------------------ CPU
def test_record_encoder_matches_the_reference_encoder(fixture_bam):
    bam_path, _, _, _ = fixture_bam
    nb = bamio.NativeBam(bam_path)
    sel = np.arange(nb.n)
    g = nb.gather(sel, want_codes=False, want_cigar=False)
    cig, off = nb.gather_cigar(sel)
    assert set(nb.hp) >= {0, 255, 256, 70_000, -1, -200} and 0 < int(nb.has_qual.sum()) < nb.n
    sam = bytes(bamio.format_sam(nb, sel, g, cig, off)).decode()
    got = bytes(bamio.format_sam(nb, sel, g, cig, off, binary=True))
    assert any(c in IUPAC for ln in sam.splitlines() for c in ln.split("\t")[9])
    assert got == b"".join(ref_record(ln, nb.refs) for ln in sam.splitlines())
    nb.close()


@pytest.mark.parametrize("kw", [{}, {"window_bytes": 20_000, "max_batch_ops": 5_000}, {"window_bytes": 0, "n_inflight": 1}])
def test_bam_pipeline_with_stand_ins(fixture_bam, stand_ins, tmp_path, kw):
    bam, fa, _, _ = fixture_bam
    made = stand_ins()
    n, sam, data, tm_s, tm_b = _sam_and_bam(bam, fa, tmp_path, "x", **kw)
    assert n == 80
    _check_bam_file(str(tmp_path / "x_b.bam"), data, sam, bamio.NativeBam(bam).refs, n)
    assert set(tm_b) == set(tm_s) | {"compress", "trace"} and "compress" not in tm_s
    assert [ev for _, ev in tm_b["trace"]].count("header written") == 1
    assert set(made) == {(None, 0)}


def test_bam_pipeline_regions_and_max_reads(fixture_bam, stand_ins, tmp_path):
    bam, fa, _, _ = fixture_bam
    stand_ins()
    refs = bamio.NativeBam(bam).refs
    for name, kw in (("reg", {"regions": [("chrB", 3_000, 9_000)], "window_bytes": 20_000, "max_batch_ops": 5_000}),
                     ("two", {"regions": [("chrA", 0, 5_000), ("chrB", 0, 4_000)], "max_batch_ops": 5_000}),
                     ("max", {"max_reads": 37, "window_bytes": 20_000, "max_batch_ops": 5_000})):
        n, sam, data, _, _ = _sam_and_bam(bam, fa, tmp_path, name, **kw)
        assert 0 < n < 80
        _check_bam_file(str(tmp_path / f"{name}_b.bam"), data, sam, refs, n)


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
def test_sharded_bam_is_the_single_device_stream(fixture_bam, stand_ins, tmp_path, devices):
    bam, fa, _, _ = fixture_bam
    made = stand_ins()
    bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "one"), argv=["t"], max_batch_ops=5_000, out_format="bam")
    tm = {}
    n = bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "many"), argv=["t"], max_batch_ops=5_000, devices=devices, timings=tm,
                          out_format="bam")
    one, many = open(tmp_path / "one.bam", "rb").read(), open(tmp_path / "many.bam", "rb").read()
    assert n == 80 and gzip.decompress(many) == gzip.decompress(one)
    assert [struct.unpack_from("<I", mb, len(mb) - 4)[0] for mb in members(many)].count(0) == 1 and many.endswith(BGZF_EOF)
    assert {slot for _, slot in made} == set(range(len(devices))) and "compress" in tm
    assert not [f for f in os.listdir(tmp_path) if ".part" in f]


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_bam_mode_failed_batch_raises_and_leaves_no_part_file(fixture_bam, stand_ins, tmp_path, devices):
    bam, fa, _, _ = fixture_bam
    stand_ins(fail_at=3)
    with pytest.raises(RuntimeError, match="stand-in batch failure"):
        bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "out"), argv=["t"], window_bytes=20_000, max_batch_ops=5_000,
                          devices=devices, out_format="bam")
    assert not [f for f in os.listdir(tmp_path) if ".part" in f]


def test_unknown_out_format_is_rejected_before_work(fixture_bam, stand_ins, tmp_path):
    bam, fa, _, _ = fixture_bam
    eng_made = stand_ins()
    with pytest.raises(ValueError, match="out_format"):
        bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "out"), argv=["t"], out_format="cram")
    assert os.listdir(tmp_path) == [] and eng_made == []


def test_compressor_kernels_do_not_spill():
    """-Xptxas -v for sm_100a: the BGZF kernels use no stack frame and spill nothing."""
    import shutil
    import subprocess
    import tempfile
    nvcc = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
    if nvcc is None:
        pytest.skip("nvcc not available")
    src = os.path.join(os.path.dirname(HERE), "npore_b200", "csrc", "bgzf.cuh")
    with tempfile.TemporaryDirectory() as d:
        unit = os.path.join(d, "k.cu")
        with open(unit, "w") as fh:
            fh.write(f'#include "{src}"\n')
        r = subprocess.run([nvcc, "-cubin", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xptxas", "-v",
                            "-o", os.path.join(d, "k.cubin"), unit], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    report = r.stderr.split("Compiling entry function")[1:]
    kernels = [blk for blk in report if "bgzf_" in blk.split("\n")[0]]
    assert len(kernels) == 2, r.stderr
    for blk in kernels:
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in blk, blk


# ------------------------------------------------------------------------------------------------ GPU end to end
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
@pytest.mark.parametrize("kw", [{}, {"window_bytes": 20_000, "max_batch_ops": 20_000}, {"regions": [("chrB", 3_000, 9_000)]},
                                {"max_reads": 45, "window_bytes": 20_000, "max_batch_ops": 20_000}])
def test_bam_output_on_device_matches_sam_output(fixture_bam, device_tables, tmp_path, kw):
    bam, fa, _, _ = fixture_bam
    n, sam, data, _, tm_b = _sam_and_bam(bam, fa, tmp_path, "e2e", **kw)
    assert n > 0 and tm_b["compress"] > 0
    _check_bam_file(str(tmp_path / "e2e_b.bam"), data, sam, bamio.NativeBam(bam).refs, n)


@pytest.mark.gpu
def test_sharded_bam_on_devices_matches_single_device(fixture_bam, device_tables, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two CUDA devices")
    bam, fa, _, _ = fixture_bam
    bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "one"), argv=["t"], max_batch_ops=20_000, out_format="bam")
    n = bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "many"), argv=["t"], max_batch_ops=20_000, devices=[0, 1], out_format="bam")
    assert n == 80
    assert gzip.decompress(open(tmp_path / "many.bam", "rb").read()) == gzip.decompress(open(tmp_path / "one.bam", "rb").read())
    assert not [f for f in os.listdir(tmp_path) if ".part" in f]
