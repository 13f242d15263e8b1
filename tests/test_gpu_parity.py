"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI (libnpore_b200.so via npore_b200.engine),
against (a) the golden vectors produced by the unmodified reference and (b) the CPU oracle on seeded inputs.
Bit-exact for CIGARs / op strings / np_info; DP scores compared bit-for-bit too (stricter than the 1e-5 relative
tolerance north_star allows: the recurrence is fp32 add + compare in the reference's order)."""
import gc
import os

import numpy as np
import pytest

import oracle
from npore_b200 import cig, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine_factory(tables):
    from npore_b200.engine import Realigner
    made = []

    def make(**kw):
        e = Realigner(tables[0], tables[1], **kw)
        made.append(e)
        return e
    yield make
    for e in made:
        e.close()


def _oracle_all(cases, S, NP, **kw):
    out = []
    for rf, sq, cg in cases:
        ir, iq = oracle.bases_to_int(rf), oracle.bases_to_int(sq)
        o, sc, st = oracle.align(ir, iq, cg, S, NP, return_scores=True, **kw)
        out.append((o, sc, st, oracle.collapse_cigar(oracle.standardize(o, ir, iq))))
    return out


def _check(eng, cases, want):
    refs = [oracle.bases_to_int(c[0]) for c in cases]
    seqs = [oracle.bases_to_int(c[1]) for c in cases]
    cigs = [c[2] for c in cases]
    outs, scores, status = eng.align_many(refs, seqs, cigs)
    std, _, _ = eng.align_many(refs, seqs, cigs, standardize=True, collapse=True)
    for k, (o, sc, st, sd) in enumerate(want):
        assert outs[k] == o, f"case {k}: op string differs"
        assert status[k] == st
        assert np.array_equal(scores[k], np.asarray(sc, dtype=np.float32)), f"case {k}: chunk scores differ"
        assert std[k] == sd, f"case {k}: standardised CIGAR differs"


def test_fuzz_golden_reference_outputs(tables, golden, engine_factory):
    """400 seeded cases; expected values come from the compiled reference itself (tests/golden/fuzz.json.gz)."""
    groups = {}
    for c in golden("fuzz.json.gz"):
        groups.setdefault((c["r"], c["max_b_rows"]), []).append(c)
    for (r, mb), cases in sorted(groups.items()):
        eng = engine_factory(max_b_rows=mb, r=r)
        want = [(c["out"], c["scores"], 0, c["std"]) for c in cases]
        _check(eng, [(c["ref"], c["seq"], c["cigar"]) for c in cases], want)


@pytest.mark.parametrize("team", ["1", "2", "4"])
def test_one_warp_and_team_forms_of_the_forward_kernel(tables, golden, monkeypatch, team):
    """forward_kernel<CPL, T>: one chunk per warp (T = 1) and a two-warp team per chunk (T = 2: band split across the warps, team
    ring, mailbox, named barrier) forced through NPORE_TEAM -- both must reproduce the reference's outputs (CIGARs, chunk scores,
    standardised CIGARs) on the golden fuzz vectors and on multi-kb reads at r = 30 / 60 / 100."""
    from npore_b200.engine import Realigner
    monkeypatch.setenv("NPORE_TEAM", team)
    S, NP = tables
    groups = {}
    for c in golden("fuzz.json.gz"):
        groups.setdefault((c["r"], c["max_b_rows"]), []).append(c)
    for (r, mb), cases in sorted(groups.items()):
        eng = Realigner(S, NP, max_b_rows=mb, r=r)
        _check(eng, [(c["ref"], c["seq"], c["cigar"]) for c in cases], [(c["out"], c["scores"], 0, c["std"]) for c in cases])
        eng.close()
    rng = np.random.default_rng(90 + int(team))
    cm = synth.call_length_model(NP)
    ref, tr = synth.make_reference_with_tracts(60_000, rng)
    cases = [(rd[9], rd[7], cig.expand_cigar(rd[5])) for rd in synth.make_reads(ref, 6, 7000, rng, cm, tracts=tr)]
    for r in (30, 60, 100):
        eng = Realigner(S, NP, r=r, max_b_rows=3000)
        _check(eng, cases, _oracle_all(cases, S, NP, r=r, max_b_rows=3000))
        eng.close()


def test_time_sliced_teams_hand_chunks_back_and_resume(tables, monkeypatch):
    """More chunks than resident teams, short slices (NPORE_RR_SLICE=64): a team of two or four warps saves its registers, team
    ring and mailbox to HBM at a slice boundary, another team resumes the chunk -- outputs stay the reference's."""
    from npore_b200.engine import Realigner
    monkeypatch.setenv("NPORE_RR_SLICE", "64")
    S, NP = tables
    rng = np.random.default_rng(97)
    cm = synth.call_length_model(NP)
    ref, tr = synth.make_reference_with_tracts(120_000, rng)
    cases = [(rd[9], rd[7], cig.expand_cigar(rd[5])) for rd in synth.make_reads(ref, 100, 4000, rng, cm, tracts=tr)]
    want = {}
    for team, r, mb in (("2", 30, 100), ("2", 60, 200), ("2", 100, 300), ("4", 100, 300)):      # <1,2>, <2,2>, <4,2>, <2,4>
        monkeypatch.setenv("NPORE_TEAM", team)
        if (r, mb) not in want:
            want[(r, mb)] = _oracle_all(cases, S, NP, r=r, max_b_rows=mb)
        eng = Realigner(S, NP, r=r, max_b_rows=mb)
        _check(eng, cases, want[(r, mb)])
        eng.close()


def test_golden_sam_through_realign_reads(tables, golden, tmp_path):
    """bam.realign_reads on test/data/reads.sam + ref.fasta reproduces test/data/npore_realigned.sam, every field."""
    from npore_b200 import bam, cfg
    g = golden("golden_sam.json")
    cfg.args.sub_scores, cfg.args.np_scores = tables
    cfg.args.max_n, cfg.args.max_l = 6, 100
    cfg.args.out_prefix = str(tmp_path / "realigned")
    lines = bam.realign_reads([tuple(r) for r in g["reads"]])
    assert lines == g["expected_sam"]
    assert open(cfg.args.out_prefix + ".sam").read().splitlines() == g["expected_sam"]
    bam.realign_read(tuple(g["reads"][3]))                                   # per-item entry appends one more line
    assert open(cfg.args.out_prefix + ".sam").read().splitlines()[-1] == g["expected_sam"][3]


def test_align_drop_in_signature(tables, golden):
    """aln.align with the reference's positional/keyword signature (test/align.py:59-60)."""
    from npore_b200 import aln, cfg
    S, NP = tables
    cfg.args.max_n, cfg.args.max_l = 6, 100
    for k in golden("align_kats.json"):
        ir, iq = cig.bases_to_int(k["ref"]), cig.bases_to_int(k["seq"])
        ex = cig.expand_cigar(k["cigar"])
        assert aln.align(ir, iq, ex, S, NP, verbose=True, max_b_rows=20, r=10) == k["small"]["out"]
        assert aln.align(ir, iq, ex, S, NP) == k["default"]["out"]
    outs, scores = aln.align_batch([cig.bases_to_int(k["ref"]) for k in golden("align_kats.json")],
                                   [cig.bases_to_int(k["seq"]) for k in golden("align_kats.json")],
                                   [k["cigar"] for k in golden("align_kats.json")], S, NP, return_scores=True)
    for k, o, sc in zip(golden("align_kats.json"), outs, scores):
        assert o == k["default"]["out"]
        assert np.array_equal(sc, np.array(k["default"]["scores"], dtype=np.float32))


def test_np_info_on_device(tables, golden, engine_factory):
    """aln.pyx:179-251 incl. the docstring example, the >max_l clamp quirk (105 x A) and N bases."""
    eng = engine_factory()
    for k in golden("np_info_kats.json"):
        info = eng.get_np_info(oracle.bases_to_int(k["seq"]))
        assert info[:, 0, :].T.tolist() == k["L"]
        assert info[:, 1, :].T.tolist() == k["L_IDX"]
    rng = np.random.default_rng(3)
    for _ in range(40):
        s = synth.make_reference(int(rng.integers(1, 3000)), rng, float(rng.choice([0.2, 0.6, 0.95])), str(rng.choice(["ACGT", "AC", "ACGTN"])))
        if rng.random() < 0.3:
            k = int(rng.integers(0, len(s)))
            s = s[:k] + "G" * int(rng.integers(101, 140)) + s[k:]
        a = oracle.bases_to_int(s)
        assert np.array_equal(eng.get_np_info(a), oracle.get_np_info(a))


def test_realign_haps(tables, golden):
    """bam.pyx:93-123 on the haplotypes of test/test_std_vcf.vcf (SURVEY.md Appendix C.3)."""
    from npore_b200 import bam, cfg
    cfg.args.sub_scores, cfg.args.np_scores = tables
    ks = golden("std_vcf_kats.json")
    res = bam.realign_haps([(k["contig"], k["hap"], k["seq"], k["ref"], cig.expand_cigar(k["cigar"])) for k in ks])
    for k, r in zip(ks, res):
        assert r == (k["contig"], k["hap"], k["seq"], k["ref"], k["out"])
    assert bam.realign_hap((ks[1]["contig"], ks[1]["hap"], ks[1]["seq"], ks[1]["ref"], cig.expand_cigar(ks[1]["cigar"])))[4] == ks[1]["out"]


@pytest.mark.parametrize("r,mb", [(3, 12), (10, 37), (16, 50), (30, 200), (31, 64), (60, 300), (100, 500), (127, 20000)])
def test_live_fuzz_vs_oracle_all_band_widths(tables, engine_factory, r, mb):
    """Fresh seeded cases per band width (covers every cells-per-lane template: W<=32, <=64, <=128, <=256)."""
    S, NP = tables
    cm = synth.call_length_model(NP)
    rng = np.random.default_rng(1000 + r)
    cases = []
    for _ in range(60):
        rf, sq, cg, _, _ = synth.fuzz_case(rng, cm)
        cases.append((rf, sq, cg))
    cases += [("", "", ""), ("A", "", "D"), ("", "C", "I"), ("ACGT", "ACGT", "MMMM")]     # empty / one-sided items
    _check(engine_factory(max_b_rows=mb, r=r), cases, _oracle_all(cases, S, NP, max_b_rows=mb, r=r))


@pytest.mark.parametrize("max_n", [0, 1, 3])
def test_reduced_max_n(tables, engine_factory, max_n):
    """cfg.args.max_n < 6 (max_n = 0 is the affine-only mode of SURVEY.md 8(c))."""
    S, NP = tables
    cm = synth.call_length_model(NP)
    rng = np.random.default_rng(77 + max_n)
    cases = [synth.fuzz_case(rng, cm)[:3] for _ in range(40)]
    _check(engine_factory(max_b_rows=150, r=10, max_n=max_n), cases, _oracle_all(cases, S, NP, max_b_rows=150, r=10, max_n=max_n))


def test_production_scale_reads_vs_oracle(tables, engine_factory):
    """48 ONT-like 10 kb reads at align()'s defaults (r=30, max_b_rows=20000), incl. reads that need a second chunk."""
    S, NP = tables
    rng = np.random.default_rng(20260101)
    cm = synth.call_length_model(NP)
    ref, tr = synth.make_reference_with_tracts(200_000, rng)
    reads = synth.make_reads(ref, 40, 10_000, rng, cm, tracts=tr) + synth.make_reads(ref, 8, 10_300, rng, cm, tracts=tr)
    cases = [(r[9], r[7], cig.expand_cigar(r[5])) for r in reads]
    want = _oracle_all(cases, S, NP)
    assert max(len(w[1]) for w in want) == 2                                   # some reads are cut into two chunks
    _check(engine_factory(), cases, want)


def test_long_indel_runs(tables, engine_factory):
    """INS/DEL runs far longer than the run field of the traceback record (their length is not stored: the
    traceback counts the 'extended' bits of the records it walks)."""
    S, NP = tables
    rng = np.random.default_rng(4)
    core = synth.make_reference(600, rng, 0.3)
    ins = "".join(rng.choice(list("ACGT"), size=9000))
    cases = [(core, core[:300] + ins + core[300:], "=" * 300 + "I" * 9000 + "=" * 300),
             (core[:300] + ins + core[300:], core, "=" * 300 + "D" * 9000 + "=" * 300)]
    _check(engine_factory(), cases, _oracle_all(cases, S, NP))


def _long_npolymer_cases():
    """(ref, seq, expanded CIGAR) items whose realignment has LEN / SHR runs of 2,047 ops or more, and one ordinary item."""
    rng = np.random.default_rng(8)
    a = synth.make_reference(300, rng, 0.0, "CGT"); b = synth.make_reference(300, rng, 0.0, "CGT")
    cases = []
    for unit, copies, extra in (("A", 12, 3000), ("AC", 9, 1200), ("A", 20, 2047), ("ACG", 8, 900)):
        tract = unit * copies
        ref = a + tract + b
        # insertion of `extra` more copies right after the tract (LEN), and the mirror image (SHR: the read lacks them)
        cases.append((ref, a + tract + unit * extra + b, "=" * (len(a) + len(tract)) + "I" * (len(unit) * extra) + "=" * len(b)))
        cases.append((a + tract + unit * extra + b, ref, "=" * (len(a) + len(tract)) + "D" * (len(unit) * extra) + "=" * len(b)))
    cases.append((a + b, a + b, "=" * 600))                       # an ordinary item in the same batch
    return cases


def test_npolymer_runs_beyond_the_record_field(tables, engine_factory):
    """LEN / SHR runs of thousands of ops (whole copies of an adjacent tract's unit inserted / deleted): the 11-bit RUN field of
    the traceback record saturates at 2047, the batch is transparently redone with the WIDE kernels (overflow list), and the
    result is the reference's -- status 0, no partial CIGAR (round 1 reported status 8 here)."""
    S, NP = tables
    cases = _long_npolymer_cases()
    want = _oracle_all(cases, S, NP)
    long_runs = [w[0] for w in want if "I" * 2047 in w[0] or "D" * 2047 in w[0]]
    assert len(long_runs) >= 4
    _check(engine_factory(), cases, want)
    small = engine_factory(max_b_rows=1500)                       # several chunks per item: runs cannot span a chunk border
    _check(small, cases, _oracle_all(cases, S, NP, max_b_rows=1500))


def _nib_pack(seqs):
    """Reads in BAM's 4-bit packing (A=1 C=2 G=4 T=8 N=15), each from the high nibble of a byte: (bytes, nibble starts)."""
    code = np.zeros(256, np.uint8)
    code[np.frombuffer(b"ACGTN", np.uint8)] = [1, 2, 4, 8, 15]
    parts, starts, at = [], [], 0
    for s in seqs:
        v = code[np.frombuffer(s.encode(), np.uint8)]
        v = np.append(v, np.zeros(len(v) & 1, np.uint8))
        parts.append((v[0::2] << 4) | v[1::2])
        starts.append(2 * at)
        at += len(v) // 2
    return np.concatenate(parts), np.array(starts, np.int64)


def test_closed_context_returns_its_device_memory(tables):
    """A closed context frees every buffer it grew: the run scratch and outputs of packed reads with run-length and standardised
    outputs, the WIDE pass and its overflow list, the np-info and confusion staging.  The device's free memory after the third
    create / use / close round equals that after the first, which absorbs the driver's one-time allocations (module loads).
    What this cannot see: the pinned host staging (host memory), and small buffers (counters, run-queue control) whose leak
    stays inside memory the driver had already reserved; the scratch, output and staging buffers are large enough to show."""
    import torch
    from npore_b200 import confusion
    from npore_b200.engine import NPORE_OUT_RLE, NPORE_OUT_STANDARDIZE, PackedBatch, Realigner, cigars_to_rle_batch
    S, NP = tables
    rng = np.random.default_rng(31)
    ref, tr = synth.make_reference_with_tracts(40_000, rng)
    reads = synth.make_reads(ref, 24, 3000, rng, synth.call_length_model(NP), tracts=tr)
    nib, nib_start = _nib_pack([r[7] for r in reads])
    words, off = cigars_to_rle_batch([r[5] for r in reads])
    packed = PackedBatch.from_flat_shared_nib(cig.bases_to_int(ref), np.array([r[3] for r in reads], np.int64),
                                              np.array([r[6] - r[3] for r in reads], np.int32), nib, nib_start,
                                              np.array([len(r[7]) for r in reads], np.int32), words, off)
    long_cases = _long_npolymer_cases()
    contig = synth.make_reference(3000, rng, p_np=0.4)
    aligned = confusion.AlignedReads([r[:5] for r in synth.make_aligned_reads(contig, 40, 600, rng)])
    pileup = confusion.PileupPack([("c", 0, 1500), ("c", 1500, 3000)], {"c": contig}, {"c": aligned}, 6)
    gc.collect()                                                  # contexts that earlier tests dropped are closed before counting
    torch.cuda.init()
    free = []
    for _ in range(3):
        eng = Realigner(S, NP)
        res = eng.align_packed(packed, NPORE_OUT_STANDARDIZE | NPORE_OUT_RLE)
        assert not res.status[:packed.n].any() and res.rle_off[packed.n] > 0
        outs, _, status = eng.align_many([oracle.bases_to_int(c[0]) for c in long_cases], [oracle.bases_to_int(c[1]) for c in long_cases],
                                         [c[2] for c in long_cases])
        # runs past the 2,047 ops of the record field with status 0 come only from the WIDE pass and its overflow list
        assert not status.any() and any("I" * 2048 in o or "D" * 2048 in o for o in outs)
        info = eng.get_np_info_batch([cig.bases_to_int(ref[:5000]), cig.bases_to_int(ref[5000:9000])])
        assert [len(x) for x in info] == [5000, 4000]
        subs, _, _, _ = eng.confusion_batch(pileup)
        assert subs.sum() > 0
        eng.close()
        free.append(torch.cuda.mem_get_info()[0])
    assert free[2] == free[0], f"free device memory after each round: {free}"


def test_bad_cigar_is_reported_not_ub(tables, engine_factory):
    eng = engine_factory()
    ok = ("ACGTACGT", "ACGTACGT", "8=")
    bad = ("ACGTACGT", "ACGTACGT", "7=")                                       # consumes 7 of 8 bases
    refs = [oracle.bases_to_int(c[0]) for c in (ok, bad, ok)]
    seqs = [oracle.bases_to_int(c[1]) for c in (ok, bad, ok)]
    outs, _, status = eng.align_many(refs, seqs, [ok[2], bad[2], ok[2]])
    assert status.tolist() == [0, 16, 0] and outs == ["=" * 8, "", "=" * 8]


def test_sub_batching_and_shared_reference_are_invisible(tables):
    """Same results when the scratch budget forces many sub-batches, and when reads index one shared reference."""
    from npore_b200.engine import PackedBatch, Realigner, cigar_to_rle, NPORE_OUT_STANDARDIZE, NPORE_OUT_RLE
    S, NP = tables
    rng = np.random.default_rng(11)
    cm = synth.call_length_model(NP)
    ref, tr = synth.make_reference_with_tracts(60_000, rng)
    reads = synth.make_reads(ref, 64, 3000, rng, cm, tracts=tr)
    refs = [cig.bases_to_int(r[9]) for r in reads]; seqs = [cig.bases_to_int(r[7]) for r in reads]
    rles = [cigar_to_rle(r[5]) for r in reads]
    flags = NPORE_OUT_STANDARDIZE | NPORE_OUT_RLE
    e1 = Realigner(S, NP, max_b_rows=1000)
    a = e1.align_packed(PackedBatch(refs, seqs, rles, pinned=False), flags)
    assert e1.stats()["n_sub_batches"] == 1
    os.environ["NPORE_SCRATCH_MB"] = "4"
    try:
        e2 = Realigner(S, NP, max_b_rows=1000)
    finally:
        del os.environ["NPORE_SCRATCH_MB"]
    shared = PackedBatch(None, seqs, rles, shared_ref=cig.bases_to_int(ref), ref_ranges=[(r[3], r[6]) for r in reads], pinned=True)
    b = e2.align_packed(shared, flags)
    assert e2.stats()["n_sub_batches"] > 3
    for k in range(len(reads)):
        assert a.ops_str(k) == b.ops_str(k) and a.cigar_text(k) == b.cigar_text(k)
        assert np.array_equal(a.scores(k), b.scores(k))
    e1.close(); e2.close()


def test_full_c2_properties(tables):
    """BASELINE.json configs[1] at full size (3,000 x 10 kb): size-independent properties of every output --
    the CIGAR consumes exactly the read and the reference span, '='/'X' agree with the bases, the run is
    deterministic, and a 64-read sample is bit-exact against the oracle."""
    import bench
    from npore_b200.engine import Realigner
    S, NP = tables
    _, reads = bench.make_workload(20260101, 1_000_000, 3000, 10_000, NP)
    packed = bench.pack_reads(reads, pinned=True)
    eng = Realigner(S, NP)
    res = eng.align_packed(packed, 0)
    assert not res.status[:packed.n].any()
    first = res.ops.copy()
    chk = 0
    for k, rd in enumerate(reads):
        ops = res.ops[res.ops_off[k]:res.ops_off[k + 1]]
        consumes_ref = int(np.count_nonzero(ops != ord("I"))); consumes_seq = int(np.count_nonzero(ops != ord("D")))
        assert consumes_ref == len(rd[9]) and consumes_seq == len(rd[7])
        rpos = np.cumsum(ops != ord("I")) - 1; spos = np.cumsum(ops != ord("D")) - 1
        diag = (ops == ord("=")) | (ops == ord("X"))
        rb = np.frombuffer(rd[9].encode(), np.uint8)[rpos[diag]]; sb = np.frombuffer(rd[7].encode(), np.uint8)[spos[diag]]
        assert np.array_equal(rb == sb, ops[diag] == ord("="))
        chk ^= hash(ops.tobytes())
    res2 = eng.align_packed(packed, 0)
    assert np.array_equal(first[:res.ops_off[packed.n]], res2.ops[:res2.ops_off[packed.n]])          # deterministic
    for k in range(0, 3000, 47):
        rd = reads[k]
        want, wsc, _ = oracle.align(oracle.bases_to_int(rd[9]), oracle.bases_to_int(rd[7]), cig.expand_cigar(rd[5]), S, NP, return_scores=True)
        assert res.ops_str(k) == want and np.array_equal(res.scores(k), wsc)
    eng.close()


def test_c3_shard_scale_properties(tables, monkeypatch):
    """BASELINE.json configs[2] is 192,000 reads over 8 GPUs; this is half of one GPU's share (12,000 x 10 kb, 14.6 G cell
    updates, ~30 GB of traceback rows) under a scratch budget that forces several sub-batches: every CIGAR consumes
    exactly its read and reference span, the result does not depend on how the reads are batched, and a sample is
    bit-exact (op strings and chunk scores) against the oracle."""
    import bench
    from npore_b200.engine import PackedBatch, Realigner
    S, NP = tables
    _, reads = bench.make_workload(20260103, 4_000_000, 12_000, 10_000, NP)
    packed = bench.pack_reads(reads, pinned=False)
    monkeypatch.setenv("NPORE_SCRATCH_MB", "12000")
    eng = Realigner(S, NP)
    res = eng.align_packed(packed, 0, eng.new_result(packed, 0, pinned=False))
    st = eng.stats()
    assert st["n_sub_batches"] >= 3 and st["n_items"] == 12_000 and not res.status[:packed.n].any()
    n = packed.n
    off = res.ops_off[:n + 1]
    ops = res.ops[:off[n]]
    not_i = np.concatenate(([0], np.cumsum(ops != ord("I"))))
    not_d = np.concatenate(([0], np.cumsum(ops != ord("D"))))
    assert np.array_equal(not_i[off[1:]] - not_i[off[:-1]], packed.ref_len) and np.array_equal(not_d[off[1:]] - not_d[off[:-1]], packed.seq_len)
    assert set(np.unique(ops).tolist()) <= {ord(c) for c in "=XID"}
    # batching invariance: the second half alone gives the same op strings and scores
    half = n // 2
    sub = PackedBatch.from_strings([r[9] for r in reads[half:]], [r[7] for r in reads[half:]], [r[5] for r in reads[half:]])
    res2 = eng.align_packed(sub, 0, eng.new_result(sub, 0, pinned=False))
    assert np.array_equal(res2.ops[:res2.ops_off[sub.n]], ops[off[half]:])
    assert np.array_equal(res2.chunk_scores[:res2.score_off[sub.n]], res.chunk_scores[res.score_off[half]:res.score_off[n]])
    for k in range(5, n, 397):
        rd = reads[k]
        want, wsc, _ = oracle.align(oracle.bases_to_int(rd[9]), oracle.bases_to_int(rd[7]), cig.expand_cigar(rd[5]), S, NP, return_scores=True)
        assert res.ops_str(k) == want and np.array_equal(res.scores(k), wsc)
    eng.close()


@pytest.mark.parametrize("r", [10, 30, 60, 100])
def test_c4_long_reads_band_and_window_sweep(tables, engine_factory, r):
    """BASELINE.json configs[3]: 50-100 kb reads, band radius x max_b_rows sweep (many chunks per read)."""
    S, NP = tables
    rng = np.random.default_rng(400 + r)
    cm = synth.call_length_model(NP)
    ref, tr = synth.make_reference_with_tracts(160_000, rng)
    reads = synth.make_reads(ref, 1, 55_000, rng, cm, tracts=tr) + synth.make_reads(ref, 1, 90_000, rng, cm, tracts=tr)
    cases = [(rd[9], rd[7], cig.expand_cigar(rd[5])) for rd in reads]
    for mb in (5000, 20000, 50000):
        want = _oracle_all(cases, S, NP, max_b_rows=mb, r=r)
        assert len(want[1][1]) == -(-(len(cases[1][0]) + len(cases[1][1])) // (mb - 1))      # chunk count (aln.pyx:344-358)
        _check(engine_factory(max_b_rows=mb, r=r), cases, want)


def test_c5_whole_contig_haplotypes(tables, golden):
    """BASELINE.json configs[4]: haplotypes carrying indels inside n-polymer tracts, one align() item per
    haplotype of a whole contig (dozens of chunks), through bam.realign_haps (bam.pyx:93-123)."""
    from npore_b200 import bam, cfg
    S, NP = tables
    cfg.args.sub_scores, cfg.args.np_scores = S, NP
    cfg.args.max_n, cfg.args.max_l = 6, 100
    rng = np.random.default_rng(55)
    cm = synth.call_length_model(NP)
    haps = []
    for ctg, length in (("chrA", 300_000), ("chrB", 120_000)):
        ref, tr = synth.make_reference_with_tracts(length, rng)
        for hap in (1, 2):
            keep = tr[rng.random(len(tr)) < 0.5]                      # variants = unit-multiple indels at tract ends only
            seq, cg = synth.make_read(ref, rng, cm, p_ins=0.0, p_sub=0.0005, p_del=0.0, tracts=keep)
            haps.append((ctg, hap, seq, ref, cg))
    got = bam.realign_haps(haps)
    for h, g in zip(haps, got):
        ir, iq = oracle.bases_to_int(h[3]), oracle.bases_to_int(h[2])
        want = oracle.standardize(oracle.align(ir, iq, h[4], S, NP), ir, iq)
        assert g[:4] == h[:4] and g[4] == want


@pytest.mark.parametrize("long_min", [1, 64])
def test_long_item_standardisation_path(tables, monkeypatch, long_min):
    """Items with many run-length groups (haplotypes) are standardised by the segment-parallel kernel; NPORE_STD_LONG_MIN
    forces that path onto ordinary reads and mid-sized haplotypes: same CIGARs as the oracle, expanded and run-length,
    incl. reads whose INDELs sit densely inside homopolymers (shifts chained through short M groups)."""
    from npore_b200.engine import Realigner
    monkeypatch.setenv("NPORE_STD_LONG_MIN", str(long_min))
    S, NP = tables
    rng = np.random.default_rng(600 + long_min)
    cm = synth.call_length_model(NP)
    ref, tr = synth.make_reference_with_tracts(260_000, rng)
    reads = synth.make_reads(ref, 12, 8000, rng, cm, tracts=tr)
    cases = [(rd[9], rd[7], cig.expand_cigar(rd[5])) for rd in reads]
    keep = tr[rng.random(len(tr)) < 0.6]
    seq, cg = synth.make_read(ref, rng, cm, p_ins=0.0, p_sub=0.0005, p_del=0.0, tracts=keep)
    cases.append((ref, seq, cg))
    # dense INDELs in a low-complexity stretch: 1-2 base M groups between runs
    poly = "A" * 40 + "C" + "A" * 30 + "GT" * 25 + "A" * 50
    noisy, _ = synth.make_read(poly * 6, rng, None, p_ins=0.08, p_sub=0.0, p_del=0.08)
    cases.append((poly * 6, noisy, _))
    cases.append(("", "", ""))
    eng = Realigner(S, NP)
    refs = [oracle.bases_to_int(c[0]) for c in cases]; seqs = [oracle.bases_to_int(c[1]) for c in cases]
    exp, _, _ = eng.align_many(refs, seqs, [c[2] for c in cases], standardize=True)
    col, _, _ = eng.align_many(refs, seqs, [c[2] for c in cases], standardize=True, collapse=True)
    wants = []
    for k, c in enumerate(cases):
        aligned = oracle.align(refs[k], seqs[k], c[2], S, NP)
        want = oracle.standardize(aligned, refs[k], seqs[k])
        wants.append((aligned, want))
        assert exp[k] == want and col[k] == oracle.collapse_cigar(want), f"case {k}"
    # the split between the two kernels is decided on the group count BEFORE standardisation (the sweeps change it): items
    # whose count crosses the threshold during the sweeps must be standardised exactly once
    crossed = 0
    for k, (aligned, want) in enumerate(wants):
        ngroups = lambda ops: sum(1 for a, b in zip(ops, ops[1:]) if a != b) + (1 if ops else 0)   # noqa: E731
        m0, m1 = ngroups(aligned.replace("=", "M").replace("X", "M")), ngroups(want)
        if m1 > m0 > 0:
            crossed += 1
            monkeypatch.setenv("NPORE_STD_LONG_MIN", str(m0 + 1))
            one, _, _ = eng.align_many([refs[k]], [seqs[k]], [cases[k][2]], standardize=True, collapse=True)
            assert one[0] == oracle.collapse_cigar(want), f"case {k} at threshold {m0 + 1}"
    assert crossed > 0 or long_min != 1
    eng.close()


def test_len_on_last_copies_of_a_read_tract(tables, golden, engine_factory):
    """aln.pyx:606-607 compares seq[i-n .. i) with ref[j .. j+n).  On the last copies of a read tract (inserted units
    followed by a different base) the unit that FOLLOWS row i is not that unit; a kernel that compares the wrong 6-mer
    loses LEN candidates there (found by tools/gpu_fuzz_live.py; 1 case in 3,700).  Expected values: compiled reference."""
    groups = {}
    for c in golden("len_tail_kats.json"):
        groups.setdefault((c["r"], c["max_n"]), []).append(c)
    for (r, max_n), cases in sorted(groups.items()):
        eng = engine_factory(r=r, max_n=max_n)
        outs, scores, status = eng.align_many([oracle.bases_to_int(c["ref"]) for c in cases], [oracle.bases_to_int(c["seq"]) for c in cases],
                                              [c["cigar"] for c in cases])
        for k, c in enumerate(cases):
            assert outs[k] == c["out"] and status[k] == 0, f"r={r} max_n={max_n} case {k}"
            assert np.array_equal(scores[k], np.array(c["scores"], dtype=np.float32)), f"r={r} max_n={max_n} case {k}: score"


def test_pipelined_realigner_matches_single_context(tables):
    """Several batches in flight on independent contexts / streams / host threads: same results as one context, whatever
    the completion order."""
    from npore_b200.engine import NPORE_OUT_RLE, NPORE_OUT_STANDARDIZE, PackedBatch, PipelinedRealigner, Realigner
    S, NP = tables
    rng = np.random.default_rng(77)
    cm = synth.call_length_model(NP)
    ref, tr = synth.make_reference_with_tracts(120_000, rng)
    batches = []
    for n, length in ((40, 3000), (3, 30_000), (25, 5000), (1, 200), (60, 1500), (8, 9000)):
        reads = synth.make_reads(ref, n, length, rng, cm, tracts=tr)
        batches.append(PackedBatch.from_strings([r[9] for r in reads], [r[7] for r in reads], [r[5] for r in reads]))
    flags = NPORE_OUT_STANDARDIZE | NPORE_OUT_RLE
    one = Realigner(S, NP)
    want = []
    for b in batches:
        r = one.align_packed(b, flags, one.new_result(b, flags, pinned=False))
        want.append((r.ops[:r.ops_off[b.n]].copy(), r.rle[:r.rle_off[b.n]].copy(), r.chunk_scores[:r.score_off[b.n]].copy()))
    one.close()
    pipe = PipelinedRealigner(S, NP, n_inflight=3)
    futs = [pipe.submit(b, flags) for b in batches] + [pipe.submit(b, flags) for b in batches[::-1]]
    got = [f.result()[0] for f in futs]
    for (ops, rle, sc), r, b in zip(want + want[::-1], got, batches + batches[::-1]):
        assert np.array_equal(r.ops[:r.ops_off[b.n]], ops) and np.array_equal(r.rle[:r.rle_off[b.n]], rle)
        assert np.array_equal(r.chunk_scores[:r.score_off[b.n]], sc) and not r.status[:b.n].any()
    pipe.close()


def test_realign_reads_streams_in_batches(tables, tmp_path):
    """The batch scheduler cuts a lazy read stream into several GPU batches; records stay in input order."""
    from npore_b200 import bam, cfg
    S, NP = tables
    cfg.args.sub_scores, cfg.args.np_scores = S, NP
    cfg.args.out_prefix = str(tmp_path / "o")
    rng = np.random.default_rng(8)
    cm = synth.call_length_model(NP)
    ref, tr = synth.make_reference_with_tracts(40_000, rng)
    reads = synth.make_reads(ref, 40, 2000, rng, cm, tracts=tr)
    lines = bam.realign_reads(iter(reads), max_batch_ops=30_000)               # ~7 reads per batch
    assert [l.split("\t")[0] for l in lines] == [r[0] for r in reads]
    for rd, line in zip(reads, lines):
        assert line.split("\t")[5] == oracle.realign_cigar(rd[9], rd[7], rd[5], S, NP)
    assert cfg.counter.value >= 40


def test_round_robin_time_slicing(tables, golden):
    """forward_kernel hands chunks back to the run queue every NPORE_RR_SLICE anti-diagonals (state saved to HBM and
    resumed by whichever warp pops it next): results must not depend on the slice length."""
    from npore_b200.engine import Realigner
    S, NP = tables
    cases = [c for c in golden("fuzz.json.gz") if c["r"] == 30 and c["max_b_rows"] == 20000]
    refs = [oracle.bases_to_int(c["ref"]) for c in cases]; seqs = [oracle.bases_to_int(c["seq"]) for c in cases]
    for sl in ("8", "37", "100000"):
        os.environ["NPORE_RR_SLICE"] = sl
        try:
            eng = Realigner(S, NP)
        finally:
            del os.environ["NPORE_RR_SLICE"]
        outs, scores, status = eng.align_many(refs, seqs, [c["cigar"] for c in cases])
        for c, o, sc in zip(cases, outs, scores):
            assert o == c["out"] and np.array_equal(sc, np.array(c["scores"], np.float32))
        eng.close()


def test_np_info_long_and_batched(tables, engine_factory):
    """Stand-alone get_np_info on sequences longer than the chunk window (global equality words) and batched (N4)."""
    eng = engine_factory()
    rng = np.random.default_rng(17)
    long_seq = synth.make_reference(150_000, rng, 0.4, "ACGTN")
    long_seq = long_seq[:70_000] + "A" * 300 + long_seq[70_000:]
    a = oracle.bases_to_int(long_seq)
    assert np.array_equal(eng.get_np_info(a), oracle.get_np_info(a))
    seqs = [oracle.bases_to_int(synth.make_reference(int(rng.integers(0, 5000)), rng, 0.5)) for _ in range(12)] + [np.zeros(0, np.uint8)]
    for got, s_ in zip(eng.get_np_info_batch(seqs), seqs):
        assert np.array_equal(got, oracle.get_np_info(s_))


def test_np_region_beds(tables, tmp_path):
    """bed.py:56-145 on the device np_info: regions = tract starts, padded, merged per n."""
    from npore_b200 import bed, cfg
    cfg.args.max_n, cfg.args.max_l = 6, 100
    rng = np.random.default_rng(23)
    refs = {"chr1": synth.make_reference(30_000, rng, 0.3), "chr2": synth.make_reference(8_000, rng, 0.6)}
    windows = [("chr1", 0, 10_000), ("chr1", 10_000, 20_000), ("chr1", 20_000, 30_000), ("chr2", 0, 8_000)]
    got = bed.get_np_regions_batch(windows, refs)
    for (ctg, a, b), per_n in zip(windows, got):
        info = oracle.get_np_info(oracle.bases_to_int(refs[ctg][a:b]))
        for n in range(1, 7):
            want = [(ctg, a + p, a + p + n * int(info[p, 0, n - 1])) for p in range(b - a) if info[p, 0, n - 1] and not info[p, 1, n - 1]]
            assert per_n[n - 1] == want
    assert bed.merge_regions([("c", 5, 9), ("c", 10, 12), ("c", 30, 31), ("b", 1, 2)], slop=1) == [("b", 0, 3), ("c", 4, 13), ("c", 29, 32)]
    bed.save_np_region_beds(got, str(tmp_path / "np"))
    assert (tmp_path / "np_1.bed").read_text().count("\n") > 0 and (tmp_path / "np_all.bed").exists()


def test_c_abi_error_behaviour(tables):
    """include/npore_b200.h conventions: negative codes, never abort; call order upload -> run -> download."""
    import ctypes as C
    from npore_b200 import _lib
    from npore_b200.engine import PackedBatch, Realigner, cigar_to_rle
    S, NP = tables
    L = _lib.lib()
    ctx = C.c_void_p()
    s32 = np.ascontiguousarray(S, np.float32); n32 = np.ascontiguousarray(NP, np.float32)
    bad_args = [dict(max_n=7), dict(max_l=128), dict(max_b_rows=1), dict(r=0), dict(r=200), dict(device=99)]
    for kw in bad_args:
        a = dict(device=0, max_n=6, max_l=100, max_b_rows=20000, r=30); a.update(kw)
        rc = L.npore_ctx_create(C.byref(ctx), a["device"], s32.ctypes.data, n32.ctypes.data, 6, 101, a["max_n"], a["max_l"], 5.0, 1.0, a["max_b_rows"], a["r"])
        assert rc == -1 and not ctx.value, kw                                   # NPORE_ERR_BAD_ARG, no context leaked
    assert L.npore_strerror(-5).startswith(b"call out of order")
    eng = Realigner(S, NP)
    packed = PackedBatch([oracle.bases_to_int("ACGTACGT")], [oracle.bases_to_int("ACGTACGT")], [cigar_to_rle("8=")], pinned=False)
    res = eng.new_result(packed, 0, pinned=False)
    r = res.c_struct()
    assert L.npore_run(eng._ctx, 0) == -5                                       # run before upload
    assert L.npore_download(eng._ctx, C.byref(r)) == -5                         # download before run
    eng.upload(packed)
    assert L.npore_download(eng._ctx, C.byref(r)) == -5
    assert L.npore_run(eng._ctx, 4) == -1                                       # NO_EXPANDED without RLE
    eng.run(0)
    r.ops_capacity = 3                                                          # caller buffer too small
    assert L.npore_download(eng._ctx, C.byref(r)) == -6 and b"too small" in L.npore_last_error(eng._ctx)
    r = res.c_struct()
    assert L.npore_download(eng._ctx, C.byref(r)) == 0 and res.ops_str(0) == "=" * 8
    # out-of-range sequence window
    packed.ref_len[0] = 100
    b = packed.c_struct()
    assert L.npore_upload(eng._ctx, C.byref(b)) == -1
    eng.close()
