"""The file pipeline of bamio.realign_bam (BAM file in, SAM file out) without a device: the engine is replaced by a stand-in whose
"realignment" returns the input CIGAR, so the native reader, the batch cut, the writer thread, region sharding and the error
path all run on a CPU.  The SAM body must equal bam.sam_record over the pure-Python decode (bamio.get_read_data)."""
import concurrent.futures
import os
import re
import threading
import time
import types

import numpy as np
import pytest

from npore_b200 import bamio, cfg, synth
from npore_b200.bam import sam_record

PHASES = {"open", "gather", "gpu_wait", "format", "write"}


class _EchoEngine:
    """submit() returns an already completed future of (result, stats): the result carries the batch's own CIGAR words.  The
    future of submit number `fail_at` (1-based) raises instead.  `consumed` counts the records of the results handed out."""

    def __init__(self, fail_at=0):
        self.fail_at, self.submitted, self.consumed = fail_at, 0, 0
        self._lock = threading.Lock()

    def submit(self, packed, flags=0):
        engine = self

        class Fut(concurrent.futures.Future):
            def result(self, timeout=None):
                out = super().result(timeout)
                with engine._lock:
                    engine.consumed += packed.n
                return out

        fut = Fut()
        with self._lock:
            self.submitted += 1
            fail = self.submitted == self.fail_at
        if fail:
            fut.set_exception(RuntimeError("stand-in batch failure"))
        else:
            t = time.perf_counter()
            res = types.SimpleNamespace(rle=packed.cigar_rle, rle_off=packed.cigar_off, status=np.zeros(max(packed.n, 1), np.int32))
            fut.set_result((res, {"ms_kernels_total": 0.0, "ms_h2d": 0.0, "ms_plan": 0.0, "ms_d2h": 0.0, "fwd_warps_per_sm": 0, "wall": (t, t, t)}))
        return fut


@pytest.fixture(scope="module")
def fixture_bam(tmp_path_factory):
    """A coordinate-sorted BAM of synthetic reads on two contigs (no clips, so the input CIGAR is what the SAM carries)."""
    t = np.load(os.path.join(os.path.dirname(__file__), "golden", "tables.npz"))
    rng = np.random.default_rng(2024)
    cm = synth.call_length_model(t["np_scores"])
    contigs, recs = [], []
    for ci, (name, length, n_reads) in enumerate((("chrA", 24_000, 60), ("chrB", 15_000, 40))):
        ref, tr = synth.make_reference_with_tracts(length, rng)
        contigs.append((name, ref))
        for rd in synth.make_reads(ref, n_reads, 1000, rng, cm, tracts=tr):
            recs.append({"name": f"{name}_{rd[0]}", "flag": 0, "ref_id": ci, "pos": rd[3], "mapq": 60, "seq": rd[7],
                         "qual": bytes(rng.integers(0, 40, len(rd[7])).astype(np.uint8)),
                         "cigar": [(int(a), b) for a, b in re.findall(r"(\d+)(\D)", rd[5])], "tags": {"HP": rd[10]}})
    path = str(tmp_path_factory.mktemp("bam") / "in.bam")
    bamio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n", [(n, len(s)) for n, s in contigs], recs)
    return path, dict(contigs), t["sub_scores"], t["np_scores"]


@pytest.fixture
def echo(fixture_bam, monkeypatch):
    """Installs a stand-in engine for every device; call it with fail_at to replace it."""
    _, _, S, NP = fixture_bam
    monkeypatch.setattr(cfg.args, "sub_scores", S)
    monkeypatch.setattr(cfg.args, "np_scores", NP)
    monkeypatch.setattr(cfg.args, "out_prefix", cfg.args.out_prefix)

    def install(fail_at=0):
        eng = _EchoEngine(fail_at)
        monkeypatch.setattr(bamio, "_pipeline", lambda sub, npt, n_inflight, device=None: eng)
        return eng
    return install


def _body(path):
    with open(path) as fh:
        return "".join(line for line in fh if not line.startswith("@"))


def _want(bam, fa, regions=None, max_reads=0):
    return "".join(sam_record(t, t[5]) + "\n" for t in bamio.get_read_data(bam, fa, regions=regions, max_reads=max_reads))


def _run(bam, fa, prefix, **kw):
    before = cfg.counter.value
    n = bamio.realign_bam(bam, fa, out_prefix=str(prefix), argv=["t"], **kw)
    assert cfg.counter.value - before == n
    return n


@pytest.mark.parametrize("kw", [{}, {"window_bytes": 20_000, "max_batch_ops": 5_000}, {"n_inflight": 1, "max_batch_ops": 5_000},
                                {"n_inflight": 3, "window_bytes": 20_000}, {"window_bytes": 0}])
def test_single_device_output_is_the_reference_record_text(fixture_bam, echo, tmp_path, kw):
    bam, fa, _, _ = fixture_bam
    eng = echo()
    tm = {"trace": []}
    n = _run(bam, fa, tmp_path / "out", timings=tm, **kw)
    want = _want(bam, fa)
    assert n == want.count("\n") == 100 and _body(tmp_path / "out.sam") == want
    assert eng.submitted >= (20 if "max_batch_ops" in kw else 1)
    assert set(tm) == PHASES | {"trace"} and tm["trace"]
    assert [ev for _, ev in tm["trace"]].count("header written") == 1


def test_regions_and_max_reads(fixture_bam, echo, tmp_path):
    bam, fa, _, _ = fixture_bam
    echo()
    region = [("chrB", 3_000, 9_000)]
    n = _run(bam, fa, tmp_path / "reg", regions=region, window_bytes=20_000, max_batch_ops=5_000)
    want = _want(bam, fa, regions=region)
    assert 0 < n < 40 and _body(tmp_path / "reg.sam") == want
    two = [("chrA", 0, 5_000), ("chrB", 0, 4_000)]
    n = _run(bam, fa, tmp_path / "two", regions=two, max_batch_ops=5_000)
    assert n and _body(tmp_path / "two.sam") == _want(bam, fa, regions=two)
    # max_reads that ends inside the second window
    nb = bamio.NativeBam(bam, window_bytes=20_000)
    first = nb.advance()
    second = nb.advance()
    nb.close()
    assert first and second > 2
    k = first + second // 2
    n = _run(bam, fa, tmp_path / "max", window_bytes=20_000, max_reads=k, max_batch_ops=5_000)
    assert n == k and _body(tmp_path / "max.sam") == _want(bam, fa, max_reads=k)


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
def test_sharded_output_is_byte_identical(fixture_bam, echo, tmp_path, devices):
    bam, fa, _, _ = fixture_bam
    echo()
    _run(bam, fa, tmp_path / "one", max_batch_ops=5_000)
    tm = {}
    n = _run(bam, fa, tmp_path / "many", max_batch_ops=5_000, devices=devices, timings=tm)
    assert open(tmp_path / "many.sam", "rb").read() == open(tmp_path / "one.sam", "rb").read()
    assert n == 100 and sum(s["reads"] for s in tm["shards"]) == n and len(tm["shards"]) == len(devices)
    assert set(tm) == PHASES | {"concat", "shards"}
    assert not [f for f in os.listdir(tmp_path) if ".part" in f]


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_a_failed_batch_is_raised_and_counted_to_the_last_record_written(fixture_bam, echo, tmp_path, devices):
    bam, fa, _, _ = fixture_bam
    eng = echo(fail_at=4)
    before = cfg.counter.value
    with pytest.raises(RuntimeError, match="stand-in batch failure"):
        bamio.realign_bam(bam, fa, out_prefix=str(tmp_path / "out"), argv=["t"], window_bytes=20_000, max_batch_ops=5_000,
                          devices=devices)
    assert eng.submitted >= 4 and 0 < eng.consumed < 100
    assert cfg.counter.value - before == eng.consumed
    assert not [f for f in os.listdir(tmp_path) if ".part" in f]
