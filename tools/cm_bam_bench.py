"""confusion.count_bam on seeded BAM files: streamed pass against a read-only pass over the same file, host peak RSS, and the
whole-file Python path (load_alignments + calc_confusion_matrices_batch) on a prefix with an equality check of the counts.

    python tools/cm_bam_bench.py [--contig-len 1000000] [--reads 750] [--read-len 10000] [--tiles 4,16] [--reps 2]

The files are made cheaply: one generated contig and its reads (synth.make_aligned_reads) are tiled onto `tiles` contigs of
the same sequence, each carrying the same reads.  Every measurement runs in a fresh child process, so that its peak RSS is
its own.  Everything is written to a temporary directory; one JSON line per measurement goes to stdout."""
import argparse
import json
import os
import resource
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _peak_mb():
    """Peak RSS of this process (VmHWM: reset by exec, unlike ru_maxrss, which a child inherits from the parent's fork)."""
    with open("/proc/self/status") as fh:
        for line in fh:
            if line.startswith("VmHWM:"):
                return int(line.split()[1]) / 1024.0
    return resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024.0


def child(mode, bam, fasta, window_bytes):
    import numpy as np
    from npore_b200 import bamio, confusion
    out = {"mode": mode, "file": os.path.basename(bam), "file_mb": os.path.getsize(bam) / 1e6}
    if mode == "read_only":
        t = time.perf_counter()
        b = bamio.NativeBam(bam, 0, window_bytes)
        n = 0
        while True:
            k = b.advance()
            if not k:
                break
            n += k
        b.close()
        out.update(wall_s=time.perf_counter() - t, records=n)
    elif mode == "count_bam":
        refs = bamio.read_fasta(fasta)
        confusion._np_engine()                       # device context set up before the clock starts
        base = _peak_mb()
        tm = {}
        t = time.perf_counter()
        res = confusion.count_bam(bam, refs, window_bytes=window_bytes, timings=tm)
        out.update(wall_s=time.perf_counter() - t, timings=tm, rss_before_mb=base, subs_sum=int(res[0].sum()))
        np.savez(bam + ".stream.npz", *res)
    elif mode == "batch_path":
        refs = bamio.read_fasta(fasta)
        confusion._np_engine()
        t = time.perf_counter()
        reads = confusion.load_alignments(bam)
        t_load = time.perf_counter() - t
        regions = [(c, 0, len(s)) for c, s in refs.items() if c in reads]
        res = confusion.calc_confusion_matrices_batch(confusion.get_ranges(regions), refs, reads)
        out.update(wall_s=time.perf_counter() - t, load_s=t_load)
        stream = np.load(bam + ".stream.npz")
        out["equal_to_count_bam"] = all(np.array_equal(a, stream[f"arr_{i}"]) for i, a in enumerate(res))
    out["peak_rss_mb"] = _peak_mb()
    if mode == "count_bam":
        out["reads_per_s"] = out["timings"]["reads"] / out["wall_s"]
    out["compressed_mb_per_s"] = out["file_mb"] / out["wall_s"]
    print(json.dumps(out), flush=True)


def make_files(d, contig_len, n_reads, read_len, tiles, seed=5):
    import numpy as np
    from npore_b200 import bamio, synth
    rng = np.random.default_rng(seed)
    t = time.perf_counter()
    contig = synth.make_reference(contig_len, rng, p_np=0.35)
    reads = synth.make_aligned_reads(contig, n_reads, read_len, rng)
    gen_s = time.perf_counter() - t
    files = {}
    for n_ctg in sorted(set(tiles) | {1}):
        names = [f"t{k}" for k in range(n_ctg)]
        recs = [{"name": f"{c}_{i}", "flag": r[4], "ref_id": k, "pos": r[0], "mapq": r[5], "cigar": r[1], "seq": r[2], "qual": r[3]}
                for k, c in enumerate(names) for i, r in enumerate(reads)]
        bam = os.path.join(d, f"tiles{n_ctg}.bam")
        bamio.write_bam(bam, "@HD\tVN:1.6\tSO:coordinate\n", [(c, len(contig)) for c in names], recs, level=1)
        fa = os.path.join(d, f"tiles{n_ctg}.fa")
        with open(fa, "w") as fh:
            fh.write("".join(f">{c}\n{contig}\n" for c in names))
        files[n_ctg] = (bam, fa)
    print(json.dumps({"mode": "make_files", "generate_s": gen_s, "make_s": time.perf_counter() - t, "reads_per_tile": n_reads,
                      "read_len": read_len, "contig_len": contig_len,
                      "files": {k: os.path.getsize(v[0]) for k, v in files.items()}}), flush=True)
    return files


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contig-len", type=int, default=1_000_000)
    ap.add_argument("--reads", type=int, default=750)
    ap.add_argument("--read-len", type=int, default=10_000)
    ap.add_argument("--tiles", default="4,16")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--window-bytes", type=int, default=16 << 20)
    ap.add_argument("--child", nargs=3, metavar=("MODE", "BAM", "FASTA"))
    a = ap.parse_args()
    if a.child:
        return child(a.child[0], a.child[1], a.child[2], a.window_bytes)
    print(json.dumps({"gpu": gpu_info(), "host_cpus": os.cpu_count()}), flush=True)
    with tempfile.TemporaryDirectory() as d:
        files = make_files(d, a.contig_len, a.reads, a.read_len, [int(x) for x in a.tiles.split(",")])
        run = lambda mode, f: subprocess.run([sys.executable, __file__, "--child", mode, *f, "--window-bytes", str(a.window_bytes)],   # noqa: E731
                                             check=True)
        for n_ctg in sorted(files):
            for _ in range(a.reps):            # alternate the two passes over the same file
                run("read_only", files[n_ctg])
                run("count_bam", files[n_ctg])
        run("batch_path", files[1])            # the prefix: the first tile alone


if __name__ == "__main__":
    main()
