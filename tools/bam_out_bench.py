"""BAM output against SAM output of bamio.realign_bam, and the BGZF compressor on its own.

The workload is C2 as a file (bench.make_workload: 10 kb reads on a 1 Mb tract-rich reference), at 3,000 and 12,000 reads, in
two variants: no qualities (QUAL 0xFF), and nanopore-like qualities (a 50-tap moving average of N(18, 6) plus N(0, 5) noise,
clipped to 2..50).  Per variant, realign_bam writes SAM and BAM in turns (one warm-up call each, then --reps timed calls each);
reported: reads/s, output bytes per read, and the forward-kernel time of every batch from the trace.  Then the compressor alone
on a >= 64 MB stream of the variant's BAM records (device ms from npore_bgzf_compress, input GB/s), and host zlib at levels 1
and 6 on all cores over the same stream.  The card's name, power limit and clock are read in the same process.

    python tools/bam_out_bench.py [--reads 3000 12000] [--reps 5] [--json out.json]
"""
import argparse
import concurrent.futures
import gzip
import json
import os
import re
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                            # noqa: E402
from npore_b200 import bamio, cfg                       # noqa: E402


def nanopore_quals(rng, n):
    m = np.convolve(rng.normal(18, 6, n + 50), np.ones(50) / 50, "valid")[:n]
    return np.clip(m + rng.normal(0, 5, n), 2, 50).astype(np.uint8).tobytes()


def write_input(path, ref, reads, with_quals, seed):
    rng = np.random.default_rng(seed)
    recs = [{"name": r[0], "flag": r[1], "ref_id": 0, "pos": r[3], "mapq": r[4], "seq": r[7],
             "qual": nanopore_quals(rng, len(r[7])) if with_quals else None,
             "cigar": [(int(a), b) for a, b in re.findall(r"(\d+)(\D)", r[5])], "tags": {"HP": r[10]}}
            for r in sorted(reads, key=lambda r: r[3])]
    bamio.write_bam(path, "@HD\tVN:1.6\tSO:coordinate\n", [("chr1", len(ref))], recs, level=1)


def kernel_ms(trace):
    """Forward-kernel milliseconds of every batch ("gpu done ... kernels_ms=")."""
    return [float(m.group(1)) for _, ev in trace for m in [re.search(r"kernels_ms=([0-9.]+)", ev)] if m]


def file_to_file(bam, fa, out_dir, n_reads, reps):
    runs = {"sam": [], "bam": []}
    for rep in range(reps + 1):                          # call 0 of each format is the warm-up
        for fmt in ("sam", "bam"):
            tm = {"trace": []}
            t = time.perf_counter()
            n = bamio.realign_bam(bam, fa, out_prefix=os.path.join(out_dir, "out"), argv=["bam_out_bench"], timings=tm, out_format=fmt)
            dt = time.perf_counter() - t
            assert n == n_reads, (n, n_reads)
            if rep:
                size = os.path.getsize(os.path.join(out_dir, f"out.{fmt}"))
                runs[fmt].append({"seconds": dt, "bytes": size, "kernels_ms": kernel_ms(tm["trace"]),
                                  "timings": {k: round(v, 4) for k, v in tm.items() if k != "trace"}})
    out = {}
    for fmt, rs in runs.items():
        secs = [r["seconds"] for r in rs]
        kms = [k for r in rs for k in r["kernels_ms"]]
        out[fmt] = {"reads_per_s_mean": round(n_reads / statistics.mean(secs)), "reads_per_s_median": round(n_reads / statistics.median(secs)),
                    "seconds": [round(s, 4) for s in secs], "bytes": rs[-1]["bytes"], "bytes_per_read": round(rs[-1]["bytes"] / n_reads, 1),
                    "batches": len(rs[-1]["kernels_ms"]), "kernels_ms_per_batch_mean": round(statistics.mean(kms), 2) if kms else None,
                    "timings_last": rs[-1]["timings"]}
    out["bam_over_sam_reads_per_s"] = round(out["bam"]["reads_per_s_mean"] / out["sam"]["reads_per_s_mean"], 3)
    if out["sam"]["kernels_ms_per_batch_mean"]:
        out["bam_over_sam_kernels_ms"] = round(out["bam"]["kernels_ms_per_batch_mean"] / out["sam"]["kernels_ms_per_batch_mean"], 3)
    return out


def compressor_alone(payload, reps):
    from npore_b200.engine import BgzfCompressor
    z = BgzfCompressor(int(getattr(cfg.args, "device", 0) or 0))
    out = bytes(z.compress(payload))                     # warm-up (and buffer growth)
    assert gzip.decompress(out) == payload
    ms, wall = [], []
    for _ in range(reps):
        t = time.perf_counter()
        z.compress(payload)
        wall.append(time.perf_counter() - t)
        ms.append(z.last_device_ms)
    z.close()
    return {"input_bytes": len(payload), "output_bytes": len(out), "ratio": round(len(out) / len(payload), 4),
            "device_ms": [round(x, 3) for x in ms], "input_GB_per_s_device": round(len(payload) / (statistics.median(ms) * 1e-3) / 1e9, 2),
            "input_GB_per_s_call": round(len(payload) / statistics.median(wall) / 1e9, 2)}


def host_zlib(payload, level, threads):
    chunks = [payload[i:i + 65280] for i in range(0, len(payload), 65280)]

    def one(c):
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        zlib.crc32(c)                                    # a BGZF writer computes each member's CRC too
        return len(co.compress(c) + co.flush()) + 26
    with concurrent.futures.ThreadPoolExecutor(threads) as pool:      # zlib releases the GIL
        sum(pool.map(one, chunks[:threads]))
        t = time.perf_counter()
        size = sum(pool.map(one, chunks))
        dt = time.perf_counter() - t
    return {"level": level, "threads": threads, "output_bytes": size, "ratio": round(size / len(payload), 4),
            "input_GB_per_s": round(len(payload) / dt / 1e9, 3)}


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    except OSError as e:
        return [f"nvidia-smi: {e}"]
    return r.stdout.strip().splitlines()[:1] if r.returncode == 0 else [f"nvidia-smi failed: {r.stderr.strip()}"]


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reads", type=int, nargs="+", default=[3000, 12000])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--stream-mb", type=int, default=64)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    S, NP = bench.load_tables()
    cfg.args.sub_scores, cfg.args.np_scores = S, NP
    result = {"gpu": gpu_info(), "host_cores": os.cpu_count(), "workloads": []}
    work = tempfile.mkdtemp(prefix="bam_out_bench_")
    try:
        for n_reads in a.reads:
            ref, reads = bench.make_workload(20260101, 1_000_000, n_reads, 10000, NP)
            for with_quals in (False, True):
                name = f"{n_reads} reads, {'nanopore-like qualities' if with_quals else 'no qualities'}"
                bam = os.path.join(work, "in.bam")
                write_input(bam, ref, reads, with_quals, seed=n_reads)
                row = {"workload": name, "file_to_file": file_to_file(bam, {"chr1": ref}, work, n_reads, a.reps)}
                if n_reads == max(a.reads):
                    raw = gzip.open(bam).read()
                    payload = (raw * (a.stream_mb * (1 << 20) // len(raw) + 1))[:max(a.stream_mb * (1 << 20), len(raw))]
                    row["compressor"] = compressor_alone(payload, a.reps)
                    row["host_zlib"] = [host_zlib(payload, lv, os.cpu_count() or 1) for lv in (1, 6)]
                result["workloads"].append(row)
                print(json.dumps(row), flush=True)
    finally:
        shutil.rmtree(work, ignore_errors=True)
    result["gpu_after"] = gpu_info()
    print(json.dumps({"gpu": result["gpu"], "gpu_after": result["gpu_after"], "host_cores": result["host_cores"]}))
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
