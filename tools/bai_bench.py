"""What the BAM index costs at write time, and what it gives a region query.

(a) realign_bam BAM output of the C2 file of tools/bam_out_bench.py (bench.make_workload: 10 kb reads on a 1 Mb tract-rich
    reference, nanopore-like qualities), index=False and index=True in turns (one warm-up call each, then --reps timed calls
    each).  Reported: reads/s of both, the writer-thread seconds of the index (timings["index"]: the device stage plus the fold
    and the write of the .bai) and the npore_bgzf_index kernel milliseconds per call.
(b) A file of --big-reads 1 kb reads on a 20 Mb reference, realigned into an indexed BAM (index=True); that BAM is then the
    input of a realignment of one 1 Mb region, with its index and with the index moved away, in turns (--reps each).
    Reported: wall time of both, the compressed bytes the reader reads (NativeBam.bytes_read) against the file size, and
    whether the two SAM outputs are identical.
The card's name, power limit and clock are read in the same process.

    python tools/bai_bench.py [--reads 3000] [--reps 5] [--big-reads 200000] [--json out.json]
"""
import argparse
import json
import os
import shutil
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench                                            # noqa: E402
from bam_out_bench import gpu_info, write_input         # noqa: E402
from npore_b200 import bamio, cfg                       # noqa: E402


def write_cost(bam, fa, out_dir, n_reads, reps):
    runs = {False: [], True: []}
    for rep in range(reps + 1):                          # call 0 of each setting is the warm-up
        for index in (False, True):
            tm = {}
            t = time.perf_counter()
            n = bamio.realign_bam(bam, fa, out_prefix=os.path.join(out_dir, "out"), argv=["bai_bench"], timings=tm, out_format="bam",
                                  index=index)
            dt = time.perf_counter() - t
            assert n == n_reads, (n, n_reads)
            if rep:
                runs[index].append({"seconds": dt, "index_s": tm.get("index", 0.0), "kernel_ms": tm.get("index_device_ms", 0.0)})
    off, on = runs[False], runs[True]
    med = lambda rs, k: statistics.median(r[k] for r in rs)   # noqa: E731
    return {"reads": n_reads, "reads_per_s_no_index": round(n_reads / med(off, "seconds")), "reads_per_s_index": round(n_reads / med(on, "seconds")),
            "seconds_no_index": [round(r["seconds"], 4) for r in off], "seconds_index": [round(r["seconds"], 4) for r in on],
            "wall_overhead_median": round(med(on, "seconds") / med(off, "seconds") - 1, 4),
            "writer_index_seconds_median": round(med(on, "index_s"), 5), "index_kernel_ms_per_call_median": round(med(on, "kernel_ms"), 3),
            }


def region_query(n_reads, out_dir, reps):
    S, NP = bench.load_tables()
    ref, reads = bench.make_workload(7, 20_000_000, n_reads, 1000, NP)
    src = os.path.join(out_dir, "big_in.bam")
    write_input(src, ref, reads, False, seed=3)
    fa = {"chr1": ref}
    n_all = bamio.realign_bam(src, fa, out_prefix=os.path.join(out_dir, "big"), argv=["bai_bench"], out_format="bam", index=True)
    path = os.path.join(out_dir, "big.bam")
    size = os.path.getsize(path)
    region = [("chr1", 9_500_000, 10_500_000)]
    runs = {True: [], False: []}
    for rep in range(reps + 1):                          # call 0 of each setting is the warm-up
        for with_index in (True, False):
            if not with_index:
                os.replace(path + ".bai", path + ".bai.away")
            try:
                t = time.perf_counter()
                n = bamio.realign_bam(path, fa, out_prefix=os.path.join(out_dir, f"reg_{with_index}"), argv=["bai_bench"], regions=region)
                dt = time.perf_counter() - t
                nb = bamio.NativeBam(path, regions=region)
                used, read = nb.index is not None, nb.bytes_read
                nb.close()
            finally:
                if not with_index:
                    os.replace(path + ".bai.away", path + ".bai")
            if rep:
                runs[with_index].append({"seconds": dt, "reads": n, "bytes_read": read, "index_used": used})
    same = open(os.path.join(out_dir, "reg_True.sam"), "rb").read() == open(os.path.join(out_dir, "reg_False.sam"), "rb").read()
    med = lambda rs: statistics.median(r["seconds"] for r in rs)   # noqa: E731
    return {"file_reads": int(n_all), "file_bytes": size, "region": region[0],
            "region_reads": runs[True][-1]["reads"], "seconds_with_index": [round(r["seconds"], 4) for r in runs[True]],
            "seconds_without_index": [round(r["seconds"], 4) for r in runs[False]], "median_speedup": round(med(runs[False]) / med(runs[True]), 2),
            "bytes_read_with_index": runs[True][-1]["bytes_read"], "bytes_read_without_index": runs[False][-1]["bytes_read"],
            "fraction_read_with_index": round(runs[True][-1]["bytes_read"] / size, 4),
            "index_used": [runs[True][-1]["index_used"], runs[False][-1]["index_used"]], "sam_outputs_identical": same}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reads", type=int, default=3000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--big-reads", type=int, default=200_000)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    S, NP = bench.load_tables()
    cfg.args.sub_scores, cfg.args.np_scores = S, NP
    result = {"gpu": gpu_info(), "host_cores": os.cpu_count()}
    work = tempfile.mkdtemp(prefix="bai_bench_")
    try:
        ref, reads = bench.make_workload(20260101, 1_000_000, a.reads, 10000, NP)
        bam = os.path.join(work, "in.bam")
        write_input(bam, ref, reads, True, seed=a.reads)
        result["write_cost"] = write_cost(bam, {"chr1": ref}, work, a.reads, a.reps)
        print(json.dumps(result["write_cost"]), flush=True)
        if a.big_reads:
            result["region_query"] = region_query(a.big_reads, work, a.reps)
            print(json.dumps(result["region_query"]), flush=True)
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
