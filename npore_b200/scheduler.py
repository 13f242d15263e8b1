"""Host-side batch scheduler pieces that replace the reference's multiprocessing.Pool (realign.py:110-114):

  iter_batches     cut a (lazy) stream of items into GPU batches bounded by total D/I ops (memory-bounded);
                   inside a batch the library sorts chunks longest-first over persistent warps (csrc/api.cu).
  n_cu             cell updates of an item (SURVEY.md 8(d)): (Lref + Lseq + n_chunks) * (2r+1)
  shard_by_region  split coordinate-sorted reads into G contiguous genomic regions of equal cell-update load,
                   one per GPU (SURVEY.md 8(e)); no collective: every shard is realigned independently and the
                   host concatenates the per-GPU outputs in region order.
  cut_balanced     the same cut for items that are ALREADY in (contig, start) order: owner shard of every item, contiguous
                   and non-decreasing, by the item's load midpoint (bamio.realign_bam with devices=[...]).
"""
import numpy as np


def iter_batches(items, size_of, max_ops):
    batch, tot = [], 0
    for it in items:
        s = size_of(it)
        if batch and tot + s > max_ops:
            yield batch
            batch, tot = [], 0
        batch.append(it)
        tot += s
    if batch:
        yield batch


def n_chunks(total_ops: int, max_b_rows: int = 20000) -> int:
    return -(-total_ops // (max_b_rows - 1)) if total_ops > 0 else 0


def n_cu(ref_len: int, seq_len: int, max_b_rows: int = 20000, r: int = 30) -> int:
    ops = ref_len + seq_len
    return (ops + n_chunks(ops, max_b_rows)) * (2 * r + 1)


def shard_by_region(starts, loads, world: int):
    """starts: reference start per read (any order); loads: n_cu per read.  Returns a list of `world` index arrays:
    reads sorted by start, cut into contiguous runs of (nearly) equal total load."""
    starts = np.asarray(starts)
    loads = np.asarray(loads, dtype=np.float64)
    order = np.argsort(starts, kind="stable")
    csum = np.cumsum(loads[order])
    total = csum[-1] if len(csum) else 0.0
    cuts = [int(np.searchsorted(csum, total * g / world, side="right")) for g in range(1, world)]
    bounds = [0] + cuts + [len(order)]
    return [order[bounds[g]:bounds[g + 1]] for g in range(world)]


def cut_balanced(loads, world: int, done: float = 0.0, total: float = None):
    """Owner shard (0 .. world-1) of every item of an ordered list: item k goes to the shard that contains the midpoint of
    its load interval [csum[k-1], csum[k]) on the axis [0, total) cut into `world` equal parts -- contiguous, non-decreasing,
    every shard's load within one item of total / world.  `done` / `total` let a caller cut a list that arrives in pieces
    (one piece per contig): pass the load already seen and the grand total."""
    loads = np.asarray(loads, dtype=np.float64)
    cs = done + np.cumsum(loads)
    tot = float(total if total is not None else (cs[-1] if len(cs) else 0.0))
    return np.minimum((cs - loads / 2.0) * world / max(tot, 1.0), world - 1).astype(np.int64)
