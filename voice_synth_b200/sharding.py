"""Static partition of independent streams over ranks/GPUs (SURVEY.md 8e): contiguous ranges, no
collective on the data path.  bench.py and the corpus driver use it; the C library applies the same
rule (balanced by samples) inside a multi-device vs_ctx."""
import numpy as np


def shard_range(n, rank, world):
    """streams [lo, hi) of rank `rank`: contiguous, sizes differ by at most one"""
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_by_samples(nsamples, world):
    """cut points [world+1] over streams such that every rank gets ~the same number of samples
    (the rule vs_split_slots in vs_batch_plan.cpp applies to the device slots of one ctx)"""
    ns = np.asarray(nsamples, dtype=np.uint64)
    total = int(ns.sum())
    cuts = [0]
    acc, g = 0, 1
    for i, v in enumerate(ns):
        acc += int(v)
        while g < world and acc * world >= total * g:
            cuts.append(i + 1)
            g += 1
    while len(cuts) < world + 1:
        cuts.append(len(ns))
    cuts[-1] = len(ns)
    return cuts


def rank_seeds(n_per_rank, rank, base=1000):
    """weak-scaling workload: every rank synthesises its own streams; seeds never collide"""
    return (base + rank * n_per_rank + np.arange(n_per_rank)).astype(np.uint32)
