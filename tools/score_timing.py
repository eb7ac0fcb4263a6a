#!/usr/bin/env python
"""Time scoring a given partition on one GPU: kp_partition_assign (owner table, overlap and gap checks) plus
kp_partition_score (per-pattern counts and terms), as PartitionPlan.partition_assign / partition_score call them, so
the times include the upload of the pattern numbers and the host synchronisations of both calls.

    python tools/score_timing.py [--reps R]

Partitions: random split trees of N^11 and N^13 (a leaf and a position drawn at random, the position's letter cut in
two), which mix a few huge patterns with many small ones, and the all-k-mers partition of N^11 (4^11 patterns of one
k-mer each).  CUDA events around each call pair; median and min of R timed runs after two warm-up runs.  Bytes are the
owner table (4 B) and the two int64 count tables (16 B) per k-mer; at N^11 they fit in L2 (84 MB), at N^13 not (1.3 GB).
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from kmerpapa_b200 import iupac
from kmerpapa_b200.engine import PartitionPlan
from kmerpapa_b200.score_partition import pattern_numbers


def random_partition(gen, nsplit, rng):
    leaves = [[iupac.MASK[c] for c in gen]]
    for _ in range(nsplit):
        j = int(rng.integers(len(leaves)))
        free = [i for i, m in enumerate(leaves[j]) if m & (m - 1)]
        if not free:
            continue
        i = free[int(rng.integers(len(free)))]
        m = leaves[j][i]
        subs = [s for s in range(1, 16) if s & m == s and s != m]
        s = subs[int(rng.integers(len(subs)))]
        a, b = list(leaves[j]), list(leaves[j])
        a[i], b[i] = s, m ^ s
        leaves[j] = a
        leaves.append(b)
    return ["".join(iupac.LETTER[m] for m in leaves[o]) for o in rng.permutation(len(leaves))]


def all_kmers_patnums(k):
    """Dense numbers of the single k-mers of N^k (A, C, G, T are digits 0-3 of N), in k-mer index order."""
    idx = np.arange(4 ** k, dtype=np.uint64)
    num = np.zeros_like(idx)
    for i in range(k):
        num += ((idx >> np.uint64(2 * i)) & np.uint64(3)) * np.uint64(15 ** i)
    return num


def gpu_identity():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:   # the numbers are still printed; say what is missing
        return f"{torch.cuda.get_device_name()} (power limit unknown: {e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("score_timing needs a CUDA device")
    print("device:", gpu_identity(), flush=True)
    rng = np.random.default_rng(2024)
    cases = []
    for k, nsplit in ((11, 5000), (13, 5000), (13, 50000)):
        gen = "N" * k
        pats = random_partition(gen, nsplit, rng)
        cases.append((f"N^{k} split tree", gen, pattern_numbers(pats, gen)))
    cases.append(("N^11 all k-mers", "N" * 11, all_kmers_patnums(11)))
    for label, gen, patnums in cases:
        plan = PartitionPlan(gen, 0, lite=True)
        nk = plan.nkmer
        U = rng.negative_binomial(1, 1e-3, nk).astype(np.int64)
        M = rng.binomial(U, 0.01).astype(np.int64)
        kM, kU = plan.upload_kmer_tables(M, U, name="st")
        rates = np.full(patnums.size, 0.01)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ta, ts = [], []
        for rep in range(args.reps + 2):
            ev[0].record()
            owner, conflict, uncovered = plan.partition_assign(patnums)
            ev[1].record()
            Mq, Uq, t = plan.partition_score(patnums, rates, kM, kU)
            ev[2].record()
            torch.cuda.synchronize()
            assert conflict is None and uncovered is None
            assert int(Mq.sum()) == int(M.sum()) and int(Uq.sum()) == int(U.sum())
            if rep >= 2:
                ta.append(ev[0].elapsed_time(ev[1]))
                ts.append(ev[1].elapsed_time(ev[2]))
        tot = np.array(ta) + np.array(ts)
        gbs = nk * 20 / (np.median(tot) * 1e-3) / 1e9
        print(f"{label}: {patnums.size} patterns, {nk} k-mers: assign {np.median(ta):.3f} ms, score {np.median(ts):.3f} ms, "
              f"together {np.median(tot):.3f} ms (min {tot.min():.3f}); {gbs:.0f} GB/s of owner + counts", flush=True)
        del plan


if __name__ == "__main__":
    main()
