#!/usr/bin/env python
"""The command line's cross-validation on a full N^9 general pattern (38.4 G patterns: the score table, 169 GB, does not
fit one GPU), under torchrun on >= 2 GPUs: every CV job is one DP sharded over the ranks (ShardedFoldRunner), then the
final fit is sharded the same way.  torchrun --nproc-per-node 2 tools/cli_n9_cv_demo.py
Prints the CV lines, the selected (alpha, penalty), the wall time and the peak device memory of every rank."""
import contextlib
import io
import os
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from kmerpapa_b200 import cli, sharded
from kmerpapa_b200.engine import get_plan

rank = int(os.environ.get("RANK", "0"))
gen_pat = "NNNNNNNNN"
n = 4 ** 9
rng = np.random.default_rng(9009)
bg = 1 + rng.negative_binomial(2, 2 / (2 + 8000.0), size=n)
idx = np.arange(n)
lograte = np.log(1e-3) + sum(rng.normal(0, s, 4)[(idx >> (2 * i)) & 3] for i, s in enumerate([0.03, 0.06, 0.12, 0.25, 0.5, 0.5, 0.25, 0.12, 0.06]))
pos = rng.binomial(bg, np.minimum(0.5, np.exp(lograte)))
letters = "ACGT"
d = os.path.join(tempfile.gettempdir(), f"n9cv_{rank}")
os.makedirs(d, exist_ok=True)
with open(f"{d}/pos.txt", "w") as fp, open(f"{d}/bg.txt", "w") as fb:
    for i in range(n):
        k = "".join(letters[(i >> (2 * j)) & 3] for j in range(9))
        fp.write(f"{k} {pos[i]}\n")
        fb.write(f"{k} {bg[i]}\n")

# peak cudaMalloc bytes of the shards (outside torch's allocator): record the largest shard this rank creates
shard_bytes = [0]
_init = sharded.ShardedDP.__init__


def _recording_init(self, *a, **k):
    _init(self, *a, **k)
    shard_bytes[0] = max(shard_bytes[0], int(self.info.table_elems) * 4 + int(self.info.kept_elems) * 2)


sharded.ShardedDP.__init__ = _recording_init

import torch

t = time.perf_counter()
err = io.StringIO()
with contextlib.redirect_stderr(err):
    rc = cli.main(["-p", f"{d}/pos.txt", "-b", f"{d}/bg.txt", "-c", "6", "8", "10", "-a", "0.5", "1", "--nfolds", "2",
                   "--seed", "1", "-o", f"{d}/out.txt"])
dt = time.perf_counter() - t
peak = torch.cuda.max_memory_allocated()
info = get_plan(gen_pat).info
mine = f"rank {rank}: peak torch {peak / 1e9:.2f} GB + shard {shard_bytes[0] / 1e9:.2f} GB = {(peak + shard_bytes[0]) / 1e9:.2f} GB"
import torch.distributed as dist

lines = [None] * dist.get_world_size() if dist.is_initialized() else [mine]
if dist.is_initialized():
    dist.all_gather_object(lines, mine)
if rank == 0:
    print(err.getvalue().strip())
    print(f"rc={rc}, {dt:.1f} s end to end (parse, plan, sampler, {2 * 3 * 2} sharded CV jobs, sharded final fit, output)")
    print(f"plan: table_elems {info.table_elems} ({info.table_elems * 4 / 1e9:.1f} GB), kept_elems {info.kept_elems}, "
          f"expanded_elems {info.expanded_elems} ({info.expanded_elems * 8 / 1e9:.2f} GB per table)")
    print("\n".join(lines))
    print(open(f"{d}/out.txt").read()[:400])
if dist.is_initialized():
    dist.barrier()
    dist.destroy_process_group()
