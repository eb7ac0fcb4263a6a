"""Sharded single DP (SURVEY 8f.3): several shards on ONE GPU in one process exercise the sharded kernel variant,
the owner/slot addressing and the cross-shard backtrack; results must equal the unsharded DP bit for bit.
The one-process-per-GPU wiring (CUDA IPC + NCCL barrier) is covered by tests/mgpu_sharded_check.py under torchrun
(test_sharded_multiprocess below runs it when the box has at least two GPUs)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _setup(gen_pat, seed):
    from kmerpapa_b200 import synthetic
    from kmerpapa_b200.engine import get_plan

    kmers, pos, neg = synthetic.negbin_counts(gen_pat, seed)
    plan = get_plan(gen_pat, 0)
    kM, kU = plan.pack_counts(synthetic.codes_of(kmers), pos, neg)
    eM, eU = plan.expand(kM, kU)
    mc = int(pos.sum() + neg.sum())
    mu = int(pos.sum()) / mc
    return plan, eM, eU, mc, 1.0 * (1 - mu) / mu


@pytest.mark.parametrize("replicate", [False, True])
@pytest.mark.parametrize("gen_pat,world", [("NNNNANN", 1), ("NNNNANN", 2), ("NNNNANN", 3), ("NNNNANN", 8),
                                           ("NNNNM", 2), ("NNNNM", 3), ("NNNNTNB", 4)])
def test_sharded_equals_unsharded(gen_pat, world, replicate):
    import torch

    from kmerpapa_b200 import sharded

    plan, eM, eU, mc, beta = _setup(gen_pat, 77)
    alpha, penalty = 1.0, 4.0
    best, kept = plan.dp_single(eM, eU, mc, alpha, beta, penalty)
    ref_part = plan.backtrack(best, kept)
    assert np.array_equal(plan.backtrack(best, kept, cap=1), ref_part)   # through the capacity retry
    rng = np.random.default_rng(5)
    pats = np.unique(np.concatenate([rng.integers(0, plan.npat, size=20000, dtype=np.uint64),
                                     np.array([0, plan.npat - 1], dtype=np.uint64), ref_part]))
    ref_codes = plan.split_codes(best, kept, pats)
    ref_vals = np.array([plan.gather(best, int(p), 1)[0] for p in pats[:50]], dtype=np.float32)
    top = plan.top_score(best)

    shards = [sharded.ShardedDP(plan, r, world, replicate=replicate) for r in range(world)]
    try:
        owner, slot = sharded.assignment(plan, world)
        assert sum(s.info.local_tiles for s in shards) == plan.info.ntiles * (world if replicate else 1)
        cells = [s.info.top_digits for s in shards]   # digits of the top position (or, replicated: (top, second) cells) owned
        assert max(cells) - min(cells) <= (1 if not replicate else max(2, max(cells) // 4))
        for s in shards:
            s.connect_local(shards)
        sharded.run_local(shards, eM, eU, mc, alpha, beta, penalty)
        torch.cuda.synchronize()
        for s in (shards[0], shards[-1]):          # any rank can read everything
            assert s.top_score() == top
            part = s.backtrack()
            assert np.array_equal(part, ref_part)
            assert np.array_equal(s.backtrack(cap=1), ref_part)
            vals, flags, codes = s.gather(pats, codes=True)
            assert np.array_equal(codes, ref_codes)
            assert np.array_equal(vals[:50], ref_vals)
            assert np.array_equal(flags == 1, ref_codes == 0xFF)
    finally:
        for s in shards:
            s.close()


def test_shard_errors():
    from kmerpapa_b200 import sharded
    from kmerpapa_b200._native import KpError
    from kmerpapa_b200.engine import get_plan

    with pytest.raises(KpError):
        sharded.ShardedDP(get_plan("NNN", 0), 0, 2)       # no high position: nothing to shard
    with pytest.raises(KpError):
        sharded.ShardedDP(get_plan("NNNNM", 0), 0, 4)     # top position has 3 digits
    with pytest.raises(KpError):
        sharded.ShardedDP(get_plan("NNNNANN", 0), 2, 2)   # rank out of range
    s = sharded.ShardedDP(get_plan("NNNNANN", 0), 0, 2)
    try:
        plan, eM, eU, mc, beta = _setup("NNNNANN", 3)
        with pytest.raises(KpError):
            s.wave(0, eM, eU, mc, 1.0, beta, 3.0)         # peer not connected
    finally:
        s.close()


def test_sharded_multiprocess():
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    world = 2 if n < 4 else 4
    from conftest import free_gpu_memory

    free_gpu_memory()
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29611", os.path.join(here, "mgpu_sharded_check.py"),
                        "NNNNANNN"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "SHARDED OK" in r.stdout


def test_cli_on_a_table_larger_than_one_gpu():
    """The command line under torchrun on the full N^9 pattern (169 GB of scores): the final fit is sharded over the
    ranks by itself; the CLI's own assertions check the counts of the partition against the input totals."""
    import torch

    if torch.cuda.device_count() < 2 or torch.cuda.get_device_properties(0).total_memory < 120e9:
        pytest.skip("needs two GPUs with at least 120 GB each")
    from conftest import free_gpu_memory

    free_gpu_memory()   # the children need (almost) all of both GPUs
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29613", os.path.join(root, "tools", "cli_n9_demo.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-6000:]
    assert "rc=0" in r.stdout and "General pattern: NNNNNNNNN" in r.stdout and "loss=" in r.stdout

