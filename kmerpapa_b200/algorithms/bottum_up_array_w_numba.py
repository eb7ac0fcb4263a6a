"""Optimal pattern partition of one data set: the single DP + backtrack, on the GPU.

Drop-in for the reference's src/kmerpapa/algorithms/bottum_up_array_w_numba.py
(`pattern_partition_bottom_up`, :67-124; called from cli.py:279): same name, arguments, return types
and partition order.  The numba array DP is replaced by the CUDA path behind libkpapa.so:
pack k-mer counts (K1) -> expand counts (K2) -> wave-front DP with fused FP64 scoring (K3+K4) ->
device backtrack (K5).
"""
import sys

import numpy as np

from .. import iupac
from ..engine import get_plan


def kmer_arrays(contextD, index_mut=0):
    """contextD {kmer: (n_pos, ..., n_neg)} -> packed codes and int64 count columns."""
    codes = iupac.kmer_codes(contextD.keys())
    vals = list(contextD.values())
    pos = np.array([t[index_mut] for t in vals], dtype=np.int64)
    neg = np.array([t[-1] for t in vals], dtype=np.int64)
    return codes, pos, neg


def count_dtype(nmut, nunmut):
    """The reference keeps counts as uint32 unless the totals need 64 bits (w_numba.py:82-85)."""
    return np.uint64 if nmut + nunmut > np.iinfo(np.uint32).max else np.uint32


def _world():
    try:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized() and dist.get_backend() == "nccl":
            return dist.get_rank(), dist.get_world_size()
    except ImportError:
        pass
    return 0, 1


def dp_buffer_bytes(plan):
    """Device bytes one unsharded DP allocates on top of the k-mer tables: score table, kept-whole masks, the two
    expanded count tables and the backtrack workspace."""
    info = plan.info
    return (int(info.table_elems) * 4 + int(info.kept_elems) * 2 + 2 * int(info.expanded_elems) * 8
            + int(info.backtrack_ws_bytes))


def cv_buffer_bytes(plan, nfolds):
    """Device bytes the unsharded cross-validation (GpuFoldRunner, pipelined jobs) allocates: two train tables and two
    kept-whole masks in rotation, the expanded totals and the expanded held-out tables of every fold, the k-mer tables
    of the totals and of one fold, and the backtrack workspace."""
    info = plan.info
    return (2 * (int(info.table_elems) * 4 + int(info.kept_elems) * 2) + (2 + 2 * int(nfolds)) * int(info.expanded_elems) * 8
            + 4 * int(info.nkmer) * 8 + int(info.backtrack_ws_bytes))


def fits_free_memory(plan, need, held_prefixes):
    """True when `need` bytes fit in what is free on the plan's device right now, counting what the plan already holds in
    the buffers whose names start with one of `held_prefixes` and the backtrack workspace (cached buffers are reused,
    not allocated again)."""
    import torch

    free, _total = torch.cuda.mem_get_info(plan.device)
    held = sum(t.numel() * t.element_size() for name, t in plan._buf.items()
               if name.startswith(tuple(held_prefixes)) or name == "btws")
    reserve = 512 << 20   # allocator slack, CUDA context growth
    return need - held + reserve <= free + _cached_free(plan.device)


def fits_one_gpu(plan):
    """True when the single DP's buffers fit in what is free on the plan's device right now."""
    return fits_free_memory(plan, dp_buffer_bytes(plan), ("best", "kept", "expM", "expU"))


def _cached_free(device):
    """Bytes torch's caching allocator holds but does not use (they count as free for a new torch allocation)."""
    import torch

    return torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)


def _sharded_partition(plan, eM, eU, max_count, alpha, beta, penalty, rank, world):
    """One DP over all ranks of the process group (kmerpapa_b200/sharded.py).  Returns None when the DP fits every rank's
    GPU or this general pattern cannot be sharded over `world` ranks (the ranks agree on both through an all_reduce)."""
    import torch

    from .. import sharded
    from .._native import KpError

    import torch.distributed as dist

    # One decision for all ranks (free memory may differ from GPU to GPU): shard as soon as ONE rank cannot hold the DP.
    fits = torch.tensor([1 if fits_one_gpu(plan) else 0], dtype=torch.int32, device=plan.device)
    dist.all_reduce(fits, op=dist.ReduceOp.MIN)
    if int(fits.item()) == 1:
        # the table fits one GPU: mapping the peers' shards (CUDA IPC, 0.1-0.3 s) costs more than the one DP gains
        # (tools/shard_overhead.py); callers that run many DPs keep a ShardedDP(replicate=True) themselves
        return None
    torch.cuda.empty_cache()   # the shards are plain cudaMalloc allocations (CUDA IPC): give them torch's cached blocks
    try:
        sh = sharded.ShardedDP(plan, rank, world, replicate=False)
    except KpError:
        sh = None
    ok = torch.tensor([0 if sh is None else 1], dtype=torch.int32, device=plan.device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # all ranks shard, or none does
    if int(ok.item()) == 0:
        if sh is not None:
            sh.close()
        return None
    # close() is collective (it must not free a table a peer's kernels still read), so every rank reaches it, also
    # when its own part failed: the error is raised after the shards are released
    res = err = None
    try:
        sh.connect()
        sh.run(eM, eU, max_count, alpha, beta, penalty)
        res = sh.top_score(), sh.backtrack()
    except Exception as e:   # noqa: BLE001 - re-raised below
        err = e
    sh.close()
    if err is not None:
        raise err
    return res


def partition_from_arrays(gen_pat, codes, pos, neg, alpha, beta, penalty, device=None, want_counts=False):
    """Array-level entry (host buffers in, host results out): returns (np.float32 loss,
    dense pattern numbers of the partition in emission order[, (M, U) per pattern]).
    Inside an NCCL process group (torchrun, one process per GPU) a DP whose table does not fit one GPU is sharded over
    the ranks (capacity mode of kmerpapa_b200/sharded.py); every rank gets the result."""
    plan = get_plan(gen_pat, device)
    plan.release_buffers(prefix="cv")   # a cross-validation that ran before the final fit keeps nothing alive
    kM, kU = plan.pack_counts(codes, pos, neg)
    eM, eU = plan.expand(kM, kU)
    max_count = int(pos.sum()) + int(neg.sum())
    rank, world = _world()
    res = _sharded_partition(plan, eM, eU, max_count, alpha, beta, penalty, rank, world) if world > 1 else None
    if res is not None:
        loss, patnums = res
    else:
        best, kept = plan.dp_single(eM, eU, max_count, alpha, beta, penalty)
        patnums = plan.backtrack(best, kept)
        loss = plan.top_score(best)
    if want_counts:
        return loss, patnums, plan.pattern_counts(kM, kU, patnums)
    return loss, patnums


def pattern_partition_bottom_up(gen_pat, contextD, alpha_, beta_, penalty_, args, nmut, nunmut, index_mut=0):
    """Returns (np.float32 loss, M, U, names): loss of the optimal partition of gen_pat, total positive
    and negative counts (numpy unsigned scalars like the reference's M_mem/U_mem entries), and the
    partition's patterns in the reference's backtrack order (c1 subtree first)."""
    gen_pat_level = iupac.pattern_level(gen_pat)
    if getattr(args, "verbosity", 0) > 1:
        for level in range(1, gen_pat_level + 1):
            print(f"level {level} of {gen_pat_level}", file=sys.stderr)
    codes, pos, neg = kmer_arrays(contextD, index_mut)
    loss, patnums = partition_from_arrays(gen_pat, codes, pos, neg, alpha_, beta_, penalty_)
    PE = iupac.PatternEnumeration(gen_pat)
    names = [PE.num2pattern(p) for p in patnums]
    itype = count_dtype(nmut, nunmut)
    return loss, itype(pos.sum()), itype(neg.sum()), names
