"""One pattern-partition DP sharded over the GPUs of a node (SURVEY 8f.3).

The score table is split by the digit of the top high position of the tile lattice; every rank runs the same
waves on its own tiles and the DP kernel reads the children that live on a peer straight from the peer's memory
over NVLink (C ABI: kp_shard_* in include/kmerpapa_b200.h).  Two ways to connect the shards:

* one process per GPU (torchrun): `ShardedDP(plan, rank, world).connect(group)` exchanges CUDA IPC handles with
  `torch.distributed.all_gather_object`; the wave barrier is an `all_reduce` on the current stream;
* several shards in one process (tests; any number of shards on one GPU): `connect_local(shards)`.

The reference has no counterpart: its tables are single numpy arrays (bottum_up_array_w_numba.py:82-91), which is
why `N^9` (38 G patterns, 770 GB in its layout) is out of its reach.
"""
import ctypes

import numpy as np

from . import _native
from ._native import KpError, check
from .engine import _torch, grow_capacity


def assignment(plan, world):
    """(owner, slot) of every digit of the top high position for `world` ranks (host logic, no GPU work)."""
    owner = np.zeros(16, dtype=np.uint8)
    slot = np.zeros(16, dtype=np.uint8)
    check(plan.lib.kp_shard_assignment(plan.handle, int(world), owner.ctypes.data, slot.ctypes.data), "kp_shard_assignment")
    return owner, slot


class ShardedDP:
    """This rank's shard of one DP.  `plan` is the PartitionPlan of the general pattern on this rank's device."""

    def __init__(self, plan, rank, world, replicate=False):
        """replicate=False (capacity mode): a rank stores its own tiles only, the kernel loads peer children over
        NVLink.  replicate=True (speed mode): every rank holds a full-size table and the kernel pushes finished
        rows to the peers that will read them, so every read is local."""
        self.plan, self.lib = plan, plan.lib
        self.rank, self.world = int(rank), int(world)
        h = ctypes.c_void_p()
        check(self.lib.kp_shard_create(plan.handle, self.rank, self.world, 1 if replicate else 0, ctypes.byref(h)),
              "kp_shard_create")
        self.handle = h
        info = _native.ShardInfo()
        check(self.lib.kp_shard_get_info(h, ctypes.byref(info)), "kp_shard_get_info")
        self.info = info
        self.nwaves = int(info.nwaves)
        self._opened = []
        self._group = None
        self._token = None
        self._local = None

    def close_peers(self):
        """Unmap the peers' shards (CUDA IPC).  Local only; see close()."""
        for ptr in self._opened:
            self.lib.kp_ipc_close(self.plan.device_index, ctypes.c_void_p(ptr))
        self._opened = []

    def close(self):
        """Release the shard.  With peers in other processes (connect()), this is a COLLECTIVE: every rank must call
        it.  A peer's kernels (backtrack, gather) may still be reading this rank's exported tables, and
        freeing an allocation that another process has mapped is undefined, so the order is: drain this rank's stream,
        wait for everyone, unmap the peers' tables, wait again, and only then free what this rank exported."""
        if not getattr(self, "handle", None):
            return
        collective = self._token is not None
        if collective:
            import torch.distributed as dist

            _torch().cuda.synchronize(self.plan.device)
            dist.barrier(group=self._group)
        self.close_peers()
        if collective:
            import torch.distributed as dist

            dist.barrier(group=self._group)
            self._token = None
        self._local = None
        self.lib.kp_shard_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:   # no collective from a finaliser: unmap, then free (callers that share shards across processes call close())
            if getattr(self, "handle", None):
                self.close_peers()
                self.lib.kp_shard_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # -- wiring --------------------------------------------------------------------------------------
    def connect_local(self, shards):
        """All shards live in this process (possibly on one GPU): hand each other the raw device pointers.  cv_job on
        any of them then runs the waves of all of them, in lock-step on one stream."""
        self._local = list(shards)
        for other in shards:
            if other.rank != self.rank:
                check(self.lib.kp_shard_set_peer(self.handle, other.rank, ctypes.c_void_p(other.info.d_best),
                                                 ctypes.c_void_p(other.info.d_kept)), "kp_shard_set_peer")

    def connect(self, group=None):
        """One process per GPU: exchange CUDA IPC handles of the shards over torch.distributed."""
        import torch.distributed as dist

        torch = _torch()
        # collective from here on (close() included), and every rank learns whether all ranks succeeded (agree())
        self._group = group
        self._token = torch.zeros(1, dtype=torch.int32, device=self.plan.device)
        hb, hk = (ctypes.c_uint8 * 64)(), (ctypes.c_uint8 * 64)()
        err = None
        try:
            check(self.lib.kp_ipc_export(ctypes.c_void_p(self.info.d_best), hb), "kp_ipc_export")
            check(self.lib.kp_ipc_export(ctypes.c_void_p(self.info.d_kept), hk), "kp_ipc_export")
        except KpError as e:
            err = e
        self.agree(err, "kp_ipc_export")
        mine = (self.rank, bytes(hb), bytes(hk))
        everyone = [None] * self.world
        dist.all_gather_object(everyone, mine, group=group)
        try:
            for r, b, k in everyone:
                if r == self.rank:
                    continue
                pb, pk = ctypes.c_void_p(), ctypes.c_void_p()
                check(self.lib.kp_ipc_open(self.plan.device_index, (ctypes.c_uint8 * 64).from_buffer_copy(b),
                                           ctypes.byref(pb)), "kp_ipc_open")
                self._opened.append(pb.value)
                check(self.lib.kp_ipc_open(self.plan.device_index, (ctypes.c_uint8 * 64).from_buffer_copy(k),
                                           ctypes.byref(pk)), "kp_ipc_open")
                self._opened.append(pk.value)
                check(self.lib.kp_shard_set_peer(self.handle, r, pb, pk), "kp_shard_set_peer")
        except KpError as e:
            err = e
        self.agree(err, "ShardedDP.connect")

    def barrier(self):
        """All ranks have finished the work they queued on their current streams (one tiny NCCL all_reduce)."""
        if self._token is not None:
            import torch.distributed as dist

            dist.all_reduce(self._token, group=self._group)

    def agree(self, err, what):
        """Barrier that also tells every rank whether all ranks succeeded (MIN all_reduce of a success flag, read back).
        err: this rank's exception or None.  Raises on every rank as soon as one rank failed, so that no rank is left
        waiting in a collective the failed rank will never join."""
        if self._token is not None:
            import torch.distributed as dist

            self._token.fill_(0 if err is not None else 1)
            dist.all_reduce(self._token, op=dist.ReduceOp.MIN, group=self._group)
            if int(self._token.item()) == 0 and err is None:
                err = KpError(f"{what}: failed on another rank")
        if err is not None:
            raise err

    # -- the DP ----------------------------------------------------------------------------------------
    def wave(self, w, eM, eU, max_count, alpha, beta, penalty):
        check(self.lib.kp_shard_dp_wave(self.handle, int(w), eM.data_ptr(), eU.data_ptr(), int(max_count), float(alpha),
                                        float(beta), float(penalty), self.plan._stream()), "kp_shard_dp_wave")

    def run(self, eM, eU, max_count, alpha, beta, penalty):
        """All waves of this rank with a barrier between them (one process per GPU)."""
        for w in range(self.nwaves):
            self.wave(w, eM, eU, max_count, alpha, beta, penalty)
            self.barrier()

    # -- cross-validation jobs -------------------------------------------------------------------------
    def cv_wave(self, w, eMtot, eUtot, eMte, eUte, max_count, alpha, beta, penalty):
        check(self.lib.kp_shard_cv_wave(self.handle, int(w), eMtot.data_ptr(), eUtot.data_ptr(), eMte.data_ptr(),
                                        eUte.data_ptr(), int(max_count), float(alpha), float(beta), float(penalty),
                                        self.plan._stream()), "kp_shard_cv_wave")

    def cv_job(self, eMtot, eUtot, eMte, eUte, max_count, alpha, beta, penalty, root=None, cap=65536):
        """One fold x alpha x penalty on the train counts total - held-out (PartitionPlan.cv_job over the shards): every
        wave, then (np.float32 train loss, np.float32 held-out loss) of `root` (default: the general pattern).  With
        in-process shards (connect_local) the waves of all of them run here, in lock-step on one stream; with one
        process per rank (connect) every rank calls this with the same arguments and the ranks meet after every wave."""
        job = (eMtot, eUtot, eMte, eUte, max_count, alpha, beta, penalty)
        if self._local is not None:
            for w in range(self.nwaves):
                for s in self._local:
                    s.cv_wave(w, *job)
        else:
            for w in range(self.nwaves):
                err = None
                try:
                    self.cv_wave(w, *job)
                except KpError as e:
                    err = e
                self.agree(err, f"kp_shard_cv_wave {w}")
        err = res = None
        try:
            res = self.cv_heldout(eMtot, eUtot, eMte, eUte, alpha, beta, penalty, root, cap)
        except KpError as e:
            err = e
        self.agree(err, "kp_shard_cv_heldout")   # no rank starts the next job's waves while a peer may still read its tables
        return res

    def cv_heldout(self, eMtot, eUtot, eMte, eUte, alpha, beta, penalty, root=None, cap=65536):
        """(train, held-out) loss of `root` after the last wave of a CV job (this rank only, reads the peers' tables)."""
        torch = _torch()
        top = (ctypes.c_float * 2)()

        def run(cap):
            ws = self.plan._buffer("btws", int(self.lib.kp_backtrack_ws_bytes(cap)), torch.uint8)
            return self.lib.kp_shard_cv_heldout(self.handle, eMtot.data_ptr(), eUtot.data_ptr(), eMte.data_ptr(),
                                                eUte.data_ptr(), float(alpha), float(beta), float(penalty),
                                                self.plan.TOP if root is None else int(root), ws.data_ptr(), cap,
                                                ctypes.cast(top, ctypes.c_void_p), self.plan._stream()), None

        grow_capacity(self.lib, "kp_shard_cv_heldout", cap, self.plan.MAX_CAP, run)
        return np.float32(top[0]), np.float32(top[1])

    def backtrack(self, cap=65536, root=None):
        torch = _torch()

        def run(cap):
            ws = self.plan._buffer("btws", int(self.lib.kp_backtrack_ws_bytes(cap)), torch.uint8)
            out = np.empty(cap, dtype=np.uint64)
            n = ctypes.c_uint64(0)
            rc = self.lib.kp_shard_backtrack(self.handle, ws.data_ptr(), cap, self.plan.TOP if root is None else int(root),
                                             out.ctypes.data, ctypes.byref(n), self.plan._stream())
            return rc, out[: n.value]

        return grow_capacity(self.lib, "kp_shard_backtrack", cap, self.plan.MAX_CAP, run).copy()

    def gather(self, patnums, codes=False):
        """(scores, kept-whole flags[, split codes]) of arbitrary patterns, wherever they are stored."""
        patnums = np.ascontiguousarray(patnums, dtype=np.uint64)
        best = np.empty(patnums.size, dtype=np.float32)
        kept = np.empty(patnums.size, dtype=np.uint8)
        cds = np.empty(patnums.size, dtype=np.uint8) if codes else None
        check(self.lib.kp_shard_gather(self.handle, patnums.ctypes.data, patnums.size, best.ctypes.data, kept.ctypes.data,
                                       cds.ctypes.data if codes else None, self.plan._stream()), "kp_shard_gather")
        return (best, kept, cds) if codes else (best, kept)

    def top_score(self):
        return self.gather(np.array([self.plan.npat - 1], dtype=np.uint64))[0][0]


def run_local(shards, eM, eU, max_count, alpha, beta, penalty):
    """Lock-step execution of several shards that live in this process (one stream: wave w of every shard is
    queued before wave w+1 of any)."""
    for w in range(shards[0].nwaves):
        for s in shards:
            s.wave(w, eM, eU, max_count, alpha, beta, penalty)
