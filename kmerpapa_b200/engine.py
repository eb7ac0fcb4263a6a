"""Host-side driver of the CUDA pattern-partition engine.

PyTorch is used for device memory and streams only; every computation goes through the C ABI of
libkpapa.so (include/kmerpapa_b200.h).  One PartitionPlan per (general pattern, device).
"""
import ctypes

import numpy as np

from . import _native
from ._native import KP_ERR_CAPACITY, KpError, check

_PLANS = {}


def _torch():
    import torch

    if not torch.cuda.is_available():
        raise KpError("no CUDA device visible: kmerpapa_b200 runs the DP on the GPU only (no CPU fallback)")
    return torch


class PartitionPlan:
    """Tables, launch geometry and reusable device buffers for one general pattern on one GPU."""

    def __init__(self, gen_pat, device=None, lite=False):
        """lite=True: no tile lattice (k-mer tables only: pack_counts, pattern_counts, the greedy estimator)."""
        torch = _torch()
        self.lite = bool(lite)
        self.lib = _native.lib()
        self.gen_pat = gen_pat
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        h = ctypes.c_void_p()
        create = self.lib.kp_plan_create_lite if self.lite else self.lib.kp_plan_create
        check(create(gen_pat.encode(), self.device_index, ctypes.byref(h)), "kp_plan_create")
        self.handle = h
        info = _native.PlanInfo()
        check(self.lib.kp_plan_get_info(h, ctypes.byref(info)), "kp_plan_get_info")
        self.info = info
        self.npat, self.nkmer = int(info.npat), int(info.nkmer)
        self._buf = {}
        self._cv_state = None
        self.top_elem = None
        if not self.lite:
            off = ctypes.c_uint64()
            check(self.lib.kp_pattern_offset(h, self.npat - 1, ctypes.byref(off), None, None), "kp_pattern_offset")
            self.top_elem = int(off.value)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.kp_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # -- helpers -------------------------------------------------------------------------------
    def _stream(self):
        torch = _torch()
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _buffer(self, name, n, dtype):
        """Reusable device buffer (torch tensor) of at least n elements."""
        torch = _torch()
        t = self._buf.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(int(n), dtype=dtype, device=self.device)
            self._buf[name] = t
        return t

    def release_buffers(self, prefix=None):
        """Drop the cached device buffers (all, or those whose name starts with `prefix`)."""
        if prefix is None:
            self._buf.clear()
        else:
            for name in [n for n in self._buf if n.startswith(prefix)]:
                del self._buf[name]
        if prefix is None or prefix == "cv":
            self._cv_state = None

    def dp_kernel_name(self, wide=False):
        """Name of the kernel family kp_dp_single / kp_dp_cv_job launch for this plan (for reports), for a max_count of
        at most 2^32 - 1 or, with wide=True, above it."""
        return self.lib.kp_dp_kernel_name(self.handle, int(bool(wide))).decode()

    @property
    def launches(self):
        return int(self.lib.kp_plan_launch_count(self.handle))

    # -- K1: k-mer tables ------------------------------------------------------------------------
    def pack_counts(self, codes, pos, neg, name="kmer"):
        """Scatter (code, positive, negative) triples into dense int64 k-mer tables on the device."""
        torch = _torch()
        codes = np.ascontiguousarray(codes, dtype=np.uint64)
        pos = np.ascontiguousarray(pos, dtype=np.int64)
        neg = np.ascontiguousarray(neg, dtype=np.int64)
        if not (codes.shape == pos.shape == neg.shape):
            raise ValueError("codes/pos/neg must have the same length")
        kM = self._buffer(name + "M", self.nkmer, torch.int64)
        kU = self._buffer(name + "U", self.nkmer, torch.int64)
        check(self.lib.kp_pack_counts(self.handle, codes.ctypes.data, pos.ctypes.data, neg.ctypes.data, codes.size,
                                      kM.data_ptr(), kU.data_ptr(), self._stream()), "kp_pack_counts")
        return kM, kU

    def upload_kmer_tables(self, kmerM, kmerU, name="kmer"):
        """Dense k-mer tables already in k-mer index order (used for the per-fold held-out counts)."""
        torch = _torch()
        kM = self._buffer(name + "M", self.nkmer, torch.int64)
        kU = self._buffer(name + "U", self.nkmer, torch.int64)
        hm = torch.from_numpy(np.ascontiguousarray(kmerM, dtype=np.int64))
        hu = torch.from_numpy(np.ascontiguousarray(kmerU, dtype=np.int64))
        kM[: self.nkmer].copy_(hm, non_blocking=False)
        kU[: self.nkmer].copy_(hu, non_blocking=False)
        return kM, kU

    # -- K2: expanded counts ---------------------------------------------------------------------
    def expand(self, kM, kU, name="exp"):
        torch = _torch()
        n = int(self.info.expanded_elems)
        eM = self._buffer(name + "M", n, torch.int64)
        eU = self._buffer(name + "U", n, torch.int64)
        check(self.lib.kp_expand_counts(self.handle, kM.data_ptr(), kU.data_ptr(), eM.data_ptr(), eU.data_ptr(),
                                        self._stream()), "kp_expand_counts")
        return eM, eU

    # -- K3+K4: single DP ------------------------------------------------------------------------
    def dp_single(self, eM, eU, max_count, alpha, beta, penalty):
        """Returns (best, kept): float32 loss table and the uint16 kept-whole bit masks (device layout)."""
        torch = _torch()
        best = self._buffer("best", int(self.info.table_elems), torch.float32)
        kept = self._buffer("kept", int(self.info.kept_elems), torch.int16)
        check(self.lib.kp_dp_single(self.handle, eM.data_ptr(), eU.data_ptr(), int(max_count), float(alpha), float(beta),
                                    float(penalty), best.data_ptr(), kept.data_ptr(), self._stream()), "kp_dp_single")
        return best, kept

    def top_score(self, table):
        """np.float32 value of the general pattern in a device table (one 4-byte device -> host read)."""
        return np.float32(table[self.top_elem].item())

    # -- K5: backtrack ---------------------------------------------------------------------------
    TOP = (1 << 64) - 1
    MAX_CAP = 1 << 26   # largest backtrack workspace (in leaves) the capacity retries grow to

    def backtrack(self, best, kept, cap=65536, root=None):
        """Dense pattern numbers of the optimal partition of `root` (default: the general pattern) in the
        reference's emission order."""
        torch = _torch()
        while True:
            ws = self._buffer("btws", int(self.lib.kp_backtrack_ws_bytes(cap)), torch.uint8)
            out = np.empty(cap, dtype=np.uint64)
            n = ctypes.c_uint64(0)
            rc = self.lib.kp_backtrack(self.handle, best.data_ptr(), kept.data_ptr(), ws.data_ptr(), cap,
                                       self.TOP if root is None else int(root), out.ctypes.data, ctypes.byref(n), self._stream())
            if rc == 0:
                return out[: n.value].copy()
            if rc == KP_ERR_CAPACITY and cap < self.MAX_CAP:
                cap *= 8
                continue
            raise KpError("kp_backtrack: " + self.lib.kp_last_error().decode())

    def split_codes(self, best, kept, patnums):
        """The reference's backtrack pointer as position*8+split codes (0xFF: kept whole)."""
        patnums = np.ascontiguousarray(patnums, dtype=np.uint64)
        out = np.empty(patnums.size, dtype=np.uint8)
        check(self.lib.kp_split_codes(self.handle, best.data_ptr(), kept.data_ptr(), patnums.ctypes.data, patnums.size,
                                      out.ctypes.data, self._stream()), "kp_split_codes")
        return out

    # -- CV job ----------------------------------------------------------------------------------
    def cv_job(self, eMtot, eUtot, eMte, eUte, max_count, alpha, beta, penalty, read_top=True, cap=65536):
        """One fold x alpha x penalty: the DP on the train counts (total - held-out).  Returns
        (np.float32 train, np.float32 held-out) loss of the general pattern; with read_top=False only the
        DP runs and the device tables (train, kept) are returned."""
        torch = _torch()
        n = int(self.info.table_elems)
        train = self._buffer("cvtrain", n, torch.float32)
        kept = self._buffer("cvkept", int(self.info.kept_elems), torch.int16)
        top = (ctypes.c_float * 2)()
        while True:
            ws = self._buffer("btws", int(self.lib.kp_backtrack_ws_bytes(cap)), torch.uint8)
            rc = self.lib.kp_dp_cv_job(self.handle, eMtot.data_ptr(), eUtot.data_ptr(), eMte.data_ptr(), eUte.data_ptr(),
                                       int(max_count), float(alpha), float(beta), float(penalty),
                                       train.data_ptr(), kept.data_ptr(), ws.data_ptr(), cap,
                                       ctypes.cast(top, ctypes.c_void_p) if read_top else None, self._stream())
            if rc == 0:
                break
            if rc == KP_ERR_CAPACITY and cap < self.MAX_CAP:
                cap *= 8
                continue
            raise KpError("kp_dp_cv_job: " + self.lib.kp_last_error().decode())
        self._cv_state = (eMtot, eUtot, eMte, eUte, float(alpha), float(beta), float(penalty))
        if not read_top:
            return train, kept
        return np.float32(top[0]), np.float32(top[1])

    # -- CV jobs without a host round trip ------------------------------------------------------
    CV_SLOTS = 3      # staging areas in rotation (a job's results are read two submissions later)

    def cv_job_submit(self, eMtot, eUtot, eMte, eUte, max_count, alpha, beta, penalty, cap=65536):
        """Queue one CV job (DP, backtrack, leaf losses, copies to pinned host memory) and return a ticket without
        waiting.  The train tables rotate over two buffers and the staging areas over CV_SLOTS, so up to two jobs may be
        outstanding: call cv_job_result on the oldest ticket before submitting a third."""
        torch = _torch()
        seq = getattr(self, "_cv_seq", 0)
        self._cv_seq = seq + 1
        train = self._buffer(f"cvtrain{seq % 2}", int(self.info.table_elems), torch.float32)
        kept = self._buffer(f"cvkept{seq % 2}", int(self.info.kept_elems), torch.int16)
        ws = self._buffer("btws", int(self.lib.kp_backtrack_ws_bytes(cap)), torch.uint8)
        stages = self.__dict__.setdefault("_cv_stage", {})
        key = (seq % self.CV_SLOTS, cap)
        if key not in stages:
            stages[key] = torch.empty(int(self.lib.kp_cv_stage_bytes(cap)), dtype=torch.uint8).pin_memory()
        stage = stages[key]
        check(self.lib.kp_cv_job_enqueue(self.handle, eMtot.data_ptr(), eUtot.data_ptr(), eMte.data_ptr(), eUte.data_ptr(),
                                         int(max_count), float(alpha), float(beta), float(penalty), train.data_ptr(),
                                         kept.data_ptr(), ws.data_ptr(), cap, stage.data_ptr(), self._stream()), "kp_cv_job_enqueue")
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        return (ev, stage, cap, (eMtot, eUtot, eMte, eUte, max_count, alpha, beta, penalty))

    def cv_job_result(self, ticket):
        """(np.float32 train, np.float32 held-out) loss of the general pattern for a submitted job (waits for it)."""
        ev, stage, cap, job = ticket
        ev.synchronize()
        top = (ctypes.c_float * 2)()
        rc = self.lib.kp_cv_job_finish(stage.data_ptr(), cap, ctypes.cast(top, ctypes.c_void_p))
        if rc == KP_ERR_CAPACITY:   # the partition has more leaves than the workspace held: run this job again, synchronously
            return self.cv_job(*job, cap=cap * 8)
        if rc != 0:
            raise KpError("kp_cv_job_finish: " + self.lib.kp_last_error().decode())
        return np.float32(top[0]), np.float32(top[1])

    def cv_heldout(self, root, cap=65536):
        """Held-out loss of the best partition of pattern `root` for the last cv_job (reference: test_score_mem[root])."""
        torch = _torch()
        if self._cv_state is None:
            raise KpError("cv_heldout: no cv_job has run on this plan yet")
        eMtot, eUtot, eMte, eUte, alpha, beta, penalty = self._cv_state
        out = ctypes.c_float(0)
        while True:
            ws = self._buffer("btws", int(self.lib.kp_backtrack_ws_bytes(cap)), torch.uint8)
            rc = self.lib.kp_cv_heldout(self.handle, self._buf["cvtrain"].data_ptr(), self._buf["cvkept"].data_ptr(),
                                        eMtot.data_ptr(), eUtot.data_ptr(), eMte.data_ptr(), eUte.data_ptr(), alpha, beta, penalty,
                                        int(root), ws.data_ptr(), cap, ctypes.byref(out), self._stream())
            if rc == 0:
                return np.float32(out.value)
            if rc == KP_ERR_CAPACITY and cap < self.MAX_CAP:
                cap *= 8
                continue
            raise KpError("kp_cv_heldout: " + self.lib.kp_last_error().decode())

    # -- output stage ----------------------------------------------------------------------------
    def pattern_counts(self, kM, kU, patnums):
        patnums = np.ascontiguousarray(patnums, dtype=np.uint64)
        M = np.empty(patnums.size, dtype=np.int64)
        U = np.empty(patnums.size, dtype=np.int64)
        check(self.lib.kp_pattern_counts(self.handle, kM.data_ptr(), kU.data_ptr(), patnums.ctypes.data, patnums.size,
                                         M.ctypes.data, U.ctypes.data, self._stream()), "kp_pattern_counts")
        return M, U

    # -- scoring a given partition ---------------------------------------------------------------
    def partition_assign(self, patnums, name="part"):
        """Owner of every k-mer for a partition given as dense pattern numbers (file order).  Returns (owner, conflict,
        uncovered): the uint32 owner table (int32 tensor, -1 = none) and the smallest k-mer index covered twice / by no
        pattern, None when there is none (kp_partition_assign)."""
        torch = _torch()
        patnums = np.ascontiguousarray(patnums, dtype=np.uint64)
        owner = self._buffer(name + "_owner", self.nkmer, torch.int32)
        conflict, uncovered = ctypes.c_uint64(0), ctypes.c_uint64(0)
        check(self.lib.kp_partition_assign(self.handle, patnums.ctypes.data, patnums.size, owner.data_ptr(),
                                           ctypes.byref(conflict), ctypes.byref(uncovered), self._stream()),
              "kp_partition_assign")
        return (owner[: self.nkmer], conflict.value - 1 if conflict.value else None,
                uncovered.value - 1 if uncovered.value else None)

    def partition_score(self, patnums, rates, kM, kU, owner=None, name="part"):
        """(M, U, t) per pattern on the k-mer tables kM / kU: int64 counts and the float64 terms
        xlogy(M, p) + xlog1py(U, -p) (kp_partition_score).  With the owner table of partition_assign, also the float64
        rate of every k-mer (device tensor) as a fourth value."""
        torch = _torch()
        patnums = np.ascontiguousarray(patnums, dtype=np.uint64)
        rates = np.ascontiguousarray(rates, dtype=np.float64)
        if rates.shape != patnums.shape:
            raise ValueError("one rate per pattern")
        n = patnums.size
        M, U, t = np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64), np.empty(n, dtype=np.float64)
        kmer_rate = self._buffer(name + "_rate", self.nkmer, torch.float64) if owner is not None else None
        check(self.lib.kp_partition_score(self.handle, patnums.ctypes.data, rates.ctypes.data, n, kM.data_ptr(), kU.data_ptr(),
                                          owner.data_ptr() if owner is not None else None,
                                          kmer_rate.data_ptr() if owner is not None else None,
                                          M.ctypes.data, U.ctypes.data, t.ctypes.data, self._stream()), "kp_partition_score")
        return (M, U, t) if owner is None else (M, U, t, kmer_rate[: self.nkmer])

    # -- applying a partition along sequences (DESIGN §4c) ---------------------------------------
    SEQ_PIECE = 1 << 16   # positions per piece of a record (kp_seq_scan)

    def kmer_rates(self, owner, rates, name="apply"):
        """float64 device tensor: the rate of every k-mer's owner (kp_kmer_rates)."""
        torch = _torch()
        rates = np.ascontiguousarray(rates, dtype=np.float64)
        out = self._buffer(name + "_kmer_rate", self.nkmer, torch.float64)
        check(self.lib.kp_kmer_rates(self.handle, owner.data_ptr(), rates.ctypes.data, rates.size, out.data_ptr(),
                                     self._stream()), "kp_kmer_rates")
        return out[: self.nkmer]

    def seq_scan(self, seq, seq_base, seq_len, rec_len, pos0, pos1, kmer_rate, both, out_sum, out_n, tasks=None,
                 track=None, count_mask=None, counts=None):
        """One kp_seq_scan call on the stream, without waiting.  seq: uint8 device tensor whose first seq_len bytes are
        the record bytes from seq_base on (at least 16 more bytes allocated); out_sum (float64) / out_n (int64): device tensors with one entry per piece of [pos0, pos1), or per
        row of tasks (int32/uint32 device tensor [ntask, 3]); track: float32 device tensor of pos1 - pos0 entries;
        count_mask: int32 device tensor of bits; counts: int64 device tensor [nkmer]."""
        ptr = lambda t: t.data_ptr() if t is not None else None   # noqa: E731
        ntask = 0 if tasks is None else int(tasks.shape[0])
        check(self.lib.kp_seq_scan(self.handle, seq.data_ptr(), int(seq_base), int(seq_len), int(rec_len), int(pos0),
                                   int(pos1), int(bool(both)), kmer_rate.data_ptr(), ptr(tasks), ntask, out_sum.data_ptr(),
                                   out_n.data_ptr(), ptr(track), ptr(count_mask), ptr(counts), self._stream()), "kp_seq_scan")

    def snv_counts(self, seq, seq_base, seq_len, rec_len, pos0, pos1, both, pos, ref_alt, alt_slot, counts, status,
                   count_mask=None):
        """One kp_snv_counts call on the stream, without waiting.  seq, seq_base, seq_len, rec_len, pos0, pos1, both and
        count_mask as in seq_scan; pos: int64 device tensor of record positions in [pos0, pos1); ref_alt: uint8 device
        tensor (REF code | ALT code << 2); alt_slot: 4 ints (-1: not counted); counts: int64 device tensor
        [slots, nkmer]; status: uint8 device tensor with one entry per SNV."""
        n = int(pos.shape[0])
        if ref_alt.shape[0] != n or status.shape[0] != n:
            raise ValueError("pos, ref_alt and status need one entry per SNV")
        if counts.numel() < (max(alt_slot) + 1) * self.nkmer:
            raise ValueError("counts needs nkmer entries for every slot")
        slots = (ctypes.c_int * 4)(*[int(x) for x in alt_slot])
        check(self.lib.kp_snv_counts(self.handle, seq.data_ptr(), int(seq_base), int(seq_len), int(rec_len), int(pos0),
                                     int(pos1), int(bool(both)), pos.data_ptr(), ref_alt.data_ptr(), n, slots,
                                     count_mask.data_ptr() if count_mask is not None else None, counts.data_ptr(),
                                     status.data_ptr(), self._stream()), "kp_snv_counts")

    def region_sums(self, piece_sum, piece_n, task_sum, task_n, regions, out_sum, out_n):
        """kp_region_sums on the stream, without waiting.  regions: int64 device tensor [n, 4]."""
        ptr = lambda t: t.data_ptr() if t is not None else None   # noqa: E731
        check(self.lib.kp_region_sums(self.handle, piece_sum.data_ptr(), piece_n.data_ptr(), ptr(task_sum), ptr(task_n),
                                      regions.data_ptr(), int(regions.shape[0]), out_sum.data_ptr(), out_n.data_ptr(),
                                      self._stream()), "kp_region_sums")

    # -- dense views (tests, exports) ------------------------------------------------------------
    def gather(self, table, first=0, n=None):
        """float32 values of patterns first..first+n-1 (dense numbering) from a device table."""
        n = self.npat - first if n is None else n
        out = np.empty(n, dtype=np.float32)
        check(self.lib.kp_gather_table(self.handle, table.data_ptr(), int(first), int(n), out.ctypes.data, self._stream()),
              "kp_gather_table")
        return out

    def gather_patterns(self, table, kept, patnums, best=True, flags=False, codes=False, chunk=1 << 25):
        """Scores / kept-whole flags / split codes of arbitrary patterns (dense numbers), pulled in chunks.
        Returns the requested arrays in the order (best, flags, codes)."""
        patnums = np.ascontiguousarray(patnums, dtype=np.uint64)
        n = patnums.size
        ob = np.empty(n, dtype=np.float32) if best else None
        of = np.empty(n, dtype=np.uint8) if flags else None
        oc = np.empty(n, dtype=np.uint8) if codes else None
        for lo in range(0, n, chunk):
            m = min(chunk, n - lo)
            check(self.lib.kp_gather_patterns(
                self.handle, table.data_ptr() if table is not None else None, kept.data_ptr() if kept is not None else None,
                patnums[lo:].ctypes.data, m, ob[lo:].ctypes.data if best else None, of[lo:].ctypes.data if flags else None,
                oc[lo:].ctypes.data if codes else None, self._stream()), "kp_gather_patterns")
        out = tuple(x for x in (ob, of, oc) if x is not None)
        return out[0] if len(out) == 1 else out

    def gather_kept(self, kept, first=0, n=None):
        n = self.npat - first if n is None else n
        out = np.empty(n, dtype=np.uint8)
        check(self.lib.kp_gather_kept(self.handle, kept.data_ptr(), int(first), int(n), out.ctypes.data, self._stream()),
              "kp_gather_kept")
        return out


def get_plan(gen_pat, device=None, lite=False):
    """Cached PartitionPlan per (general pattern, device).  lite=True accepts a full plan too (it can do everything a
    lattice-free plan can) and otherwise builds one without the DP's tile lattice."""
    torch = _torch()
    dev = torch.cuda.current_device() if device is None else int(device)
    plan = _PLANS.get((gen_pat, dev, False))
    if plan is None and lite:
        plan = _PLANS.get((gen_pat, dev, True))
    if plan is None:
        plan = PartitionPlan(gen_pat, dev, lite=lite)
        _PLANS[(gen_pat, dev, bool(lite))] = plan
    return plan


def clear_plans():
    _PLANS.clear()
