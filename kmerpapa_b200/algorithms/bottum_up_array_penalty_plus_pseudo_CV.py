"""Cross-validation grid over (pseudo-count alpha, penalty): one GPU DP per fold x alpha x penalty.

Drop-in for the reference's src/kmerpapa/algorithms/bottum_up_array_penalty_plus_pseudo_CV.py
(`pattern_partition_bottom_up`, :81-177; called from cli.py:232): same name, arguments, return
values, CVfile rows and stderr lines.

What changed underneath: the reference carries all folds on the last axis of one numba DP; folds never
interact inside that DP (_CV.py:46-51, :63-78), so here a job is one (iteration, fold, alpha, penalty)
and runs as an independent single-fold DP on the GPU (kp_dp_cv_job), with train counts formed on the
device as total - held-out.  Jobs are dealt to the ranks of torch.distributed (one process per GPU)
in contiguous fold-major chunks and the per-job (train, held-out) losses of the general pattern are
all-gathered (NCCL on GPUs); every rank then does the reference's float32 fold sum and selection.
A general pattern whose CV tables do not fit one GPU is cross-validated with every job as one DP sharded over all
ranks instead (ShardedFoldRunner, chosen by sharded_cv_runner).
"""
import sys

import numpy as np

from .. import CV_tools, iupac
from ..score_utils import get_betas
from .bottum_up_array_w_numba import count_dtype, kmer_arrays


# ---------------------------------------------------------------------------------------------
# job sharding (pure host logic; exercised on CPU with gloo in tests/)
# ---------------------------------------------------------------------------------------------
def job_list(nit, nfolds, n_alpha, n_penalty):
    """All jobs, fold-major so that a contiguous chunk touches as few folds as possible."""
    return [(it, f, a_i, p_i) for it in range(nit) for f in range(nfolds) for a_i in range(n_alpha)
            for p_i in range(n_penalty)]


def shard_bounds(njobs, rank, world):
    """Contiguous chunk [lo, hi) of rank; chunks differ by at most one job."""
    base, extra = divmod(njobs, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def dist_info():
    try:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except ImportError:
        pass
    return 0, 1


def gather_job_results(local, njobs, rank, world, device=None):
    """local: float32 [hi-lo, 2] results of this rank's chunk -> float32 [njobs, 2] on every rank.
    One all_gather of equally padded chunks (NCCL when the tensors live on a GPU, gloo on CPU)."""
    if world == 1:
        return local
    import torch
    import torch.distributed as dist

    chunk = -(-njobs // world)
    pad = np.zeros((chunk, 2), dtype=np.float32)
    pad[: local.shape[0]] = local
    t = torch.from_numpy(pad)
    if device is not None:
        t = t.to(device)
    out = torch.empty((world * chunk, 2), dtype=torch.float32, device=t.device)
    dist.all_gather_into_tensor(out, t)
    out = out.cpu().numpy().reshape(world, chunk, 2)
    full = np.empty((njobs, 2), dtype=np.float32)
    for r in range(world):
        lo, hi = shard_bounds(njobs, r, world)
        full[lo:hi] = out[r, : hi - lo]
    return full


# ---------------------------------------------------------------------------------------------
# host-side reduction and selection (reference :165-177)
# ---------------------------------------------------------------------------------------------
def fold_sum(values, nit):
    """Python sum() over np.float32 values then / nit: sequential float32 accumulation (SURVEY H8)."""
    return sum(list(values)) / nit


def select_best(alphas, penalties, results, nit, nfolds, k, cvfile=None):
    """results: float32 [nit, nfolds, n_alpha, n_penalty, 2].  Writes one CVfile row per grid point and
    returns (alpha, penalty, test) of the first strict minimum, alpha outer / penalty inner."""
    best_test_loss = 1e100
    best_values = (None, None)
    for a_i, alpha in enumerate(alphas):
        for p_i, penalty in enumerate(penalties):
            vals = [results[it, f, a_i, p_i, 1] for it in range(nit) for f in range(nfolds)]
            test = fold_sum(vals, nit)
            if cvfile is not None:
                print(k, alpha, penalty, test, file=cvfile)
            with np.errstate(over="ignore"):   # float32 test against the 1e100 start value, as in the reference
                better = test < best_test_loss
            if better:
                best_values = (alpha, penalty)
                best_test_loss = test
    return best_values[0], best_values[1], best_test_loss


def covering_patterns_per_kmer(gen_pat):
    """Number of sub-patterns of gen_pat that contain a given k-mer (8 per N, 4 per 3-letter, 2 per 2-letter)."""
    c = 1
    for ch in gen_pat:
        c *= 1 << (len(iupac.CODE[ch]) - 1)
    return c


class GpuFoldRunner:
    """Runs single-fold DP jobs of one CV iteration on this process's GPU."""

    def __init__(self, gen_pat, codes, pos, neg, device=None):
        from ..engine import get_plan

        self.plan = get_plan(gen_pat, device)
        self.codes = codes
        self.max_count = int(pos.sum()) + int(neg.sum())
        kM, kU = self.plan.pack_counts(codes, pos, neg, name="cvtot_k")
        self.tot = self.plan.expand(kM, kU, name="cvtot_e")
        self.folds = {}
        self.pending = []

    def set_folds(self, Mf, Uf):
        self.Mf, self.Uf = Mf, Uf
        self.folds = {}

    def begin_folds(self, nkmer, nfolds):
        """Folds arrive one at a time (set_fold) while earlier folds' jobs already run."""
        self.Mf = np.zeros((nkmer, nfolds), dtype=np.uint64)
        self.Uf = np.zeros((nkmer, nfolds), dtype=np.uint64)
        self.folds = {}

    def set_fold(self, f, M, U):
        self.Mf[:, f], self.Uf[:, f] = M, U

    def _fold(self, f):
        if f not in self.folds:
            kM, kU = self.plan.pack_counts(self.codes, self.Mf[:, f], self.Uf[:, f], name="cvfold_k")
            self.folds[f] = self.plan.expand(kM, kU, name=f"cvfold{f}_e")
        return self.folds[f]

    def run(self, f, alpha, beta, penalty):
        eMte, eUte = self._fold(f)
        return self.plan.cv_job(self.tot[0], self.tot[1], eMte, eUte, self.max_count, alpha, beta, penalty)

    # pipelined interface: the next job's DP is queued before the previous job's results are read back, so the GPU
    # does not idle during the host round trip (backtrack results, float32 tree sum) of every job
    DEPTH = 2

    def submit(self, tag, f, alpha, beta, penalty):
        """Queue a job; returns the (tag, train, held-out) results that became due (oldest first)."""
        eMte, eUte = self._fold(f)
        self.pending.append((tag, self.plan.cv_job_submit(self.tot[0], self.tot[1], eMte, eUte, self.max_count, alpha, beta,
                                                          penalty)))
        out = []
        while len(self.pending) >= self.DEPTH:
            out.append(self._pop())
        return out

    def flush(self):
        out = []
        while self.pending:
            out.append(self._pop())
        return out

    def _pop(self):
        tag, ticket = self.pending.pop(0)
        tr, te = self.plan.cv_job_result(ticket)
        return tag, tr, te

    @property
    def device(self):
        return self.plan.device


class ShardedFoldRunner:
    """GpuFoldRunner's run / begin_folds / set_fold / set_folds over ONE capacity-mode DP sharded over several shards, for a
    general pattern whose CV tables do not fit one GPU: every job is a sharded CV job (ShardedDP.cv_job).  It is a
    collective runner: every rank runs every job, so run_grid neither deals the jobs to the ranks nor gathers them.
    It keeps the expanded held-out tables of one fold only (the jobs are fold-major: each fold is expanded once) and has
    no pipelined interface.  `shards`: this process's connected shards, either one per rank of the NCCL group (connect())
    or all shards of the DP in this process (connect_local(), see local())."""

    collective = True

    def __init__(self, shards, codes, pos, neg):
        self.shards = list(shards)
        self.plan = self.shards[0].plan
        self.codes = codes
        self.max_count = int(pos.sum()) + int(neg.sum())
        kM, kU = self.plan.pack_counts(codes, pos, neg, name="cvtot_k")
        self.tot = self.plan.expand(kM, kU, name="cvtot_e")
        self.fold = None   # (f, expanded M, expanded U) of the resident fold

    @classmethod
    def local(cls, gen_pat, codes, pos, neg, world, device=None):
        """`world` in-process shards on one GPU (the sharded CV without a process group)."""
        from .. import sharded
        from ..engine import get_plan

        plan = get_plan(gen_pat, device)
        shards = []
        try:
            for r in range(world):
                shards.append(sharded.ShardedDP(plan, r, world, replicate=False))
            for s in shards:
                s.connect_local(shards)
            return cls(shards, codes, pos, neg)
        except BaseException:
            for s in shards:
                s.close()
            raise

    def set_folds(self, Mf, Uf):
        self.Mf, self.Uf = Mf, Uf
        self.fold = None

    def begin_folds(self, nkmer, nfolds):
        self.Mf = np.zeros((nkmer, nfolds), dtype=np.uint64)
        self.Uf = np.zeros((nkmer, nfolds), dtype=np.uint64)
        self.fold = None

    def set_fold(self, f, M, U):
        self.Mf[:, f], self.Uf[:, f] = M, U

    def run(self, f, alpha, beta, penalty):
        if self.fold is None or self.fold[0] != f:
            err = None
            try:
                kM, kU = self.plan.pack_counts(self.codes, self.Mf[:, f], self.Uf[:, f], name="cvfold_k")
                self.fold = (f,) + self.plan.expand(kM, kU, name="cvfold_e")
            except Exception as e:   # noqa: BLE001 - raised on every rank by agree()
                err = e
            self.shards[0].agree(err, "ShardedFoldRunner: held-out tables")
        return self.shards[0].cv_job(self.tot[0], self.tot[1], self.fold[1], self.fold[2], self.max_count, alpha, beta,
                                     penalty)

    def close(self):
        """Release the shards (collective with peers in other processes: every rank calls it) and the CV buffers."""
        self.fold = self.tot = None
        for s in self.shards:
            s.close()
        self.shards = []
        self.plan.release_buffers(prefix="cv")

    @property
    def device(self):
        return self.plan.device


def sharded_cv_runner(gen_pat, codes, pos, neg, nfolds):
    """A ShardedFoldRunner over the ranks of the NCCL group when the CV tables GpuFoldRunner would allocate do not fit
    one rank's GPU (or KP_SHARD_CV=1 asks for it) and every rank can hold its shard; else None: the jobs are dealt to
    the ranks as usual.  The ranks agree on every decision through an all_reduce."""
    import os

    from .bottum_up_array_w_numba import _world, cv_buffer_bytes, fits_free_memory

    rank, world = _world()
    if world == 1:
        return None
    import torch
    import torch.distributed as dist

    from .. import sharded
    from .._native import KpError
    from ..engine import get_plan

    plan = get_plan(gen_pat)
    forced = os.environ.get("KP_SHARD_CV") == "1"
    fits = torch.tensor([0 if forced else int(fits_free_memory(plan, cv_buffer_bytes(plan, nfolds), ("cv",)))],
                        dtype=torch.int32, device=plan.device)
    dist.all_reduce(fits, op=dist.ReduceOp.MIN)   # shard as soon as ONE rank cannot hold the CV
    if int(fits.item()) == 1:
        return None
    torch.cuda.empty_cache()   # the shards are plain cudaMalloc allocations (CUDA IPC): give them torch's cached blocks
    try:
        sh = sharded.ShardedDP(plan, rank, world, replicate=False)
    except KpError:
        sh = None
    ok = torch.tensor([0 if sh is None else 1], dtype=torch.int32, device=plan.device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)     # all ranks shard, or none does
    if int(ok.item()) == 0:
        if sh is not None:
            sh.close()
        return None
    runner = err = None
    try:
        sh.connect()   # raises on every rank when one rank cannot map its peers
        try:
            runner = ShardedFoldRunner([sh], codes, pos, neg)
        except Exception as e:   # noqa: BLE001 - e.g. no memory left for the count tables on this rank; raised by agree()
            err = e
        sh.agree(err, "ShardedFoldRunner")
    except BaseException:
        sh.close()     # collective: every rank is here
        raise
    return runner


def run_grid(gen_pat, kmers, codes, pos, neg, alphas, penalties, nfolds, nit, seed, verbosity=0, runner=None,
             gather_device="auto", presampled=None, progress=None):
    """Core of the CV: returns float32 results [nit, nfolds, n_alpha, n_penalty, 2] (train, held-out).
    presampled: optional list (one per iteration) of (Mf, Uf) held-out tables to use instead of sampling.
    progress(it, results_of_iteration): called once per iteration, in order — right after the iteration's jobs in
    a single process (the reference's interleaving of its stderr lines), after the gather when the jobs are sharded."""
    rank, world = dist_info()
    if getattr(runner, "collective", False):   # every rank runs every job (one DP over all ranks): nothing to deal or gather
        rank, world = 0, 1
    prng = np.random.RandomState(seed)
    if runner is None:
        runner = GpuFoldRunner(gen_pat, codes, pos, neg)
    if gather_device == "auto":
        gather_device = getattr(runner, "device", None)
    na, npen = len(alphas), len(penalties)
    jobs = job_list(nit, nfolds, na, npen)
    lo, hi = shard_bounds(len(jobs), rank, world)
    local = np.zeros((hi - lo, 2), dtype=np.float32)
    cover = covering_patterns_per_kmer(gen_pat)
    prev_M = prev_U = None
    pipelined = hasattr(runner, "submit")

    def run_job(slot, f, alpha, beta, penalty):
        if pipelined:   # results arrive a job or two later; the GPU already has the next DP queued by then
            for tag, tr, te in runner.submit(slot, f, alpha, beta, penalty):
                local[tag, 0], local[tag, 1] = tr, te
        else:
            local[slot, 0], local[slot, 1] = runner.run(f, alpha, beta, penalty)

    def drain():
        if pipelined:
            for tag, tr, te in runner.flush():
                local[tag, 0], local[tag, 1] = tr, te

    for it in range(nit):
        if verbosity > 0 and nit > 1:
            print("CV Iteration", it, file=sys.stderr)
        jlo, jhi = max(lo, it * nfolds * na * npen), min(hi, (it + 1) * nfolds * na * npen)
        if presampled is None and hasattr(runner, "set_fold"):
            # The host sampler (numpy's legacy RandomState, about 0.3 s per fold for 9-mers) runs on a thread, one
            # fold ahead of the GPU: the jobs are fold-major and fold f is final once drawn.  A fold's beta needs the
            # fold's own totals and the grand totals only, and the latter are known beforehand (H7 quirk included).
            import queue
            import threading

            q = queue.Queue()

            def produce(prng=prng):
                try:
                    for item in CV_tools.iter_fold_counts(kmers, pos, neg, nfolds, prng):
                        q.put(item)
                except BaseException as e:   # surface sampler errors in the consumer
                    q.put(e)

            th = threading.Thread(target=produce, daemon=True)
            th.start()
            M_tot, U_tot = np.uint64(int(np.sum(pos))), np.uint64(int(np.sum(neg)))
            if prev_M is not None:
                M_tot = M_tot + np.uint64(cover - 1) * prev_M.sum()
                U_tot = U_tot + np.uint64(cover - 1) * prev_U.sum()
            runner.begin_folds(len(kmers), nfolds)
            cur_M, cur_U = np.zeros(nfolds, dtype=np.uint64), np.zeros(nfolds, dtype=np.uint64)
            j = jlo
            for _ in range(nfolds):
                item = q.get()
                if isinstance(item, BaseException):
                    raise item
                f, M, U = item
                runner.set_fold(f, M, U)
                cur_M[f], cur_U[f] = M.sum(), U.sum()
                mt, ut = cur_M[f], cur_U[f]
                if prev_M is not None:
                    mt, ut = mt + np.uint64(cover - 1) * prev_M[f], ut + np.uint64(cover - 1) * prev_U[f]
                Mtr, Utr = np.array([M_tot - mt]), np.array([U_tot - ut])
                while j < jhi and jobs[j][1] == f:
                    _, _, a_i, p_i = jobs[j]
                    beta = get_betas(alphas[a_i], Mtr, Utr)[0]
                    run_job(j - lo, f, alphas[a_i], beta, penalties[p_i])
                    j += 1
            drain()
            th.join()
            prev_M, prev_U = cur_M, cur_U
            if verbosity > 0:
                print("CV sampling DONE", file=sys.stderr)
            if progress is not None and world == 1:
                progress(it, local.reshape(nit, nfolds, na, npen, 2)[it])
            continue
        if presampled is not None:
            Mf, Uf = presampled[it]
        else:
            Mf, Uf = CV_tools.sample_fold_counts(kmers, pos, neg, nfolds, prng)
        if verbosity > 0:
            print("CV sampling DONE", file=sys.stderr)
        # per-fold held-out totals.  The reference sums ALL rows of its np.empty tables (_CV.py:134-135):
        # zero pages on the first iteration, the previous iteration's upper-level rows afterwards (SURVEY H7).
        M_sum_test = Mf.sum(axis=0)
        U_sum_test = Uf.sum(axis=0)
        if prev_M is not None:
            M_sum_test = M_sum_test + np.uint64(cover - 1) * prev_M
            U_sum_test = U_sum_test + np.uint64(cover - 1) * prev_U
        prev_M, prev_U = Mf.sum(axis=0), Uf.sum(axis=0)
        M_sum_train = M_sum_test.sum() - M_sum_test
        U_sum_train = U_sum_test.sum() - U_sum_test
        betas = [get_betas(alpha, M_sum_train, U_sum_train) for alpha in alphas]
        runner.set_folds(Mf, Uf)
        for j in range(jlo, jhi):
            _, f, a_i, p_i = jobs[j]
            run_job(j - lo, f, alphas[a_i], betas[a_i][f], penalties[p_i])
        drain()
        if progress is not None and world == 1:
            progress(it, local.reshape(nit, nfolds, na, npen, 2)[it])
    full = gather_job_results(local, len(jobs), rank, world, gather_device).reshape(nit, nfolds, na, npen, 2)
    if progress is not None and world > 1:
        for it in range(nit):
            progress(it, full[it])
    return full


def pattern_partition_bottom_up(gen_pat, contextD, alphas, args, nmut, nunmut, penalties, index_mut=0):
    """Returns (best_alpha, best_penalty, np.float32 best_test_loss); writes the CVfile rows
    `k alpha penalty test` and the reference's progress lines on stderr."""
    nf, nit = args.nfolds, args.iterations
    kmers = list(contextD.keys())
    codes, pos, neg = kmer_arrays(contextD, index_mut)
    verbosity = getattr(args, "verbosity", 0)
    rank, _ = dist_info()
    gen_pat_level = iupac.pattern_level(gen_pat)

    def progress(it, res_it):   # the reference's per-grid-point lines (_CV.py:157-160)
        if verbosity > 0 and rank == 0:
            for a_i, alpha in enumerate(alphas):
                for p_i, penalty in enumerate(penalties):
                    row = res_it[:, a_i, p_i, 1]
                    if verbosity > 1:   # the reference reports every level of every grid point's DP (_CV.py:154-155)
                        for level in range(1, gen_pat_level + 1):
                            print(f"level {level} of {gen_pat_level}", file=sys.stderr)
                    print(f"CV on k={len(gen_pat)} alpha={alpha} penalty={penalty} i={it} test_LL={sum(row)}", file=sys.stderr)
                    if verbosity > 1:
                        print(f"test LL for each fold: {row}", file=sys.stderr)

    runner = sharded_cv_runner(gen_pat, codes, pos, neg, nf)   # None: the jobs are dealt to the ranks (or one GPU runs them)
    try:
        results = run_grid(gen_pat, kmers, codes, pos, neg, alphas, penalties, nf, nit, args.seed, verbosity, runner=runner,
                           progress=progress)
    finally:
        if runner is not None:   # collective: every rank gets here, also when the grid raised (on all ranks alike)
            runner.close()
    cvfile = args.CVfile if rank == 0 else None
    return select_best(alphas, penalties, results, nit, nf, len(gen_pat), cvfile)
