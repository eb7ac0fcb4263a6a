"""run_grid with a collective runner (one that runs every job on every rank, like the sharded CV runner) over
torch.distributed with the gloo backend, world size 2, on CPU: every rank runs every job itself, nothing is dealt or
all-gathered, every rank returns the single-process result and reports its progress in the single-process order."""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GEN_PAT, ALPHAS, PENS, NF, SEED, NIT = "NNN", [0.5, 2.0], [2.0, 5.0, 7.0], 3, 4, 2


@pytest.fixture(scope="module")
def built_oracle():
    sys.path.insert(0, ROOT)
    from oracle import kp_oracle

    kp_oracle.build()
    return kp_oracle


def _data():
    rng = np.random.default_rng(3)
    U = 1 + rng.negative_binomial(2, 2 / (2 + 900.0), size=64)
    M = rng.binomial(U, 0.03)
    return M.astype(np.int64), U.astype(np.int64)


class CollectiveOracleRunner:
    """The sharded runner's interface (set_folds / begin_folds / set_fold / run, no submit) on top of the CPU oracle."""

    collective = True
    device = None

    def __init__(self, gen_pat, M, U):
        from oracle import kp_oracle

        self.O, self.gp, self.M, self.U = kp_oracle, gen_pat, M, U
        self.calls = 0

    def set_folds(self, Mf, Uf):
        self.Mf, self.Uf = Mf, Uf

    def begin_folds(self, nkmer, nfolds):
        self.Mf = np.zeros((nkmer, nfolds), dtype=np.uint64)
        self.Uf = np.zeros((nkmer, nfolds), dtype=np.uint64)

    def set_fold(self, f, M, U):
        self.Mf[:, f], self.Uf[:, f] = M, U

    def run(self, f, alpha, beta, penalty):
        self.calls += 1
        tr, te = self.O.cv_job(self.gp, self.M, self.U, self.Mf[:, f], self.Uf[:, f], alpha, beta, penalty, nthreads=1)
        return tr[-1], te[-1]


def _grid():
    from kmerpapa_b200 import iupac
    from kmerpapa_b200.algorithms import bottum_up_array_penalty_plus_pseudo_CV as cv

    M, U = _data()
    runner = CollectiveOracleRunner(GEN_PAT, M, U)
    events = []

    def progress(it, res_it):
        events.append((it, runner.calls, res_it.tobytes()))

    res = cv.run_grid(GEN_PAT, iupac.matches(GEN_PAT), None, M, U, ALPHAS, PENS, NF, NIT, SEED, runner=runner,
                      gather_device=None, progress=progress)
    return res, runner.calls, events


def _worker(rank, world, port, q):
    import torch.distributed as dist

    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from kmerpapa_b200.algorithms import bottum_up_array_penalty_plus_pseudo_CV as cv

    gather = cv.gather_job_results

    def no_gather(local, njobs, rank, world, device=None):
        assert world == 1, "a collective runner's results must not be gathered"
        return gather(local, njobs, rank, world, device)

    cv.gather_job_results = no_gather
    res, calls, events = _grid()
    q.put((rank, res.tobytes(), calls, events))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_collective_runner_runs_every_job_on_every_rank(built_oracle):
    single, calls, events = _grid()
    njobs = NIT * NF * len(ALPHAS) * len(PENS)
    assert calls == njobs
    # progress after each iteration's own jobs, as in one process
    assert [(it, c) for it, c, _ in events] == [(it, (it + 1) * njobs // NIT) for it in range(NIT)]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=240) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(r for r, *_ in got) == [0, 1]
    for rank, blob, c, ev in got:
        assert blob == single.tobytes()   # the full, identical result on every rank
        assert c == njobs                 # every job ran on this rank
        assert ev == events               # and the progress came in the single-process order
