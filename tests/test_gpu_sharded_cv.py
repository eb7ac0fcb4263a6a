"""Cross-validation of a sharded DP (ShardedDP.cv_job, ShardedFoldRunner): several shards on ONE GPU in one process run the
sharded CV job, whose train and held-out losses must equal the unsharded CV job (PartitionPlan.cv_job) bit for bit.
The one-process-per-GPU wiring is covered by tests/mgpu_sharded_cv_check.py under torchrun when the box has two GPUs."""
import contextlib
import glob
import io
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")


@pytest.fixture(scope="module")
def oracle():
    from oracle import kp_oracle

    kp_oracle.build()
    return kp_oracle


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _worlds(plan, candidates):
    """The shard counts of `candidates` the plan accepts."""
    from kmerpapa_b200 import sharded
    from kmerpapa_b200._native import KpError

    out = []
    for w in candidates:
        try:
            sharded.assignment(plan, w)
            out.append(w)
        except KpError:
            pass
    return out


@contextlib.contextmanager
def _shards(plan, world, replicate=False):
    from kmerpapa_b200 import sharded

    shards = [sharded.ShardedDP(plan, r, world, replicate=replicate) for r in range(world)]
    try:
        for s in shards:
            s.connect_local(shards)
        yield shards
    finally:
        for s in shards:
            s.close()


def _cv_setup(gen_pat, seed):
    """Synthetic counts, one held-out fold of a 3-fold split; expanded total and held-out tables."""
    from kmerpapa_b200 import CV_tools, synthetic
    from kmerpapa_b200.engine import get_plan
    from kmerpapa_b200.score_utils import get_betas

    kmers, pos, neg = synthetic.negbin_counts(gen_pat, seed)
    Mf, Uf = CV_tools.sample_fold_counts(kmers, pos, neg, 3, np.random.RandomState(seed))
    plan = get_plan(gen_pat, 0)
    codes = synthetic.codes_of(kmers)
    tot = plan.expand(*plan.pack_counts(codes, pos, neg, name="t_tot"), name="t_tot_e")
    fold = plan.expand(*plan.pack_counts(codes, Mf[:, 0], Uf[:, 0], name="t_fold"), name="t_fold_e")
    Ms, Us = Mf.sum(axis=0), Uf.sum(axis=0)
    beta = get_betas(1.0, Ms.sum() - Ms, Us.sum() - Us)[0]
    return plan, tot, fold, int(pos.sum() + neg.sum()), beta


@pytest.mark.parametrize("wide", [False, True])
@pytest.mark.parametrize("replicate", [False, True])
@pytest.mark.parametrize("gen_pat", ["NNNNANN", "NNNNM", "NNNNTNB"])
def test_sharded_cv_job_equals_unsharded(gen_pat, replicate, wide):
    plan, tot, fold, mc, beta = _cv_setup(gen_pat, 21)
    job = (tot[0], tot[1], fold[0], fold[1], 1 << 40 if wide else mc, 1.0, beta, 4.0)
    ref = plan.cv_job(*job)
    ref_table = plan.gather(plan._buf["cvtrain"])
    roots = np.random.default_rng(4).choice(plan.npat, size=40, replace=False)
    ref_roots = [plan.cv_heldout(int(r)) for r in roots]
    ref_train_roots = ref_table[roots]
    worlds = _worlds(plan, (1, 2, 3, 8))
    assert 2 in worlds and 3 in worlds
    for world in worlds:
        with _shards(plan, world, replicate) as shards:
            tr, te = shards[0].cv_job(*job)
            assert (tr.tobytes(), te.tobytes()) == (ref[0].tobytes(), ref[1].tobytes()), (world, tr, te, ref)
            table, _ = shards[-1].gather(np.arange(plan.npat, dtype=np.uint64))
            bad = np.flatnonzero(_bits(table) != _bits(ref_table))
            assert bad.size == 0, f"world {world}: {bad.size} train cells differ, first {bad[:5]}"
            for i, r in enumerate(roots):
                tr, te = shards[0].cv_job(*job, root=int(r))
                assert te.tobytes() == ref_roots[i].tobytes() and tr.tobytes() == ref_train_roots[i].tobytes(), (world, r)
                tr, te = shards[-1].cv_heldout(*job[:4], *job[5:], root=int(r))   # the same tables, read from the last shard
                assert te.tobytes() == ref_roots[i].tobytes() and tr.tobytes() == ref_train_roots[i].tobytes(), (world, r)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "cv_*.npz"))), ids=os.path.basename)
def test_sharded_cv_jobs_against_reference_tables(oracle, path):
    """The recorded reference CV tables (those of test_cv_jobs_against_reference_tables) from a sharded DP."""
    from kmerpapa_b200._native import KpError
    from kmerpapa_b200 import sharded
    from kmerpapa_b200.engine import get_plan

    g = np.load(path)
    gp, nf = str(g["gen_pat"]), int(g["nfolds"])
    plan = get_plan(gp, 0)
    worlds = _worlds(plan, (2, 3))
    try:
        sharded.ShardedDP(plan, 0, 2).close()
    except KpError:
        worlds = []
    if not worlds:   # a pattern that cannot be sharded must say so, not compute something else
        with pytest.raises(KpError):
            sharded.ShardedDP(plan, 0, 2)
        return
    pn = oracle.kmer_patnums(gp).astype(np.int64)
    Mf, Uf = g["M_folds"][pn], g["U_folds"][pn]
    Mtot, Utot = Mf.sum(axis=1), Uf.sum(axis=1)
    Ms, Us = Mf.sum(axis=0), Uf.sum(axis=0)
    Mtr, Utr = Ms.sum() - Ms, Us.sum() - Us
    alphas, pens = [float(a) for a in g["alphas"]], [float(c) for c in g["penalties"]]
    tot = plan.expand(*plan.upload_kmer_tables(Mtot, Utot, name="t_tot"), name="t_tot_e")
    mc = int(Mtot.sum() + Utot.sum())
    folds = [plan.expand(*plan.upload_kmer_tables(Mf[:, f], Uf[:, f], name=f"t_fold{f}"), name=f"t_fold{f}_e") for f in range(nf)]
    ref_te = {}
    for world in worlds:
        with _shards(plan, world) as shards:
            gi = 0
            for alpha in alphas:
                my = Mtr / (Mtr + Utr)
                betas = (alpha * (1.0 - my)) / my
                for pen in pens:
                    for f in range(nf):
                        ref_tr = g["train_tables"][gi][:, f]
                        if (gi, f) not in ref_te:
                            ref_te[gi, f] = (g["last_test_table"][-1, f] if gi == len(alphas) * len(pens) - 1 else
                                             oracle.cv_job(gp, Mtot, Utot, Mf[:, f], Uf[:, f], alpha, betas[f], pen)[1][-1])
                        tr, te = shards[0].cv_job(tot[0], tot[1], folds[f][0], folds[f][1], mc, alpha, betas[f], pen)
                        table, _ = shards[-1].gather(np.arange(plan.npat, dtype=np.uint64))
                        assert np.array_equal(_bits(table), _bits(ref_tr)), (world, gi, f)
                        assert tr.tobytes() == ref_tr[-1].tobytes() and te.tobytes() == ref_te[gi, f].tobytes(), (world, gi, f)
                    gi += 1


def _cfg2_inputs():
    """The inputs of BASELINE config 2 (tests/golden/cli_cfg2_7mers.json), read the way the command line reads them."""
    from kmerpapa_b200 import iupac
    from kmerpapa_b200.algorithms.bottum_up_array_w_numba import kmer_arrays
    from kmerpapa_b200.io_utils import read_postive_and_other

    with open(os.path.join(GOLDEN, "data", "mutated_7mers.txt")) as fp, \
            open(os.path.join(GOLDEN, "data", "background_7mers.txt")) as fb:
        contextD, _, _ = read_postive_and_other(fp, fb, None, n_scale=1, background=True)
    gen_pat = iupac.lca_pattern(list(contextD.keys()))
    for kmer in iupac.matches(gen_pat):
        contextD.setdefault(kmer, (0, 0))
    codes, pos, neg = kmer_arrays(contextD)
    return gen_pat, list(contextD.keys()), codes, pos, neg


@pytest.mark.parametrize("nit", [1, 2])
def test_sharded_cv_grid_equals_unsharded(nit):
    import json

    from kmerpapa_b200.algorithms import bottum_up_array_penalty_plus_pseudo_CV as cv
    from kmerpapa_b200.engine import get_plan

    gen_pat, kmers, codes, pos, neg = _cfg2_inputs()
    alphas, pens, nf, seed = [0.5, 1.0, 10.0], [3.0, 5.0, 6.0], 5, 1
    world = max(_worlds(get_plan(gen_pat, 0), (1, 2, 3)))
    assert world > 1
    runner = cv.ShardedFoldRunner.local(gen_pat, codes, pos, neg, world, device=0)
    try:
        got = cv.run_grid(gen_pat, kmers, codes, pos, neg, alphas, pens, nf, nit, seed, runner=runner)
    finally:
        runner.close()
    ref = cv.run_grid(gen_pat, kmers, codes, pos, neg, alphas, pens, nf, nit, seed,
                      runner=cv.GpuFoldRunner(gen_pat, codes, pos, neg, 0))
    assert got.tobytes() == ref.tobytes()
    if nit == 1:
        out = io.StringIO()
        print("k alpha P LL_test", file=out)
        cv.select_best(alphas, pens, got, nit, nf, len(gen_pat), out)
        assert out.getvalue() == json.load(open(os.path.join(GOLDEN, "cli_cfg2_7mers.json")))["cvfile"]


def test_sharded_cv_errors():
    from kmerpapa_b200 import sharded
    from kmerpapa_b200._native import KpError

    plan, tot, fold, mc, beta = _cv_setup("NNNNANN", 8)
    job = (tot[0], tot[1], fold[0], fold[1], mc, 0.5, beta, 3.0)
    s = sharded.ShardedDP(plan, 0, 2)
    try:
        with pytest.raises(KpError, match="peer"):
            s.cv_job(*job)                       # the peer's shard was never set
    finally:
        s.close()
    ref = plan.cv_job(*job)
    with _shards(plan, 2) as shards:
        tr, te = shards[0].cv_job(*job, cap=1)   # far too small a workspace: grown by the capacity retries
        assert (tr.tobytes(), te.tobytes()) == (ref[0].tobytes(), ref[1].tobytes())


def _torchrun(nproc, port, script, *args, timeout=900, env=None):
    from conftest import free_gpu_memory

    free_gpu_memory()
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
                           "--master-addr", "127.0.0.1", "--master-port", str(port), script, *args],
                          capture_output=True, text=True, timeout=timeout, env=env)


def test_cli_sharded_cv_over_gpus():
    """The command line under torchrun with KP_SHARD_CV=1: every CV job is one DP sharded over the ranks; stdout, CVfile
    and stderr lines must be those of the recorded single-process reference runs."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    r = _torchrun(2, 29617, os.path.join(HERE, "mgpu_sharded_cv_check.py"), env=dict(os.environ, KP_SHARD_CV="1"))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "CLI SHARDED CV OK" in r.stdout


def test_cli_cv_on_a_table_larger_than_one_gpu():
    """tools/cli_n9_cv_demo.py: a CV grid on the full N^9 pattern (169 GB of scores) over two GPUs."""
    import torch

    if torch.cuda.device_count() < 2 or torch.cuda.get_device_properties(0).total_memory < 120e9:
        pytest.skip("needs two GPUs with at least 120 GB each")
    r = _torchrun(2, 29618, os.path.join(ROOT, "tools", "cli_n9_cv_demo.py"), timeout=1800)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-6000:]
    assert "rc=0" in r.stdout and "General pattern: NNNNNNNNN" in r.stdout and "CV DONE." in r.stdout
