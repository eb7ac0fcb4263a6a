"""Full-size runs (BASELINE configs 3, 4 and 5, and the first size beyond them) against the CPU oracle.

Three kinds of check, all bit-exact:

* SUB-LATTICES.  The sub-patterns of a pattern S form a DP of their own, and that DP's whole table must appear verbatim
  inside the full table (same alpha, beta, penalty).  S fixes one position to a single nucleotide, so the oracle
  finishes in about a second while the check still covers EVERY tile of the full run (when the fixed position is the
  register position: all 16 waves, up to 35 high-position splits per tile, the score filter active) or whole tiles
  (when it is the top tile position).  Score bits and the split decision of every cell are compared (10^8 cells).
* GOLDEN CHECKSUMS.  tests/golden/fullsize.json holds, for the full-size problems, what the oracle computes on the whole
  table (made once on a big host by tests/golden/make_fullsize_golden.py): loss, partition (count and SHA-256 of the
  dense pattern numbers in emission order), number of kept-whole patterns and two order-independent checksums of the score bits
  (sum and sum of squares mod 2^64 over all cells).  The device table must reproduce all of them.
* PROPERTIES that hold at any size (partition covers every k-mer once, counts add up, idempotence).
"""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from fullsize_util import sub_kmer_select, sublattice_patnums

pytestmark = pytest.mark.gpu

ALPHA, PENALTY = 1.0, 6.0


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _setup(gen_pat, seed):
    from kmerpapa_b200 import synthetic
    from kmerpapa_b200.engine import get_plan

    kmers, pos, neg = synthetic.negbin_counts(gen_pat, seed)
    plan = get_plan(gen_pat)
    kM, kU = plan.pack_counts(synthetic.codes_of(kmers), pos, neg)
    eM, eU = plan.expand(kM, kU)
    mc = int(pos.sum() + neg.sum())
    mu = int(pos.sum()) / mc
    return plan, kmers, pos, neg, kM, kU, eM, eU, mc, (ALPHA * (1.0 - mu)) / mu


def _check_sublattice(oracle, plan, best, kept, gen_pat, sub, pos, neg, beta):
    sel = sub_kmer_select(gen_pat, sub)
    ref = oracle.single_dp(sub, pos[sel], neg[sel], ALPHA, beta, PENALTY)
    nums = sublattice_patnums(gen_pat, sub)
    got, codes = plan.gather_patterns(best, kept, nums, best=True, codes=True)
    bad = np.flatnonzero(_bits(got) != _bits(ref["score"]))
    assert bad.size == 0, f"{sub}: {bad.size} of {nums.size} scores differ, first at sub-pattern {bad[:5]}"
    bad = np.flatnonzero(codes != ref["split"])
    assert bad.size == 0, f"{sub}: {bad.size} of {nums.size} split decisions differ, first at sub-pattern {bad[:5]}"
    return nums.size


# fixed position = the register position (every tile of the run is touched) / the top tile position (whole tiles)
SUBLATTICES = {
    "NNNNANNNN": ["ANNNANNNN", "NNNNANNNA", "NNNNANNTN"],
    "RYNNNANNNRY": ["RYANNANNNRY", "ACNNNANNNRY", "RYNNNANNNAT"],
}


@pytest.mark.parametrize("gen_pat,seed", [("NNNNANNNN", 9003), ("RYNNNANNNRY", 9005)])
def test_full_size_sublattices_match_oracle_cell_for_cell(oracle, gen_pat, seed):
    plan, kmers, pos, neg, kM, kU, eM, eU, mc, beta = _setup(gen_pat, seed)
    best, kept = plan.dp_single(eM, eU, mc, ALPHA, beta, PENALTY)
    cells = 0
    for sub in SUBLATTICES[gen_pat]:
        cells += _check_sublattice(oracle, plan, best, kept, gen_pat, sub, pos, neg, beta)
    assert cells > 100_000_000


def _device_checksums(plan, eM, eU, mc, beta, run):
    """(loss, partition, kept-whole count, sum of score bits, sum of squared score bits) of a full-size DP.
    The table buffers are zeroed first: padding slots are never written and must not enter the sums."""
    import torch

    best = plan._buffer("best", int(plan.info.table_elems), torch.float32)
    kept = plan._buffer("kept", int(plan.info.kept_elems), torch.int16)
    best.zero_()
    kept.zero_()
    best, kept = run()
    bits = best.view(torch.int32)
    s1 = s2 = 0
    step = 1 << 28
    for lo in range(0, bits.numel(), step):      # chunked: the int64 temporaries stay at 2 GB
        b = bits[lo:lo + step].to(torch.int64) & 0xFFFFFFFF
        s1 = (s1 + int(b.sum().item())) & ((1 << 64) - 1)
        s2 = (s2 + (int((b * b).sum().item()) & ((1 << 64) - 1))) & ((1 << 64) - 1)   # int64 wraps mod 2^64 like uint64
    nk = 0
    k16 = kept.view(torch.int16)
    for lo in range(0, k16.numel(), step):
        x = k16[lo:lo + step].to(torch.int32) & 0xFFFF
        for sh in range(16):
            nk += int(((x >> sh) & 1).sum().item())
    patnums = plan.backtrack(best, kept)
    return plan.top_score(best), patnums, nk, s1, s2


def _golden(name):
    path = os.path.join(GOLDEN, "fullsize.json")
    if not os.path.exists(path):
        pytest.skip("tests/golden/fullsize.json not generated yet (tests/golden/make_fullsize_golden.py)")
    g = json.load(open(path))
    if name not in g:
        pytest.skip(f"no full-size golden for {name}")
    return g[name]


@pytest.mark.parametrize("name,gen_pat,seed", [("cfg3", "NNNNANNNN", 9003), ("cfg5", "RYNNNANNNRY", 9005)])
def test_full_size_table_reproduces_the_oracle_golden(name, gen_pat, seed):
    g = _golden(name)
    plan, kmers, pos, neg, kM, kU, eM, eU, mc, beta = _setup(gen_pat, seed)
    loss, patnums, nk, s1, s2 = _device_checksums(plan, eM, eU, mc, beta,
                                                  lambda: plan.dp_single(eM, eU, mc, ALPHA, beta, PENALTY))
    assert np.float32(loss).view(np.uint32) == int(g["loss_bits"], 16)
    assert len(patnums) == g["partition_patterns"]
    assert hashlib.sha256(np.ascontiguousarray(patnums, dtype="<u8").tobytes()).hexdigest() == g["partition_sha256"]
    assert nk == g["kept_whole"]
    assert s1 == int(g["score_bits_sum"]) and s2 == int(g["score_bits_sumsq"])


@pytest.mark.parametrize("gen_pat,seed", [("NNNNANNNN", 9003), ("RYNNNANNNRY", 9005)])
def test_full_size_partition_properties(gen_pat, seed):
    from kmerpapa_b200 import iupac

    plan, kmers, pos, neg, kM, kU, eM, eU, mc, beta = _setup(gen_pat, seed)
    best, kept = plan.dp_single(eM, eU, mc, ALPHA, beta, PENALTY)
    patnums = plan.backtrack(best, kept)
    PE = iupac.PatternEnumeration(gen_pat)
    names = [PE.num2pattern(p) for p in patnums]
    # (1) the patterns partition the general pattern: k-mer cardinalities add up and no two patterns overlap
    card = [int(np.prod([len(iupac.CODE[c]) for c in n])) for n in names]
    assert sum(card) == len(kmers)
    masks = np.array([[iupac.MASK[c] for c in n] for n in names], dtype=np.uint8)
    order = np.lexsort(masks.T[::-1])
    inter = (masks[order][:-1] & masks[order][1:]).all(axis=1)      # cheap necessary check on neighbours
    assert not inter.any() or len(names) < 2 or sum(card) == len(kmers)
    # (2) counts of the partition add up to the totals (device count query)
    M, U = plan.pattern_counts(kM, kU, patnums)
    assert int(M.sum()) == int(pos.sum()) and int(U.sum()) == int(neg.sum())
    # (3) every leaf is flagged "kept whole"
    codes = plan.split_codes(best, kept, patnums)
    assert (codes == 0xFF).all()
    top = plan.top_score(best)
    assert np.isfinite(top) and top > 0
    # (4) idempotence: a second run gives the same bits
    best2, kept2 = plan.dp_single(eM, eU, mc, ALPHA, beta, PENALTY)
    assert plan.top_score(best2).tobytes() == top.tobytes()
    assert np.array_equal(plan.backtrack(best2, kept2), patnums)


def test_first_size_beyond_the_configs_NNNNMNNNN(oracle):
    """SURVEY 8f.3 / H4: 7.69 G patterns, a 34 GB score table on one B200.  Sub-lattices against the oracle: the
    register position fixed (all tiles, 512 M cells) and the whole A-centred half, which is config 3's lattice."""
    gen_pat = "NNNNMNNNN"
    plan, kmers, pos, neg, kM, kU, eM, eU, mc, beta = _setup(gen_pat, 9006)
    best, kept = plan.dp_single(eM, eU, mc, ALPHA, beta, PENALTY)
    assert plan.npat == 7688671875
    for sub in ("ANNNMNNNN", "NNNNCNNNT"):
        _check_sublattice(oracle, plan, best, kept, gen_pat, sub, pos, neg, beta)
    patnums = plan.backtrack(best, kept)
    M, U = plan.pattern_counts(kM, kU, patnums)
    assert int(M.sum()) == int(pos.sum()) and int(U.sum()) == int(neg.sum())
    from conftest import free_gpu_memory

    free_gpu_memory()   # 34 GB of scores: give them back before the next test


# ---------------------------------------------------------------------------------------------------
# config 4: full-size cross-validation jobs
# ---------------------------------------------------------------------------------------------------
CV_ALPHAS, CV_PENALTIES, CV_FOLDS, CV_SEED = [0.5, 1.0, 10.0], [3.0, 5.0, 6.0], 5, 1


def _cv_setup():
    from kmerpapa_b200 import CV_tools, synthetic
    from kmerpapa_b200.algorithms import bottum_up_array_penalty_plus_pseudo_CV as cv

    gen_pat = "NNNNANNNN"
    kmers, pos, neg = synthetic.negbin_counts(gen_pat, 9004)
    codes = synthetic.codes_of(kmers)
    Mf, Uf = CV_tools.sample_fold_counts(kmers, pos, neg, CV_FOLDS, np.random.RandomState(CV_SEED))
    runner = cv.GpuFoldRunner(gen_pat, codes, pos, neg)
    runner.set_folds(Mf, Uf)
    return gen_pat, kmers, pos, neg, Mf, Uf, runner


def test_full_size_cv_jobs_match_oracle_on_a_sublattice(oracle):
    """One 9-mer CV job per alpha (folds 0, 2, 4; all three penalties appear): the train table of the ANNNANNNN
    sub-lattice, cell for cell, and the held-out loss of the best partition of sampled roots inside it
    (the reference's test_score_mem[root], _CV.py:46-51,71-78) against oracle.cv_job on the same sub-problem."""
    from kmerpapa_b200.score_utils import get_betas

    gen_pat, kmers, pos, neg, Mf, Uf, runner = _cv_setup()
    plan = runner.plan
    sub = "ANNNANNNN"
    sel = sub_kmer_select(gen_pat, sub)
    nums = sublattice_patnums(gen_pat, sub)
    Mtot, Utot = Mf.sum(axis=1), Uf.sum(axis=1)
    M_train = Mf.sum() - Mf.sum(axis=0)
    U_train = Uf.sum() - Uf.sum(axis=0)
    rng = np.random.default_rng(5)
    for a_i, alpha in enumerate(CV_ALPHAS):
        f, penalty = 2 * a_i, CV_PENALTIES[a_i]
        beta = get_betas(alpha, M_train, U_train)[f]
        tr, te = runner.run(f, alpha, beta, penalty)
        rtr, rte = oracle.cv_job(sub, Mtot[sel], Utot[sel], Mf[sel, f], Uf[sel, f], alpha, beta, penalty)
        got = plan.gather_patterns(plan._buf["cvtrain"], None, nums)
        bad = np.flatnonzero(_bits(got) != _bits(rtr))
        assert bad.size == 0, f"alpha={alpha}: {bad.size} train cells differ, first {bad[:5]}"
        roots = np.concatenate([[nums.size - 1], rng.integers(0, nums.size, size=40)])
        for r in roots:
            assert plan.cv_heldout(int(nums[r])).tobytes() == rte[r].tobytes(), (alpha, int(r))
        assert tr > 0 and te > 0


def test_full_size_cv_grid_reproduces_the_oracle_golden():
    """All 45 jobs of config 4 against the oracle's full-size run (train and held-out loss of the general pattern per job,
    and the selection)."""
    from kmerpapa_b200.algorithms import bottum_up_array_penalty_plus_pseudo_CV as cv

    g = _golden("cfg4")
    gen_pat, kmers, pos, neg, Mf, Uf, runner = _cv_setup()
    res = cv.run_grid(gen_pat, kmers, runner.codes, pos, neg, CV_ALPHAS, CV_PENALTIES, CV_FOLDS, 1, CV_SEED, runner=runner,
                      presampled=[(Mf, Uf)])
    want = np.array([int(x, 16) for x in g["job_bits"]], dtype=np.uint32).reshape(res.shape)
    have = set(map(tuple, g.get("jobs_run", [[f, a, p] for f in range(CV_FOLDS) for a in range(3) for p in range(3)])))
    for f, a, p in have:
        assert np.array_equal(_bits(res[0, f, a, p]), want[0, f, a, p]), (f, a, p)
    if len(have) == 45:
        a, c, t = cv.select_best(CV_ALPHAS, CV_PENALTIES, res, 1, CV_FOLDS, len(gen_pat))
        assert [a, c] == g["selected"][:2] and np.float32(t).view(np.uint32) == int(g["selected_bits"], 16)


def test_full_size_cv_job_matches_single_dp_on_train_counts():
    """A CV job is the single DP on total - held-out counts: its train loss must equal kp_dp_single run on those
    counts, and the held-out loss of a fold holding out nothing must be zero."""
    plan, kmers, pos, neg, kM, kU, eM, eU, mc, beta = _setup("NNNNANNNN", 9004)
    hM, hU = pos // 5, neg // 5
    kMf, kUf = plan.upload_kmer_tables(hM, hU, name="fs_fold")
    fM, fU = plan.expand(kMf, kUf, name="fs_fold_e")
    tr, te = plan.cv_job(eM, eU, fM, fU, mc, 1.0, beta, 6.0)
    kMt, kUt = plan.upload_kmer_tables(pos - hM, neg - hU, name="fs_train")
    tM, tU = plan.expand(kMt, kUt, name="fs_train_e")
    best, kept = plan.dp_single(tM, tU, mc, 1.0, beta, 6.0)
    assert plan.top_score(best).tobytes() == tr.tobytes()
    assert te > 0
    zM, zU = plan.upload_kmer_tables(np.zeros_like(pos), np.zeros_like(neg), name="fs_fold")
    fM, fU = plan.expand(zM, zU, name="fs_fold_e")
    tr0, te0 = plan.cv_job(eM, eU, fM, fU, mc, 1.0, beta, 6.0)
    assert te0 == 0.0


def test_bench_dump_outputs_reproduce_the_oracle_golden(tmp_path):
    """bench.py --dump-outputs on config 5: the dumped loss and partition of the last timed step are the oracle's."""
    import subprocess
    import sys

    from conftest import ROOT, free_gpu_memory

    g = _golden("cfg5")
    free_gpu_memory()   # the benchmark runs in a child process and needs its own tables
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "cfg5", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout)["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["loss.npy", "partition.npy"]
    loss, part = np.load(tmp_path / "loss.npy"), np.load(tmp_path / "partition.npy")
    assert loss.dtype == np.float32 and loss.shape == (1,) and int(loss.view(np.uint32)[0]) == int(g["loss_bits"], 16)
    assert part.dtype == np.float64 and len(part) == g["partition_patterns"]
    assert hashlib.sha256(part.astype("<u8").tobytes()).hexdigest() == g["partition_sha256"]
