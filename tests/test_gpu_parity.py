"""GPU parity tests: the CUDA path (through the C ABI) against the reference's golden tables and the
CPU oracle.  Bit-exact everywhere: float32 score tables, split decisions, partitions, counts, CV losses.
"""
import ctypes

import numpy as np
import pytest

from conftest import GOLDEN, golden_files

pytestmark = pytest.mark.gpu


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


@pytest.fixture(scope="module")
def eng():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kmerpapa_b200 import engine

    return engine


def _codes(gen_pat):
    from kmerpapa_b200 import iupac

    return np.array([iupac.kmer_code(k) for k in iupac.matches(gen_pat)], dtype=np.uint64)


def _run_single(eng, gen_pat, M, U, alpha, beta, penalty, max_count=None):
    plan = eng.get_plan(gen_pat)
    kM, kU = plan.pack_counts(_codes(gen_pat), M, U)
    eM, eU = plan.expand(kM, kU)
    mc = int(np.sum(M, dtype=np.uint64) + np.sum(U, dtype=np.uint64)) if max_count is None else max_count
    best, kept = plan.dp_single(eM, eU, mc, alpha, beta, penalty)
    split = plan.split_codes(best, kept, np.arange(plan.npat, dtype=np.uint64))   # the reference's backtrack pointer, as a code
    assert np.array_equal(plan.gather_kept(kept) == 1, split == 0xFF)
    return plan, plan.gather(best), split, plan.backtrack(best, kept)


def test_device_log_is_glibc_log(eng, oracle):
    from kmerpapa_b200 import _native

    rng = np.random.default_rng(5)
    n = 1_000_000
    xs = np.concatenate([
        rng.random(n), 1.0 - rng.random(n) * 0.07, 1.0 + (rng.random(n) - 0.5) * 0.2,
        np.exp(rng.uniform(-700, 700, n)), rng.random(n) * 1e-300,
        np.abs(rng.integers(0, 2**63 - 1, n, dtype=np.int64).view(np.float64)),
        np.array([0.0, 1.0, np.inf, 5e-324, 2.2250738585072014e-308, 0.9375, 1.064697265625, -1.0, np.nan]),
    ])
    xs = np.ascontiguousarray(xs)
    y = np.empty_like(xs)
    _native.check(_native.lib().kp_debug_log(0, xs.ctypes.data, y.ctypes.data, xs.size), "kp_debug_log")
    ref = np.empty_like(xs)
    oracle.lib().kpo_log_array(xs.ctypes.data, ref.ctypes.data, xs.size)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(y), nan)
    assert np.array_equal(_bits(y[~nan]), _bits(ref[~nan]))


def test_device_leaf_score_is_scipy(eng):
    import scipy.special as sp

    from kmerpapa_b200 import _native

    rng = np.random.default_rng(6)
    n = 300_000
    U = rng.integers(0, 5_000_000, n)
    M = rng.binomial(U, rng.random(n) * 0.6)
    M[:1000] = 0
    U[500:1500] = 0
    alpha, beta, pen = 0.8, 1234.5, 5.0
    out = np.empty(n, dtype=np.float64)
    M64, U64 = M.astype(np.int64), U.astype(np.int64)
    _native.check(_native.lib().kp_debug_leaf_score(0, M64.ctypes.data, U64.ctypes.data, n, alpha, beta, pen,
                                                    out.ctypes.data), "kp_debug_leaf_score")
    p = (M64 + alpha) / (M64 + U64 + alpha + beta)
    ref = -2 * (sp.xlogy(M64, p) + sp.xlog1py(U64, -p)) + pen
    assert np.array_equal(_bits(out), _bits(ref))


@pytest.mark.parametrize("path", golden_files("single"), ids=lambda p: p.split("single_")[-1][:-4])
def test_single_dp_against_reference_tables(eng, oracle, path):
    g = np.load(path)
    gp = str(g["gen_pat"])
    plan, best, split, patnums = _run_single(eng, gp, g["kmerM"], g["kmerU"], float(g["alpha"]), float(g["beta"]),
                                             float(g["penalty"]))
    assert np.array_equal(_bits(best), _bits(g["score"]))
    kept = g["bt"] == np.arange(len(g["bt"]), dtype=np.uint64)
    assert np.array_equal(split == 0xFF, kept)
    from kmerpapa_b200 import iupac

    PE = iupac.PatternEnumeration(gp)
    assert [PE.num2pattern(p) for p in patnums] == [str(x) for x in g["names"]]
    # split codes decode to the reference's c1 pointer
    ref = oracle.single_dp(gp, g["kmerM"], g["kmerU"], float(g["alpha"]), float(g["beta"]), float(g["penalty"]))
    assert np.array_equal(split, ref["split"])
    # counts of the partition's patterns straight from the device k-mer tables
    M, U = plan.pattern_counts(plan._buf["kmerM"], plan._buf["kmerU"], patnums)
    assert np.array_equal(M.astype(np.uint64), g["M"][patnums.astype(np.int64)])
    assert np.array_equal(U.astype(np.uint64), g["U"][patnums.astype(np.int64)])


@pytest.mark.parametrize("path", golden_files("single"), ids=lambda p: p.split("single_")[-1][:-4])
def test_single_dp_wide_counts_path(eng, path):
    """Same data through the 64-bit on-chip count path (selected by max_count)."""
    g = np.load(path)
    gp = str(g["gen_pat"])
    _, best, split, _ = _run_single(eng, gp, g["kmerM"], g["kmerU"], float(g["alpha"]), float(g["beta"]),
                                    float(g["penalty"]), max_count=1 << 40)
    assert np.array_equal(_bits(best), _bits(g["score"]))


@pytest.mark.parametrize("path", golden_files("cv"), ids=lambda p: p.split("cv_")[-1][:-4])
def test_cv_jobs_against_reference_tables(eng, oracle, path):
    g = np.load(path)
    gp, nf = str(g["gen_pat"]), int(g["nfolds"])
    pn = oracle.kmer_patnums(gp).astype(np.int64)
    Mf, Uf = g["M_folds"][pn], g["U_folds"][pn]            # held-out counts per k-mer and fold
    Mtot, Utot = Mf.sum(axis=1), Uf.sum(axis=1)
    Ms, Us = Mf.sum(axis=0), Uf.sum(axis=0)
    Mtr, Utr = Ms.sum() - Ms, Us.sum() - Us
    alphas, pens = [float(a) for a in g["alphas"]], [float(c) for c in g["penalties"]]
    plan = eng.get_plan(gp)
    kM, kU = plan.upload_kmer_tables(Mtot, Utot, name="t_tot")
    tot = plan.expand(kM, kU, name="t_tot_e")
    mc = int(Mtot.sum() + Utot.sum())
    gi = 0
    for a_i, alpha in enumerate(alphas):
        my = Mtr / (Mtr + Utr)
        betas = (alpha * (1.0 - my)) / my
        for p_i, pen in enumerate(pens):
            for f in range(nf):
                kMf, kUf = plan.upload_kmer_tables(Mf[:, f], Uf[:, f], name="t_fold")
                fold = plan.expand(kMf, kUf, name="t_fold_e")
                ref_tr = g["train_tables"][gi][:, f]
                if gi == len(alphas) * len(pens) - 1:
                    ref_te = g["last_test_table"][:, f]
                else:
                    _, ref_te = oracle.cv_job(gp, Mtot, Utot, Mf[:, f], Uf[:, f], alpha, betas[f], pen)
                for wide_mc in (mc, 1 << 40):
                    top = plan.cv_job(tot[0], tot[1], fold[0], fold[1], wide_mc, alpha, betas[f], pen)
                    # train table: every cell; held-out loss: the general pattern (all the reference reads) ...
                    assert np.array_equal(_bits(plan.gather(plan._buf["cvtrain"])), _bits(ref_tr))
                    assert top[0].tobytes() == ref_tr[-1].tobytes() and top[1].tobytes() == ref_te[-1].tobytes()
                # ... and a spread of other patterns, against the reference's whole test table
                rng = np.random.default_rng(gi * 31 + f)
                for root in rng.choice(plan.npat, size=min(40, plan.npat), replace=False):
                    assert plan.cv_heldout(int(root)).tobytes() == ref_te[root].tobytes()
            gi += 1


@pytest.mark.parametrize("gen_pat,seed", [("NNNNN", 1), ("NNNMNN", 2), ("RYNNANNKM", 3), ("VNNNH", 4), ("NNNNNN", 5),
                                          ("SWNNBNA", 6), ("MMMMMMMMMM", 7), ("RYNNNANRY", 8), ("BBDHVVB", 9),
                                          ("KNSNWNMN", 10), ("N", 11), ("ACGT", 12), ("RA", 13), ("NB", 14)])
def test_random_against_oracle(eng, oracle, gen_pat, seed):
    """Larger general patterns (several tile waves, mixed radices) against the CPU oracle."""
    rng = np.random.default_rng(seed)
    _, nk, _ = oracle.plan_info(gen_pat)
    U = (1 + rng.negative_binomial(2, 2 / (2 + 800.0), size=nk)) * (rng.random(nk) < 0.9)
    M = rng.binomial(U, np.minimum(0.5, 0.02 * np.exp(rng.normal(0, 0.8, size=nk))))
    U[0], M[0] = max(U[0], 50), max(M[0], 2)      # never an all-zero table (beta would be NaN)
    alpha, pen = 1.0, 4.0
    mu = M.sum() / (M.sum() + U.sum())
    beta = alpha * (1 - mu) / mu
    _, best, split, patnums = _run_single(eng, gen_pat, M, U, alpha, beta, pen)
    ref = oracle.single_dp(gen_pat, M, U, alpha, beta, pen)
    assert np.array_equal(_bits(best), _bits(ref["score"]))
    assert np.array_equal(split, ref["split"])
    assert np.array_equal(patnums, oracle.backtrack(gen_pat, ref["split"]))


@pytest.mark.parametrize("regime", ["rate_near_one", "half", "tiny_counts", "huge_counts", "zeros", "penalty_ties", "low_rates",
                                    "kept_whole", "negative_penalty"])
@pytest.mark.parametrize("gen_pat", ["NNNNN", "NNMNNN", "NNNNNN"])
def test_count_regimes_against_oracle(eng, oracle, gen_pat, regime):
    """Regimes that stress the score filter (a float32 bound decides whether the exact FP64 score is computed): rates
    near 1 (absolute error of the fast log), rates around 1/2, counts of a few units, counts near 2^31, mostly empty
    tables, penalties that make many self-scores tie with split sums, and negative penalties (the filter's estimate
    pen + t1 + t2 then cancels).  Full table + split codes vs the oracle."""
    import zlib

    rng = np.random.default_rng(zlib.crc32((gen_pat + regime).encode()))
    _, nk, _ = oracle.plan_info(gen_pat)
    if regime == "rate_near_one":
        M = rng.integers(10 ** 5, 10 ** 6, size=nk)
        U = rng.integers(0, 30, size=nk) * (rng.random(nk) < 0.5)
    elif regime == "half":
        U = rng.integers(10 ** 4, 10 ** 5, size=nk)
        M = rng.binomial(2 * U, 0.5)
    elif regime == "tiny_counts":
        U = rng.integers(0, 4, size=nk)
        M = rng.integers(0, 3, size=nk)
    elif regime == "huge_counts":
        hi = (2 ** 31 - 10 ** 6) // nk
        U = rng.integers(min(10 ** 6, hi // 2), hi, size=nk)
        M = rng.binomial(U, 0.001)
    elif regime == "zeros":
        keep = rng.random(nk) < 0.02
        U = rng.integers(1, 5000, size=nk) * keep
        M = rng.binomial(U, 0.05)
    elif regime == "low_rates":     # the fast score path (kp_self_score_fast): rates on both sides of its 2^-8 switch, up to 2^-4
        U = rng.integers(10 ** 4, 10 ** 6, size=nk)
        M = rng.binomial(U, np.exp(rng.uniform(np.log(1e-6), np.log(0.07), size=nk)))
    elif regime in ("kept_whole", "negative_penalty"):   # kept_whole: a penalty so large that every pattern is kept whole
        U = 1 + rng.negative_binomial(2, 2 / (2 + 33000.0), size=nk)
        M = rng.binomial(U, np.minimum(0.5, 1e-3 * np.exp(rng.normal(0, 0.7, size=nk))))
    else:
        U = np.full(nk, 1000)
        M = np.full(nk, 10)
    U[0], M[0] = max(U[0], 5), max(M[0], 1)
    grid = {"penalty_ties": ((1.0, 0.0), (1.0, 2.0)), "kept_whole": ((1.0, 1e6), (0.01, 3e3)),
            "negative_penalty": ((1.0, -0.5), (10.0, -3.0))}.get(regime, ((1.0, 4.0), (0.5, 0.0)))
    for alpha, pen in grid:
        mu = M.sum() / (M.sum() + U.sum())
        beta = alpha * (1 - mu) / mu
        _, best, split, patnums = _run_single(eng, gen_pat, M, U, alpha, beta, pen)
        ref = oracle.single_dp(gen_pat, M, U, alpha, beta, pen)
        assert np.array_equal(_bits(best), _bits(ref["score"]))
        assert np.array_equal(split, ref["split"])
        assert np.array_equal(patnums, oracle.backtrack(gen_pat, ref["split"]))


@pytest.mark.parametrize("gen_pat,seed", [("NNNNN", 21), ("RYNNANNKM", 22), ("VNNNH", 23), ("MMMMMMMMMM", 24),
                                          ("RYNNNANRY", 25), ("BBDHVVB", 26), ("N", 27), ("ACGT", 28), ("NNNSNN", 29),
                                          ("NNNNNN", 30)])
def test_random_cv_job_against_oracle(eng, oracle, gen_pat, seed):
    """One held-out fold on larger / oddly shaped general patterns: train and held-out tables, both widths.  Seed 30: a
    negative penalty."""
    rng = np.random.default_rng(seed)
    _, nk, _ = oracle.plan_info(gen_pat)
    U = (1 + rng.negative_binomial(2, 2 / (2 + 800.0), size=nk)) * (rng.random(nk) < 0.9)
    M = rng.binomial(U, np.minimum(0.5, 0.02 * np.exp(rng.normal(0, 0.8, size=nk))))
    if seed % 2:                      # provoke ties: few distinct values
        U = rng.choice([0, 40, 80, 800], size=nk)
        M = np.minimum(U, rng.choice([0, 1, 2, 4], size=nk))
        M[0], U[0] = 3, 50
    Mte, Ute = rng.binomial(M, 0.3), rng.binomial(U, 0.3)
    alpha, pen = (1.0, 3.0) if seed < 30 else (1.0, -2.0)
    mu = (M.sum() - Mte.sum()) / ((M.sum() - Mte.sum()) + (U.sum() - Ute.sum()))
    beta = alpha * (1 - mu) / mu
    plan = eng.get_plan(gen_pat)
    kM, kU = plan.upload_kmer_tables(M, U, name="r_tot")
    tot = plan.expand(kM, kU, name="r_tot_e")
    kMf, kUf = plan.upload_kmer_tables(Mte, Ute, name="r_fold")
    fold = plan.expand(kMf, kUf, name="r_fold_e")
    otr, ote = oracle.cv_job(gen_pat, M, U, Mte, Ute, alpha, beta, pen)
    for mc in (int(M.sum() + U.sum()), 1 << 40):
        top = plan.cv_job(tot[0], tot[1], fold[0], fold[1], mc, alpha, beta, pen)
        assert np.array_equal(_bits(plan.gather(plan._buf["cvtrain"])), _bits(otr))
        assert top[0].tobytes() == otr[-1].tobytes() and top[1].tobytes() == ote[-1].tobytes()
    rng2 = np.random.default_rng(seed + 100)
    for root in rng2.choice(plan.npat, size=min(60, plan.npat), replace=False):
        assert plan.cv_heldout(int(root)).tobytes() == ote[root].tobytes()


def test_7mer_test_data_final_dp(eng, oracle):
    """BASELINE config 2's final DP (test_data 7-mers, alpha=10, penalty=6): 34 171 875 patterns."""
    from kmerpapa_b200 import iupac

    gp = "NNNMNNN"
    kmers = iupac.matches(gp)
    pos, bg = {}, {}
    for line in open(f"{GOLDEN}/data/mutated_7mers.txt"):
        k, c = line.split()
        pos[k] = int(c)
    for line in open(f"{GOLDEN}/data/background_7mers.txt"):
        k, c = line.split()
        bg[k] = int(c)
    M = np.array([pos.get(k, 0) for k in kmers], dtype=np.int64)
    U = np.array([bg.get(k, 0) for k in kmers], dtype=np.int64) - M
    alpha = 10.0
    mu = int(M.sum()) / (int(M.sum()) + int(U.sum()))
    beta = (alpha * (1.0 - mu)) / mu
    _, best, split, patnums = _run_single(eng, gp, M, U, alpha, beta, 6.0)
    ref = oracle.single_dp(gp, M, U, alpha, beta, 6.0)
    assert np.array_equal(_bits(best), _bits(ref["score"]))
    assert np.array_equal(split, ref["split"])
    PE = iupac.PatternEnumeration(gp)
    names = [PE.num2pattern(p) for p in patnums]
    assert len(names) == 270 and names[0] == "RCAATNT"       # recorded from the reference CLI (SURVEY 8c)
    assert float(best[-1]) == 1324533.625


def test_pack_counts_sums_duplicates_and_rejects_bad_codes(eng):
    from kmerpapa_b200 import iupac
    from kmerpapa_b200._native import KpError

    gp = "NAN"
    plan = eng.get_plan(gp)
    kmers = iupac.matches(gp)
    codes = np.array([iupac.kmer_code(k) for k in kmers] + [iupac.kmer_code("CAG")], dtype=np.uint64)
    pos = np.arange(len(codes), dtype=np.int64)
    neg = 10 * np.arange(len(codes), dtype=np.int64)
    kM, kU = plan.pack_counts(codes, pos, neg)
    hM = kM[: plan.nkmer].cpu().numpy()
    idx = kmers.index("CAG")
    assert hM[idx] == idx + len(kmers)
    with pytest.raises(KpError):
        plan.pack_counts(np.array([iupac.kmer_code("CCG")], dtype=np.uint64), np.ones(1, np.int64), np.ones(1, np.int64))


@pytest.mark.parametrize("gen_pat,seed", [("NNN", 1), ("NNMNN", 2), ("RYNAN", 3), ("BDHV", 4), ("NNNNN", 5), ("SWKMN", 6),
                                          ("A", 7), ("NTNBN", 8)])
def test_greedy_against_oracle(eng, oracle, gen_pat, seed):
    """kp_greedy (one launch per depth, one CTA per pattern) against the plain-Python restatement of the reference's
    greedy recursion: same leaves in the same order, float64 losses / held-out LLs / score bit for bit."""
    from kmerpapa_b200 import iupac
    from kmerpapa_b200.algorithms import greedy_penalty_plus_pseudo as gr

    rng = np.random.default_rng(seed)
    km = oracle.kmers_of(gen_pat)
    U = rng.integers(0, 4000, size=len(km)) * (rng.random(len(km)) < 0.9)
    M = rng.binomial(np.maximum(U, 1), 0.03)
    if M.sum() == 0:
        M[0] = 3
    Mt, Ut = rng.binomial(M, 0.3), rng.binomial(U, 0.3)
    plan = eng.get_plan(gen_pat)
    PE = iupac.PatternEnumeration(gen_pat)
    for alpha, pen in ((0.8, 4.0), (10.0, 0.5), (1.0, 30.0)):
        mu = M.sum() / (M.sum() + U.sum())
        beta = (alpha * (1.0 - mu)) / mu
        kM, kU = plan.upload_kmer_tables(M - Mt, U - Ut, name="g_tr")
        tM, tU = plan.upload_kmer_tables(Mt, Ut, name="g_te")
        pats, loss, tst, score = gr._greedy(plan, kM, kU, alpha, beta, pen, test=(tM, tU))
        rscore, rnames, rloss, rtest = oracle.greedy(gen_pat, M - Mt, U - Ut, alpha, beta, pen, Mt, Ut)
        assert [PE.num2pattern(p) for p in pats] == rnames
        assert np.array_equal(loss.view(np.uint64), np.array(rloss, dtype=np.float64).view(np.uint64))
        assert np.array_equal(tst.view(np.uint64), np.array(rtest, dtype=np.float64).view(np.uint64))
        assert np.float64(score).tobytes() == np.float64(rscore).tobytes()


def test_lattice_free_plan(eng):
    """kp_plan_create_lite: the greedy estimator and the count queries work without the DP's tile lattice (and so for
    general patterns far beyond the DP's reach); the DP entry points refuse such a plan."""
    from kmerpapa_b200 import iupac, synthetic
    from kmerpapa_b200._native import KpError
    from kmerpapa_b200.algorithms import greedy_penalty_plus_pseudo as gr
    from kmerpapa_b200.engine import PartitionPlan

    gen_pat = "NNNANNN"
    kmers, pos, neg = synthetic.negbin_counts(gen_pat, 5)
    mu = pos.sum() / (pos.sum() + neg.sum())
    full, lite = eng.get_plan(gen_pat), PartitionPlan(gen_pat, 0, lite=True)
    res = []
    for plan in (full, lite):
        kM, kU = plan.upload_kmer_tables(pos, neg, name="lf")
        res.append(gr._greedy(plan, kM, kU, 1.0, (1 - mu) / mu, 5.0))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1]) and res[0][3] == res[1][3]
    M, U = lite.pattern_counts(kM, kU, res[1][0])
    assert M.sum() == pos.sum() and U.sum() == neg.sum()
    with pytest.raises(KpError):
        lite.expand(kM, kU)
    # 12 free positions: 15^12 = 1.3e14 patterns, no DP table could hold them; the greedy needs the 4^10 k-mers only
    big = "NNNNNANNNNN"
    plan = PartitionPlan(big, 0, lite=True)
    assert plan.npat == 15 ** 10
    rng = np.random.default_rng(3)
    n = 4 ** 10
    U = 1 + rng.negative_binomial(2, 2 / (2 + 2000.0), size=n)
    first = np.arange(n) % 4
    M = rng.binomial(U, 0.002 * (1 + first))     # the rate depends on the first position only
    kM, kU = plan.upload_kmer_tables(M, U, name="lfbig")
    mu = M.sum() / (M.sum() + U.sum())
    pats, loss, _, score = gr._greedy(plan, kM, kU, 1.0, (1 - mu) / mu, 8.0)
    PE = iupac.PatternEnumeration(big)
    names = [PE.num2pattern(p) for p in pats]
    assert sum(int(np.prod([len(iupac.CODE[c]) for c in nm])) for nm in names) == n      # a partition of the k-mers
    Mp, Up = plan.pattern_counts(kM, kU, pats)
    assert Mp.sum() == M.sum() and Up.sum() == U.sum()
    assert all(nm[0] != "N" for nm in names) and len(names) < 200      # the signal sits in position 0: it is always split


def test_7mer_matches_the_recorded_numba_reference():
    """bench.py's comparison with the unmodified numba reference (NNNMNNN, 34 M patterns), against that reference's
    recorded result: same loss bits and the same partition, name for name."""
    import importlib.util
    import json
    import os

    from conftest import ROOT

    nb = json.load(open(os.path.join(GOLDEN, "numba_NNNMNNN.json")))
    spec = importlib.util.spec_from_file_location("kp_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert (bench.NUMBA_GEN_PAT, bench.NUMBA_SEED, bench.NUMBA_ALPHA, bench.NUMBA_PENALTY) == (
        nb["gen_pat"], nb["seed"], nb["alpha"], nb["penalty"])
    assert bench.gpu_matches_numba(nb, 0)
