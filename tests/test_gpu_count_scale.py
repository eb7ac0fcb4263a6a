"""Counts at genome scale, on both sides of the 32-bit count limit, against the CPU oracle (uint64 counts, float64 scores).

Every count-consuming kernel picks its on-chip count width from the caller's max_count: 32-bit counts while the total is
at most 2^32 - 1, 64-bit counts above.  One strand of a human genome (about 2.9e9 positions) lies between 2^31 and 2^32;
both strands, several genomes or the tables `apply_partition --kmer_counts` writes lie above 2^32.  The bands below put
the totals, and single k-mers, right there:

- narrow_top:   total 2^32 - 1 exactly, one k-mer with U >= 2^31 (32-bit path, its largest total)
- narrow_top_m: total in (1.5 * 2^31, 2^32 - 1), one k-mer with M >= 2^31
- wide_edge:    total 2^32 exactly (the smallest total on the 64-bit path), one k-mer with U >= 2^31
- wide:         total from 2^33 to 2^40
- wide_heavy:   total from 2^48 to 2^50, single k-mers with M >= 2^32 and U >= 2^45

Elsewhere the tables are genome-like: per-k-mer totals spread log-normally, mutation rates from 1e-4 to 1e-2.  Every
count stays below 2^53, so it is exact in float64 in the kernels, the oracle and the references here.  At these totals a
loss is 1e10 to 1e16 and one float32 ulp of it is 1e3 to 1e9, so self-scores tie with split sums far more often than at
small counts: the DP's tie rule and rounded-up bit decide many cells.  Everything is compared bit for bit, or exactly for
integers.
"""
import contextlib
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NARROW_MAX = 2 ** 32 - 1
BANDS = ("narrow_top", "narrow_top_m", "wide_edge", "wide", "wide_heavy")
GRID = ((1.0, 4.0), (10.0, -3.0), (1.0, 0.0))   # (alpha, penalty): the negative and zero penalties drive the filter and ties


def band_counts(band, nk, seed):
    """(M, U, max_count) of one band: int64 k-mer tables of nk k-mers and their exact total."""
    rng = np.random.default_rng(seed)
    heavy = []   # (table, count) of single k-mers above the 31- or 32-bit line
    if band == "narrow_top":
        total = NARROW_MAX
        heavy = [("U", 2 ** 31 + int(rng.integers(0, 2 ** 28)))]
    elif band == "narrow_top_m":
        total = int(rng.integers(3 * 2 ** 30, NARROW_MAX))
        heavy = [("M", 2 ** 31 + int(rng.integers(0, 2 ** 28)))]
    elif band == "wide_edge":
        total = 2 ** 32
        heavy = [("U", 2 ** 31 + int(rng.integers(0, 2 ** 28)))]
    elif band == "wide":
        total = int(2.0 ** rng.uniform(33, 40))
    elif band == "wide_heavy":
        total = int(2.0 ** rng.uniform(48, 50))
        heavy = [("M", 2 ** 32 + int(rng.integers(0, 2 ** 40))), ("U", 2 ** 45 + int(rng.integers(0, 2 ** 46)))]
    else:
        raise ValueError(band)
    M = np.zeros(nk, dtype=np.int64)
    U = np.zeros(nk, dtype=np.int64)
    where = rng.permutation(nk)
    for i, (table, c) in enumerate(heavy):
        (M if table == "M" else U)[where[i % nk]] += c
    rest = total - sum(c for _, c in heavy)
    w = rng.lognormal(0.0, 1.0, nk) * (rng.random(nk) < 0.97)
    w[where[-1]] += 1.0
    c = np.floor(w / w.sum() * rest).astype(np.int64)
    c[np.argmax(w)] += rest - int(c.sum())
    m = rng.binomial(c, np.exp(rng.uniform(np.log(1e-4), np.log(1e-2), nk)))
    M += m
    U += c - m
    assert int(M.sum()) + int(U.sum()) == total and M.min() >= 0 and U.min() >= 0 and M.sum() > 0
    assert (total <= NARROW_MAX) == band.startswith("narrow")
    return M, U, total


def _beta(alpha, M, U):
    """beta from the totals, as the command line derives it (Python ints: exact division)."""
    from kmerpapa_b200.score_utils import beta_from_totals

    return beta_from_totals(alpha, int(M.sum()), int(U.sum()))


def _seed(*parts):
    return zlib.crc32("/".join(map(str, parts)).encode())


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def _codes(gen_pat):
    from kmerpapa_b200 import iupac

    return np.array([iupac.kmer_code(k) for k in iupac.matches(gen_pat)], dtype=np.uint64)


def _fresh_plan(gen_pat, monkeypatch, coop_tail=True, lite=False):
    """A new plan (not the cached one) with the rows kernel family and, with coop_tail=False, the multi-warp launch for
    every wave: both are read from the environment when the plan is created."""
    from kmerpapa_b200.engine import PartitionPlan

    monkeypatch.setenv("KP_DP_KERNEL", "rows")
    if coop_tail:
        monkeypatch.delenv("KP_NO_COOP_TAIL", raising=False)
    else:
        monkeypatch.setenv("KP_NO_COOP_TAIL", "1")
    return PartitionPlan(gen_pat, 0, lite=lite)


def _wave_sizes(gen_pat, plan):
    """Tiles per wave (high-position level) of a plan: the product of the per-position level counts of the high
    positions, i.e. C(n, j + 1) patterns of level j for a position of n letters."""
    from math import comb

    from kmerpapa_b200 import iupac

    radices = sorted(((2 ** len(iupac.CODE[ch]) - 1, i) for i, ch in enumerate(gen_pat) if len(iupac.CODE[ch]) > 1),
                     key=lambda x: -x[0])
    cells, high = 1, []
    for r, i in radices:          # the plan's choice of low positions: largest radix first, at most 4096 cells a tile
        if cells * r <= 4096:
            cells *= r
        else:
            high.append(len(iupac.CODE[gen_pat[i]]))
    waves = np.ones(1, dtype=np.int64)
    for n in high:
        waves = np.convolve(waves, [comb(n, j + 1) for j in range(n)])
    assert int(waves.sum()) == plan.info.ntiles
    return waves


# -------------------------------------------------------------------------------------------------------------------
# 1. DP kernel instantiations
# -------------------------------------------------------------------------------------------------------------------
# case -> (general pattern, register radix, rows of a tile, cooperative tail launch)
DP_CASES = {
    "r1_rows1": ("ACGT", 1, 1, True),
    "r3_rows729": ("RYSWKMRY", 3, 729, True),
    "r7_rows343": ("BDHVBDH", 7, 343, True),
    "r15_rows225_coop": ("NNNNN", 15, 225, True),          # 225 rows pad to 232: the KP_RP_NN instantiation
    "r15_rows225_multiwarp": ("NNNNN", 15, 225, False),
    "r15_rows135_coop": ("NNRRRRR", 15, 135, True),
}
DP_BANDS = BANDS + ("narrow_top_forced_wide",)


@pytest.mark.parametrize("band", DP_BANDS)
@pytest.mark.parametrize("case", list(DP_CASES))
def test_dp_instantiations_at_band_counts(oracle, monkeypatch, case, band):
    gen_pat, radix, rows, coop = DP_CASES[case]
    plan = _fresh_plan(gen_pat, monkeypatch, coop_tail=coop)
    info = plan.info
    assert (info.register_radix, info.rows) == (radix, rows), (info.register_radix, info.rows)
    assert ((info.rows + 7) & ~7 == 232) == (rows == 225)
    if radix == 15:
        # every wave has at most one tile per SM, so with the cooperative tail every wave runs one CTA per tile, and
        # without it every wave runs the multi-warp launch
        assert _wave_sizes(gen_pat, plan).max() <= info.sm_count and (rows + 31) // 32 <= 12
    M, U, total = band_counts(band.replace("_forced_wide", ""), plan.nkmer, _seed(gen_pat, band))
    max_count = 1 << 40 if band.endswith("forced_wide") else total
    wide = max_count > NARROW_MAX
    assert plan.dp_kernel_name(wide) == "kp_dp_rows_kernel"
    kM, kU = plan.pack_counts(_codes(gen_pat), M, U)
    eM, eU = plan.expand(kM, kU)
    allpat = np.arange(plan.npat, dtype=np.uint64)
    # and a penalty that keeps every pattern whole: then the general pattern's own self-score, on counts that sum to
    # the total, decides its cell
    for alpha, pen in GRID + ((1.0, 1e15),):
        beta = _beta(alpha, M, U)
        best, kept = plan.dp_single(eM, eU, max_count, alpha, beta, pen)
        ref = oracle.single_dp(gen_pat, M, U, alpha, beta, pen)
        got = plan.gather(best)
        bad = np.flatnonzero(_bits(got) != _bits(ref["score"]))
        assert bad.size == 0, f"alpha={alpha} pen={pen}: {bad.size} of {got.size} scores differ, first {bad[:8]}"
        split = plan.split_codes(best, kept, allpat)
        bad = np.flatnonzero(split != ref["split"])
        assert bad.size == 0, f"alpha={alpha} pen={pen}: {bad.size} split codes differ, first {bad[:8]}"
        assert np.array_equal(plan.gather_kept(kept) == 1, ref["split"] == 0xFF)
        assert np.array_equal(plan.backtrack(best, kept), oracle.backtrack(gen_pat, ref["split"]))


# -------------------------------------------------------------------------------------------------------------------
# 2. Counts out
# -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lite", [False, True], ids=["full", "lite"])
@pytest.mark.parametrize("band", BANDS)
def test_pattern_counts_at_band_counts(oracle, monkeypatch, band, lite):
    """kp_pattern_counts over every pattern of NNNNN equals the oracle's per-pattern M and U."""
    gen_pat = "NNNNN"
    plan = _fresh_plan(gen_pat, monkeypatch, lite=lite)
    M, U, _ = band_counts(band, plan.nkmer, _seed(gen_pat, band, "counts"))
    kM, kU = plan.pack_counts(_codes(gen_pat), M, U)
    ref = oracle.single_dp(gen_pat, M, U, 1.0, _beta(1.0, M, U), 4.0)
    gM, gU = plan.pattern_counts(kM, kU, np.arange(plan.npat, dtype=np.uint64))
    assert np.array_equal(gM.astype(np.uint64), ref["M"]) and np.array_equal(gU.astype(np.uint64), ref["U"])
    assert int(gM[-1]) == int(M.sum()) and int(gU[-1]) == int(U.sum())


@pytest.mark.parametrize("band", ["narrow_top", "wide_heavy"])
def test_pack_counts_sums_duplicates_across_2_32(band):
    """Duplicate codes whose counts sum past 2^32 (and, wide_heavy, past 2^50) are summed exactly by the pack atomics."""
    from kmerpapa_b200.engine import get_plan

    gen_pat = "NNAN"
    plan = get_plan(gen_pat, 0)
    rng = np.random.default_rng(_seed(band, "pack"))
    codes = _codes(gen_pat)
    idx = np.concatenate([np.arange(plan.nkmer), rng.integers(0, plan.nkmer, 4000), np.full(6, 5)])
    hi = 2 ** 31 if band == "narrow_top" else 2 ** 40
    pos = rng.integers(hi // 2, hi, idx.size, dtype=np.int64)
    neg = rng.integers(hi, 2 * hi, idx.size, dtype=np.int64)
    kM, kU = plan.pack_counts(codes[idx], pos, neg)
    refM = np.zeros(plan.nkmer, dtype=np.int64)
    refU = np.zeros(plan.nkmer, dtype=np.int64)
    np.add.at(refM, idx, pos)
    np.add.at(refU, idx, neg)
    assert refM[5] > 2 ** 32 and refU.max() < 2 ** 53
    assert np.array_equal(kM[: plan.nkmer].cpu().numpy(), refM)
    assert np.array_equal(kU[: plan.nkmer].cpu().numpy(), refU)


# -------------------------------------------------------------------------------------------------------------------
# 3. CV jobs
# -------------------------------------------------------------------------------------------------------------------
def _cv_tables(gen_pat, band, nk):
    """Band tables and one held-out fold drawn by binomial thinning (train = total - held-out stays in the band)."""
    M, U, total = band_counts(band, nk, _seed(gen_pat, band, "cv"))
    rng = np.random.default_rng(_seed(gen_pat, band, "fold"))
    Mte, Ute = rng.binomial(M, 0.3), rng.binomial(U, 0.3)
    return M, U, Mte, Ute, total


@pytest.mark.parametrize("band", BANDS)
@pytest.mark.parametrize("gen_pat", ["NNNNN", "BDHVBDH"])
def test_cv_jobs_at_band_counts(oracle, monkeypatch, gen_pat, band):
    plan = _fresh_plan(gen_pat, monkeypatch)
    M, U, Mte, Ute, total = _cv_tables(gen_pat, band, plan.nkmer)
    tot = plan.expand(*plan.upload_kmer_tables(M, U, name="s_tot"), name="s_tot_e")
    fold = plan.expand(*plan.upload_kmer_tables(Mte, Ute, name="s_fold"), name="s_fold_e")
    Mtr, Utr = M - Mte, U - Ute
    rng = np.random.default_rng(_seed(gen_pat, band, "roots"))
    roots = np.concatenate([[plan.npat - 1], rng.choice(plan.npat, size=47, replace=False)])
    for alpha, pen in GRID:
        beta = _beta(alpha, Mtr, Utr)
        otr, ote = oracle.cv_job(gen_pat, M, U, Mte, Ute, alpha, beta, pen)
        job = (tot[0], tot[1], fold[0], fold[1], total, alpha, beta, pen)
        top = plan.cv_job(*job)
        got = plan.gather(plan._buf["cvtrain"])
        bad = np.flatnonzero(_bits(got) != _bits(otr))
        assert bad.size == 0, f"alpha={alpha} pen={pen}: {bad.size} train cells differ, first {bad[:8]}"
        assert (top[0].tobytes(), top[1].tobytes()) == (otr[-1].tobytes(), ote[-1].tobytes())
        for r in roots:
            assert plan.cv_heldout(int(r)).tobytes() == ote[r].tobytes(), (alpha, pen, int(r))
        # the pipelined path the grid search takes: two jobs in flight
        t1 = plan.cv_job_submit(*job)
        t2 = plan.cv_job_submit(*job)
        for t in (t1, t2):
            tr, te = plan.cv_job_result(t)
            assert (tr.tobytes(), te.tobytes()) == (otr[-1].tobytes(), ote[-1].tobytes())


# -------------------------------------------------------------------------------------------------------------------
# 4. Sharded DP and CV job, several shards on one GPU
# -------------------------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def _shards(plan, world, replicate):
    from kmerpapa_b200 import sharded

    shards = [sharded.ShardedDP(plan, r, world, replicate=replicate) for r in range(world)]
    try:
        for s in shards:
            s.connect_local(shards)
        yield shards
    finally:
        for s in shards:
            s.close()


@pytest.mark.parametrize("replicate", [False, True], ids=["capacity", "replicate"])
@pytest.mark.parametrize("band", ["narrow_top", "wide"])
def test_sharded_at_band_counts(monkeypatch, band, replicate):
    """The sharded DP and CV job are the same bytes as the unsharded ones (which the tests above pin to the oracle)."""
    from kmerpapa_b200 import sharded
    from kmerpapa_b200._native import KpError

    gen_pat = "NNNNNN"
    plan = _fresh_plan(gen_pat, monkeypatch)
    worlds = []
    for w in range(2, 9):
        try:
            sharded.assignment(plan, w)
            worlds.append(w)
        except KpError:
            pass
    assert 2 in worlds and len(worlds) >= 3, worlds
    M, U, Mte, Ute, total = _cv_tables(gen_pat, band, plan.nkmer)
    tot = plan.expand(*plan.upload_kmer_tables(M, U, name="h_tot"), name="h_tot_e")
    fold = plan.expand(*plan.upload_kmer_tables(Mte, Ute, name="h_fold"), name="h_fold_e")
    alpha, pen = 10.0, -3.0
    beta = _beta(alpha, M, U)
    best, kept = plan.dp_single(tot[0], tot[1], total, alpha, beta, pen)
    ref_part = plan.backtrack(best, kept)
    pats = np.arange(plan.npat, dtype=np.uint64)
    ref_vals, ref_codes = plan.gather(best), plan.split_codes(best, kept, pats)
    cbeta = _beta(alpha, M - Mte, U - Ute)
    job = (tot[0], tot[1], fold[0], fold[1], total, alpha, cbeta, pen)
    ref_cv = plan.cv_job(*job)
    for world in worlds:
        with _shards(plan, world, replicate) as shards:
            sharded.run_local(shards, tot[0], tot[1], total, alpha, beta, pen)
            vals, _, codes = shards[-1].gather(pats, codes=True)
            assert np.array_equal(_bits(vals), _bits(ref_vals)), world
            assert np.array_equal(codes, ref_codes), world
            assert np.array_equal(shards[0].backtrack(), ref_part), world
            tr, te = shards[0].cv_job(*job)
            assert (tr.tobytes(), te.tobytes()) == (ref_cv[0].tobytes(), ref_cv[1].tobytes()), world


# -------------------------------------------------------------------------------------------------------------------
# 5. Greedy at scale
# -------------------------------------------------------------------------------------------------------------------
def greedy_by_index(gen_pat, kmerM, kmerU, alpha, beta, penalty, testM=None, testU=None):
    """oracle.greedy restated with numpy index subsets instead of string enumeration: the same recursion, candidate
    order and float64 arithmetic (oracle._greedy_loss, _greedy_test_ll), integer counts summed exactly."""
    from oracle import kp_oracle as O

    bases = "ACGT"
    # digit of every k-mer at every free position (k-mer index order: first free position fastest)
    nk = len(kmerM)
    digit = np.empty((len(gen_pat), nk), dtype=np.int8)
    stride = 1
    for i, ch in enumerate(gen_pat):
        letters = O.CODE[ch]
        digit[i] = np.array([bases.index(b) for b in letters], dtype=np.int8)[(np.arange(nk) // stride) % len(letters)]
        stride *= len(letters)
    tabs = [np.asarray(t, dtype=np.int64) for t in ([kmerM, kmerU] + ([testM, testU] if testM is not None else []))]
    letter_bits = {ch: sum(1 << bases.index(b) for b in O.CODE[ch]) for ch in O.CODE}

    def sums(idx, k):
        return [int(t[idx].sum()) for t in tabs[:k]]

    def rec(pattern, idx):
        c = sums(idx, len(tabs))
        best = O._greedy_loss(c[0], c[1], alpha, beta, penalty)
        mine = (best, [pattern], [best],
                [O._greedy_test_ll(c[0], c[1], c[2], c[3], alpha, beta)] if testM is not None else None)
        if all(ch in bases for ch in pattern):
            return mine
        choice = None
        for i, ch in enumerate(pattern):
            for c1, c2 in O.COMPLEMENTS.get(ch, []):
                in1 = ((letter_bits[c1] >> digit[i, idx]) & 1).astype(bool)
                a, b = sums(idx[in1], 2), sums(idx[~in1], 2)
                s = O._greedy_loss(a[0], a[1], alpha, beta, penalty) + O._greedy_loss(b[0], b[1], alpha, beta, penalty)
                if s < best:
                    best, choice = s, (pattern[:i] + c1 + pattern[i + 1:], pattern[:i] + c2 + pattern[i + 1:], idx[in1],
                                       idx[~in1])
        if choice is None:
            return mine
        s1, n1, l1, t1 = rec(choice[0], choice[2])
        s2, n2, l2, t2 = rec(choice[1], choice[3])
        return s1 + s2, n1 + n2, l1 + l2, (t1 + t2 if testM is not None else None)

    return rec(gen_pat, np.arange(nk))


@pytest.mark.parametrize("gen_pat,seed", [("NNN", 1), ("NNMNN", 2), ("RYNAN", 3), ("BDHV", 4), ("SWKMN", 6), ("A", 7)])
def test_greedy_restatement_is_the_oracle(oracle, gen_pat, seed):
    rng = np.random.default_rng(seed)
    km = oracle.kmers_of(gen_pat)
    U = rng.integers(0, 4000, size=len(km)) * (rng.random(len(km)) < 0.9)
    M = rng.binomial(np.maximum(U, 1), 0.03)
    M[0] += 3
    Mt, Ut = rng.binomial(M, 0.3), rng.binomial(U, 0.3)
    for alpha, pen in ((0.8, 4.0), (10.0, 0.5), (1.0, 30.0)):
        beta = _beta(alpha, M, U)
        assert greedy_by_index(gen_pat, M - Mt, U - Ut, alpha, beta, pen, Mt, Ut) == \
            oracle.greedy(gen_pat, M - Mt, U - Ut, alpha, beta, pen, Mt, Ut)


def _signal_tables(band, nk, seed):
    """Band tables whose rate depends on the first two positions only, so that the greedy partition stays small."""
    M, U, total = band_counts(band, nk, seed)
    c = M + U
    rng = np.random.default_rng(seed + 1)
    rate = np.array([2e-4, 1e-3, 3e-3, 1e-2])[np.arange(nk) % 4] * np.array([1.0, 1.5, 1.0, 0.7])[(np.arange(nk) // 4) % 4]
    M = rng.binomial(c, rate)
    return M, c - M, total


@pytest.mark.parametrize("band", ["narrow_top", "wide", "wide_heavy"])
def test_greedy_shared_path_at_band_counts(band):
    """8 free positions (65 536 k-mers): the root and every node of at least 32 768 k-mers take the marginals path
    shared by all CTAs.  wide_heavy has a single k-mer of more than 2^45 counts."""
    from kmerpapa_b200 import iupac
    from kmerpapa_b200.algorithms import greedy_penalty_plus_pseudo as gr
    from kmerpapa_b200.engine import PartitionPlan

    gen_pat = "NNNNANNNN"
    plan = PartitionPlan(gen_pat, 0, lite=True)
    assert plan.nkmer == 4 ** 8
    M, U, _ = _signal_tables(band, plan.nkmer, _seed(gen_pat, band, "greedy"))
    rng = np.random.default_rng(_seed(band, "greedy_fold"))
    Mt, Ut = rng.binomial(M, 0.3), rng.binomial(U, 0.3)
    PE = iupac.PatternEnumeration(gen_pat)
    for alpha, pen in ((1.0, 2000.0), (10.0, 400.0)):
        beta = _beta(alpha, M - Mt, U - Ut)
        kM, kU = plan.upload_kmer_tables(M - Mt, U - Ut, name="gs_tr")
        tM, tU = plan.upload_kmer_tables(Mt, Ut, name="gs_te")
        pats, loss, tst, score = gr._greedy(plan, kM, kU, alpha, beta, pen, test=(tM, tU))
        rscore, rnames, rloss, rtest = greedy_by_index(gen_pat, M - Mt, U - Ut, alpha, beta, pen, Mt, Ut)
        assert 4 <= len(rnames) < 2000
        assert [PE.num2pattern(p) for p in pats] == rnames
        assert np.array_equal(loss.view(np.uint64), np.array(rloss, dtype=np.float64).view(np.uint64))
        assert np.array_equal(tst.view(np.uint64), np.array(rtest, dtype=np.float64).view(np.uint64))
        assert np.float64(score).tobytes() == np.float64(rscore).tobytes()


def test_greedy_capacity_retry_at_band_counts(oracle):
    """A greedy partition of more than 65 536 leaves (every k-mer of 9 free positions, wide counts): the first call
    runs out of workspace and _greedy retries with a larger one.  Same leaves, order and bits as one call with room
    for all of them; every leaf's loss and held-out LL is the oracle's formula on its k-mer counts."""
    import ctypes

    import torch

    from kmerpapa_b200._native import KP_ERR_CAPACITY
    from kmerpapa_b200.algorithms import greedy_penalty_plus_pseudo as gr
    from kmerpapa_b200.engine import PartitionPlan

    gen_pat = "NNNNNNNNN"
    plan = PartitionPlan(gen_pat, 0, lite=True)
    M, U, _ = band_counts("wide", plan.nkmer, _seed(gen_pat, "retry"))
    rng = np.random.default_rng(5)
    Mt, Ut = rng.binomial(M, 0.3), rng.binomial(U, 0.3)
    Mtr, Utr = M - Mt, U - Ut
    alpha, pen = 1.0, -1e16          # every split pays: the partition is every k-mer
    beta = _beta(alpha, Mtr, Utr)
    kM, kU = plan.upload_kmer_tables(Mtr, Utr, name="gr_tr")
    tM, tU = plan.upload_kmer_tables(Mt, Ut, name="gr_te")
    # the overflowing call itself: its frontier outgrows the workspace from depth 17 on; nothing past the workspace
    # may be read or written (a guard region follows it)
    cap = 65536
    ws_bytes = int(plan.lib.kp_greedy_ws_bytes(cap))
    ws = torch.full((4 * ws_bytes,), 0xA5, dtype=torch.uint8, device=plan.device)
    out = np.empty(cap, dtype=np.uint64)
    n = ctypes.c_uint64(0)
    rc = plan.lib.kp_greedy(plan.handle, kM.data_ptr(), kU.data_ptr(), tM.data_ptr(), tU.data_ptr(), alpha, beta, pen,
                            ws.data_ptr(), cap, out.ctypes.data, None, None, ctypes.byref(n), None, plan._stream())
    assert rc == KP_ERR_CAPACITY
    assert bool((ws[ws_bytes:] == 0xA5).all()), "kp_greedy wrote past its workspace"
    pats, loss, tst, score = gr._greedy(plan, kM, kU, alpha, beta, pen, test=(tM, tU))
    assert len(pats) == plan.nkmer > 65536
    big = gr._greedy(plan, kM, kU, alpha, beta, pen, test=(tM, tU), cap=1 << 19)
    assert np.array_equal(pats, big[0]) and np.array_equal(_bits(loss), _bits(big[1]))
    assert np.array_equal(_bits(tst), _bits(big[2])) and np.float64(score).tobytes() == np.float64(big[3]).tobytes()
    kidx = {int(p): i for i, p in enumerate(oracle.kmer_patnums(gen_pat))}
    kidx = [kidx[int(p)] for p in pats]
    assert sorted(kidx) == list(range(plan.nkmer))
    rl = np.array([oracle._greedy_loss(Mtr[i], Utr[i], alpha, beta, pen) for i in kidx])
    rt = np.array([oracle._greedy_test_ll(Mtr[i], Utr[i], Mt[i], Ut[i], alpha, beta) for i in kidx])
    assert np.array_equal(_bits(loss), _bits(rl)) and np.array_equal(_bits(tst), _bits(rt))


# -------------------------------------------------------------------------------------------------------------------
# 6. All-k-mers CV terms
# -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("band", BANDS)
def test_all_kmers_fold_terms_at_band_counts(band):
    import scipy.special as sp

    from kmerpapa_b200.algorithms import all_kmers_CV

    nk, nf = 4096, 3
    M, U, _ = band_counts(band, nk, _seed(band, "terms"))
    rng = np.random.default_rng(_seed(band, "terms_folds"))
    Mte = np.stack([rng.binomial(M, 1 / nf) for _ in range(nf)], axis=1)
    Ute = np.stack([rng.binomial(U, 1 / nf) for _ in range(nf)], axis=1)
    Mtr, Utr = M[:, None] - Mte, U[:, None] - Ute
    alpha = 10.0
    betas = np.array([_beta(alpha, Mtr[:, f], Utr[:, f]) for f in range(nf)])
    tr, te = all_kmers_CV.fold_terms(Mtr, Utr, Mte, Ute, betas, alpha)
    p = (Mtr + alpha) / (Mtr + Utr + alpha + betas)
    rtr = -2 * (sp.xlogy(Mtr, p) + sp.xlog1py(Utr, -p)) + 0.0   # the train term is a leaf score with penalty 0
    rte = -2 * (sp.xlogy(Mte, p) + sp.xlog1py(Ute, -p))
    for name, got, ref in (("train", tr, rtr), ("held-out", te, rte)):
        bad = np.argwhere(_bits(got) != _bits(ref))
        assert bad.size == 0, f"{name}: {len(bad)} terms differ, first {bad[:4].tolist()}: " \
                              f"{[(got[tuple(i)], ref[tuple(i)]) for i in bad[:4]]}"


# -------------------------------------------------------------------------------------------------------------------
# 7. The command line, end to end
# -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("band", ["narrow", "wide"])
def test_cli_at_band_counts(oracle, tmp_path, band):
    """A 5-mer positive and background file with a total in (2^31, 2^32) (uint32 counts, the 32-bit DP) or in
    (2^33, 2^40] (uint64, the 64-bit DP): CV rows, the selected (alpha, penalty) and the final partition with its counts against
    the oracle."""
    from kmerpapa_b200 import cli, iupac
    from kmerpapa_b200.algorithms.bottum_up_array_w_numba import count_dtype

    gen_pat = "NNNNN"
    kmers = oracle.kmers_of(gen_pat)
    M, U, total = band_counts("narrow_top_m" if band == "narrow" else "wide", len(kmers), _seed("cli", band))
    if band == "wide":
        assert 2 ** 33 < total <= 2 ** 40
    assert count_dtype(int(M.sum()), int(U.sum())) == (np.uint32 if band == "narrow" else np.uint64)
    pos, bg = tmp_path / "pos.txt", tmp_path / "bg.txt"
    pos.write_text("".join(f"{k} {int(m)}\n" for k, m in zip(kmers, M)))
    bg.write_text("".join(f"{k} {int(m) + int(u)}\n" for k, m, u in zip(kmers, M, U)))
    out, cv = tmp_path / "out.txt", tmp_path / "cv.txt"
    alphas, pens, seed = (1.0, 10.0), (0.0, 4.0), 17
    rc = cli.main(["-p", str(pos), "-b", str(bg), "-a", *map(str, alphas), "-c", *map(str, pens), "--nfolds", "2",
                   "--seed", str(seed), "--CVfile", str(cv), "-o", str(out), "--verbosity", "0"])
    assert rc == 0
    ref = oracle.cv_grid(gen_pat, M, U, alphas, pens, 2, seed)
    rows = [line.split() for line in cv.read_text().splitlines()[1:]]
    assert len(rows) == len(ref["rows"])
    for row, (alpha, pen, test) in zip(rows, ref["rows"]):
        assert (int(row[0]), float(row[1]), float(row[2])) == (5, alpha, pen)
        assert np.float32(row[3]).tobytes() == np.float32(test).tobytes(), (row, test)
    best_alpha, best_pen, _ = ref["best"]
    fit = oracle.single_dp(gen_pat, M, U, best_alpha, _beta(best_alpha, M, U), best_pen)
    patnums = oracle.backtrack(gen_pat, fit["split"])
    lines = out.read_text().splitlines()
    assert lines[0] == "pattern p_neg p_pos p_rate"
    got = [line.split() for line in lines[1:]]
    PE = iupac.PatternEnumeration(gen_pat)
    assert [g[0] for g in got] == [PE.num2pattern(p) for p in patnums]
    assert [int(g[1]) for g in got] == [int(x) for x in fit["U"][patnums.astype(np.int64)]]
    assert [int(g[2]) for g in got] == [int(x) for x in fit["M"][patnums.astype(np.int64)]]
