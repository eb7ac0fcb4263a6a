"""The fiber kernel (kmerpapa_b200/csrc/kp_fiber.cuh: a fourth position on chip) against the CPU oracle, bit for bit:
score tables, split decisions, partitions, CV jobs — on every shape of general pattern it accepts (fiber position at
tile weight 1 and above, radix-3/7 positions among the other high positions), on the 32- and 64-bit count paths, and
against the rows kernel on the same inputs.  The full-size configs run through it in test_gpu_fullsize.py when
KP_DP_KERNEL=fiber (or when it is the default)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPES = ["NNNN", "NNNNN", "RNNNNY", "NNANNN", "NNNNRN", "VNNNNB", "NNNNNN"]


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _plan(gen_pat, kernel, monkeypatch):
    from kmerpapa_b200.engine import PartitionPlan

    monkeypatch.setenv("KP_DP_KERNEL", kernel)
    plan = PartitionPlan(gen_pat)
    assert plan.dp_kernel_name(wide=False) == f"kp_dp_{kernel}_kernel", (gen_pat, plan.dp_kernel_name())
    return plan


def _counts(gen_pat, seed, regime):
    from kmerpapa_b200 import iupac

    n = len(iupac.matches(gen_pat))
    rng = np.random.default_rng(seed)
    if regime == "dense":
        U = 1 + rng.negative_binomial(2, 2 / (2 + 30000.0), size=n)
        M = rng.binomial(U, np.minimum(0.5, 1e-3 * np.exp(rng.normal(0, 0.6, size=n))))
    elif regime == "sparse":
        U = rng.poisson(3.0, size=n)
        M = rng.binomial(U, 0.2)
    else:   # ties: few distinct counts, many exactly equal scores
        U = rng.integers(0, 3, size=n) * 10
        M = rng.integers(0, 2, size=n) * (U > 0)
    return M.astype(np.int64), U.astype(np.int64)


def _codes(gen_pat):
    from kmerpapa_b200 import iupac

    return np.array([iupac.kmer_code(k) for k in iupac.matches(gen_pat)], dtype=np.uint64)


@pytest.mark.parametrize("regime", ["dense", "sparse", "ties", "negative_penalty", "narrow_top", "wide_edge", "wide"])
@pytest.mark.parametrize("gen_pat", SHAPES)
def test_fiber_kernel_against_oracle(oracle, monkeypatch, gen_pat, regime):
    """The count bands of test_gpu_count_scale (totals 2^32 - 1, 2^32 and 2^33..2^40) run with max_count = the true
    total, so the band selects the count width; the fiber kernel runs at both widths on every shape."""
    from test_gpu_count_scale import GRID, band_counts

    if regime in ("narrow_top", "wide_edge", "wide"):
        M, U, _ = band_counts(regime, len(_codes(gen_pat)), 77 + len(gen_pat))
        grid = GRID
    else:
        M, U = _counts(gen_pat, 77 + len(gen_pat), "dense" if regime == "negative_penalty" else regime)
        grid = ({"ties": (1.0, 0.5), "negative_penalty": (10.0, -3.0)}.get(regime, (0.8, 4.0)),)
    mc = int(M.sum() + U.sum())
    plan = _plan(gen_pat, "fiber", monkeypatch)
    assert plan.dp_kernel_name(wide=True) == "kp_dp_fiber_kernel", gen_pat
    kM, kU = plan.pack_counts(_codes(gen_pat), M, U)
    eM, eU = plan.expand(kM, kU)
    for alpha, penalty in grid:
        mu = max(int(M.sum()), 1) / max(mc, 2)
        beta = alpha * (1.0 - mu) / mu
        best, kept = plan.dp_single(eM, eU, mc, alpha, beta, penalty)
        ref = oracle.single_dp(gen_pat, M, U, alpha, beta, penalty)
        got = plan.gather(best)
        bad = np.flatnonzero(_bits(got) != _bits(ref["score"]))
        assert bad.size == 0, f"{bad.size} of {got.size} scores differ, first {bad[:8]}"
        codes = plan.split_codes(best, kept, np.arange(plan.npat, dtype=np.uint64))
        assert np.array_equal(codes, ref["split"])
        assert np.array_equal(plan.gather_kept(kept) == 1, ref["split"] == 0xFF)
        assert np.array_equal(plan.backtrack(best, kept), oracle.backtrack(gen_pat, ref["split"]))
        # the 64-bit on-chip count path (selected by max_count) gives the same table
        best64, _ = plan.dp_single(eM, eU, 1 << 40, alpha, beta, penalty)
        assert np.array_equal(_bits(plan.gather(best64)), _bits(ref["score"]))


@pytest.mark.parametrize("gen_pat", ["NNNNN", "RNNNNY", "NNNNNN"])
def test_fiber_kernel_cv_job_against_oracle(oracle, monkeypatch, gen_pat):
    M, U = _counts(gen_pat, 5, "dense")
    rng = np.random.default_rng(9)
    Mte, Ute = rng.binomial(M, 0.2), rng.binomial(U, 0.2)
    alpha, beta, penalty = 0.5, 300.0, 3.0
    plan = _plan(gen_pat, "fiber", monkeypatch)
    tot = plan.expand(*plan.upload_kmer_tables(M, U, name="t"), name="te")
    fold = plan.expand(*plan.upload_kmer_tables(Mte, Ute, name="f"), name="fe")
    tr, te = plan.cv_job(tot[0], tot[1], fold[0], fold[1], int(M.sum() + U.sum()), alpha, beta, penalty)
    rtr, rte = oracle.cv_job(gen_pat, M, U, Mte, Ute, alpha, beta, penalty)
    assert np.array_equal(_bits(plan.gather(plan._buf["cvtrain"])), _bits(rtr))
    assert tr.tobytes() == rtr[-1].tobytes() and te.tobytes() == rte[-1].tobytes()
    for root in rng.integers(0, plan.npat, size=30):
        assert plan.cv_heldout(int(root)).tobytes() == rte[root].tobytes()


def test_fiber_and_rows_kernels_write_the_same_bytes(monkeypatch):
    """Both kernel families fill the same HBM layout: the raw device tables (scores and kept-whole masks) are equal."""
    import torch

    gen_pat = "NNNNNN"
    M, U = _counts(gen_pat, 3, "dense")
    mc = int(M.sum() + U.sum())
    out = []
    for kernel in ("rows", "fiber"):
        plan = _plan(gen_pat, kernel, monkeypatch)
        eM, eU = plan.expand(*plan.pack_counts(_codes(gen_pat), M, U))
        plan._buffer("best", int(plan.info.table_elems), torch.float32).zero_()
        plan._buffer("kept", int(plan.info.kept_elems), torch.int16).zero_()
        best, kept = plan.dp_single(eM, eU, mc, 1.0, 500.0, 6.0)
        out.append((best.view(torch.int32).clone(), kept.clone()))
    assert torch.equal(out[0][0], out[1][0])
    assert torch.equal(out[0][1], out[1][1])
