"""Scoring fitted partitions on the GPU (kmerpapa_b200.score_partition, kp_partition_assign / kp_partition_score):
the recorded reference runs, random valid partitions against host sums, and invalid partitions against a host check."""
import contextlib
import glob
import io
import json
import os
import time

import numpy as np
import pytest
from scipy.special import xlog1py, xlogy

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

INPUT_FLAGS = {"-p", "-b", "-n", "-j", "-s"}


def _input_argv(argv):
    """The input flags of a recorded argv, with the recorded data paths moved under this checkout's tests/golden."""
    out = []
    for i, a in enumerate(argv):
        if a in INPUT_FLAGS:
            value = argv[i + 1]
            cut = value.find("/tests/golden/")
            out += [a, GOLDEN + value[cut + len("/tests/golden"):] if cut >= 0 else value]
    return out


def _main(argv):
    from kmerpapa_b200 import score_partition

    out, err = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(out), contextlib.redirect_stderr(err):
        rc = score_partition.main(argv)
    return rc, out.getvalue(), err.getvalue()


@pytest.mark.parametrize("name", [os.path.basename(f) for f in sorted(glob.glob(os.path.join(GOLDEN, "cli_*.json")))])
def test_recorded_runs_reproduce_their_LL(name, tmp_path):
    """A partition scored on the data it was fitted on gives the fitting run's `LL=` line, byte for byte."""
    g = json.load(open(os.path.join(GOLDEN, name)))
    part = tmp_path / "partition.txt"
    part.write_text(g["stdout"])
    rc, out, err = _main(_input_argv(g["argv"]) + ["--partition", str(part)])
    assert rc == 0, err
    want = [l for l in g["stderr"] if l.startswith("LL=")]
    assert [l for l in err.splitlines() if l.startswith("LL=")] == want
    head, row = out.splitlines()
    assert head == "partition k n_patterns LL_test"
    assert row.split()[3] == want[0][3:]


def test_per_pattern_and_per_kmer_files(tmp_path):
    """On its training data the per-pattern counts are the partition file's, and the per-k-mer rows are the -l rows."""
    g = json.load(open(os.path.join(GOLDEN, "cli_5mers_joint.json")))
    part = tmp_path / "partition.txt"
    part.write_text(g["stdout"])
    pp, pk = tmp_path / "pp.txt", tmp_path / "pk.txt"
    rc, _, err = _main(_input_argv(g["argv"]) + ["--partition", str(part), "--per_pattern", str(pp), "--per_kmer", str(pk)])
    assert rc == 0, err
    rows = [l.split() for l in g["stdout"].splitlines()[1:]]
    patrows = {r[4]: (r[7], r[5], r[6]) for r in rows}   # pattern -> p_rate, p_neg, p_pos
    got = [l.split() for l in pp.read_text().splitlines()]
    assert got[0] == ["pattern", "p_rate", "t_neg", "t_pos", "LL"]
    assert [r[0] for r in got[1:]] == list(dict.fromkeys(r[4] for r in rows))
    for r in got[1:]:
        assert tuple(r[1:4]) == patrows[r[0]]
    from kmerpapa_b200 import iupac

    got = [l.split() for l in pk.read_text().splitlines()]
    assert got[0] == ["context", "c_neg", "c_pos", "pattern", "p_rate"]
    gen = iupac.lca_pattern(list(patrows))
    assert [r[0] for r in got[1:]] == iupac.matches(gen)
    want = {r[0]: (r[1], r[2], r[4], r[7]) for r in rows}
    assert {r[0]: tuple(r[1:]) for r in got[1:]} == want


def test_several_partitions_and_usage_errors(tmp_path):
    names = ["cli_5mers_single.json", "cli_5mers_greedy.json"]
    paths = []
    for i, name in enumerate(names):
        paths.append(tmp_path / f"p{i}.txt")
        paths[-1].write_text(json.load(open(os.path.join(GOLDEN, name)))["stdout"])
    argv = _input_argv(json.load(open(os.path.join(GOLDEN, names[0])))["argv"])
    rc, out, err = _main(argv + ["--partition"] + [str(p) for p in paths])
    assert rc == 0 and "LL=" not in err
    rows = [l.split() for l in out.splitlines()[1:]]
    assert [r[0] for r in rows] == [str(p) for p in paths]
    for r, name in zip(rows, names):
        ll = [l for l in json.load(open(os.path.join(GOLDEN, name)))["stderr"] if l.startswith("LL=")][0]
        assert r[1] == "5" and r[3] == ll[3:]
    bad = tmp_path / "bad.txt"
    bad.write_text("pattern p_neg p_pos p_rate\nNNNNN 1 1 1.5\n")
    rc, _, err = _main(argv + ["--partition", str(bad)])
    assert rc == 1 and "not in (0, 1)" in err


# ---- random valid partitions -------------------------------------------------------------------------------------
def _random_partition(gen, nsplit, rng):
    """Leaves of a random split tree: a leaf and one of its positions are drawn at random, and the position's letter
    is cut into two non-empty subsets.  Returned in random file order."""
    from kmerpapa_b200 import iupac

    leaves = [[iupac.MASK[c] for c in gen]]
    for _ in range(nsplit):
        j = int(rng.integers(len(leaves)))
        free = [i for i, m in enumerate(leaves[j]) if m & (m - 1)]
        if not free:
            continue
        i = free[int(rng.integers(len(free)))]
        m = leaves[j][i]
        subs = [s for s in range(1, 16) if s & m == s and s != m]
        s = subs[int(rng.integers(len(subs)))]
        a, b = list(leaves[j]), list(leaves[j])
        a[i], b[i] = s, m ^ s
        leaves[j] = a
        leaves.append(b)
    order = rng.permutation(len(leaves))
    return ["".join(iupac.LETTER[m] for m in leaves[o]) for o in order]


def _members(gen, pat):
    """k-mer indices of a pattern in the device's member order (position 0 fastest, bases in A, C, G, T order)."""
    from kmerpapa_b200.iupac import CODE

    out, w, parts = np.zeros(1, dtype=np.int64), 1, []
    for g, c in zip(gen, pat):
        parts.append(np.array([CODE[g].index(b) * w for b in "ACGT" if b in CODE[c]], dtype=np.int64))
        w *= len(CODE[g])
    for p in reversed(parts):
        out = (out[:, None] + p[None, :]).ravel()
    return out


def _nkmer(gen):
    from kmerpapa_b200.iupac import CODE

    return int(np.prod([len(CODE[c]) for c in gen]))


def _host_check(gen, patterns):
    """The first k-mer covered twice (members claimed in file order, in chunks of nkmer, stopping after the first chunk
    with a conflict) else the first k-mer covered by none; None for a partition."""
    nk = _nkmer(gen)
    seen = np.zeros(nk, dtype=np.int64)
    buf, nbuf, pats = [], 0, iter(patterns)
    while True:
        while nbuf < nk:
            p = next(pats, None)
            if p is None:
                break
            buf.append(_members(gen, p))
            nbuf += buf[-1].size
        if not buf:
            break
        flat = np.concatenate(buf)
        chunk, rest = flat[:nk], flat[nk:]
        np.add.at(seen, chunk, 1)
        dup = np.flatnonzero(seen >= 2)
        if dup.size:
            return "overlap", int(dup.min())
        buf, nbuf = ([rest], rest.size) if rest.size else ([], 0)
    gap = np.flatnonzero(seen == 0)
    return ("gap", int(gap.min())) if gap.size else None


GENS = [("A", 0), ("N", 3), ("RN", 4), ("NBN", 10), ("NNSNN", 40), ("DNNVNK", 120), ("NNNNRNNN", 600), ("NNNNNNNNN", 2000),
        ("NNNNNYNNNNN", 3000), ("NNNNNNNNNNNNN", 4000)]


@pytest.mark.parametrize("gen,nsplit", GENS)
def test_random_partition_against_host(gen, nsplit):
    from kmerpapa_b200 import iupac
    from kmerpapa_b200.engine import get_plan
    from kmerpapa_b200.score_partition import covering, pattern_numbers

    rng = np.random.default_rng(len(gen) * 1000 + nsplit)
    patterns = _random_partition(gen, nsplit, rng)
    assert iupac.lca_pattern(patterns) == gen
    rates = 10.0 ** rng.uniform(-7, -0.05, len(patterns))
    nk = _nkmer(gen)
    U = rng.negative_binomial(1, 1e-3, nk).astype(np.int64)
    M = rng.binomial(U, 0.01).astype(np.int64)
    U[rng.random(nk) < 0.05] = 0
    M[rng.random(nk) < 0.05] = 0
    big = rng.random(nk) < 0.001
    U[big] = rng.integers(1 << 36, 1 << 40, int(big.sum()))
    plan = get_plan(gen, lite=True)
    kM, kU = plan.upload_kmer_tables(M, U, name="t_rand")
    patnums = pattern_numbers(patterns, gen)
    owner_t, conflict, uncovered = plan.partition_assign(patnums)
    assert conflict is None and uncovered is None
    owner = owner_t.cpu().numpy().view(np.uint32).copy()
    Md, Ud, t, krate = plan.partition_score(patnums, rates, kM, kU, owner=owner_t)
    krate = krate.cpu().numpy()
    # host sums per pattern, and the host owner table
    hM, hU = np.empty(len(patterns), np.int64), np.empty(len(patterns), np.int64)
    howner = np.full(nk, -1, dtype=np.int64) if len(gen) <= 9 else None
    for q, p in enumerate(patterns):
        idx = _members(gen, p)
        hM[q], hU[q] = M[idx].sum(), U[idx].sum()
        if howner is not None:
            howner[idx] = q
    assert np.array_equal(Md, hM) and np.array_equal(Ud, hU)
    ht = xlogy(hM, rates) + xlog1py(hU, -rates)
    assert np.array_equal(t.view(np.uint64), ht.view(np.uint64))
    total = 0.0
    for x in (xlogy(int(m), float(p)) + xlog1py(int(u), -float(p)) for m, u, p in zip(hM, hU, rates)):
        total += x
    from kmerpapa_b200.score_utils import loss_from_terms

    assert repr(loss_from_terms(t)) == repr(-2 * total)
    if howner is not None:
        assert np.array_equal(owner.astype(np.int64), howner)
    else:
        sample = rng.integers(0, nk, 4096)
        for i in sample:
            assert covering(patterns, iupac.kmer_of_index(gen, int(i))).tolist() == [owner[i]]
    assert np.array_equal(krate.view(np.uint64), rates[owner].view(np.uint64))
    # the same bits on a second run
    owner2 = plan.partition_assign(patnums)[0].cpu().numpy().view(np.uint32)
    M2, U2, t2 = plan.partition_score(patnums, rates, kM, kU)
    assert np.array_equal(owner2, owner) and np.array_equal(M2, Md) and np.array_equal(U2, Ud)
    assert t2.tobytes() == t.tobytes()


def test_rates_from_counts_give_get_loss():
    """With p = (M + a) / (M + U + a + b) from the same counts, LL_test is score_utils.get_loss bit for bit."""
    from kmerpapa_b200 import iupac, score_partition
    from kmerpapa_b200.score_utils import get_loss

    rng = np.random.default_rng(11)
    gen = "NNRNN"
    patterns = _random_partition(gen, 60, rng)
    kmers = iupac.matches(gen)
    U = rng.integers(0, 100000, len(kmers))
    M = rng.binomial(U, 0.003)
    contextD = {k: (int(m), int(u)) for k, m, u in zip(kmers, M, U) if m + u > 0}
    counts = []
    for p in patterns:
        idx = [i for i, k in enumerate(kmers) if iupac.contains(p, k)]
        counts.append((int(M[idx].sum()), int(U[idx].sum())))
    alpha, beta = 0.8, 250.0
    rates = np.array([(m + alpha) / (m + u + alpha + beta) for m, u in counts])
    res = score_partition.score(patterns, rates, contextD)
    assert repr(res.LL) == repr(get_loss(counts, alpha, beta))


def test_longer_kmers_are_collapsed():
    from kmerpapa_b200 import iupac, score_partition

    rng = np.random.default_rng(12)
    patterns = _random_partition("NRN", 8, rng)
    rates = rng.uniform(0.01, 0.5, len(patterns))
    long = iupac.matches("NNRNN")
    contextD = {k: (int(rng.integers(0, 20)), int(rng.integers(0, 2000))) for k in long}
    short = {}
    for k, (m, u) in contextD.items():
        a = short.setdefault(k[1:4], [0, 0])
        a[0] += m
        a[1] += u
    res = score_partition.score(patterns, rates, contextD)
    for q, p in enumerate(patterns):
        ks = [k for k in short if iupac.contains(p, k)]
        assert (res.M[q], res.U[q]) == (sum(short[k][0] for k in ks), sum(short[k][1] for k in ks))


# ---- invalid partitions ------------------------------------------------------------------------------------------
def _invalid_cases():
    from kmerpapa_b200 import iupac

    rng = np.random.default_rng(21)
    cases = []
    for gen, nsplit in (("NNNNN", 150), ("NNNANNN", 900), ("NNNNNNNNN", 2500)):
        good = _random_partition(gen, nsplit, rng)
        # a pattern whose removal leaves the general pattern as it is (else the rest may partition a smaller one)
        j = next(j for j in range(len(good)) if iupac.lca_pattern(good[:j] + good[j + 1:]) == gen)
        i = next(i for i, (c, g) in enumerate(zip(good[j], gen)) if c != g)
        overlap = list(good)
        overlap[j] = good[j][:i] + gen[i] + good[j][i + 1:]
        gap = good[:j] + good[j + 1:]
        dup = good[: j + 1] + [good[j]] + good[j + 1:]
        cases += [(gen, "overlap", overlap), (gen, "gap", gap), (gen, "duplicate", dup)]
        cases.append((gen, "over-covering", [gen] * (200000 if len(gen) == 9 else 1000) + good))
    return cases


def test_invalid_partitions_name_the_host_kmer():
    from kmerpapa_b200 import iupac, score_partition

    for gen, what, patterns in _invalid_cases():
        kind, kidx = _host_check(gen, patterns)
        kmer = iupac.kmer_of_index(gen, kidx)
        rates = np.full(len(patterns), 0.25)
        t = time.perf_counter()
        with pytest.raises(score_partition.PartitionError) as e:
            score_partition.score(patterns, rates, {kmer: (1, 1)})
        dt = time.perf_counter() - t
        msg = str(e.value)
        assert f"k-mer {kmer} " in msg, (gen, what, msg)
        assert ("overlap" in msg) == (kind == "overlap"), (gen, what, msg)
        if kind == "overlap":
            a, b = [i for i, p in enumerate(patterns) if iupac.contains(p, kmer)][:2]
            assert f"pattern {a + 1} ({patterns[a]})" in msg and f"pattern {b + 1} ({patterns[b]})" in msg
        assert dt < 30, (gen, what, dt)


def test_test_kmer_outside_the_general_pattern():
    from kmerpapa_b200 import iupac, score_partition

    rng = np.random.default_rng(22)
    patterns = _random_partition("NNANN", 30, rng)
    contextD = {k: (1, 10) for k in rng.permutation(iupac.matches("NNNNN")).tolist()}
    first = min(k for k in contextD if k[2] != "A")
    with pytest.raises(score_partition.PartitionError, match=f"test k-mer {first} is outside"):
        score_partition.score(patterns, np.full(len(patterns), 0.1), contextD)
