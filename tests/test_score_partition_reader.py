"""Reader of fitted partition files (kmerpapa_b200.score_partition.read_partition) and its host helpers; no GPU."""
import io
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from kmerpapa_b200 import iupac
from kmerpapa_b200.score_partition import PartitionError, covering, pattern_numbers, read_partition
from kmerpapa_b200.score_utils import get_loss, loss_from_terms


def _read(text):
    return read_partition(io.StringIO(text), "f")


def test_both_formats_of_the_recorded_runs():
    for name, long in (("cli_5mers_single.json", False), ("cli_5mers_joint.json", True), ("cli_5mers_superpattern.json", True)):
        g = json.load(open(os.path.join(GOLDEN, name)))
        patterns, rates = _read(g["stdout"])
        rows = [l.split() for l in g["stdout"].splitlines()[1:]]
        col = 4 if long else 0
        want = list(dict.fromkeys(r[col] for r in rows))   # first-seen order, once each
        assert patterns == want
        assert rates.dtype == np.float64
        by_pat = {r[col]: r[-1] for r in rows}
        assert [repr(float(p)) for p in rates] == [by_pat[p] for p in patterns]   # exact round trip


def test_duplicate_rows():
    long = "context c_neg c_pos c_rate pattern p_neg p_pos p_rate\n"
    text = long + "AA 1 0 0.0 AN 2 0 0.25\nCA 1 0 0.0 NC 1 0 0.5\nAC 1 0 0.0 AN 2 0 0.25\n"
    pats, rates = _read(text)
    assert pats == ["AN", "NC"] and rates.tolist() == [0.25, 0.5]
    with pytest.raises(PartitionError, match="two rates"):
        _read(long + "AA 1 0 0.0 AN 2 0 0.25\nAC 1 0 0.0 AN 2 0 0.3\n")
    # in the one-row-per-pattern format a repeated pattern is kept: it overlaps itself, which the GPU check reports
    pats, _ = _read("pattern p_neg p_pos p_rate\nAN 1 2 0.1\nAN 1 2 0.1\n")
    assert pats == ["AN", "AN"]


@pytest.mark.parametrize("text,match", [
    ("", "empty file"),
    ("\n\n", "empty file"),
    ("pattern p_neg p_pos p_rate\n", "no patterns"),
    ("pat p_neg p_pos p_rate\nA 1 1 0.5\n", "header"),
    ("pattern p_neg p_pos p_rate\nAN 1 1 0.5\nNNN 1 1 0.5\n", "length 3"),
    ("pattern p_neg p_pos p_rate\nAX 1 1 0.5\n", "not IUPAC: 'X'"),
    ("pattern p_neg p_pos p_rate\nan 1 1 0.5\n", "not IUPAC"),
    ("pattern p_neg p_pos p_rate\nAN 1 1 0\n", "not in"),
    ("pattern p_neg p_pos p_rate\nAN 1 1 1.0\n", "not in"),
    ("pattern p_neg p_pos p_rate\nAN 1 1 -0.5\n", "not in"),
    ("pattern p_neg p_pos p_rate\nAN 1 1 nan\n", "not in"),
    ("pattern p_neg p_pos p_rate\nAN 1 1 x\n", "not a number"),
    ("pattern p_neg p_pos p_rate\nAN 1 0.5\n", "3 columns"),
])
def test_rejected_files(text, match):
    with pytest.raises(PartitionError, match=match):
        _read(text)


def test_line_numbers_in_messages():
    with pytest.raises(PartitionError, match="f:4:"):
        _read("pattern p_neg p_pos p_rate\nAN 1 1 0.5\n\nCN 1 1 2\n")


def test_pattern_numbers_and_covering():
    rng = np.random.default_rng(5)
    gen = "NRSNB"
    PE = iupac.PatternEnumeration(gen)
    nums = rng.integers(0, PE.npat, 300)
    pats = [PE.num2pattern(x) for x in nums]
    assert np.array_equal(pattern_numbers(pats, gen), nums.astype(np.uint64))
    kmer = "AGCTC"
    assert covering(pats, kmer).tolist() == [i for i, p in enumerate(pats) if iupac.contains(p, kmer)]


def test_kmer_of_index():
    for gen in ("A", "NSN", "RNDY"):
        assert [iupac.kmer_of_index(gen, i) for i in range(len(iupac.matches(gen)))] == iupac.matches(gen)


def test_loss_from_terms_is_get_loss():
    rng = np.random.default_rng(1)
    counts = [(int(m), int(u)) for m, u in zip(rng.integers(0, 50, 40), rng.integers(0, 5000, 40))]
    alpha, beta = 0.8, 321.5
    from scipy.special import xlog1py, xlogy
    terms = []
    for m, u in counts:
        p = (m + alpha) / (m + u + alpha + beta)
        terms.append(xlogy(m, p) + xlog1py(u, -p))
    assert repr(loss_from_terms(terms)) == repr(get_loss(counts, alpha, beta))
    assert repr(loss_from_terms(terms, 3.0)) == repr(get_loss(counts, alpha, beta, 3.0))
