"""Host side of kmerpapa_b200.apply_partition: the FASTA and BED readers, the region bookkeeping and the argument
checks that run before any GPU work; no GPU."""
import contextlib
import gzip
import io

import numpy as np
import pytest

from kmerpapa_b200 import apply_partition as A
from kmerpapa_b200 import iupac


def _records(path):
    return list(A.read_fasta(str(path)))


def test_fasta_multiline_crlf_lowercase_and_empty_records(tmp_path):
    p = tmp_path / "g.fa"
    p.write_bytes(b">chr1 first record\r\nACGTN\r\nacgtn\r\n\r\nRYK-\r\n>empty\r\n>chr2\tdescription\nA\nC\n>last\n")
    assert _records(p) == [("chr1", b"ACGTNacgtnRYK-"), ("empty", b""), ("chr2", b"AC"), ("last", b"")]


def test_fasta_gzip(tmp_path):
    p = tmp_path / "g.fa.gz"
    with gzip.open(p, "wb") as f:
        f.write(b">a\nAC\nGT\n>b\nTTT\n")
    assert _records(p) == [("a", b"ACGT"), ("b", b"TTT")]


def test_fasta_streams_one_record_at_a_time(tmp_path):
    p = tmp_path / "g.fa"
    p.write_bytes(b">a\nAC\n>a\nGT\n")
    it = A.read_fasta(str(p))
    assert next(it) == ("a", b"AC")   # the first record is handed out before the duplicate is read
    with pytest.raises(A.InputError, match=r"g.fa:3: duplicate record name a"):
        next(it)


@pytest.mark.parametrize("text, msg", [
    (b"ACGT\n>a\nAC\n", r":1: sequence before the first '>' header"),
    (b">a\nAC\n> \nAC\n", r":3: header line without a name"),
])
def test_fasta_errors_name_the_line(tmp_path, text, msg):
    p = tmp_path / "g.fa"
    p.write_bytes(text)
    with pytest.raises(A.InputError, match=msg):
        _records(p)


def test_bed_parsing_skips_headers_and_keeps_order():
    text = "track name=x\nbrowser position chr1\n# comment\n\nchr2\t5\t9\tname\t0\t+\nchr1 0 1\n"
    assert A.read_regions(io.StringIO(text), "r.bed") == [("chr2", 5, 9, "r.bed:5"), ("chr1", 0, 1, "r.bed:6")]


@pytest.mark.parametrize("line, msg", [
    ("chr1 5", r"r.bed:2: expected 'chrom start end'"),
    ("chr1 a 9", r"r.bed:2: start and end must be integers"),
    ("chr1 1.5 9", r"r.bed:2: start and end must be integers"),
    ("chr1 -1 9", r"r.bed:2: negative start -1"),
    ("chr1 9 9", r"r.bed:2: start 9 is not below end 9"),
    ("chr1 10 9", r"r.bed:2: start 10 is not below end 9"),
])
def test_bed_errors_name_the_line(line, msg):
    with pytest.raises(A.InputError, match=msg):
        A.read_regions(io.StringIO("chr1 0 5\n" + line + "\n"), "r.bed")


def test_merge_intervals_and_mask_words():
    s, e = A.merge_intervals(np.array([10, 0, 3, 12, 40, 20]), np.array([15, 5, 8, 13, 41, 21]))
    assert s.tolist() == [0, 10, 20, 40] and e.tolist() == [8, 15, 21, 41]
    s, e = A.merge_intervals(np.array([0, 5]), np.array([5, 9]))   # touching intervals merge
    assert s.tolist() == [0] and e.tolist() == [9]
    rng = np.random.default_rng(1)
    starts = rng.integers(0, 5000, 300)
    ends = starts + rng.integers(1, 200, 300)
    us, ue = A.merge_intervals(starts, ends)
    want = np.zeros(6000, bool)
    for a, b in zip(starts, ends):
        want[a:b] = True
    for pos0, pos1 in ((0, 6000), (64, 1000), (1024, 4097), (4096, 4096 + 33)):
        words = A.mask_words(us, ue, pos0, pos1)
        bits = np.unpackbits(words.view(np.uint8), bitorder="little").astype(bool)
        assert len(words) == (pos1 - pos0 + 31) // 32
        assert np.array_equal(bits[: pos1 - pos0], want[pos0:pos1])
        assert not bits[pos1 - pos0:].any()


def test_region_tasks_cover_each_region_once():
    """Every region's pieces: the clipped ones through a task with the right range, the others whole."""
    P = A.PIECE
    L = 5 * P + 123
    rng = np.random.default_rng(2)
    starts = np.concatenate([rng.integers(0, L - 1, 400), [0, 0, P, P - 1, 5 * P, 2 * P]])
    ends = np.concatenate([np.minimum(L, starts[:400] + rng.integers(1, 3 * P, 400)), [L, P, 2 * P, P + 1, L, 2 * P + 1]])
    tasks, reg = A.region_tasks(starts, ends, L)
    assert np.all(np.diff(tasks[:, 0].astype(np.int64)) >= 0)
    for s, e, (pa, pb, ta, tb) in zip(starts, ends, reg):
        assert pa == s // P and pb == (e - 1) // P
        for q in range(pa, pb + 1):
            lo, hi = max(s, q * P) - q * P, min(e, (q + 1) * P, L) - q * P
            t = ta if q == pa else tb if q == pb else -1
            if t >= 0:
                assert tasks[t].tolist() == [q, lo, hi]
                assert (lo, hi) != (0, min(P, L - q * P))   # a task never stands for a whole piece
            else:
                assert (lo, hi) == (0, min(P, L - q * P))


def test_kmers_of_indices_is_matches_order():
    for gen_pat in ("A", "SWN", "NRNCNYN"):
        kmers = iupac.matches(gen_pat)
        idx = np.arange(len(kmers))[::-1]
        assert [x.decode() for x in A.kmers_of_indices(gen_pat, idx)] == [kmers[i] for i in idx]


def test_kmer_count_file_reads_back():
    from kmerpapa_b200.io_utils import read_dict

    gen_pat = "NSN"
    counts = np.zeros(len(iupac.matches(gen_pat)), np.int64)
    counts[[0, 5, 31]] = [3, 1, 12]
    f = io.StringIO()
    A.write_kmer_counts(f, gen_pat, counts)
    table, total = read_dict(io.StringIO(f.getvalue()), None)
    kmers = iupac.matches(gen_pat)
    assert table == {kmers[0]: 3, kmers[5]: 1, kmers[31]: 12} and total == 16
    assert list(table) == [kmers[0], kmers[5], kmers[31]]


def test_even_k_rejected_with_both_strands():
    with pytest.raises(A.InputError, match=r"needs an odd k.*k = 4"):
        A.apply(["NNNN"], [0.1], [("a", b"ACGT")], strand="both")
    with pytest.raises(A.InputError, match="strand must be one of"):
        A.apply(["NNN"], [0.1], [("a", b"ACGT")], strand="reverse")
    with pytest.raises(A.InputError, match="multiple of 65536"):
        A.apply(["NNN"], [0.1], [("a", b"ACGT")], chunk_bases=1000)


def test_cli_errors_exit_1(tmp_path):
    part = tmp_path / "p.txt"
    part.write_text("pattern p_neg p_pos p_rate\nNNAN 10 1 0.1\n")
    fa = tmp_path / "g.fa"
    fa.write_bytes(b">a\nACGT\n")
    bed = tmp_path / "r.bed"
    bed.write_text("a 3 2\n")
    for argv, msg in (
        (["--partition", str(part), "--fasta", str(fa), "--strand", "both"], "needs an odd k"),
        (["--partition", str(part), "--fasta", str(fa), "--regions", str(bed)], "r.bed:1: start 3 is not below end 2"),
        (["--partition", str(tmp_path / "missing.txt"), "--fasta", str(fa)], "missing.txt"),
    ):
        err = io.StringIO()
        with contextlib.redirect_stderr(err), contextlib.redirect_stdout(io.StringIO()):
            assert A.main(argv) == 1
        assert err.getvalue().startswith("apply_partition: error: ") and msg in err.getvalue()
