"""Host side of kmerpapa_b200.burden: the --model parser, the model-set checks, --scale, the Poisson columns, the output
format and the input errors that are found before any GPU work; no GPU."""
import re

import numpy as np
import pytest
from scipy.stats import poisson

from kmerpapa_b200 import burden as B
from kmerpapa_b200.apply_partition import InputError

# a partition of NNCNN (any partition of the general pattern will do for the host checks)
PART_C = "pattern p_neg p_pos p_rate\nNNCNN 100 5 0.047619047619047616\n"


def model(name, alt, *patterns):
    return B.Model(name, alt, list(patterns), np.full(len(patterns), 0.01))


def write(tmp_path, name, text):
    p = tmp_path / name
    p.write_text(text)
    return str(p)


def test_model_parser(tmp_path):
    f = write(tmp_path, "ct.txt", PART_C)
    args = B.get_parser().parse_args(["--fasta", "g.fa", "--vcf", "v.vcf", "--model", "CT", "T", f,
                                      "--model", "CA", "a", f])
    assert args.model == [["CT", "T", f], ["CA", "a", f]]
    assert args.strand == "forward" and args.scale == 1.0 and args.regions is None
    m = B.read_model("CT", "T", f)
    assert m.name == "CT" and m.alt == "T" and m.patterns == ["NNCNN"] and m.rates.tolist() == [0.047619047619047616]
    long = "context c_neg c_pos c_rate pattern p_neg p_pos p_rate\n" + "".join(
        f"A{b}CAA 1 0 0.0 ANCAA 4 1 0.25\n" for b in "ACGT")
    m = B.read_model("x", "G", write(tmp_path, "long.txt", long))
    assert m.patterns == ["ANCAA"] and m.rates.tolist() == [0.25]
    with pytest.raises(SystemExit):   # NAME ALT FILE: three values
        B.get_parser().parse_args(["--fasta", "g", "--vcf", "v", "--model", "CT", "T"])
    with pytest.raises(SystemExit):   # at least one --model
        B.get_parser().parse_args(["--fasta", "g", "--vcf", "v"])


def test_revcomp_and_intersects():
    assert B.revcomp("ACGTN") == "NACGT"
    assert B.revcomp("RYSWKMBDHV") == "BDHVKMWSRY"
    assert B.intersects("NNCGN", "NNCHN") is False
    assert B.intersects("NNCNN", "NNCGN") is True
    assert B.intersects("NNCAN", "NNNWN") is True


def test_cpg_split_accepted():
    cpg = model("CpG", "T", "NNNNCGNNN")
    noncpg = model("nonCpG", "T", "NNNNCANNN", "NNNNCCNNN", "NNNNCTNNN")
    for strand in B.STRANDS:
        assert B.check_models([cpg, noncpg], strand) == ["NNNNCGNNN", "NNNNCHNNN"]
    six = [model("CA", "A", "NNNNCNNNN"), model("CG", "G", "NNNNCNNNN"), model("CT", "T", "NNNNCNNNN"),
           model("AC", "C", "NNNNANNNN"), model("AG", "G", "NNNNANNNN"), model("AT", "T", "NNNNANNNN")]
    assert len(B.check_models(six, "both")) == 6
    # G>A next to C>T is fine on the forward strand alone
    assert B.check_models([model("CT", "T", "NNCNN"), model("GA", "A", "NNGNN")], "forward")


@pytest.mark.parametrize("models, strand, msg", [
    ([model("CT", "T", "NNNNCNNNN"), model("GA", "A", "NNNNGNNNN")], "both",
     r"models CT \(NNNNCNNNN >T\) and GA \(NNNNGNNNN >A\) can count the same SNV on opposite strands"),
    ([model("a", "T", "NNCNN"), model("b", "T", "NNCNN")], "forward",
     r"models a \(NNCNN >T\) and b \(NNCNN >T\) can count the same SNV on the same strand"),
    ([model("a", "T", "NNCGN"), model("b", "T", "NNMNN")], "forward", r"models a .* and b .* same strand"),
    ([model("a", "C", "NNCNN")], "forward", r"model a: ALT C is a base of the centre letter C of NNCNN"),
    ([model("a", "T", "NNYNN")], "forward", r"model a: ALT T is a base of the centre letter Y"),
    ([model("a", "T", "NNCNN"), model("b", "T", "NNNGNNN")], "forward", r"model b has k = 7, model a k = 5"),
    ([model("a", "T", "NNCN")], "both", r"model a \(NNCN\): --strand both needs an odd k"),
    ([model("a", "T", "NNSNN")], "both", r"model a \(NNSNN\): --strand both needs a centre letter"),
    ([model("a", "T", "NNNNN")], "both", r"centre letter"),
    ([model("a", "X", "NNCNN")], "forward", r"model a: ALT must be one letter of ACGT, not 'X'"),
    ([model("a", "TG", "NNCNN")], "forward", r"ALT must be one letter"),
    ([model("a", "T", "NNCNN"), model("a", "A", "NNCNN")], "forward", r"two models are named a"),
    ([model("a b", "T", "NNCNN")], "forward", r"without white space"),
    ([], "forward", r"at least one --model"),
    ([model("a", "T", "NNCNN")], "reverse", r"strand must be one of"),
])
def test_model_set_rejected(models, strand, msg):
    with pytest.raises(InputError, match=msg):
        B.check_models(models, strand)


def test_strand_both_accepts_models_without_a_reverse_overlap():
    # A>G on NNANN next to C>T on NNCNN: revcomp(NNCNN) = NNGNN does not meet NNANN
    assert B.check_models([model("AG", "G", "NNANN"), model("CT", "T", "NNCNN")], "both")
    # C>T next to G>T: the reverse of a G>T is a C>A, which C>T does not count
    assert B.check_models([model("CT", "T", "NNCNN"), model("GT", "T", "NNGNN")], "both")


@pytest.mark.parametrize("scale", [0.0, -1.0, float("nan"), float("inf"), -float("inf")])
def test_scale_rejected(scale):
    with pytest.raises(InputError, match="--scale must be finite and > 0"):
        B.check_scale(scale)


def test_scale_accepted():
    for s in (1.0, 1e-300, 2.5, 1e300):
        B.check_scale(s)


def test_poisson_columns_against_scipy_stats():
    o = np.repeat(np.array([0, 1, 2, 3, 7, 20, 100, 1000, 10 ** 5], np.int64), 7)
    lam = np.tile(np.array([1e-6, 0.5, 1.0, 3.0, 50.0, 1000.0, 1e5]), 9)
    pe, pd = B.poisson_tails(o, lam)
    ref_e = np.where(o > 0, poisson.sf(o - 1, lam), 1.0)
    np.testing.assert_allclose(pe, ref_e, rtol=1e-12, atol=0)
    np.testing.assert_allclose(pd, poisson.cdf(o, lam), rtol=1e-12, atol=0)
    assert np.all(pe[o == 0] == 1.0)
    assert not np.isnan(pe).any() and not np.isnan(pd).any()


def test_poisson_edges():
    pe, pd = B.poisson_tails(np.array([0, 0, 3]), np.array([0.0, 2.0, 0.0]))
    assert pe.tolist() == [1.0, 1.0, 0.0]    # P(X >= 0) = 1; P(X >= 3) = 0 at lambda 0
    assert pd[0] == 1.0 and pd[2] == 1.0     # P(X <= o) = 1 at lambda 0
    assert pd[1] == poisson.cdf(0, 2.0)
    # counts above 2^32 are exact in float64 and give the same tails as scipy.stats
    big = np.array([2 ** 32 + 1, 2 ** 33, 3 * 2 ** 32 + 7], np.int64)
    lam = np.array([2.0 ** 32, 2.0 ** 33 + 2 ** 17, 3.0 * 2 ** 32 - 2 ** 18])
    pe, pd = B.poisson_tails(big, lam)
    np.testing.assert_allclose(pe, poisson.sf(big - 1, lam), rtol=1e-9)
    np.testing.assert_allclose(pd, poisson.cdf(big, lam), rtol=1e-9)
    assert 0.05 < pd[1] < 0.5 < pe[1] < 0.95   # 2^17 = 1.4 sd below lambda: significant neither way


def test_output_format():
    res = B.BurdenResult(chrom=["chr1", "chr2"], start=np.array([0, 5]), end=np.array([10, 9]),
                         observed=np.array([3, 0]), expected=np.array([0.1 + 0.2, 1.5]),
                         p_excess=np.array([0.25, 1.0]), p_deficit=np.array([0.75, 0.1]),
                         model_observed=np.array([[1, 0], [2, 0]]), model_expected=np.array([[0.1, 1.0], [0.2, 0.5]]),
                         model_n=np.array([[4, 2], [3, 1]]), names=["CpG", "nonCpG"])
    assert B.format_rows(res) == [
        "chrom start end observed expected p_excess p_deficit observed.CpG expected.CpG n.CpG observed.nonCpG "
        "expected.nonCpG n.nonCpG",
        "chr1 0 10 3 0.30000000000000004 0.25 0.75 1 0.1 4 2 0.2 3",
        "chr2 5 9 0 1.5 1.0 0.1 0 1.0 2 0 0.5 1",
    ]


VCF = b"#CHROM\tPOS\tID\tREF\tALT\nchr1\t3\t.\tA\tC\n"
FASTA = ">chr1\nACGTACGTAC\n"


@pytest.mark.parametrize("what, text, msg", [
    ("partition", "pattern p_neg p_pos p_rate\nNNCNN 1 2 1.5\n", r"ct.txt:2: rate 1.5 of pattern NNCNN is not in"),
    ("partition", "pattern p_neg p_pos p_rate\nNNCNN 1 2\n", r"ct.txt:2: 3 columns, expected 4"),
    ("regions", "chr1 5\n", r"r.bed:1: expected 'chrom start end'"),
    ("regions", "chr1 5 5\n", r"r.bed:1: start 5 is not below end 5"),
    ("vcf", "#h\nchr1\tx\t.\tA\tC\n", r"v.vcf:2: POS 'x' is not an integer >= 1"),
    ("vcf", "chr1\t3\t.\tA\n", r"v.vcf:1: expected at least 5 tab-separated columns"),
])
def test_input_errors_exit_1_with_file_line(tmp_path, capsys, what, text, msg):
    files = {"partition": PART_C, "regions": "chr1 0 5\n", "vcf": VCF.decode()}
    files[what] = text
    part = write(tmp_path, "ct.txt", files["partition"])
    bed = write(tmp_path, "r.bed", files["regions"])
    vcf = write(tmp_path, "v.vcf", files["vcf"])
    fa = write(tmp_path, "g.fa", FASTA)
    rc = B.main(["--fasta", fa, "--vcf", vcf, "--regions", bed, "--model", "CT", "T", part])
    assert rc == 1
    err = capsys.readouterr().err
    assert err.startswith("burden: error: ")
    assert re.search(msg, err), err


@pytest.mark.parametrize("argv, msg", [
    (["--scale", "0"], "--scale must be finite and > 0"),
    (["--scale", "nan"], "--scale must be finite and > 0"),
    (["--model", "CA", "C", "@"], "model CA: ALT C is a base of the centre letter"),
    (["--model", "CT2", "t", "@"], "models CT .* and CT2 .* can count the same SNV"),
    (["--model", "x", "T", "missing.txt"], "missing.txt"),
])
def test_argument_errors_exit_1(tmp_path, capsys, argv, msg):
    part = write(tmp_path, "ct.txt", PART_C)
    argv = [part if a == "@" else a for a in argv]
    base = ["--fasta", write(tmp_path, "g.fa", FASTA), "--vcf", write(tmp_path, "v.vcf", VCF.decode()),
            "--model", "CT", "T", part]
    assert B.main(base + argv) == 1
    err = capsys.readouterr().err
    assert err.startswith("burden: error: ") and re.search(msg, err), err
