"""Host side of kmerpapa_b200.count_mutations: the VCF reader, the argument checks that run before any GPU work and the
joint count file; no GPU."""
import contextlib
import gzip
import io

import numpy as np
import pytest

from kmerpapa_b200 import count_mutations as C
from kmerpapa_b200 import iupac
from kmerpapa_b200.apply_partition import InputError

VCF = (b"##fileformat=VCFv4.2\n"
       b"##INFO=<ID=DP,Number=1,Type=Integer,Description=\"a, b\">\n"
       b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"
       b"chr1\t10\t.\tA\tG\t.\tPASS\tDP=3,4\n"
       b"chr1\t12\trs7\ta\tc,T,AT,*,<DEL>,,g\t.\tLowQual\t.\n"
       b"\n"
       b"chr2\t5\t.\tAC\tA\t.\t.\t.\n"
       b"chr2\t7\t.\tG\tt\r\n"
       b"chr2\t9\t.\tN\tA\n"
       b"chr1\t3\t.\tT\tC\n"
       b"chr2\t7\t.\tG\tT")   # a duplicate, and no newline at the end


def test_vcf_plain_gzip_and_any_block_size(tmp_path):
    """Headers and blank lines skipped, multi-allelic records split, lowercase and CRLF read, duplicates kept, every
    other allele skipped and counted; the same for gzip and for blocks that cut lines anywhere."""
    p = tmp_path / "v.vcf"
    p.write_bytes(VCF)
    g = tmp_path / "v.vcf.gz"
    with gzip.open(g, "wb") as f:
        f.write(VCF)
    for path in (p, g):
        for block in (1, 7, 64, C.VCF_BLOCK):
            s = C.read_vcf(str(path), block=block)
            assert s.chroms == ["chr1", "chr2"] and s.name == str(path)
            assert s.chrom_line.tolist() == [4, 7]   # chr2's first line has no SNV allele
            assert s.chrom.tolist() == [0, 0, 0, 0, 1, 0, 1]
            assert s.pos.tolist() == [9, 11, 11, 11, 6, 2, 6]
            assert s.ref.tolist() == [0, 0, 0, 0, 2, 3, 2]
            assert s.alt.tolist() == [2, 1, 3, 2, 3, 1, 3]
            assert s.line.tolist() == [4, 5, 5, 5, 8, 10, 11]
            assert s.skipped == 6   # AT, *, <DEL> and the empty allele of line 5; AC>A; N>A
            assert len(s) == 7


def test_vcf_empty_and_header_only(tmp_path):
    p = tmp_path / "v.vcf"
    p.write_bytes(b"##x\n#CHROM\tPOS\tID\tREF\tALT\n")
    s = C.read_vcf(str(p))
    assert len(s) == 0 and s.skipped == 0 and s.chroms == []
    p.write_bytes(b"")
    assert len(C.read_vcf(str(p))) == 0


@pytest.mark.parametrize("line, msg", [
    (b"chr1\t5\t.\tA", r"v.vcf:3: expected at least 5 tab-separated columns"),
    (b"chr1 5 . A C", r"v.vcf:3: expected at least 5 tab-separated columns"),
    (b"chr1\t5.0\t.\tA\tC", r"v.vcf:3: POS '5.0' is not an integer >= 1"),
    (b"chr1\tx\t.\tA\tC", r"v.vcf:3: POS 'x' is not an integer >= 1"),
    (b"chr1\t\t.\tA\tC", r"v.vcf:3: POS '' is not an integer >= 1"),
    (b"chr1\t0\t.\tA\tC", r"v.vcf:3: POS '0' is not an integer >= 1"),
    (b"chr1\t-4\t.\tA\tC", r"v.vcf:3: POS '-4' is not an integer >= 1"),
    (b"chr1\t1234567890123456789\t.\tA\tC", r"v.vcf:3: POS '1234567890123456789' is not an integer >= 1"),
    (b"chr\xff1\t5\t.\tA\tC", r"v.vcf:3: CHROM is not valid UTF-8"),
])
def test_vcf_errors_name_the_line(tmp_path, line, msg):
    p = tmp_path / "v.vcf"
    p.write_bytes(b"#CHROM\tPOS\tID\tREF\tALT\nchr1\t1\t.\tA\tC\n" + line + b"\nchr1\t2\t.\tA\tC\n")
    for block in (5, C.VCF_BLOCK):
        with pytest.raises(InputError, match=msg):
            C.read_vcf(str(p), block=block)


def test_vcf_many_lines_match_a_line_by_line_parse(tmp_path):
    """Random lines across many blocks, chromosome changes and multi-allelic records, against a plain split()."""
    rng = np.random.default_rng(4)
    lines, want = [], []
    alleles = ["A", "C", "G", "T", "a", "t", "AC", "*", "<INS>", "N", ""]
    for i in range(3000):
        chrom = f"c{int(rng.integers(0, 4)) * 7}" if rng.integers(5) == 0 or not lines else lines[-1].split("\t")[0]
        ref = ["A", "c", "G", "T", "N", "AG"][int(rng.integers(6))]
        alts = [alleles[int(rng.integers(len(alleles)))] for _ in range(int(rng.integers(1, 4)))]
        pos = int(rng.integers(1, 10 ** int(rng.integers(1, 12))))
        lines.append(f"{chrom}\t{pos}\tid{i}\t{ref}\t{','.join(alts)}\t.\tPASS\tX=1,2")
    text = "##h\n" + "\n".join(lines) + "\n"
    p = tmp_path / "v.vcf"
    p.write_text(text)
    names, first, skipped = {}, [], 0
    for ln, line in enumerate(text.splitlines(), 1):
        if line.startswith("#"):
            continue
        c = line.split("\t")
        if c[0] not in names:   # chromosomes in first-seen order, SNVs or not
            first.append(ln)
        ci = names.setdefault(c[0], len(names))
        for alt in c[4].split(","):
            if len(c[3]) == 1 and len(alt) == 1 and c[3].upper() in "ACGT" and alt.upper() in "ACGT":
                want.append((ci, int(c[1]) - 1, "ACGT".index(c[3].upper()),
                             "ACGT".index(alt.upper()), ln))
            else:
                skipped += 1
    for block in (100, 4096, C.VCF_BLOCK):
        s = C.read_vcf(str(p), block=block)
        got = list(zip(s.chrom.tolist(), s.pos.tolist(), s.ref.tolist(), s.alt.tolist(), s.line.tolist()))
        assert got == want and s.skipped == skipped and s.chroms == list(names) and s.chrom_line.tolist() == first


@pytest.mark.parametrize("pattern, strand, alts, msg", [
    ("NNNNCNNN", "both", None, r"needs an odd k.*k = 8"),
    ("NNNNNNNNN", "both", None, r"centre letter.*centre is N"),
    *[(f"NN{x}NN", "both", None, f"centre is {x}") for x in "SWBDHV"],
    ("NNCNN", "both", ["T", "X"], r"--alt takes letters of ACGT"),
    ("NNCNN", "forward", ["TT"], r"--alt takes letters of ACGT"),
    ("NNCNN", "forward", ["T", "t"], r"--alt names a letter twice"),
    ("NNCNX", "forward", None, r"IUPAC letters"),
    ("", "forward", None, r"IUPAC letters"),
    ("N" * 33, "forward", None, r"at most 32"),
    ("NNCNN", "reverse", None, r"strand must be one of"),
])
def test_argument_checks(pattern, strand, alts, msg):
    with pytest.raises(InputError, match=msg):
        C.check_args(pattern, strand, alts)


def test_argument_slots():
    for x in "ACGTMKRY":
        C.check_args(f"NN{x}NN", "both", None)
    assert C.check_args("NNNN", "forward", None) == (["all"], [0, 0, 0, 0])
    assert C.check_args("NNCNN", "both", ["t", "A", "G"]) == (["T", "A", "G"], [1, -1, 2, 0])


def test_joint_file_reads_back():
    from kmerpapa_b200.io_utils import read_joint_kmer_counts

    gen_pat = "NSN"
    kmers = iupac.matches(gen_pat)
    bg = np.zeros(len(kmers), np.int64)
    pos = np.zeros(len(kmers), np.int64)
    bg[[0, 5, 31, 7]] = [3, 1, 12, 9]
    pos[[0, 31]] = [2, 12]
    f = io.StringIO()
    C.write_joint(f, gen_pat, pos, bg)
    assert f.getvalue().splitlines()[0] == f"{kmers[0]} 2 3"
    table, n_unmut, n_mut = read_joint_kmer_counts(io.StringIO(f.getvalue()), gen_pat)
    assert table == {kmers[0]: (2, 1), kmers[5]: (0, 1), kmers[7]: (0, 9), kmers[31]: (12, 0)}
    assert list(table) == [kmers[0], kmers[5], kmers[7], kmers[31]]
    assert n_mut == 14 and n_unmut == 25 - 14


def test_cli_errors_exit_1(tmp_path):
    fa = tmp_path / "g.fa"
    fa.write_bytes(b">a\nACGT\n")
    vcf = tmp_path / "v.vcf"
    vcf.write_bytes(b"a\t1\t.\tA\n")
    bed = tmp_path / "r.bed"
    bed.write_text("a 3 2\n")
    base = ["--fasta", str(fa), "--prefix", str(tmp_path / "out")]
    for argv, msg in (
        (["--pattern", "NNCN", "--vcf", str(vcf), "--strand", "both"], "needs an odd k"),
        (["--pattern", "NNNNN", "--vcf", str(vcf), "--strand", "both"], "centre letter"),
        (["--pattern", "NNCNN", "--vcf", str(vcf), "--alt", "U"], "--alt takes letters of ACGT"),
        (["--pattern", "NNCNN", "--vcf", str(vcf)], "v.vcf:1: expected at least 5 tab-separated columns"),
        (["--pattern", "NNCNN", "--vcf", str(vcf), "--regions", str(bed)], "r.bed:1: start 3 is not below end 2"),
        (["--pattern", "NNCNN", "--vcf", str(tmp_path / "missing.vcf")], "missing.vcf"),
    ):
        err = io.StringIO()
        with contextlib.redirect_stderr(err), contextlib.redirect_stdout(io.StringIO()):
            assert C.main(argv + base) == 1
        assert err.getvalue().startswith("count_mutations: error: ") and msg in err.getvalue()
