"""Counting SNV contexts on the GPU (kmerpapa_b200.count_mutations, kp_snv_counts) against a plain-Python per-SNV
reference kept here, and the background table against apply_partition's k-mer counts."""
import contextlib
import io
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 1 << 16
COMP = bytes.maketrans(b"ACGT", b"TGCA")


# ---- plain-Python reference, one SNV at a time ---------------------------------------------------------------------
def _index(gen, w):
    from kmerpapa_b200.iupac import CODE

    idx, wt = 0, 1
    for g, ch in zip(gen, w):
        idx += CODE[g].index(ch) * wt
        wt *= len(CODE[g])
    return idx


def _ref_snv(gen, seq, i, ref, alt, in_regions, both, slot):
    """(status name, (table, k-mer index) or None) of one SNV with REF / ALT letters at record position i."""
    from kmerpapa_b200.iupac import contains

    k, c = len(gen), len(gen) // 2
    b = seq[i:i + 1].upper().decode()
    if b in "ACGT" and b != ref:
        return "ref_mismatch", None
    if not in_regions:
        return "outside_regions", None
    if i < c or i - c + k > len(seq):
        return "no_context", None
    w = seq[i - c: i - c + k].upper()
    if any(ch not in b"ACGT" for ch in w):
        return "no_context", None
    if contains(gen, w.decode()):
        idx, a = _index(gen, w.decode()), alt
    elif both and contains(gen, w.translate(COMP)[::-1].decode()):
        idx, a = _index(gen, w.translate(COMP)[::-1].decode()), "ACGT"["TGCA".index(alt)]
    else:
        return "no_match", None
    s = slot["ACGT".index(a)]
    return ("alt_not_selected", None) if s < 0 else ("counted", (s, idx))


def _reference(gen, recs, vcf_rows, regions, both, alts):
    from kmerpapa_b200 import count_mutations as C
    from kmerpapa_b200 import iupac

    labels, slot = C.check_args(gen, "both" if both else "forward", alts)
    seqs = dict(recs)
    pos = np.zeros((len(labels), len(iupac.matches(gen))), np.int64)
    status = []
    for chrom, p1, ref, alt in vcf_rows:
        if regions is None:
            inr = True
        elif not any(r[0] == chrom for r in regions):   # a record with no region is not scanned
            status.append("outside_regions")
            continue
        else:
            inr = any(r[0] == chrom and r[1] <= p1 - 1 < r[2] for r in regions)
        st, hit = _ref_snv(gen, seqs[chrom], p1 - 1, ref.upper(), alt.upper(), inr, both, slot)
        status.append(st)
        if hit:
            pos[hit] += 1
    return labels, pos, status


# ---- seeded inputs -------------------------------------------------------------------------------------------------
def _genome(rng, gen):
    """Records with N runs, other IUPAC letters, lowercase stretches, one shorter than k, and two over several pieces;
    k-mers of gen (and their reverse complements) planted so that long patterns match."""
    from kmerpapa_b200.iupac import CODE

    k = len(gen)
    recs = []
    for i, n in enumerate([3 * P + 101, k - 1, 5000, 2 * P - 3, 140_000]):
        s = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=n)
        for _ in range(n // 4000):
            a = int(rng.integers(n))
            kind = rng.integers(3)
            if kind == 0:
                s[a: a + int(rng.integers(1, 300))] = ord("N")
            elif kind == 1:
                s[a] = rng.choice(np.frombuffer(b"RYKn-", np.uint8))
            else:
                s[a: a + int(rng.integers(1, 3000))] |= 0x20
        if n > 4 * k:
            for _ in range(n // 300):
                km = bytes(ord(CODE[g][int(rng.integers(len(CODE[g])))]) for g in gen)
                if rng.integers(2):
                    km = km.translate(COMP)[::-1]
                a = int(rng.integers(n - k))
                s[a: a + k] = np.frombuffer(km, np.uint8)
        recs.append((f"chr{i}", s.tobytes()))
    return recs


def _snv_rows(rng, recs, k, n, unique=True):
    """(chrom, POS, REF, ALT) rows: random positions plus record ends, neighbours of non-bases and chunk and piece
    boundaries; REF is the genome base (a random letter where it is not a base), in random case."""
    rows = []
    for name, s in recs:
        L = len(s)
        if L == 0:
            continue
        want = set(int(x) for x in rng.integers(0, L, n * L // 400_000 + 3))
        want |= {0, 1, k // 2 - 1, k // 2, L - 1, L - 2, L - k // 2, L - k // 2 - 1}
        want |= {b + d for b in range(P, L, P) for d in (-k, -1, 0, 1, k)}
        bad = [i for i in range(L) if s[i:i + 1].upper() not in (b"A", b"C", b"G", b"T")]
        for i in bad[:: max(1, len(bad) // 40)]:
            want |= {i - 1, i + 1, i - k // 2, i + k // 2, i}
        for i in sorted(x for x in want if 0 <= x < L):
            b = s[i:i + 1].upper().decode()
            ref = b if b in "ACGT" else "ACGT"[int(rng.integers(4))]
            alt = [x for x in "ACGT" if x != ref][int(rng.integers(3))]
            if rng.integers(2):
                ref, alt = ref.lower(), alt.lower()
            rows.append((name, i + 1, ref, alt))
            if not unique and rng.integers(10) == 0:
                rows.append((name, i + 1, ref, alt))
    order = rng.permutation(len(rows))   # the VCF need not be sorted
    return [rows[o] for o in order]


def _write_vcf(path, rows):
    lines = ["##fileformat=VCFv4.2", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"]
    for c, p, r, a in rows:
        lines.append(f"{c}\t{p}\t.\t{r}\t{a}\t.\tPASS\t.")
    lines.append(f"{rows[0][0]}\t{rows[0][1]}\t.\t{rows[0][2]}\t{rows[0][3]}C,*\t.\tPASS\t.")   # skipped alleles
    path.write_text("\n".join(lines) + "\n")


def _regions(rng, recs):
    out = []
    for name, s in recs[:-1]:   # the last record has none: it is not scanned
        L = len(s)
        if L < 2:
            continue
        out += [(name, 0, 1), (name, L - 1, L), (name, 0, min(L, 50))]
        for _ in range(6):
            a = int(rng.integers(L - 1))
            out.append((name, a, int(min(L, a + rng.integers(1, 40_000)))))
        out.append((name, out[-1][1] + 1, min(L, out[-1][2] + 7)))   # overlaps the one before
    return out


CASES = [("NNNNCNNNN", True), ("NNNNANNNN", True), ("NNRNN", False), ("ACGTTNNCNNRTGCA", True),
         ("ACGTTGCANNNCNNAGTTRYC", False)]
ALTS = [None, ["T"], ["A", "G", "T"]]


@pytest.mark.parametrize("gen,both", CASES)
@pytest.mark.parametrize("with_regions", [False, True])
def test_counts_against_reference(tmp_path, gen, both, with_regions):
    from kmerpapa_b200 import apply_partition as A
    from kmerpapa_b200 import count_mutations as C

    rng = np.random.default_rng(zlib.crc32(f"{gen} {both} {with_regions}".encode()))
    recs = _genome(rng, gen)
    rows = _snv_rows(rng, recs, len(gen), 3000)
    vcf = tmp_path / "v.vcf"
    _write_vcf(vcf, rows)
    snvs = C.read_vcf(str(vcf))
    assert len(snvs) == len(rows) and snvs.skipped == 2
    regions = _regions(rng, recs) if with_regions else None
    strand = "both" if both else "forward"
    for alts in ALTS:
        labels, want_pos, want_status = _reference(gen, recs, rows, regions, both, alts)
        runs = [C.count_mutations(gen, recs, snvs, regions, strand, alts, chunk_bases=cb)
                for cb in (C.CHUNK_BASES, P, 3 * P)]
        res = runs[0]
        assert res.alts == labels
        assert [C.STATUS[x] for x in res.status] == want_status
        assert np.array_equal(res.positive, want_pos)
        assert res.status_counts == {s: want_status.count(s) for s in C.STATUS}
        assert res.skipped == 2
        for r in runs[1:]:
            assert np.array_equal(r.positive, res.positive) and np.array_equal(r.background, res.background)
            assert np.array_equal(r.status, res.status)
        assert res.positive.sum() == want_status.count("counted")
        assert (res.positive <= res.background).all()   # one allele per position
        if alts is None:
            assert want_status.count("counted") > 0 and want_status.count("no_context") > 0
            assert want_status.count("outside_regions") > 0 or not with_regions
            bg = A.apply([gen], [0.5], recs, regions=regions, strand=strand, kmer_counts=True).counts
            assert np.array_equal(res.background, bg)


def test_duplicates_count_twice_and_can_pass_the_background(tmp_path):
    from kmerpapa_b200 import count_mutations as C

    gen = "NNCNN"
    recs = [("a", b"ACGTACCCAGT" * 20)]
    rows = [("a", 7, "C", "T")] * 30   # one position, 30 times
    vcf = tmp_path / "v.vcf"
    _write_vcf(vcf, rows)
    res = C.count_mutations(gen, recs, C.read_vcf(str(vcf)), strand="both")
    assert res.positive.sum() == 30 and (res.positive > res.background).sum() == 1


def test_errors_after_the_pass(tmp_path):
    from kmerpapa_b200 import count_mutations as C
    from kmerpapa_b200.apply_partition import InputError

    recs = [("a", b"ACGTACGTAC"), ("b", b"GGGGG")]

    def run(text, **kw):
        vcf = tmp_path / "v.vcf"
        vcf.write_text("#CHROM\tPOS\tID\tREF\tALT\n" + text)
        return C.count_mutations("NCN", recs, C.read_vcf(str(vcf)), **kw)

    with pytest.raises(InputError, match=r"v.vcf:4: REF A does not match the genome base G at b:2; 2 SNV alleles mismatch"):
        run("a\t1\t.\tA\tC\na\t2\t.\tC\tT\nb\t2\t.\ta\tC\na\t3\t.\tT\tA\n")
    with pytest.raises(InputError, match=r"v.vcf:3: unknown chrom c \(no FASTA record of that name\)"):
        run("a\t1\t.\tA\tC\nc\t2\t.\tC\tT\nc\t1\t.\tC\tT\n")
    # a CHROM whose only line is an indel is still a CHROM of the VCF
    with pytest.raises(InputError, match=r"v.vcf:3: unknown chrom chrM \(no FASTA record of that name\)"):
        run("a\t1\t.\tA\tC\nchrM\t7\t.\tAC\tA\n")
    with pytest.raises(InputError, match=r"v.vcf:3: POS 11 is past the end of a \(2 SNV alleles in all\)"):
        run("a\t10\t.\tC\tA\na\t11\t.\tC\tA\na\t12\t.\tC\tT\n")
    # regions on a only: b is not scanned, so its REF is not checked
    res = run("b\t2\t.\tA\tC\na\t2\t.\tC\tT\n", regions=[("a", 0, 10)])
    assert [C.STATUS[x] for x in res.status] == ["outside_regions", "counted"]


def test_cli_unknown_chrom_without_snvs_exits_1(tmp_path):
    """An unknown CHROM whose only allele is an indel is an input error on the command line, not a traceback."""
    from kmerpapa_b200 import count_mutations as C

    fa = tmp_path / "g.fa"
    fa.write_bytes(b">chr1\nACGTACGTAC\n")
    vcf = tmp_path / "v.vcf"
    vcf.write_bytes(b"#CHROM\tPOS\tID\tREF\tALT\nchr1\t5\t.\tA\tG\nchrM\t7\t.\tAC\tA\n")
    err = io.StringIO()
    with contextlib.redirect_stderr(err):
        rc = C.main(["--pattern", "NCN", "--fasta", str(fa), "--vcf", str(vcf), "--prefix", str(tmp_path / "out")])
    assert rc == 1
    assert err.getvalue() == f"count_mutations: error: {vcf}:3: unknown chrom chrM (no FASTA record of that name)\n"


def test_cli_joint_file_fits_like_the_reference(tmp_path):
    """count_mutations' joint file and one written from the reference counts give the same kmerpapa -j output."""
    from kmerpapa_b200 import apply_partition as A
    from kmerpapa_b200 import cli
    from kmerpapa_b200 import count_mutations as C

    rng = np.random.default_rng(31)
    gen = "NNCNN"
    recs = _genome(rng, "NNNNN")
    fa = tmp_path / "g.fa"
    with open(fa, "wb") as f:
        for name, s in recs:
            f.write(b">" + name.encode() + b"\n" + b"\n".join(s[i: i + 60] for i in range(0, len(s), 60)) + b"\n")
    rows = _snv_rows(rng, recs, 5, 60_000)
    vcf = tmp_path / "v.vcf"
    _write_vcf(vcf, rows)
    err = io.StringIO()
    with contextlib.redirect_stderr(err):
        assert C.main(["--pattern", gen, "--fasta", str(fa), "--vcf", str(vcf), "--strand", "both", "--alt", "T", "A",
                       "--prefix", str(tmp_path / "out")]) == 0
    labels, want_pos, want_status = _reference(gen, recs, rows, None, True, ["T", "A"])
    text = err.getvalue()
    assert "ref_mismatch 0" in text and f"counted {want_status.count('counted')}" in text
    assert "0 k-mers with n_pos > n_bg" in text
    bg = A.apply([gen], [0.5], recs, strand="both", kmer_counts=True).counts
    ref_joint = tmp_path / "ref.T.txt"
    with open(ref_joint, "w") as f:
        C.write_joint(f, gen, want_pos[0], bg)
    assert (tmp_path / "out.T.txt").read_text() == ref_joint.read_text()
    outs = []
    for j in (tmp_path / "out.T.txt", ref_joint):
        o = tmp_path / (j.name + ".partition")
        assert cli.main(["-j", str(j), "-s", gen, "-c", "5", "-a", "1", "-o", str(o), "--seed", "1",
                         "--verbosity", "0"]) == 0
        outs.append(o.read_text())
    assert outs[0] == outs[1] and len(outs[0].splitlines()) > 1
