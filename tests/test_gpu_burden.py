"""Observed against expected SNV counts of a model set on the GPU (kmerpapa_b200.burden, kp_snv_region_counts): the
expected columns against apply_partition, the observed ones against a plain-Python per-allele reference kept here and
against count_mutations, chunk-size independence, the errors after the pass and the command line end to end."""
import contextlib
import io
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 1 << 16
COMP = bytes.maketrans(b"ACGT", b"TGCA")


# ---- plain-Python reference, one allele at a time ------------------------------------------------------------------
def _counts(gen, seq, i, ref, alt, both, model_alt):
    """count_mutations' status of one SNV allele for one model, without regions: 'counted' or another name."""
    from kmerpapa_b200.iupac import contains

    k, c = len(gen), len(gen) // 2
    b = seq[i:i + 1].upper().decode()
    if b in "ACGT" and b != ref:
        return "ref_mismatch"
    if i < c or i - c + k > len(seq):
        return "no_context"
    w = seq[i - c: i - c + k].upper()
    if any(ch not in b"ACGT" for ch in w):
        return "no_context"
    if contains(gen, w.decode()):
        a = alt
    elif both and contains(gen, w.translate(COMP)[::-1].decode()):
        a = "ACGT"["TGCA".index(alt)]
    else:
        return "no_match"
    return "counted" if a == model_alt else "alt_not_selected"


def _reference(gens, alts, recs, alleles, regions, both):
    """(status per allele, model id per allele (None: none), observed [model, row]) of burden."""
    seqs = dict(recs)
    status, ids = [], []
    for chrom, i, ref, alt in alleles:
        per = [_counts(g, seqs[chrom], i, ref.upper(), alt.upper(), both, a) for g, a in zip(gens, alts)]
        hit = [m for m, s in enumerate(per) if s == "counted"]
        assert len(hit) <= 1
        ids.append(hit[0] if hit else None)
        inside = regions is None or any(r[0] == chrom and r[1] <= i < r[2] for r in regions)
        if regions is not None and not any(r[0] == chrom for r in regions):
            status.append("outside_regions")   # a record with no region is not scanned
        elif per[0] == "ref_mismatch":
            status.append("ref_mismatch")
        elif not inside:
            status.append("outside_regions")
        elif per[0] == "no_context":
            status.append("no_context")
        else:
            status.append("counted" if hit else "not_modelled")
    rows = [(name, 0, len(s)) for name, s in recs] if regions is None else regions
    obs = np.zeros((len(gens), len(rows)), np.int64)
    for (chrom, i, _, _), m, st in zip(alleles, ids, status):
        if m is None or st != "counted":
            continue
        for r, (c, a, b) in enumerate(rows):
            if c == chrom and a <= i < b:
                obs[m, r] += 1
    return status, ids, obs


# ---- seeded inputs -------------------------------------------------------------------------------------------------
def _partition(rng, gen, depth=5):
    """A random partition of gen: split a multi-base letter into two sub-letters, recursively."""
    from kmerpapa_b200 import iupac

    multi = [i for i, ch in enumerate(gen) if len(iupac.CODE[ch]) > 1]
    if depth == 0 or not multi or rng.random() < 0.25:
        return [gen]
    i = multi[int(rng.integers(len(multi)))]
    bases = list(iupac.CODE[gen[i]])
    rng.shuffle(bases)
    cut = int(rng.integers(1, len(bases)))
    out = []
    for part in (bases[:cut], bases[cut:]):
        letter = iupac.LETTER[sum(iupac.MASK[b] for b in part)]
        out += _partition(rng, gen[:i] + letter + gen[i + 1:], depth - 1)
    return out


def _models(rng, specs):
    from kmerpapa_b200 import burden as B

    out = []
    for name, gen, alt in specs:
        pats = _partition(rng, gen)
        out.append(B.Model(name, alt, pats, np.exp(rng.uniform(np.log(1e-4), np.log(0.2), len(pats)))))
    return out


def _genome(rng, k):
    """Records with N runs, other IUPAC letters and lowercase stretches, one shorter than k, two over several pieces."""
    recs = []
    for i, n in enumerate([3 * P + 101, k - 1, 5000, 2 * P - 3, 90_000]):
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
        recs.append((f"chr{i}", s.tobytes()))
    return recs


def _regions(rng, recs, with_last=False):
    """Overlapping regions in any order, one- and two-base regions at record ends, a whole-record region; the last
    record gets none unless with_last."""
    out = []
    for name, s in (recs if with_last else recs[:-1]):
        L = len(s)
        if L < 2:
            continue
        out += [(name, 0, 1), (name, L - 2, L), (name, 0, L)]
        for _ in range(8):
            a = int(rng.integers(L - 1))
            out.append((name, a, int(min(L, a + rng.integers(1, 40_000)))))
        out.append((name, out[-1][1] + 1, min(L, out[-1][2] + 7)))   # overlaps the one before
    order = rng.permutation(len(out))
    return [out[o] for o in order]


def _vcf_lines(rng, recs, k, regions, n):
    """VCF lines (chrom, POS, REF, [ALT, ...]): random positions, record ends, neighbours of non-bases, piece
    boundaries and region edges; multi-allelic lines and duplicate lines; REF in random case."""
    lines = []
    edges = {}
    for c, a, b in regions or []:
        edges.setdefault(c, set()).update({a - 1, a, b - 1, b})
    for name, s in recs:
        L = len(s)
        if L == 0:
            continue
        want = set(int(x) for x in rng.integers(0, L, n * L // 400_000 + 3))
        want |= {0, 1, k // 2 - 1, k // 2, L - 1, L - 2, L - k // 2, L - k // 2 - 1} | edges.get(name, set())
        want |= {b + d for b in range(P, L, P) for d in (-k, -1, 0, 1, k)}
        bad = [i for i in range(L) if s[i:i + 1].upper() not in (b"A", b"C", b"G", b"T")]
        for i in bad[:: max(1, len(bad) // 40)]:
            want |= {i - 1, i + 1, i - k // 2, i + k // 2, i}
        for i in sorted(x for x in want if 0 <= x < L):
            b = s[i:i + 1].upper().decode()
            ref = b if b in "ACGT" else "ACGT"[int(rng.integers(4))]
            others = [x for x in "ACGT" if x != ref]
            alts = [others[int(rng.integers(3))]] if rng.integers(4) else others   # some lines are multi-allelic
            if rng.integers(2):
                ref, alts = ref.lower(), [x.lower() for x in alts]
            lines.append((name, i + 1, ref, alts))
            if rng.integers(12) == 0:
                lines.append((name, i + 1, ref, alts))   # a duplicate line
    order = rng.permutation(len(lines))   # the VCF need not be sorted
    return [lines[o] for o in order]


def _write_vcf(path, lines):
    out = ["##fileformat=VCFv4.2", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"]
    out += [f"{c}\t{p}\t.\t{r}\t{','.join(a)}\t.\tPASS\t." for c, p, r, a in lines]
    path.write_text("\n".join(out) + "\n")


def _alleles(lines):
    return [(c, p - 1, r, a) for c, p, r, alts in lines for a in alts]


def _write_fasta(path, recs):
    with open(path, "wb") as f:
        for name, s in recs:
            f.write(b">" + name.encode() + b"\n" + b"\n".join(s[i: i + 60] for i in range(0, len(s), 60)) + b"\n")


COLUMNS = ("observed", "expected", "p_excess", "p_deficit", "model_observed", "model_expected", "model_n", "status")
SETS = {
    "forward": [("CT", "NNNCNNN", "T"), ("CA", "NNNCNNN", "A"), ("GA", "NNNGNNN", "A"), ("AG", "NNNANNN", "G")],
    "both": [("CT", "NNNCNNN", "T"), ("CA", "NNNCNNN", "A"), ("AG", "NNNANNN", "G"), ("AT", "NNNANNN", "T")],
}


@pytest.mark.parametrize("strand", ["forward", "both"])
@pytest.mark.parametrize("with_regions", [False, True])
def test_against_apply_partition_and_reference(tmp_path, strand, with_regions):
    from kmerpapa_b200 import apply_partition as A
    from kmerpapa_b200 import burden as B
    from kmerpapa_b200 import count_mutations as C

    rng = np.random.default_rng(zlib.crc32(f"{strand} {with_regions}".encode()))
    models = _models(rng, SETS[strand])
    recs = _genome(rng, 7)
    regions = _regions(rng, recs) if with_regions else None
    lines = _vcf_lines(rng, recs, 7, regions, 3000)
    vcf = tmp_path / "v.vcf"
    _write_vcf(vcf, lines)
    snvs = C.read_vcf(str(vcf))
    alleles = _alleles(lines)
    assert len(snvs) == len(alleles)
    runs = [B.burden(models, recs, snvs, regions, strand, scale=1.5, chunk_bases=cb) for cb in (A.CHUNK_BASES, P, 3 * P)]
    runs.append(B.burden(models, recs, snvs, regions, strand, scale=1.5))
    res = runs[0]
    for r in runs[1:]:   # the same bits for every chunk size and run
        for col in COLUMNS:
            assert np.asarray(getattr(r, col)).tobytes() == np.asarray(getattr(res, col)).tobytes(), col
    for m, mod in enumerate(models):
        ap = A.apply(mod.patterns, mod.rates, recs, regions=regions, strand=strand)
        assert ap.expected.tobytes() == res.model_expected[m].tobytes()
        assert np.array_equal(ap.n_contexts, res.model_n[m])
    gens = [B.check_models([mod], strand)[0] for mod in models]
    status, ids, obs = _reference(gens, [m.alt for m in models], recs, alleles, regions, strand == "both")
    assert [B.STATUS[x] for x in res.status] == status
    assert np.array_equal(res.model_observed, obs)
    assert res.status_counts == {s: status.count(s) for s in B.STATUS}
    assert status.count("counted") > 0 and status.count("not_modelled") > 0 and status.count("no_context") > 0
    assert len({i for i in ids if i is not None}) == len(models)   # every model counts some allele
    assert np.array_equal(res.observed, obs.sum(axis=0))
    want = res.model_expected[0]
    for m in range(1, len(models)):
        want = want + res.model_expected[m]
    assert res.expected.tobytes() == want.tobytes()
    pe, pd = B.poisson_tails(res.observed, 1.5 * want)
    assert res.p_excess.tobytes() == pe.tobytes() and res.p_deficit.tobytes() == pd.tobytes()
    if regions is None:
        assert res.observed.sum() == status.count("counted")


@pytest.mark.parametrize("strand", ["forward", "both"])
def test_sums_equal_count_mutations(tmp_path, strand):
    """On disjoint regions, summed observed.NAME / n.NAME equal count_mutations' positive / background totals."""
    from kmerpapa_b200 import burden as B
    from kmerpapa_b200 import count_mutations as C

    rng = np.random.default_rng(zlib.crc32(f"cm {strand}".encode()))
    models = _models(rng, SETS[strand])
    recs = _genome(rng, 7)
    pieces = [(name, a, b) for name, s in recs[:-1] if len(s) > 100
              for a, b in [(0, 40), (60, len(s) // 2), (len(s) // 2, len(s) - 30)]]
    lines = _vcf_lines(rng, recs, 7, pieces, 3000)
    vcf = tmp_path / "v.vcf"
    _write_vcf(vcf, lines)
    snvs = C.read_vcf(str(vcf))
    res = B.burden(models, recs, snvs, pieces, strand)
    for m, mod in enumerate(models):
        gen = B.check_models([mod], strand)[0]
        cm = C.count_mutations(gen, recs, snvs, pieces, strand, alts=[mod.alt])
        assert res.model_observed[m].sum() == cm.positive.sum() > 0
        assert res.model_n[m].sum() == cm.background.sum()
    assert res.status_counts["outside_regions"] > 0


@pytest.mark.parametrize("strand", ["forward", "both"])
def test_cpg_split_adds_up(tmp_path, strand):
    from kmerpapa_b200 import burden as B
    from kmerpapa_b200 import count_mutations as C

    rng = np.random.default_rng(zlib.crc32(f"cpg {strand}".encode()))
    recs = _genome(rng, 9)
    regions = _regions(rng, recs, with_last=True)
    lines = _vcf_lines(rng, recs, 9, regions, 6000)
    vcf = tmp_path / "v.vcf"
    _write_vcf(vcf, lines)
    snvs = C.read_vcf(str(vcf))
    split = _models(rng, [("CpG", "NNNNCGNNN", "T"), ("nonCpG", "NNNNCHNNN", "T")])
    one = _models(rng, [("CT", "NNNNCNNNN", "T")])
    a = B.burden(split, recs, snvs, regions, strand)
    b = B.burden(one, recs, snvs, regions, strand)
    assert np.array_equal(a.observed, b.observed) and a.observed.sum() > 0
    assert a.model_observed[0].sum() > 0 and a.model_observed[1].sum() > 0
    assert np.array_equal(a.model_n.sum(axis=0), b.model_n[0])
    assert a.status_counts == b.status_counts


def test_errors_after_the_pass(tmp_path):
    """REF mismatch, unknown CHROM and POS past the end: count_mutations' messages."""
    from kmerpapa_b200 import burden as B
    from kmerpapa_b200 import count_mutations as C
    from kmerpapa_b200.apply_partition import InputError

    recs = [("a", b"ACGTACGTAC"), ("b", b"GGGGG")]
    models = [B.Model("CT", "T", ["NCN"], np.array([0.01])), B.Model("AG", "G", ["NAN"], np.array([0.02]))]
    cases = [
        ("a\t1\t.\tA\tC\na\t2\t.\tC\tT\nb\t2\t.\ta\tC\na\t3\t.\tT\tA\n",
         r"v.vcf:4: REF A does not match the genome base G at b:2; 2 SNV alleles mismatch"),
        ("a\t1\t.\tA\tC\nc\t2\t.\tC\tT\nc\t1\t.\tC\tT\n", r"v.vcf:3: unknown chrom c \(no FASTA record of that name\)"),
        ("a\t10\t.\tC\tA\na\t11\t.\tC\tA\na\t12\t.\tC\tT\n", r"v.vcf:3: POS 11 is past the end of a \(2 SNV alleles in all\)"),
    ]
    vcf = tmp_path / "v.vcf"
    for text, msg in cases:
        vcf.write_text("#CHROM\tPOS\tID\tREF\tALT\n" + text)
        snvs = C.read_vcf(str(vcf))
        with pytest.raises(InputError, match=msg) as e1:
            B.burden(models, recs, snvs)
        with pytest.raises(InputError) as e2:
            C.count_mutations("NCN", recs, snvs)
        assert str(e1.value) == str(e2.value)
    # regions on a only: b is not scanned, so its REF is not checked
    vcf.write_text("#CHROM\tPOS\tID\tREF\tALT\nb\t2\t.\tA\tC\na\t2\t.\tC\tT\na\t5\t.\tA\tG\na\t9\t.\tA\tC\n")
    res = B.burden(models, recs, C.read_vcf(str(vcf)), [("a", 0, 6)])
    assert [B.STATUS[x] for x in res.status] == ["outside_regions", "counted", "counted", "outside_regions"]
    assert res.model_observed.tolist() == [[1], [1]] and res.observed.tolist() == [2]


def test_cli_end_to_end(tmp_path):
    """count_mutations writes -j files for three alts, kmerpapa fits each, burden runs on the fitted partitions."""
    from kmerpapa_b200 import burden as B
    from kmerpapa_b200 import cli
    from kmerpapa_b200 import count_mutations as C

    rng = np.random.default_rng(57)
    gen = "NNCNN"
    recs = _genome(rng, 5)
    fa = tmp_path / "g.fa"
    _write_fasta(fa, recs)
    lines = [x for x in _vcf_lines(rng, recs, 5, None, 60_000) if len(x[3]) == 1]
    lines = list({(c, p): (c, p, r, a) for c, p, r, a in lines}.values())   # one allele per position
    vcf = tmp_path / "v.vcf"
    _write_vcf(vcf, lines)
    with contextlib.redirect_stderr(io.StringIO()):
        assert C.main(["--pattern", gen, "--fasta", str(fa), "--vcf", str(vcf), "--strand", "both",
                       "--alt", "T", "A", "G", "--prefix", str(tmp_path / "out")]) == 0
    argv = ["--fasta", str(fa), "--vcf", str(vcf), "--strand", "both"]
    for alt in "TAG":
        part = tmp_path / f"C{alt}.partition"
        assert cli.main(["-j", str(tmp_path / f"out.{alt}.txt"), "-s", gen, "-c", "5", "-a", "1", "-o", str(part),
                         "--seed", "1", "--verbosity", "0"]) == 0
        argv += ["--model", f"C{alt}", alt, str(part)]
    out, err = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(out), contextlib.redirect_stderr(err):
        assert B.main(argv) == 0
    rows = out.getvalue().splitlines()
    assert rows[0] == ("chrom start end observed expected p_excess p_deficit observed.CT expected.CT n.CT "
                       "observed.CA expected.CA n.CA observed.CG expected.CG n.CG")
    assert [r.split()[0] for r in rows[1:]] == [name for name, _ in recs]
    counted = int(err.getvalue().split("counted ")[1].split()[0])
    assert sum(int(r.split()[3]) for r in rows[1:]) == counted > 0
    assert "ref_mismatch 0" in err.getvalue()
