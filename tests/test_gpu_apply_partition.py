"""Applying fitted partitions along sequences on the GPU (kmerpapa_b200.apply_partition, kp_seq_scan / kp_region_sums)
against a numpy reference kept here: sliding windows over the record, per-position lookup tables and the owner table of
a host assignment."""
import contextlib
import io
import json
import math
import os
import zlib

import numpy as np
import pytest
from numpy.lib.stride_tricks import sliding_window_view

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
P = 1 << 16
# Region sums against math.fsum.  A region's sum is a tree of float64 additions of non-negative terms: in a piece,
# a thread adds its <= 256 positions in order (255 roundings; the first add is to 0), a warp adds its 32 thread sums by
# a 5-level shuffle tree, the block adds its 8 warp sums in order (7 roundings), and the region adds its m clipped
# piece sums left to right (m - 1 roundings).  Every term passes through at most h = 255 + 5 + 7 + m - 1 roundings, so
# |sum - exact| <= h u / (1 - h u) * sum of terms, and fsum adds one more rounding of the exact sum.
TREE_ROUNDINGS = 255 + 5 + 7


def _bound(total, npieces):
    h = TREE_ROUNDINGS + max(npieces, 1) - 1
    return (h * U / (1 - h * U) + U) * total


# ---- host reference ------------------------------------------------------------------------------------------------
LUT = np.full(256, 4, np.uint8)
for _i, _b in enumerate(b"ACGT"):
    LUT[_b] = LUT[_b + 32] = _i


def _random_partition(gen, nsplit, rng):
    """Leaves of a random split tree in random file order (a leaf and one of its multi-letter positions are drawn at
    random and the letter is cut into two non-empty subsets)."""
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


def _offsets(gen):
    """[k, 5] k-mer index contribution of base code (A, C, G, T, other) at each position, -1 where not allowed."""
    from kmerpapa_b200.iupac import CODE

    off, w = np.full((len(gen), 5), -1, np.int64), 1
    for j, g in enumerate(gen):
        for b, base in enumerate("ACGT"):
            if base in CODE[g]:
                off[j, b] = CODE[g].index(base) * w
        w *= len(CODE[g])
    return off, w


def _host_owner(gen, patterns):
    """Owner pattern of every k-mer index, from the patterns' members."""
    from kmerpapa_b200.iupac import CODE

    off, nk = _offsets(gen)
    owner = np.full(nk, -1, np.int64)
    for q, pat in enumerate(patterns):
        idx = np.zeros(1, np.int64)
        for j in reversed(range(len(gen))):
            part = np.array([off[j, b] for b, base in enumerate("ACGT") if base in CODE[pat[j]]], np.int64)
            idx = (part[:, None] + idx[None, :]).ravel()
        assert (owner[idx] == -1).all()
        owner[idx] = q
    assert (owner >= 0).all()
    return owner


def _host_record(gen, owner, rates, seq, both):
    """(rate float64 [L] with NaN where no context, matches per position, forward k-mer index or -1, reverse or -1)."""
    k, c, L = len(gen), len(gen) // 2, len(seq)
    rate, nmatch = np.full(L, np.nan), np.zeros(L, np.int64)
    kf_pos, kr_pos = np.full(L, -1, np.int64), np.full(L, -1, np.int64)
    if L < k:
        return rate, nmatch, kf_pos, kr_pos
    off, _ = _offsets(gen)
    W = sliding_window_view(LUT[np.frombuffer(seq, np.uint8)], k)   # window starting at i - c
    ctx = (W < 4).all(1)
    cols = np.arange(k)

    def side(codes):
        o = off[cols, codes]
        m = ctx & (o >= 0).all(1)
        kidx = np.where(m, o.sum(1), 0)
        return m, kidx, np.where(m, rates[owner[kidx]], 0.0)

    mf, kf, pf = side(W)
    if both:
        mr, kr, pr = side(np.where(W < 4, 3 - W, 4)[:, ::-1])
    else:
        mr, kr, pr = np.zeros_like(mf), kf, np.zeros_like(pf)
    sl = slice(c, c + len(ctx))
    rate[sl] = np.where(ctx, pf + pr, np.nan)
    nmatch[sl] = mf.astype(np.int64) + mr
    kf_pos[sl] = np.where(mf, kf, -1)
    kr_pos[sl] = np.where(mr, kr, -1)
    return rate, nmatch, kf_pos, kr_pos


def _genome(rng, total, k, plant=None):
    """Seeded records: random bases with N runs, other IUPAC letters, soft-masked stretches, records shorter than k
    and exactly k long, an empty record and one record longer than two pieces.  plant: a general pattern of which
    random k-mers and their reverse complements are written at random places (a long pattern has few chance matches)."""
    from kmerpapa_b200.iupac import CODE
    sizes = [0, 1, max(k - 1, 0), k, k + 1, 37, 3 * P + 17]
    while sum(sizes) < total:
        sizes.append(int(rng.integers(1000, 400000)))
    recs = []
    for i, n in enumerate(sizes):
        s = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=n)
        for _ in range(n // 20000):
            a = int(rng.integers(n))
            kind = rng.integers(3)
            if kind == 0:
                s[a: a + int(rng.integers(1, 2000))] = ord("N")
            elif kind == 1:
                s[a] = rng.choice(np.frombuffer(b"RYKMSWBDHVn-", np.uint8))
            else:
                b = a + int(rng.integers(1, 5000))
                s[a:b] = s[a:b] | 0x20
        if plant is not None and n > 4 * k:
            for _ in range(n // 500):
                km = np.array([ord(CODE[g][int(rng.integers(len(CODE[g])))]) for g in plant], np.uint8)
                if rng.integers(2):
                    km = np.frombuffer(bytes(km).translate(bytes.maketrans(b"ACGT", b"TGCA"))[::-1], np.uint8)
                a = int(rng.integers(n - k))
                s[a: a + k] = km
        recs.append((f"r{i}", s.tobytes()))
    return recs


def _regions(rng, recs, n):
    """Regions at record ends, overlapping ones, one without a context, whole records and random ones over many pieces."""
    out = []
    for name, s in recs:
        L = len(s)
        if L == 0:
            continue
        out += [(name, 0, L), (name, 0, 1), (name, L - 1, L), (name, max(0, L - 5), L)]
        if L > 2 * P:
            out += [(name, P - 3, 2 * P + 5), (name, P, 2 * P), (name, 1, L - 1)]
    for _ in range(n):
        name, s = recs[int(rng.integers(len(recs)))]
        if len(s) < 2:
            continue
        a = int(rng.integers(len(s) - 1))
        out.append((name, a, int(min(len(s), a + rng.integers(1, 150000)))))
    out.append(("r0" if len(recs[0][1]) else recs[1][0], 0, 1))
    return out


def _host_apply(gen, patterns, rates, recs, regions, both):
    owner = _host_owner(gen, patterns)
    by = {name: _host_record(gen, owner, rates, s, both) for name, s in recs}
    return owner, by


def _check_regions(res, by, regions):
    for i, (name, a, b) in enumerate(regions):
        rate, nmatch = by[name][0][a:b], by[name][1][a:b]
        r = np.nan_to_num(rate)
        assert res.n_contexts[i] == nmatch.sum(), (name, a, b)
        want = math.fsum(r)
        npieces = (b - 1) // P - a // P + 1
        assert abs(res.expected[i] - want) <= _bound(want, npieces), (name, a, b, res.expected[i], want)
        if not (r > 0).any():
            assert res.expected[i] == 0.0


GENS = [("A", 0, False), ("SWN", 6, False), ("NRN", 6, True), ("NNRNCNYNN", 80, False), ("NNRNCNYNN", 80, True),
        ("NNNNCNNNN", 200, True), ("NNNNCNNNN", 200, False), ("NNNNNNNNNNNNN", 400, True), ("NNNNNNNNNNNN", 300, False),
        ("ACGTTGCANNAACCGGTTRY", 5, False), ("ACGTTGCANNAACCGGTTRYC", 5, True)]


@pytest.mark.parametrize("gen,nsplit,both", GENS)
def test_tracks_counts_and_region_sums_against_host(gen, nsplit, both):
    from kmerpapa_b200 import apply_partition as A

    rng = np.random.default_rng(zlib.crc32(f"{gen} {both}".encode()))
    k = len(gen)
    patterns = _random_partition(gen, nsplit, rng)
    rates = rng.uniform(1e-6, 0.3, len(patterns))
    recs = _genome(rng, 1_500_000, k, plant=gen if k > 16 else None)
    regions = _regions(rng, recs, 300)
    res = A.apply(patterns, rates, recs, regions=regions, strand="both" if both else "forward", track=True,
                  kmer_counts=True)
    owner, by = _host_apply(gen, patterns, rates, recs, regions, both)
    assert res.gen_pat == gen
    for name, s in recs:
        assert np.array_equal(res.tracks[name].view(np.uint32), by[name][0].astype(np.float32).view(np.uint32)), name
    _check_regions(res, by, regions)
    # counts over the union of the regions
    want = np.zeros(len(owner), np.int64)
    for name, s in recs:
        use = np.zeros(len(s), bool)
        for rn, a, b in regions:
            if rn == name:
                use[a:b] = True
        for kp in by[name][2:]:
            want += np.bincount(kp[use & (kp >= 0)], minlength=len(owner))
    assert np.array_equal(res.counts, want)


def test_whole_records_identity_and_written_counts(tmp_path):
    """Without regions: one row per record, and sum(count * rate) = sum(expected), sum(counts) = sum(n_contexts); the
    written --kmer_counts file reads back as the same table."""
    from kmerpapa_b200 import apply_partition as A
    from kmerpapa_b200.io_utils import read_dict
    from kmerpapa_b200 import iupac

    rng = np.random.default_rng(11)
    gen = "NNNNCNNNN"
    patterns = _random_partition(gen, 150, rng)
    rates = rng.uniform(1e-6, 0.3, len(patterns))
    recs = _genome(rng, 1_000_000, 9)
    res = A.apply(patterns, rates, recs, strand="both", kmer_counts=True)
    owner, by = _host_apply(gen, patterns, rates, recs, None, True)
    assert res.chrom == [n for n, _ in recs] and res.start.tolist() == [0] * len(recs)
    assert res.end.tolist() == [len(s) for _, s in recs]
    _check_regions(res, by, [(n, 0, len(s)) for n, s in recs])   # one row per record, the empty one too
    assert res.counts.sum() == res.n_contexts.sum()
    total = math.fsum(res.expected)
    npieces = max((len(s) + P - 1) // P for _, s in recs)
    ident = math.fsum(res.counts * rates[owner])
    assert abs(ident - total) <= _bound(total, npieces) + 2 * U * total
    f = io.StringIO()
    A.write_kmer_counts(f, gen, res.counts)
    table, _ = read_dict(io.StringIO(f.getvalue()), None)
    kmers = iupac.matches(gen)
    assert table == {kmers[i]: int(res.counts[i]) for i in np.flatnonzero(res.counts)}


def test_deterministic_for_runs_and_chunk_sizes():
    from kmerpapa_b200 import apply_partition as A

    rng = np.random.default_rng(5)
    gen = "NNRNCNYNN"
    patterns = _random_partition(gen, 60, rng)
    rates = rng.uniform(1e-6, 0.3, len(patterns))
    recs = _genome(rng, 2_000_000, 9)
    regions = _regions(rng, recs, 500)
    runs = [A.apply(patterns, rates, recs, regions=regions, strand="both", track=True, kmer_counts=True, chunk_bases=cb)
            for cb in (A.CHUNK_BASES, A.CHUNK_BASES, P, 3 * P)]
    for r in runs[1:]:
        assert r.expected.tobytes() == runs[0].expected.tobytes()
        assert np.array_equal(r.n_contexts, runs[0].n_contexts)
        assert np.array_equal(r.counts, runs[0].counts)
        for name in r.tracks:
            assert r.tracks[name].tobytes() == runs[0].tracks[name].tobytes()


def test_regions_errors_and_duplicates():
    from kmerpapa_b200 import apply_partition as A

    recs = [("a", b"ACGTACGTAC"), ("b", b"AC")]
    with pytest.raises(A.InputError, match=r"r.bed:7: end 11 is past the end of a \(length 10\)"):
        A.apply(["NNN"], [0.1], recs, regions=[("a", 0, 11, "r.bed:7")])
    with pytest.raises(A.InputError, match=r"r.bed:2: unknown chrom c"):
        A.apply(["NNN"], [0.1], recs, regions=[("a", 0, 5, "r.bed:1"), ("c", 0, 1, "r.bed:2")])
    with pytest.raises(A.InputError, match="duplicate record name a"):
        A.apply(["NNN"], [0.1], recs + [("a", b"A")])


def _run(argv):
    from kmerpapa_b200 import apply_partition

    out, err = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(out), contextlib.redirect_stderr(err):
        rc = apply_partition.main(argv)
    return rc, out.getvalue(), err.getvalue()


def _write_fasta(path, recs, width=60):
    with open(path, "wb") as f:
        for name, s in recs:
            f.write(b">" + name.encode() + b" synthetic\n")
            for i in range(0, len(s), width):
                f.write(s[i: i + width] + b"\n")


def test_cli_recorded_partition(tmp_path):
    """The partition a recorded kmerpapa run printed, applied from the command line: rows, track files and errors."""
    g = json.load(open(os.path.join(GOLDEN, "cli_7mers_single.json")))
    part = tmp_path / "partition.txt"
    part.write_text(g["stdout"])
    from kmerpapa_b200 import iupac
    from kmerpapa_b200.score_partition import read_partition

    patterns, rates = read_partition(open(part))
    gen = iupac.lca_pattern(patterns)
    rng = np.random.default_rng(3)
    recs = _genome(rng, 300_000, 7)[:12]
    fa = tmp_path / "g.fa"
    _write_fasta(fa, recs)
    bed = tmp_path / "r.bed"
    regions = _regions(rng, recs, 40)
    bed.write_text("track name=test\n" + "".join(f"{n}\t{a}\t{b}\tx\n" for n, a, b in regions))
    tdir = tmp_path / "tracks"
    rc, out, err = _run(["--partition", str(part), "--fasta", str(fa), "--regions", str(bed), "--track", str(tdir),
                         "--strand", "both", "--kmer_counts", str(tmp_path / "counts.txt")])
    assert rc == 0, err
    lines = out.splitlines()
    assert lines[0] == "chrom start end n_contexts expected"
    owner, by = _host_apply(gen, patterns, rates, recs, regions, True)
    res = type("Rows", (), {})()
    rows = [l.split() for l in lines[1:]]
    assert [(r[0], int(r[1]), int(r[2])) for r in rows] == regions
    res.n_contexts = np.array([int(r[3]) for r in rows])
    res.expected = np.array([float(r[4]) for r in rows])
    assert [r[4] for r in rows] == [repr(float(x)) for x in res.expected]   # printed with repr, round-trips
    _check_regions(res, by, regions)
    for name, s in recs:
        t = np.fromfile(tdir / (name + ".f32"), dtype="<f4")
        assert np.array_equal(t.view(np.uint32), by[name][0].astype(np.float32).view(np.uint32)), name
    # errors come out as `apply_partition: error: ...` with exit code 1
    bad = tmp_path / "bad.bed"
    bad.write_text("r1 0 1\nnope 0 5\n")
    rc, out, err = _run(["--partition", str(part), "--fasta", str(fa), "--regions", str(bad)])
    assert rc == 1 and err == f"apply_partition: error: {bad}:2: unknown chrom nope (no record of that name)\n"
    over = tmp_path / "over.txt"
    over.write_text("pattern p_neg p_pos p_rate\n" + f"{gen} 1 1 0.5\n" + f"{patterns[0]} 1 1 0.5\n")
    rc, out, err = _run(["--partition", str(over), "--fasta", str(fa)])
    assert rc == 1 and err.startswith("apply_partition: error: the patterns overlap: k-mer ")


def test_end_to_end_counts_fit_and_apply(tmp_path):
    """Background counts of a synthetic genome feed kmerpapa with seeded positive counts; the fitted partition is applied
    to the same genome and sum(count * rate) = sum(expected) holds for it."""
    from kmerpapa_b200 import apply_partition as A
    from kmerpapa_b200 import cli
    from kmerpapa_b200.io_utils import read_dict
    from kmerpapa_b200.score_partition import read_partition

    rng = np.random.default_rng(21)
    recs = _genome(rng, 2_000_000, 5)
    fa = tmp_path / "g.fa"
    _write_fasta(fa, recs)
    seed_part = ["NNNNN"]
    (tmp_path / "seed.txt").write_text("pattern p_neg p_pos p_rate\nNNNNN 1 1 0.5\n")
    bg = tmp_path / "bg.txt"
    rc, out, err = _run(["--partition", str(tmp_path / "seed.txt"), "--fasta", str(fa), "--kmer_counts", str(bg)])
    assert rc == 0, err
    table, _ = read_dict(open(bg), None)
    kmers = sorted(table)
    true_rate = {km: 0.002 * (1 + 5 * (km[2] == "C") + 3 * (km[1] == "T")) for km in kmers}
    pos = tmp_path / "pos.txt"
    pos.write_text("".join(f"{km} {rng.binomial(table[km], true_rate[km])}\n" for km in kmers))
    fitted = tmp_path / "fitted.txt"
    assert cli.main(["-p", str(pos), "-b", str(bg), "-c", "5", "-a", "1", "-o", str(fitted), "--seed", "1",
                     "--verbosity", "0"]) == 0
    patterns, rates = read_partition(open(fitted))
    assert len(patterns) > 1 and seed_part != patterns
    res = A.apply(patterns, rates, A.read_fasta(str(fa)), kmer_counts=True)
    from kmerpapa_b200 import iupac

    gen = iupac.lca_pattern(patterns)
    owner = _host_owner(gen, patterns)
    total = math.fsum(res.expected)
    ident = math.fsum(res.counts * rates[owner])
    npieces = max((len(s) + P - 1) // P for _, s in recs)
    assert abs(ident - total) <= _bound(total, npieces) + U * total
    assert res.counts.sum() == res.n_contexts.sum() == sum(table.values())
