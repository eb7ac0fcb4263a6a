"""Count the k-mer contexts of mutations and of the genome they were called in:
`python -m kmerpapa_b200.count_mutations --pattern P --fasta G --vcf V [--regions BED] [--strand forward|both]
[--alt A [A ...]] --prefix OUT`.

kmerpapa fits a model from the k-mers around mutations (the positive set) and the k-mers of the genome (the
background).  This module makes both tables from a genome and a VCF on the GPU and writes them as the joint
`kmer n_pos n_bg` file that `kmerpapa -j` reads, one file OUT.<ALT>.txt per positive table (OUT.all.txt without
--alt).  The background pass is apply_partition's (kp_seq_scan with the one-pattern partition [P]); the SNVs of each
chunk are counted from the same device bytes by kp_snv_counts (DESIGN §4d).

Conventions (those of apply_partition, DESIGN §4c, plus):
- P is the general IUPAC pattern (kmerpapa's -s); k = len(P), c = k // 2.  The context of position i is the window
  seq[i - c : i - c + k]; a window of a byte other than A, C, G, T (either case), or one that leaves the record, is no
  context.  The background table is the one `apply_partition --kmer_counts` writes for the same pattern, FASTA,
  regions and strand.
- --strand both (odd k only) also counts reverse-complement windows.  It refuses a pattern whose centre letter is
  self-complementary (N S W B D H V: its bases and their complements overlap), so that at most one strand puts a
  given genome base at the centre and each SNV lands in at most one table entry.
- VCF (plain or .gz): lines starting with '#' and blank lines are skipped.  Columns are tab-separated: CHROM, POS
  (1-based: position i = POS - 1), ID, REF, ALT; further columns, FILTER included, are ignored.  Each comma-separated
  ALT is one allele.  An allele is an SNV when REF and ALT are each one letter of ACGT in either case; any other
  allele (indel, MNV, '*', '<...>') is skipped and counted.  A line with fewer than 5 columns, or a POS that is not an
  integer >= 1, is an error naming file:line.  Every line counts: duplicates are not merged.
- Each SNV allele gets the first status that applies, in this order (STATUS):
  ref_mismatch      the genome base is in ACGT and differs from REF (case-insensitive); an error after the pass;
  outside_regions   the position is not in the union of the regions;
  no_context        the position has no context;
  no_match          neither allowed strand's window matches P;
  alt_not_selected  the ALT (as counted below) is not one of --alt;
  counted.
  With regions given, a record with no region on it is not scanned: its SNVs are outside_regions and their REF is not
  checked.
- A counted SNV adds 1 to the forward window's k-mer index under ALT when the forward window matches, and otherwise
  (--strand both) to the reverse window's index under complement(ALT).  So with NNNNCNNNN --strand both --alt T, a
  G>A on the + strand counts as C>T.
- Both tables select positions with the same region bits, so n_pos <= n_bg holds for every k-mer whenever each
  (position, allele) appears once in the VCF.
- A CHROM with no FASTA record (also one whose lines have no SNV allele), a POS past the end of its record and a REF
  mismatch are errors after the FASTA pass.  A CHROM that is not valid UTF-8 is an error naming its line.

Every output is an integer count, the same whatever the chunk size or thread order.
"""
import argparse
import gzip
import sys

import numpy as np

from . import iupac
from .apply_partition import (CHUNK_BASES, MAXK, STRANDS, Applier, InputError, kmers_of_indices, read_fasta,
                              read_regions)

STATUS = ("ref_mismatch", "outside_regions", "no_context", "no_match", "alt_not_selected", "counted")   # KP_SNV_* codes
OUTSIDE_REGIONS = STATUS.index("outside_regions")
REF_MISMATCH = STATUS.index("ref_mismatch")
BAD_POSITION = 255                       # KP_SNV_BAD_POSITION: never left once a record is counted
SELF_COMPLEMENTARY = set("NSWBDHV")      # letters whose bases and their complements overlap
VCF_BLOCK = 1 << 24                      # bytes of VCF text parsed at a time

_CODE = np.full(256, 4, np.uint8)        # byte -> base code A, C, G, T = 0..3 (either case), 4 otherwise
for _i, _b in enumerate(b"ACGT"):
    _CODE[_b] = _CODE[_b + 32] = _i


class Snvs:
    """SNV alleles of a VCF in file order: chrom (int32 index into chroms), pos (int64, 0-based), ref and alt (uint8
    base codes A, C, G, T = 0..3), line (int64, 1-based VCF line); chroms = every CHROM of the file in first-seen order,
    whether or not its lines have SNVs, and chrom_line = the first line of each; skipped = the number of other alleles;
    name = the file name used in messages."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def __len__(self):
        return len(self.pos)


def _parse_block(b, line0, name, cidx, chrom_line, out):
    """Parse whole lines b (bytes ending in a newline) whose first line is line0 + 1; append the SNV arrays to out, new
    CHROM names to cidx (name -> index) and their first lines to chrom_line.  Returns the number of skipped alleles."""
    a = np.frombuffer(b, np.uint8)
    nl = np.flatnonzero(a == 10)
    starts = np.concatenate(([0], nl[:-1] + 1))
    ends = nl.copy()
    cr = (ends > starts) & (a[np.maximum(ends - 1, 0)] == 13)
    ends[cr] -= 1
    keep = (ends > starts) & (a[starts] != ord("#"))
    s, e, ln = starts[keep], ends[keep], line0 + 1 + np.flatnonzero(keep)
    if len(s) == 0:
        return 0
    tabs = np.concatenate((np.flatnonzero(a == 9), np.full(5, len(a) + 1)))
    ti = np.searchsorted(tabs, s)
    t = [tabs[ti + j] for j in range(5)]            # the first five tabs at or after each line start
    few = t[3] >= e
    if few.any():
        raise InputError(f"{name}:{ln[np.argmax(few)]}: expected at least 5 tab-separated columns "
                         f"(CHROM POS ID REF ALT)")
    # POS: 1 to 18 decimal digits, >= 1
    p0, p1 = t[0] + 1, t[1]
    w = p1 - p0
    bad = (w < 1) | (w > 18)
    pos = np.zeros(len(s), np.int64)
    for d in range(18):
        valid = d < w
        ch = a[np.where(valid, p1 - 1 - d, 0)].astype(np.int64) - 48
        bad |= valid & ((ch < 0) | (ch > 9))
        pos += np.where(valid & ~bad, ch * 10 ** d, 0)
    bad |= pos < 1
    if bad.any():
        j = int(np.argmax(bad))
        raise InputError(f"{name}:{ln[j]}: POS {b[p0[j]:p1[j]].decode(errors='replace')!r} is not an integer >= 1")
    # CHROM: names are looked up where they differ from the line before (compared byte for byte where lengths agree)
    c0, cl = s, t[0] - s
    new = np.ones(len(s), bool)
    cand = np.flatnonzero(cl[1:] == cl[:-1]) + 1
    lens = cl[cand]
    ramp = np.arange(lens.sum()) - np.repeat(np.cumsum(lens) - lens, lens)
    differ = a[np.repeat(c0[cand], lens) + ramp] != a[np.repeat(c0[cand - 1], lens) + ramp]
    new[cand] = np.bincount(np.repeat(np.arange(len(cand)), lens), weights=differ, minlength=len(cand)) > 0
    first = np.flatnonzero(new)
    ids = np.empty(len(first), np.int32)
    for x, j in enumerate(first):
        try:
            nm = b[c0[j]: c0[j] + cl[j]].decode()
        except UnicodeDecodeError:
            raise InputError(f"{name}:{ln[j]}: CHROM is not valid UTF-8") from None
        if nm not in cidx:
            cidx[nm] = len(cidx)
            chrom_line.append(int(ln[j]))
        ids[x] = cidx[nm]
    chrom = ids[np.cumsum(new) - 1]
    # REF, then the ALT alleles: the pieces of the ALT column between commas
    r0 = t[2] + 1
    ref_ok = (t[3] - r0 == 1) & (_CODE[a[r0]] < 4)
    a0, a1 = t[3] + 1, np.minimum(t[4], e)
    commas = np.flatnonzero(a == ord(","))
    li = np.searchsorted(a0, commas, "right") - 1
    inside = li >= 0
    inside[inside] = commas[inside] < a1[li[inside]]
    ci, cline = commas[inside], li[inside]
    S = np.concatenate((a0, ci + 1))
    which = np.concatenate((np.arange(len(s)), cline))
    o = np.argsort(S, kind="stable")
    S, which = S[o], which[o]
    E = np.sort(np.concatenate((ci, a1)))
    snv = (E - S == 1) & (_CODE[a[S]] < 4) & ref_ok[which]
    sel = which[snv]
    out["chrom"].append(chrom[sel])
    out["pos"].append(pos[sel] - 1)
    out["ref"].append(_CODE[a[r0[sel]]])
    out["alt"].append(_CODE[a[S[snv]]])
    out["line"].append(ln[sel])
    return int(len(S) - snv.sum())


def read_vcf(path, block=VCF_BLOCK):
    """The SNV alleles of a plain or gzip (.gz) VCF file (see the module docstring), as Snvs.  The text is parsed with
    numpy a block of whole lines at a time."""
    opener = gzip.open if path.endswith(".gz") else open
    cidx, chrom_line = {}, []
    out = {x: [] for x in ("chrom", "pos", "ref", "alt", "line")}
    skipped, nlines, tail = 0, 0, b""
    with opener(path, "rb") as f:
        while True:
            data = f.read(block)
            buf = tail + data
            if not data:
                if buf and not buf.endswith(b"\n"):
                    buf += b"\n"
                cut = len(buf)
            else:
                cut = buf.rfind(b"\n") + 1
            tail = buf[cut:]
            if cut:
                skipped += _parse_block(buf[:cut], nlines, path, cidx, chrom_line, out)
                nlines += buf.count(b"\n", 0, cut)
            if not data:
                break
    cat = lambda x, dt: np.concatenate(out[x]).astype(dt, copy=False) if out[x] else np.zeros(0, dt)   # noqa: E731
    return Snvs(chroms=list(cidx), chrom_line=np.array(chrom_line, np.int64), chrom=cat("chrom", np.int32), pos=cat("pos", np.int64), ref=cat("ref", np.uint8),
                alt=cat("alt", np.uint8), line=cat("line", np.int64), skipped=skipped, name=path)


def check_args(gen_pat, strand, alts):
    """The checks that need no GPU.  Returns (alt labels, alt_slot): one label per positive table ('all' without
    alts) and the table of each ALT base code (-1: not counted)."""
    if not gen_pat or any(ch not in iupac.MASK for ch in gen_pat):
        raise InputError(f"the pattern {gen_pat!r} must be a non-empty string of IUPAC letters")
    k = len(gen_pat)
    if k > MAXK:
        raise InputError(f"the pattern has length {k}; at most {MAXK} is supported")
    if strand not in STRANDS:
        raise InputError(f"strand must be one of {', '.join(STRANDS)}, not {strand!r}")
    if strand == "both":
        if k % 2 == 0:
            raise InputError(f"--strand both needs an odd k, so that the reverse context is centred on the same base "
                             f"(the pattern has k = {k})")
        if gen_pat[k // 2] in SELF_COMPLEMENTARY:
            raise InputError(f"--strand both needs a centre letter whose bases and their complements do not overlap "
                             f"(A C G T M K R Y); the pattern's centre is {gen_pat[k // 2]}")
    if alts is None:
        return ["all"], [0, 0, 0, 0]
    labels = [x.upper() for x in alts]
    if not labels or any(x not in ("A", "C", "G", "T") for x in labels):
        raise InputError(f"--alt takes letters of ACGT, got {' '.join(alts)}")
    if len(set(labels)) != len(labels):
        raise InputError(f"--alt names a letter twice: {' '.join(alts)}")
    slot = [-1] * 4
    for i, x in enumerate(labels):
        slot["ACGT".index(x)] = i
    return labels, slot


class CountResult:
    """gen_pat, k, alts (one label per positive table), background (int64 [nkmer]), positive (int64 [nalt, nkmer]),
    status (uint8 per SNV of the input, STATUS codes), status_counts ({STATUS name: count}), skipped (non-SNV
    alleles).  k-mers are in k-mer index order (iupac.matches(gen_pat))."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


class _Counter:
    """The per-record SNV state of count_mutations (a snv_pass hook): the record's SNVs sorted by position on the
    device and the on_chunk hook that counts those of each chunk."""

    def __init__(self, ap, snvs, slot, counts):
        self.ap, self.snvs, self.slot, self.counts = ap, snvs, slot, counts

    def start(self, name, idx, L):
        torch, dev = self.ap.torch, self.ap.dev
        self.L = L
        self.pos = self.snvs.pos[idx]
        ra = self.snvs.ref[idx] | (self.snvs.alt[idx] << 2)
        self.dpos = torch.from_numpy(self.pos).to(dev)
        self.dra = torch.from_numpy(ra).to(dev)
        self.dstatus = torch.full((len(idx),), BAD_POSITION, dtype=torch.uint8, device=dev)
        self.scanned = False

    def __call__(self, dseq, b0, b1, pos0, pos1, mask):
        self.scanned = True
        lo, hi = np.searchsorted(self.pos, [pos0, pos1])
        if hi > lo:
            self.ap.plan.snv_counts(dseq, b0, b1 - b0, self.L, pos0, pos1, self.ap.both, self.dpos[lo:hi], self.dra[lo:hi],
                                    self.slot, self.counts, self.dstatus[lo:hi], count_mask=mask)

    def finish(self, name):
        return self.dstatus.cpu().numpy()


def snv_pass(ap, records, snvs, hook):
    """The record loop of count_mutations and burden: stream records, an iterable of (name, bytes) pairs, through the
    Applier ap with the SNV alleles snvs (Snvs).  Per record, hook.start(name, idx, L) gets the indices of the record's
    SNVs that lie inside it, sorted by position; ap.record(name, seq, on_chunk=hook) scans the record, and the hook sets
    hook.scanned when a chunk was scanned; then hook.finish(name) returns the uint8 status of those SNVs.  The status
    codes are the caller's, except that REF_MISMATCH, OUTSIDE_REGIONS and BAD_POSITION mean what they mean in STATUS:
    SNVs of a record that is not scanned are OUTSIDE_REGIONS.  Returns (status of every SNV, ap.finish()).  Raises
    InputError after the pass for an unknown CHROM, a POS past the end of its record and a REF mismatch, in that order,
    and AssertionError when a scanned SNV is left BAD_POSITION."""
    n = len(snvs)
    status = np.full(n, BAD_POSITION, np.uint8)
    dc = np.diff(snvs.chrom)
    if ((dc > 0) | ((dc == 0) & (np.diff(snvs.pos) >= 0))).all():   # a sorted VCF: chrom indices are first-seen order
        order = np.arange(n)
    else:
        order = np.lexsort((snvs.pos, snvs.chrom))
    bounds = np.searchsorted(snvs.chrom[order], np.arange(len(snvs.chroms) + 1))
    chrom_of = {nm: i for i, nm in enumerate(snvs.chroms)}
    past_end, mismatch, seen = [], [], set()
    for name, seq in records:
        if isinstance(seq, str):
            seq = seq.encode("ascii")
        ci = chrom_of.get(name)
        idx = order[bounds[ci]: bounds[ci + 1]] if ci is not None else order[:0]
        seen.add(ci)
        L = len(seq)
        over = snvs.pos[idx] >= L
        if over.any():
            past_end.append(idx[over])
            idx = idx[~over]
        hook.start(name, idx, L)
        ap.record(name, seq, on_chunk=hook)
        if not hook.scanned:
            status[idx] = OUTSIDE_REGIONS
            continue
        st = hook.finish(name)
        if (st == BAD_POSITION).any():
            raise AssertionError("kp_snv_counts left an SNV of a scanned record uncounted")
        status[idx] = st
        bad = idx[st == REF_MISMATCH]
        if len(bad):
            j = bad[np.argmin(snvs.line[bad])]
            mismatch.append((int(snvs.line[j]), name, int(snvs.pos[j]), seq[snvs.pos[j]: snvs.pos[j] + 1].decode(), j))
    res = ap.finish()
    where = snvs.name
    lost = [i for i in range(len(snvs.chroms)) if i not in seen]
    if lost:   # every CHROM of the VCF, also one whose lines have no SNV allele
        i = min(lost, key=lambda i: snvs.chrom_line[i])
        raise InputError(f"{where}:{snvs.chrom_line[i]}: unknown chrom {snvs.chroms[i]} (no FASTA record of that name)")
    if past_end:
        sel = np.concatenate(past_end)
        j = sel[np.argmin(snvs.line[sel])]
        raise InputError(f"{where}:{snvs.line[j]}: POS {snvs.pos[j] + 1} is past the end of "
                         f"{snvs.chroms[snvs.chrom[j]]} ({len(sel)} SNV alleles in all)")
    if mismatch:
        line, name, pos, base, j = min(mismatch)
        total = int((status == REF_MISMATCH).sum())
        raise InputError(f"{where}:{line}: REF {'ACGT'[snvs.ref[j]]} does not match the genome base {base} at "
                         f"{name}:{pos + 1}; {total} SNV alleles mismatch in all (is the VCF from another genome build?)")
    return status, res


def count_mutations(gen_pat, records, snvs, regions=None, strand="forward", alts=None, device=None,
                    chunk_bases=CHUNK_BASES):
    """Background and positive k-mer counts of gen_pat over records, an iterable of (name, bytes) pairs, and the SNVs
    snvs (Snvs, as read_vcf returns).  regions: None (whole records) or (chrom, start, end[, where]) tuples; alts: None
    (one table of every SNV) or ALT letters (one table each).  chunk_bases (a multiple of 65536) changes no result.
    Returns a CountResult; see the module docstring for the conventions.  Raises InputError on bad input."""
    labels, slot = check_args(gen_pat, strand, alts)
    ap = Applier([gen_pat], [0.0], regions, strand, kmer_counts=True, device=device, chunk_bases=chunk_bases)
    torch = ap.torch
    counts = torch.zeros((len(labels), ap.plan.nkmer), dtype=torch.int64, device=ap.dev)
    status, res = snv_pass(ap, records, snvs, _Counter(ap, snvs, slot, counts))
    hist = np.bincount(status, minlength=len(STATUS))
    return CountResult(gen_pat=gen_pat, k=len(gen_pat), alts=labels, background=res.counts, positive=counts.cpu().numpy(),
                       status=status, status_counts={s: int(hist[i]) for i, s in enumerate(STATUS)},
                       skipped=snvs.skipped)


def write_joint(f, gen_pat, n_pos, n_bg):
    """`kmer n_pos n_bg` lines (io_utils.read_joint_kmer_counts reads them, kmerpapa -j) for the k-mers with a
    non-zero count, in k-mer index order."""
    nz = np.flatnonzero((n_pos > 0) | (n_bg > 0))
    for lo in range(0, len(nz), 1 << 20):
        part = nz[lo: lo + (1 << 20)]
        kmers = kmers_of_indices(gen_pat, part)
        f.write("".join(f"{km.decode()} {int(p)} {int(b)}\n" for km, p, b in zip(kmers, n_pos[part], n_bg[part])))


def get_parser():
    p = argparse.ArgumentParser(prog="python -m kmerpapa_b200.count_mutations",
                                description="k-mer counts of SNV contexts and of the genome background, written as "
                                            "kmerpapa -j input")
    p.add_argument("--pattern", required=True, metavar="P", help="General IUPAC pattern, e.g. NNNNCNNNN (kmerpapa -s)")
    p.add_argument("--fasta", required=True, metavar="G", help="FASTA file, plain or gzip (.gz)")
    p.add_argument("--vcf", required=True, metavar="V", help="VCF file, plain or gzip (.gz)")
    p.add_argument("--regions", metavar="BED", help="Regions 'chrom start end' (0-based, half-open); default: whole records")
    p.add_argument("--strand", choices=STRANDS, default="forward",
                   help="both: also count reverse-complement contexts (odd k, centre letter not self-complementary)")
    p.add_argument("--alt", nargs="+", metavar="A", help="One positive table per ALT letter; default: one of every SNV")
    p.add_argument("--prefix", required=True, metavar="OUT", help="Write OUT.<ALT>.txt (OUT.all.txt without --alt)")
    return p


def main(argv=None):
    args = get_parser().parse_args(argv)
    try:
        check_args(args.pattern, args.strand, args.alt)
        regions = None
        if args.regions:
            with open(args.regions) as f:
                regions = read_regions(f, args.regions)
        snvs = read_vcf(args.vcf)
        res = count_mutations(args.pattern, read_fasta(args.fasta), snvs, regions, args.strand, args.alt)
    except (OSError, InputError) as e:
        print(f"count_mutations: error: {e}", file=sys.stderr)
        return 1
    sc = res.status_counts
    err = sys.stderr
    err.write(f"count_mutations: {len(snvs) + res.skipped} alleles, {res.skipped} not SNVs (skipped)\n")
    err.write("count_mutations: SNV alleles: " + ", ".join(f"{s} {sc[s]}" for s in STATUS) + "\n")
    for i, label in enumerate(res.alts):
        path = f"{args.prefix}.{label}.txt"
        with open(path, "w") as f:
            write_joint(f, res.gen_pat, res.positive[i], res.background)
        over = int((res.positive[i] > res.background).sum())
        err.write(f"count_mutations: {path}: {int(res.positive[i].sum())} SNVs; {over} k-mers with n_pos > n_bg"
                  + (" (kmerpapa -j will refuse this file)" if over else "") + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
