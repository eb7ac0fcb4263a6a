"""Count observed SNVs against the expected counts of fitted models per region:
`python -m kmerpapa_b200.burden --fasta G --vcf V [--regions BED] [--strand forward|both] [--scale F]
--model NAME ALT FILE [--model NAME ALT FILE ...]`.

A kmerpapa model is fitted for one mutation type: a partition of the contexts of a general pattern (C>T on NNNNCNNNN,
say) with a rate per pattern.  A set of such models, one per type, predicts how many SNVs a region should carry given
its sequence.  This module counts the SNVs each model covers in every region, sums each model's expected count there
(apply_partition's), and gives the Poisson tails of the total observed count under the total expected one, in one pass
over the genome on the GPU (DESIGN §4e).

Conventions (those of apply_partition, DESIGN §4c, and count_mutations, DESIGN §4d, plus):
- --model NAME ALT FILE: FILE is a partition written by kmerpapa (either format); its general pattern gen is the LCA of
  its patterns; ALT is the alternative base it was fitted for, in the model's own orientation (count_mutations --alt).
  NAME labels the model's output columns.
- expected.NAME and n.NAME are apply_partition's `expected` and `n_contexts` of the model's partition alone, bit for
  bit.  observed.NAME counts the SNV alleles of the region that `count_mutations --pattern gen --alt ALT` gives the
  status counted: same windows, strand rule and REF check.
- Every model has the same k.  --strand both needs an odd k and, for every model, a centre letter that is not
  self-complementary.  ALT is one of ACGT and not a base of the model's centre letter.  Two models conflict, which is an
  error, when they can claim the same (forward window, ALT): ALT_a = ALT_b and gen_a intersects gen_b, or (--strand
  both) ALT_a = complement(ALT_b) and gen_a intersects revcomp(gen_b); two patterns intersect when their letters share a
  base at every position.  So each allele is counted by at most one model (asserted on the device result too), and
  `observed` counts no allele twice.  A CpG split (C>T on NNNNCGNNN next to C>T on NNNNCHNNN) is allowed.
- observed is the integer sum over the models, expected the left-to-right float64 sum of the expected.NAME in model
  order.  With lambda = F * expected (--scale F, finite and > 0, default 1): p_excess = P(X >= observed) =
  pdtrc(observed - 1, lambda), 1.0 when observed = 0; p_deficit = P(X <= observed) = pdtr(observed, lambda).
- Each SNV allele gets the first status that applies (STATUS): ref_mismatch (an error after the pass), outside_regions
  (not in the union of the regions, or on a record without regions), no_context, not_modelled (no model counts it),
  counted.

Every output is the same bits on every run, whatever the chunk size: the counts are integers and the expected counts
are apply_partition's.
"""
import argparse
import math
import sys
from collections import namedtuple

import numpy as np

from . import iupac
from .apply_partition import CHUNK_BASES, STRANDS, Applier, InputError, merge_intervals, read_fasta, read_regions
from .count_mutations import BAD_POSITION, REF_MISMATCH, check_args, read_vcf, snv_pass
from .score_partition import PartitionError, read_partition

STATUS = ("ref_mismatch", "outside_regions", "no_context", "not_modelled", "counted")   # the first three as in count_mutations
OUTSIDE_REGIONS, NO_CONTEXT, NOT_MODELLED, COUNTED = 1, 2, 3, 4
KP_SNV_NO_CONTEXT, KP_SNV_COUNTED = 2, 5   # kp_snv_counts status codes
NO_MODEL = 255                             # model id of an allele no model counts
_COMPLEMENT = {"A": "T", "C": "G", "G": "C", "T": "A"}

Model = namedtuple("Model", "name alt patterns rates")


def read_model(name, alt, path):
    """Model(name, ALT letter, patterns, float64 rates) from a partition file of the kmerpapa command."""
    with open(path) as f:
        patterns, rates = read_partition(f, path)
    return Model(name, alt, patterns, rates)


def revcomp(pattern):
    """The reverse complement of an IUPAC pattern (each letter's bases complemented)."""
    comp = {m: sum(1 << (3 - b) for b in range(4) if m >> b & 1) for m in range(16)}   # A<->T, C<->G on the masks
    return "".join(iupac.LETTER[comp[iupac.MASK[ch]]] for ch in reversed(pattern))


def intersects(p, q):
    """True when some k-mer lies in both patterns: their letters share a base at every position."""
    return all(iupac.MASK[a] & iupac.MASK[b] for a, b in zip(p, q))


def check_models(models, strand):
    """The checks of a model set that need no GPU (see the module docstring).  Returns the general pattern of each
    model.  Raises InputError naming the model, or both models of a conflict."""
    if strand not in STRANDS:
        raise InputError(f"strand must be one of {', '.join(STRANDS)}, not {strand!r}")
    if not models:
        raise InputError("give at least one --model")
    names = set()
    for m in models:
        if not m.name or any(ch.isspace() for ch in m.name):
            raise InputError(f"model name {m.name!r} must be non-empty and without white space")
        if m.name in names:
            raise InputError(f"two models are named {m.name}")
        names.add(m.name)
    gens = [iupac.lca_pattern(m.patterns) for m in models]
    k = len(gens[0])
    for m, gen in zip(models, gens):
        if len(gen) != k:
            raise InputError(f"model {m.name} has k = {len(gen)}, model {models[0].name} k = {k}: every model needs "
                             f"the same k")
        try:
            check_args(gen, strand, None)
        except InputError as e:
            raise InputError(f"model {m.name} ({gen}): {e}") from None
        if m.alt not in _COMPLEMENT:
            raise InputError(f"model {m.name}: ALT must be one letter of ACGT, not {m.alt!r}")
        if m.alt in iupac.CODE[gen[k // 2]]:
            raise InputError(f"model {m.name}: ALT {m.alt} is a base of the centre letter {gen[k // 2]} of {gen}")
    for a in range(len(models)):
        for b in range(a + 1, len(models)):
            ma, mb = models[a], models[b]
            same = ma.alt == mb.alt and intersects(gens[a], gens[b])
            flip = strand == "both" and ma.alt == _COMPLEMENT[mb.alt] and intersects(gens[a], revcomp(gens[b]))
            if same or flip:
                how = "on the same strand" if same else "on opposite strands"
                raise InputError(f"models {ma.name} ({gens[a]} >{ma.alt}) and {mb.name} ({gens[b]} >{mb.alt}) can count "
                                 f"the same SNV {how}")
    return gens


def check_scale(scale):
    if not (math.isfinite(scale) and scale > 0):
        raise InputError(f"--scale must be finite and > 0, got {scale!r}")


def poisson_tails(observed, lam):
    """(p_excess, p_deficit) per region: P(X >= o) and P(X <= o) for X ~ Poisson(lam), o = observed (int64)."""
    from scipy.special import pdtr, pdtrc

    o = np.asarray(observed, np.int64)
    lam = np.asarray(lam, np.float64)
    p_excess = np.where(o > 0, pdtrc(np.maximum(o - 1, 0).astype(np.float64), lam), 1.0)
    return p_excess, pdtr(o.astype(np.float64), lam)


class BurdenResult:
    """Per region (input order; per record without regions): chrom, start, end, observed (int64), expected (float64),
    p_excess, p_deficit, and per model [model, region]: model_observed (int64), model_expected (float64), model_n
    (int64).  status (uint8 per SNV of the input, STATUS codes), status_counts ({STATUS name: count}), skipped (non-SNV
    alleles), names (the model names)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


class _Classifier:
    """The per-record SNV state of burden (a count_mutations.snv_pass hook): every model's kp_snv_counts on each chunk,
    then one model id per allele and the per-region counts of the record (kp_snv_region_counts)."""

    def __init__(self, ap, snvs, plans, models, regions):
        torch = ap.torch
        self.ap, self.snvs, self.plans = ap, snvs, plans
        self.slots = [[0 if x == m.alt else -1 for x in "ACGT"] for m in models]
        self.counts = [torch.zeros(p.nkmer, dtype=torch.int64, device=ap.dev) for p in plans]   # not read
        self.regions = regions
        self.observed = {}   # record name -> int64 [nmodels, regions of the record]
        if regions is not None:
            self.by_chrom = {}
            for i, r in enumerate(regions):
                self.by_chrom.setdefault(r[0], []).append(i)

    def start(self, name, idx, L):
        torch, dev = self.ap.torch, self.ap.dev
        self.L = L
        self.pos = self.snvs.pos[idx]
        ra = self.snvs.ref[idx] | (self.snvs.alt[idx] << 2)
        self.dpos = torch.from_numpy(self.pos).to(dev)
        self.dra = torch.from_numpy(ra).to(dev)
        self.dstatus = torch.full((len(self.plans), len(idx)), BAD_POSITION, dtype=torch.uint8, device=dev)
        self.scanned = False

    def __call__(self, dseq, b0, b1, pos0, pos1, mask):
        self.scanned = True
        lo, hi = np.searchsorted(self.pos, [pos0, pos1])
        if hi > lo:
            for m, plan in enumerate(self.plans):
                plan.snv_counts(dseq, b0, b1 - b0, self.L, pos0, pos1, self.ap.both, self.dpos[lo:hi], self.dra[lo:hi],
                                self.slots[m], self.counts[m], self.dstatus[m, lo:hi])

    def finish(self, name):
        torch, st, nm = self.ap.torch, self.dstatus, len(self.plans)
        hit = st == KP_SNV_COUNTED
        if bool((hit.sum(0) > 1).any()):
            raise AssertionError("two models counted one SNV allele")
        model = torch.full((st.shape[1],), NO_MODEL, dtype=torch.uint8, device=self.ap.dev)
        for m in range(nm):
            model.masked_fill_(hit[m], m)
        code = lambda x: torch.tensor(x, dtype=torch.uint8, device=self.ap.dev)   # noqa: E731
        out = torch.where(model == NO_MODEL, code(NOT_MODELLED), code(COUNTED))
        out = torch.where(st[0] == KP_SNV_NO_CONTEXT, code(NO_CONTEXT), out)   # k, so the context, is every model's
        out = torch.where(st[0] == REF_MISMATCH, code(REF_MISMATCH), out)
        out = torch.where((st == BAD_POSITION).any(0), code(BAD_POSITION), out)
        if self.regions is None:
            ridx, bounds = None, np.array([[0, self.L]], np.int64)
        else:
            ridx = self.by_chrom.get(name, [])
            bounds = np.array([self.regions[i][1:3] for i in ridx], np.int64).reshape(-1, 2)
        obs = torch.empty((len(bounds), nm), dtype=torch.int64, device=self.ap.dev)
        self.plans[0].snv_region_counts(self.dpos, model, nm, torch.from_numpy(bounds).to(self.ap.dev), obs)
        self.observed[name] = obs.cpu().numpy().T
        status = out.cpu().numpy()
        if self.regions is not None:   # outside the union of the record's regions (the REF check comes first)
            us, ue = merge_intervals(bounds[:, 0], bounds[:, 1])
            j = np.searchsorted(us, self.pos, "right") - 1
            inside = (j >= 0) & (self.pos < ue[np.maximum(j, 0)])
            status[~inside & (status != REF_MISMATCH) & (status != BAD_POSITION)] = OUTSIDE_REGIONS
        return status


def burden(models, records, snvs, regions=None, strand="forward", scale=1.0, device=None, chunk_bases=CHUNK_BASES):
    """Observed and expected SNV counts of a model set per region, with their Poisson tails.  models: Model tuples
    (read_model); records: an iterable of (name, bytes) pairs; snvs: Snvs (count_mutations.read_vcf); regions: None (one
    row per record) or (chrom, start, end[, where]) tuples.  chunk_bases (a multiple of 65536) changes no result.
    Returns a BurdenResult; see the module docstring for the conventions.  Raises InputError on bad input and
    PartitionError when a model's patterns do not partition their general pattern."""
    models = [m._replace(alt=str(m.alt).upper()) for m in models]
    check_models(models, strand)
    check_scale(scale)
    ap = Applier(models[0].patterns, models[0].rates, regions, strand, device=device, chunk_bases=chunk_bases)
    plans = [ap.plan] + [ap.add_model(m.patterns, m.rates)[2] for m in models[1:]]
    hook = _Classifier(ap, snvs, plans, models, ap.regions)
    status, res = snv_pass(ap, records, snvs, hook)
    nm = len(models)
    model_observed = np.zeros((nm, len(res.chrom)), np.int64)
    cols = hook.by_chrom if regions is not None else {c: [j] for j, c in enumerate(res.chrom)}
    for name, obs in hook.observed.items():   # records that were not scanned have no SNV in a region
        model_observed[:, cols[name]] = obs
    expected = res.model_expected[0].copy()
    for m in range(1, nm):
        expected = expected + res.model_expected[m]
    observed = model_observed.sum(axis=0)
    p_excess, p_deficit = poisson_tails(observed, float(scale) * expected)
    hist = np.bincount(status, minlength=len(STATUS))
    return BurdenResult(chrom=res.chrom, start=res.start, end=res.end, observed=observed, expected=expected,
                        p_excess=p_excess, p_deficit=p_deficit, model_observed=model_observed,
                        model_expected=res.model_expected, model_n=res.model_n_contexts, status=status,
                        status_counts={s: int(hist[i]) for i, s in enumerate(STATUS)}, skipped=snvs.skipped,
                        names=[m.name for m in models])


def format_rows(res):
    """The output lines: header, then one row per region (floats printed with repr)."""
    head = "chrom start end observed expected p_excess p_deficit"
    head += "".join(f" observed.{n} expected.{n} n.{n}" for n in res.names)
    out = [head]
    per = list(zip(res.model_observed.T.tolist(), res.model_expected.T.tolist(), res.model_n.T.tolist()))
    for c, s, e, o, x, pe, pd, (mo, mx, mn) in zip(res.chrom, res.start.tolist(), res.end.tolist(), res.observed.tolist(),
                                                   res.expected.tolist(), res.p_excess.tolist(), res.p_deficit.tolist(), per):
        out.append(f"{c} {s} {e} {o} {x!r} {pe!r} {pd!r}" + "".join(f" {a} {b!r} {n}" for a, b, n in zip(mo, mx, mn)))
    return out


def get_parser():
    p = argparse.ArgumentParser(prog="python -m kmerpapa_b200.burden",
                                description="Observed SNVs against the expected counts of fitted kmerpapa models per "
                                            "region, with Poisson tails")
    p.add_argument("--fasta", required=True, metavar="G", help="FASTA file, plain or gzip (.gz)")
    p.add_argument("--vcf", required=True, metavar="V", help="VCF file, plain or gzip (.gz)")
    p.add_argument("--regions", metavar="BED", help="Regions 'chrom start end' (0-based, half-open); default: whole records")
    p.add_argument("--strand", choices=STRANDS, default="forward",
                   help="both: also the reverse-complement contexts (odd k, centre letters not self-complementary)")
    p.add_argument("--scale", type=float, default=1.0, metavar="F",
                   help="Poisson mean = F * expected (finite, > 0; default 1)")
    p.add_argument("--model", nargs=3, action="append", required=True, metavar=("NAME", "ALT", "FILE"),
                   help="A partition file written by kmerpapa, fitted for the alternative base ALT; NAME labels its "
                        "columns.  Repeat for every model")
    return p


def main(argv=None):
    args = get_parser().parse_args(argv)
    try:
        check_scale(args.scale)
        models = [read_model(name, alt.upper(), path) for name, alt, path in args.model]
        check_models(models, args.strand)
        regions = None
        if args.regions:
            with open(args.regions) as f:
                regions = read_regions(f, args.regions)
        snvs = read_vcf(args.vcf)
        res = burden(models, read_fasta(args.fasta), snvs, regions, args.strand, args.scale)
    except (OSError, InputError, PartitionError) as e:
        print(f"burden: error: {e}", file=sys.stderr)
        return 1
    sc = res.status_counts
    sys.stderr.write(f"burden: {len(snvs) + res.skipped} alleles, {res.skipped} not SNVs (skipped)\n")
    sys.stderr.write("burden: SNV alleles: " + ", ".join(f"{s} {sc[s]}" for s in STATUS) + "\n")
    sys.stdout.write("\n".join(format_rows(res)) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
