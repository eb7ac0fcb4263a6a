"""Score a fitted pattern partition on k-mer counts: `python -m kmerpapa_b200.score_partition --partition F [F ...]`.

The kmerpapa command writes a model: IUPAC patterns that partition the k-mers, each with a rate `p_rate`.  This module
reads such a file (either of the two formats the command writes), checks on the GPU that its patterns form a partition
of their general pattern (their LCA), and gives the -2 log-likelihood of new counts under the model,

    LL_test = -2 * sum over patterns q of  xlogy(M_q, p_q) + xlog1py(U_q, -p_q),

with (M_q, U_q) the positive and negative counts of the k-mers of pattern q, summed in file order exactly as
score_utils.get_loss sums (so a partition scored on its own training data reproduces the `LL=` line of the run that
fitted it).  This is how kmerPaPa compares models: on held-out data, another sample, another penalty or k.  It replaces
the reference's papa.PatternPartition check.  There is no CPU path: the member enumeration, the owner table and the
scores are CUDA kernels (kp_partition_assign / kp_partition_score).
"""
import argparse
import sys

import numpy as np

from . import iupac
from .io_utils import downsize_contextD_device, read_input
from .score_utils import loss_from_terms

HEADER = ["pattern", "p_neg", "p_pos", "p_rate"]
LONG_HEADER = ["context", "c_neg", "c_pos", "c_rate", "pattern", "p_neg", "p_pos", "p_rate"]   # kmerpapa -l


class PartitionError(ValueError):
    pass


def read_partition(f, name="partition"):
    """(patterns, float64 rates) from a partition file of the kmerpapa command, in file order.  The -l format has one
    row per k-mer: its patterns are taken once each, in first-seen order.  Rates round-trip exactly (the command prints
    them with repr)."""
    rows = [(i, line.split()) for i, line in enumerate(f, 1) if line.strip()]
    if not rows:
        raise PartitionError(f"{name}: empty file")
    head = rows[0][1]
    if head not in (HEADER, LONG_HEADER):
        raise PartitionError(f"{name}: header is neither '{' '.join(HEADER)}' nor '{' '.join(LONG_HEADER)}'")
    long = head == LONG_HEADER
    col_pat, col_rate = len(head) - 4, len(head) - 1
    patterns, rates, seen = [], [], {}
    for lineno, row in rows[1:]:
        where = f"{name}:{lineno}"
        if len(row) != len(head):
            raise PartitionError(f"{where}: {len(row)} columns, expected {len(head)}")
        pat = row[col_pat]
        try:
            p = float(row[col_rate])
        except ValueError:
            raise PartitionError(f"{where}: p_rate {row[col_rate]!r} is not a number") from None
        if long and pat in seen:
            if seen[pat] != p:
                raise PartitionError(f"{where}: pattern {pat} appears with two rates ({seen[pat]!r} and {p!r})")
            continue
        seen[pat] = p
        bad = [c for c in pat if c not in iupac.MASK]
        if bad:
            raise PartitionError(f"{where}: pattern {pat} has a letter that is not IUPAC: {bad[0]!r}")
        if patterns and len(pat) != len(patterns[0]):
            raise PartitionError(f"{where}: pattern {pat} has length {len(pat)}, the first pattern {len(patterns[0])}")
        if not 0.0 < p < 1.0:
            raise PartitionError(f"{where}: rate {p!r} of pattern {pat} is not in (0, 1)")
        patterns.append(pat)
        rates.append(p)
    if not patterns:
        raise PartitionError(f"{name}: no patterns")
    return patterns, np.array(rates, dtype=np.float64)


def _letters(strings):
    """uint8 [n, k] ASCII codes of strings of one length."""
    k = len(strings[0])
    return np.frombuffer("".join(strings).encode("ascii"), dtype=np.uint8).reshape(len(strings), k)


def pattern_numbers(patterns, gen_pat):
    """Dense pattern numbers (iupac.PatternEnumeration) of many sub-patterns of gen_pat at once."""
    letters = _letters(patterns)
    PE = iupac.PatternEnumeration(gen_pat)
    num = np.zeros(len(patterns), dtype=np.uint64)
    for i, c in enumerate(gen_pat):
        lut = np.zeros(256, dtype=np.uint64)
        for d, x in enumerate(iupac.PERM[c]):
            lut[ord(x)] = d
        num += lut[letters[:, i]] * np.uint64(PE.weight[i])
    return num


def covering(patterns, kmer):
    """Indices of the patterns that contain kmer, in file order."""
    lut = np.zeros(256, dtype=np.uint8)
    for c, m in iupac.MASK.items():
        lut[ord(c)] = m
    masks = lut[_letters(patterns)]
    want = lut[np.frombuffer(kmer.encode("ascii"), dtype=np.uint8)]
    return np.flatnonzero((masks & want).all(axis=1))


class PartitionScore:
    """Result of score(): the partition, its general pattern, per-pattern test counts (M, U) and terms t, LL_test, and,
    when asked for, the owner of every k-mer (index into patterns, in iupac.matches(gen_pat) order) and the k-mer
    counts."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def assign(patterns, device=None):
    """Check on the GPU that `patterns` partition their general pattern (their LCA).  Returns (gen_pat, plan, patnums,
    owner): the lite plan of the general pattern, the dense pattern numbers and the device owner table of
    PartitionPlan.partition_assign.  Raises PartitionError naming the first k-mer that is covered twice or not at all."""
    from .engine import get_plan

    gen_pat = iupac.lca_pattern(patterns)
    plan = get_plan(gen_pat, device, lite=True)
    patnums = pattern_numbers(patterns, gen_pat)
    owner, conflict, uncovered = plan.partition_assign(patnums)
    if conflict is not None:
        kmer = iupac.kmer_of_index(gen_pat, conflict)
        a, b = covering(patterns, kmer)[:2]
        raise PartitionError(f"the patterns overlap: k-mer {kmer} is in pattern {a + 1} ({patterns[a]}) and in pattern "
                             f"{b + 1} ({patterns[b]})")
    if uncovered is not None:
        raise PartitionError(f"the patterns leave a gap: k-mer {iupac.kmer_of_index(gen_pat, uncovered)} of their general "
                             f"pattern {gen_pat} is in none of them")
    return gen_pat, plan, patnums, owner


def score(patterns, rates, contextD, device=None, per_kmer=False):
    """Check that `patterns` partition their general pattern and score the counts contextD {kmer: (n_pos, n_neg)}.
    Longer k-mers are collapsed around their centre to the patterns' length (as kmerpapa --test_smaller_k does);
    k-mers of the partition that contextD lacks count as zero.  Raises PartitionError naming the first k-mer that is
    covered twice or not at all, or a test k-mer outside the general pattern."""
    from .algorithms.bottum_up_array_w_numba import kmer_arrays

    gen_pat, plan, patnums, owner = assign(patterns, device)
    k = len(gen_pat)
    if not contextD:
        raise PartitionError("the input has no k-mers")
    have = len(next(iter(contextD)))
    if have < k:
        raise PartitionError(f"the input k-mers have length {have}, shorter than the partition's patterns ({k})")
    if have > k:
        contextD, _ = downsize_contextD_device(contextD, iupac.lca_pattern(list(contextD)), k)
    codes, pos, neg = kmer_arrays(contextD)
    outside = (codes & ~np.uint64(iupac.kmer_code(gen_pat))) != 0
    if outside.any():
        kmers = list(contextD)
        first = min(kmers[i] for i in np.flatnonzero(outside))
        raise PartitionError(f"test k-mer {first} is outside the partition's general pattern {gen_pat}")
    kM, kU = plan.pack_counts(codes, pos, neg, name="score_k")
    M, U, t = plan.partition_score(patnums, rates, kM, kU)
    res = PartitionScore(patterns=patterns, rates=rates, gen_pat=gen_pat, k=k, M=M, U=U, t=t, LL=loss_from_terms(t))
    if per_kmer:
        res.owner = owner.cpu().numpy().view(np.uint32)
        res.kmerM = kM[: plan.nkmer].cpu().numpy()
        res.kmerU = kU[: plan.nkmer].cpu().numpy()
    return res


def get_parser():
    p = argparse.ArgumentParser(prog="python -m kmerpapa_b200.score_partition",
                                description="-2 log-likelihood of k-mer counts under fitted kmerpapa partitions")
    p.add_argument("--partition", nargs="+", required=True, metavar="F",
                   help="Partition file(s) written by kmerpapa (with or without -l)")
    p.add_argument("-p", "--positive", type=argparse.FileType("r"), help="File with k-mer counts in positive set")
    p.add_argument("-n", "--negative", type=argparse.FileType("r"),
                   help="File with k-mer counts in negative set. Longer k-mers are collapsed around their centre to the "
                        "length of the positive k-mers.")
    p.add_argument("-b", "--background", type=argparse.FileType("r"),
                   help="File with k-mer counts in background set (positive and negative regions together). Longer "
                        "k-mers are collapsed around their centre to the length of the positive k-mers.")
    p.add_argument("-j", "--joint_context_counts", type=argparse.FileType("r"),
                   help="File with three columns: k-mer, positive count, background count. Replaces -p/-b.")
    p.add_argument("-s", "--super_pattern", type=str, help="Only k-mers matching this IUPAC pattern are used.")
    p.add_argument("--per_pattern", type=argparse.FileType("w"), metavar="FILE",
                   help="Write 'pattern p_rate t_neg t_pos LL' per pattern (one partition only)")
    p.add_argument("--per_kmer", type=argparse.FileType("w"), metavar="FILE",
                   help="Write 'context c_neg c_pos pattern p_rate' per k-mer of the general pattern (one partition only)")
    return p


def main(argv=None):
    parser = get_parser()
    args = parser.parse_args(argv)
    if (args.per_pattern or args.per_kmer) and len(args.partition) > 1:
        parser.error("--per_pattern and --per_kmer take a single --partition file")
    try:
        contextD, _, _ = read_input(args, args.super_pattern)
        rows = []
        for path in args.partition:
            with open(path) as f:
                patterns, rates = read_partition(f, path)
            res = score(patterns, rates, contextD, per_kmer=args.per_kmer is not None)
            rows.append((path, res))
    except (AssertionError, PartitionError) as e:
        print(f"score_partition: error: {e}", file=sys.stderr)
        return 1
    print("partition", "k", "n_patterns", "LL_test")
    for path, res in rows:
        print(path, res.k, len(res.patterns), res.LL)
    if len(rows) == 1:
        print(f"LL={rows[0][1].LL}", file=sys.stderr)
    res = rows[0][1]
    if args.per_pattern:
        print("pattern", "p_rate", "t_neg", "t_pos", "LL", file=args.per_pattern)
        for pat, p, m, u, t in zip(res.patterns, res.rates, res.M, res.U, res.t):
            print(pat, float(p), int(u), int(m), float(-2 * t), file=args.per_pattern)
        args.per_pattern.close()
    if args.per_kmer:
        print("context", "c_neg", "c_pos", "pattern", "p_rate", file=args.per_kmer)
        for kmer, o, m, u in zip(iupac.matches(res.gen_pat), res.owner, res.kmerM, res.kmerU):
            print(kmer, int(u), int(m), res.patterns[o], float(res.rates[o]), file=args.per_kmer)
        args.per_kmer.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
