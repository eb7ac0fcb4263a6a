"""IUPAC tables of the host side.

Restated from the reference's src/kmerpapa/pattern_utils.py: `code` (:5-19), `perm_code` (:86-100),
dense pattern numbering (:237-266), `matches` (:415-429), `LCA_pattern_of_kmers` (:382-388),
`pattern_level` (:219-230), `pattern_max` (:587-599).  Letters are handled as nucleotide-subset
masks A=1, C=2, G=4, T=8.
"""
MASK = {"A": 1, "C": 2, "G": 4, "T": 8, "R": 5, "Y": 10, "S": 6, "W": 9, "K": 12, "M": 3, "B": 14, "D": 13, "H": 11,
        "V": 7, "N": 15}
LETTER = {m: c for c, m in MASK.items()}
# nucleotides of a letter in the reference's order (note S = G,C)
CODE = {"A": "A", "C": "C", "G": "G", "T": "T", "R": "AG", "Y": "CT", "S": "GC", "W": "AT", "K": "GT", "M": "AC",
        "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGT"}
# sub-letters of a general letter in digit order
PERM = {"A": "A", "C": "C", "G": "G", "T": "T", "R": "AGR", "Y": "CTY", "S": "GCS", "W": "ATW", "K": "GTK",
        "M": "ACM", "B": "CGTSYKB", "D": "AGTRWKD", "H": "ACTMWYH", "V": "ACGMRSV", "N": "ACGTRYSWKMBDHVN"}
NUCLEOTIDES = "ACGT"


def pattern_level(pattern):
    return sum(len(CODE[c]) - 1 for c in pattern)


def pattern_max(gen_pat):
    n = 1
    for c in gen_pat:
        n *= len(PERM[c])
    return n


def matches(pattern):
    """All k-mers of a pattern, first position fastest (the reference's enumeration order)."""
    out = [""]
    for ch in reversed(pattern):
        out = [b + s for s in out for b in CODE[ch]]
    return out


def kmer_of_index(pattern, idx):
    """matches(pattern)[idx] without the list: the k-mer index is mixed radix over the positions, first fastest."""
    out = []
    for ch in pattern:
        bases = CODE[ch]
        out.append(bases[idx % len(bases)])
        idx //= len(bases)
    return "".join(out)


def lca_pattern(kmers):
    """Smallest pattern covering all the given k-mers."""
    k = len(kmers[0])
    masks = [0] * k
    for km in kmers:
        for i, c in enumerate(km):
            masks[i] |= MASK[c]
    return "".join(LETTER[m] for m in masks)


def contains(pattern, kmer):
    return all(MASK[c] & MASK[p] for p, c in zip(pattern, kmer))


class PatternEnumeration:
    """Dense pattern number <-> IUPAC string for the sub-patterns of one general pattern."""

    def __init__(self, gen_pat):
        self.genpat = gen_pat
        self.radix = [len(PERM[c]) for c in gen_pat]
        self.weight = []
        w = 1
        for r in self.radix:
            self.weight.append(w)
            w *= r
        self.npat = w
        self._digit = [{x: d for d, x in enumerate(PERM[c])} for c in gen_pat]

    def pattern2num(self, pattern):
        return sum(self._digit[i][pattern[i]] * self.weight[i] for i in range(len(self.genpat)))

    def num2pattern(self, num):
        num = int(num)
        out = []
        for i, c in enumerate(self.genpat):
            out.append(PERM[c][num % self.radix[i]])
            num //= self.radix[i]
        return "".join(out)


def kmer_code(kmer):
    """4 bits per position, one-hot, position 0 in the low nibble (the packing kp_pack_counts reads)."""
    code = 0
    for i, c in enumerate(kmer):
        code |= MASK[c] << (4 * i)
    return code


def kmer_codes(kmers):
    """kmer_code of many k-mers of one length at once (numpy): one byte table lookup and k shifted ORs."""
    import numpy as np

    kmers = list(kmers)
    if not kmers:
        return np.empty(0, dtype=np.uint64)
    k = len(kmers[0])
    if k > 16 or any(len(x) != k for x in kmers):
        return np.array([kmer_code(x) for x in kmers], dtype=np.uint64)
    raw = np.frombuffer("".join(kmers).encode("ascii"), dtype=np.uint8).reshape(len(kmers), k)
    lut = np.zeros(256, dtype=np.uint64)
    for c, m in MASK.items():
        lut[ord(c)] = m
    nib = lut[raw]
    assert nib.all(), "k-mer with a letter outside the IUPAC alphabet"
    codes = np.zeros(len(kmers), dtype=np.uint64)
    for i in range(k):
        codes |= nib[:, i] << np.uint64(4 * i)
    return codes

