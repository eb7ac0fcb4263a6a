"""Apply a fitted pattern partition along genome sequences:
`python -m kmerpapa_b200.apply_partition --partition F --fasta G [--regions BED] [--strand forward|both] [--track DIR]
[--kmer_counts OUT]`.

A kmerpapa model is a list of IUPAC patterns, each with a mutation rate.  This module gives every position of a
sequence the rate of the pattern its context falls in, sums the rates over regions (the expected number of mutations
there) and counts the contexts, on the GPU (kp_seq_scan / kp_region_sums, DESIGN §4c).  Its k-mer counts are the `-b`
background input of kmerpapa.

Conventions:
- k is the partition's length and c = k // 2.  Position i of a record (0-based) has the forward window
  seq[i - c : i - c + k]; this is the centre io_utils._centre_window keeps when it collapses longer k-mers.
- A window is a context when it lies inside the record and all its bytes are A, C, G or T, in either case.  Any other
  byte (N, other IUPAC letters, '-') makes every window that contains it no context.
- A context matches when every base lies in the general pattern's letter at its position (kp_pack_kernel's test); its
  k-mer index is kp_pack_kernel's (mixed radix over the general pattern's multi-letter positions, first position
  fastest, the bases of a letter in iupac.matches order).
- --strand both also looks up the reverse complement of the window.  It needs an odd k, so that the reverse context is
  centred on the same base.  The position's rate is p_fwd + p_rev as one float64 addition, where a side that does not
  match adds 0, and every matching (position, strand) pair is one context.  This is the pyrimidine-centred model:
  NNNNCNNNN covers C on the + strand and G on the + strand (as a C on the - strand).
- A position's rate is 0 when it has a context that does not match, and it has no rate (NaN in the track) when it has
  no context.
- A region `chrom start end [anything]` is 0-based and half-open and sums over the positions start <= i < end.  A
  position's context is read from the record, so it may reach past the region's ends.  Regions may overlap; each is
  summed on its own.  BED lines starting with '#', 'track' or 'browser' are skipped.
- --kmer_counts counts each context (each strand's, with --strand both) at a position in the union of the regions once,
  or at every position when no regions are given.

Every output is the same bits on every run, whatever the chunk size: a region's expected count is the left-to-right
float64 sum of its clipped piece sums (pieces are 65536 positions at fixed record coordinates, each summed by a fixed
reduction tree), and the counts are integers.
"""
import argparse
import gzip
import os
import sys

import numpy as np

from . import iupac
from .score_partition import PartitionError, assign, read_partition

PIECE = 1 << 16          # positions per piece of a record (kp_seq_scan)
CHUNK_BASES = 1 << 26    # positions uploaded and scanned per call
MAXK = 32                # longest partition (KP_MAXK)
STRANDS = ("forward", "both")


class InputError(ValueError):
    pass


def read_fasta(path):
    """(name, bytes) per record of a plain or gzip (.gz) FASTA file, one record at a time.  The name is the first word
    of the header line; sequence lines lose their line ends and surrounding white space.  Duplicate names are an error."""
    opener = gzip.open if path.endswith(".gz") else open
    seen = set()
    with opener(path, "rb") as f:
        name, parts = None, []
        for lineno, line in enumerate(f, 1):
            if line.startswith(b">"):
                if name is not None:
                    yield name, b"".join(parts)
                words = line[1:].split()
                if not words:
                    raise InputError(f"{path}:{lineno}: header line without a name")
                name, parts = words[0].decode(), []
                if name in seen:
                    raise InputError(f"{path}:{lineno}: duplicate record name {name}")
                seen.add(name)
                continue
            s = line.strip()
            if not s:
                continue
            if name is None:
                raise InputError(f"{path}:{lineno}: sequence before the first '>' header")
            parts.append(s)
        if name is not None:
            yield name, b"".join(parts)


def read_regions(f, name="regions"):
    """[(chrom, start, end, 'file:line')] from BED lines, in file order.  Malformed lines, negative starts and empty
    regions are errors that name the line; chromosome names and lengths are checked against the records later."""
    out = []
    for lineno, line in enumerate(f, 1):
        s = line.strip()
        if not s or s.startswith(("#", "track", "browser")):
            continue
        where = f"{name}:{lineno}"
        cols = s.split()
        if len(cols) < 3:
            raise InputError(f"{where}: expected 'chrom start end', got {s!r}")
        try:
            start, end = int(cols[1]), int(cols[2])
        except ValueError:
            raise InputError(f"{where}: start and end must be integers, got {cols[1]!r} {cols[2]!r}") from None
        if start < 0:
            raise InputError(f"{where}: negative start {start}")
        if start >= end:
            raise InputError(f"{where}: start {start} is not below end {end}")
        out.append((cols[0], start, end, where))
    return out


def merge_intervals(starts, ends):
    """Sorted, disjoint, non-touching (start, end) arrays of the union of the half-open intervals."""
    if len(starts) == 0:
        return np.empty(0, np.int64), np.empty(0, np.int64)
    o = np.argsort(starts, kind="stable")
    s, e = np.asarray(starts, np.int64)[o], np.asarray(ends, np.int64)[o]
    reach = np.maximum.accumulate(e)
    new = np.ones(len(s), bool)
    new[1:] = s[1:] > reach[:-1]
    first = np.flatnonzero(new)
    last = np.append(first[1:], len(s)) - 1
    return s[first], reach[last]


def mask_words(ustart, uend, pos0, pos1):
    """uint32 words whose bit i - pos0 is set for the positions i of [pos0, pos1) in the union (ustart, uend)."""
    n = pos1 - pos0
    nbits = (n + 31) // 32 * 32
    d = np.zeros(nbits + 1, np.int8)
    lo, hi = np.searchsorted(uend, pos0, "right"), np.searchsorted(ustart, pos1, "left")
    s = np.clip(ustart[lo:hi], pos0, pos1) - pos0
    e = np.clip(uend[lo:hi], pos0, pos1) - pos0
    d[s] += 1
    d[e] -= 1
    bits = np.cumsum(d[:nbits], dtype=np.int8) > 0
    return np.packbits(bits, bitorder="little").view(np.uint32)


def region_tasks(starts, ends, rec_len):
    """The clipped piece sums the regions of one record need.  Returns (tasks, reg): tasks uint32 [t, 3] (piece, lo, hi
    in the piece), sorted by piece; reg int64 [r, 4] = (first piece, last piece, task of the first or -1, task of the
    last or -1) for kp_region_sums."""
    s, e = np.asarray(starts, np.int64), np.asarray(ends, np.int64)
    pa, pb = s // PIECE, (e - 1) // PIECE
    pend_a = np.minimum((pa + 1) * PIECE, rec_len)
    a_lo, a_hi = s - pa * PIECE, np.minimum(e, pend_a) - pa * PIECE
    clip_a = (a_lo != 0) | (a_hi != pend_a - pa * PIECE)
    clip_b = (pb > pa) & (e != np.minimum((pb + 1) * PIECE, rec_len))
    ia, ib = np.flatnonzero(clip_a), np.flatnonzero(clip_b)
    piece = np.concatenate([pa[ia], pb[ib]])
    lo = np.concatenate([a_lo[ia], np.zeros(len(ib), np.int64)])
    hi = np.concatenate([a_hi[ia], e[ib] - pb[ib] * PIECE])
    order = np.argsort(piece, kind="stable")
    slot = np.empty(len(order), np.int64)
    slot[order] = np.arange(len(order))
    reg = np.full((len(s), 4), -1, np.int64)
    reg[:, 0], reg[:, 1] = pa, pb
    reg[ia, 2] = slot[: len(ia)]
    reg[ib, 3] = slot[len(ia):]
    tasks = np.stack([piece, lo, hi], axis=1)[order].astype(np.uint32)
    return tasks, reg


class ApplyResult:
    """Per region (input order; per record without regions): chrom, start, end, n_contexts (int64), expected
    (float64); model_n_contexts and model_expected hold them for every model of Applier.add_model, [model, region],
    the first model's row being n_contexts / expected.  tracks: {name: float32 array} when asked for; counts: int64 per
    k-mer of gen_pat in k-mer index order when asked for."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


class Applier:
    """Streams records through the scan: a plan and a device rate table per model (one model unless add_model is
    called), double-buffered pinned uploads."""

    def __init__(self, patterns, rates, regions=None, strand="forward", track=False, kmer_counts=False, device=None,
                 chunk_bases=CHUNK_BASES):
        import torch

        if strand not in STRANDS:
            raise InputError(f"strand must be one of {', '.join(STRANDS)}, not {strand!r}")
        if chunk_bases < PIECE or chunk_bases % PIECE:
            raise InputError(f"chunk_bases must be a positive multiple of {PIECE}")
        rates = np.ascontiguousarray(rates, dtype=np.float64)
        if len(rates) != len(patterns):
            raise InputError("one rate per pattern")
        k = len(patterns[0])
        if strand == "both" and k % 2 == 0:
            raise InputError(f"--strand both needs an odd k, so that the reverse context is centred on the same base "
                             f"(the partition has k = {k})")
        self.gen_pat, self.plan, _, owner = assign(patterns, device)
        self.k, self.c, self.both, self.track, self.chunk = k, k // 2, strand == "both", bool(track), int(chunk_bases)
        self.torch, self.dev = torch, self.plan.device
        self.kmer_rate = self.plan.kmer_rates(owner, rates)
        self.scans = [(self.plan, self.kmer_rate)]   # (plan, device rate table) per model
        self.counts = torch.zeros(self.plan.nkmer, dtype=torch.int64, device=self.dev) if kmer_counts else None
        self.regions = None
        if regions is not None:
            regions = [tuple(r) + (f"region {i + 1}",) if len(r) == 3 else tuple(r) for i, r in enumerate(regions)]
            self.regions = regions
            self.by_chrom = {}
            for i, r in enumerate(regions):
                self.by_chrom.setdefault(r[0], []).append(i)
            n = len(regions)
            self.n_contexts, self.expected = np.zeros((1, n), np.int64), np.zeros((1, n), np.float64)
        else:
            self.rows = []
        self.names = set()
        cap = self.chunk + MAXK + 32
        self.pinned = [torch.empty(cap, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.dseq = [torch.empty(cap, dtype=torch.uint8, device=self.dev) for _ in range(2)]
        self.pmask = [torch.empty(self.chunk // 32, dtype=torch.int32).pin_memory() for _ in range(2)]
        self.dmask = [torch.empty(self.chunk // 32, dtype=torch.int32, device=self.dev) for _ in range(2)]
        self.ev = [None, None]
        self.nchunks = 0

    def add_model(self, patterns, rates):
        """Scan one more partition of the same k with the first, from the same uploaded bytes: kp_seq_scan and
        kp_region_sums run once per model on its own plan (shared by models of one general pattern) and rate table.
        Returns (model index, general pattern, plan).  Call it before the first record, on an Applier without tracks
        and k-mer counts.  Raises PartitionError as the constructor does."""
        if self.track or self.counts is not None:
            raise InputError("tracks and k-mer counts are of one partition only")
        if self.nchunks or self.names:
            raise InputError("add every model before the first record")
        rates = np.ascontiguousarray(rates, dtype=np.float64)
        if len(rates) != len(patterns):
            raise InputError("one rate per pattern")
        if len(patterns[0]) != self.k:
            raise InputError(f"every partition needs the same k ({self.k}), not {len(patterns[0])}")
        gen_pat, plan, _, owner = assign(patterns, self.dev.index)
        m = len(self.scans)
        self.scans.append((plan, plan.kmer_rates(owner, rates, name=f"apply{m}")))
        if self.regions is not None:
            n = len(self.regions)
            self.n_contexts = np.concatenate([self.n_contexts, np.zeros((1, n), np.int64)])
            self.expected = np.concatenate([self.expected, np.zeros((1, n), np.float64)])
        return m, gen_pat, plan

    def record(self, name, seq, on_chunk=None):
        """Scan one record.  Returns its float32 track (numpy) when tracks are asked for, else None.  A record that has
        no region, when regions are given and tracks are not asked for, is not scanned.  on_chunk(dseq, b0, b1, pos0,
        pos1, mask) is called after the scan of each chunk is enqueued, on the same stream: dseq holds the record bytes
        [b0, b1), which cover the windows of the positions [pos0, pos1), and mask is the region-union bit mask of those
        positions (None without regions).  Work it enqueues on that stream may read both until it ends."""
        torch = self.torch
        if isinstance(seq, str):
            seq = seq.encode("ascii")
        if name in self.names:
            raise InputError(f"duplicate record name {name}")
        self.names.add(name)
        L = len(seq)
        if self.regions is not None:
            idx = np.array(self.by_chrom.pop(name, []), np.int64)
            starts = np.array([self.regions[i][1] for i in idx], np.int64)
            ends = np.array([self.regions[i][2] for i in idx], np.int64)
            past = np.flatnonzero(ends > L)
            if len(past):
                r = self.regions[idx[past[0]]]
                raise InputError(f"{r[3]}: end {r[2]} is past the end of {name} (length {L})")
            if len(idx) == 0 and not self.track:
                return None
        else:
            starts, ends = np.zeros(1, np.int64), np.array([L], np.int64)
        with torch.cuda.device(self.dev):
            out = self._scan(seq, L, starts, ends, on_chunk)
        if self.regions is not None:
            if len(idx):
                self.n_contexts[:, idx], self.expected[:, idx] = out[0], out[1]
        else:
            self.rows.append((name, 0, L, out[0][:, 0], out[1][:, 0]))
        return out[2]

    def _scan(self, seq, L, starts, ends, on_chunk):
        torch, P, nm = self.torch, PIECE, len(self.scans)
        stream = torch.cuda.current_stream(self.dev)
        npieces = (L + P - 1) // P
        psum = torch.empty((nm, max(npieces, 1)), dtype=torch.float64, device=self.dev)
        pn = torch.empty((nm, max(npieces, 1)), dtype=torch.int64, device=self.dev)
        tasks, reg = region_tasks(starts, ends, L) if len(starts) else (np.zeros((0, 3), np.uint32), np.zeros((0, 4), np.int64))
        dtasks = torch.from_numpy(tasks.view(np.int32)).to(self.dev) if len(tasks) else None
        tsum = torch.empty((nm, max(len(tasks), 1)), dtype=torch.float64, device=self.dev)
        tn = torch.empty((nm, max(len(tasks), 1)), dtype=torch.int64, device=self.dev)
        track = torch.empty(L, dtype=torch.float32, device=self.dev) if self.track else None
        masked = self.counts is not None and self.regions is not None
        if masked:
            ustart, uend = merge_intervals(starts, ends)
        src = np.frombuffer(seq, dtype=np.uint8)
        tpiece = tasks[:, 0].astype(np.int64)
        for pos0 in range(0, L, self.chunk):
            pos1 = min(L, pos0 + self.chunk)
            b0, b1 = max(0, pos0 - self.c), min(L, pos1 + self.k - 1 - self.c)
            slot = self.nchunks % 2
            self.nchunks += 1
            if self.ev[slot] is not None:
                self.ev[slot].synchronize()   # the scan that read this slot's buffers is done
            self.pinned[slot].numpy()[: b1 - b0] = src[b0:b1]
            self.dseq[slot][: b1 - b0].copy_(self.pinned[slot][: b1 - b0], non_blocking=True)
            mask = None
            if masked:
                words = mask_words(ustart, uend, pos0, pos1)
                self.pmask[slot].numpy()[: len(words)] = words.view(np.int32)
                mask = self.dmask[slot][: len(words)]
                mask.copy_(self.pmask[slot][: len(words)], non_blocking=True)
            t0, t1 = np.searchsorted(tpiece, pos0 // P), np.searchsorted(tpiece, (pos1 + P - 1) // P)
            for m, (plan, kmer_rate) in enumerate(self.scans):
                plan.seq_scan(self.dseq[slot], b0, b1 - b0, L, pos0, pos1, kmer_rate, self.both, psum[m, pos0 // P:],
                              pn[m, pos0 // P:], track=track[pos0:pos1] if track is not None else None, count_mask=mask,
                              counts=self.counts)
                if t1 > t0:
                    plan.seq_scan(self.dseq[slot], b0, b1 - b0, L, pos0, pos1, kmer_rate, self.both, tsum[m, t0:],
                                  tn[m, t0:], tasks=dtasks[t0:t1])
            if on_chunk is not None:
                on_chunk(self.dseq[slot], b0, b1, pos0, pos1, mask)
            ev = torch.cuda.Event()
            ev.record(stream)
            self.ev[slot] = ev
        res_n = res_s = None
        if len(reg):
            dreg = torch.from_numpy(reg).to(self.dev)
            osum = torch.empty((nm, len(reg)), dtype=torch.float64, device=self.dev)
            on = torch.empty((nm, len(reg)), dtype=torch.int64, device=self.dev)
            for m, (plan, _) in enumerate(self.scans):
                plan.region_sums(psum[m], pn[m], tsum[m] if len(tasks) else None, tn[m] if len(tasks) else None, dreg,
                                 osum[m], on[m])
            res_n, res_s = on.cpu().numpy(), osum.cpu().numpy()
        return res_n, res_s, track.cpu().numpy() if track is not None else None

    def finish(self):
        """The result once every record has been scanned (unknown region chromosomes are errors here)."""
        if self.regions is not None:
            left = sorted(i for idx in self.by_chrom.values() for i in idx)
            if left:
                r = self.regions[left[0]]
                raise InputError(f"{r[3]}: unknown chrom {r[0]} (no record of that name)")
            chrom = [r[0] for r in self.regions]
            start = np.array([r[1] for r in self.regions], np.int64)
            end = np.array([r[2] for r in self.regions], np.int64)
            n_contexts, expected = self.n_contexts, self.expected
        else:
            chrom = [r[0] for r in self.rows]
            start = np.array([r[1] for r in self.rows], np.int64)
            end = np.array([r[2] for r in self.rows], np.int64)
            nm = len(self.scans)
            n_contexts = np.ascontiguousarray(np.array([r[3] for r in self.rows], np.int64).reshape(-1, nm).T)
            expected = np.ascontiguousarray(np.array([r[4] for r in self.rows], np.float64).reshape(-1, nm).T)
        counts = self.counts.cpu().numpy() if self.counts is not None else None
        return ApplyResult(gen_pat=self.gen_pat, k=self.k, chrom=chrom, start=start, end=end, n_contexts=n_contexts[0],
                           expected=expected[0], model_n_contexts=n_contexts, model_expected=expected, counts=counts)


def apply(patterns, rates, records, regions=None, strand="forward", track=False, kmer_counts=False, device=None,
          chunk_bases=CHUNK_BASES):
    """Apply a partition (patterns, float64 rates) to records, an iterable of (name, bytes) pairs.  regions: None (one
    row per record) or (chrom, start, end[, where]) tuples.  Returns an ApplyResult; see the module docstring for the
    conventions.  chunk_bases (a multiple of 65536) is the number of positions scanned per call; it changes no result.
    Raises PartitionError when the patterns do not partition their general pattern and InputError on bad input."""
    ap = Applier(patterns, rates, regions, strand, track, kmer_counts, device, chunk_bases)
    tracks = {} if track else None
    for name, seq in records:
        t = ap.record(name, seq)
        if track:
            tracks[name] = t
    res = ap.finish()
    res.tracks = tracks
    return res


def kmers_of_indices(gen_pat, idx):
    """numpy bytes array: the k-mers of gen_pat with the given k-mer indices (iupac.kmer_of_index, vectorised)."""
    idx = np.array(idx, dtype=np.int64)
    out = np.empty((len(idx), len(gen_pat)), np.uint8)
    for s, ch in enumerate(gen_pat):
        bases = np.frombuffer(iupac.CODE[ch].encode("ascii"), np.uint8)
        out[:, s] = bases[idx % len(bases)]
        idx //= len(bases)
    return out.view(f"S{len(gen_pat)}").ravel()


def write_kmer_counts(f, gen_pat, counts):
    """`kmer count` lines (io_utils.read_dict reads them) for the k-mers with a non-zero count, in k-mer index order."""
    nz = np.flatnonzero(counts)
    for lo in range(0, len(nz), 1 << 20):
        part = nz[lo: lo + (1 << 20)]
        kmers = kmers_of_indices(gen_pat, part)
        f.write("".join(f"{km.decode()} {int(c)}\n" for km, c in zip(kmers, counts[part])))


def get_parser():
    p = argparse.ArgumentParser(prog="python -m kmerpapa_b200.apply_partition",
                                description="Expected mutation counts, rate tracks and k-mer counts of a fitted kmerpapa "
                                            "partition along genome sequences")
    p.add_argument("--partition", required=True, metavar="F", help="Partition file written by kmerpapa (with or without -l)")
    p.add_argument("--fasta", required=True, metavar="G", help="FASTA file, plain or gzip (.gz)")
    p.add_argument("--regions", metavar="BED", help="Regions 'chrom start end' (0-based, half-open); default: whole records")
    p.add_argument("--strand", choices=STRANDS, default="forward",
                   help="both: add the rate of the reverse-complement context (odd k only)")
    p.add_argument("--track", metavar="DIR", help="Write DIR/<record>.f32: float32 rate per position, NaN without a context")
    p.add_argument("--kmer_counts", metavar="OUT",
                   help="Write 'kmer count' lines of the contexts in the regions (kmerpapa -b input)")
    return p


def main(argv=None):
    args = get_parser().parse_args(argv)
    try:
        with open(args.partition) as f:
            patterns, rates = read_partition(f, args.partition)
        regions = None
        if args.regions:
            with open(args.regions) as f:
                regions = read_regions(f, args.regions)
        ap = Applier(patterns, rates, regions, args.strand, track=args.track is not None,
                     kmer_counts=args.kmer_counts is not None)
        if args.track:
            os.makedirs(args.track, exist_ok=True)
        for name, seq in read_fasta(args.fasta):
            t = ap.record(name, seq)
            if args.track:
                t.astype("<f4").tofile(os.path.join(args.track, name + ".f32"))
        res = ap.finish()
    except (OSError, PartitionError, InputError) as e:
        print(f"apply_partition: error: {e}", file=sys.stderr)
        return 1
    if args.kmer_counts:
        with open(args.kmer_counts, "w") as f:
            write_kmer_counts(f, res.gen_pat, res.counts)
    out = ["chrom start end n_contexts expected"]
    out += [f"{c} {s} {e} {n} {x!r}" for c, s, e, n, x in zip(res.chrom, res.start.tolist(), res.end.tolist(),
                                                               res.n_contexts.tolist(), res.expected.tolist())]
    sys.stdout.write("\n".join(out) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
