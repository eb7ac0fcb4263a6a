"""Times count_mutations on one GPU: the SNV kernel (kp_snv_counts) on its own, the whole chunk loop with and without
positives, and the host VCF reader.

    python tools/count_timing.py [--gbases 3.1] [--snvs 100000000] [--vcf_lines 10000000] [--reps 3] [--out FILE.json]

The genome is apply_timing.py's: --gbases seeded random bases made on the device and cut into 24 records of equal
length.  --snvs seeded random SNVs are spread uniformly over it, REF the genome base and ALT one of the other three.
The pattern is k = 9 NNNNCNNNN with both strands.  Rows:
- the SNV kernel alone over the device-resident genome (one call per record), with each record's SNVs sorted by
  position (as count_mutations passes them) and in a random order;
- the background scan with k-mer counts alone (kp_seq_scan, as apply_timing.py's k-mer-count row), for scale;
- Applier's chunk loop from host bytes with k-mer counts (the background table alone: pinned copies, upload, scan);
- count_mutations() from host bytes: the same loop plus the per-record SNV upload, the SNV kernel per chunk and the
  status copy-back, and its host grouping of the SNVs by record (the SNVs come sorted, as from a sorted VCF).  The VCF
  parse is not included;
- read_vcf alone on a written VCF of --vcf_lines seeded SNV lines (22 chromosomes, sorted, 8 columns), a host time
  (perf_counter) reported with the host CPU's name.
Each case runs once to warm up, then --reps times between CUDA events (the loops end in a device synchronise); the
median is reported.  The card's name and power limit are read in the same run.  --out also writes the rows as JSON.
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from apply_timing import device_genome, gpu_info   # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbases", type=float, default=3.1)
    ap.add_argument("--snvs", type=int, default=100_000_000)
    ap.add_argument("--vcf_lines", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also write the rows as JSON to this file")
    args = ap.parse_args()
    import torch

    from kmerpapa_b200 import count_mutations as C
    from kmerpapa_b200.apply_partition import PIECE, Applier
    from kmerpapa_b200.score_partition import assign

    name, power = gpu_info()
    print(f"GPU: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    gen = "NNNNCNNNN"
    nrec = 24
    rec_len = int(args.gbases * 1e9) // nrec // 64 * 64
    n = rec_len * nrec
    seq = device_genome(torch, n, 1)
    g = torch.Generator(device="cuda").manual_seed(2)
    gpos = torch.sort(torch.randint(0, n, (args.snvs,), generator=g, device="cuda")).values
    code = torch.full((256,), 4, dtype=torch.uint8, device="cuda")
    code[torch.tensor([65, 67, 71, 84], device="cuda")] = torch.arange(4, dtype=torch.uint8, device="cuda")
    ref = code[seq[gpos].long()]
    alt = (ref + torch.randint(1, 4, (args.snvs,), generator=g, device="cuda", dtype=torch.uint8)) % 4
    ra = ref | (alt << 2)
    bounds = torch.searchsorted(gpos, torch.arange(nrec + 1, device="cuda") * rec_len).tolist()
    rpos = [gpos[bounds[r]: bounds[r + 1]] - r * rec_len for r in range(nrec)]
    rra = [ra[bounds[r]: bounds[r + 1]] for r in range(nrec)]
    status = torch.empty(args.snvs, dtype=torch.uint8, device="cuda")
    _, plan, _, owner = assign([gen])
    krate = plan.kmer_rates(owner, np.array([0.5]))
    npieces = (rec_len + PIECE - 1) // PIECE
    psum = torch.empty(nrec * npieces, dtype=torch.float64, device="cuda")
    pn = torch.empty(nrec * npieces, dtype=torch.int64, device="cuda")
    pos_counts = torch.zeros((1, plan.nkmer), dtype=torch.int64, device="cuda")
    bg_counts = torch.zeros(plan.nkmer, dtype=torch.int64, device="cuda")
    rows = []

    def timed(label, fn, bases):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        t = float(np.median(ts))
        rows.append(dict(case=label, bases=bases, snvs=args.snvs, seconds=t, times=ts))
        print(f"{label:70s} {t * 1e3:10.2f} ms  {args.snvs / t / 1e9:6.2f} G SNVs/s  {bases / t / 1e9:7.1f} Gbases/s",
              flush=True)

    def snv_kernel():
        for r in range(nrec):
            lo = r * rec_len
            plan.snv_counts(seq[lo:], 0, rec_len, rec_len, 0, rec_len, True, rpos[r], rra[r], [0, 0, 0, 0], pos_counts,
                            status[bounds[r]: bounds[r + 1]])

    def bg_scan():
        for r in range(nrec):
            lo = r * rec_len
            plan.seq_scan(seq[lo:], 0, rec_len, rec_len, 0, rec_len, krate, True, psum[r * npieces:], pn[r * npieces:],
                          counts=bg_counts)

    tag = f"k=9 {gen} both, {nrec} records of {rec_len} b"
    timed(f"{tag}: SNV kernel alone, SNVs sorted by position, device genome", snv_kernel, n)
    st = status.cpu().numpy()
    print("  statuses:", {s: int(c) for s, c in zip(C.STATUS, np.bincount(st, minlength=len(C.STATUS)))}, flush=True)
    sorted_counts = pos_counts.clone()
    for r in range(nrec):   # the same SNVs, each record's in a random order: scattered window reads
        perm = torch.randperm(len(rpos[r]), generator=g, device="cuda")
        rpos[r], rra[r] = rpos[r][perm], rra[r][perm]
    pos_counts.zero_()
    timed(f"{tag}: SNV kernel alone, SNVs in random order, device genome", snv_kernel, n)
    assert torch.equal(pos_counts, sorted_counts), "the SNV order changed the counts"
    timed(f"{tag}: background scan with k-mer counts alone, device genome", bg_scan, n)

    # from host bytes: the chunk loop without and with positives
    host = seq[:n].cpu().numpy()
    recs = [(f"r{r}", host[r * rec_len: (r + 1) * rec_len].tobytes()) for r in range(nrec)]
    del host
    hp = gpos.cpu().numpy()
    snvs = C.Snvs(chroms=[nm for nm, _ in recs], chrom_line=np.zeros(nrec, np.int64), chrom=(hp // rec_len).astype(np.int32), pos=hp % rec_len,
                  ref=ref.cpu().numpy(), alt=alt.cpu().numpy(), line=np.arange(1, args.snvs + 1, dtype=np.int64),
                  skipped=0, name="synthetic")
    del gpos, ref, alt, ra, rpos, rra, status, seq
    torch.cuda.empty_cache()

    def loop_bg():
        a = Applier([gen], [0.5], strand="both", kmer_counts=True)
        for nm, s in recs:
            a.record(nm, s)
        a.finish()

    timed(f"{tag}: Applier chunk loop with k-mer counts, host bytes", loop_bg, n)
    res = None

    def loop_pos():
        nonlocal res
        res = None   # one result alive at a time: each holds a status byte per SNV
        res = C.count_mutations(gen, recs, snvs, strand="both")

    timed(f"{tag}: count_mutations() chunk loop with {args.snvs} SNVs, host bytes", loop_pos, n)
    print("  statuses:", res.status_counts, flush=True)
    statuses = res.status_counts
    del res, recs, snvs

    # the host VCF reader on its own
    cpu = host_cpu()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "calls.vcf")
        write_vcf(path, args.vcf_lines)
        nbytes = os.path.getsize(path)
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            got = C.read_vcf(path)
            ts.append(time.perf_counter() - t0)
        assert len(got) == args.vcf_lines
    t = float(np.median(ts))
    rows.append(dict(case=f"read_vcf, {args.vcf_lines} lines", host_cpu=cpu, lines=args.vcf_lines, bytes=nbytes,
                     seconds=t, times=ts))
    print(f"{'read_vcf, ' + str(args.vcf_lines) + ' lines, ' + str(nbytes) + ' B':70s} {t * 1e3:10.2f} ms  "
          f"{args.vcf_lines / t / 1e6:6.2f} M lines/s  (host: {cpu})", flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(gpu=name, power_limit_max_sm_clock=power, host_cpu=cpu, records=nrec, rec_len=rec_len,
                           statuses=statuses, rows=rows), f, indent=1)


def host_cpu():
    try:
        with open("/proc/cpuinfo") as f:
            model = next(line.split(":", 1)[1].strip() for line in f if line.startswith("model name"))
    except (OSError, StopIteration):
        model = "unknown CPU"
    return f"{model}, {os.cpu_count()} logical CPUs"


def write_vcf(path, n, seed=1):
    """n seeded SNV lines over 22 chromosomes, sorted by chromosome and position, with the 8 fixed VCF columns."""
    rng = np.random.default_rng(seed)
    chrom = np.sort(rng.integers(1, 23, n))
    pos = rng.integers(1, 250_000_000, n)
    o = np.lexsort((pos, chrom))
    chrom, pos = chrom[o], pos[o]
    ref = rng.integers(0, 4, n)
    alt = (ref + rng.integers(1, 4, n)) % 4
    with open(path, "w") as f:
        f.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n")
        for lo in range(0, n, 1_000_000):
            sl = slice(lo, lo + 1_000_000)
            f.write("".join(f"chr{c}\t{p}\t.\t{'ACGT'[r]}\t{'ACGT'[a]}\t50\tPASS\tDP=30\n"
                            for c, p, r, a in zip(chrom[sl].tolist(), pos[sl].tolist(), ref[sl].tolist(),
                                                  alt[sl].tolist())))


if __name__ == "__main__":
    main()
