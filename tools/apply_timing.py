"""Times the sequence scan of apply_partition (kp_seq_scan / kp_region_sums) on one GPU, and the host FASTA reader.

    python tools/apply_timing.py [--gbases 3.1] [--reps 3] [--out FILE.json]

A random genome of --gbases bases (seeded torch generator) is made on the device and cut into 24 records of equal
length, so the host parse is not in the scan times.  Each case runs once to warm up, then --reps times between CUDA
events; the median is reported as bases/s and bytes/s (1 byte read per base, plus 4 written per base with the track).
The genome is far larger than L2.  The host FASTA reader is timed on its own on a written 300 Mb file, and apply()
from host bytes (double-buffered pinned uploads, parse excluded) on the first 300 Mb of the genome.  The table is
printed; --out also writes it as JSON.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def random_partition(gen, nsplit, rng):
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
    return ["".join(iupac.LETTER[m] for m in leaf) for leaf in leaves]


def device_genome(torch, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    seq = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    step = 1 << 28
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        x = torch.randint(0, 4, (hi - lo,), generator=g, device="cuda", dtype=torch.uint8)
        seq[lo:hi] = 65 + 2 * x + 2 * (x >= 2).to(torch.uint8) + 11 * (x == 3).to(torch.uint8)   # A C G T
    return seq


def gpu_info():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:   # the numbers are then reported without it
        q = f"unavailable ({e})"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbases", type=float, default=3.1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--regions", type=int, default=1_000_000)
    ap.add_argument("--out", help="also write the rows as JSON to this file")
    args = ap.parse_args()
    import torch

    from kmerpapa_b200 import apply_partition as A
    from kmerpapa_b200.score_partition import assign

    name, power = gpu_info()
    print(f"GPU: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    nrec = 24
    rec_len = int(args.gbases * 1e9) // nrec // 64 * 64
    n = rec_len * nrec
    seq = device_genome(torch, n, 1)
    rng = np.random.default_rng(1)
    P = A.PIECE
    npieces = (rec_len + P - 1) // P
    rows = []

    def timed(label, fn, bytes_per_base):
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
        row = dict(case=label, bases=n, seconds=t, times=ts, gbases_per_s=n / t / 1e9,
                   gbytes_per_s=n * bytes_per_base / t / 1e9)
        rows.append(row)
        print(f"{label:58s} {t * 1e3:9.2f} ms  {row['gbases_per_s']:7.1f} Gbases/s  {row['gbytes_per_s']:7.1f} GB/s", flush=True)

    for gen, nsplit, both in (("NNNNCNNNN", 200, True), ("NNNNNNNNNNNNN", 400, False)):
        patterns = random_partition(gen, nsplit, rng)
        rates = rng.uniform(1e-6, 0.3, len(patterns))
        _, plan, _, owner = assign(patterns)
        krate = plan.kmer_rates(owner, rates)
        psum = torch.empty(nrec * npieces, dtype=torch.float64, device="cuda")
        pn = torch.empty(nrec * npieces, dtype=torch.int64, device="cuda")
        tag = f"k={len(gen)} {gen} {'both' if both else 'forward'}"

        def scan(track=None, counts=None):
            for r in range(nrec):
                lo = r * rec_len
                plan.seq_scan(seq[lo:], 0, rec_len, rec_len, 0, rec_len, krate, both, psum[r * npieces:],
                              pn[r * npieces:], track=track[lo: lo + rec_len] if track is not None else None,
                              counts=counts)

        timed(f"{tag}: piece sums ({len(patterns)} patterns)", scan, 1)
        if not both:
            continue
        # 10^6 random regions (lengths 1 .. 20 kb) over the records: clipped-piece pass and region sums
        rr = rng.integers(0, nrec, args.regions)
        starts = rng.integers(0, rec_len - 1, args.regions)
        ends = np.minimum(rec_len, starts + rng.integers(1, 20_000, args.regions))
        per = []
        for r in range(nrec):
            sel = rr == r
            tasks, reg = A.region_tasks(starts[sel], ends[sel], rec_len)
            reg[:, :2] += r * npieces
            per.append((torch.from_numpy(tasks.view(np.int32)).cuda(), torch.from_numpy(reg).cuda()))
        tsum = [torch.empty(len(t), dtype=torch.float64, device="cuda") for t, _ in per]
        tn = [torch.empty(len(t), dtype=torch.int64, device="cuda") for t, _ in per]
        osum = torch.empty(args.regions, dtype=torch.float64, device="cuda")
        on = torch.empty(args.regions, dtype=torch.int64, device="cuda")

        def regions():
            scan()
            for r, (tasks, reg) in enumerate(per):
                lo = r * rec_len
                plan.seq_scan(seq[lo:], 0, rec_len, rec_len, 0, rec_len, krate, both, tsum[r], tn[r], tasks=tasks)
                plan.region_sums(psum, pn, tsum[r], tn[r], reg, osum, on)

        timed(f"{tag}: piece sums + {args.regions} regions", regions, 1)
        track = torch.empty(n, dtype=torch.float32, device="cuda")
        timed(f"{tag}: piece sums + track", lambda: scan(track=track), 5)
        del track
        counts = torch.zeros(plan.nkmer, dtype=torch.int64, device="cuda")
        timed(f"{tag}: piece sums + k-mer counts", lambda: scan(counts=counts), 1)

        # apply() from host bytes: double-buffered pinned uploads of 64 Mb chunks (the parse is not timed)
        host = seq[: 300_000_000 // rec_len * rec_len if rec_len < 300_000_000 else 300_000_000].cpu().numpy().tobytes()
        recs = [(f"h{i}", host[i: i + rec_len]) for i in range(0, len(host), rec_len)]
        A.apply(patterns, rates, recs[:1], strand="both")
        t0 = time.perf_counter()
        A.apply(patterns, rates, recs, strand="both")
        t = time.perf_counter() - t0
        rows.append(dict(case=f"{tag}: apply() from host bytes", bases=len(host), seconds=t,
                         gbases_per_s=len(host) / t / 1e9))
        print(f"{tag + ': apply() from host bytes, ' + str(len(host)) + ' b':58s} {t * 1e3:9.2f} ms  "
              f"{len(host) / t / 1e9:7.2f} Gbases/s", flush=True)
        del host, recs
    del seq
    torch.cuda.empty_cache()

    # the host FASTA reader on its own, on a written 300 Mb file
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "g.fa")
        lines = np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(2).integers(0, 4, 300_000_000)].reshape(-1, 60)
        body = np.concatenate([lines, np.full((len(lines), 1), ord("\n"), np.uint8)], axis=1)
        with open(path, "wb") as f:
            for r in range(10):
                part = body[r * len(body) // 10: (r + 1) * len(body) // 10]
                f.write(b">chr%d\n" % r)
                f.write(part.tobytes())
        t0 = time.perf_counter()
        nb = sum(len(s) for _, s in A.read_fasta(path))
        t = time.perf_counter() - t0
    rows.append(dict(case="host FASTA reader, 300 Mb in 60-column lines", bases=nb, seconds=t, gbases_per_s=nb / t / 1e9))
    print(f"{'host FASTA reader, 300 Mb in 60-column lines':58s} {t * 1e3:9.2f} ms  {nb / t / 1e9:7.3f} Gbases/s")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(gpu=name, power_limit_max_sm_clock=power, records=nrec, rec_len=rec_len, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
