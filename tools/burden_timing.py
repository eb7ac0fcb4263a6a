"""Times burden on one GPU: the six scans with their region sums, the six SNV classification calls and the region-count
kernel (kp_snv_region_counts) over a device-resident genome, then burden() and, for comparison, six apply() calls from
host bytes.

    python tools/burden_timing.py [--gbases 3.1] [--snvs 100000000] [--regions 1000000] [--reps 3] [--out FILE.json]

The genome is apply_timing.py's: --gbases seeded random bases made on the device and cut into 24 records of equal
length.  --snvs seeded random SNVs are spread uniformly over it, REF the genome base and ALT one of the other three;
--regions seeded regions of 1 b to 20 kb lie on random records.  The models are the usual six, k = 9 with both strands:
C>A, C>G, C>T on NNNNCNNNN and A>C, A>G, A>T on NNNNANNNN, each a seeded random partition of 200 splits.  Rows:
- the six scans with their region sums (per record and model: kp_seq_scan's piece pass and clipped-task pass, then
  kp_region_sums), device genome;
- the six classification calls (kp_snv_counts per record and model, SNVs sorted by position), device genome;
- the region-count kernel alone (kp_snv_region_counts per record: the prefix-count scan and the region kernel), on the
  model ids the classification gave;
- burden() from host bytes: the chunk loop with pinned uploads, the scans, the classification, the model ids, the
  region counts and the host work per record (the FASTA and VCF parses are not included);
- six apply() calls from host bytes, one per model: what burden replaces for the expected counts.
Each case runs once to warm up, then --reps times between CUDA events (every case ends in a device synchronise); the
median is reported.  The card's name and power limit are read in the same run.  --out also writes the rows as JSON.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from apply_timing import device_genome, gpu_info, random_partition   # noqa: E402

SPECS = [("CA", "NNNNCNNNN", "A"), ("CG", "NNNNCNNNN", "G"), ("CT", "NNNNCNNNN", "T"),
         ("AC", "NNNNANNNN", "C"), ("AG", "NNNNANNNN", "G"), ("AT", "NNNNANNNN", "T")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gbases", type=float, default=3.1)
    ap.add_argument("--snvs", type=int, default=100_000_000)
    ap.add_argument("--regions", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also write the rows as JSON to this file")
    args = ap.parse_args()
    import torch

    from kmerpapa_b200 import apply_partition as A
    from kmerpapa_b200 import burden as B
    from kmerpapa_b200 import count_mutations as C
    from kmerpapa_b200.score_partition import assign

    name, power = gpu_info()
    print(f"GPU: {name}; power.limit, clocks.max.sm: {power}", flush=True)
    rng = np.random.default_rng(3)
    models = []
    for nm, gen, alt in SPECS:
        pats = random_partition(gen, 200, rng)
        models.append(B.Model(nm, alt, pats, rng.uniform(1e-6, 0.3, len(pats))))
    nrec = 24
    rec_len = int(args.gbases * 1e9) // nrec // 64 * 64
    n = rec_len * nrec
    P = A.PIECE
    npieces = (rec_len + P - 1) // P
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
    rr = rng.integers(0, nrec, args.regions)
    starts = rng.integers(0, rec_len - 1, args.regions)
    ends = np.minimum(rec_len, starts + rng.integers(1, 20_001, args.regions))

    scans = []   # (plan, device rate table) per model
    for i, m in enumerate(models):
        _, plan, _, owner = assign(m.patterns)
        scans.append((plan, plan.kmer_rates(owner, m.rates, name=f"timing{i}")))
    slots = [[0 if x == m.alt else -1 for x in "ACGT"] for m in models]
    psum = torch.empty(nrec * npieces, dtype=torch.float64, device="cuda")
    pn = torch.empty(nrec * npieces, dtype=torch.int64, device="cuda")
    per = []
    for r in range(nrec):
        sel = rr == r
        tasks, reg = A.region_tasks(starts[sel], ends[sel], rec_len)
        reg[:, :2] += r * npieces
        bnd = np.stack([starts[sel], ends[sel]], axis=1)
        per.append((torch.from_numpy(tasks.view(np.int32)).cuda(), torch.from_numpy(reg).cuda(),
                    torch.from_numpy(bnd).cuda()))
    tsum = [torch.empty(len(t), dtype=torch.float64, device="cuda") for t, _, _ in per]
    tn = [torch.empty(len(t), dtype=torch.int64, device="cuda") for t, _, _ in per]
    osum = torch.empty(args.regions, dtype=torch.float64, device="cuda")
    on = torch.empty(args.regions, dtype=torch.int64, device="cuda")
    counts = [torch.zeros(p.nkmer, dtype=torch.int64, device="cuda") for p, _ in scans]
    status = torch.empty((len(models), args.snvs), dtype=torch.uint8, device="cuda")
    model_id = torch.empty(args.snvs, dtype=torch.uint8, device="cuda")
    obs = [torch.empty((len(b), len(models)), dtype=torch.int64, device="cuda") for _, _, b in per]
    rows = []

    def timed(label, fn):
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
        rows.append(dict(case=label, bases=n, snvs=args.snvs, regions=args.regions, seconds=t, times=ts))
        print(f"{label:78s} {t * 1e3:10.2f} ms", flush=True)

    def scans_and_sums():
        for plan, krate in scans:
            for r, (tasks, reg, _) in enumerate(per):
                lo = r * rec_len
                plan.seq_scan(seq[lo:], 0, rec_len, rec_len, 0, rec_len, krate, True, psum[r * npieces:],
                              pn[r * npieces:])
                plan.seq_scan(seq[lo:], 0, rec_len, rec_len, 0, rec_len, krate, True, tsum[r], tn[r], tasks=tasks)
                plan.region_sums(psum, pn, tsum[r], tn[r], reg, osum, on)

    def classify():
        for m, (plan, _) in enumerate(scans):
            for r in range(nrec):
                lo = r * rec_len
                plan.snv_counts(seq[lo:], 0, rec_len, rec_len, 0, rec_len, True, rpos[r], rra[r], slots[m], counts[m],
                                status[m, bounds[r]: bounds[r + 1]])

    def region_counts():
        for r, (_, _, bnd) in enumerate(per):
            scans[0][0].snv_region_counts(rpos[r], model_id[bounds[r]: bounds[r + 1]], len(models), bnd, obs[r])

    tag = f"six k=9 models, both strands, {nrec} records of {rec_len} b, {args.regions} regions"
    timed(f"{tag}: six scans + region sums, device genome", scans_and_sums)
    timed(f"{tag}: six classification calls ({args.snvs} SNVs), device genome", classify)
    hit = status == B.KP_SNV_COUNTED
    assert int(hit.sum(0).max()) <= 1, "two models counted one SNV"
    model_id.fill_(B.NO_MODEL)
    for m in range(len(models)):
        model_id.masked_fill_(hit[m], m)
    del hit
    timed(f"{tag}: region-count kernel alone", region_counts)
    dev_obs = torch.cat(obs).sum(0).tolist()
    print("  observed per model:", dict(zip([m.name for m in models], dev_obs)), flush=True)

    # from host bytes
    host = seq[:n].cpu().numpy()
    recs = [(f"r{r}", host[r * rec_len: (r + 1) * rec_len].tobytes()) for r in range(nrec)]
    del host
    regions = [(f"r{c}", int(s), int(e)) for c, s, e in zip(rr.tolist(), starts.tolist(), ends.tolist())]
    hp = gpos.cpu().numpy()
    snvs = C.Snvs(chroms=[nm for nm, _ in recs], chrom_line=np.zeros(nrec, np.int64), chrom=(hp // rec_len).astype(np.int32),
                  pos=hp % rec_len, ref=ref.cpu().numpy(), alt=alt.cpu().numpy(),
                  line=np.arange(1, args.snvs + 1, dtype=np.int64), skipped=0, name="synthetic")
    del gpos, ref, alt, ra, rpos, rra, status, model_id, obs, seq, per, tsum, tn, psum, pn
    torch.cuda.empty_cache()
    res = None

    def run_burden():
        nonlocal res
        res = None   # one result alive at a time
        res = B.burden(models, recs, snvs, regions, "both")

    timed(f"{tag}: burden() from host bytes", run_burden)
    print("  statuses:", res.status_counts, flush=True)
    assert res.model_observed.sum(1).tolist() == dev_obs, "burden() and the device-genome path disagree"
    statuses = res.status_counts
    del res

    def six_apply():
        for m in models:
            A.apply(m.patterns, m.rates, recs, regions=regions, strand="both")

    timed(f"{tag}: six apply() calls from host bytes", six_apply)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(gpu=name, power_limit_max_sm_clock=power, records=nrec, rec_len=rec_len, statuses=statuses,
                           rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
