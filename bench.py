#!/usr/bin/env python
"""Benchmark of the pattern-partition DP on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config auto|cfg3|cfg4|cfg5|n9m]
                  [--dump-outputs DIR]

--config auto (default):
  N = 1  : BASELINE config 3 — one full 9-mer DP (`NNNNANNNN`, 2 562 890 625 patterns) + backtrack.
           A step = count expansion (K2) + wave-front DP with fused scoring (K3+K4) + backtrack (K5), k-mer count
           tables already resident in HBM.  metric = pattern-scores/sec.  The same line carries, under `cv_grid`, the
           45-job CV grid of config 4 on this one GPU: the N = 1 point of the N > 1 curve.
  N > 1  : BASELINE config 4 — the 3x3 (alpha, penalty) grid x 5 folds = 45 single-fold DP jobs of the same size, dealt to
           the ranks by job, one all_gather (NCCL) of the per-job losses.  A step = fold count expansion + this rank's
           jobs + gather + selection, held-out fold tables already sampled.  metric = pattern-scores/sec over all jobs
           (strong scaling: the 45 jobs are fixed); the grid wall time is `ms_per_step`.
--config cfg5 / n9m: the 11-mer `RYNNNANNNRY` (config 5) / `NNNNMNNNN` (7.69 G patterns, the first size beyond the configs) as
           a single DP, same step as config 3 (N > 1: independent replicas).
--impl reference : the reference's CPU path on the host cores — the oracle's C restatement of the numba DP with ALL host
           threads (an explicit count: torchrun exports OMP_NUM_THREADS=1) — on a bounded sample of the same config: the
           sub-problem of k-mers starting with A (1/15 of the patterns); for config 4 a step is two of the 45 jobs on
           that sample.  At N = 1 it also times the UNMODIFIED numba reference (baseline/_ref, one core, fresh process)
           on the 7-mer `NNNMNNN` and reports it under cpu_baseline.numba.

Results are checked, not just timed: loss, partition and per-job CV losses are compared with tests/golden/fullsize.json
(the oracle's full-size run) and the line carries "parity_checked".  A mismatch aborts the benchmark.

Prints ONE JSON line on rank 0.  Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max
over ranks.  Every GPU measurement of the line runs W warm-up steps, then K timed steps.  Tables (>= 4 GB) are far
larger than the 126 MB L2, so no explicit flush.

--dump-outputs DIR: after the timed steps rank 0 writes what the last timed step of each GPU measurement returned, as
DIR/<name>.npy (float32 or float64), so that two builds can be compared output for output; the inputs are seeded and
identical from run to run.  Single DP: loss (float32), partition (its pattern numbers, float64, exact below 2^53).
CV grid: cv_losses (float32 [1, folds, alphas, penalties, (train, held-out)]), cv_selected (float64 [alpha, penalty,
held-out loss]).  Sharded DP (N > 1): sharded_loss, sharded_partition.  A partition has at most one pattern per k-mer,
so all of it stays far below 64 MB and is written whole.

The benchmark compiles nothing and writes nothing into the tree: it loads the libraries __graft_entry__.build() made.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALPHA, PENALTY = 1.0, 6.0
CV_ALPHAS, CV_PENALTIES, CV_FOLDS, CV_SEED = [0.5, 1.0, 10.0], [3.0, 5.0, 6.0], 5, 1
ALGO_BYTES_SINGLE = 41.0   # SURVEY 8(d): f32 best W+R (8) + int64 M,U W+R (32) + u8 split W (1)
ALGO_BYTES_CV = 48.0       # SURVEY 8(d): f32 train+test W+R (16) + read 4 int64 counts (32)
NUMBA_GEN_PAT, NUMBA_SEED, NUMBA_ALPHA, NUMBA_PENALTY = "NNNMNNN", 9002, 1.0, 6.0

# name -> (general pattern, seed of the synthetic counts, CPU sample = the sub-problem with the first free position fixed to A)
SINGLE = {
    "cfg3": ("NNNNANNNN", 9003, "ANNNANNNN",
             "cfg3 synthetic 9-mer (neg-binomial), single penalty+pseudo, full DP + backtrack"),
    "cfg5": ("RYNNNANNNRY", 9005, "RYANNANNNRY",
             "cfg5 synthetic super-pattern-restricted 11-mer RYNNNANNNRY, single penalty+pseudo, full DP + backtrack"),
    "n9m": ("NNNNMNNNN", 9006, "ANNNMNNNN",
            "synthetic 9-mer NNNNMNNNN (7.69 G patterns, beyond the configs), single penalty+pseudo, full DP + backtrack"),
}
CV_GEN_PAT, CV_DATA_SEED, CV_SAMPLE = "NNNNANNNN", 9004, "ANNNANNNN"


def config_for(name, world):
    """The `config` object of the JSON line: a description of the workload only, identical for both arms."""
    if name == "cfg4":
        return {"workload": "cfg4 synthetic 9-mer, 3x3 penalty x pseudo grid, 5-fold CV sharded by job",
                "gen_pat": CV_GEN_PAT, "npat": 15 ** 8, "jobs": CV_FOLDS * len(CV_ALPHAS) * len(CV_PENALTIES),
                "alphas": CV_ALPHAS, "penalties": CV_PENALTIES, "nfolds": CV_FOLDS, "data_seed": CV_DATA_SEED,
                "cv_seed": CV_SEED, "l2": "train table 11 GB per job >> 126 MB L2, no flush needed"}
    gen_pat, seed, _sample, text = SINGLE[name]
    from kmerpapa_b200 import iupac

    return {"workload": text, "gen_pat": gen_pat, "npat": iupac.pattern_max(gen_pat), "alpha": ALPHA, "penalty": PENALTY,
            "data_seed": seed, "replicas": world, "l2": "score table >= 4 GB >> 126 MB L2, no flush needed"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def host_threads():
    """All host cores, as an explicit number (torch.distributed.run exports OMP_NUM_THREADS=1 to its workers)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler:
    """Samples SM clocks and throttle reasons through NVML (in-process thread) while the timed region runs.
    NVML is initialised in __init__, well before the timed region: spawning nvidia-smi or initialising NVML
    next to the timed steps stalls the driver for tens of milliseconds and would distort the measurement."""

    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index, period_s=0.025):
        self.rows, self.period, self.running, self.thread = [], period_s, False, None
        self.handle = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # NVML missing: report it, do not guess
            self.error = repr(e)

    def _loop(self):
        nv = self.nv
        while self.running:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append((float(mhz), int(rs)))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.handle is None:
            return
        self.running = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.handle is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "error", "?")]}
        self.running = False
        self.thread.join(timeout=2)
        sm = [r[0] for r in self.rows]
        reasons = sorted({name for _, bits in self.rows for name, bit in self.REASONS.items() if bits & bit})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(sm)}


def dist_setup(ngpus):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return rank, world, local


def barrier_sync(world):
    import torch

    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms, world, device):
    if world == 1:
        return ms
    import torch
    import torch.distributed as dist

    t = torch.tensor([ms], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def pinned(arr):
    """Copy a numpy array into page-locked host memory (still a numpy view)."""
    import torch

    t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
    return t.numpy(), t


def golden(name):
    p = os.path.join(ROOT, "tests", "golden", "fullsize.json")
    if os.path.exists(p):
        return json.load(open(p)).get(name)
    return None


def load_traffic(kind):
    """DRAM bytes per DP / per CV job from the committed ncu capture (profiles/traffic.json): (bytes, capture id) or
    (None, None).  The number is a profile of the same kernels at the commit named there, not measured in this run."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        t = json.load(open(p))
        v = t.get(kind)
        if isinstance(v, dict):
            return v.get("bytes"), v.get("capture")
        return v, t.get("capture")
    return None, None


# ---------------------------------------------------------------------------------------------
# CPU legs (the oracle is only ever the baseline/checker here, never the product path)
# ---------------------------------------------------------------------------------------------
def sample_inputs(gen_pat, seed, sample):
    """k-mer counts of the sample sub-problem and the (alpha-independent) rate of the FULL data set."""
    from kmerpapa_b200 import iupac, synthetic

    kmers, pos, neg = synthetic.negbin_counts(gen_pat, seed)
    keep = np.array([i for i, km in enumerate(kmers) if iupac.contains(sample, km)])   # k-mer index order is preserved
    mu = int(pos.sum()) / (int(pos.sum()) + int(neg.sum()))
    return pos[keep].astype(np.uint64), neg[keep].astype(np.uint64), mu


def cpu_single_sample(name, threads, inputs=None):
    """One full DP + backtrack of the oracle on the sample of a single-DP config."""
    from oracle import kp_oracle as O

    gen_pat, seed, sample, _ = SINGLE[name]
    M, U, mu = inputs if inputs is not None else sample_inputs(gen_pat, seed, sample)
    beta = (ALPHA * (1.0 - mu)) / mu
    npat, _, _ = O.plan_info(sample)
    t0 = time.perf_counter()
    res = O.single_dp(sample, M, U, ALPHA, beta, PENALTY, nthreads=threads)
    n = len(O.backtrack(sample, res["split"]))
    dt = time.perf_counter() - t0
    return {"npat": npat, "seconds": dt, "threads": threads, "partition": n, "sample": sample, "jobs": 1}


_CV_SAMPLE_JOBS = [(0, 0, 0), (3, 2, 2)]   # (fold, alpha index, penalty index): two of the 45 jobs per step


def cpu_cv_sample(threads, inputs=None):
    """Two of config 4's 45 jobs on the sample sub-problem (oracle.cv_job: train DP carrying the held-out loss)."""
    from kmerpapa_b200 import CV_tools, iupac, synthetic
    from kmerpapa_b200.score_utils import get_betas
    from oracle import kp_oracle as O

    if inputs is None:
        kmers, pos, neg = synthetic.negbin_counts(CV_GEN_PAT, CV_DATA_SEED)
        keep = np.array([i for i, km in enumerate(kmers) if iupac.contains(CV_SAMPLE, km)])
        Mf, Uf = CV_tools.sample_fold_counts(kmers, pos, neg, CV_FOLDS, np.random.RandomState(CV_SEED))
        inputs = (Mf, Uf, keep)
    Mf, Uf, keep = inputs
    M_train, U_train = Mf.sum() - Mf.sum(axis=0), Uf.sum() - Uf.sum(axis=0)
    Mtot, Utot = Mf.sum(axis=1)[keep], Uf.sum(axis=1)[keep]
    npat, _, _ = O.plan_info(CV_SAMPLE)
    t0 = time.perf_counter()
    for f, a_i, p_i in _CV_SAMPLE_JOBS:
        beta = get_betas(CV_ALPHAS[a_i], M_train, U_train)[f]
        O.cv_job(CV_SAMPLE, Mtot, Utot, Mf[keep, f], Uf[keep, f], CV_ALPHAS[a_i], beta, CV_PENALTIES[p_i], nthreads=threads)
    dt = time.perf_counter() - t0
    return {"npat": npat, "seconds": dt, "threads": threads, "sample": CV_SAMPLE, "jobs": len(_CV_SAMPLE_JOBS), "inputs": inputs}


def numba_reference_timing():
    """The unmodified numba reference (baseline/_ref) on the 7-mer NNNMNNN, one core, fresh process; JIT share from a
    second fresh process on a tiny general pattern.  Returns a dict for cpu_baseline.numba."""
    script = os.path.join(ROOT, "oracle", "ref_numba_timing.py")
    env = dict(os.environ)
    env.pop("OMP_NUM_THREADS", None)

    def run(gen_pat, seed):
        try:
            r = subprocess.run([sys.executable, script, gen_pat, str(seed), str(NUMBA_ALPHA), str(NUMBA_PENALTY)],
                               stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, env=env)
            if r.returncode != 0:
                return {"unavailable": "reference run failed: " + (r.stderr.strip().splitlines() or ["?"])[-1][:200]}
            return json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:  # noqa: BLE001
            return {"unavailable": repr(e)[:200]}

    big = run(NUMBA_GEN_PAT, NUMBA_SEED)
    if "unavailable" in big:
        return big
    tiny = run("NAN", 1)
    jit_s = tiny.get("seconds") if "unavailable" not in tiny else None
    return {"value": big["npat"] / big["seconds"], "unit": "patterns/s", "cores": f"1 of {host_threads()}",
            "seconds": big["seconds"], "jit_s": jit_s,
            "value_without_jit": big["npat"] / (big["seconds"] - jit_s) if jit_s and big["seconds"] > jit_s else None,
            "workload": f"{NUMBA_GEN_PAT} single DP + backtrack ({big['npat']} patterns), synthetic counts seed {NUMBA_SEED}, "
                        f"alpha {NUMBA_ALPHA}, penalty {NUMBA_PENALTY}: kmerpapa.algorithms.bottum_up_array_w_numba."
                        "pattern_partition_bottom_up of the unmodified reference v0.2.4, fresh process",
            "loss_bits": big["loss_bits"], "patterns": big["patterns"], "partition_sha256": big["partition_sha256"],
            "numba": big["numba"]}


def gpu_matches_numba(nb, local):
    """The GPU path on the numba run's input: same loss bits and the same partition, name for name."""
    from kmerpapa_b200 import iupac, synthetic
    from kmerpapa_b200.algorithms import bottum_up_array_w_numba as single

    kmers, pos, neg = synthetic.negbin_counts(NUMBA_GEN_PAT, NUMBA_SEED)
    mu = int(pos.sum()) / (int(pos.sum()) + int(neg.sum()))
    beta = (NUMBA_ALPHA * (1.0 - mu)) / mu
    loss, patnums = single.partition_from_arrays(NUMBA_GEN_PAT, synthetic.codes_of(kmers), pos, neg, NUMBA_ALPHA, beta,
                                                 NUMBA_PENALTY, device=local)
    PE = iupac.PatternEnumeration(NUMBA_GEN_PAT)
    names = [PE.num2pattern(p) for p in patnums]
    same = (f"{int(np.float32(loss).view(np.uint32)):08x}" == nb["loss_bits"]
            and hashlib.sha256("\n".join(names).encode()).hexdigest() == nb["partition_sha256"])
    if not same:
        raise AssertionError(f"GPU result differs from the numba reference on {NUMBA_GEN_PAT}: loss {loss} / {len(names)} patterns "
                             f"vs bits {nb['loss_bits']} / {nb['patterns']} patterns")
    return True


def run_reference(args, emit):
    """--impl reference: the reference's CPU path (oracle port, all host threads) on the bounded sample of the config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    name = args.config if args.config != "auto" else ("cfg3" if world == 1 else "cfg4")
    threads = host_threads()
    if name == "cfg4":
        inputs = cpu_cv_sample(threads)["inputs"]
        step = lambda: cpu_cv_sample(threads, inputs)   # noqa: E731
        what = (f"two of the 45 CV jobs (fold, alpha, penalty index {_CV_SAMPLE_JOBS}) per step on the sub-problem of k-mers starting "
                f"with A ({CV_SAMPLE}, 170859375 patterns each): train DP carrying the held-out loss")
    else:
        gen_pat, seed, sample, _ = SINGLE[name]
        inputs = sample_inputs(gen_pat, seed, sample)
        step = lambda: cpu_single_sample(name, threads, inputs)   # noqa: E731
        what = f"the DP restricted to k-mers whose first free position is A ({sample}), full DP + backtrack per step"
    for _ in range(max(0, args.warmup - 1)):   # the inputs call above was one warm-up of the cfg4 sample
        step()
    times = []
    for _ in range(args.steps):
        r = step()
        times.append(r["seconds"])
    ms = 1e3 * sum(times) / len(times)
    value = r["jobs"] * r["npat"] / (ms / 1e3)
    sample = f"{what}; {r['jobs'] * r['npat']} pattern-scores per step; oracle C restatement of the numba path, OpenMP"
    cpu = {"value": value, "unit": "patterns/s", "cores": r["threads"], "kind": "port", "sample": sample}
    if world == 1 and not args.no_numba:
        cpu["numba"] = numba_reference_timing()
    line = {
        "impl": "reference", "metric": "pattern-scores/sec", "value": value, "unit": "patterns/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if name == "cfg4" else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_for(name, world),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "patterns/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# GPU legs
# ---------------------------------------------------------------------------------------------
def check_single_against_golden(name, loss, patnums):
    """Loss bits, partition size and SHA-256 of the partition against the oracle's full-size run.  Returns the
    `parity` object of the line; raises on a mismatch."""
    g = golden(name)
    if g is None:
        return {"checked": False, "why": f"no golden for {name} in tests/golden/fullsize.json"}
    got = {"loss_bits": f"{int(np.float32(loss).view(np.uint32)):08x}", "partition_patterns": int(len(patnums)),
           "partition_sha256": hashlib.sha256(np.ascontiguousarray(patnums, dtype="<u8").tobytes()).hexdigest()}
    for k, v in got.items():
        if g[k] != v:
            raise AssertionError(f"{name}: {k} = {v} differs from the oracle golden {g[k]}")
    return {"checked": True, "against": "tests/golden/fullsize.json (CPU oracle, full size)", **got}


def bench_single(args, name, rank, world, local):
    import torch

    from kmerpapa_b200 import synthetic
    from kmerpapa_b200.algorithms import bottum_up_array_w_numba as single
    from kmerpapa_b200.engine import get_plan

    gen_pat, seed, _sample, _text = SINGLE[name]
    dev = torch.device("cuda", local)
    kmers, pos, neg = synthetic.negbin_counts(gen_pat, seed)
    codes, _c = pinned(synthetic.codes_of(kmers))
    pos_p, _p = pinned(pos)
    neg_p, _n = pinned(neg)
    mu = int(pos.sum()) / (int(pos.sum()) + int(neg.sum()))
    beta = (ALPHA * (1.0 - mu)) / mu
    max_count = int(pos.sum()) + int(neg.sum())
    plan = get_plan(gen_pat, local)
    npat = plan.npat
    kM, kU = plan.pack_counts(codes, pos_p, neg_p)

    def device_step(ev=None):
        eM, eU = plan.expand(kM, kU)
        if ev:
            ev[0].record()
        best, kept = plan.dp_single(eM, eU, max_count, ALPHA, beta, PENALTY)
        if ev:
            ev[1].record()
        patnums = plan.backtrack(best, kept)
        return plan.top_score(best), patnums

    sampler = ClockSampler(local)
    for _ in range(args.warmup):
        loss, patnums = device_step()
    barrier_sync(world)
    sampler.start()
    l0 = plan.launches
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    start.record()
    for s in range(args.steps):
        loss, patnums = device_step(kev[s])
    end.record()
    barrier_sync(world)
    clocks = sampler.stop()
    launches = plan.launches - l0
    ms_total = max_over_ranks(start.elapsed_time(end), world, dev)
    ms_step = ms_total / args.steps
    dp_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps        # the DP wave kernels alone
    value = world * npat / (ms_step / 1e3)
    parity = check_single_against_golden(name, loss, patnums)

    # end to end through the public array API: host buffers in, partition out
    def e2e_step():
        return single.partition_from_arrays(gen_pat, codes, pos_p, neg_p, ALPHA, beta, PENALTY, device=local)

    e2e_step()
    barrier_sync(world)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        loss2, pat2 = e2e_step()
    barrier_sync(world)
    e2e_ms = max_over_ranks(1e3 * (time.perf_counter() - t0), world, dev) / args.steps
    assert loss2 == loss and np.array_equal(pat2, patnums)

    peak, peak_kind = measured_peak()
    achieved = ALGO_BYTES_SINGLE * npat / (dp_ms / 1e3) / 1e9
    info = plan.info
    traffic, capture = load_traffic(f"{name}_single_dp")
    line = {
        "metric": "pattern-scores/sec", "value": value, "unit": "patterns/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_for(name, world),
        "result": {"loss": float(loss), "partition_patterns": int(len(patnums))},
        "parity_checked": bool(parity["checked"]), "parity": parity,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_capture": capture,
                     "kernel": f"{plan.dp_kernel_name()} (fused lazy score + min-plus), all {int(info.high_levels)} wave launches of one DP",
                     "kernel_ms": dp_ms, "algorithmic_bytes_per_pattern": ALGO_BYTES_SINGLE, "peak_kind": peak_kind},
        "e2e": {"value": world * npat / (e2e_ms / 1e3), "unit": "patterns/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(codes.nbytes + pos_p.nbytes + neg_p.nbytes),
                "d2h_bytes_per_step": int(4 + 8 * len(patnums) + 16)},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    return line, {"loss": np.array([loss], dtype=np.float32), "partition": patnums.astype(np.float64)}


def check_cv_against_golden(res, best):
    g = golden("cfg4")
    if g is None:
        return {"checked": False, "why": "no golden for cfg4 in tests/golden/fullsize.json"}
    want = np.array([int(x, 16) for x in g["job_bits"]], dtype=np.uint32).reshape(res.shape)
    got = np.ascontiguousarray(res).view(np.uint32)
    for f, a, p in g["jobs_run"]:
        if not np.array_equal(got[0, f, a, p], want[0, f, a, p]):
            raise AssertionError(f"cfg4 job (fold {f}, alpha {CV_ALPHAS[a]}, penalty {CV_PENALTIES[p]}): (train, held-out) bits "
                                 f"{got[0, f, a, p]} differ from the oracle golden {want[0, f, a, p]}")
    out = {"checked": True, "against": "tests/golden/fullsize.json (CPU oracle, full size)", "jobs_compared": len(g["jobs_run"])}
    if "selected" in g:
        if [best[0], best[1]] != g["selected"][:2] or f"{int(np.float32(best[2]).view(np.uint32)):08x}" != g["selected_bits"]:
            raise AssertionError(f"cfg4 selection {best} differs from the oracle golden {g['selected']}")
        out["selected_compared"] = True
    return out


def bench_cv(args, rank, world, local):
    import torch

    from kmerpapa_b200 import CV_tools, synthetic
    from kmerpapa_b200.algorithms import bottum_up_array_penalty_plus_pseudo_CV as cv
    from kmerpapa_b200.engine import get_plan

    steps, warmup = args.steps, args.warmup
    dev = torch.device("cuda", local)
    kmers, pos, neg = synthetic.negbin_counts(CV_GEN_PAT, CV_DATA_SEED)
    codes = synthetic.codes_of(kmers)
    plan = get_plan(CV_GEN_PAT, local)
    npat = plan.npat
    prng = np.random.RandomState(CV_SEED)
    folds = CV_tools.sample_fold_counts(kmers, pos, neg, CV_FOLDS, prng)      # host sampler, outside the timed region
    njobs = CV_FOLDS * len(CV_ALPHAS) * len(CV_PENALTIES)

    def step():
        runner = cv.GpuFoldRunner(CV_GEN_PAT, codes, pos, neg, device=local)
        res = cv.run_grid(CV_GEN_PAT, kmers, codes, pos, neg, CV_ALPHAS, CV_PENALTIES, CV_FOLDS, 1, CV_SEED, runner=runner,
                          presampled=[folds])
        return res, cv.select_best(CV_ALPHAS, CV_PENALTIES, res, 1, CV_FOLDS, len(CV_GEN_PAT))

    sampler = ClockSampler(local)
    for _ in range(warmup):
        res, best = step()
    barrier_sync(world)
    sampler.start()
    l0 = plan.launches
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    start.record()
    for _ in range(steps):
        res, best = step()
    end.record()
    barrier_sync(world)
    wall_ms = 1e3 * (time.perf_counter() - t0)     # host clock around the same steps, barrier included: the end-to-end time
    clocks = sampler.stop()
    launches = plan.launches - l0
    ms_step = max_over_ranks(start.elapsed_time(end), world, dev) / steps
    e2e_ms_step = max_over_ranks(wall_ms, world, dev) / steps
    value = njobs * npat / (ms_step / 1e3)
    peak, peak_kind = measured_peak()
    achieved = ALGO_BYTES_CV * njobs * npat / (ms_step / 1e3) / 1e9 / world
    parity = check_cv_against_golden(res, best)
    out = {"jobs": njobs, "steps": steps, "warmup": warmup, "wall_s": ms_step / 1e3, "pattern_scores_per_s": value,
           "e2e_wall_s": e2e_ms_step / 1e3, "e2e_pattern_scores_per_s": njobs * npat / (e2e_ms_step / 1e3),
           "selected": [best[0], best[1], float(best[2])], "parity_checked": bool(parity["checked"]), "parity": parity,
           "launches": int(launches), "clocks": clocks, "achieved_gbs_per_gpu": achieved, "frac_per_gpu": achieved / peak,
           "peak": peak, "peak_kind": peak_kind}
    return out, {"cv_losses": np.asarray(res, dtype=np.float32),
                 "cv_selected": np.array([best[0], best[1], best[2]], dtype=np.float64)}


def bench_sharded_dp(args, rank, world, local):
    """Secondary N>1 measurement: ONE 9-mer DP (config 3) sharded over the ranks (kmerpapa_b200/sharded.py, replicated
    mode: rows pushed to their readers over NVLink inside the DP kernel).  Device time, max over ranks, best of the
    timed steps."""
    import torch
    import torch.distributed as dist

    from kmerpapa_b200 import sharded, synthetic
    from kmerpapa_b200.engine import get_plan

    gen_pat, seed = SINGLE["cfg3"][:2]
    kmers, pos, neg = synthetic.negbin_counts(gen_pat, seed)
    plan = get_plan(gen_pat, local)
    kM, kU = plan.pack_counts(synthetic.codes_of(kmers), pos, neg)
    eM, eU = plan.expand(kM, kU)
    mc = int(pos.sum() + neg.sum())
    mu = int(pos.sum()) / mc
    beta = ALPHA * (1.0 - mu) / mu
    sh = sharded.ShardedDP(plan, rank, world, replicate=True)
    sh.connect()
    ms = []
    for _ in range(args.warmup + args.steps):
        sh.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sh.run(eM, eU, mc, ALPHA, beta, PENALTY)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=plan.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms.append(float(t.item()))
    part = sh.backtrack()
    top = float(sh.top_score())
    parity = check_single_against_golden("cfg3", np.float32(top), part)
    sh.close()
    ms = ms[args.warmup:]
    best = min(ms)
    return ({"workload": "cfg3 single 9-mer DP sharded by the top high digit, replicated mode", "ms": best,
             "pattern_scores_per_s": plan.npat / (best / 1e3), "partition_patterns": int(len(part)), "loss": top,
             "parity_checked": bool(parity["checked"]), "reps_ms": [round(x, 3) for x in ms]},
            {"sharded_loss": np.array([top], dtype=np.float32), "sharded_partition": part.astype(np.float64)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto", "cfg3", "cfg4", "cfg5", "n9m"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numba", action="store_true", help="skip the timing of the unmodified numba reference (about a minute)")
    ap.add_argument("--no-cv", action="store_true", help="N=1: skip the secondary CV-grid measurement")
    ap.add_argument("--no-sharded", action="store_true", help="N>1: skip the secondary sharded single-DP measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of each GPU measurement to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    # stdout carries exactly one JSON line: everything else that writes to file descriptor 1 (the NCCL banner,
    # stray prints of libraries) is sent to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    if args.impl == "reference":
        run_reference(args, emit)
        return
    rank, world, local = dist_setup(args.gpus)
    name = args.config if args.config != "auto" else ("cfg3" if world == 1 else "cfg4")
    if name != "cfg4":
        line, outputs = bench_single(args, name, rank, world, local)
        if world == 1 and name == "cfg3" and not args.no_cv:
            line["cv_grid"], cv_outputs = bench_cv(args, rank, world, local)
            line["cv_grid"]["note"] = ("config 4 on this one GPU: the N = 1 point of the strong-scaling curve whose N > 1 points are "
                                       "the `value` of `bench.py --gpus N`")
            outputs.update(cv_outputs)
    else:
        cvres, outputs = bench_cv(args, rank, world, local)
        traffic, capture = load_traffic("cfg4_cv_job")
        line = {
            "metric": "pattern-scores/sec", "value": cvres["pattern_scores_per_s"], "unit": "patterns/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cvres["wall_s"] * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_for("cfg4", world),
            "result": {"selected": cvres["selected"]},
            "parity_checked": cvres["parity_checked"], "parity": cvres["parity"],
            "roofline": {"bound": "hbm", "achieved": cvres["achieved_gbs_per_gpu"], "peak": cvres["peak"], "unit": "GB/s",
                         "frac": cvres["frac_per_gpu"], "traffic": traffic, "traffic_capture": capture,
                         "kernel": "the single-DP kernel on train counts + backtrack/leaf kernels, per GPU, per job",
                         "algorithmic_bytes_per_pattern": ALGO_BYTES_CV, "peak_kind": cvres["peak_kind"]},
            "e2e": {"value": cvres["e2e_pattern_scores_per_s"], "unit": "patterns/s", "ms_per_step": cvres["e2e_wall_s"] * 1e3,
                    "h2d_bytes_per_step": int(65536 * 8 * 3 * 6), "d2h_bytes_per_step": int(8 * cvres["jobs"]),
                    "note": "host clock around the same steps (every step packs the host fold tables, H2D, runs its jobs, reads "
                            "every job's losses back, D2H, and gathers them over NCCL), max over ranks"},
            "cv_grid": cvres, "gpu_launches": cvres["launches"], "clocks": cvres["clocks"],
        }
        if not args.no_sharded and 1 < world <= 8:
            line["sharded_single_dp"], sharded_outputs = bench_sharded_dp(args, rank, world, local)
            outputs.update(sharded_outputs)
    if rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for key, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, key + ".npy"), arr)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        r = cpu_single_sample(name, threads) if name != "cfg4" else cpu_cv_sample(threads)
        line["cpu_baseline"] = {
            "value": r["jobs"] * r["npat"] / r["seconds"], "unit": "patterns/s", "cores": r["threads"], "kind": "port",
            "sample": f"{r['sample']}: the DP restricted to k-mers whose first free position is A, {r['jobs']} x {r['npat']} patterns, "
                      f"{r['seconds']:.1f} s, oracle C restatement of the numba path with OpenMP"}
        if not args.no_numba:
            nb = numba_reference_timing()
            if "unavailable" not in nb:
                nb["gpu_result_identical"] = gpu_matches_numba(nb, local)
            line["cpu_baseline"]["numba"] = nb
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)


if __name__ == "__main__":
    main()
