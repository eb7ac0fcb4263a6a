"""Run under torchrun on N GPUs with KP_SHARD_CV=1: the CLI's cross-validation runs every job as one DP sharded over the
ranks (ShardedFoldRunner) and must write the stdout, CVfile and stderr lines of the recorded single-process reference
runs, byte for byte (a collective runner keeps the single-process order of the progress lines).
Usage: KP_SHARD_CV=1 torchrun --nproc-per-node N tests/mgpu_sharded_cv_check.py"""
import contextlib
import io
import json
import os
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")


def _golden_path(arg):
    """An input file of a recorded run, found under this checkout's tests/golden (the run recorded its own absolute path)."""
    _, sep, rest = arg.partition("/tests/golden/")
    return os.path.join(GOLDEN, rest) if sep else arg


def main():
    from kmerpapa_b200 import cli
    from kmerpapa_b200.algorithms import bottum_up_array_penalty_plus_pseudo_CV as cv

    runners = []
    choose = cv.sharded_cv_runner

    def recording(*a, **k):   # which runner the CV picked
        r = choose(*a, **k)
        runners.append(type(r).__name__)
        return r

    cv.sharded_cv_runner = recording
    rank = int(os.environ.get("RANK", "0"))
    ok = True
    for name in ("cli_cfg2_7mers.json", "cli_5mers_iterations2.json"):
        g = json.load(open(os.path.join(GOLDEN, name)))
        argv = [_golden_path(a) for a in g["argv"]]
        d = tempfile.mkdtemp()
        out, cvf = os.path.join(d, "out.txt"), os.path.join(d, "cv.txt")
        err = io.StringIO()
        del runners[:]
        with contextlib.redirect_stderr(err):
            rc = cli.main(argv + ["-o", out, "--CVfile", cvf])
        if rank == 0:
            lines = [l for l in err.getvalue().splitlines() if "Warning" not in l and not l.startswith("  ")]
            ref = [l for l in g["stderr"] if not l.startswith("  ")]
            same = (rc == g["rc"] and open(out).read() == g["stdout"] and open(cvf).read() == g["cvfile"] and lines == ref
                    and runners == ["ShardedFoldRunner"])
            print(name, "OK" if same else "MISMATCH", runners, flush=True)
            if lines != ref:
                print("\n".join(lines), flush=True)
            ok = ok and same
    if rank == 0:
        print("CLI SHARDED CV OK" if ok else "CLI SHARDED CV MISMATCH", flush=True)
    import torch.distributed as dist

    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
