"""Cost and host memory of segmented input: the file-level calls on a config-#1-size FASTA (0.5 Gbases) and on a
5-Gbase FASTA, each read as one segment and in 4 and 16 forced segments (LRB_SEGMENT_BASES), plus the 5-Gbase file at
the budget of config #1's 4 segments (the same fixed budget on both sizes).  Every run is a child process: its wall time
per file-level call, its peak resident memory (VmHWM), its stderr notice, and the sha256 of every file it wrote, which
must equal the one-segment run's.  One JSON line per run on stdout (and appended to --out).

Usage: bench_segments.py [--out FILE] [--big-reads N] [--threads T]
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from lrbinner_b200.synth import CONFIGS, SynthSpec  # noqa: E402

K, BS, BC = 3, 32, 10

CHILD = r"""
import json, os, sys, time
sys.path.insert(0, sys.argv[1])
from lrbinner_b200 import runners_utils
mode, fasta, out, threads = sys.argv[2], sys.argv[3], sys.argv[4], int(sys.argv[5])
k, bs, bc = %d, %d, %d
calls = {}
def timed(name, fn, *a, **kw):
    t = time.perf_counter()
    fn(*a, **kw)
    calls[name] = time.perf_counter() - t
if mode == "fused":
    timed("run_profile", runners_utils.run_profile, fasta, out, k, bs, bc, threads, write_table=True)
else:
    timed("run_kmers", runners_utils.run_kmers, fasta, out, k, threads)
    timed("run_15mer_counts", runners_utils.run_15mer_counts, fasta, out, threads)
    timed("run_15mer_vecs", runners_utils.run_15mer_vecs, fasta, out, bs, bc, threads)
hwm = [l for l in open("/proc/self/status") if l.startswith("VmHWM:")][0].split()[1]
print(json.dumps({"calls_s": calls, "vmhwm_kb": int(hwm)}))
""" % (K, BS, BC)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power}


def write_reads(path, spec):
    """FASTA of a synthetic read set, one line per sequence, written from the generator's ASCII buffer"""
    bases, offsets = spec.host_ascii()
    mv = memoryview(bases)
    with open(path, "wb", buffering=1 << 24) as f:
        for i in range(spec.n_reads):
            f.write(b">r%d\n" % i)
            f.write(mv[int(offsets[i]):int(offsets[i + 1])])
            f.write(b"\n")
    return int(offsets[-1])


def sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    return h.hexdigest()


def run(mode, fasta, work, threads, budget):
    out = os.path.join(work, "out")
    shutil.rmtree(out, ignore_errors=True)
    env = dict(os.environ)
    env.pop("LRB_SEGMENT_BASES", None)
    if budget:
        env["LRB_SEGMENT_BASES"] = str(budget)
    p = subprocess.run([sys.executable, "-c", CHILD, ROOT, mode, fasta, out, str(threads)], env=env, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"{mode} budget={budget}: rc {p.returncode}\n{p.stdout}\n{p.stderr}")
    rec = json.loads(p.stdout.strip().splitlines()[-1])
    rec["notice"] = [line for line in p.stderr.splitlines() if "segments" in line]
    rec["files"] = {name: sha(f"{out}/profiles/{name}") for name in ("com_profs", "cov_profs", "15mers-counts")}
    shutil.rmtree(out, ignore_errors=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--big-reads", type=int, default=1_000_000, help="reads of the large FASTA (gamma 5 kb: ~5 Gbases)")
    ap.add_argument("--small-reads", type=int, default=CONFIGS["cfg1_100k_5kb_k3"]["n_reads"])
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
    args = ap.parse_args()
    info = gpu_info()
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 24 * 2 ** 30 else None
    work = tempfile.mkdtemp(prefix="lrb_bench_seg_", dir=base)
    fixed = None
    try:
        cfg = CONFIGS["cfg1_100k_5kb_k3"]
        for label, n, seed in (("cfg1_0.5G", args.small_reads, cfg["seed"]), ("ont_5G", args.big_reads, 1234)):
            fasta = os.path.join(work, f"{label}.fa")
            bases = write_reads(fasta, SynthSpec(n, lengths="gamma5k", errors="ont", seed=seed))
            budgets = [("one_segment", None), ("4_segments", -(-bases // 4)), ("16_segments", -(-bases // 16))]
            if fixed is None:
                fixed = budgets[1][1]
            else:
                budgets.append(("fixed_budget_of_cfg1_4_segments", fixed))
            want = None
            for blabel, budget in budgets:
                for mode in ("fused", "three"):
                    rec = run(mode, fasta, work, args.threads, budget)
                    if want is None:
                        want = rec["files"]
                    rec.update({"input": label, "reads": n, "bases": bases, "file_bytes": os.path.getsize(fasta),
                                "segments": blabel, "segment_bases": budget, "mode": mode, "files_equal_one_segment": rec["files"] == want,
                                "k": K, "bin_size": BS, "bins": BC, "threads": args.threads, **info})
                    del rec["files"]
                    line = json.dumps(rec)
                    print(line, flush=True)
                    if args.out:
                        with open(args.out, "a") as f:
                            f.write(line + "\n")
            os.remove(fasta)
    finally:
        shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
