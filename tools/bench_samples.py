"""Cost of searching reads against several samples' 15-mer tables in one pass, against one search per table in the same
process.  One JSON line per measurement on stdout (and appended to --out).
Usage: bench_samples.py [--out FILE] [--reps N] [--file-reps N] [--parent-tree DIR]

(a) Config #2 (1 M ONT reads, 5 Gbases) resident on the device, against n = 1, 2, 4, 8 sample tables (the reads' own table
    and tables counted from other synthetic communities), all with -bs 10 -bc 32: CUDA-event time of
    lrb_dev_partition_search_samples over all 64 buckets (one walk per table, G = 1) and of n single-table searches
    (lrb_dev_partition_apply_range mode 2 against the full-layout tables) over the same lists; the two are timed
    alternately, rep by rep, with the rows zeroed outside the timed window.  The tables (2 GiB compact, 4 GiB full) and the
    312 MB entry stream are larger than the 126 MB L2.  Every rep's blocks are checked against the single searches.
    (Two tables per walk, G = 2, was measured 1.28-1.30x slower than G = 1: profiles/r06_samples_bench.jsonl.)
(b) Loading a page-cached table file: lrb_ctx_sample_table_load (canonical rows, 2 GiB read) against lrb_ctx_table_load
    (4 GiB), alternately.
(c) Config #1 (100 k reads, 0.5 Gbases) as a FASTA file against 3 tables: one lrb_search_15mers_samples call against
    3 lrb_search_15mers calls plus pasting their columns, alternately; the files must be equal byte for byte.
(d) With --parent-tree: the bench.py step of the parent commit's tree and of this tree, alternated.
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from lrbinner_b200 import _lib  # noqa: E402
from lrbinner_b200.profile import Context, PartitionWorkspace, dev_count, dev_table_compact  # noqa: E402
from lrbinner_b200.synth import CONFIGS, SynthSpec, write_fasta  # noqa: E402

DEV = "cuda:0"
BS, BC = 10, 32


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power}


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def stats(ms):
    return {"ms_median": float(np.median(ms)), "ms_min": float(min(ms)), "ms_max": float(max(ms))}


def other_community(cfg, i, n_reads):
    return SynthSpec(n_reads, lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"] + 1000 + i)


def device_resident(emit, reps):
    cfg = CONFIGS["cfg2_1M_5kb_ont_k4"]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, _ = spec.device_reads(DEV)
    full = [torch.zeros(2 ** 30, dtype=torch.int32, device=DEV) for _ in range(8)]
    dev_count(dr, full[0])
    for i in range(1, 8):   # other communities, a fifth of config #2's size each
        dri, _ = other_community(cfg, i, cfg["n_reads"] // 5).device_reads(DEV)
        dev_count(dri, full[i])
        del dri
    compact = [dev_table_compact(t) for t in full]
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    n = spec.n_reads
    for nt in (1, 2, 4, 8):
        S = [(BS, BC)] * nt
        hist = torch.zeros((n, BC * nt), dtype=torch.int32, device=DEV)
        sums = torch.zeros(n, dtype=torch.int32, device=DEV)
        singles = [torch.zeros((n, BC), dtype=torch.int32, device=DEV) for _ in range(nt)]
        s1 = torch.zeros(n, dtype=torch.int32, device=DEV)

        def run_samples():
            ws.search_samples(compact[:nt], S, hist, sums)

        def run_singles():
            for t, h in enumerate(singles):
                ws.apply(full[t], count=False, search=True, bin_size=BS, bins=BC, hist=h, sums=s1)

        t = {1: [], "single": []}
        for rep in range(reps + 2):                   # two warm-up reps
            hist.zero_()
            sums.zero_()
            for h in singles:
                h.zero_()
            s1.zero_()
            torch.cuda.synchronize()
            ms = {1: event_ms(run_samples), "single": event_ms(run_singles)}
            if rep >= 2:
                for k, v in ms.items():
                    t[k].append(v)
        for i, h in enumerate(singles):
            assert torch.equal(hist[:, i * BC:(i + 1) * BC], h), (nt, i)
        assert torch.equal(sums, s1)
        emit({"what": "samples_search_device", "config": "cfg2_1M_5kb_ont_k4", "n_tables": nt, "W": BC * nt, "setting": [BS, BC],
              "reps": reps, "G1": stats(t[1]), "single_calls": stats(t["single"]),
              "single_calls_over_G1": float(np.median(t["single"]) / np.median(t[1])), "results_equal": True})
        del hist, sums, singles, s1
        torch.cuda.empty_cache()
    del ws, full, compact, dr
    torch.cuda.empty_cache()


def work_dir():
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 24 * 2 ** 30 else None
    return tempfile.mkdtemp(prefix="lrb_samples_", dir=base)


def count_file(work, name, spec, threads):
    fasta = os.path.join(work, f"{name}.fa")
    write_fasta(fasta, spec.host_sequences())
    tbl = os.path.join(work, f"{name}.15mers-counts")
    _lib.check(_lib.lib.lrb_count_15mers(fasta.encode(), tbl.encode(), threads))
    return fasta, tbl


def load_times(emit, reps, tbl):
    ctx = Context(0)
    ctx.table_load(tbl)                              # page cache warm, buffers allocated
    ctx.sample_table_load(0, tbl)
    for rep in range(reps):
        t0 = time.perf_counter()
        ctx.sample_table_load(0, tbl)
        t_slot = time.perf_counter() - t0
        t0 = time.perf_counter()
        ctx.table_load(tbl)
        t_table = time.perf_counter() - t0
        emit({"what": "table_load", "rep": rep, "page_cached": True, "wall_s_sample_table_load_2GiB": t_slot,
              "wall_s_table_load_4GiB": t_table, "table_over_sample": t_table / t_slot})
    ctx.close()


def file_level(emit, reps, threads, work):
    cfg = CONFIGS["cfg1_100k_5kb_k3"]
    fasta, own = count_file(work, "cfg1", SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"]), threads)
    tables = [own] + [count_file(work, f"other{i}", other_community(cfg, i, cfg["n_reads"] // 2), threads)[1] for i in (1, 2)]
    load_times(emit, reps, own)
    n = len(tables)
    multi = os.path.join(work, "cov_profs_samples")
    single = [os.path.join(work, f"single{t}") for t in range(n)]
    pasted = os.path.join(work, "pasted")
    paths = (C.c_char_p * n)(*[t.encode() for t in tables])
    bs = (C.c_long * n)(*[BS] * n)
    bc = (C.c_int * n)(*[BC] * n)
    for rep in range(reps):
        t0 = time.perf_counter()
        _lib.check(_lib.lib.lrb_search_15mers_samples(paths, n, bs, bc, fasta.encode(), multi.encode(), None, threads))
        t_multi = time.perf_counter() - t0
        t0 = time.perf_counter()
        for tbl, out in zip(tables, single):
            _lib.check(_lib.lib.lrb_search_15mers(tbl.encode(), fasta.encode(), out.encode(), BS, BC, threads))
        files = [open(p, "rb") for p in single]
        with open(pasted, "wb") as f:
            for lines in zip(*files):
                f.write(b" ".join(x.rstrip(b"\n") for x in lines) + b"\n")
        for fh in files:
            fh.close()
        t_single = time.perf_counter() - t0
        equal = open(multi, "rb").read() == open(pasted, "rb").read()
        assert equal, "files differ"
        emit({"what": "samples_search_file", "config": "cfg1_100k_5kb_k3", "input": "FASTA", "n_tables": n, "setting": [BS, BC],
              "rep": rep, "threads": threads, "wall_s_one_samples_call": t_multi, "wall_s_three_search_calls_and_paste": t_single,
              "three_calls_over_one": t_single / t_multi, "files_equal": equal, "bytes": os.path.getsize(multi)})


def bench_py_steps(emit, parent_tree, rounds):
    cmd = ["--gpus", "1", "--steps", "5", "--warmup", "3", "--no-cpu-baseline"]
    order = 0
    for _ in range(rounds):
        for build, tree in (("parent", parent_tree), ("branch", ROOT)):
            tree = os.path.abspath(tree)
            out = subprocess.run([sys.executable, os.path.join(tree, "bench.py")] + cmd, capture_output=True, text=True, check=True,
                                 cwd=tree).stdout
            line = [json.loads(x) for x in out.splitlines() if x.startswith("{")][-1]
            emit({"what": "bench_py_step", "build": build, "order": order, "command": "bench.py " + " ".join(cmd),
                  "config": line.get("config"), "ms_per_step": line.get("ms_per_step"), "Gbases_per_s": line.get("Gbases_per_s"),
                  "e2e_ms_per_step": line.get("e2e_ms_per_step")})
            order += 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--file-reps", type=int, default=3)
    ap.add_argument("--parent-tree", default=None, help="a built checkout of the parent commit: time its bench.py step beside this one")
    ap.add_argument("--bench-rounds", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_samples.py needs a CUDA device")
    info = gpu_info()
    lines = []

    def emit(d):
        d = {**info, **d}
        print(json.dumps(d), flush=True)
        lines.append(d)

    try:
        device_resident(emit, args.reps)
        work = work_dir()
        try:
            file_level(emit, args.file_reps, os.cpu_count() or 8, work)
        finally:
            shutil.rmtree(work, ignore_errors=True)
        if args.parent_tree:
            bench_py_steps(emit, args.parent_tree, args.bench_rounds)
    finally:
        if args.out:
            with open(args.out, "a") as f:
                for d in lines:
                    f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
