"""Cost of binning several coverage settings in one search, against one search per setting in the same process.  One JSON
line per measurement on stdout (and appended to --out).  Usage: bench_cov_settings.py [--out FILE] [--reps N]

(a) Config #2 (1 M ONT reads, 5 Gbases) resident on the device: CUDA-event time of lrb_dev_partition_search_settings over
    all 64 buckets with the first M of eight settings (M = 1, 2, 4, 6, 8), and of M single-setting searches
    (lrb_dev_partition_apply_range mode 2) over the same lists; the two are timed alternately, rep by rep.  The histogram
    rows are zeroed before every rep, outside the timed window.  The 4 GiB table and the 312 MB entry stream are larger
    than the 126 MB L2.  Every rep's column blocks are checked against the single searches.
(b) Config #1 (100 k reads, 0.5 Gbases) as a FASTA file: wall clock of one lrb_search_15mers_settings call with the six
    golden settings against six lrb_search_15mers calls, alternately; the files of the two must be equal byte for byte.
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

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from lrbinner_b200 import _lib  # noqa: E402
from lrbinner_b200.profile import PartitionWorkspace, dev_count  # noqa: E402
from lrbinner_b200.synth import CONFIGS, SynthSpec, write_fasta  # noqa: E402

DEV = "cuda:0"
GOLDEN_SETTINGS = [(10, 8), (32, 10), (1, 5), (3, 1), (10, 32), (2, 3)]
EIGHT = GOLDEN_SETTINGS + [(5, 20), (64, 16)]


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


def device_resident(emit, reps):
    cfg = CONFIGS["cfg2_1M_5kb_ont_k4"]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, _ = spec.device_reads(DEV)
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, table)
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    n = spec.n_reads
    for M in (1, 2, 4, 6, 8):
        S = EIGHT[:M]
        W = sum(b for _, b in S)
        hist = torch.zeros((n, W), dtype=torch.int32, device=DEV)
        sums = torch.zeros(n, dtype=torch.int32, device=DEV)
        singles = [torch.zeros((n, b), dtype=torch.int32, device=DEV) for _, b in S]
        s1 = torch.zeros_like(sums)

        def run_settings():
            ws.search_settings(table, S, hist, sums)

        def run_singles():
            for (bs, bc), h in zip(S, singles):
                ws.apply(table, count=False, search=True, bin_size=bs, bins=bc, hist=h, sums=s1)

        t_set, t_one = [], []
        for rep in range(reps + 2):                   # two warm-up reps
            hist.zero_(); sums.zero_()
            for h in singles:
                h.zero_()
            s1.zero_()
            torch.cuda.synchronize()
            a = event_ms(run_settings)
            b = event_ms(run_singles)
            if rep >= 2:
                t_set.append(a)
                t_one.append(b)
        off = 0
        for (bs, bc), h in zip(S, singles):
            assert torch.equal(hist[:, off:off + bc], h), (M, bs, bc)
            off += bc
        assert torch.equal(sums, s1)
        emit({"what": "settings_search_device", "config": "cfg2_1M_5kb_ont_k4", "M": M, "W": W, "settings": S, "reps": reps,
              "settings_call": stats(t_set), "single_calls": stats(t_one),
              "single_calls_over_settings_call": float(np.median(t_one) / np.median(t_set)), "results_equal": True})
        del hist, sums, singles, s1
        torch.cuda.empty_cache()
    del ws, table, dr
    torch.cuda.empty_cache()


def file_level(emit, reps, threads):
    cfg = CONFIGS["cfg1_100k_5kb_k3"]
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 12 * 2 ** 30 else None
    work = tempfile.mkdtemp(prefix="lrb_cov_settings_", dir=base)
    try:
        spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
        fasta = os.path.join(work, "cfg1.fa")
        write_fasta(fasta, spec.host_sequences())
        tbl = os.path.join(work, "15mers-counts").encode()
        _lib.check(_lib.lib.lrb_count_15mers(fasta.encode(), tbl, threads))
        n = len(GOLDEN_SETTINGS)
        multi = [os.path.join(work, f"multi_bs{s}_bc{b}").encode() for s, b in GOLDEN_SETTINGS]
        single = [os.path.join(work, f"single_bs{s}_bc{b}").encode() for s, b in GOLDEN_SETTINGS]
        bs = (C.c_long * n)(*[s for s, _ in GOLDEN_SETTINGS])
        bc = (C.c_int * n)(*[b for _, b in GOLDEN_SETTINGS])
        outs = (C.c_char_p * n)(*multi)
        for rep in range(reps):
            t0 = time.perf_counter()
            _lib.check(_lib.lib.lrb_search_15mers_settings(tbl, fasta.encode(), n, bs, bc, outs, None, threads))
            t_multi = time.perf_counter() - t0
            t0 = time.perf_counter()
            for (s, b), path in zip(GOLDEN_SETTINGS, single):
                _lib.check(_lib.lib.lrb_search_15mers(tbl, fasta.encode(), path, s, b, threads))
            t_single = time.perf_counter() - t0
            equal = all(open(a, "rb").read() == open(b, "rb").read() for a, b in zip(multi, single))
            assert equal, "files differ"
            emit({"what": "settings_search_file", "config": "cfg1_100k_5kb_k3", "input": "FASTA", "settings": GOLDEN_SETTINGS,
                  "rep": rep, "threads": threads, "wall_s_one_settings_call": t_multi, "wall_s_six_search_calls": t_single,
                  "six_calls_over_one": t_single / t_multi, "files_equal": equal,
                  "bytes": [os.path.getsize(p) for p in multi]})
    finally:
        shutil.rmtree(work, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--file-reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_cov_settings.py needs a CUDA device")
    info = gpu_info()
    lines = []

    def emit(d):
        d = {**info, **d}
        print(json.dumps(d), flush=True)
        lines.append(d)

    device_resident(emit, args.reps)
    file_level(emit, args.file_reps, os.cpu_count() or 8)
    if args.out:
        with open(args.out, "a") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
