"""Cost of binning coverage by count edges (k_search_edges) against the (bin size, bin count) rule (k_search_keys).  One
JSON line per measurement on stdout (and appended to --out).  Usage: bench_edges.py [--out FILE] [--reps N]

(a) Config #2 (1 M ONT reads, 5 Gbases) resident on the device: CUDA-event time of lrb_dev_partition_search_edges over all
    64 buckets against lrb_dev_partition_apply_range mode 2 with -bs 32 -bc 10 over the same lists, timed alternately rep
    by rep, for four edge sets: {2..10}, 16 geometric bins from 2, 32 equal-mass bins from the table's spectrum
    (spectrum_quantile_edges) and 4095 edges.  The rows are zeroed before every rep, outside the timed window.  The 4 GiB
    table and the 312 MB entry stream are larger than the 126 MB L2.  Each set's column sums are checked against
    spectrum_edge_mass.  Then edges {2..B} against -bs 1 -bc B (B = 10, 20, 32), the same rows both ways, so the difference
    is the binning alone and not the number of distinct cells the REDs hit.
(b) Config #1 (100 k reads, 0.5 Gbases) as a FASTA file: wall clock of run_15mer_vecs_edges (16 geometric bins) against
    run_15mer_vecs (-bs 32 -bc 10), alternately; edges {2..5} are checked to write the -bs 1 -bc 5 file byte for byte.
"""
import argparse
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

from lrbinner_b200 import _lib, runners_utils  # noqa: E402
from lrbinner_b200.profile import (PartitionWorkspace, dev_count, dev_table_spectrum, spectrum_edge_mass,  # noqa: E402
                                   spectrum_quantile_edges)
from lrbinner_b200.synth import CONFIGS, SynthSpec, write_fasta  # noqa: E402

DEV = "cuda:0"
GEOMETRIC16 = [2 << i for i in range(15)]      # 16 bins: [0, 2), [2, 4), ..., [32768, inf)


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
    s = dev_table_spectrum(table, 65536).cpu().numpy().view(np.uint64)
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    n = spec.n_reads
    sets = {"2..10": list(range(2, 11)), "geometric16": GEOMETRIC16, "quantile32": spectrum_quantile_edges(s, 32),
            "4095": list(range(2, 2002)) + [2002 + 7 * i for i in range(_lib.MAX_BINS - 1 - 2000)]}
    # the same rows both ways: edges {2..B} against -bs 1 -bc B, so the two kernels issue the same REDs
    same = {f"2..{B}": B for B in (10, 20, 32)}
    for name, edges in list(sets.items()) + [(f"same {k}", list(range(2, B + 1))) for k, B in same.items()]:
        bs, bc = (1, len(edges) + 1) if name.startswith("same") else (32, 10)
        hk = torch.zeros((n, bc), dtype=torch.int32, device=DEV)
        sk = torch.zeros(n, dtype=torch.int32, device=DEV)
        he = torch.zeros((n, len(edges) + 1), dtype=torch.int32, device=DEV)
        se = torch.zeros(n, dtype=torch.int32, device=DEV)

        def run_edges():
            ws.search_edges(table, edges, he, se)

        def run_keys():
            ws.apply(table, count=False, search=True, bin_size=bs, bins=bc, hist=hk, sums=sk)

        t_e, t_k = [], []
        for rep in range(reps + 2):                   # two warm-up reps
            he.zero_(); se.zero_(); hk.zero_(); sk.zero_()
            torch.cuda.synchronize()
            a = event_ms(run_edges)
            b = event_ms(run_keys)
            if rep >= 2:
                t_e.append(a)
                t_k.append(b)
        col = he.sum(dim=0, dtype=torch.int64).cpu().numpy().astype(np.uint64)
        mass_ok = bool(np.array_equal(col, spectrum_edge_mass(s, edges)))
        assert mass_ok and torch.equal(se, sk), name
        if bs == 1:
            assert torch.equal(he, hk), name
        emit({"what": "edges_search_device", "config": "cfg2_1M_5kb_ont_k4", "edges": name, "bins": len(edges) + 1,
              "reps": reps, "k_search_edges": stats(t_e), "k_search_keys": stats(t_k), "keys_setting": [bs, bc],
              "rows_equal": bs == 1,
              "edges_over_keys": float(np.median(t_e) / np.median(t_k)), "column_sums_equal_edge_mass": mass_ok,
              "edge_list": edges if len(edges) <= 32 else f"{len(edges)} edges, {edges[0]}..{edges[-1]}"})
        del he, se, hk, sk
        torch.cuda.empty_cache()
    del ws, table, dr
    torch.cuda.empty_cache()


def file_level(emit, reps, threads):
    cfg = CONFIGS["cfg1_100k_5kb_k3"]
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 12 * 2 ** 30 else None
    work = tempfile.mkdtemp(prefix="lrb_edges_", dir=base)
    try:
        spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
        fasta = os.path.join(work, "cfg1.fa")
        write_fasta(fasta, spec.host_sequences())
        runners_utils.run_15mer_counts(fasta, work, threads)
        prof = os.path.join(work, "profiles")
        runners_utils.run_15mer_vecs_edges(fasta, work, [2, 3, 4, 5], threads)
        runners_utils.run_15mer_vecs(fasta, work, 1, 5, threads)
        equal = open(f"{prof}/cov_profs_edges", "rb").read() == open(f"{prof}/cov_profs", "rb").read()
        assert equal, "edges {2..5} differ from -bs 1 -bc 5"
        for rep in range(reps):
            t0 = time.perf_counter()
            runners_utils.run_15mer_vecs_edges(fasta, work, GEOMETRIC16, threads)
            t_edges = time.perf_counter() - t0
            t0 = time.perf_counter()
            runners_utils.run_15mer_vecs(fasta, work, 32, 10, threads)
            t_keys = time.perf_counter() - t0
            emit({"what": "edges_search_file", "config": "cfg1_100k_5kb_k3", "input": "FASTA", "rep": rep, "threads": threads,
                  "wall_s_run_15mer_vecs_edges_geometric16": t_edges, "wall_s_run_15mer_vecs_bs32_bc10": t_keys,
                  "edges_over_keys": t_edges / t_keys, "edges_2_to_5_equal_bs1_bc5": equal})
    finally:
        shutil.rmtree(work, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--file-reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_edges.py needs a CUDA device")
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
