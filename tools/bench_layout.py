"""Cost of mixed coverage rows (k_search_layout) against the kernels of the single shapes.  One JSON line per measurement on
stdout (and appended to --out).  Usage: bench_layout.py [--out FILE] [--reps N]

Config #2 (1 M ONT reads, 5 Gbases) resident on the device, the lists of all 64 buckets built once; CUDA-event times, the
two sides alternated rep by rep after two warm-up reps, rows zeroed before every rep outside the timed window.  The 4 GiB
table, its 2 GiB compact form and the 312 MB entry stream are larger than the 126 MB L2.
(a) One table, the row [(-bs 32 -bc 10), 16 geometric edges] in one call of lrb_dev_partition_search_layout (one walk)
    against k_search_keys (-bs 32 -bc 10) plus k_search_edges (the same 16 edges): two walks.  The rows must be equal.
(b) n = 2, 4, 8 compact tables, each block binned by 16 equal-mass edges from its own table's spectrum (the counted table
    copied into n slots: the same counts, separate memory) against k_search_samples with -bs 10 -bc 32 on every table.
    Both make one walk per table; the ratio is per walk.  The column sums of each block must equal spectrum_edge_mass.
    The same binning both ways separates the kernel from the binning: one slot with those edges (k_search_layout, compact
    load) against k_search_edges with the same edges on the full-layout table; the rows must be equal.
(c) k_table_spectrum in compact form (lrb_dev_compact_spectrum) against the full form on the same table.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from lrbinner_b200.profile import (CovBlock, PartitionWorkspace, dev_compact_spectrum, dev_count, dev_table_compact,  # noqa: E402
                                   dev_table_spectrum, spectrum_edge_mass, spectrum_quantile_edges)
from lrbinner_b200.synth import CONFIGS, SynthSpec  # noqa: E402

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


def alternate(reps, zero, first, second):
    t1, t2 = [], []
    for rep in range(reps + 2):                   # two warm-up reps
        zero()
        torch.cuda.synchronize()
        a = event_ms(first)
        b = event_ms(second)
        if rep >= 2:
            t1.append(a)
            t2.append(b)
    return t1, t2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_layout.py needs a CUDA device")
    info = gpu_info()
    lines = []

    def emit(d):
        d = {**info, "config": "cfg2_1M_5kb_ont_k4", "reps": args.reps, **d}
        print(json.dumps(d), flush=True)
        lines.append(d)

    cfg = CONFIGS["cfg2_1M_5kb_ont_k4"]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, _ = spec.device_reads(DEV)
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, table)
    s = dev_table_spectrum(table, 65536).cpu().numpy().view(np.uint64)
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    n = spec.n_reads

    def z(w):
        return torch.zeros((n, w), dtype=torch.int32, device=DEV), torch.zeros(n, dtype=torch.int32, device=DEV)

    # (a) one table, two blocks: one walk against two
    hl, sl = z(26)
    hk, sk = z(10)
    he, se = z(16)
    layout = [CovBlock(None, 32, 10), CovBlock(None, edges=GEOMETRIC16)]

    def zero_a():
        for t in (hl, sl, hk, sk, he, se):
            t.zero_()

    def separate():
        ws.apply(table, count=False, search=True, bin_size=32, bins=10, hist=hk, sums=sk)
        ws.search_edges(table, GEOMETRIC16, he, se)

    t_l, t_s = alternate(args.reps, zero_a, lambda: ws.search_layout(table, None, layout, hl, sl), separate)
    equal = bool(torch.equal(hl, torch.cat([hk, he], dim=1)) and torch.equal(sl, sk))
    assert equal
    emit({"what": "layout_one_table", "layout": "[(None, -bs 32 -bc 10), (None, 16 geometric edges)]", "k_search_layout": stats(t_l),
          "k_search_keys+k_search_edges": stats(t_s), "layout_over_separate": float(np.median(t_l) / np.median(t_s)), "rows_equal": equal})
    del hl, sl, hk, sk, he, se
    torch.cuda.empty_cache()

    # (b) n slots, each with equal-mass edges from its own spectrum, against k_search_samples (10, 32) per slot
    compact = dev_table_compact(table)
    own = dev_compact_spectrum(compact, 65536).cpu().numpy().view(np.uint64)
    assert np.array_equal(own, s)
    q = spectrum_quantile_edges(own, 16)
    hl, sl = z(len(q) + 1)
    he, se = z(len(q) + 1)

    def zero_s():
        for t in (hl, sl, he, se):
            t.zero_()

    t_l, t_e = alternate(args.reps, zero_s, lambda: ws.search_layout(None, [compact], [CovBlock(0, edges=q)], hl, sl),
                         lambda: ws.search_edges(table, q, he, se))
    equal = bool(torch.equal(hl, he) and torch.equal(sl, se))
    assert equal
    emit({"what": "layout_slot_same_binning", "edges_per_block": len(q), "edge_list": q, "k_search_layout_compact": stats(t_l),
          "k_search_edges_full": stats(t_e), "layout_over_edges": float(np.median(t_l) / np.median(t_e)), "rows_equal": equal})
    del hl, sl, he, se
    slots = [compact] + [compact.clone() for _ in range(7)]
    for k in (2, 4, 8):
        hl, sl = z(k * (len(q) + 1))
        hs, ss = z(k * 32)
        layout = [CovBlock(t, edges=q) for t in range(k)]

        def zero_b():
            for t in (hl, sl, hs, ss):
                t.zero_()

        t_l, t_s = alternate(args.reps, zero_b, lambda: ws.search_layout(None, slots[:k], layout, hl, sl),
                             lambda: ws.search_samples(slots[:k], [(10, 32)] * k, hs, ss))
        col = hl.sum(dim=0, dtype=torch.int64).cpu().numpy().astype(np.uint64).reshape(k, -1)
        mass_ok = all(np.array_equal(c, spectrum_edge_mass(s, q)) for c in col) and bool(torch.equal(sl, ss))
        assert mass_ok
        emit({"what": "layout_slots", "tables": k, "edges_per_block": len(q), "edge_list": q,
              "k_search_layout": stats(t_l), "k_search_samples_bs10_bc32": stats(t_s),
              "layout_over_samples_per_walk": float(np.median(t_l) / np.median(t_s)), "column_sums_equal_edge_mass": mass_ok})
        del hl, sl, hs, ss
        torch.cuda.empty_cache()
    del slots

    # (c) the spectrum of the compact form against the full form
    spec_c = torch.zeros(65539, dtype=torch.int64, device=DEV)
    spec_f = torch.zeros(65539, dtype=torch.int64, device=DEV)

    def zero_c():
        spec_c.zero_()
        spec_f.zero_()

    t_c, t_f = alternate(args.reps, zero_c, lambda: dev_compact_spectrum(compact, 65536, out=spec_c),
                         lambda: dev_table_spectrum(table, 65536, out=spec_f))
    equal = bool(torch.equal(spec_c, spec_f))
    assert equal
    emit({"what": "spectrum_compact", "k_table_spectrum_compact": stats(t_c), "k_table_spectrum_full": stats(t_f),
          "compact_over_full": float(np.median(t_c) / np.median(t_f)), "spectra_equal": equal})
    if args.out:
        with open(args.out, "a") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
