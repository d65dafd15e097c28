"""bench.py's bookkeeping on the CPU: the per-kernel table, the choice of the dominant single kernel and the committed
DRAM-traffic record it quotes (no GPU, no timing here)."""
import json
import os

from conftest import ROOT

import bench


def test_kernel_table_gives_every_kernel_its_8d_bytes_and_bound():
    L, V, n, P, B, hbm = 5.0e9, 4.986e9, 1_000_000, 136, 10, 6550.4
    steps = 5
    prof = {"k_composition": (5, 11.7), "k_step_hist": (15, 12.4), "k_group_scan": (15, 0.3), "k_partition": (15, 36.5),
            "k_sample_cells": (5, 0.65), "k_plan_cells": (5, 0.6), "k2_partition": (15, 55.5), "k_count_smem": (5, 15.2),
            "k_count_keys": (5, 0.2), "k_count_spill": (5, 0.05), "k_search_keys": (5, 102.4), "k_row_sums": (5, 0.06), "k_mirror": (5, 3.4)}
    traffic, src = bench.load_traffic("cfg2_1M_5kb_ont_k4", 1_000_000)
    assert src and traffic["k_search_keys"]["dram_bytes_per_step"] > 4e10       # profiles/traffic.json is of the headline workload
    rows = bench.kernel_table(prof, steps, L, V, n, P, B, hbm, traffic)
    assert set(rows) == set(prof)
    dom = max(rows, key=lambda k: rows[k]["ms_per_step"])
    assert dom == "k_search_keys"                                               # the dominant SINGLE kernel, not a group
    s = rows["k_search_keys"]
    assert abs(s["algorithmic_bytes"] - (0.375 * L + 4 * V + 4 * n * B)) < 1      # SURVEY 8(d): 0.375 L + 4 V + 4 N B
    assert 0.15 < s["frac_of_hbm"] < 0.18 and 0.8 < s["alt_bound"]["frac"] < 0.9
    assert s["dram_traffic_bytes_per_step"] == traffic["k_search_keys"]["dram_bytes_per_step"]
    for name in ("k_step_hist", "k_group_scan", "k_partition", "k_sample_cells", "k_plan_cells", "k2_partition"):
        assert rows[name]["overhead"] and rows[name]["algorithmic_bytes"] == 0     # the partition chain: no bytes in 8(d)
    assert abs(rows["k_count_smem"]["algorithmic_bytes"] - (0.375 * L + 16 * V)) < 1
    assert abs(rows["k_composition"]["algorithmic_bytes"] - (0.25 * L + 4 * n * P)) < 1
    assert rows["k_mirror"]["algorithmic_bytes"] == 2.0 ** 32 and rows["k_mirror"]["launches_per_step"] == 1


def test_dump_outputs_is_a_fixed_exact_sample_under_64_mb(tmp_path):
    """--dump-outputs: the same rows and table entries every run, u32 values exact (the table's above 2^31 too), <= 64 MB at k = 5"""
    import numpy as np
    import torch
    n, P, B = 40000, 512, 10
    comp = torch.randint(0, 5000, (n, P), dtype=torch.int32)
    comp[:, 0] = torch.arange(n, dtype=torch.int32)                     # row i carries i
    hist = comp[:, :B] * 3
    sums = comp[:, 0] + 7
    table = torch.from_numpy((np.arange(1 << 22, dtype=np.uint32) * np.uint32(1021)).view(np.int32))   # entry i holds 1021 i < 2^32
    a = bench.sample_outputs(comp, hist, sums, table)
    b = bench.sample_outputs(comp, hist, sums, table)
    assert set(a) == {"comp", "hist", "sums", "table"} and all(np.array_equal(a[x], b[x]) for x in a)
    rows = a["comp"][:, 0].astype(np.int64)
    assert len(rows) == bench.DUMP_ROWS and np.all(np.diff(rows) > 0)
    assert np.array_equal(a["comp"], comp.numpy()[rows]) and np.array_equal(a["hist"], hist.numpy()[rows])
    assert np.array_equal(a["sums"], sums.numpy()[rows])
    keys = a["table"] / 1021
    assert a["table"].dtype == np.float64 and len(keys) == bench.DUMP_KEYS and a["table"].max() > 2 ** 31
    assert np.array_equal(keys, np.floor(keys)) and np.all(np.diff(keys) > 0)
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    bench.write_outputs(str(tmp_path / "out"), a)
    for name, x in a.items():
        y = np.load(tmp_path / "out" / f"{name}.npy")
        assert y.dtype in (np.float32, np.float64) and np.array_equal(x, y)


def test_committed_bench_lines_carry_the_contract_keys():
    """the lines kept under profiles/ (what DESIGN.md quotes) have the keys the contract names"""
    for name in ("r02_bench_n1_final.json", "r02_bench_n2_final.json", "r02_bench_n4_final.json", "r02_bench_n8_final.json"):
        d = json.loads(open(os.path.join(ROOT, "profiles", name)).read())
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                    "data", "config", "e2e", "gpu_launches", "roofline", "clocks"):
            assert key in d, (name, key)
        assert d["dtype"] == "u32" and d["vs_baseline"] is None and d["gpu_launches"] > 0
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
        if d["n_gpus"] == 1:
            assert d["roofline"]["kernel"] == "k_search_keys" and d["cpu_baseline"]["kind"] == "reference"
            assert d["file_level"]["parity_vs_reference_tools"] is True
        else:
            assert d["verify"]["ok"] is True and d["verify"]["oracle_spot_check"]["mismatches"] == 0
            assert len(d["north_star"]) == 3 and all(r["verify"]["digests_equal_across_plans"] for r in d["north_star"])
