"""Kernel time of lrb_dev_table_spectrum on five tables against a 2 GiB device-to-device copy in the same process, and
the wall time of the file-level lrb_table_spectrum on a 15mers-counts file.  One JSON line per measurement on stdout
(and appended to --out).  Usage: bench_spectrum.py [--out FILE] [--reps N]

Tables: (a) config #2 (1 M ONT reads, counted on the device), (b) config #4 (500 k HiFi reads), (c) all zeros,
(d) every entry 1, (e) uniform random values in [0, 64).  The kernel reads the canonical half, 2^31 bytes, which is far
larger than the 126 MB L2, so every launch streams from HBM.  The copy moves 2^31 bytes each way; its rate counts both
directions (what HBM carries), and `fraction_of_copy` is the kernel's read rate over that.
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
from lrbinner_b200.profile import _ptr, dev_count, dev_table_spectrum  # noqa: E402
from lrbinner_b200.synth import CONFIGS, SynthSpec  # noqa: E402

DEV = "cuda:0"
M = 65536
CANON_BYTES = 2 ** 31


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return {"gpu": name, "power_limit": power}


def median_ms(fn, reps, before=None):
    for _ in range(3):                     # warm-up
        if before:
            before()
        fn()
    ms = []
    for _ in range(reps):
        if before:
            before()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), float(min(ms)), float(max(ms))


def config_table(name):
    cfg = CONFIGS[name]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, _ = spec.device_reads(DEV)
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, table)
    torch.cuda.synchronize()
    del dr
    return table


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_spectrum.py needs a CUDA device")
    info = gpu_info()
    lines = []

    def emit(d):
        d = {**info, **d}
        print(json.dumps(d), flush=True)
        lines.append(d)

    src = torch.empty(CANON_BYTES // 4, dtype=torch.int32, device=DEV)
    dst = torch.empty_like(src)
    src.fill_(1)
    c_med, c_min, c_max = median_ms(lambda: dst.copy_(src), args.reps)
    copy_rate = 2 * CANON_BYTES / (c_med * 1e-3) / 1e9
    emit({"what": "copy_2GiB_d2d", "ms_median": c_med, "ms_min": c_min, "ms_max": c_max, "GBps_read_plus_write": copy_rate})
    del src, dst
    torch.cuda.empty_cache()

    spec = torch.zeros(M + 3, dtype=torch.int64, device=DEV)
    work = None
    tables = [("a_cfg2_ont", lambda: config_table("cfg2_1M_5kb_ont_k4")),
              ("b_cfg4_hifi", lambda: config_table("cfg4_500k_15kb_hifi_k5")),
              ("c_zeros", lambda: torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)),
              ("d_ones", lambda: torch.ones(2 ** 30, dtype=torch.int32, device=DEV)),
              ("e_uniform_0_64", lambda: torch.randint(0, 64, (2 ** 30,), dtype=torch.int32, device=DEV,
                                                        generator=torch.Generator(device=DEV).manual_seed(7)))]
    for name, make in tables:
        table = make()
        ms, mn, mx = median_ms(lambda: dev_table_spectrum(table, M, out=spec), args.reps, before=spec.zero_)
        s = spec.cpu().numpy().view(np.uint64)
        assert int(s[:M + 1].sum()) == 2 ** 29, name       # every canonical key counted once
        rate = CANON_BYTES / (ms * 1e-3) / 1e9
        emit({"what": "k_table_spectrum", "table": name, "max_count": M, "ms_median": ms, "ms_min": mn, "ms_max": mx,
              "GBps_read": rate, "fraction_of_copy": rate / copy_rate, "n0_fraction": float(s[0]) / 2 ** 29,
              "n1_fraction": float(s[1]) / 2 ** 29, "max_count_seen": int(s[M + 2]), "keys_over_max": int(s[M])})
        if name == "a_cfg2_ont":           # keep a file of this table for the file-level call
            base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 12 * 2 ** 30 else None
            work = tempfile.mkdtemp(prefix="lrb_spectrum_", dir=base)
            host = table.cpu().numpy()
            _lib.check(_lib.lib.lrb_table_write_file(f"{work}/15mers-counts".encode(), _ptr(host)))
            del host
        del table
        torch.cuda.empty_cache()

    try:
        for rep in range(2):
            t0 = time.perf_counter()
            _lib.check(_lib.lib.lrb_table_spectrum(f"{work}/15mers-counts".encode(), f"{work}/15mers-histo".encode(), M))
            dt = time.perf_counter() - t0
            emit({"what": "lrb_table_spectrum_file", "table": "a_cfg2_ont", "rep": rep, "wall_s": dt,
                  "file_bytes": os.path.getsize(f"{work}/15mers-counts"), "histo_lines": sum(1 for _ in open(f"{work}/15mers-histo"))})
    finally:
        shutil.rmtree(work, ignore_errors=True)
    if args.out:
        with open(args.out, "a") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
