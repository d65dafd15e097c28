"""Kernel launches of one call of each coverage search entry point, and a digest of what it returned.

Usage: launch_counts.py [--tree DIR] [--parent-tree DIR] [--out FILE]

For every call (lrb_profile_host, lrb_profile_host_settings with 3 settings, lrb_profile_host_samples with 2 slots,
lrb_profile_host_edges, and each lrb_dev_partition_search_*) the library's launch profiler (lrb_prof_enable) reports the
kernel names and launch counts, and the rows and sums are hashed.  Where the package has mixed coverage rows (CovBlock), a
mixed layout goes through lrb_profile_host_layout and lrb_dev_partition_search_layout, and the 3 settings and the 2 slots are
given once more as layouts: those must launch and return exactly what the settings and samples calls did.  --tree imports
the package of another built checkout instead of this one.  --parent-tree runs this script against that tree too and exits
non-zero unless both trees launch the same kernels the same number of times and return the same rows for every call the
other tree has, and the layouts of existing shapes match their calls.  Needs one CUDA device.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def measure():
    import numpy as np
    import torch
    from lrbinner_b200 import _lib
    from lrbinner_b200.profile import (Context, PartitionWorkspace, dev_count, dev_mirror, dev_table_compact)
    from lrbinner_b200.synth import SynthSpec
    try:
        from lrbinner_b200.profile import CovBlock
    except ImportError:                  # a tree without mixed coverage rows
        CovBlock = None

    dev = "cuda:0"
    spec = SynthSpec(4000, seed=11, n_rate=1e-3, lowercase_frac=0.02, edge_lengths=True, scale=0.01)
    reads = spec.host_packed(threads=4)
    settings = [(32, 10), (8, 5), (1, 16)]
    edges = [2, 3, 5, 9, 17, 33, 65]
    results = {}

    def digest(*arrays):
        h = hashlib.sha256()
        for a in arrays:
            a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
            h.update(np.ascontiguousarray(a).tobytes())
        return h.hexdigest()[:16]

    def record(name, fn):
        torch.cuda.synchronize()
        _lib.lib.lrb_prof_enable(1)
        outs = fn()
        torch.cuda.synchronize()
        _lib.lib.lrb_prof_enable(0)
        results[name] = {"launches": {k: n for k, (n, _) in sorted(_lib.prof_report().items())}, "digest": digest(*outs)}

    ctx = Context(0)
    ctx.profile(reads, k=4, bin_size=32, bins=10)   # warm-up: module load, buffers
    record("lrb_profile_host", lambda: [(r := ctx.profile(reads, k=4, bin_size=32, bins=10))["comp"], r["hist"], r["sums"]])
    record("lrb_profile_host_settings[3]", lambda: [(r := ctx.profile(reads, coverage=settings))["hist"], r["sums"]])
    record("lrb_profile_host_edges", lambda: [(r := ctx.profile(reads, edges=edges))["hist"], r["sums"]])
    ctx.profile(reads, keep_table=True)
    ctx.sample_table_keep(0)
    ctx.sample_table_keep(3)
    record("lrb_profile_host_samples[2]", lambda: [(r := ctx.profile(reads, samples=[(0, 32, 10), (3, 8, 5)]))["hist"], r["sums"]])
    if CovBlock:
        record("layout as lrb_profile_host_settings[3]",
               lambda: [(r := ctx.profile(reads, layout=[CovBlock(None, s_, b) for s_, b in settings]))["hist"], r["sums"]])
        record("layout as lrb_profile_host_samples[2]",
               lambda: [(r := ctx.profile(reads, layout=[CovBlock(0, 32, 10), CovBlock(3, 8, 5)]))["hist"], r["sums"]])
        mixed = [CovBlock(3, edges=edges), CovBlock(None, 32, 10), CovBlock(0, 8, 5), CovBlock(3, 1, 16)]
        record("lrb_profile_host_layout[4]", lambda: [(r := ctx.profile(reads, layout=mixed))["hist"], r["sums"]])
    ctx.close()

    dr, _ = spec.device_reads(dev)
    table = torch.zeros(_lib.TABLE_ENTRIES, dtype=torch.int32, device=dev)
    dev_count(dr, table)
    dev_mirror(table)
    compact = [dev_table_compact(table), dev_table_compact(table)]
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)

    def rows(width):
        return (torch.zeros((dr.n_reads, width), dtype=torch.int32, device=dev), torch.zeros(dr.n_reads, dtype=torch.int32, device=dev))

    def search(method, width, *args):
        hist, sums = rows(width)
        getattr(ws, method)(*args, hist, sums)
        return [hist, sums]

    record("lrb_dev_partition_search_settings[1]", lambda: search("search_settings", 10, table, settings[:1]))
    record("lrb_dev_partition_search_settings[3]", lambda: search("search_settings", 31, table, settings))
    record("lrb_dev_partition_search_samples[2]", lambda: search("search_samples", 15, compact, [(32, 10), (8, 5)]))
    record("lrb_dev_partition_search_edges", lambda: search("search_edges", len(edges) + 1, table, edges))
    if CovBlock:
        record("lrb_dev_partition_search_layout[4]", lambda: search("search_layout", 39, table, [compact[0], None, None, compact[1]], mixed))
    return results


# layouts of existing shapes and the calls whose launches and rows they must repeat
SAME_AS = {"layout as lrb_profile_host_settings[3]": "lrb_profile_host_settings[3]",
           "layout as lrb_profile_host_samples[2]": "lrb_profile_host_samples[2]"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=None, help="import the package from this built checkout")
    ap.add_argument("--parent-tree", default=None, help="a built checkout to compare with")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.tree or ROOT))
    if args.parent_tree:
        got = {}
        for build, tree in (("parent", args.parent_tree), ("branch", args.tree or ROOT)):
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--tree", os.path.abspath(tree)], capture_output=True,
                                 text=True, check=True, cwd=os.path.abspath(tree)).stdout
            got[build] = json.loads(out.splitlines()[-1])
        parent, branch = got["parent"], got["branch"]
        ref = {name: parent.get(name, branch.get(SAME_AS.get(name))) for name in branch}   # what each call must equal
        verdict = {name: "same" if ref[name] == branch[name] else "new" if ref[name] is None else "DIFFERENT" for name in branch}
        same = all(name in branch for name in parent) and "DIFFERENT" not in verdict.values()
        report = {"same": same, **got}
        for name in branch:
            print(f"{name:40s} {verdict[name]} {json.dumps(branch[name])}")
        if args.out:
            with open(args.out, "w") as f:
                json.dump(report, f, indent=1)
        sys.exit(0 if same else 1)
    print(json.dumps(measure()))


if __name__ == "__main__":
    main()
