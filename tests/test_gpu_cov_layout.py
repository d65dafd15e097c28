"""GPU tier (-m gpu): mixed coverage rows (layouts of blocks, each on any table and binned by (bin_size, bins) or by edges).

Edges {2, 3, 4, 5} are the rule of -bs 1 -bc 5, so the golden files of -bs 1 -bc 5, -bs 3 -bc 1 and -bs 32 -bc 10 joined
by one space check the file-level path byte for byte in every input mode.  Other layouts are checked against the oracle's
window keys (numpy searchsorted and the reference's bin rule), against the single-block calls, and at full size against
the spectrum's bin and edge mass."""
import gzip
import os
import shutil

import numpy as np
import pytest

from conftest import GOLDEN, golden_inputs
from edge_inputs import plant, value_pool

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

from oracle import oracle  # noqa: E402
from lrbinner_b200 import _lib, runners_utils  # noqa: E402
from lrbinner_b200.profile import (Context, CovBlock, DeviceReads, PackedReads, PartitionWorkspace, dev_compact_spectrum,  # noqa: E402
                                   dev_count, dev_mirror, dev_table_compact, dev_table_spectrum, spectrum_bin_mass,
                                   spectrum_edge_mass, spectrum_quantile_edges)
from lrbinner_b200.synth import CONFIGS, SynthSpec  # noqa: E402

DEV = "cuda:0"
GEOMETRIC = [2 ** i for i in range(1, 17)]
GOLDEN_LAYOUT = [CovBlock(0, edges=[2, 3, 4, 5]), CovBlock(0, 3, 1), CovBlock(0, 32, 10)]
GOLDEN_PARTS = [(1, 5), (3, 1), (32, 10)]


class _env:
    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kw}
        os.environ.update({k: str(v) for k, v in self.kw.items()})

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _z(*shape):
    return torch.zeros(shape, dtype=torch.int32, device=DEV)


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _golden_joined(stem):
    parts = []
    for bs, bc in GOLDEN_PARTS:
        with gzip.open(os.path.join(GOLDEN, f"{stem}.cov_bs{bs}_bc{bc}.txt.gz"), "rb") as f:
            parts.append(f.read().splitlines())
    assert len({len(p) for p in parts}) == 1
    return b"".join(b" ".join(line) + b"\n" for line in zip(*parts))


def _layout_files_equal_golden(reads, out, stem, table_reads=None):
    """count the table of `table_reads` (default: the reads), then the golden layout on it; text and .npy against the
    golden lines of -bs 1 -bc 5, -bs 3 -bc 1 and -bs 32 -bc 10 joined by one space"""
    runners_utils.run_15mer_counts(table_reads or reads, out, 4)
    table = f"{out}/profiles/15mers-counts"
    runners_utils.run_15mer_vecs_layout(reads, out, [table], GOLDEN_LAYOUT, 4, write_npy=True)
    path = f"{out}/profiles/cov_profs_layout"
    txt = open(path, "rb").read()
    assert txt == _golden_joined(stem), stem
    want = np.array([[float(x) for x in line.split()] for line in txt.decode().splitlines() if line.strip()]).reshape(-1, 16)
    assert np.array_equal(np.load(path + ".npy"), want), stem
    assert open(path + ".layout").read() == f"{table}\tedges 2 3 4 5\n{table}\tbs 3 bc 1\n{table}\tbs 32 bc 10\n"
    assert not os.path.exists(f"{out}/profiles/cov_profs")
    shutil.rmtree(f"{out}/profiles")     # the 4 GiB table


# ---- 1. file level against the reference's bytes -------------------------------------------------------------

@pytest.mark.parametrize("name", golden_inputs())
def test_layout_writes_the_golden_lines(name, tmp_path):
    _layout_files_equal_golden(os.path.join(GOLDEN, name), str(tmp_path), name.split(".")[0])


def test_tiny_segments_gzip_and_batches(tmp_path, capfd):
    src = os.path.join(GOLDEN, "g06_community.fa")
    with _env(LRB_SEGMENT_BASES=max(1, PackedReads.from_file(src).total_bases // 5)):
        _layout_files_equal_golden(src, str(tmp_path / "seg"), "g06_community")
    assert "segments" in capfd.readouterr().err
    gz = tmp_path / "g04_format.gz"
    with gzip.open(gz, "wb") as f:
        f.write(open(os.path.join(GOLDEN, "g04_format.fq"), "rb").read())
    with _env(LRB_SEGMENT_BASES=max(1, PackedReads.from_file(str(gz)).total_bases // 4)):
        _layout_files_equal_golden(str(gz), str(tmp_path / "gz"), "g04_format")
    with _env(LRB_BATCH_BASES=9000):
        _layout_files_equal_golden(src, str(tmp_path / "batched"), "g06_community")
    assert "batch(es)" in capfd.readouterr().err


def test_contigs_mode(tmp_path):
    reads = os.path.join(GOLDEN, "g06_community.fa")
    frags = os.path.join(GOLDEN, "g10_fragments.fasta")
    _layout_files_equal_golden(frags, str(tmp_path / "whole"), "g10_contigs_mode", table_reads=reads)
    with _env(LRB_SEGMENT_BASES=3000):
        _layout_files_equal_golden(frags, str(tmp_path / "seg"), "g10_contigs_mode", table_reads=reads)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus(tmp_path, capfd):
    with _env(LRB_GPUS=2, LRB_MIN_BLOCKS_PER_DEVICE=1, LRB_VERBOSE=1):
        _layout_files_equal_golden(os.path.join(GOLDEN, "g06_community.fa"), str(tmp_path), "g06_community")
    assert "on 2 GPU(s)" in capfd.readouterr().err
    seqs, pr = _synthetic(17)
    layout = [CovBlock(None, 32, 10), CovBlock(0, edges=GEOMETRIC), CovBlock(None, edges=[2, 5, 9])]
    one, two = Context(0), Context([0, 1])
    for c in (one, two):
        c.profile(_synthetic(5)[1], keep_table=True)
        c.sample_table_keep(0)
    with _env(LRB_MIN_BLOCKS_PER_DEVICE=1):
        a = one.profile(pr, k=4, layout=layout)
        b = two.profile(pr, k=4, layout=layout)
        assert two.info()["n_devices"] == 2
    for key in ("comp", "hist", "sums"):
        assert np.array_equal(a[key], b[key]), key
    one.close()
    two.close()


def test_runner_leaves_cov_profs_alone(tmp_path):
    src = os.path.join(GOLDEN, "g06_community.fa")
    out = str(tmp_path)
    runners_utils.run_15mer_counts(src, out, 4)
    runners_utils.run_15mer_vecs(src, out, 32, 10, 4)
    before = open(f"{out}/profiles/cov_profs", "rb").read()
    runners_utils.run_15mer_vecs_layout(src, out, [f"{out}/profiles/15mers-counts"], [CovBlock(0, edges=GEOMETRIC)], 4)
    assert open(f"{out}/profiles/cov_profs", "rb").read() == before
    assert sorted(os.listdir(f"{out}/profiles")) == ["15mers-counts", "cov_profs", "cov_profs_layout", "cov_profs_layout.layout"]
    shutil.rmtree(f"{out}/profiles")


# ---- 2. against the oracle: every block over the window keys ------------------------------------------------------

def _synthetic(seed):
    spec = SynthSpec(2500, seed=seed, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.005)
    seqs = spec.host_sequences() + [b"", b"ACGT", b"N" * 40, b"acgtacgtacgtacgtacgtacgt", b"ACGTTGCA" * 3000]
    return seqs, PackedReads.from_sequences(seqs, threads=4)


def _bin(cnt, block):
    """the bins of counts `cnt` (u64) under one block's rule"""
    if block.edges is not None:
        return np.searchsorted(np.asarray(block.edges, np.uint64), cnt, side="right")
    S, B = int(block.bin_size), int(block.bins)
    c = np.where(cnt < 2, 0, cnt).astype(np.int64)
    pos = c // S - 1
    return np.where(c <= S, 0, np.where((pos > 0) & (pos < B), pos, B - 1))


def _oracle_block(keys, table, block):
    """hist [n, width] of one block: the table's count of every window key, binned"""
    w = len(block.edges) + 1 if block.edges is not None else int(block.bins)
    hist = np.zeros((len(keys), w), np.uint32)
    for i, k in enumerate(keys):
        hist[i] = np.bincount(_bin(table[k].astype(np.uint64), block), minlength=w)
    return hist


def _oracle_rows(keys, tables, layout):
    hist = np.concatenate([_oracle_block(keys, tables[b.table], b) for b in layout], axis=1)
    return hist, np.array([k.size for k in keys], np.uint32)


@pytest.fixture(scope="module")
def three_tables():
    """a context with two other samples' counted tables in slots 0 and 1 and the reads' own table as its table; the
    oracle's table of each (None = the context's)"""
    seqs, pr = _synthetic(17)
    c = Context(0)
    host = {}
    for slot, seed in ((0, 5), (1, 6)):
        s2, p2 = _synthetic(seed)
        host[slot] = c.profile(p2, want_table=True)["table"].copy()
        c.sample_table_keep(slot)
    host[None] = c.profile(pr, want_table=True)["table"].copy()
    for key, src in ((0, _synthetic(5)[0]), (None, seqs)):     # the counted tables are the oracle's
        t = oracle.Table()
        for s in src:
            t.count(s)
        assert np.array_equal(t.array, host[key]), key
        t.close()
    keys = [oracle.window_keys(s) for s in seqs]
    yield c, seqs, pr, keys, host
    c.close()


def _layouts(c, host):
    q = {t: spectrum_quantile_edges(c.sample_table_spectrum(t), 16) for t in (0, 1)}
    q[None] = spectrum_quantile_edges(c.table_spectrum(), 16)
    top = int(max(h.max() for h in host.values()))
    return {
        "per-slot quantiles": [CovBlock(0, edges=q[0]), CovBlock(1, edges=q[1]), CovBlock(None, edges=q[None])],
        "one table twice": [CovBlock(0, edges=GEOMETRIC), CovBlock(0, edges=q[0]), CovBlock(None, 32, 10)],
        "interleaved 1 0 1": [CovBlock(1, 32, 10), CovBlock(0, edges=GEOMETRIC), CovBlock(1, edges=[2, 3, 4, 5])],
        "eight": [CovBlock(None, 32, 10), CovBlock(0, edges=GEOMETRIC), CovBlock(1, 8, 5), CovBlock(None, edges=q[None]),
                  CovBlock(0, 1, 16), CovBlock(1, edges=[2]), CovBlock(None, edges=[]), CovBlock(0, 10, 8)],
        "W 4096": [CovBlock(0, edges=list(range(2, 2 + 2047))), CovBlock(None, edges=list(range(2, 2 + 2046))), CovBlock(1, 3, 1)],
        "above": [CovBlock(0, edges=[top + 1, top + 2, 2 ** 32 - 1]), CovBlock(None, 32, 10), CovBlock(1, edges=[top + 5])],
    }


def test_layouts_against_the_oracle_and_the_single_block_calls(three_tables):
    c, seqs, pr, keys, host = three_tables
    layouts = _layouts(c, host)
    assert all(len(e) >= 4 for e in (layouts["per-slot quantiles"][m].edges for m in range(3)))
    assert sum(b.bins if b.edges is None else len(b.edges) + 1 for b in layouts["W 4096"]) == _lib.MAX_BINS
    for name, layout in layouts.items():
        got = c.profile(pr, layout=layout, use_loaded_table=True)
        want_hist, want_sums = _oracle_rows(keys, host, layout)
        assert np.array_equal(got["sums"], want_sums), name
        assert np.array_equal(got["hist"], want_hist), name
        # each block is the single-block call's row
        for m, b in enumerate(layout):
            one = c.profile(pr, layout=[b], use_loaded_table=True)
            assert np.array_equal(got["hists"][m], one["hist"]) and np.array_equal(got["sums"], one["sums"]), (name, m)


def test_existing_shapes_take_their_kernels(three_tables):
    """a layout one of the settings, samples or edges calls could take launches that call's kernels and returns its rows"""
    c, seqs, pr, keys, host = three_tables
    cases = [
        ([CovBlock(None, 32, 10)], dict(bin_size=32, bins=10), "k_search_keys"),
        ([CovBlock(None, 32, 10), CovBlock(None, 8, 5)], dict(coverage=[(32, 10), (8, 5)]), "k_search_settings"),
        ([CovBlock(0, 32, 10), CovBlock(1, 8, 5), CovBlock(0, 1, 5)], dict(samples=[(0, 32, 10), (1, 8, 5), (0, 1, 5)]), "k_search_samples"),
        ([CovBlock(None, edges=GEOMETRIC)], dict(edges=GEOMETRIC), "k_search_edges"),
        ([CovBlock(None, 32, 10), CovBlock(None, edges=GEOMETRIC)], None, "k_search_layout"),
    ]
    for layout, kw, kernel in cases:
        runs = []
        for args in ([dict(layout=layout)] + ([kw] if kw else [])):
            torch.cuda.synchronize()
            _lib.lib.lrb_prof_enable(1)
            r = c.profile(pr, use_loaded_table=True, **args)
            _lib.lib.lrb_prof_enable(0)
            runs.append((r, {k: n for k, (n, _) in _lib.prof_report().items()}))
        assert kernel in runs[0][1], (kernel, runs[0][1])
        if kw:
            assert "k_search_layout" not in runs[0][1] and runs[0][1] == runs[1][1], (runs[0][1], runs[1][1])
            assert np.array_equal(runs[0][0]["hist"], runs[1][0]["hist"]) and np.array_equal(runs[0][0]["sums"], runs[1][0]["sums"])


def test_slot_spectrum_equals_the_table_spectrum(three_tables, tmp_path):
    c, seqs, pr, keys, host = three_tables
    c.sample_table_keep(2)      # the context's (counted) table
    assert np.array_equal(c.sample_table_spectrum(2), c.table_spectrum())
    assert np.array_equal(c.sample_table_spectrum(2, 40), c.table_spectrum(40))
    # a planted table with counts over the whole u32 range, through a file
    rng = np.random.default_rng(29)
    nz = np.flatnonzero(host[None][: _lib.TABLE_ENTRIES]).astype(np.int64)
    canon = nz[(nz & (1 << 15)) == 0]
    planted = np.zeros(_lib.TABLE_ENTRIES, np.uint32)
    planted[canon] = plant(canon, rng, value_pool(rng))
    path = str(tmp_path / "planted")
    _lib.check(_lib.lib.lrb_table_write_file(path.encode(), planted.ctypes.data))
    del planted
    d = Context(0)
    d.table_load(path)
    d.sample_table_keep(0)
    d.sample_table_load(1, path)
    for mc in (65536, 2 ** 24, 2):
        want = d.table_spectrum(mc)
        assert np.array_equal(d.sample_table_spectrum(0, mc), want) and np.array_equal(d.sample_table_spectrum(1, mc), want), mc
    with pytest.raises(_lib.LrbError) as e:
        d.sample_table_spectrum(5)
    assert e.value.code == _lib.LRB_EINVAL and "empty" in str(e.value)
    d.close()
    os.remove(path)


def test_planted_tables_against_the_oracle():
    """u32 counts over the whole range (edge_inputs.value_pool) through the device-level search, full and compact tables
    together, in key shards"""
    seqs, pr = _synthetic(17)
    dr = DeviceReads(pr, DEV)
    rng = np.random.default_rng(71)
    canon = _z(2 ** 30)
    dev_count(dr, canon)
    keys = torch.nonzero(canon).flatten()
    fulls, compacts, hosts = [], [], {}
    for t in range(2):
        canon.zero_()
        canon[keys] = torch.from_numpy(plant(keys, rng, value_pool(rng)).view(np.int32)).to(DEV)
        full = canon.clone()
        dev_mirror(full)
        fulls.append(full)
        compacts.append(dev_table_compact(full))
        hosts[t] = _u32(full)
    del canon
    hosts[None] = hosts[1]
    top = [2 ** 32 - 1]
    quant = sorted(set(np.quantile(hosts[0][keys.cpu().numpy()].astype(np.float64), np.linspace(0, 1, 34)[1:-1]).astype(np.int64).tolist()) - {0, 1})
    layouts = [
        [CovBlock(0, edges=GEOMETRIC), CovBlock(None, 32, 10), CovBlock(1, edges=quant), CovBlock(0, 2 ** 31, 3)],
        [CovBlock(1, edges=top), CovBlock(0, edges=quant), CovBlock(1, 1, _lib.MAX_BINS - 2 - (len(quant) + 1))],
        [CovBlock(None, edges=GEOMETRIC), CovBlock(0, 7, 300)],
    ]
    wkeys = [oracle.window_keys(s) for s in seqs]
    ws = PartitionWorkspace(dr, sub_capacity=0)
    for layout in layouts:
        W = sum(b.bins if b.edges is None else len(b.edges) + 1 for b in layout)
        hist, sums = _z(pr.n_reads, W), _z(pr.n_reads)
        for lo in range(0, 2 ** 30, 2 ** 28):    # four partitions of 16 buckets each
            ws.build(True, key_lo=lo, key_hi=lo + 2 ** 28, log2_bucket_keys=24, count=False)
            ws.check()
            ws.search_layout(fulls[1], compacts, layout, hist, sums)
        want_hist, want_sums = _oracle_rows(wkeys, hosts, layout)
        assert np.array_equal(_u32(sums), want_sums)
        assert np.array_equal(_u32(hist), want_hist), [tuple(b.table for b in layout)]
    # the compact spectrum is the full one
    for t in range(2):
        assert torch.equal(dev_compact_spectrum(compacts[t], 65536), dev_table_spectrum(fulls[t], 65536))
    del fulls, compacts, ws, dr
    torch.cuda.empty_cache()


# ---- 3. in memory: every flag and part beside a layout -------------------------------------------------------------

@pytest.mark.parametrize("batch_bases", [None, 20000])
def test_context_layout_with_every_flag(batch_bases):
    seqs, pr = _synthetic(17)
    other = _synthetic(5)[1]
    layout = [CovBlock(0, edges=GEOMETRIC), CovBlock(None, 32, 10), CovBlock(0, 8, 5), CovBlock(None, edges=[2, 9, 40])]
    slots_only = [CovBlock(0, edges=GEOMETRIC), CovBlock(0, 8, 5)]
    with _env(**({"LRB_BATCH_BASES": batch_bases} if batch_bases else {})):
        c = Context(0)
        c.profile(other, keep_table=True)
        c.sample_table_keep(0)
        ref = c.profile(pr, k=5, want_table=True)                       # composition and table alone
        singles = [c.profile(pr, layout=[b], use_loaded_table=True)["hist"] for b in layout]
        want = np.concatenate(singles, axis=1)
        # a layout with a block on the context's table counts the table from the reads
        c.profile(other, keep_table=True)
        got = c.profile(pr, k=5, layout=layout, want_table=True)
        if batch_bases:
            assert c.info()["n_batches"] > 1
        assert np.array_equal(got["comp"], ref["comp"]) and np.array_equal(got["table"], ref["table"])
        assert np.array_equal(got["hist"], want)
        assert np.array_equal(c.profile(pr, layout=layout, use_loaded_table=True)["hist"], want)
        kept = c.profile(pr, k=5, layout=layout, keep_table=True)
        assert np.array_equal(kept["hist"], want) and np.array_equal(kept["comp"], ref["comp"])
        # the table of two halves added one after the other, with the layout searched in the second call
        n = pr.n_reads
        c.profile(pr.slice(0, n // 2), keep_table=True)
        added = c.profile(pr.slice(n // 2, n), layout=layout, add_to_table=True, want_table=True)
        assert np.array_equal(added["table"], ref["table"]) and np.array_equal(added["hist"], want[n // 2:])
        # a layout of slots alone leaves the context's table as it was, composition and count flags beside it
        c.profile(other, keep_table=True)
        before = c.table_spectrum()
        want_slots = np.concatenate([singles[0], singles[2]], axis=1)
        s = c.profile(pr, k=5, layout=slots_only)
        assert np.array_equal(s["hist"], want_slots) and np.array_equal(s["comp"], ref["comp"])
        assert np.array_equal(c.table_spectrum(), before)
        s = c.profile(pr, layout=slots_only, keep_table=True, want_table=True)
        assert np.array_equal(s["table"], ref["table"]) and np.array_equal(s["hist"], want_slots)
        c.close()


def test_refusals_leave_the_context_usable(three_tables):
    c, seqs, pr, keys, host = three_tables
    layout = [CovBlock(0, edges=GEOMETRIC), CovBlock(None, 32, 10)]
    before = c.profile(pr, layout=layout, use_loaded_table=True)
    for bad in ([CovBlock(6, 32, 10)], [CovBlock(None, 32, 10), CovBlock(None, 32, 10)]):   # empty slot, repeated block
        with pytest.raises(_lib.LrbError) as e:
            c.profile(pr, layout=bad, use_loaded_table=True)
        assert e.value.code == _lib.LRB_EINVAL
    with _env(LRB_TABLE_PATH="direct"):
        with pytest.raises(_lib.LrbError) as e:
            c.profile(pr, layout=layout, use_loaded_table=True)
        assert e.value.code == _lib.LRB_EINVAL and "direct" in str(e.value)
    after = c.profile(pr, layout=layout, use_loaded_table=True)
    assert np.array_equal(after["hist"], before["hist"]) and np.array_equal(after["sums"], before["sums"])


# ---- 4. full size: the column sums of the blocks on the reads' own table are the spectrum's mass ----------------------

def test_full_size_mass():
    torch.cuda.empty_cache()
    cfg = CONFIGS["cfg2_1M_5kb_ont_k4"]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, _ = spec.device_reads(DEV)
    table = _z(2 ** 30)
    dev_count(dr, table)
    compact = dev_table_compact(table)
    s = dev_table_spectrum(table, 65536).cpu().numpy().view(np.uint64)
    assert np.array_equal(dev_compact_spectrum(compact, 65536).cpu().numpy().view(np.uint64), s)
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    valid = np.clip(spec.lengths.astype(np.int64) - 14, 0, None)            # all-ACGT reads
    q = spectrum_quantile_edges(s, 16)
    layout = [CovBlock(None, 32, 10), CovBlock(0, edges=q), CovBlock(None, edges=GEOMETRIC), CovBlock(0, 1, 16)]
    masses = [spectrum_bin_mass(s, 32, 10), spectrum_edge_mass(s, q), spectrum_edge_mass(s, GEOMETRIC), spectrum_bin_mass(s, 1, 16)]
    W = sum(m.size for m in masses)
    hist, sums = _z(spec.n_reads, W), _z(spec.n_reads)
    ws.search_layout(table, [compact], layout, hist, sums)
    col = hist.sum(dim=0, dtype=torch.int64).cpu().numpy().astype(np.uint64)
    assert np.array_equal(col, np.concatenate(masses))
    assert np.array_equal(sums.cpu().numpy().astype(np.int64), valid)
    del hist, sums, table, compact, dr, ws
    torch.cuda.empty_cache()
