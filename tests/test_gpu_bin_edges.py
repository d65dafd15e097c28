"""GPU tier (-m gpu): coverage profiles with bins given by count edges.

Edges {2, 3, 4, 5} are the rule of -bs 1 -bc 5 and no edges that of -bc 1, so the golden files of those settings check
the file-level path byte for byte in every input mode.  Other edge sets are checked against numpy's searchsorted over
the oracle's window keys, on a counted and on a planted table, and at full size the column sums must equal the
spectrum's edge mass."""
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
from lrbinner_b200.profile import (Context, DeviceReads, PackedReads, PartitionWorkspace, dev_count, dev_mirror,  # noqa: E402
                                   dev_table_spectrum, spectrum_edge_mass, spectrum_quantile_edges)
from lrbinner_b200.synth import CONFIGS, SynthSpec  # noqa: E402

DEV = "cuda:0"
GEOMETRIC = [2 ** i for i in range(1, 17)]


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


def _golden(stem, bs, bc):
    with gzip.open(os.path.join(GOLDEN, f"{stem}.cov_bs{bs}_bc{bc}.txt.gz"), "rb") as f:
        return f.read()


def _edges_files_equal_golden(reads, out, stem, table_reads=None):
    """count the table of `table_reads` (default: the reads), then edges {2..5} and no edges; each file and .npy against
    the golden text of -bs 1 -bc 5 and -bs 3 -bc 1"""
    runners_utils.run_15mer_counts(table_reads or reads, out, 4)
    for edges, (bs, bc) in (([2, 3, 4, 5], (1, 5)), ([], (3, 1))):
        runners_utils.run_15mer_vecs_edges(reads, out, edges, 4, write_npy=True)
        path = f"{out}/profiles/cov_profs_edges"
        txt = open(path, "rb").read()
        assert txt == _golden(stem, bs, bc), (stem, edges)
        want = np.array([[float(x) for x in line.split()] for line in txt.decode().splitlines() if line.strip()]).reshape(-1, bc)
        assert np.array_equal(np.load(path + ".npy"), want), (stem, edges)
        assert open(path + ".edges").read() == " ".join(map(str, edges)) + "\n"
    assert not os.path.exists(f"{out}/profiles/cov_profs")
    shutil.rmtree(f"{out}/profiles")     # the 4 GiB table


# ---- 1. file level against the reference's bytes -------------------------------------------------------------

@pytest.mark.parametrize("name", golden_inputs())
def test_edges_write_the_golden_files(name, tmp_path):
    _edges_files_equal_golden(os.path.join(GOLDEN, name), str(tmp_path), name.split(".")[0])


def test_tiny_segments_gzip_and_batches(tmp_path, capfd):
    src = os.path.join(GOLDEN, "g06_community.fa")
    with _env(LRB_SEGMENT_BASES=max(1, PackedReads.from_file(src).total_bases // 5)):
        _edges_files_equal_golden(src, str(tmp_path / "seg"), "g06_community")
    assert "segments" in capfd.readouterr().err
    for name in ("g06_community.fa", "g04_format.fq"):
        stem = name.split(".")[0]
        gz = tmp_path / f"{stem}.gz"
        with gzip.open(gz, "wb") as f:
            f.write(open(os.path.join(GOLDEN, name), "rb").read())
        with _env(LRB_SEGMENT_BASES=max(1, PackedReads.from_file(str(gz)).total_bases // 4)):
            _edges_files_equal_golden(str(gz), str(tmp_path / f"gz_{stem}"), stem)
    with _env(LRB_BATCH_BASES=9000):
        _edges_files_equal_golden(src, str(tmp_path / "batched"), "g06_community")
    assert "batch(es)" in capfd.readouterr().err


def test_contigs_mode(tmp_path):
    reads = os.path.join(GOLDEN, "g06_community.fa")
    frags = os.path.join(GOLDEN, "g10_fragments.fasta")
    _edges_files_equal_golden(frags, str(tmp_path / "whole"), "g10_contigs_mode", table_reads=reads)
    with _env(LRB_SEGMENT_BASES=3000):
        _edges_files_equal_golden(frags, str(tmp_path / "seg"), "g10_contigs_mode", table_reads=reads)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus(tmp_path, capfd):
    with _env(LRB_GPUS=2, LRB_MIN_BLOCKS_PER_DEVICE=1, LRB_VERBOSE=1):
        _edges_files_equal_golden(os.path.join(GOLDEN, "g06_community.fa"), str(tmp_path), "g06_community")
    assert "on 2 GPU(s)" in capfd.readouterr().err
    pr = _synthetic()[1]
    one, two = Context(0), Context([0, 1])
    with _env(LRB_MIN_BLOCKS_PER_DEVICE=1):
        a = one.profile(pr, k=4, edges=GEOMETRIC)
        b = two.profile(pr, k=4, edges=GEOMETRIC)
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
    runners_utils.run_15mer_vecs_edges(src, out, GEOMETRIC, 4)
    assert open(f"{out}/profiles/cov_profs", "rb").read() == before
    assert sorted(os.listdir(f"{out}/profiles")) == ["15mers-counts", "cov_profs", "cov_profs_edges", "cov_profs_edges.edges"]
    shutil.rmtree(f"{out}/profiles")


# ---- 2. against the oracle: searchsorted over the window keys ----------------------------------------------------

def _synthetic():
    spec = SynthSpec(2500, seed=17, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.005)
    seqs = spec.host_sequences() + [b"", b"ACGT", b"N" * 40, b"acgtacgtacgtacgtacgtacgt", b"ACGTTGCA" * 3000]
    return seqs, PackedReads.from_sequences(seqs, threads=4)


def _oracle_rows(seqs, table, edges):
    """hist [n, len(edges) + 1] and sums of the rule: bin = searchsorted(edges, T[key], side="right")"""
    e = np.asarray(edges, dtype=np.uint64)
    hist = np.zeros((len(seqs), len(edges) + 1), dtype=np.uint32)
    sums = np.zeros(len(seqs), dtype=np.uint32)
    for i, s in enumerate(seqs):
        cnt = table[oracle.window_keys(s)].astype(np.uint64)
        hist[i] = np.bincount(np.searchsorted(e, cnt, side="right"), minlength=len(edges) + 1)
        sums[i] = cnt.size
    return hist, sums


def _edge_sets(spectrum, top, rng):
    """geometric, quantile (32 bins), random, 4095 edges, edges above every count, a single edge of 2"""
    many = sorted(set(range(2, 2002)) | set(rng.integers(2002, 2 ** 32, size=4000).tolist()))[:_lib.MAX_BINS - 1]
    return {
        "geometric": GEOMETRIC,
        "quantile": spectrum_quantile_edges(spectrum, 32),
        "random": sorted(set(rng.integers(2, max(top, 3) * 2, size=40).tolist())),
        "4095": many,
        "above": [top + 1, top + 2, 2 ** 32 - 1],
        "two": [2],
    }


def test_counted_table_against_the_oracle():
    seqs, pr = _synthetic()
    table = oracle.Table()
    for s in seqs:
        table.count(s)
    c = Context(0)
    c.profile(pr, keep_table=True)
    spec = c.table_spectrum(65536)
    sets = _edge_sets(spec, int(table.array.max()), np.random.default_rng(3))
    assert len(sets["quantile"]) >= 4 and len(sets["4095"]) == _lib.MAX_BINS - 1
    for name, edges in sets.items():
        got = c.profile(pr, edges=edges, use_loaded_table=True)
        want_hist, want_sums = _oracle_rows(seqs, table.array, edges)
        assert np.array_equal(got["sums"], want_sums), name
        assert np.array_equal(got["hist"], want_hist), name
        if name in ("geometric", "quantile", "4095", "two"):   # the counted table's exact identity
            assert np.array_equal(got["hist"].sum(0, dtype=np.uint64), spectrum_edge_mass(spec, edges)), name
    table.close()
    c.close()


def test_planted_table_against_the_oracle():
    """u32 counts over the whole range (edge_inputs.value_pool) through the device-level search, in key shards"""
    seqs, pr = _synthetic()
    dr = DeviceReads(pr, DEV)
    rng = np.random.default_rng(71)
    canon = _z(2 ** 30)
    dev_count(dr, canon)
    keys = torch.nonzero(canon).flatten()
    canon.zero_()
    canon[keys] = torch.from_numpy(plant(keys, rng, value_pool(rng)).view(np.int32)).to(DEV)
    full = canon.clone()
    dev_mirror(full)
    host = _u32(full)
    sets = _edge_sets(np.zeros(65539, np.uint64), 2 ** 20, rng)
    sets["above"] = [2 ** 32 - 1]
    sets["quantile"] = sorted(set(np.quantile(_u32(canon[keys]).astype(np.float64), np.linspace(0, 1, 34)[1:-1]).astype(np.int64).tolist()) - {0, 1})
    ws = PartitionWorkspace(dr, sub_capacity=0)
    for name, edges in sets.items():
        hist, sums = _z(pr.n_reads, len(edges) + 1), _z(pr.n_reads)
        for lo in range(0, 2 ** 30, 2 ** 28):    # four partitions of 16 buckets each
            ws.build(True, key_lo=lo, key_hi=lo + 2 ** 28, log2_bucket_keys=24, count=False)
            ws.check()
            ws.search_edges(canon, edges, hist, sums)
        want_hist, want_sums = _oracle_rows(seqs, host, edges)
        assert np.array_equal(_u32(sums), want_sums), name
        assert np.array_equal(_u32(hist), want_hist), name
    del canon, full, ws, dr
    torch.cuda.empty_cache()


# ---- 3. in memory: every flag and part beside the edges ----------------------------------------------------------

@pytest.mark.parametrize("batch_bases", [None, 20000])
def test_context_edges_with_every_flag(batch_bases):
    seqs, pr = _synthetic()
    edges = GEOMETRIC
    with _env(**({"LRB_BATCH_BASES": batch_bases} if batch_bases else {})):
        c = Context(0)
        ref = c.profile(pr, k=5, want_table=True)                       # composition and table alone
        got = c.profile(pr, k=5, edges=edges, want_table=True)
        if batch_bases:
            assert c.info()["n_batches"] > 1
        assert np.array_equal(got["comp"], ref["comp"]) and np.array_equal(got["table"], ref["table"])
        spec = c.table_spectrum(65536)
        assert np.array_equal(got["hist"].sum(0, dtype=np.uint64), spectrum_edge_mass(spec, edges))
        assert np.array_equal(got["hist"], _oracle_rows(seqs, ref["table"], edges)[0])
        # use_loaded_table and keep_table give the same rows
        assert np.array_equal(c.profile(pr, edges=edges, use_loaded_table=True)["hist"], got["hist"])
        kept = c.profile(pr, k=5, edges=edges, keep_table=True)
        assert np.array_equal(kept["hist"], got["hist"]) and np.array_equal(kept["comp"], ref["comp"])
        # the table of two halves added one after the other, with the edges searched in the second call
        n = pr.n_reads
        c.profile(pr.slice(0, n // 2), keep_table=True)
        added = c.profile(pr.slice(n // 2, n), edges=edges, add_to_table=True, want_table=True)
        assert np.array_equal(added["table"], ref["table"])
        assert np.array_equal(added["hist"], got["hist"][n // 2:])
        # edges {2..B} equal -bs 1 -bc B, and no edges equal -bc 1
        for B in (2, 5, 33):
            a = c.profile(pr, edges=list(range(2, B + 1)), use_loaded_table=True)
            b = c.profile(pr, bin_size=1, bins=B, use_loaded_table=True)
            assert np.array_equal(a["hist"], b["hist"]) and np.array_equal(a["sums"], b["sums"]), B
        a = c.profile(pr, edges=[], use_loaded_table=True)
        assert np.array_equal(a["hist"], c.profile(pr, bin_size=7, bins=1, use_loaded_table=True)["hist"])
        c.close()


def test_invalid_edges_are_refused_and_the_table_stays_usable():
    seqs, pr = _synthetic()
    c = Context(0)
    c.profile(pr, keep_table=True)
    before = c.profile(pr, edges=GEOMETRIC, use_loaded_table=True)
    edges = np.array([5, 3], np.uint32)
    hist, sums = np.zeros((pr.n_reads, 3), np.uint32), np.zeros(pr.n_reads, np.uint32)
    for flags in (_lib.PROFILE_USE_LOADED_TABLE, 0):
        rc = _lib.lib.lrb_profile_host_edges(c._h, pr._h, 4, edges.ctypes.data, 2, None, hist.ctypes.data, sums.ctypes.data, None, flags)
        assert rc == _lib.LRB_EINVAL and "strictly increasing" in _lib.last_error()
    assert not hist.any() and not sums.any()
    with _env(LRB_TABLE_PATH="direct"):
        with pytest.raises(_lib.LrbError) as e:
            c.profile(pr, edges=GEOMETRIC, use_loaded_table=True)
        assert e.value.code == _lib.LRB_EINVAL and "direct" in str(e.value)
    after = c.profile(pr, edges=GEOMETRIC, use_loaded_table=True)
    assert np.array_equal(after["hist"], before["hist"]) and np.array_equal(after["sums"], before["sums"])
    c.close()


# ---- 4. full size: the column sums are the spectrum's edge mass --------------------------------------------------

@pytest.mark.parametrize("name", ["cfg1_100k_5kb_k3", "cfg2_1M_5kb_ont_k4"])
def test_full_size_edge_mass(name):
    torch.cuda.empty_cache()
    cfg = CONFIGS[name]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, _ = spec.device_reads(DEV)
    table = _z(2 ** 30)
    dev_count(dr, table)
    s = dev_table_spectrum(table, 65536).cpu().numpy().view(np.uint64)
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    valid = np.clip(spec.lengths.astype(np.int64) - 14, 0, None)            # all-ACGT reads
    for edges in (GEOMETRIC, spectrum_quantile_edges(s, 32), list(range(2, 11)),
                  list(range(2, 2002)) + [2002 + 7 * i for i in range(_lib.MAX_BINS - 1 - 2000)]):
        hist, sums = _z(spec.n_reads, len(edges) + 1), _z(spec.n_reads)
        ws.search_edges(table, edges, hist, sums)
        col = hist.sum(dim=0, dtype=torch.int64).cpu().numpy().astype(np.uint64)
        assert np.array_equal(col, spectrum_edge_mass(s, edges)), (name, len(edges))
        assert np.array_equal(sums.cpu().numpy().astype(np.int64), valid)
        if edges == list(range(2, 11)):   # the rule of -bs 1 -bc 10, row for row
            h1, s1 = _z(spec.n_reads, 10), _z(spec.n_reads)
            ws.apply(table, count=False, search=True, bin_size=1, bins=10, hist=h1, sums=s1)
            assert torch.equal(hist, h1) and torch.equal(sums, s1)
        del hist, sums
    del table, dr, ws
    torch.cuda.empty_cache()
