"""GPU tier (-m gpu): coverage profiles for several (-bs, -bc) settings in one search.

One call with the six golden settings must leave, for every setting, the bytes the reference's search-15mers writes for
it (file level, in every input mode); in memory, the column block of setting m must equal a single-setting search with
it, and at full size the column sums must equal the spectrum's bin mass for every setting."""
import gzip
import os
import random
import shutil

import numpy as np
import pytest

from conftest import COV_PARAMS, GOLDEN, golden_inputs

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

from lrbinner_b200 import _lib, runners_utils  # noqa: E402
from lrbinner_b200.profile import (Context, PackedReads, PartitionWorkspace, dev_count, dev_table_spectrum,  # noqa: E402
                                   spectrum_bin_mass)
from lrbinner_b200.synth import CONFIGS, SynthSpec  # noqa: E402

DEV = "cuda:0"
EIGHT = COV_PARAMS + [(5, 20), (64, 16)]


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


def _golden(stem, bs, bc):
    with gzip.open(os.path.join(GOLDEN, f"{stem}.cov_bs{bs}_bc{bc}.txt.gz"), "rb") as f:
        return f.read()


def _shuffled(seed):
    s = list(COV_PARAMS)
    random.Random(seed).shuffle(s)
    return s


def _settings_files_equal_golden(reads, out, stem, seed, table_reads=None):
    """count the table of `table_reads` (default: the reads), then one settings call over `reads`; every file and .npy
    against the golden coverage text of its setting.  Returns the settings in the order they were passed."""
    runners_utils.run_15mer_counts(table_reads or reads, out, 4)
    settings = _shuffled(seed)
    runners_utils.run_15mer_vecs_settings(reads, out, settings, 4, write_npy=True)
    for bs, bc in settings:
        path = f"{out}/profiles/cov_profs_bs{bs}_bc{bc}"
        txt = open(path, "rb").read()
        assert txt == _golden(stem, bs, bc), (stem, bs, bc)
        want = np.array([[float(x) for x in line.split()] for line in txt.decode().splitlines() if line.strip()]).reshape(-1, bc)
        assert np.array_equal(np.load(path + ".npy"), want), (stem, bs, bc)
    assert not os.path.exists(f"{out}/profiles/cov_profs")
    return settings


# ---- 1. file level against the reference's bytes -------------------------------------------------------------

@pytest.mark.parametrize("name", golden_inputs())
def test_one_call_writes_the_six_golden_files(name, tmp_path):
    _settings_files_equal_golden(os.path.join(GOLDEN, name), str(tmp_path), name.split(".")[0], seed=len(name))


def test_tiny_segments_gzip_and_batches(tmp_path, capfd):
    src = os.path.join(GOLDEN, "g06_community.fa")
    budget = max(1, PackedReads.from_file(src).total_bases // 5)
    with _env(LRB_SEGMENT_BASES=budget):
        _settings_files_equal_golden(src, str(tmp_path / "seg"), "g06_community", seed=1)
    assert "segments" in capfd.readouterr().err
    for name in ("g06_community.fa", "g04_format.fq"):
        stem = name.split(".")[0]
        gz = tmp_path / f"{stem}.gz"
        with gzip.open(gz, "wb") as f:
            f.write(open(os.path.join(GOLDEN, name), "rb").read())
        with _env(LRB_SEGMENT_BASES=max(1, PackedReads.from_file(str(gz)).total_bases // 4)):
            _settings_files_equal_golden(str(gz), str(tmp_path / f"gz_{stem}"), stem, seed=2)
    with _env(LRB_BATCH_BASES=9000):
        _settings_files_equal_golden(src, str(tmp_path / "batched"), "g06_community", seed=3)
    assert "batch(es)" in capfd.readouterr().err


def test_contigs_mode(tmp_path):
    """the table of the READS, the fragments searched against it (pipelines.py:139-175), whole and in segments"""
    reads = os.path.join(GOLDEN, "g06_community.fa")
    frags = os.path.join(GOLDEN, "g10_fragments.fasta")
    _settings_files_equal_golden(frags, str(tmp_path / "whole"), "g10_contigs_mode", seed=4, table_reads=reads)
    with _env(LRB_SEGMENT_BASES=3000):
        _settings_files_equal_golden(frags, str(tmp_path / "seg"), "g10_contigs_mode", seed=5, table_reads=reads)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus(tmp_path, capfd):
    with _env(LRB_GPUS=2, LRB_MIN_BLOCKS_PER_DEVICE=1, LRB_VERBOSE=1):
        _settings_files_equal_golden(os.path.join(GOLDEN, "g06_community.fa"), str(tmp_path), "g06_community", seed=6)
    assert "on 2 GPU(s)" in capfd.readouterr().err
    spec = SynthSpec(3000, seed=12, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.006)
    pr = spec.host_packed(threads=4)
    one, two = Context(0), Context([0, 1])
    with _env(LRB_MIN_BLOCKS_PER_DEVICE=1):
        a = one.profile(pr, k=4, coverage=EIGHT)
        b = two.profile(pr, k=4, coverage=EIGHT)
        assert two.info()["n_devices"] == 2
    for key in ("comp", "hist", "sums"):
        assert np.array_equal(a[key], b[key]), key
    one.close()
    two.close()


# ---- 2. in memory: each column block == a single-setting search ------------------------------------------------

def _synthetic():
    spec = SynthSpec(2500, seed=17, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.005)
    seqs = spec.host_sequences() + [b"", b"ACGT", b"N" * 40, b"acgtacgtacgtacgtacgtacgt", b"ACGTTGCA" * 3000]
    return PackedReads.from_sequences(seqs, threads=4)


@pytest.mark.parametrize("batch_bases", [None, 20000])
def test_context_settings_equal_separate_searches(batch_bases):
    pr = _synthetic()
    c = Context(0)
    c.profile(pr, keep_table=True)
    with _env(**({"LRB_BATCH_BASES": batch_bases} if batch_bases else {})):
        for settings in (EIGHT, _shuffled(7), [(3, 1), (1, 5)], [(10, 4000), (2, 96)]):
            r = c.profile(pr, coverage=settings, use_loaded_table=True)
            if batch_bases:
                assert c.info()["n_batches"] > 1
            assert r["hist"].shape == (pr.n_reads, sum(b for _, b in settings))
            for (bs, bc), h in zip(settings, r["hists"]):
                one = c.profile(pr, bin_size=bs, bins=bc, use_loaded_table=True)
                assert np.array_equal(h, one["hist"]), (bs, bc)
                assert np.array_equal(r["sums"], one["sums"]), (bs, bc)
    c.close()


def test_count_composition_and_settings_in_one_call():
    pr = _synthetic()
    c = Context(0)
    got = c.profile(pr, k=5, coverage=EIGHT, want_table=True)
    table = got["table"].copy()
    for (bs, bc), h in zip(EIGHT, got["hists"]):
        one = c.profile(pr, k=5, bin_size=bs, bins=bc, want_table=True)
        assert np.array_equal(h, one["hist"]) and np.array_equal(got["sums"], one["sums"]), (bs, bc)
        assert np.array_equal(got["comp"], one["comp"])
        assert np.array_equal(table, one["table"])
    # adding to a table and keeping it, with settings searched in the same call
    n = pr.n_reads
    c.profile(pr.slice(0, n // 2), keep_table=True)
    added = c.profile(pr.slice(n // 2, n), coverage=EIGHT[:3], add_to_table=True, want_table=True)
    assert np.array_equal(added["table"], table)
    c.close()


def test_one_setting_equals_profile_host():
    pr = _synthetic()
    c = Context(0)
    c.profile(pr, keep_table=True)
    for bs, bc in COV_PARAMS:
        a = c.profile(pr, coverage=[(bs, bc)], use_loaded_table=True)
        b = c.profile(pr, bin_size=bs, bins=bc, use_loaded_table=True)
        assert np.array_equal(a["hist"], b["hist"]) and np.array_equal(a["hists"][0], b["hist"]) and np.array_equal(a["sums"], b["sums"])
    c.close()


# ---- 3. full size: every setting's column sums == the spectrum's bin mass ----------------------------------------

@pytest.mark.parametrize("name", ["cfg1_100k_5kb_k3", "cfg2_1M_5kb_ont_k4"])
def test_full_size_bin_mass_of_every_setting(name):
    torch.cuda.empty_cache()
    cfg = CONFIGS[name]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, _ = spec.device_reads(DEV)
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, table)
    s = dev_table_spectrum(table, 65536).cpu().numpy().view(np.uint64)
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    W = sum(b for _, b in EIGHT)
    hist = torch.zeros((spec.n_reads, W), dtype=torch.int32, device=DEV)
    sums = torch.zeros(spec.n_reads, dtype=torch.int32, device=DEV)
    ws.search_settings(table, EIGHT, hist, sums)
    col = hist.to(torch.int64).sum(dim=0).cpu().numpy().astype(np.uint64)
    off = 0
    for bs, bc in EIGHT:
        assert np.array_equal(spectrum_bin_mass(s, bs, bc), col[off:off + bc]), (name, bs, bc)
        off += bc
    valid = np.clip(spec.lengths.astype(np.int64) - 14, 0, None)            # all-ACGT reads
    assert np.array_equal(sums.cpu().numpy().astype(np.int64), valid)
    # the last setting alone, through the single-setting search, gives the same block row for row
    h1 = torch.zeros((spec.n_reads, EIGHT[-1][1]), dtype=torch.int32, device=DEV)
    s1 = torch.zeros_like(sums)
    ws.apply(table, count=False, search=True, bin_size=EIGHT[-1][0], bins=EIGHT[-1][1], hist=h1, sums=s1)
    assert torch.equal(hist[:, W - EIGHT[-1][1]:], h1) and torch.equal(sums, s1)
    del table, dr, ws, hist, sums, h1, s1
    torch.cuda.empty_cache()


# ---- 4. refused inputs --------------------------------------------------------------------------------------------

BAD = [[], [(10, 8)] * 9, [(0, 5)], [(10, 8), (3, 0)], [(10, 4097)], [(10, 8), (2, 3), (10, 8)], [(1, 4000), (2, 97)]]


def test_invalid_settings_are_refused_and_the_table_stays_usable():
    pr = _synthetic()
    c = Context(0)
    c.profile(pr, keep_table=True)
    before = c.profile(pr, coverage=EIGHT, use_loaded_table=True)
    for bad in BAD:
        for kw in ({"use_loaded_table": True}, {"k": 4}, {"k": 4, "want_table": True}):
            with pytest.raises(_lib.LrbError) as e:
                c.profile(pr, coverage=bad, **kw)
            assert e.value.code == _lib.LRB_EINVAL, (bad, kw)
        after = c.profile(pr, coverage=EIGHT, use_loaded_table=True)
        assert np.array_equal(after["hist"], before["hist"]) and np.array_equal(after["sums"], before["sums"]), bad
    with _env(LRB_TABLE_PATH="direct"):
        with pytest.raises(_lib.LrbError) as e:
            c.profile(pr, coverage=EIGHT[:2], use_loaded_table=True)
        assert e.value.code == _lib.LRB_EINVAL and "direct" in str(e.value)
        one = c.profile(pr, coverage=EIGHT[:1], use_loaded_table=True)     # one setting still runs there
    assert np.array_equal(one["hist"], before["hists"][0])
    assert np.array_equal(c.profile(pr, coverage=EIGHT, use_loaded_table=True)["hist"], before["hist"])
    c.close()
    # device level
    dr, _ = SynthSpec(300, seed=2, scale=0.002).device_reads(DEV)
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, table)
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    hist = torch.zeros((dr.n_reads, 4096), dtype=torch.int32, device=DEV)
    sums = torch.zeros(dr.n_reads, dtype=torch.int32, device=DEV)
    for bad in BAD:
        with pytest.raises(_lib.LrbError) as e:
            ws.search_settings(table, bad, hist, sums)
        assert e.value.code == _lib.LRB_EINVAL, bad
    torch.cuda.synchronize()
    assert not hist.any() and not sums.any()
    del table, ws, dr, hist, sums
    torch.cuda.empty_cache()


def test_runner_leaves_cov_profs_alone(tmp_path):
    src = os.path.join(GOLDEN, "g06_community.fa")
    out = str(tmp_path)
    runners_utils.run_15mer_counts(src, out, 4)
    runners_utils.run_15mer_vecs(src, out, 32, 10, 4)
    before = open(f"{out}/profiles/cov_profs", "rb").read()
    runners_utils.run_15mer_vecs_settings(src, out, [(10, 8), (2, 3)], 4)
    assert open(f"{out}/profiles/cov_profs", "rb").read() == before
    assert sorted(os.listdir(f"{out}/profiles")) == ["15mers-counts", "cov_profs", "cov_profs_bs10_bc8", "cov_profs_bs2_bc3"]
    shutil.rmtree(f"{out}/profiles")
