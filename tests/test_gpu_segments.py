"""GPU tier (-m gpu) of segmented input: the file-level drop-ins read a file larger than one segment segment by segment
(count: each segment added to the table; search: each segment against the loaded table; fused: two passes over the file)
and must leave the reference tools' bytes on disk for every segmentation; LRB_PROFILE_ADD_TO_TABLE at context level."""
import gzip
import hashlib
import os

import numpy as np
import pytest

from conftest import COV_PARAMS, GOLDEN, golden_inputs

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

from lrbinner_b200 import _lib, runners_utils  # noqa: E402
from lrbinner_b200.profile import Context, PackedReads, read_segments  # noqa: E402
from lrbinner_b200.synth import CONFIGS, SynthSpec, write_fasta  # noqa: E402


def _gz(path):
    with gzip.open(path, "rb") as f:
        return f.read()


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


def _golden(stem, what):
    return _gz(os.path.join(GOLDEN, f"{stem}.{what}.txt.gz"))


def _table_file_equals_golden(path, stem):
    gold = np.load(os.path.join(GOLDEN, f"{stem}.table.npz"))
    assert os.path.getsize(path) == int(gold["file_bytes"])
    head = np.fromfile(path, dtype=np.uint64, count=1)
    assert head[0] == 2 ** 30
    t = np.memmap(path, dtype=np.uint32, mode="r", offset=8)
    keys = gold["keys"].astype(np.int64)
    assert np.array_equal(np.flatnonzero(t), keys) and np.array_equal(t[keys], gold["counts"])
    del t


def _budget_for(path):
    """a budget that cuts the input into several segments"""
    return max(1, PackedReads.from_file(path).total_bases // 5)


def _n_segments(path, budget):
    return sum(1 for _ in read_segments(path, budget, 2))


def _all_files(src, stem, out, capfd, fused=True):
    """the three drop-ins for every k and every (-bs, -bc), then run_profile; every file against the golden bytes"""
    for k in (3, 4, 5):
        runners_utils.run_kmers(src, out, k, 4)
        assert open(f"{out}/profiles/com_profs", "rb").read() == _golden(stem, f"com_k{k}"), (stem, k)
    runners_utils.run_15mer_counts(src, out, 4)
    _table_file_equals_golden(f"{out}/profiles/15mers-counts", stem)
    for bs, bc in COV_PARAMS:
        runners_utils.run_15mer_vecs(src, out, bs, bc, 4)
        assert open(f"{out}/profiles/cov_profs", "rb").read() == _golden(stem, f"cov_bs{bs}_bc{bc}"), (stem, bs, bc)
    os.remove(f"{out}/profiles/15mers-counts")
    if fused:
        for i, k in enumerate((3, 4, 5)):
            bs, bc = COV_PARAMS[(2 * i) % len(COV_PARAMS)]
            fo = f"{out}/fused{k}"
            runners_utils.run_profile(src, fo, k, bs, bc, 4, write_table=(i == 0), write_npy=True)
            assert open(f"{fo}/profiles/com_profs", "rb").read() == _golden(stem, f"com_k{k}"), (stem, "fused", k)
            cov = open(f"{fo}/profiles/cov_profs", "rb").read()
            assert cov == _golden(stem, f"cov_bs{bs}_bc{bc}"), (stem, "fused", bs, bc)
            want = np.array([[float(x) for x in line.split()] for line in cov.decode().splitlines() if line.strip()]).reshape(-1, bc)
            assert np.array_equal(np.load(f"{fo}/profiles/cov_profs.npy"), want)
            comp = np.load(f"{fo}/profiles/com_profs.npy")
            assert comp.shape[0] == want.shape[0]
            if i == 0:
                _table_file_equals_golden(f"{fo}/profiles/15mers-counts", stem)
                os.remove(f"{fo}/profiles/15mers-counts")
    return capfd.readouterr().err


@pytest.mark.parametrize("name", golden_inputs())
def test_dropins_in_tiny_segments_write_the_golden_bytes(name, tmp_path, capfd):
    stem = name.split(".")[0]
    src = os.path.join(GOLDEN, name)
    budget = _budget_for(src)
    with _env(LRB_SEGMENT_BASES=budget):
        err = _all_files(src, stem, str(tmp_path), capfd)
    if _n_segments(src, budget) > 1:
        assert "segments" in err and "2 passes over the file" in err, err


def test_gzip_input_and_batches_inside_segments(tmp_path, capfd):
    """gzip input in segments, and segments that are themselves processed in device batches (LRB_BATCH_BASES)"""
    for name in ("g06_community.fa", "g04_format.fq"):
        stem = name.split(".")[0]
        gz = tmp_path / f"{stem}.gz"
        with gzip.open(gz, "wb") as f:
            f.write(open(os.path.join(GOLDEN, name), "rb").read())
        budget = _budget_for(str(gz))
        with _env(LRB_SEGMENT_BASES=budget):
            err = _all_files(str(gz), stem, str(tmp_path / f"o_{stem}"), capfd, fused=(stem == "g06_community"))
        assert "segments" in err, err
    src = os.path.join(GOLDEN, "g06_community.fa")
    with _env(LRB_SEGMENT_BASES=40000, LRB_BATCH_BASES=9000):
        out = str(tmp_path / "batched")
        runners_utils.run_profile(src, out, 4, 10, 8, 4, write_table=True)
        assert open(f"{out}/profiles/com_profs", "rb").read() == _golden("g06_community", "com_k4")
        assert open(f"{out}/profiles/cov_profs", "rb").read() == _golden("g06_community", "cov_bs10_bc8")
        _table_file_equals_golden(f"{out}/profiles/15mers-counts", "g06_community")
    err = capfd.readouterr().err
    assert "segments" in err and "batch(es)" in err, err


def test_contigs_mode_in_segments(tmp_path, capfd):
    """contigs mode (pipelines.py:139-175): the table of the READS, fragments profiled against it; both sides segmented"""
    reads = os.path.join(GOLDEN, "g06_community.fa")
    frags = os.path.join(GOLDEN, "g10_fragments.fasta")
    out = str(tmp_path)
    with _env(LRB_SEGMENT_BASES=25000):
        runners_utils.run_15mer_counts(reads, out, 4)
    with _env(LRB_SEGMENT_BASES=3000):
        for k in (3, 4, 5):
            runners_utils.run_kmers(frags, out, k, 4)
            assert open(f"{out}/profiles/com_profs", "rb").read() == _golden("g10_contigs_mode", f"com_k{k}"), k
        for bs, bc in COV_PARAMS:
            runners_utils.run_15mer_vecs(frags, out, bs, bc, 4)
            assert open(f"{out}/profiles/cov_profs", "rb").read() == _golden("g10_contigs_mode", f"cov_bs{bs}_bc{bc}"), (bs, bc)
    os.remove(f"{out}/profiles/15mers-counts")
    assert capfd.readouterr().err.count("segments") >= 1 + 3 + len(COV_PARAMS)


def test_config1_full_size_in_segments_against_stored_digests():
    """BASELINE.json config #1 in full (100 k reads, 0.5 Gbases) in segments of 50 Mbases: fused and three calls leave the
    sizes and sha256 of tests/golden/cfg1_100k_5kb_k3.files.json"""
    import json
    import shutil
    import tempfile
    cfg = CONFIGS["cfg1_100k_5kb_k3"]
    with open(os.path.join(GOLDEN, "cfg1_100k_5kb_k3.files.json")) as f:
        want = json.load(f)["files"]
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 12 * 2 ** 30 else None
    work = tempfile.mkdtemp(prefix="lrb_seg_cfg1_", dir=base)

    def digest(path):
        h = hashlib.sha256()
        with open(path, "rb") as f:
            for blk in iter(lambda: f.read(1 << 24), b""):
                h.update(blk)
        return {"bytes": os.path.getsize(path), "sha256": h.hexdigest()}

    try:
        spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
        fasta = os.path.join(work, "cfg1.fa")
        write_fasta(fasta, spec.host_sequences())
        assert digest(fasta) == want["reads.fa"]
        threads = os.cpu_count() or 8
        with _env(LRB_SEGMENT_BASES=50_000_000):
            assert _n_segments(fasta, 50_000_000) >= 10
            out = os.path.join(work, "fused")
            runners_utils.run_profile(fasta, out, cfg["k"], 32, 10, threads, write_table=True)
            for name in ("com_profs", "cov_profs", "15mers-counts"):
                assert digest(f"{out}/profiles/{name}") == want[name], ("fused", name)
            shutil.rmtree(out)
            out = os.path.join(work, "three")
            runners_utils.run_kmers(fasta, out, cfg["k"], threads)
            runners_utils.run_15mer_counts(fasta, out, threads)
            runners_utils.run_15mer_vecs(fasta, out, 32, 10, threads)
            for name in ("com_profs", "cov_profs", "15mers-counts"):
                assert digest(f"{out}/profiles/{name}") == want[name], ("three calls", name)
    finally:
        shutil.rmtree(work, ignore_errors=True)


def _add_slices(ctx, pr, cuts, **kw):
    ctx.profile(pr.slice(cuts[0], cuts[1]), keep_table=True, **kw)
    for a, b in zip(cuts[1:-2], cuts[2:-1]):
        ctx.profile(pr.slice(a, b), add_to_table=True, **kw)
    return ctx.profile(pr.slice(cuts[-2], cuts[-1]), add_to_table=True, want_table=True, **kw)["table"]


def test_add_to_table_equals_the_table_of_the_whole_set():
    """tables counted from k slices added one after another == the table of the whole set, entry for entry: resident,
    in device batches, on the direct kernels, and with composition / coverage rows requested beside the count"""
    spec = SynthSpec(3000, seed=21, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.006)
    pr = spec.host_packed(threads=4)
    c = Context(0)
    whole = c.profile(pr, want_table=True)["table"].copy()
    n = pr.n_reads
    for cuts, env, kw in (([0, n // 3, n // 2, n - 1, n], {}, {}),
                          ([0, 1, 2, n // 2, n], {}, {"k": 5, "bin_size": 3, "bins": 7}),
                          ([0, n // 4, n], {"LRB_BATCH_BASES": 30000}, {}),
                          ([0, 700, 1400, 2100, n], {"LRB_TABLE_PATH": "direct"}, {"k": 3})):
        with _env(**env):
            got = _add_slices(c, pr, cuts, **kw)
        assert np.array_equal(got, whole), (cuts, env, kw)
    # the spectrum of the added table is that of the whole set
    c.profile(pr, keep_table=True)
    spec_whole = c.table_spectrum(4096)
    _add_slices(c, pr, [0, n // 2, n])
    assert np.array_equal(c.table_spectrum(4096), spec_whole)
    c.close()


def test_failed_add_leaves_no_table():
    pr = SynthSpec(200, seed=4, scale=0.002).host_packed(threads=2)
    c = Context(0)
    with pytest.raises(_lib.LrbError, match="no table"):
        c.profile(pr, add_to_table=True)           # nothing to add to
    c.profile(pr, keep_table=True)
    c.table_spectrum(64)                           # a table is there
    with pytest.raises(_lib.LrbError):
        c.profile(pr, bin_size=2, bins=0, add_to_table=True)
    with pytest.raises(_lib.LrbError, match="no table"):
        c.table_spectrum(64)
    with pytest.raises(_lib.LrbError, match="no table"):
        c.profile(pr, add_to_table=True)
    with pytest.raises(_lib.LrbError, match="exclude"):
        c.profile(pr, bin_size=2, bins=3, use_loaded_table=True, add_to_table=True)
    c.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_in_segments_write_the_golden_bytes(tmp_path, capfd):
    """LRB_GPUS=2: every segment is sharded over two devices; ADD_TO_TABLE adds device 0's share to the complete table and
    counts device 1's share from zero, the exchange sums them"""
    src = os.path.join(GOLDEN, "g06_community.fa")
    with _env(LRB_GPUS=2, LRB_MIN_BLOCKS_PER_DEVICE=1, LRB_SEGMENT_BASES=30000, LRB_VERBOSE=1):
        err = _all_files(src, "g06_community", str(tmp_path), capfd)
    assert "segments" in err and "on 2 GPU(s)" in err, err
    spec = SynthSpec(4000, seed=9, n_rate=1e-3, lowercase_frac=0.01, edge_lengths=True, scale=0.01)
    pr = spec.host_packed(threads=4)
    one, two = Context(0), Context([0, 1])
    whole = one.profile(pr, want_table=True)["table"]
    with _env(LRB_MIN_BLOCKS_PER_DEVICE=1):
        got = _add_slices(two, pr, [0, 1000, 2500, pr.n_reads])
        assert two.info()["n_devices"] == 2
    assert np.array_equal(got, whole)
    one.close()
    two.close()
