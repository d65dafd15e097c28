"""GPU tier (-m gpu): coverage against several samples' 15-mer tables in one search (differential coverage).

Block t of every row must equal the single-table search against table t: the reference's bytes for a read set's own
table (golden files), the C oracle's for every other pair, and in memory a single-table Context.profile.  At full size
the own-table block's column sums equal the spectrum's bin mass."""
import gzip
import hashlib
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

from oracle import oracle  # noqa: E402
from lrbinner_b200 import _lib, runners_utils  # noqa: E402
from lrbinner_b200.profile import (Context, PackedReads, PartitionWorkspace, dev_count, dev_mirror,  # noqa: E402
                                   dev_table_compact, dev_table_spectrum, spectrum_bin_mass)
from lrbinner_b200.synth import CONFIGS, SynthSpec  # noqa: E402

DEV = "cuda:0"
G06 = os.path.join(GOLDEN, "g06_community.fa")
G01 = os.path.join(GOLDEN, "g01_identical25.fa")
TABLE_BYTES = 8 + 4 * _lib.TABLE_ENTRIES


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


def _table_file(reads_path, path):
    """The 15mers-counts file of a read file (u64 2^30, then the 2^30 u32 counts), counted on the device and written with
    its all-zero pages left as holes: the same bytes as run_15mer_counts writes, but the tables of these small inputs take
    megabytes of disk instead of 4 GiB each.  Returns the path."""
    c = Context(0)
    t = c.profile(PackedReads.from_file(reads_path), want_table=True)["table"]
    c.close()
    os.makedirs(os.path.dirname(path), exist_ok=True)
    used = np.flatnonzero(t.reshape(-1, 1024).any(axis=1))          # 4 KiB pages holding a count
    cut = np.flatnonzero(np.diff(used) != 1) + 1
    with open(path, "wb") as f:
        f.write(np.uint64(_lib.TABLE_ENTRIES).tobytes())
        f.truncate(TABLE_BYTES)
        for run in np.split(used, cut) if used.size else []:
            f.seek(8 + 4096 * int(run[0]))
            f.write(t[1024 * int(run[0]):1024 * (int(run[-1]) + 1)].tobytes())
    del t
    return path


@pytest.fixture(autouse=True)
def _free_tmp(tmp_path):
    """every test's files go when it ends: the suite's disk use stays what it was without this module"""
    yield
    shutil.rmtree(tmp_path, ignore_errors=True)


@pytest.fixture(scope="module")
def sample_tables(tmp_path_factory):
    """15mers-counts of g06_community and g01_identical25, counted once"""
    d = tmp_path_factory.mktemp("samples")
    out = {}
    for src in (G06, G01):
        stem = os.path.basename(src).split(".")[0]
        out[stem] = _table_file(src, str(d / stem / "15mers-counts"))
    yield out
    shutil.rmtree(d, ignore_errors=True)


def _golden(stem, bs, bc):
    with gzip.open(os.path.join(GOLDEN, f"{stem}.cov_bs{bs}_bc{bc}.txt.gz"), "rb") as f:
        return f.read()


def _blocks(txt, widths):
    """text of n blocks per line -> n texts of one block per line (the writer joins values by one space)"""
    out = [[] for _ in widths]
    for line in txt.decode().splitlines():
        vals = line.split(" ")
        assert len(vals) == sum(widths), (len(vals), widths)
        off = 0
        for t, w in enumerate(widths):
            out[t].append(" ".join(vals[off:off + w]))
            off += w
    return [("\n".join(b) + "\n").encode() if b else b"" for b in out]


def _single(table, reads, bs, bc, tmp):
    """the single-table file: lrb_search_15mers"""
    path = str(tmp / f"single_{abs(hash((table, reads, bs, bc)))}")
    assert _lib.lib.lrb_search_15mers(table.encode(), reads.encode(), path.encode(), bs, bc, 4) == 0, _lib.last_error()
    return open(path, "rb").read()


def _oracle(table, reads, bs, bc, tmp):
    path = str(tmp / f"oracle_{abs(hash((table, reads, bs, bc)))}")
    assert oracle.search_15mers_file(table, reads, path, bs, bc) == 0
    return open(path, "rb").read()


def _check_npy(out, width):
    txt = open(out, "rb").read()
    want = np.array([[float(x) for x in line.split()] for line in txt.decode().splitlines() if line.strip()]).reshape(-1, width)
    assert np.array_equal(np.load(out + ".npy"), want)


def _runner(reads, out, paths, bs, bc, npy=True):
    runners_utils.run_15mer_vecs_samples(reads, out, paths, bs, bc, 4, write_npy=npy)
    f = f"{out}/profiles/cov_profs_samples"
    if npy:
        _check_npy(f, bc * len(paths))
    assert not os.path.exists(f"{out}/profiles/cov_profs")
    return open(f, "rb").read()


# ---- 1. file level against the reference's bytes and the oracle -------------------------------------------------

def _three_tables(reads, own, stem, sample_tables, tmp, seed):
    paths = [("own", own), ("g06", sample_tables["g06_community"]), ("g01", sample_tables["g01_identical25"])]
    random.Random(seed).shuffle(paths)
    bs, bc = COV_PARAMS[seed % len(COV_PARAMS)]
    txt = _runner(reads, str(tmp / "run"), [p for _, p in paths], bs, bc)
    for (who, path), block in zip(paths, _blocks(txt, [bc] * 3)):
        want = _golden(stem, bs, bc) if who == "own" else _oracle(path, reads, bs, bc, tmp)
        assert block == want, (stem, who, bs, bc)
    return txt


@pytest.mark.parametrize("name", golden_inputs())
def test_every_golden_input_against_three_tables(name, tmp_path, sample_tables):
    src = os.path.join(GOLDEN, name)
    own = _table_file(src, str(tmp_path / "own" / "15mers-counts"))
    _three_tables(src, own, name.split(".")[0], sample_tables, tmp_path, len(name))


def test_contigs_mode(tmp_path, sample_tables):
    """fragments against the table counted on the reads (g10 goldens), beside the other samples (the reads' table a
    second time under another path)"""
    frags = os.path.join(GOLDEN, "g10_fragments.fasta")
    own = _table_file(G06, str(tmp_path / "own" / "15mers-counts"))
    _three_tables(frags, own, "g10_contigs_mode", sample_tables, tmp_path, 4)


def test_a_setting_per_table(tmp_path, sample_tables):
    """different (S, B) per table, the same table twice with two settings, through the C entry point"""
    t06, t01 = sample_tables["g06_community"], sample_tables["g01_identical25"]
    tables = [(t06, 10, 8), (t01, 32, 10), (t06, 2, 3), (t01, 1, 5), (t06, 10, 32)]
    out = str(tmp_path / "cov")
    n = len(tables)
    import ctypes as C
    paths = (C.c_char_p * n)(*[p.encode() for p, _, _ in tables])
    bs = (C.c_long * n)(*[s for _, s, _ in tables])
    bc = (C.c_int * n)(*[b for _, _, b in tables])
    assert _lib.lib.lrb_search_15mers_samples(paths, n, bs, bc, G06.encode(), out.encode(), (out + ".npy").encode(), 4) == 0, _lib.last_error()
    txt = open(out, "rb").read()
    _check_npy(out, sum(b for _, _, b in tables))
    for (path, s, b), block in zip(tables, _blocks(txt, [b for _, _, b in tables])):
        want = _golden("g06_community", s, b) if path == t06 else _oracle(path, G06, s, b, tmp_path)
        assert block == want, (path, s, b)


# ---- 2. the same bytes in every input mode --------------------------------------------------------------------------

def test_segments_gzip_batches_and_eight_slots(tmp_path, sample_tables, capfd):
    paths = [sample_tables["g01_identical25"], sample_tables["g06_community"]]
    plain = _runner(G06, str(tmp_path / "plain"), paths, 32, 10)
    budget = max(1, PackedReads.from_file(G06).total_bases // 5)
    with _env(LRB_SEGMENT_BASES=budget):
        assert _runner(G06, str(tmp_path / "seg"), paths, 32, 10) == plain
    assert "segments" in capfd.readouterr().err
    gz = tmp_path / "g06.fa.gz"
    with gzip.open(gz, "wb") as f:
        f.write(open(G06, "rb").read())
    assert _runner(str(gz), str(tmp_path / "gz"), paths, 32, 10) == plain
    with _env(LRB_SEGMENT_BASES=max(1, budget // 2)):
        assert _runner(str(gz), str(tmp_path / "gzseg"), paths, 32, 10) == plain
    with _env(LRB_BATCH_BASES=9000):
        assert _runner(G06, str(tmp_path / "batched"), paths, 32, 10) == plain
    assert "batch(es)" in capfd.readouterr().err
    # eight slots, W = 4090: every block equals the single-table file
    import ctypes as C
    t06, t01 = sample_tables["g06_community"], sample_tables["g01_identical25"]
    tables = [(t06, 1, 4000), (t01, 1, 60), (t06, 2, 10), (t01, 3, 8), (t06, 10, 4), (t01, 32, 4), (t06, 5, 2), (t01, 7, 2)]
    n = len(tables)
    out = str(tmp_path / "eight")
    ok = _lib.lib.lrb_search_15mers_samples((C.c_char_p * n)(*[p.encode() for p, _, _ in tables]), n,
                                            (C.c_long * n)(*[s for _, s, _ in tables]), (C.c_int * n)(*[b for _, _, b in tables]),
                                            G04.encode(), out.encode(), None, 4)
    assert ok == 0, _lib.last_error()
    for (p, s, b), block in zip(tables, _blocks(open(out, "rb").read(), [b for _, _, b in tables])):
        assert block == _single(p, G04, s, b, tmp_path), (p, s, b)


G04 = os.path.join(GOLDEN, "g04_format.fq")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus(tmp_path, sample_tables, capfd):
    paths = [sample_tables["g01_identical25"], sample_tables["g06_community"]]
    plain = _runner(G06, str(tmp_path / "one"), paths, 10, 8)
    with _env(LRB_GPUS=2, LRB_MIN_BLOCKS_PER_DEVICE=1, LRB_VERBOSE=1):
        assert _runner(G06, str(tmp_path / "two"), paths, 10, 8) == plain
    assert "on 2 GPU(s)" in capfd.readouterr().err


# ---- 3. in memory: each column block == a single-table Context.profile --------------------------------------------

def _synthetic(seed):
    spec = SynthSpec(2500, seed=seed, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.005)
    seqs = spec.host_sequences() + [b"", b"ACGT", b"N" * 40, b"acgtacgtacgtacgtacgtacgt", b"ACGTTGCA" * 3000]
    return PackedReads.from_sequences(seqs, threads=4)


def _reference(table_source, pr, bs, bc):
    """single-table search of pr against a table given as a read set (counted) or a file (loaded)"""
    c = Context(0)
    if isinstance(table_source, str):
        c.table_load(table_source)
    else:
        c.profile(table_source, keep_table=True)
    r = c.profile(pr, bin_size=bs, bins=bc, use_loaded_table=True)
    c.close()
    return r


@pytest.mark.parametrize("batch_bases", [None, 20000])
def test_context_samples_equal_single_table_searches(sample_tables, batch_bases, capfd):
    pr, other = _synthetic(17), _synthetic(18)
    c = Context(0)
    c.profile(other, keep_table=True)
    c.sample_table_keep(0)                          # a table counted in the context, no file round trip
    c.profile(pr, keep_table=True)
    c.sample_table_keep(1)
    c.sample_table_load(2, sample_tables["g06_community"])
    sources = {0: other, 1: pr, 2: sample_tables["g06_community"]}
    samples = [(2, 10, 8), (0, 32, 10), (1, 1, 5), (0, 2, 3)]   # slot 0 twice, with two settings
    env = {"LRB_BATCH_BASES": batch_bases} if batch_bases else {}
    with _env(**env):
        got = c.profile(pr, k=4, samples=samples)
    if batch_bases:
        assert c.info()["n_batches"] > 1 and "batch(es)" in capfd.readouterr().err
    assert got["hist"].shape == (pr.n_reads, sum(b for _, _, b in samples))
    plain = c.profile(pr, k=4)
    assert np.array_equal(got["comp"], plain["comp"])
    for (slot, bs, bc), h in zip(samples, got["hists"]):
        ref = _reference(sources[slot], pr, bs, bc)
        assert np.array_equal(h, ref["hist"]), (slot, bs, bc)
        assert np.array_equal(got["sums"], ref["sums"])
    c.close()


def test_samples_beside_count_keep_and_add(sample_tables):
    pr, other = _synthetic(21), _synthetic(22)
    samples = [(3, 10, 8), (5, 32, 10)]
    c = Context(0)
    c.profile(other, keep_table=True)
    c.sample_table_keep(3)
    c.sample_table_load(5, sample_tables["g01_identical25"])
    full = c.profile(pr, want_table=True)["table"].copy()     # the table of pr, for comparison
    # count (keep_table) and composition in the same call as the sample search
    got = c.profile(pr, k=5, samples=samples, keep_table=True, want_table=True)
    assert np.array_equal(got["table"], full)
    assert np.array_equal(got["comp"], c.profile(pr, k=5)["comp"])
    refs = [_reference(other, pr, 10, 8), _reference(sample_tables["g01_identical25"], pr, 32, 10)]
    for h, ref in zip(got["hists"], refs):
        assert np.array_equal(h, ref["hist"]) and np.array_equal(got["sums"], ref["sums"])
    # adding the second half to the first half's table, the sample search of the second half in the same call
    n = pr.n_reads
    c.profile(pr.slice(0, n // 2), keep_table=True)
    half = pr.slice(n // 2, n)
    added = c.profile(half, samples=samples, add_to_table=True, want_table=True)
    assert np.array_equal(added["table"], full)
    for h, ref in zip(added["hists"], refs):
        assert np.array_equal(h, ref["hist"][n // 2:]) and np.array_equal(added["sums"], ref["sums"][n // 2:])
    # a search of the slots alone leaves the context's own table as it was
    c.profile(pr, samples=samples)
    assert np.array_equal(c.profile(pr, want_table=True, use_loaded_table=True)["table"], full)
    c.close()


# ---- 4. full size -----------------------------------------------------------------------------------------------

def test_full_size_config1_against_itself_and_a_second_community():
    torch.cuda.empty_cache()
    cfg = CONFIGS["cfg1_100k_5kb_k3"]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    other = SynthSpec(cfg["n_reads"] // 2, lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"] + 1000)
    dr, _ = spec.device_reads(DEV)
    dr2, _ = other.device_reads(DEV)
    own = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    foreign = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, own)
    dev_count(dr2, foreign)
    dev_mirror(own)
    dev_mirror(foreign)
    del dr2
    compact = [dev_table_compact(own), dev_table_compact(foreign)]
    spec_own = dev_table_spectrum(own, 65536).cpu().numpy().view(np.uint64)
    ws = PartitionWorkspace(dr, sub_capacity=0)
    ws.build(with_rids=True, count=False)
    bs, bc = 10, 32
    hist = torch.zeros((spec.n_reads, 2 * bc), dtype=torch.int32, device=DEV)
    sums = torch.zeros(spec.n_reads, dtype=torch.int32, device=DEV)
    ws.search_samples(compact, [(bs, bc), (bs, bc)], hist, sums)
    col = hist[:, :bc].to(torch.int64).sum(dim=0).cpu().numpy().astype(np.uint64)
    assert np.array_equal(spectrum_bin_mass(spec_own, bs, bc), col)
    h1 = torch.zeros((spec.n_reads, bc), dtype=torch.int32, device=DEV)
    s1 = torch.zeros_like(sums)
    ws.apply(foreign, count=False, search=True, bin_size=bs, bins=bc, hist=h1, sums=s1)

    def digest(t):
        return hashlib.sha256(t.contiguous().cpu().numpy().tobytes()).hexdigest()
    assert digest(hist[:, bc:]) == digest(h1) and torch.equal(sums, s1)
    del own, foreign, compact, dr, ws, hist, sums, h1, s1
    torch.cuda.empty_cache()


# ---- 5. refusals ------------------------------------------------------------------------------------------------

def test_refusals_leave_the_table_and_slots_usable(sample_tables, tmp_path):
    pr = _synthetic(31)
    c = Context(0)
    c.profile(pr, keep_table=True)
    c.sample_table_load(0, sample_tables["g06_community"])
    c.sample_table_keep(1)
    samples = [(0, 10, 8), (1, 32, 10)]
    before = c.profile(pr, samples=samples)
    own = c.profile(pr, bin_size=10, bins=8, use_loaded_table=True)

    def refused(code, f, *a, **kw):
        with pytest.raises(_lib.LrbError) as e:
            f(*a, **kw)
        assert e.value.code == code, (code, str(e.value))
    refused(_lib.LRB_EINVAL, c.profile, pr, samples=[(0, 10, 8), (4, 10, 8)])              # empty slot
    refused(_lib.LRB_EINVAL, c.profile, pr, samples=[(0, 10, 8), (0, 10, 8)])              # repeated
    refused(_lib.LRB_EINVAL, c.profile, pr, samples=[(0, 0, 8)])
    refused(_lib.LRB_EINVAL, c.profile, pr, samples=[(0, 10, 4097)])
    refused(_lib.LRB_EINVAL, c.profile, pr, k=4, samples=[(0, 1, 4000), (1, 1, 97)])
    refused(_lib.LRB_EIO, c.sample_table_load, 0, str(tmp_path / "missing"))
    for cut in (1, 4096):                                                                   # sparse truncated copies
        bad = tmp_path / f"cut{cut}"
        with open(bad, "wb") as f:
            f.write(np.uint64(_lib.TABLE_ENTRIES).tobytes())
            f.truncate(TABLE_BYTES - cut)
        refused(_lib.LRB_EFORMAT, c.sample_table_load, 0, str(bad))
        refused(_lib.LRB_EFORMAT, c.sample_table_load, 6, str(bad))
    with _env(LRB_TABLE_PATH="direct"):
        refused(_lib.LRB_EINVAL, c.profile, pr, samples=samples)
    c.sample_table_free(1)
    refused(_lib.LRB_EINVAL, c.profile, pr, samples=samples)
    c.sample_table_keep(1)
    after = c.profile(pr, samples=samples)
    assert np.array_equal(after["hist"], before["hist"]) and np.array_equal(after["sums"], before["sums"])
    again = c.profile(pr, bin_size=10, bins=8, use_loaded_table=True)
    assert np.array_equal(again["hist"], own["hist"])
    c.close()
    # a context without a table cannot keep one
    e = Context(0)
    refused(_lib.LRB_EINVAL, e.sample_table_keep, 0)
    e.close()
    # file level: a missing table file, after the arguments passed
    out = str(tmp_path / "cov")
    with pytest.raises(SystemExit) as ex:
        runners_utils.run_15mer_vecs_samples(G06, str(tmp_path), [sample_tables["g06_community"], str(tmp_path / "missing")], 10, 8, 4)
    assert ex.value.code == _lib.LRB_EIO
    assert not os.path.exists(out)
    # and a following file-level search gives the golden bytes
    txt = _runner(G06, str(tmp_path / "after"), [sample_tables["g06_community"]], 10, 8)
    assert txt == _golden("g06_community", 10, 8)
