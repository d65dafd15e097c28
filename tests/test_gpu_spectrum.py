"""GPU tier (-m gpu): the 15-mer abundance spectrum (lrb_dev_table_spectrum and the calls above it).

The spectrum is checked against numpy on tables built without the count kernels, on planted values that reach every
path of the kernel (shared-memory bins, global tail, overflow, u64 sums, key-range edges), and through the identity that
ties it to the search: for a table counted from read set R and a search of R with (S, B),
    sum over reads of hist[r][b] == sum_c c * n_c * [bin(c) == b]   for every bin b.
"""
import os

import numpy as np
import pytest

from conftest import COV_PARAMS, GOLDEN

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

from lrbinner_b200 import _lib, runners_utils  # noqa: E402
from lrbinner_b200.profile import (Context, PackedReads, dev_count, dev_mirror, dev_search, dev_table_spectrum,  # noqa: E402
                                   spectrum_bin_mass)
from lrbinner_b200.synth import CONFIGS, SynthSpec  # noqa: E402

DEV = "cuda:0"
HALF = 2 ** 29
GOLDEN_TABLES = sorted(f for f in os.listdir(GOLDEN) if f.endswith(".table.npz"))


def _halves(table):
    """(canonical, bit-15-set) views of a 2^30-entry table: rows of 2^15 entries at a pitch of 2^16."""
    v = table.view(2 ** 14, 2, 2 ** 15)
    return v[:, 0, :], v[:, 1, :]


def _u64(t):
    return t.cpu().numpy().view(np.uint64)


def _spectrum_np(canon_counts, M, n_keys=HALF):
    """Spectrum of a key set given the u32 counts of its nonzero keys (zeros implied up to n_keys)."""
    c = np.asarray(canon_counts, dtype=np.uint64)
    spec = np.zeros(M + 3, dtype=np.uint64)
    low = c[c < M]
    spec[:M] = np.bincount(low.astype(np.int64), minlength=M).astype(np.uint64)
    spec[0] += n_keys - len(c)
    over = c[c >= M]
    spec[M], spec[M + 1] = len(over), int(over.sum(dtype=np.uint64))
    spec[M + 2] = int(c.max()) if len(c) else 0
    return spec


def _windows_mass(spec):
    M = len(spec) - 3
    return sum(int(c) * int(spec[c]) for c in np.flatnonzero(spec[:M])) + int(spec[M + 1])


def _env(**kw):
    import contextlib

    @contextlib.contextmanager
    def cm():
        old = {k: os.environ.get(k) for k in kw}
        os.environ.update({k: str(v) for k, v in kw.items()})
        try:
            yield
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    return cm()


# ---- 1. golden tables, scattered into the device without the count kernels ------------------------------------

def test_golden_tables_equal_numpy():
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    for name in GOLDEN_TABLES:
        g = np.load(os.path.join(GOLDEN, name))
        keys, counts = g["keys"].astype(np.int64), g["counts"]
        table.zero_()
        table[torch.from_numpy(keys).to(DEV)] = torch.from_numpy(counts.view(np.int32)).to(DEV)
        M = 65536
        got = _u64(dev_table_spectrum(table, M))
        canon = (keys & 0x8000) == 0
        assert np.array_equal(got, _spectrum_np(counts[canon], M)), name
        # T[x] == T[rc x] and exactly one of each pair has bit 15 clear: the full table holds every count twice
        full = np.bincount(counts.astype(np.int64))
        assert got[0] * 2 == 2 ** 30 - len(keys), name
        assert np.array_equal(got[1:len(full)] * 2, full[1:].astype(np.uint64)), name
    del table
    torch.cuda.empty_cache()


def test_golden_community_through_the_context():
    g = np.load(os.path.join(GOLDEN, "g06_community.table.npz"))
    keys, counts = g["keys"].astype(np.int64), g["counts"]
    c = Context(0)
    c.profile(PackedReads.from_file(os.path.join(GOLDEN, "g06_community.fa"), threads=2), keep_table=True)
    for M in (2, 7, 65536):
        assert np.array_equal(c.table_spectrum(M), _spectrum_np(counts[(keys & 0x8000) == 0], M)), M
    c.close()


# ---- 2. planted values: shared-memory bins, global tail, overflow, u64 sum, max; the other half ignored --------

@pytest.mark.parametrize("M", [65536, 2 ** 24])
def test_planted_values(M):
    rng = np.random.default_rng(M)
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    canon, other = _halves(table)
    garbage = 77777                                             # >= 65536 and absent from the planted set
    other.fill_(garbage)
    planted = {2: 3, M - 1: 2, M: 2, M + 1: 1, 2 ** 32 - 1: 2, 9000: 5, 40000: 1}
    vals = [v for v, n in planted.items() for _ in range(n)] + [1] * 3000
    pos = rng.choice(HALF, size=len(vals), replace=False)
    flat = torch.from_numpy(pos).to(DEV)
    row, col = flat // 2 ** 15, flat % 2 ** 15
    canon[row, col] = torch.from_numpy(np.array(vals, dtype=np.uint32).view(np.int32)).to(DEV)
    got = _u64(dev_table_spectrum(table, M))
    want = _spectrum_np(vals, M)
    assert np.array_equal(got, want)
    over = [v for v in vals if v >= M]
    assert int(got[M]) == len(over) and int(got[M + 1]) == sum(over) > 2 ** 32 and int(got[M + 2]) == 2 ** 32 - 1
    if M > garbage:
        assert got[garbage] == 0
    # all zeros, then every canonical entry 1 (one hot bin: the contention path)
    table.zero_()
    got = _u64(dev_table_spectrum(table, M))
    assert got[0] == HALF and got.sum() == HALF
    canon.fill_(1)
    got = _u64(dev_table_spectrum(table, M))
    assert got[1] == HALF and got[0] == 0 and got[M + 2] == 1 and got.sum() == HALF + 1
    del table, canon, other
    torch.cuda.empty_cache()


# ---- 3. key shards: disjoint ranges accumulated into one buffer == the whole range -----------------------------

def test_key_shards_sum_to_the_whole_range():
    M = 65536
    g = torch.Generator(device=DEV).manual_seed(5)
    table = torch.randint(0, 64, (2 ** 30,), dtype=torch.int32, device=DEV, generator=g)
    table[::1000003] = 70000                                    # a sprinkle of overflow keys
    table[12346] = -1                                           # 2^32 - 1 inside a two-key range
    whole = dev_table_spectrum(table, M)
    canon = _halves(table)[0].reshape(-1).to(torch.int64) & 0xFFFFFFFF
    ref = _spectrum_np([], M, n_keys=0)
    ref[:M] = torch.bincount(canon.clamp(max=M), minlength=M + 1)[:M].cpu().numpy().astype(np.uint64)
    over = canon[canon >= M]
    ref[M], ref[M + 1], ref[M + 2] = over.numel(), int(over.sum().item()), int(canon.max().item())
    del canon, over
    assert np.array_equal(_u64(whole), ref)
    bounds = [0, 12345, 12347, 2 ** 29 + 7, 2 ** 29 + 7 + 3 * 2 ** 16 + 40000, 2 ** 30]  # unaligned, bit-15-set edge too
    acc = torch.zeros(M + 3, dtype=torch.int64, device=DEV)
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        dev_table_spectrum(table, M, lo, hi, out=acc)
    assert np.array_equal(_u64(acc), _u64(whole))
    # a range inside one 4-key unit, and an empty one
    small = dev_table_spectrum(table, M, 12345, 12347)
    assert int(_u64(small)[:M + 1].sum()) == 2 and int(_u64(small)[M + 2]) == 2 ** 32 - 1
    assert not _u64(dev_table_spectrum(table, M, 77, 77)).any()
    del table, acc, whole
    torch.cuda.empty_cache()


# ---- 4. the identity: spectrum projected onto bins == column sums of the search -------------------------------

@pytest.mark.parametrize("batch_bases", [None, 9000])
def test_bin_mass_identity_on_synthetic_reads(batch_bases):
    spec = SynthSpec(1500, seed=8, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.004)
    pr = spec.host_packed(threads=4)
    c = Context(0)
    with _env(**({"LRB_BATCH_BASES": batch_bases} if batch_bases else {})):
        c.profile(pr, keep_table=True)
        if batch_bases:
            assert c.info()["n_batches"] > 1
        s = c.table_spectrum()
        for bs, bc in COV_PARAMS:
            r = c.profile(pr, bin_size=bs, bins=bc, use_loaded_table=True)
            assert np.array_equal(spectrum_bin_mass(s, bs, bc), r["hist"].sum(axis=0, dtype=np.uint64)), (bs, bc)
            assert _windows_mass(s) == int(r["sums"].sum(dtype=np.uint64)), (bs, bc)
    c.close()


# ---- 5. full size ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["cfg1_100k_5kb_k3", "cfg2_1M_5kb_ont_k4", "cfg4_500k_15kb_hifi_k5"])
def test_full_size_identity(name):
    torch.cuda.empty_cache()
    cfg = CONFIGS[name]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, _ = spec.device_reads(DEV)
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, table)
    s = _u64(dev_table_spectrum(table, 65536))
    assert _windows_mass(s) == int(np.clip(spec.lengths.astype(np.int64) - 14, 0, None).sum())   # all-ACGT reads
    dev_mirror(table)
    for bs, bc in ((32, 10), (10, 32)):
        hist = torch.zeros((spec.n_reads, bc), dtype=torch.int32, device=DEV)
        sums = torch.zeros(spec.n_reads, dtype=torch.int32, device=DEV)
        dev_search(dr, table, bs, bc, hist, sums)
        col = hist.to(torch.int64).sum(dim=0).cpu().numpy().astype(np.uint64)
        assert np.array_equal(spectrum_bin_mass(s, bs, bc), col), (name, bs, bc)
        del hist, sums
    del table, dr
    torch.cuda.empty_cache()


# ---- 6. context and file level --------------------------------------------------------------------------------

def test_context_spectrum_leaves_the_table_alone(tmp_path):
    pr = PackedReads.from_file(os.path.join(GOLDEN, "g06_community.fa"), threads=2)
    c = Context(0)
    c.profile(pr, keep_table=True)
    before = c.profile(pr, bin_size=10, bins=8, use_loaded_table=True)
    s1 = c.table_spectrum()
    s2 = c.table_spectrum()
    assert np.array_equal(s1, s2)
    after = c.profile(pr, bin_size=10, bins=8, use_loaded_table=True)
    assert np.array_equal(before["hist"], after["hist"]) and np.array_equal(before["sums"], after["sums"])
    c.table_save(str(tmp_path / "t"))                       # still a complete table
    os.remove(tmp_path / "t")
    for bad in (1, _lib.SPECTRUM_MAX_COUNT + 1):
        with pytest.raises(_lib.LrbError) as e:
            c.table_spectrum(bad)
        assert e.value.code == _lib.LRB_EINVAL
    c.close()
    empty = Context(0)
    with pytest.raises(_lib.LrbError) as e:
        empty.table_spectrum()
    assert e.value.code == _lib.LRB_EINVAL and "no table" in str(e.value)
    empty.close()
    table = torch.zeros(2 ** 16, dtype=torch.int32, device=DEV)   # never launched on: the arguments fail first
    for bad in (1, _lib.SPECTRUM_MAX_COUNT + 1):
        with pytest.raises(_lib.LrbError) as e:
            dev_table_spectrum(table, bad, 0, 2 ** 16)
        assert e.value.code == _lib.LRB_EINVAL


def test_runner_writes_the_histo_file(tmp_path):
    src = os.path.join(GOLDEN, "g06_community.fa")
    out = str(tmp_path)
    runners_utils.run_15mer_counts(src, out, 4)
    runners_utils.run_15mer_histo(out, 4)
    g = np.load(os.path.join(GOLDEN, "g06_community.table.npz"))
    counts = g["counts"][(g["keys"] & 0x8000) == 0]
    vals, n = np.unique(counts, return_counts=True)
    want = "".join(f"{v} {k}\n" for v, k in zip(vals, n) if v < 65536)
    if (counts >= 65536).any():
        want += f"65536 {(counts >= 65536).sum()}\n"
    assert open(f"{out}/profiles/15mers-histo").read() == want
    assert _lib.lib.lrb_table_spectrum(f"{out}/profiles/15mers-counts".encode(), f"{out}/h".encode(), 1) == _lib.LRB_EINVAL
    assert _lib.lib.lrb_table_spectrum(f"{out}/profiles/15mers-counts".encode(), f"{out}/h".encode(),
                                       _lib.SPECTRUM_MAX_COUNT + 1) == _lib.LRB_EINVAL
    with open(f"{out}/bad", "wb") as f:
        f.write(b"\x00" * 64)
    assert _lib.lib.lrb_table_spectrum(f"{out}/bad".encode(), f"{out}/h".encode(), 65536) == _lib.LRB_EFORMAT
    os.remove(f"{out}/profiles/15mers-counts")
    with pytest.raises(SystemExit):
        runners_utils.run_15mer_histo(out, 4)                # missing table file -> check_proc -> sys.exit
    assert _lib.lib.lrb_table_spectrum(f"{out}/profiles/15mers-counts".encode(), f"{out}/h".encode(), 65536) == _lib.LRB_EIO


# ---- 7. multi-GPU ---------------------------------------------------------------------------------------------

@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_multi_gpu_context_spectrum_equals_single():
    pr = PackedReads.from_file(os.path.join(GOLDEN, "g06_community.fa"), threads=2)
    one = Context(0)
    one.profile(pr, keep_table=True)
    want = one.table_spectrum()
    one.close()
    two = Context([0, 1])
    two.profile(pr, keep_table=True)
    assert two.info()["n_devices"] == 2
    assert np.array_equal(two.table_spectrum(), want)
    two.close()
