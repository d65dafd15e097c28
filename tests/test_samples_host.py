"""CPU tier: the multi-table (sample) coverage search without a device.

- the argument checks of lrb_search_15mers_samples, lrb_profile_host_samples, Context.profile(samples=...) and
  run_15mer_vecs_samples, which all run before any file or device is touched;
- the compact index the search gathers at, over the whole canonical key space, for every bucket size;
- the canonical-row reader of sample slots against np.memmap slicing of a (sparse) 4 GiB table file, and its refusal of
  truncated files."""
import ctypes as C
import os
import types

import numpy as np
import pytest

from conftest import GOLDEN

from lrbinner_b200 import _lib, runners_utils
from lrbinner_b200.profile import Context, PackedReads, read_table_canonical

lib = _lib.lib
READS = os.path.join(GOLDEN, "g06_community.fa")
TABLE_BYTES = 8 + 4 * _lib.TABLE_ENTRIES
ROWS = _lib.TABLE_ENTRIES >> 16

# (tables as (path, bin_size, bins), what the message names); paths are never opened
A, B = "/nonexistent/a/15mers-counts", "/nonexistent/b/15mers-counts"
BAD = [
    ([], "number of sample tables"),
    ([(A, 10, 8)] + [(B, s, 8) for s in range(1, 9)], "number of sample tables"),
    ([(A, 10, 8), (B, 0, 5)], "bin_size"),
    ([(A, 10, 0)], "bins"),
    ([(A, 10, 8), (B, 2, 4097)], "bins"),
    ([(A, 1, 4000), (B, 1, 97)], "add up to 4097"),
    ([(A, 10, 8), (B, 10, 8), (A, 10, 8)], "repeats"),
]


def _file_call(tables, reads=READS, out=b"/nonexistent/out", npy=None):
    n = len(tables)
    paths = (C.c_char_p * max(n, 1))(*[p.encode() if p is not None else None for p, _, _ in tables])
    bs = (C.c_long * max(n, 1))(*[s for _, s, _ in tables])
    bc = (C.c_int * max(n, 1))(*[b for _, _, b in tables])
    return lib.lrb_search_15mers_samples(paths, n, bs, bc, reads.encode() if reads else None, out, npy, 2)


@pytest.mark.parametrize("tables,what", BAD)
def test_file_level_refuses_bad_arguments_before_any_work(tables, what):
    assert _file_call(tables) == _lib.LRB_EINVAL
    msg = _lib.last_error()
    assert "lrb_search_15mers_samples" in msg and what in msg, msg


def test_file_level_refuses_null_paths():
    good = [(A, 10, 8), (B, 10, 8)]
    assert _file_call(good, reads=None) == _lib.LRB_EINVAL
    assert _file_call(good, out=None) == _lib.LRB_EINVAL
    assert _file_call([(A, 10, 8), (None, 10, 8)]) == _lib.LRB_EINVAL
    assert "table 1" in _lib.last_error()
    bs, bc = (C.c_long * 1)(10), (C.c_int * 1)(8)
    assert lib.lrb_search_15mers_samples(None, 1, bs, bc, READS.encode(), b"/nonexistent/out", None, 2) == _lib.LRB_EINVAL


def test_file_level_accepts_a_table_twice_with_different_settings_and_every_limit():
    """past the checks (the call then fails on the missing table file or device, never with LRB_EINVAL)"""
    assert _file_call([(A, 10, 8), (A, 32, 10), (B, 10, 8)]) != _lib.LRB_EINVAL
    eight = [(A, 1, 4089)] + [(B if i % 2 else A, 2 + i, 1) for i in range(7)]
    assert sum(b for _, _, b in eight) == _lib.MAX_BINS and len(eight) == _lib.MAX_SAMPLE_TABLES
    assert _file_call(eight) != _lib.LRB_EINVAL


def test_file_level_refuses_the_direct_table_path(monkeypatch, tmp_path):
    monkeypatch.setenv("LRB_TABLE_PATH", "direct")
    out = tmp_path / "out"
    assert _file_call([(A, 10, 8)], out=str(out).encode()) == _lib.LRB_EINVAL
    assert "LRB_TABLE_PATH=direct" in _lib.last_error()
    assert not out.exists()


def _ctx_call(slots, settings, ctx=None):
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    n = len(slots)
    sl = (C.c_int * max(n, 1))(*slots)
    bs = (C.c_long * max(n, 1))(*[s for s, _ in settings])
    bc = (C.c_int * max(n, 1))(*[b for _, b in settings])
    hist = np.zeros(4096, dtype=np.uint32)
    sums = np.zeros(1, dtype=np.uint32)
    return lib.lrb_profile_host_samples(ctx, reads._h, 0, n, sl, bs, bc, None, hist.ctypes.data, sums.ctypes.data, None, 0)


@pytest.mark.parametrize("slots,settings,what", [
    ([], [], "number of sample tables"),
    (list(range(8)) + [0], [(s, 4) for s in range(1, 10)], "number of sample tables"),
    ([0, 1], [(10, 8), (0, 8)], "bin_size"),
    ([0], [(10, 0)], "bins"),
    ([0, 1], [(10, 8), (10, 4097)], "bins"),
    ([0, 1, 2], [(1, 2000), (1, 2000), (1, 97)], "add up to 4097"),
    ([3, 1, 3], [(10, 8), (10, 8), (10, 8)], "repeats"),
    ([0, 8], [(10, 8), (10, 8)], "slot must be in [0, 8)"),
    ([-1], [(10, 8)], "slot must be in [0, 8)"),
])
def test_context_level_refuses_bad_arguments_before_the_context(slots, settings, what):
    assert _ctx_call(slots, settings) == _lib.LRB_EINVAL
    assert what in _lib.last_error(), _lib.last_error()


def test_context_level_checks_the_context_after_the_arguments():
    assert _ctx_call([0, 0, 1], [(10, 8), (32, 10), (10, 8)]) == _lib.LRB_EINVAL
    assert "null context" in _lib.last_error()


def test_python_level_refusals():
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    no_device = types.SimpleNamespace(_h=None)   # a context that was never created: the library refuses before using it
    for kw in ({"coverage": [(10, 8)]}, {"bin_size": 10}, {"bins": 8}):
        with pytest.raises(_lib.LrbError) as e:
            Context.profile(no_device, reads, samples=[(0, 10, 8)], **kw)
        assert e.value.code == _lib.LRB_EINVAL and "samples=" in str(e.value)
    for samples, what in [([(0, 10, 8), (0, 10, 8)], "repeats"), ([(0, 0, 8)], "bin_size"), ([(9, 10, 8)], "slot"),
                          ([], "number of sample tables"), ([(t % 8, 1, 600) for t in range(7)], "add up to 4200")]:
        with pytest.raises(_lib.LrbError) as e:
            Context.profile(no_device, reads, samples=samples)
        assert e.value.code == _lib.LRB_EINVAL and what in str(e.value), str(e.value)


@pytest.mark.parametrize("paths,setting,what", [
    ([], (10, 8), "number of sample tables"),
    ([A, B] * 4 + [A], (10, 8), "number of sample tables"),
    ([A, B], (0, 8), "bin_size"),
    ([A], (10, 0), "bins"),
    ([A, B], (10, 2049), "add up to 4098"),
    ([A, B, A], (10, 8), "repeats"),
])
def test_runner_exits_before_writing_anything(paths, setting, what, tmp_path):
    """the runner has one (bin_size, bin_count) for every table"""
    with pytest.raises(SystemExit) as e:
        runners_utils.run_15mer_vecs_samples(READS, str(tmp_path), paths, *setting, 2, write_npy=True)
    assert e.value.code == _lib.LRB_EINVAL
    assert what in _lib.last_error()
    assert os.listdir(tmp_path / "profiles") == []


# ---- the compact index ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("shift", range(20, 26))
def test_compact_index_of_every_canonical_key(shift):
    """Every bit-15-clear key c: the entry the partition stores for it (partition.cu, k_partition: bit 15 dropped, a read
    delta above bit shift - 2) gathers, through (bucket_base >> 1) | (e & (2^(shift-1) - 1)), the compact position where
    lrb_dev_table_compact puts T[c]."""
    lo15, hi_mask = 0x7FFF, ((1 << (shift - 1)) - 1) & ~0x7FFF
    emask = (1 << (shift - 1)) - 1
    rng = np.random.default_rng(shift)
    step = 1 << 24
    for i0 in range(0, 1 << 29, step):   # canonical index i <-> key ((i >> 15) << 16) | (i & 0x7FFF)
        i = np.arange(i0, i0 + step, dtype=np.uint64)
        c = ((i >> 15) << 16) | (i & lo15)
        assert not np.any(c & 0x8000)
        bucket_base = (c >> shift) << shift
        delta = rng.integers(0, 256, size=step, dtype=np.uint64)
        e = ((c & lo15) | ((c >> 1) & hi_mask) | (delta << (shift - 1))) & 0xFFFFFFFF
        gathered = (bucket_base >> 1) | (e & emask)
        assert np.array_equal(gathered, i), (shift, i0)
        # a bucket's slice of a compact table is one contiguous range
        assert np.array_equal(gathered >> (shift - 1), c >> shift)


# ---- the canonical-row reader ---------------------------------------------------------------------------------------

def _sparse_table(path, n_pokes=4000, seed=7):
    """A 4 GiB 15mers-counts file that costs no disk: header, ftruncate, values written at scattered entries (both
    halves of rows, row edges included).  Returns {entry: value}."""
    rng = np.random.default_rng(seed)
    pokes = {int(k): int(v) for k, v in zip(rng.integers(0, _lib.TABLE_ENTRIES, n_pokes), rng.integers(1, 1 << 32, n_pokes))}
    for row in (0, 1, 511, 512, 513, ROWS - 1):
        for off in (0, 1, 0x7FFE, 0x7FFF, 0x8000, 0xFFFF):
            pokes[(row << 16) | off] = (row * 65536 + off) % (1 << 32) or 1
    with open(path, "wb") as f:
        f.write(np.uint64(_lib.TABLE_ENTRIES).tobytes())
        f.truncate(TABLE_BYTES)
        for k, v in sorted(pokes.items()):
            f.seek(8 + 4 * k)
            f.write(np.uint32(v).tobytes())
    return pokes


@pytest.fixture(scope="module")
def sparse_table(tmp_path_factory):
    path = tmp_path_factory.mktemp("sparse") / "15mers-counts"
    pokes = _sparse_table(str(path))
    yield str(path), pokes
    os.unlink(path)


@pytest.mark.parametrize("rows", [(0, 3), (509, 515), (1000, 2024), (ROWS - 2, ROWS), (7, 7)])
def test_canonical_rows_equal_memmap_slicing(sparse_table, rows):
    path, _ = sparse_table
    lo, hi = rows
    got = read_table_canonical(path, lo, hi)
    mm = np.memmap(path, dtype=np.uint32, mode="r", offset=8, shape=(ROWS, 1 << 16))
    assert np.array_equal(got, np.asarray(mm[lo:hi, : 1 << 15]).reshape(-1))


def test_canonical_rows_hold_exactly_the_bit15_clear_values(sparse_table):
    path, pokes = sparse_table
    want = {((k >> 16) << 15) | (k & 0x7FFF): v for k, v in pokes.items() if not k & 0x8000}
    for lo in range(0, ROWS, 2048):   # 2048 rows = 256 MiB at a time
        got = read_table_canonical(path, lo, lo + 2048)
        nz = np.flatnonzero(got)
        base = lo << 15
        assert {int(i) + base: int(got[i]) for i in nz} == {i: v for i, v in want.items() if base <= i < base + got.size}


def test_reader_refusals(sparse_table, tmp_path):
    path, _ = sparse_table
    out = np.empty(1 << 15, dtype=np.uint32)
    assert lib.lrb_table_read_canonical(b"/nonexistent/15mers-counts", 0, 1, out.ctypes.data) == _lib.LRB_EIO
    assert lib.lrb_table_read_canonical(path.encode(), 0, ROWS + 1, out.ctypes.data) == _lib.LRB_EINVAL
    assert lib.lrb_table_read_canonical(path.encode(), 3, 2, out.ctypes.data) == _lib.LRB_EINVAL
    bad = tmp_path / "bad"
    for size, header in [(TABLE_BYTES - 1, _lib.TABLE_ENTRIES), (TABLE_BYTES - 4096, _lib.TABLE_ENTRIES),
                         (TABLE_BYTES - (1 << 17) + 4, _lib.TABLE_ENTRIES), (TABLE_BYTES + 1, _lib.TABLE_ENTRIES),
                         (TABLE_BYTES, _lib.TABLE_ENTRIES - 1), (4, _lib.TABLE_ENTRIES)]:
        with open(bad, "wb") as f:
            f.write(np.uint64(header).tobytes()[: min(8, size)])
            f.truncate(size)
        # the rows asked for exist in every one of these files: only the header and size checks can refuse them
        assert lib.lrb_table_read_canonical(str(bad).encode(), 0, 1, out.ctypes.data) == _lib.LRB_EFORMAT, (size, header)
        assert "15mers-counts" in _lib.last_error()
        os.unlink(bad)
