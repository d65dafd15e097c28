"""CPU tier: mixed coverage rows (layouts of blocks).  The checks of every level (device, context, file, Python, the runner)
run before any file or device is touched, so a machine without a GPU gets LRB_EINVAL, not LRB_ECUDA, and no output file
appears.  The .layout file says how each block was made."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN

from lrbinner_b200 import _lib, runners_utils
from lrbinner_b200.profile import CovBlock, Context, PackedReads, PartitionWorkspace

lib = _lib.lib
READS = os.path.join(GOLDEN, "g06_community.fa")
WIDE = list(range(2, 2 + 2047))      # 2047 edges: a block of 2048 bins

# (layout as CovBlock, what the refusal names); table indices are valid at the file level (two tables)
BAD = [
    ([], "number of blocks"),
    ([CovBlock(0, 1, m + 1) for m in range(9)], "number of blocks"),
    ([CovBlock(8, 32, 10)], "table must be"),
    ([CovBlock(0, 32, 10), CovBlock(-2, 32, 10)], "table must be"),
    ([CovBlock(0, 0, 10)], "bin_size must be >= 1"),
    ([CovBlock(0, 32, 0)], "bins must be in"),
    ([CovBlock(1, 32, _lib.MAX_BINS + 1)], "bins must be in"),
    ([CovBlock(0, edges=[5, 3])], "strictly increasing"),
    ([CovBlock(0, 32, 10), CovBlock(1, edges=[1, 5])], "first edge"),
    ([CovBlock(0, edges=list(range(2, 2 + _lib.MAX_BINS)))], "number of edges"),
    ([CovBlock(0, edges=WIDE), CovBlock(1, edges=WIDE), CovBlock(0, 1, 1)], "add up to 4097"),
    ([CovBlock(0, 32, 10), CovBlock(1, edges=[2, 4]), CovBlock(0, 32, 10)], "repeats block 0"),
    ([CovBlock(1, edges=[2, 4, 8]), CovBlock(0, 32, 10), CovBlock(1, edges=[2, 4, 8])], "repeats block 0"),
]


def _c_blocks(layout, keep):
    """lrb_cov_block array of a layout without the Python checks (table None = -1)"""
    arr = (_lib.CovBlockC * max(len(layout), 1))()
    for m, b in enumerate(layout):
        t = -1 if b.table is None else int(b.table)
        if b.edges is not None:
            e = np.array(b.edges, np.uint32)
            keep.append(e)
            arr[m] = _lib.CovBlockC(t, 1, 1, 1, e.ctypes.data if e.size else None, int(e.size))
        else:
            arr[m] = _lib.CovBlockC(t, 0, int(b.bin_size), int(b.bins), None, 0)
    return arr


def _file_call(layout, paths=(b"/nonexistent/t0", b"/nonexistent/t1"), txt=b"/nonexistent/out", reads=READS.encode(), keep=None):
    keep = [] if keep is None else keep
    arr = _c_blocks(layout, keep)
    tp = (C.c_char_p * max(len(paths), 1))(*paths)
    return lib.lrb_search_15mers_layout(tp, len(paths), reads, arr, len(layout), txt, None, 2)


@pytest.mark.parametrize("layout,what", BAD)
def test_c_levels_refuse_bad_layouts_before_any_work(layout, what):
    assert _file_call(layout) == _lib.LRB_EINVAL
    assert "lrb_search_15mers_layout" in _lib.last_error() and what in _lib.last_error(), _lib.last_error()
    keep = []
    arr = _c_blocks(layout, keep)
    # the context call checks the layout before it looks at the context
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    hist = np.zeros((1, 4096), np.uint32)
    sums = np.zeros(1, np.uint32)
    rc = lib.lrb_profile_host_layout(None, reads._h, 0, arr, len(layout), None, hist.ctypes.data, sums.ctypes.data, None, 0)
    assert rc == _lib.LRB_EINVAL and "lrb_profile_host_layout" in _lib.last_error() and what in _lib.last_error(), _lib.last_error()
    # the device-level call too, before it launches anything
    part = _lib.Partition()
    slots = (C.c_void_p * 8)(*([16] * 8))
    rc = lib.lrb_dev_partition_search_layout(C.byref(part), 0, 64, C.c_void_p(16), slots, arr, len(layout), C.c_void_p(16), C.c_void_p(16),
                                             None)
    assert rc == _lib.LRB_EINVAL and "lrb_dev_partition_search_layout" in _lib.last_error() and what in _lib.last_error()


@pytest.mark.parametrize("layout,what", BAD)
def test_python_levels_refuse_bad_layouts(layout, what, tmp_path):
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    with pytest.raises(_lib.LrbError) as e:   # before a context (and a device) is needed
        Context.profile(None, reads, layout=layout)
    assert e.value.code == _lib.LRB_EINVAL and what in str(e.value), str(e.value)
    with pytest.raises(_lib.LrbError) as e:
        PartitionWorkspace.search_layout(None, None, None, layout, None, None)
    assert e.value.code == _lib.LRB_EINVAL
    with pytest.raises(SystemExit) as e:
        runners_utils.run_15mer_vecs_layout(READS, str(tmp_path), ["/nonexistent/t0", "/nonexistent/t1"], layout, 2, write_npy=True)
    assert e.value.code == _lib.LRB_EINVAL
    assert not os.path.exists(tmp_path / "profiles") or os.listdir(tmp_path / "profiles") == []


def test_file_level_refuses_the_context_table_and_bad_table_indices(tmp_path):
    for layout in ([CovBlock(None, 32, 10)], [CovBlock(0, 32, 10), CovBlock(None, edges=[2, 3])], [CovBlock(2, 32, 10)]):
        assert _file_call(layout) == _lib.LRB_EINVAL
        assert "names its table by its index" in _lib.last_error(), _lib.last_error()
        with pytest.raises(SystemExit) as e:
            runners_utils.run_15mer_vecs_layout(READS, str(tmp_path), ["/nonexistent/t0", "/nonexistent/t1"], layout, 2)
        assert e.value.code == _lib.LRB_EINVAL
    assert not os.path.exists(tmp_path / "profiles")
    for paths in ((), tuple(b"/nonexistent/t%d" % i for i in range(9))):
        assert _file_call([CovBlock(0, 32, 10)], paths=paths) == _lib.LRB_EINVAL
        assert "number of tables" in _lib.last_error()
    # a path listed twice is one table: the same binning on both is a repeated block
    assert _file_call([CovBlock(0, 32, 10), CovBlock(1, 32, 10)], paths=(b"/nonexistent/t", b"/nonexistent/t")) == _lib.LRB_EINVAL
    assert "repeats block 0" in _lib.last_error()
    assert _file_call([CovBlock(0, 32, 10)], paths=(b"/nonexistent/t", None)) == _lib.LRB_EINVAL
    assert "null table path" in _lib.last_error()
    assert _file_call([CovBlock(0, 32, 10)], txt=None) == _lib.LRB_EINVAL and "null path" in _lib.last_error()
    assert _file_call([CovBlock(0, 32, 10)], reads=None) == _lib.LRB_EINVAL


def test_null_blocks_and_null_tables():
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    assert lib.lrb_profile_host_layout(None, reads._h, 0, None, 2, None, None, None, None, 0) == _lib.LRB_EINVAL
    assert "null blocks" in _lib.last_error()
    part = _lib.Partition()
    keep = []
    full = _c_blocks([CovBlock(None, 32, 10), CovBlock(3, edges=[2])], keep)
    rc = lib.lrb_dev_partition_search_layout(C.byref(part), 0, 64, None, (C.c_void_p * 8)(*([16] * 8)), full, 2, C.c_void_p(16),
                                             C.c_void_p(16), None)
    assert rc == _lib.LRB_EINVAL and "null table" in _lib.last_error()
    rc = lib.lrb_dev_partition_search_layout(C.byref(part), 0, 64, C.c_void_p(16), (C.c_void_p * 8)(), full, 2, C.c_void_p(16),
                                             C.c_void_p(16), None)
    assert rc == _lib.LRB_EINVAL and "null compact table 3" in _lib.last_error()
    rc = lib.lrb_dev_partition_search_layout(C.byref(part), 0, 64, C.c_void_p(16), None, full, 2, C.c_void_p(16), C.c_void_p(16), None)
    assert rc == _lib.LRB_EINVAL and "null compact table 3" in _lib.last_error()


def test_context_refusals_without_a_context():
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    good = [CovBlock(None, 32, 10), CovBlock(0, edges=[2, 5])]
    keep = []
    arr = _c_blocks(good, keep)
    rc = lib.lrb_profile_host_layout(None, reads._h, 0, arr, 2, None, None, None, None, 0)
    assert rc == _lib.LRB_EINVAL and "null context" in _lib.last_error()
    spec = np.zeros(19, np.uint64)
    for slot, what in ((-1, "slot must be"), (8, "slot must be")):
        assert lib.lrb_ctx_sample_table_spectrum(C.c_void_p(16), slot, 16, spec.ctypes.data) == _lib.LRB_EINVAL
        assert what in _lib.last_error()
    assert lib.lrb_ctx_sample_table_spectrum(None, 0, 16, spec.ctypes.data) == _lib.LRB_EINVAL and "null context" in _lib.last_error()
    assert lib.lrb_dev_compact_spectrum(None, 16, None, None) == _lib.LRB_EINVAL
    assert lib.lrb_dev_compact_spectrum(C.c_void_p(16), 1, C.c_void_p(16), None) == _lib.LRB_EINVAL and "max_count" in _lib.last_error()
    assert lib.lrb_dev_compact_spectrum(C.c_void_p(20), 16, C.c_void_p(16), None) == _lib.LRB_EINVAL and "aligned" in _lib.last_error()


def test_direct_table_path_is_refused(monkeypatch, tmp_path):
    monkeypatch.setenv("LRB_TABLE_PATH", "direct")
    assert _file_call([CovBlock(0, 32, 10), CovBlock(1, edges=[2, 3])]) == _lib.LRB_EINVAL
    assert "LRB_TABLE_PATH=direct" in _lib.last_error() and "layout of 2 blocks" in _lib.last_error()
    with pytest.raises(SystemExit) as e:
        runners_utils.run_15mer_vecs_layout(READS, str(tmp_path), ["/nonexistent/t0"], [CovBlock(0, 32, 10)], 2, write_npy=True)
    assert e.value.code == _lib.LRB_EINVAL
    assert os.listdir(tmp_path / "profiles") == []


def test_layout_limits_pass_the_checks():
    """8 blocks, a row of exactly 4096 bins, every slot, edges up to 2^32 - 1: past the checks (the call then fails on the
    missing tables, never with LRB_EINVAL)"""
    paths = tuple(b"/nonexistent/t%d" % i for i in range(8))
    eight = [CovBlock(t, 32, 10) if t % 2 else CovBlock(t, edges=[2 ** 32 - 2, 2 ** 32 - 1]) for t in range(8)]
    full = [CovBlock(0, edges=WIDE), CovBlock(1, edges=WIDE[:-1]), CovBlock(0, 3, 1)]
    assert sum(len(b.edges) + 1 if b.edges is not None else b.bins for b in full) == _lib.MAX_BINS
    for layout in (eight, full, [CovBlock(0, edges=[2, 3]), CovBlock(0, edges=[2, 4])], [CovBlock(1, edges=[]), CovBlock(0, edges=[])]):
        assert _file_call(layout, paths=paths) != _lib.LRB_EINVAL, _lib.last_error()


def test_context_refuses_layout_with_other_coverage_arguments():
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    for kw in (dict(bins=8), dict(bin_size=10), dict(coverage=[(10, 8)]), dict(samples=[(0, 10, 8)]), dict(edges=[2, 3])):
        with pytest.raises(_lib.LrbError) as e:
            Context.profile(None, reads, layout=[CovBlock(None, 32, 10)], **kw)
        assert e.value.code == _lib.LRB_EINVAL and "layout=" in str(e.value), kw
    for bad in ([(None, 32, 10)], [CovBlock(None, 32)], [CovBlock(None, 32, 10, [2, 3])]):
        with pytest.raises(_lib.LrbError) as e:
            Context.profile(None, reads, layout=bad)
        assert e.value.code == _lib.LRB_EINVAL


def test_layout_file_lines():
    paths = ["/data/s1/profiles/15mers-counts", "/data/s2/profiles/15mers-counts"]
    blocks = [CovBlock(1, edges=[2, 7, 40]), CovBlock(0, 32, 10), CovBlock(1, edges=[])]
    assert runners_utils.layout_lines(paths, blocks) == [
        "/data/s2/profiles/15mers-counts\tedges 2 7 40\n",
        "/data/s1/profiles/15mers-counts\tbs 32 bc 10\n",
        "/data/s2/profiles/15mers-counts\tedges\n",
    ]
