"""CPU tier: coverage bins given by count edges.  The argument checks of every level (device, context, file, Python, the
runner) run before any file or device is touched, so a machine without a GPU gets LRB_EINVAL, not LRB_ECUDA, and no
output file appears.  spectrum_edge_mass is compared with numpy's searchsorted, and spectrum_quantile_edges with its
defining inequality."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN

from lrbinner_b200 import _lib, runners_utils
from lrbinner_b200.profile import Context, PackedReads, PartitionWorkspace, spectrum_edge_mass, spectrum_quantile_edges

lib = _lib.lib
READS = os.path.join(GOLDEN, "g06_community.fa")

BAD_EDGES = [
    ([5, 3], "strictly increasing"),
    ([2, 7, 7, 9], "strictly increasing"),
    ([1, 5], "first edge"),
    ([0], "first edge"),
    (list(range(2, 2 + _lib.MAX_BINS)), "number of edges"),
]


def _u32(edges):
    return (C.c_uint32 * max(len(edges), 1))(*edges)


def _file_call(edges, n=None, txt=b"/nonexistent/out", table=b"/nonexistent/15mers-counts", reads=READS.encode()):
    return lib.lrb_search_15mers_edges(table, reads, _u32(edges), len(edges) if n is None else n, txt, None, 2)


@pytest.mark.parametrize("edges,what", BAD_EDGES)
def test_c_levels_refuse_bad_edges_before_any_work(edges, what):
    assert _file_call(edges) == _lib.LRB_EINVAL
    assert "lrb_search_15mers_edges" in _lib.last_error() and what in _lib.last_error(), _lib.last_error()
    # the context call checks the edges before it looks at the context
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    hist = np.zeros((1, len(edges) + 1), np.uint32)
    sums = np.zeros(1, np.uint32)
    rc = lib.lrb_profile_host_edges(None, reads._h, 0, _u32(edges), len(edges), None, hist.ctypes.data, sums.ctypes.data, None, 0)
    assert rc == _lib.LRB_EINVAL and "lrb_profile_host_edges" in _lib.last_error() and what in _lib.last_error()
    # the device-level call too, before it launches anything
    part = _lib.Partition()
    rc = lib.lrb_dev_partition_search_edges(C.byref(part), 0, 64, C.c_void_p(16), _u32(edges), len(edges), C.c_void_p(16),
                                            C.c_void_p(16), None)
    assert rc == _lib.LRB_EINVAL and "lrb_dev_partition_search_edges" in _lib.last_error() and what in _lib.last_error()
    spec = np.zeros(19, np.uint64)
    mass = np.zeros(_lib.MAX_BINS + 1, np.uint64)
    assert lib.lrb_spectrum_edge_mass(spec.ctypes.data, 16, _u32(edges), len(edges), mass.ctypes.data) == _lib.LRB_EINVAL
    assert what in _lib.last_error()


def test_c_levels_refuse_null_edges_and_counts_out_of_range():
    for n, what in ((3, "null edges"), (-1, "number of edges"), (_lib.MAX_BINS, "number of edges")):
        assert lib.lrb_search_15mers_edges(b"t", READS.encode(), None, n, b"/nonexistent/out", None, 2) == _lib.LRB_EINVAL
        assert what in _lib.last_error(), (n, _lib.last_error())
        reads = PackedReads.from_sequences([b"ACGT" * 10])
        assert lib.lrb_profile_host_edges(None, reads._h, 0, None, n, None, None, None, None, 0) == _lib.LRB_EINVAL
        assert what in _lib.last_error()
    assert _file_call([2, 3], table=None) == _lib.LRB_EINVAL
    assert _file_call([2, 3], reads=None) == _lib.LRB_EINVAL
    assert _file_call([2, 3], txt=None) == _lib.LRB_EINVAL and "null path" in _lib.last_error()


def test_direct_table_path_is_refused(monkeypatch):
    monkeypatch.setenv("LRB_TABLE_PATH", "direct")
    assert _file_call([2, 3, 4]) == _lib.LRB_EINVAL
    assert "LRB_TABLE_PATH=direct" in _lib.last_error()


def test_edge_limits_pass_the_checks():
    """4095 edges up to 2^32 - 1, no edges, a single edge of 2: past the checks (the call then fails on the missing table
    or device, never with LRB_EINVAL)"""
    top = list(range(2 ** 32 - _lib.MAX_BINS + 1, 2 ** 32))
    assert len(top) == _lib.MAX_BINS - 1
    for edges in (top, [], [2], list(range(2, _lib.MAX_BINS + 1))):
        assert _file_call(edges) != _lib.LRB_EINVAL, _lib.last_error()
    assert lib.lrb_search_15mers_edges(b"/nonexistent/t", READS.encode(), None, 0, b"/nonexistent/out", None, 2) != _lib.LRB_EINVAL


@pytest.mark.parametrize("edges,what", BAD_EDGES + [([2, 2 ** 32], "u32")])
def test_python_levels_refuse_bad_edges(edges, what, tmp_path):
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    with pytest.raises(_lib.LrbError) as e:   # before a context (and a device) is needed
        Context.profile(None, reads, edges=edges)
    assert e.value.code == _lib.LRB_EINVAL and what in str(e.value)
    with pytest.raises(_lib.LrbError) as e:
        spectrum_edge_mass(np.zeros(19, np.uint64), edges)
    assert e.value.code == _lib.LRB_EINVAL
    with pytest.raises(_lib.LrbError) as e:
        PartitionWorkspace.search_edges(None, None, edges, None, None)
    assert e.value.code == _lib.LRB_EINVAL
    with pytest.raises(SystemExit) as e:
        runners_utils.run_15mer_vecs_edges(READS, str(tmp_path), edges, 2, write_npy=True)
    assert e.value.code == _lib.LRB_EINVAL
    assert not os.path.exists(tmp_path / "profiles") or os.listdir(tmp_path / "profiles") == []


def test_runner_refusal_from_the_library_writes_nothing(tmp_path, monkeypatch):
    monkeypatch.setenv("LRB_TABLE_PATH", "direct")
    with pytest.raises(SystemExit) as e:
        runners_utils.run_15mer_vecs_edges(READS, str(tmp_path), [2, 3], 2, write_npy=True)
    assert e.value.code == _lib.LRB_EINVAL
    assert os.listdir(tmp_path / "profiles") == []


def test_context_refuses_edges_with_other_coverage_arguments():
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    for kw in (dict(bins=8), dict(bin_size=10), dict(coverage=[(10, 8)]), dict(samples=[(0, 10, 8)])):
        with pytest.raises(_lib.LrbError) as e:
            Context.profile(None, reads, edges=[2, 3], **kw)
        assert e.value.code == _lib.LRB_EINVAL and "edges=" in str(e.value), kw


# ---- spectrum_edge_mass against numpy ---------------------------------------------------------------------------

def _random_spectrum(rng, M, over):
    spec = np.zeros(M + 3, np.uint64)
    spec[1:M] = rng.integers(0, 1000, size=M - 1) * (rng.random(M - 1) < 0.3)
    if over:
        spec[M] = rng.integers(1, 50)
        spec[M + 1] = int(spec[M]) * (M + int(rng.integers(0, 1000)))
        spec[M + 2] = M + 999
    return spec


def _numpy_mass(spec, edges):
    M = spec.size - 3
    c = np.arange(M, dtype=np.uint64)
    mass = np.zeros(len(edges) + 1, np.uint64)
    np.add.at(mass, np.searchsorted(np.asarray(edges, np.int64), c.astype(np.int64), side="right"), c * spec[:M])
    mass[-1] += spec[M + 1]
    return mass


def _edge_sets(rng, M):
    yield []
    yield [2]
    yield list(range(2, 11))
    yield [2 ** i for i in range(1, 17)]
    yield sorted(set(rng.integers(2, 3 * M, size=20).tolist()))
    yield list(range(2, _lib.MAX_BINS + 1))
    yield [M - 1, M]


@pytest.mark.parametrize("seed", range(6))
def test_spectrum_edge_mass_matches_searchsorted(seed):
    rng = np.random.default_rng(seed)
    M = int(rng.choice([16, 300, 5000]))
    for over in (False, True):
        spec = _random_spectrum(rng, M, over)
        for edges in _edge_sets(rng, M):
            determined = not over or not edges or edges[-1] <= M
            if not determined:
                with pytest.raises(_lib.LrbError) as e:
                    spectrum_edge_mass(spec, edges)
                assert "below the last edge" in str(e.value)
                continue
            got = spectrum_edge_mass(spec, edges)
            assert np.array_equal(got, _numpy_mass(spec, edges)), (seed, over, edges[:5])
            assert int(got.sum()) == int((np.arange(M, dtype=np.uint64) * spec[:M]).sum()) + int(spec[M + 1])


def test_spectrum_edge_mass_equals_bin_mass_where_the_rules_agree():
    """-bs 1 -bc B is edges {2, ..., B}, and -bc 1 is no edges"""
    from lrbinner_b200.profile import spectrum_bin_mass
    spec = _random_spectrum(np.random.default_rng(9), 400, True)
    for B in (1, 2, 5, 32, 300):
        assert np.array_equal(spectrum_edge_mass(spec, list(range(2, B + 1))), spectrum_bin_mass(spec, 1, B)), B
    assert np.array_equal(spectrum_edge_mass(spec, []), spectrum_bin_mass(spec, 3, 1))


# ---- spectrum_quantile_edges ----------------------------------------------------------------------------------

def _check_quantiles(spec, B, edges):
    M = spec.size - 3
    prefix = [0]                   # prefix[c] = sum_{c' < c} c' n_c', in Python integers
    for c in range(M):
        prefix.append(prefix[-1] + c * int(spec[c]))
    total = prefix[M] + int(spec[M + 1])
    assert len(edges) <= B - 1
    assert all(isinstance(t, int) for t in edges)
    assert all(b > a for a, b in zip(edges, edges[1:]))
    assert not edges or (edges[0] >= 2 and edges[-1] <= M)
    # the t_i of the definition, repeats dropped
    want = []
    for i in range(1, B):
        c = next((c for c in range(2, M + 1) if B * prefix[c] >= i * total), None)
        if c is None:
            break
        assert B * prefix[c] >= i * total and (c == 2 or B * prefix[c - 1] < i * total)
        if not want or want[-1] != c:
            want.append(c)
    assert edges == want


@pytest.mark.parametrize("seed", range(8))
def test_quantile_edges_follow_the_definition(seed):
    rng = np.random.default_rng(100 + seed)
    M = int(rng.choice([8, 64, 700]))
    spec = _random_spectrum(rng, M, over=bool(seed % 2))
    for B in (1, 2, 3, 7, 16, 32, 100):
        _check_quantiles(spec, B, spectrum_quantile_edges(spec, B))


def test_quantile_edges_of_special_spectra():
    M = 64
    empty = np.zeros(M + 3, np.uint64)
    _check_quantiles(empty, 8, spectrum_quantile_edges(empty, 8))
    one_count = np.zeros(M + 3, np.uint64)
    one_count[10] = 500            # all the mass at one count: a single edge just above it
    e = spectrum_quantile_edges(one_count, 16)
    _check_quantiles(one_count, 16, e)
    assert e == [11]
    flat = np.zeros(M + 3, np.uint64)
    flat[1:M] = 1
    e = spectrum_quantile_edges(flat, 4)
    _check_quantiles(flat, 4, e)
    assert len(e) == 3
    mostly_over = np.zeros(M + 3, np.uint64)
    mostly_over[3], mostly_over[M], mostly_over[M + 1] = 5, 1, 70   # 15 of 85 windows below M
    e = spectrum_quantile_edges(mostly_over, 8)
    _check_quantiles(mostly_over, 8, e)
    assert e == [4]                # the rest of the mass is above M: fewer bins
    with pytest.raises(_lib.LrbError):
        spectrum_quantile_edges(flat, 0)
