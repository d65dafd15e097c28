"""CPU tier: argument checks of the multi-setting coverage search (lrb_search_15mers_settings, run_15mer_vecs_settings,
Context.profile(coverage=...)).  Every check runs before any file or device is touched, so a machine without a GPU
gets LRB_EINVAL, not LRB_ECUDA, and no output file appears."""
import ctypes as C
import os

import pytest

from conftest import COV_PARAMS, GOLDEN

from lrbinner_b200 import _lib, runners_utils

lib = _lib.lib
READS = os.path.join(GOLDEN, "g06_community.fa")

BAD_SETTINGS = [
    ([], "number of settings"),
    ([(10, 8)] * 9, "number of settings"),
    ([(10, 8), (0, 5)], "bin_size"),
    ([(-3, 5)], "bin_size"),
    ([(10, 0)], "bins"),
    ([(10, 8), (2, 4097)], "bins"),
    ([(10, 8), (3, -1)], "bins"),
    ([(10, 8), (32, 10), (10, 8)], "repeats"),
    ([(1, 4096), (2, 1)], "add up to 4097"),
    ([(s, 1000) for s in range(1, 6)], "add up to 5000"),
]


def _call(settings, txts=None, npys=None, table=b"/nonexistent/15mers-counts", reads=READS.encode()):
    n = len(settings)
    bs = (C.c_long * max(n, 1))(*[s for s, _ in settings])
    bc = (C.c_int * max(n, 1))(*[b for _, b in settings])
    if txts is None:
        txts = [f"/nonexistent/out{m}".encode() for m in range(n)]
    t = (C.c_char_p * max(len(txts), 1))(*txts)
    p = (C.c_char_p * max(len(npys), 1))(*npys) if npys is not None else None
    return lib.lrb_search_15mers_settings(table, reads, n, bs, bc, t, p, 2)


@pytest.mark.parametrize("settings,what", BAD_SETTINGS)
def test_file_level_refuses_bad_settings_before_any_work(settings, what):
    assert _call(settings) == _lib.LRB_EINVAL
    msg = _lib.last_error()
    assert "lrb_search_15mers_settings" in msg and what in msg, msg


def test_file_level_refuses_null_paths():
    good = list(COV_PARAMS)
    assert _call(good, table=None) == _lib.LRB_EINVAL
    assert _call(good, reads=None) == _lib.LRB_EINVAL
    txts = [f"/nonexistent/out{m}".encode() for m in range(len(good))]
    txts[3] = None
    assert _call(good, txts=txts) == _lib.LRB_EINVAL
    assert "setting 3" in _lib.last_error()
    bs = (C.c_long * 1)(10)
    assert lib.lrb_search_15mers_settings(b"t", b"r", 1, bs, None, None, None, 2) == _lib.LRB_EINVAL


def test_direct_table_path_refuses_several_settings(monkeypatch):
    monkeypatch.setenv("LRB_TABLE_PATH", "direct")
    assert _call(list(COV_PARAMS)) == _lib.LRB_EINVAL
    assert "LRB_TABLE_PATH=direct" in _lib.last_error() and "6 settings" in _lib.last_error()


def test_every_setting_limit_is_accepted_by_the_checks():
    """eight settings, bins adding up to exactly 4096, the largest bin_size: past the checks (the call then fails on the
    missing table or device, never with LRB_EINVAL)"""
    settings = [(1, 4089), (2 ** 40, 1), (2, 1), (3, 1), (4, 1), (5, 1), (6, 1), (7, 1)]
    assert sum(b for _, b in settings) == _lib.MAX_BINS and len(settings) == _lib.MAX_COV_SETTINGS
    assert _call(settings) != _lib.LRB_EINVAL


@pytest.mark.parametrize("settings,what", BAD_SETTINGS)
def test_runner_exits_before_writing_anything(settings, what, tmp_path):
    with pytest.raises(SystemExit) as e:
        runners_utils.run_15mer_vecs_settings(READS, str(tmp_path), settings, 2, write_npy=True)
    assert e.value.code == _lib.LRB_EINVAL
    assert what in _lib.last_error()
    assert os.listdir(tmp_path / "profiles") == []


def test_context_rejects_coverage_together_with_bin_size():
    from lrbinner_b200.profile import Context, PackedReads
    reads = PackedReads.from_sequences([b"ACGT" * 10])
    # the mixed call is refused in Python, before a context (and a device) is needed
    with pytest.raises(_lib.LrbError) as e:
        Context.profile(None, reads, bin_size=10, coverage=[(10, 8)])
    assert e.value.code == _lib.LRB_EINVAL
    with pytest.raises(_lib.LrbError):
        Context.profile(None, reads, bins=8, coverage=[(10, 8)])

