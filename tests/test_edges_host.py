"""CPU tier: the kernels' per-lane search arithmetic (csrc/lane_core.cuh, run by tests/host_emul.cpp) at the edges of its
count range and bin settings, and on a read set that fills the partition's list layout, against the oracle.  The GPU
counterpart is tests/test_gpu_edges.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from edge_inputs import (SETTINGS, STEP_BLOCKS, TASK_BLOCKS, canonical_keys, dense_lengths, dense_occupancy, oracle_coverage,
                         oracle_table_from, plant, revcomp15, value_pool)
from oracle import oracle

from lrbinner_b200.synth import SynthSpec

EMUL_SO = os.path.join(ROOT, "tests", "_build", "libemul.so")


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul.cpp")
    deps = [src, os.path.join(ROOT, "lrbinner_b200", "csrc", "lane_core.cuh"), os.path.join(ROOT, "lrbinner_b200", "csrc", "fixed6.h")]
    if not os.path.exists(EMUL_SO) or os.path.getmtime(EMUL_SO) < max(os.path.getmtime(d) for d in deps):
        os.makedirs(os.path.dirname(EMUL_SO), exist_ok=True)
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wno-unknown-pragmas", "-fPIC", "-shared", "-o", EMUL_SO, src])
    return C.CDLL(EMUL_SO)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _emul_table(emul, pr):
    """the mirrored 15-mer table of pr, and its bit-15-clear keys"""
    table = np.zeros(2 ** 30, dtype=np.uint32)
    emul.emul_count(C.byref(pr.view), _p(table), C.c_uint32(0), C.c_uint32(2 ** 30))
    canon = np.flatnonzero(table).astype(np.uint32)
    return table, canon


def _emul_search(emul, pr, table, bs, bc):
    hist = np.zeros((pr.n_reads, bc), dtype=np.uint32)
    sums = np.zeros(pr.n_reads, dtype=np.uint32)
    emul.emul_search(C.byref(pr.view), _p(table), C.c_long(bs), bc, _p(hist), _p(sums), C.c_uint32(0), C.c_uint32(2 ** 30))
    return hist, sums


def test_planted_counts_every_edge_setting(emul):
    """every bit-15-clear key the reads hit holds a count at an edge of the bucket rule (up to 2^32 - 1); the emulated
    search bins them as the oracle does for S up to 2^40 and B up to 4096"""
    spec = SynthSpec(300, seed=61, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.01)
    seqs = spec.host_sequences()
    pr = spec.host_packed(threads=4)
    rng = np.random.default_rng(61)
    canon = canonical_keys(seqs)
    vals = plant(canon, rng, value_pool(rng))
    assert int((vals >= 2 ** 31).sum()) > 1000
    table = np.zeros(2 ** 30, dtype=np.uint32)
    table[canon] = vals
    assert emul.emul_mirror_keys(_p(table), _p(canon), C.c_uint64(len(canon))) == 0
    want_table = oracle_table_from(np.concatenate([canon, revcomp15(canon)]), np.concatenate([vals, vals]))
    for bs, bc in SETTINGS:
        hist, sums = _emul_search(emul, pr, table, bs, bc)
        want_hist, want_sums = oracle_coverage(want_table, seqs, bs, bc)
        assert np.array_equal(hist, want_hist) and np.array_equal(sums, want_sums), (bs, bc)
    want_table.close()


def test_dense_layout(emul):
    """the read set whose steps hold 256 reads and whose tasks hold 4096: layout as intended, count and search equal
    the oracle"""
    lens = dense_lengths()
    spec = SynthSpec(len(lens), lengths=lens, seed=62, n_rate=1e-3, lowercase_frac=0.01)
    seqs = spec.host_sequences()
    pr = spec.host_packed(threads=4)
    assert 38000 <= pr.n_reads <= 45000
    per_step, per_task, full = dense_occupancy(pr.read_blk, seqs)
    assert per_step.max() == STEP_BLOCKS and len(full) >= 6, (per_step.max(), full)
    assert per_task.max() == TASK_BLOCKS
    blk = np.asarray(pr.read_blk, dtype=np.int64)
    assert (blk[:-1] % STEP_BLOCKS == 0).sum() >= 40 and (blk[1:] % STEP_BLOCKS == 0).sum() >= 40
    table = np.zeros(2 ** 30, dtype=np.uint32)
    emul.emul_count(C.byref(pr.view), _p(table), C.c_uint32(0), C.c_uint32(2 ** 30))
    want = oracle.Table()
    for s in seqs:
        want.count(s)
    keys = np.flatnonzero(want.array)
    canon = keys[(keys & 0x8000) == 0].astype(np.uint32)
    assert np.count_nonzero(table) == len(canon) and np.array_equal(table[canon], want.array[canon])
    assert emul.emul_mirror_keys(_p(table), _p(canon), C.c_uint64(len(canon))) == 0
    assert np.count_nonzero(table) == len(keys) and np.array_equal(table[keys], want.array[keys])
    for bs, bc in ((1, 4096), (32, 10)):
        hist, sums = _emul_search(emul, pr, table, bs, bc)
        want_hist, want_sums = oracle_coverage(want, seqs, bs, bc)
        assert np.array_equal(hist, want_hist) and np.array_equal(sums, want_sums), (bs, bc)
    want.close()
