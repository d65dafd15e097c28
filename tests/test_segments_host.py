"""Host tier of the segment reader (lrb_reader_*) and of the append forms of the row writers: no device needed.

A segment is a contiguous run of whole records of at most `segment_bases` bases (a longer record forms a segment on its
own); concatenated, the segments must be exactly the read set of lrb_reads_from_file, for every budget and every chunking
of the input, plain and gzip.
"""
import ctypes as C
import gzip
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_inputs
from oracle import oracle

from lrbinner_b200 import _lib
from lrbinner_b200.profile import COMP_WIDTH, PackedReads, SegmentReader, read_segments

INPUTS = golden_inputs() + ["g10_fragments.fasta"]


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class _env:
    def __init__(self, **kw):
        self.kw = {k: v for k, v in kw.items()}

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kw}
        for k, v in self.kw.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = str(v)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _raw(path):
    if path.endswith(".gz"):
        with gzip.open(path, "rb") as f:
            return f.read()
    return open(path, "rb").read()


def _valid_from_exceptions(pr):
    """validity words rebuilt from the read lengths + the exception list (what the device does)"""
    blk, ln = np.asarray(pr.read_blk, dtype=np.int64), np.asarray(pr.read_len, dtype=np.int64)
    want = np.zeros(pr.n_blocks, dtype=np.uint32)
    for r in range(pr.n_reads):
        for b in range(blk[r], blk[r + 1]):
            n_in = min(32, max(0, ln[r] - 32 * (b - blk[r])))
            want[b] = 0xFFFFFFFF if n_in == 32 else (1 << n_in) - 1
    eb, ew = pr.exceptions()
    if len(eb):
        want[eb] = ew
    return want


def _segments(path, budget, threads):
    rd = SegmentReader(path, budget, threads)
    segs = list(rd)
    info = rd.tell()
    return rd, segs, info


def _check_against_whole(whole, segs, budget, what):
    assert sum(s.n_reads for s in segs) == whole.n_reads, what
    r0 = b0 = 0
    for i, s in enumerate(segs):
        assert s.n_reads > 0, what
        # the budget holds, except for a single read longer than it; and the next read would not have fitted
        assert s.total_bases <= budget or s.n_reads == 1, (what, i, s.total_bases)
        if i + 1 < len(segs):
            assert s.total_bases + int(segs[i + 1].read_len[0]) > budget, (what, i)
        n, nb = s.n_reads, s.n_blocks
        assert np.array_equal(s.read_len, whole.read_len[r0:r0 + n]), (what, i)
        assert np.array_equal(s.read_blk, whole.read_blk[r0:r0 + n + 1] - whole.read_blk[r0]), (what, i)
        assert np.array_equal(s.codes[:2 * nb], whole.codes[2 * b0:2 * (b0 + nb)]), (what, i)
        assert np.array_equal(_valid_from_exceptions(s), whole.valid[b0:b0 + nb]), (what, i)
        r0 += n
        b0 += nb
    assert b0 == whole.n_blocks, what


# (LRB_GZ_CHUNK, LRB_PARSE_CHUNK, threads, segment budget in bases): chunks down to one byte, budgets from one base to
# more than the file
_SMALL_FILE_CASES = [(1, None, 1, 1), (1, None, 2, 300), (3, 2, 2, 50), (64, 16, 4, 1000), (1000, 100, 3, 7),
                     (4096, None, 8, 20000), (None, None, 8, 10 ** 12)]
_LARGE_FILE_CASES = [(7, 3, 2, 5000), (64, 16, 4, 1), (1000, 100, 3, 7), (4096, None, 8, 20000), (65536, 1000, 8, 40000),
                     (None, None, 8, 10 ** 12)]


@pytest.mark.parametrize("gz", [False, True], ids=["plain", "gzip"])
@pytest.mark.parametrize("name", INPUTS)
def test_segments_concatenate_to_the_whole_file(name, gz, tmp_path):
    src = os.path.join(GOLDEN, name)
    raw = _raw(src)
    path = tmp_path / ("in.gz" if gz else "in.txt")
    if gz:
        with gzip.open(path, "wb") as f:
            f.write(raw)
    else:
        path.write_bytes(raw)
    seqs, _ = oracle.parse_reads(raw)
    whole = PackedReads.from_file(src, threads=2)
    assert list(whole.read_len) == [len(s) for s in seqs]
    cases = _SMALL_FILE_CASES if len(raw) < 10000 else _LARGE_FILE_CASES
    for chunk, pchunk, threads, budget in cases:
        what = (name, gz, chunk, pchunk, threads, budget)
        with _env(LRB_GZ_CHUNK=chunk, LRB_PARSE_CHUNK=pchunk):
            rd, segs, info = _segments(str(path), budget, threads)
            _check_against_whole(whole, segs, budget, what)
            assert info == {"reads": whole.n_reads, "bases": whole.total_bases, "segments": len(segs), "at_end": True}, what
            # a rewind yields the same segments
            rd.rewind()
            assert rd.tell()["reads"] == 0
            again = list(rd)
            assert len(again) == len(segs), what
            for a, b in zip(segs, again):
                assert np.array_equal(a.read_len, b.read_len) and np.array_equal(a.codes, b.codes), what
                assert all(np.array_equal(x, y) for x, y in zip(a.exceptions(), b.exceptions())), what
            rd.close()


def _soup(rng, n_max):
    alphabet = np.frombuffer(b"ACGTacgtN>@+\n\r \t;-", dtype=np.uint8)
    probs = np.array([8, 8, 8, 8, 1, 1, 1, 1, 1, .6, .6, .6, 4, 1.5, .5, .3, .2, .2])
    probs /= probs.sum()
    return rng.choice(alphabet, size=int(rng.integers(0, n_max)), p=probs).tobytes()


def test_segment_reader_fuzz_against_oracle(tmp_path):
    """the byte soups of the whole-file ingest tests (headers, quality-like lines, CR, well-formed FASTQ records), plain and
    gzip, through the reader at budgets of a few bases with chunks of a few bytes"""
    rng = np.random.default_rng(2024)
    for it in range(160):
        data = _soup(rng, 500)
        if it % 5 == 0:
            data = b">" + data
        if it % 7 == 0:
            data = data.replace(b"+", b"+\n")
        if it % 3 == 0:
            s = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=int(rng.integers(1, 40))).tobytes()
            data = b"@r\n" + s + b"\n+\n" + b"@" * len(s) + b"\n" + data
        seqs, _ = oracle.parse_reads(data)
        gz = it % 2 == 1
        path = tmp_path / f"s{it}.{'gz' if gz else 'txt'}"
        if gz:
            with gzip.open(path, "wb") as f:
                f.write(data)
        else:
            path.write_bytes(data)
        for chunk, pchunk, threads, budget in ((1, None, 1, 1), (5, 3, 4, 5), (37, 8, 3, 40)):
            with _env(LRB_GZ_CHUNK=chunk, LRB_PARSE_CHUNK=pchunk):
                segs = list(read_segments(str(path), budget, threads))
            got = [(seg.unpack(i), int(seg.read_len[i])) for seg in segs for i in range(seg.n_reads)]
            assert [g[1] for g in got] == [len(x) for x in seqs], (it, chunk, budget, data)
            for (u, _), x in zip(got, seqs):
                assert u == bytes(b"ACTG"[(c >> 1) & 3] for c in x), (it, chunk, budget)
            for seg in segs:
                assert seg.total_bases <= budget or seg.n_reads == 1, (it, chunk, budget)


@pytest.mark.parametrize("data,want", [
    # a FASTQ record with a short quality block ends the stream for good, also when it falls in a later segment
    (b"@a\nACGT\n+\nIIII\n@b\nAC\n+\nI\n@c\nGG\n+\nII\n", [b"ACGT"]),
    (b">x\nAC\n>y\nGT\n>w\nT\n@b\nAC\n+\nI\n>z\nAAAA\n", [b"AC", b"GT", b"T"]),
    (b">x\nACG\n>y\nGT\n@b\nACGTACGT\n+\n", [b"ACG", b"GT"]),
    # empty records still produce reads (rows); a sequence is cut at its first NUL; CR is stripped
    (b">a\n>b\nAC\n>c\n", [b"", b"AC", b""]),
    (b">a\nAC\0GT\n>b\nGG\r\n>c\r\nA\r\nC\r\n", [b"AC", b"GG", b"AC"]),
])
def test_segment_boundaries_keep_the_record_rules(data, want, tmp_path):
    assert oracle.parse_reads(data)[0] == want
    for gz in (False, True):
        path = tmp_path / ("f.gz" if gz else "f.txt")
        if gz:
            with gzip.open(path, "wb") as f:
                f.write(data)
        else:
            path.write_bytes(data)
        for chunk in (1, 2, 3, 5, 8, 1 << 20):
            for budget in (1, 2, 3, 4, 100):
                with _env(LRB_GZ_CHUNK=chunk, LRB_PARSE_CHUNK=1):
                    segs = list(read_segments(str(path), budget, 2))
                got = [seg.unpack(i) for seg in segs for i in range(seg.n_reads)]
                assert [len(g) for g in got] == [len(w) for w in want], (gz, chunk, budget)
                assert got == [bytes(b"ACTG"[(c >> 1) & 3] for c in w) for w in want], (gz, chunk, budget)


def test_automatic_budget_and_its_override(tmp_path):
    src = os.path.join(GOLDEN, "g06_community.fa")
    whole = PackedReads.from_file(src)
    with _env(LRB_SEGMENT_BASES=None):
        segs = list(read_segments(src))                # automatic: sized from MemAvailable, far above this file
    assert len(segs) == 1 and np.array_equal(segs[0].read_len, whole.read_len)
    with _env(LRB_SEGMENT_BASES=30000):
        segs = list(read_segments(src))
    assert len(segs) > 1
    _check_against_whole(whole, segs, 30000, "override")
    # an explicit budget is not overridden
    with _env(LRB_SEGMENT_BASES=30000):
        assert len(list(read_segments(src, segment_bases=10 ** 9))) == 1


def test_missing_and_empty_files_are_empty_streams(tmp_path):
    rd = SegmentReader(str(tmp_path / "nope.fa"), 10)
    assert rd.next() is None and rd.tell() == {"reads": 0, "bases": 0, "segments": 0, "at_end": True}
    rd.rewind()
    assert rd.next() is None
    (tmp_path / "empty.fa").write_bytes(b"")
    assert list(read_segments(str(tmp_path / "empty.fa"), 10)) == []
    (tmp_path / "noise.fa").write_bytes(b"no header here\n")
    assert list(read_segments(str(tmp_path / "noise.fa"), 10)) == []


# ---- append forms of the writers -------------------------------------------------------------------------------------

def _splits(rng, n):
    cuts = sorted(set(int(x) for x in rng.integers(0, n + 1, size=int(rng.integers(0, 6)))))
    edges = [0] + cuts + [n]
    return [(a, b) for a, b in zip(edges[:-1], edges[1:])]


@pytest.mark.parametrize("kind", ["composition", "coverage"])
def test_append_writers_equal_the_one_shot_writers(kind, tmp_path):
    rng = np.random.default_rng(11 if kind == "composition" else 12)
    for it, n in enumerate([0, 1, 7, 300, 1000]):
        if kind == "composition":
            k = (3, 4, 5)[it % 3]
            width, arg = COMP_WIDTH[k], k
            read_len = rng.integers(0, 3000, size=n).astype(np.uint32)
            counts = rng.integers(0, 40, size=(n, width)).astype(np.uint32)
            denom = read_len
        else:
            bins = (1, 3, 10, 32, 64)[it]
            width, arg = bins, bins
            counts = rng.integers(0, 500, size=(n, bins)).astype(np.uint32)
            denom = counts.sum(axis=1).astype(np.uint32) + rng.integers(0, 3, size=n).astype(np.uint32)
        counts = np.ascontiguousarray(counts)
        for ext in ("txt", "npy"):
            one = str(tmp_path / f"one.{ext}")
            f_one = getattr(_lib.lib, f"lrb_write_{kind}_{ext}")
            f_app = getattr(_lib.lib, f"lrb_append_{kind}_{ext}")
            assert f_one(one.encode(), _ptr(counts), _ptr(denom), n, arg, 3) == 0
            for rep in range(4):
                parts = str(tmp_path / f"parts{rep}.{ext}")
                with open(parts, "wb") as f:
                    f.write(b"x" * 5000)          # whatever was there before is truncated by the first part
                for a, b in _splits(rng, n) if rep else [(0, n)]:
                    c = np.ascontiguousarray(counts[a:b])
                    d = np.ascontiguousarray(denom[a:b])
                    assert f_app(parts.encode(), _ptr(c), _ptr(d), b - a, arg, 1 + rep, a) == 0
                assert open(parts, "rb").read() == open(one, "rb").read(), (kind, ext, n, rep)
                if ext == "npy":
                    got = np.load(parts)
                    assert got.shape == (n, width) and np.array_equal(got, np.load(one))
