"""Pins oracle/ (the CPU restatement) to the outputs of the UNMODIFIED reference tools.

tests/golden/* were produced by tests/golden/make_golden.py running oracle/_ref/{count-kmers,
count-15mers,search-15mers} (compiled from /root/reference).  The reference ships no tests of its own
(SURVEY.md section 4), so these fixtures are the known-answer vectors for the whole path.
"""
import gzip
import os

import numpy as np
import pytest

from conftest import COV_PARAMS, GOLDEN, golden_inputs
from oracle import oracle


def _gz(path):
    with gzip.open(path, "rb") as f:
        return f.read()


def _com_text(seqs, k):
    lut, width = oracle.kmer_lut(k)
    out = []
    for s in seqs:
        _, _, prof = oracle.composition(s, k)
        out.append("".join(oracle.format_f(v) + " " for v in prof) + "\n")
    return "".join(out).encode()


@pytest.mark.parametrize("name", golden_inputs())
def test_oracle_matches_reference_tools(name, tmp_path):
    stem = name.split(".")[0]
    src = os.path.join(GOLDEN, name)
    seqs, _ = oracle.load_reads(src)
    # composition text, all k
    for k in (3, 4, 5):
        assert _com_text(seqs, k) == _gz(os.path.join(GOLDEN, f"{stem}.com_k{k}.txt.gz")), (name, k)
    # 15-mer table
    gold = np.load(os.path.join(GOLDEN, f"{stem}.table.npz"))
    t = oracle.Table()
    for s in seqs:
        t.count(s)
    keys = gold["keys"].astype(np.int64)
    assert np.array_equal(t.array[keys], gold["counts"])
    assert int(t.array[keys].astype(np.uint64).sum()) == sum(int(v) for v in gold["counts"].astype(np.uint64))
    # nothing outside the golden support: total mass must match 2 * valid windows
    nwin = sum(oracle.Table.coverage(t, s, 1, 1)[1] for s in seqs)
    assert int(gold["counts"].astype(np.uint64).sum()) == 2 * nwin
    # coverage text
    for bs, bc in COV_PARAMS:
        rows = []
        for s in seqs:
            _, _, vec = t.coverage(s, bs, bc)
            rows.append(" ".join(oracle.format_f(v) for v in vec) + "\n")
        assert "".join(rows).encode() == _gz(os.path.join(GOLDEN, f"{stem}.cov_bs{bs}_bc{bc}.txt.gz")), (name, bs, bc)
    t.close()


def test_oracle_file_drivers_byte_identical(tmp_path):
    # the file-level drivers reproduce the tools' files (text outputs; the 4 GiB table is checked sparsely above)
    src = os.path.join(GOLDEN, "g03_edge.fa")
    out = str(tmp_path / "com")
    for k in (3, 4, 5):
        assert oracle.count_kmers_file(src, out, k) == 0
        assert open(out, "rb").read() == _gz(os.path.join(GOLDEN, f"g03_edge.com_k{k}.txt.gz"))


@pytest.mark.parametrize("name", ["g03_edge.fa", "g06_community.fa"])
def test_oracle_table_and_search_file_drivers_byte_identical(name, tmp_path):
    # the whole 15mers-counts file (size + sha256 of the reference's) and search-15mers' text read back from it
    import hashlib
    import shutil
    import tempfile
    stem = name.split(".")[0]
    src = os.path.join(GOLDEN, name)
    gold = np.load(os.path.join(GOLDEN, f"{stem}.table.npz"))
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 6 * 2 ** 30 else str(tmp_path)
    work = tempfile.mkdtemp(prefix="lrb_pins_", dir=base)
    try:
        table, cov = os.path.join(work, "15mers-counts"), os.path.join(work, "cov_profs")
        assert oracle.count_15mers_file(src, table) == 0
        h = hashlib.sha256()
        with open(table, "rb") as f:
            for blk in iter(lambda: f.read(1 << 24), b""):
                h.update(blk)
        assert os.path.getsize(table) == int(gold["file_bytes"]) and h.hexdigest() == str(gold["sha256"])
        for bs, bc in COV_PARAMS:
            assert oracle.search_15mers_file(table, src, cov, bs, bc) == 0
            assert open(cov, "rb").read() == _gz(os.path.join(GOLDEN, f"{stem}.cov_bs{bs}_bc{bc}.txt.gz")), (name, bs, bc)
    finally:
        shutil.rmtree(work, ignore_errors=True)


def test_known_answers_survey_section4():
    # SURVEY.md section 4 probes, observed on the reference binaries
    assert _gz(os.path.join(GOLDEN, "g01_identical25.cov_bs10_bc8.txt.gz")).splitlines()[0] == b"0.000000 1.000000 0.000000 0.000000 0.000000 0.000000 0.000000 0.000000"
    assert _gz(os.path.join(GOLDEN, "g02_identical12.cov_bs10_bc8.txt.gz")).splitlines()[0] == b"0.000000 0.000000 0.000000 0.000000 0.000000 0.000000 0.000000 1.000000"
    t = oracle.Table()
    t.count("A" * 20)
    assert t.array[0] == 6 and t.array[oracle.revcomp(0, 15)] == 6   # polyA and polyT
    t.close()
    lut, width = oracle.kmer_lut(3)
    assert width == 32
    assert list(lut) == [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 2, 10, 11, 12, 6, 13, 14, 15, 10, 16, 17, 18, 13, 19, 20, 21, 3, 16, 22,
                         23, 7, 19, 24, 25, 8, 20, 26, 27, 11, 22, 24, 28, 0, 14, 26, 29, 4, 17, 28, 30, 9, 21, 29, 31, 12, 23,
                         25, 30, 1, 15, 27, 31, 5, 18]
    assert oracle.kmer_lut(4)[1] == 136 and oracle.kmer_lut(5)[1] == 512
    # bucket quirks (kmer_utils.h:54-69): singleton -> 0 -> bin 0; (S, 2S) -> last bin; pos >= bins -> last bin
    assert oracle.bucket(1, 10, 8) == 0 and oracle.bucket(10, 10, 8) == 0
    assert oracle.bucket(12, 10, 8) == 7 and oracle.bucket(25, 10, 8) == 1 and oracle.bucket(10**6, 10, 8) == 7
