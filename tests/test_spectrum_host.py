"""CPU tier: the host side of the 15-mer abundance spectrum — the projection onto coverage bins
(lrb_spectrum_bin_mass) against the oracle's bucket rule, and the jellyfish-style text writer."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import COV_PARAMS, GOLDEN
from oracle import oracle

from lrbinner_b200 import _lib
from lrbinner_b200.profile import spectrum_bin_mass


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _mass_oracle(spec, S, B):
    """mass[b] = sum_c c * n_c over counts in bin b (oracle.bucket), overflow sum into the last bin; exact, mod 2^64."""
    M = len(spec) - 3
    mass = [0] * B
    for c in np.flatnonzero(spec[:M]):
        mass[oracle.bucket(int(c), S, B)] += int(c) * int(spec[c])
    mass[B - 1] += int(spec[M + 1])
    return np.array([m % 2 ** 64 for m in mass], dtype=np.uint64)


def _random_spectrum(rng, M, overflow):
    spec = np.zeros(M + 3, dtype=np.uint64)
    # a Poisson-like floor, a few genomic peaks and sparse high counts
    spec[:M] = rng.integers(0, 1 << 20, size=M, dtype=np.uint64) * (rng.random(M) < 0.3)
    spec[0] = 1 << 29
    if overflow:
        n_over = int(rng.integers(1, 5000))
        spec[M] = n_over
        spec[M + 1] = n_over * M + int(rng.integers(0, 1 << 40))        # above 2^32 on purpose
        spec[M + 2] = 2 ** 32 - 1
    else:
        spec[M + 2] = int(np.flatnonzero(spec[:M]).max())
    return spec


def _pairs(M):
    pairs = list(COV_PARAMS) + [(1, 1)]
    # S * (B + 1) == M exactly: the smallest M whose overflow bin is determined
    pairs += [(S, M // S - 1) for S in (1, 2, 8, 64) if M % S == 0 and 1 <= M // S - 1 <= _lib.MAX_BINS]
    return pairs


@pytest.mark.parametrize("M", [2, 33, 512, 4096])
@pytest.mark.parametrize("overflow", [False, True])
def test_bin_mass_matches_oracle_bucket_rule(M, overflow):
    rng = np.random.default_rng(M * 2 + overflow)
    for rep in range(3):
        spec = _random_spectrum(rng, M, overflow)
        for S, B in _pairs(M):
            mass = np.zeros(B, dtype=np.uint64)
            rc = _lib.lib.lrb_spectrum_bin_mass(_p(spec), M, S, B, _p(mass))
            if overflow and M < S * (B + 1):
                assert rc == _lib.LRB_EINVAL, (M, S, B)
                continue
            assert rc == 0, (M, S, B, _lib.last_error())
            assert np.array_equal(mass, _mass_oracle(spec, S, B)), (M, S, B)
            assert np.array_equal(spectrum_bin_mass(spec, S, B), mass)


def test_bin_mass_overflow_rule_boundary():
    M = 4096
    spec = np.zeros(M + 3, dtype=np.uint64)
    spec[5], spec[M], spec[M + 1] = 7, 3, 3 * (2 ** 32 - 1)
    assert np.array_equal(spectrum_bin_mass(spec, 32, 127), [35] + [0] * 125 + [3 * (2 ** 32 - 1)])   # 32 * 128 == M
    with pytest.raises(_lib.LrbError) as e:
        spectrum_bin_mass(spec, 32, 128)                                                              # 32 * 129 > M
    assert e.value.code == _lib.LRB_EINVAL
    with pytest.raises(_lib.LrbError):
        spectrum_bin_mass(spec, 2 ** 40, 3)                                                           # S far above M
    spec[M] = spec[M + 1] = 0                                                                         # no overflow: any (S, B)
    assert np.array_equal(spectrum_bin_mass(spec, 32, 128)[:1], [35])


def test_bin_mass_rejects_bad_parameters():
    spec = np.zeros(16 + 3, dtype=np.uint64)
    mass = np.zeros(_lib.MAX_BINS + 1, dtype=np.uint64)
    for S, B in ((0, 4), (-3, 4), (10, 0), (10, -1), (10, _lib.MAX_BINS + 1)):
        assert _lib.lib.lrb_spectrum_bin_mass(_p(spec), 16, S, B, _p(mass)) == _lib.LRB_EINVAL, (S, B)
    assert _lib.lib.lrb_spectrum_bin_mass(None, 16, 10, 4, _p(mass)) == _lib.LRB_EINVAL


def test_spectrum_text_is_jellyfish_histo_layout(tmp_path):
    M = 8
    spec = np.zeros(M + 3, dtype=np.uint64)
    spec[[0, 1, 3, 7]] = [1 << 29, 5, 2 ** 40, 1]
    spec[M + 2] = 7
    path = str(tmp_path / "histo")
    assert _lib.lib.lrb_write_spectrum_txt(path.encode(), _p(spec), M) == 0
    assert open(path, "rb").read() == b"1 5\n3 1099511627776\n7 1\n"       # c = 0 and n_c = 0 lines omitted
    spec[M], spec[M + 1], spec[M + 2] = 4, 4 * 100, 100
    assert _lib.lib.lrb_write_spectrum_txt(path.encode(), _p(spec), M) == 0
    assert open(path, "rb").read() == b"1 5\n3 1099511627776\n7 1\n8 4\n"
    spec[:] = 0
    assert _lib.lib.lrb_write_spectrum_txt(path.encode(), _p(spec), M) == 0
    assert open(path, "rb").read() == b""
    assert _lib.lib.lrb_write_spectrum_txt(str(tmp_path / "no" / "such").encode(), _p(spec), M) == _lib.LRB_EIO


def test_file_level_spectrum_fails_without_a_device(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out = str(tmp_path / "histo")
    assert _lib.lib.lrb_table_spectrum(os.path.join(GOLDEN, "g03_edge.fa").encode(), out.encode(), 65536) != 0
    assert not os.path.exists(out)
