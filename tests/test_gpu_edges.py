"""GPU tier (-m gpu): the search kernels and the device "%f" code at the edges the read-derived tests never reach, against
the oracle.

A. Planted counts: every bit-15-clear key the reads hit holds a count at an edge of the bucket rule (0 .. 2^32 - 1), and
   every search path bins them as oracle.Table.coverage does for bin sizes up to 2^40 and bin counts up to 4096 (both
   sides of k_search15's 48 KiB shared-memory opt-in): the direct kernel on the mirrored table and over key shards of the
   canonical half, the partitioned walk at every bucket size, several settings in one pass, compact sample tables, and a
   table loaded from a file.
B. Device "%f": k_profile_values and k_format_rows on the numerator / denominator pairs where fixed6 can go wrong.
C. Dense list layout: steps of 256 one-block reads (the 8-bit read field of a list entry full) and 16-step search tasks of
   4096 reads (hist cells up to ~2^24), through every partitioned path and a partition of 64 chunks."""
import ctypes as C
import os
import shutil

import numpy as np
import pytest

from edge_inputs import (SETTINGS, SETTINGS8, STEP_BLOCKS, TASK_BLOCKS, dense_lengths, dense_occupancy, oracle_coverage,
                         oracle_table_from, plant, value_pool)

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

from oracle import oracle  # noqa: E402
from lrbinner_b200 import _lib  # noqa: E402
from lrbinner_b200.profile import (COMP_WIDTH, Context, DeviceReads, PartitionWorkspace, dev_count, dev_format_composition,  # noqa: E402
                                   dev_format_coverage, dev_mirror, dev_search, dev_table_compact, _ptr)
from lrbinner_b200.synth import SynthSpec  # noqa: E402

DEV = "cuda:0"


def _z(*shape):
    return torch.zeros(shape, dtype=torch.int32, device=DEV)


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(DEV)


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


def _canon(t):
    """the bit-15-clear half of a full-layout table, [2^14, 2^15]"""
    return t.view(-1, 2, 1 << 15)[:, 0, :]


# ---- A. planted counts -------------------------------------------------------------------------------------------

class Planted:
    """reads, the planted table (canonical half only, and mirrored) on the device, and the oracle's search of it"""

    def __init__(self):
        spec = SynthSpec(2000, seed=71, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.02)
        self.seqs = spec.host_sequences()
        self.pr = spec.host_packed(threads=8)
        self.dr = DeviceReads(self.pr, DEV)
        self.n = self.pr.n_reads
        self.rng = np.random.default_rng(71)
        self.pool = value_pool(self.rng)
        self.canon = _z(2 ** 30)
        dev_count(self.dr, self.canon)
        self.keys = torch.nonzero(self.canon).flatten()
        self.canon.zero_()
        self.canon[self.keys] = _dev(plant(self.keys, self.rng, self.pool))
        self.full = self.canon.clone()
        dev_mirror(self.full)
        self.table = self.oracle_of(self.full)
        self.want = {}

    @staticmethod
    def oracle_of(full):
        nz = torch.nonzero(full).flatten()
        return oracle_table_from(nz.cpu().numpy(), _u32(full[nz]))

    def oracle(self, bs, bc):
        if (bs, bc) not in self.want:
            self.want[(bs, bc)] = oracle_coverage(self.table, self.seqs, bs, bc)
        return self.want[(bs, bc)]

    def check(self, hist, sums, bs, bc, what):
        want_hist, want_sums = self.oracle(bs, bc)
        got_hist = _u32(hist)
        assert np.array_equal(_u32(sums), want_sums), (what, bs, bc)
        bad = np.flatnonzero((got_hist != want_hist).any(axis=1))
        assert bad.size == 0, (what, bs, bc, bad[:5], got_hist[bad[:1]].nonzero(), want_hist[bad[:1]].nonzero())


@pytest.fixture(scope="module")
def planted():
    p = Planted()
    assert int((_u32(p.canon[p.keys]) >= 2 ** 31).sum()) > 10000
    yield p
    p.table.close()
    torch.cuda.empty_cache()


def test_direct_search_planted_counts(planted):
    """k_search15 on the mirrored table, and summed over 4 key shards of the canonical half"""
    p = planted
    bounds = [0, 2 ** 28, 2 ** 29, 3 * 2 ** 28, 2 ** 30]
    for bs, bc in SETTINGS:
        hist, sums = _z(p.n, bc), _z(p.n)
        dev_search(p.dr, p.full, bs, bc, hist, sums)
        p.check(hist, sums, bs, bc, "mirrored")
        hist.zero_(), sums.zero_()
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            dev_search(p.dr, p.canon, bs, bc, hist, sums, key_lo=lo, key_hi=hi)
        p.check(hist, sums, bs, bc, "key shards")


def _shards(shift):
    """key ranges of a whole-table partitioned pass at this bucket size: at most 64 buckets of 2^shift keys each"""
    step = min(2 ** 30, 2 ** (shift + 6))
    return [(lo, lo + step) for lo in range(0, 2 ** 30, step)]


@pytest.mark.parametrize("shift", [20, 21, 22, 23, 24, 25])
def test_partitioned_search_planted_counts(planted, shift):
    """k_search_keys at every bucket size; k_search_settings with 8 extreme settings, W = 4096"""
    p = planted
    ws = PartitionWorkspace(p.dr, sub_capacity=0)
    hists = {s: _z(p.n, s[1]) for s in SETTINGS}
    sums = {s: _z(p.n) for s in SETTINGS}
    h8, s8 = _z(p.n, 4096), _z(p.n)
    for lo, hi in _shards(shift):
        ws.build(True, key_lo=lo, key_hi=hi, log2_bucket_keys=shift, count=False)
        ws.check()
        for s in SETTINGS:
            ws.apply(p.full, count=False, search=True, bin_size=s[0], bins=s[1], hist=hists[s], sums=sums[s])
        ws.search_settings(p.canon, SETTINGS8, h8, s8)
    for s in SETTINGS:
        p.check(hists[s], sums[s], s[0], s[1], f"partitioned {shift}")
    off = 0
    for bs, bc in SETTINGS8:
        p.check(h8[:, off:off + bc], s8, bs, bc, f"settings {shift}")
        off += bc


def test_sample_tables_planted_counts(planted):
    """k_search_samples over 8 compact tables, each planted with its own values and binned with its own setting"""
    p = planted
    ws = PartitionWorkspace(p.dr, sub_capacity=0)
    ws.build(True, count=False)
    scratch = _z(2 ** 30)
    compact, wants = [], []
    for t, (bs, bc) in enumerate(SETTINGS8):
        scratch.zero_()
        scratch[p.keys] = _dev(plant(p.keys, p.rng, p.pool))
        compact.append(dev_table_compact(scratch))
        dev_mirror(scratch)
        tab = Planted.oracle_of(scratch)
        wants.append(oracle_coverage(tab, p.seqs, bs, bc))
        tab.close()
    del scratch
    hist, sums = _z(p.n, 4096), _z(p.n)
    ws.search_samples(compact, SETTINGS8, hist, sums)
    off = 0
    for (bs, bc), (want_hist, want_sums) in zip(SETTINGS8, wants):
        assert np.array_equal(_u32(hist[:, off:off + bc]), want_hist) and np.array_equal(_u32(sums), want_sums), (bs, bc)
        off += bc
    del compact
    torch.cuda.empty_cache()


def test_sample_table_reads_only_the_canonical_half(planted):
    """a sample table is its bit-15-clear half: other values in the bit-15-set half do not change the search"""
    p = planted
    t = p.canon.clone()
    t.view(-1, 2, 1 << 15)[:, 1, :] = torch.randint(-2 ** 31, 2 ** 31 - 1, (1 << 14, 1 << 15), dtype=torch.int32, device=DEV)
    compact = dev_table_compact(t)
    del t
    ws = PartitionWorkspace(p.dr, sub_capacity=0)
    for bs, bc in ((2 ** 31, 1537), (3, 4096)):
        hist, sums = _z(p.n, bc), _z(p.n)
        for lo, hi in _shards(22):
            ws.build(True, key_lo=lo, key_hi=hi, log2_bucket_keys=22, count=False)
            ws.search_samples([compact], [(bs, bc)], hist, sums)
        p.check(hist, sums, bs, bc, "canonical half")


def test_loaded_table_file_planted_counts(planted, tmp_path):
    """the planted table through a 15mers-counts file: Context.table_load, one multi-setting profile (partitioned) and
    single settings at B = 4096 through the direct kernels"""
    p = planted
    path = str(tmp_path / "15mers-counts")
    try:
        host = p.full.cpu().numpy()
        assert _lib.lib.lrb_table_write_file(path.encode(), _ptr(host)) == 0, _lib.last_error()
        del host
        ctx = Context(0)
        ctx.table_load(path)
        res = ctx.profile(p.pr, use_loaded_table=True, coverage=SETTINGS8)
        for (bs, bc), h in zip(SETTINGS8, res["hists"]):
            want_hist, want_sums = p.oracle(bs, bc)
            assert np.array_equal(h, want_hist) and np.array_equal(res["sums"], want_sums), (bs, bc)
        with _env(LRB_TABLE_PATH="direct"):
            for bs in (1, 65537, 2 ** 31, 2 ** 32 - 1, 2 ** 40):
                res = ctx.profile(p.pr, bin_size=bs, bins=4096, use_loaded_table=True)
                assert ctx.info()["table_path"] == 0
                want_hist, want_sums = p.oracle(bs, 4096)
                assert np.array_equal(res["hist"], want_hist) and np.array_equal(res["sums"], want_sums), bs
        ctx.close()
        if oracle.ref_available():      # the unmodified reference tool on counts >= 2^31, against the oracle's file
            reads = str(tmp_path / "reads.fa")
            from lrbinner_b200.synth import write_fasta
            write_fasta(reads, p.seqs)
            for bs, bc in ((2 ** 31, 10), (2 ** 32 - 1, 3), (7, 1537)):
                oracle.ref_search_15mers(path, reads, str(tmp_path / "ref.txt"), bs, bc)
                assert oracle.search_15mers_file(path, reads, str(tmp_path / "orc.txt"), bs, bc) == 0
                assert open(tmp_path / "ref.txt", "rb").read() == open(tmp_path / "orc.txt", "rb").read(), (bs, bc)
    finally:
        shutil.rmtree(tmp_path, ignore_errors=True)


# ---- B. device "%f" ----------------------------------------------------------------------------------------------

def _fixed6_pairs():
    """(num, den) pairs where the exact "%f" of num / max(den, 1) can go wrong: the list of the host test, den = 0 and
    2^32 - 1, ratios below 2^-11 (fixed6's s >= 64 branch), exact ties n / 2^7 with large denominators, and the
    neighbours of the 1e-4 cut of the coverage rows"""
    rng = np.random.default_rng(11)
    pairs = [(0, 0), (0, 5), (1, 1), (5, 5), (1, 3), (2, 3), (1, 8), (1, 16), (1, 64), (3, 64), (1, 2 ** 20), (1, 2 ** 31),
             (1, 4294967295), (4294967295, 4294967295), (1, 10000), (1, 10001), (1, 9999), (5, 49999), (5, 50000), (5, 50001),
             (1, 2000000), (3, 2000000), (1, 1000000), (15, 32), (1, 32), (9, 16)]
    dens = rng.integers(1, 200000, size=60000)
    nums = (rng.random(60000) * (dens + 1)).astype(np.int64).clip(0, dens)
    pairs += list(zip(nums.tolist(), dens.tolist()))
    big = rng.integers(1, 2 ** 32, size=20000)
    pairs += [(int(rng.integers(0, d + 1)), int(d)) for d in big]
    pairs += [(n, 2 ** s) for s in range(1, 25) for n in (1, 3, 5, 7, 2 ** s - 1) if n <= 2 ** s]
    # den = 0 and 2^32 - 1
    pairs += [(1, 0)] + [(n, 2 ** 32 - 1) for n in (0, 1, 2, 429496, 429497, 2 ** 31, 2 ** 32 - 2, 2 ** 32 - 1)]
    pairs += [(int(n), 2 ** 32 - 1) for n in rng.integers(0, 2 ** 32, size=2000)]
    # ratios in [2^-32, 2^-11): d = m 2^-s with s >= 64
    for d in rng.integers(2 ** 12, 2 ** 32, size=5000):
        pairs.append((int(max(1, int(d) * rng.uniform(2.0 ** -31, 2.0 ** -11))), int(d)))
    # exact ties: odd n / 2^7 (six decimals and a 5), with the denominator scaled up to 2^32 - 1
    for a in [1, 3, 1000, 2 ** 20, 2 ** 25 - 1] + rng.integers(1, 2 ** 25, size=300).tolist():
        for n in (1, 3, 5, 63, 127):
            pairs.append((n * int(a), 128 * int(a)))
    # the neighbours of 1e-4
    for d in [10000, 10001, 9999, 20000, 2 ** 31, 2 ** 32 - 1] + rng.integers(10000, 2 ** 32, size=3000).tolist():
        n0 = int(d) // 10000
        pairs += [(n, int(d)) for n in (n0 - 1, n0, n0 + 1, n0 + 2) if 0 <= n <= int(d)]
    return pairs


def test_device_fixed6_matches_printf():
    pairs = _fixed6_pairs()
    num = np.array([n for n, _ in pairs], dtype=np.uint32)
    den = np.array([d for _, d in pairs], dtype=np.uint32)
    n = len(pairs)
    vals = [float(a) / float(max(b, 1)) for a, b in pairs]
    cov = [0.0 if v < 1e-4 else v for v in vals]
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    # k = 0 (coverage rows): value = float of the "%f" text after the 1e-4 rule
    num_d, den_d = _dev(num), _dev(den)
    out = torch.zeros(n, dtype=torch.float64, device=DEV)
    _lib.check(_lib.lib.lrb_dev_profile_values(C.c_void_p(num_d.data_ptr()), C.c_void_p(den_d.data_ptr()), n, 1, 0,
                                               C.c_void_p(out.data_ptr()), st))
    got = out.cpu().numpy()
    want = np.array([float("%f" % v) for v in cov])
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, [(pairs[i], got[i], want[i]) for i in bad[:5]]
    text = torch.zeros(n * 9, dtype=torch.uint8, device=DEV)
    dev_format_coverage(num_d, den_d, n, 1, text)
    lines = text.cpu().numpy().tobytes().split(b"\n")[:-1]
    for i, v in enumerate(cov):
        assert lines[i] == b"%f" % v, (pairs[i], lines[i])
    # k = 3 (composition rows, total = read_len - 2): no 1e-4 rule, the pair in column 0 of a row of 32
    keep = np.flatnonzero(den <= 2 ** 32 - 3)
    m = len(keep)
    counts = np.zeros((m, COMP_WIDTH[3]), dtype=np.uint32)
    counts[:, 0] = num[keep]
    read_len = den[keep] + 2
    counts_d, len_d = _dev(counts), _dev(read_len)
    out = torch.zeros(m * COMP_WIDTH[3], dtype=torch.float64, device=DEV)
    _lib.check(_lib.lib.lrb_dev_profile_values(C.c_void_p(counts_d.data_ptr()), C.c_void_p(len_d.data_ptr()), m,
                                               COMP_WIDTH[3], 3, C.c_void_p(out.data_ptr()), st))
    got = out.cpu().numpy().reshape(m, COMP_WIDTH[3])
    want = np.array([float("%f" % vals[i]) for i in keep])
    assert not got[:, 1:].any()
    bad = np.flatnonzero(got[:, 0] != want)
    assert bad.size == 0, [(pairs[keep[i]], got[i, 0], want[i]) for i in bad[:5]]
    text = torch.zeros(m * (9 * COMP_WIDTH[3] + 1), dtype=torch.uint8, device=DEV)
    dev_format_composition(counts_d, len_d, m, 3, text)
    rows = text.cpu().numpy().tobytes().split(b"\n")[:-1]
    rest = b"0.000000 " * (COMP_WIDTH[3] - 1)
    for r, i in enumerate(keep):
        assert rows[r] == b"%f " % vals[i] + rest, (pairs[i], rows[r][:20])


# ---- C. dense list layout ----------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def dense():
    lens = dense_lengths()
    spec = SynthSpec(len(lens), lengths=lens, seed=62, n_rate=1e-3, lowercase_frac=0.01)
    seqs = spec.host_sequences()
    pr = spec.host_packed(threads=8)
    per_step, per_task, full = dense_occupancy(pr.read_blk, seqs)
    assert per_step.max() == STEP_BLOCKS and len(full) >= 6 and per_task.max() == TASK_BLOCKS, (per_step.max(), full, per_task.max())
    table = oracle.Table()
    for s in seqs:
        table.count(s)
    yield seqs, pr, table
    table.close()
    torch.cuda.empty_cache()


def test_dense_layout_profile(dense):
    """table, composition k = 3/4/5 and coverage (1, 4096) / (32, 10) through Context.profile"""
    seqs, pr, table = dense
    want = {s: oracle_coverage(table, seqs, *s) for s in ((1, 4096), (32, 10))}
    ctx = Context(0)
    for k, (bs, bc) in ((3, (1, 4096)), (4, (32, 10)), (5, (1, 4096))):
        res = ctx.profile(pr, k=k, bin_size=bs, bins=bc, want_table=(k == 3))
        assert ctx.info()["table_path"] != 0
        comp = np.stack([oracle.composition(s, k)[0] for s in seqs]).astype(np.uint32)
        assert np.array_equal(res["comp"], comp), k
        assert np.array_equal(res["hist"], want[(bs, bc)][0]) and np.array_equal(res["sums"], want[(bs, bc)][1]), (k, bs, bc)
        if k == 3:
            nz = np.flatnonzero(table.array)
            assert np.array_equal(np.flatnonzero(res["table"]), nz) and np.array_equal(res["table"][nz], table.array[nz])
    ctx.close()


def test_dense_layout_partitioned_passes(dense):
    """count (shared-memory and L2-atomic, adding and writing) and search (one setting, several settings, sample tables)
    of the partitioned passes at every bucket size, and a partition of 64 chunks"""
    seqs, pr, table = dense
    dr = DeviceReads(pr, DEV)
    n = pr.n_reads
    want_canon = _dev(np.ascontiguousarray(table.array.reshape(-1, 2, 1 << 15)[:, 0, :]))
    full = _z(2 ** 30)
    _canon(full).copy_(want_canon)
    dev_mirror(full)
    w4096 = oracle_coverage(table, seqs, 1, 4096)
    w10 = oracle_coverage(table, seqs, 32, 10)

    def check_wide(hist, sums, bc, what):          # bc <= 4096 bins of S = 1 from the 4096-bin oracle rows
        got, (wh, ws_) = _u32(hist), w4096
        assert np.array_equal(_u32(sums), ws_), what
        assert np.array_equal(got[:, :bc - 1], wh[:, :bc - 1]) and np.array_equal(got[:, bc - 1], wh[:, bc - 1:].sum(axis=1)), what

    def check10(hist, sums, what):
        assert np.array_equal(_u32(hist), w10[0]) and np.array_equal(_u32(sums), w10[1]), what

    ws = PartitionWorkspace(dr)
    for shift in (24, 25):
        for smem in (True, False):
            t = _z(2 ** 30)
            ws.build(True, log2_bucket_keys=shift)
            ws.apply(t, count=True, smem_count=smem)
            assert torch.equal(_canon(t), want_canon) and not t.view(-1, 2, 1 << 15)[:, 1, :].any(), (shift, smem)
            t.fill_(-559038737)
            ws.apply(t, count=True, overwrite=True, smem_count=smem)
            assert torch.equal(_canon(t), want_canon), (shift, smem, "writing")
            del t
    compact = dev_table_compact(full)
    for shift in (20, 21, 22, 23, 24, 25):
        h1, s1 = _z(n, 4096), _z(n)
        h10, s10 = _z(n, 10), _z(n)
        h8, s8 = _z(n, 4096), _z(n)
        hs, ss = _z(n, 4010), _z(n)
        for lo, hi in _shards(shift):
            ws.build(True, key_lo=lo, key_hi=hi, log2_bucket_keys=shift, count=False)
            ws.apply(full, count=False, search=True, bin_size=1, bins=4096, hist=h1, sums=s1)
            ws.apply(full, count=False, search=True, bin_size=32, bins=10, hist=h10, sums=s10)
            ws.search_settings(full, [(32, 10), (1, 4086)], h8, s8)
            ws.search_samples([compact, compact], [(1, 4000), (32, 10)], hs, ss)
        check_wide(h1, s1, 4096, ("search", shift))
        check10(h10, s10, ("search", shift))
        check10(h8[:, :10], s8, ("settings", shift))
        check_wide(h8[:, 10:], s8, 4086, ("settings", shift))
        check_wide(hs[:, :4000], ss, 4000, ("samples", shift))
        check10(hs[:, 4000:4010], ss, ("samples", shift))
        del h1, s1, h10, s10, h8, s8, hs, ss
    del compact
    # 64 chunks: cuts one block before, at and after step boundaries (one-block chunks among them)
    nb = pr.n_blocks
    rng = np.random.default_rng(3)
    steps = rng.choice(np.arange(1, nb // STEP_BLOCKS), size=20, replace=False)
    cuts = {0, nb}
    for s in steps:
        cuts.update([int(s) * STEP_BLOCKS - 1, int(s) * STEP_BLOCKS, int(s) * STEP_BLOCKS + 1])
    while len(cuts) < 65:
        cuts.add(int(rng.integers(1, nb)))
    cuts = sorted(cuts)
    assert len(cuts) == 65 and sum(b - a == 1 for a, b in zip(cuts[:-1], cuts[1:])) >= 40
    t, h1, s1 = _z(2 ** 30), _z(n, 4096), _z(n)
    ws.begin(True)
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        ws.add(lo, hi)
    assert ws.part.n_chunks == 64
    with pytest.raises(_lib.LrbError) as e:
        ws.add(0, 1)
    assert e.value.code == _lib.LRB_EINVAL
    ws.apply(t, count=True, search=False)
    assert torch.equal(_canon(t), want_canon)
    ws.apply(full, count=False, search=True, bin_size=1, bins=4096, hist=h1, sums=s1)
    check_wide(h1, s1, 4096, "64 chunks")
