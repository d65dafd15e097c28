"""GPU tier (-m gpu): the second-level partition (k2_partition) copies each staging row into its list segment as an
entry-wise head and whole 16-byte words, from a staging ring aligned with the destination.  Every case counts the same
reads through the second-level lists and with the direct kernel (dev_count) and compares the tables key for key:
rows of every length and destination offset modulo 8 (many partial tiles, fills carried over many chunks), rows that
wrap around the ring, rows that overflow into the per-tile overflow list, full segments that go to the spill area, the
uniform-capacity plan of a small input, and 128 / 256 / 512 sub-slices per bucket."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

from lrbinner_b200.profile import DeviceReads, PackedReads, PartitionWorkspace, dev_count  # noqa: E402
from lrbinner_b200.synth import SynthSpec  # noqa: E402

DEV = "cuda:0"
_META_O2 = 2 * 64 * 64 + 65 + 2     # PartMeta (csrc/partition.cu) in u64 units: ..., overflow2 u32[64] (32 u64), spill_n, spill_dropped


def _zeros(n):
    return torch.zeros(n, dtype=torch.int32, device=DEV)


def _meta(ws):
    """(buckets fallen back to the L2-atomic count, entries through the spill area, spill area overflowed)"""
    m = ws.small.cpu().numpy()
    o2 = m[_META_O2:_META_O2 + 32].view(np.uint32)[:ws.part.n_buckets].astype(bool)
    return int(o2.sum()), int(m[_META_O2 + 32]), int(m[_META_O2 + 33])


def _fills(ws):
    """segment fill counters of every (CTA, cell) of the last partition"""
    n = ws.part.l2_ncta * ws.part.n_buckets * (1 << (ws.part.shift - 16))
    return ws.sub[:2 * n].view(torch.int32).cpu().numpy()


def _count_partitioned(ws, n_blocks, cuts, log2_bucket_keys=24, key_ranges=((0, 2 ** 30),)):
    """the table counted through the second-level lists, each key range built in the chunks `cuts` (block bounds)"""
    table = _zeros(2 ** 30)
    for lo_k, hi_k in key_ranges:
        ws.begin(True, key_lo=lo_k, key_hi=hi_k, log2_bucket_keys=log2_bucket_keys)
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            ws.add(lo, hi)
        assert ws.part.l2_enabled
        ws.apply(table, count=True)
        ws.check()
    return table


def _reads(seqs):
    pr = PackedReads.from_sequences(seqs)
    dr = DeviceReads(pr, DEV)
    direct = _zeros(2 ** 30)
    dev_count(dr, direct)
    return pr, dr, direct


@pytest.fixture(scope="module")
def mixed():
    spec = SynthSpec(6000, seed=41, scale=0.05)
    return _reads(spec.host_sequences())


@pytest.mark.parametrize("log2_bucket_keys", [23, 24, 25])
def test_many_chunks_every_offset(mixed, log2_bucket_keys):
    """40 chunks: every chunk's bucket regions end in partial tiles, and the segment fills carry over from chunk to chunk,
    so rows start at every offset modulo 8 and have every length modulo 8; about a quarter of the rows wrap the ring."""
    pr, dr, direct = mixed
    nb = pr.n_blocks
    cuts = sorted(set([0, nb] + list(np.linspace(0, nb, 41).astype(int))))
    ws = PartitionWorkspace(dr)
    # 2^23-key buckets: 128 of them cover the key space, so it is counted in two halves of 64 buckets
    ranges = ((0, 2 ** 29), (2 ** 29, 2 ** 30)) if log2_bucket_keys == 23 else ((0, 2 ** 30),)
    table = _count_partitioned(ws, nb, cuts, log2_bucket_keys, ranges)
    fb, spilled, dropped = _meta(ws)
    assert fb == 0 and not dropped, (fb, spilled, dropped)
    fills = _fills(ws)
    assert set(np.unique(fills[fills > 0] % 8)) == set(range(8))
    assert torch.equal(table, direct)


def test_overflow_list_rows():
    """Tandem repeats of a 5..7-base unit put a few hundred windows of a handful of keys into one tile: their rows pass
    the ring's capacity and the rest goes through the per-tile overflow list, appended after the row's whole words
    (roomy segments and short repeats, so that these rows are listed rather than spilled)."""
    rng = np.random.default_rng(5)
    seqs = SynthSpec(1500, seed=43, scale=0.05).host_sequences()
    for _ in range(60):
        unit = bytes(rng.choice(list(b"ACGT"), size=int(rng.integers(5, 8))).tolist())
        seqs.append((unit * 400)[:int(rng.integers(800, 1400))])
    seqs = [seqs[i] for i in rng.permutation(len(seqs))]
    pr, dr, direct = _reads(seqs)
    ws = PartitionWorkspace(dr, sub_capacity=40 * pr.n_blocks * 32)
    table = _count_partitioned(ws, pr.n_blocks, [0, pr.n_blocks // 3, pr.n_blocks])
    fb, spilled, dropped = _meta(ws)
    assert fb == 0 and not dropped, (fb, spilled, dropped)
    assert torch.equal(table, direct)


def test_full_segments_spill(mixed):
    """Little room for the lists: many segments fill, and the rows that find theirs full go to the spill area (read
    back from the ring at the row's own rotation); the spill area holds them all, so every bucket is still counted from
    its segments plus the spill area.  (With less room the plan falls back to one capacity and the spill area overflows.)"""
    pr, dr, direct = mixed
    ws = PartitionWorkspace(dr, sub_capacity=int(2.4 * pr.n_blocks * 32) + (1 << 20))
    table = _count_partitioned(ws, pr.n_blocks, [0, pr.n_blocks // 2, pr.n_blocks])
    fb, spilled, dropped = _meta(ws)
    assert fb == 0 and spilled > 10000 and not dropped, (fb, spilled, dropped)
    assert torch.equal(table, direct)


@pytest.mark.parametrize("log2_bucket_keys", [24, 25])
def test_uniform_plan_small_input(log2_bucket_keys):
    """Too few windows for a sampled plan: every cell gets the same capacity, so the rows of a CTA's first tile (all
    fills zero) start at offsets that differ only by multiples of that capacity."""
    pr, dr, direct = _reads(SynthSpec(120, seed=47, scale=0.01).host_sequences())
    ws = PartitionWorkspace(dr)
    cuts = sorted(set([0, pr.n_blocks // 4, pr.n_blocks // 2, pr.n_blocks]))
    table = _count_partitioned(ws, pr.n_blocks, cuts, log2_bucket_keys)
    assert torch.equal(table, direct)
