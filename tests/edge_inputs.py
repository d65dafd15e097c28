"""Inputs shared by tests/test_edges_host.py and tests/test_gpu_edges.py: table values planted at the edges of the bucket
rule, the (bin size, bin count) settings they are checked with, and a read set that fills the partition's list layout.

A list entry of the partitioned passes (csrc/partition.cu) carries the read's index relative to the first read of its
256-block step in 8 bits, and the search walk turns entries back into rows of a 16-step task; the dense read set puts 256
reads into whole steps and 4096 into a whole task, so those fields and rows are used up to their last value."""
import numpy as np

from oracle import oracle

STEP_BLOCKS = 256              # blocks of 32 slots per step of the partition
TASK_BLOCKS = 16 * STEP_BLOCKS  # a search task of the walk: 16 consecutive steps of a chunk

BIN_SIZES = [1, 2, 3, 7, 65535, 65537, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1, 2 ** 32, 2 ** 40]
BIN_COUNTS = [1, 2, 10, 1536, 1537, 4096]
SETTINGS = [(s, b) for s in BIN_SIZES for b in BIN_COUNTS]

# eight settings whose bins sum to 4096, the widest row a multi-setting search takes
SETTINGS8 = [(1, 1537), (2 ** 40, 1536), (2, 600), (2 ** 31, 200), (65537, 100), (2 ** 32 - 1, 80), (3, 33), (7, 10)]
assert sum(b for _, b in SETTINGS8) == 4096


def value_pool(rng, n_uniform=64):
    """u32 counts at the edges of the bucket rule of every setting in SETTINGS, plus the top of the u32 range and
    uniform values"""
    vals = {2 ** 31 - 1, 2 ** 31, 2 ** 31 + 1, 2 ** 32 - 2, 2 ** 32 - 1}
    for s, b in SETTINGS:
        vals.update([0, 1, 2, 3, s - 1, s, s + 1, 2 * s - 1, 2 * s, 2 * s + 1, b * s - 1, b * s, (b + 1) * s - 1, (b + 1) * s + 1])
    vals.update(rng.integers(0, 2 ** 32, size=n_uniform).tolist())
    return np.array(sorted(v for v in vals if 0 <= v < 2 ** 32), dtype=np.uint32)


def revcomp15(keys):
    """reverse complement of 30-bit 15-mer keys (A=0 C=1 T=2 G=3: the complement is XOR 2)"""
    keys = np.asarray(keys, dtype=np.uint32)
    out = np.zeros_like(keys)
    for i in range(15):
        out |= (((keys >> np.uint32(2 * i)) & np.uint32(3)) ^ np.uint32(2)) << np.uint32(2 * (14 - i))
    return out


def canonical_keys(seqs):
    """the distinct bit-15-clear keys of {x, rc(x)} over every 15-mer window of the reads"""
    fwd = np.unique(np.concatenate([oracle.window_keys(s) for s in seqs] + [np.zeros(0, np.uint32)]))
    return np.unique(np.where(fwd & 0x8000, revcomp15(fwd), fwd))


def plant(canon_keys, rng, pool):
    """a value from the pool for each bit-15-clear key"""
    return pool[rng.integers(0, len(pool), size=len(canon_keys))]


def oracle_table_from(keys, vals):
    """oracle.Table holding vals at keys (a mirrored table: both strands of every key listed)"""
    t = oracle.Table()
    t.array[keys] = vals
    return t


def oracle_coverage(table, seqs, bin_size, bins):
    """(hist u32[n, bins], sums u32[n]) of the oracle's search"""
    hist = np.zeros((len(seqs), bins), dtype=np.uint32)
    sums = np.zeros(len(seqs), dtype=np.uint32)
    for i, s in enumerate(seqs):
        raw, total, _ = table.coverage(s, bin_size, bins)
        hist[i] = raw
        sums[i] = total
    return hist, sums


def dense_lengths(seed=5):
    """~40 k read lengths: long runs of one-block reads (a run of 8200, runs of 600 starting at several offsets inside a
    step), reads of 8192 m + {-1, 0, 1, 14, 15} bases, reads that start and end on step boundaries, between them
    ordinary reads of 100-2000 bases"""
    rng = np.random.default_rng(seed)
    out = []
    blocks = [0]

    def add(n):
        out.append(int(n))
        blocks[0] += int(n) // 32 + 1

    def ordinary(n):
        for x in rng.integers(100, 2000, size=n):
            add(x)

    def one_block_run(n):                       # mostly 15..31 bases (windows), some 0..14 (none)
        short = rng.random(n) < 0.1
        for x in np.where(short, rng.integers(0, 15, size=n), rng.integers(15, 32, size=n)):
            add(x)

    def to_step_offset(off):                    # one filler read so that the next read starts at block `off` of a step
        d = (off - blocks[0]) % STEP_BLOCKS
        if d:
            add(32 * (d - 1) + int(rng.integers(0, 32)))

    ordinary(6000)
    one_block_run(8200)
    ordinary(3000)
    for off in (0, 1, 37, 128, 255):
        to_step_offset(off)
        one_block_run(600)
        ordinary(1500)
    for m in (1, 2, 3):
        for d in (-1, 0, 1, 14, 15):
            add(8192 * m + d)
        ordinary(200)
    for _ in range(40):                         # a read starting on a step boundary and ending on the next one, or two later
        to_step_offset(0)
        add(32 * STEP_BLOCKS * int(rng.integers(1, 3)) - 1 - int(rng.integers(0, 32)))
    ordinary(12000)
    return np.array(out, dtype=np.uint32)


def dense_occupancy(read_blk, seqs):
    """(reads starting in each step, reads starting in each 16-step task aligned to block 0, steps that hold 256 reads
    whose last read has a 15-mer window)"""
    first = np.asarray(read_blk[:-1], dtype=np.int64)
    nb = int(read_blk[-1])
    per_step = np.bincount(first // STEP_BLOCKS, minlength=(nb + STEP_BLOCKS - 1) // STEP_BLOCKS)
    per_task = np.bincount(first // TASK_BLOCKS)
    full = []
    for s in np.flatnonzero(per_step == STEP_BLOCKS):
        last = int(np.searchsorted(first, (s + 1) * STEP_BLOCKS)) - 1
        if len(oracle.window_keys(seqs[last])):
            full.append(int(s))
    return per_step, per_task, full
