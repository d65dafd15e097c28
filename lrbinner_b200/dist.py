"""Multi-GPU profile stage: one process per GPU, torch.distributed (NCCL over NVLink) for the exchanges.

Reads are independent for composition; the 15-mer table is a commutative u32 sum; the search is a gather
against the finished table (SURVEY.md section 8e).  Three decompositions are implemented and timed
(bench.py keeps the fastest on measured numbers, as BASELINE.json's north star asks):

  plan "keyshard_rs" (A)  key space split by the high bits of the 30-bit key: rank g owns
        T[g*2^30/G, (g+1)*2^30/G).  COUNT: every rank scans all reads and increments only its own keys —
        no communication.  SEARCH: every rank buckets only the windows whose key it owns into partial
        u32[N,B] histograms (+ partial sums[N]); reduce-scatter(sum) leaves each rank the final rows of its
        own N/G reads.
  plan "keyshard_ag" (B)  COUNT as in A, then all-gather of the table slices (4 GiB in total), local
        mirror, read-sharded SEARCH with no further communication.
  plan "readshard_ar" (X) every rank counts only ITS reads into a private full table; all-reduce(sum) of the
        canonical half of the tables (2 GiB: count touches only the bit-15-clear member of {x, rc x}); local mirror;
        read-sharded SEARCH.  No rank needs another rank's reads.

        The exchange is PIPELINED with the search: the table is summed slice by slice (one slice = one bucket of the
        key partition, 32 MiB of canonical entries) on a side stream, and the main stream searches slice i as soon as
        it has arrived while slices i+1.. are still on NVLink — the search of a slice reads only that slice.

u32 sums are associative mod 2^32, so every plan is bit-exact whatever the reduction order.
Composition is read-sharded in all plans.  Each rank returns the rows of its own reads
[own_lo, own_hi) = equal contiguous chunks of ceil(N/G) reads.

The engine argument does the per-GPU work.  The product engine is CudaEngine (lrb_dev_* kernels); the
CPU tests inject an oracle-backed engine to check the sharding / collective logic over gloo.
"""
import os

import numpy as np

TABLE_ENTRIES = 1 << 30
PLANS = ("keyshard_rs", "keyshard_ag", "readshard_ar")


def chunk_size(n, world):
    return (n + world - 1) // world


def own_range(n, world, rank):
    c = chunk_size(n, world)
    return min(n, rank * c), min(n, (rank + 1) * c)


def key_range(world, rank, entries=TABLE_ENTRIES):
    return rank * entries // world, (rank + 1) * entries // world


class CudaEngine:
    """Per-GPU work through the C ABI kernels on torch CUDA tensors (the product path).

    Table passes go through the key-partitioned, L2-resident kernels (csrc/partition.cu): count() builds the
    partition of the requested (reads x keys) rectangle and applies it; search() re-uses that partition when it
    covers the same rectangle (plans A and X: count -> exchange -> search on the same lists), else builds its own."""

    def __init__(self, device_reads, workspace_entries=None, log2_bucket_keys=24):
        import torch
        from . import profile
        self.torch, self.p, self.dr = torch, profile, device_reads
        self.n_reads = device_reads.n_reads
        self.device = device_reads.device
        self.table_entries = TABLE_ENTRIES          # 4^15 (count-15mers.cpp:99)
        self.canon_bit = 15                         # count() touches only keys with this bit clear; mirror() fills the rest
        self.shift = log2_bucket_keys
        self._rb = None
        self.ws = profile.PartitionWorkspace(device_reads, capacity=workspace_entries)
        self._rect = None
        self._verified = set()
        self.can_overwrite = True                   # count(..., overwrite=True) writes the table slices: no table.zero_() needed

    def zeros(self, shape):
        return self.torch.zeros(shape, dtype=self.torch.int32, device=self.device)

    def zeros_rows(self, shape, lo, hi):
        """A tensor indexed by GLOBAL read of which only rows [lo, hi) will be written and returned: only those are zeroed
        (at N = 8 the composition rows of the whole global set are 4.4 GB — 0.7 ms of memset per step for rows no kernel
        touches; the row sums of foreign reads are computed from uninitialised rows and never looked at)."""
        t = self.torch.empty(shape, dtype=self.torch.int32, device=self.device)
        t[lo:hi].zero_()
        return t

    def _blocks(self, lo, hi):
        if self._rb is None:
            self._rb = self.dr.read_blk.cpu().numpy().view(np.uint32)
        return int(self._rb[lo]), int(self._rb[hi])

    def _partition(self, read_lo, read_hi, key_lo, key_hi, count=True):
        rect = (read_lo, read_hi, key_lo, key_hi)
        if self._rect != rect:
            blo, bhi = self._blocks(read_lo, read_hi)
            shift = self.shift
            while (key_hi - key_lo) >> shift > 64:
                shift += 1
            self.ws.build(True, blo, bhi, key_lo, key_hi, shift, grow=rect not in self._verified, count=count)
            self._verified.add(rect)       # same reads, same rectangle -> same size: later steps stay asynchronous
            self._rect = rect

    def composition(self, k, comp, read_lo, read_hi):
        tlo, thi = self.dr.tile_range_for_reads(read_lo, read_hi)
        self.p.dev_composition(self.dr, k, comp, tlo, thi)

    def count(self, table, key_lo, key_hi, read_lo, read_hi, overwrite=False):
        self._rect = None                            # new step: the reads may have been re-uploaded
        self._partition(read_lo, read_hi, key_lo, key_hi)
        self.ws.apply(table, count=True, overwrite=overwrite)

    def count_fed(self, table, read_lo, read_hi, chunks, per_chunk, overwrite=False):
        """count() over the whole key space with the reads arriving in chunks (the e2e pipeline: the partition of chunk j
        runs while chunk j+1 is still on PCIe).  chunks = [(read_lo_j, read_hi_j), ...] covering [read_lo, read_hi);
        per_chunk(j) is called before chunk j is touched (it makes the stream wait for the chunk and may run other
        per-chunk work, e.g. the composition)."""
        rect = (read_lo, read_hi, 0, self.table_entries)
        dbg = os.environ.get("LRB_FEED_DEBUG") == "1"
        tl = []
        def stamp(name):
            if dbg:
                e = self.torch.cuda.Event(enable_timing=True)
                e.record()
                tl.append((name, e))
        stamp("begin")
        self.ws.begin(True, 0, self.table_entries, self.shift, count=True)
        for j, (rlo, rhi) in enumerate(chunks):
            per_chunk(j)
            stamp(f"c{j}")
            blo, bhi = self._blocks(rlo, rhi)
            self.ws.add(blo, bhi)
            stamp(f"a{j}")
        if rect not in self._verified:               # first time for this rectangle: verify the workspace (synchronises)
            try:
                self.ws.check()
            except self.p._lib.LrbError:             # too small: every chunk has arrived by now, redo in one piece and grow
                blo, bhi = self._blocks(read_lo, read_hi)
                self.ws.build(True, blo, bhi, 0, self.table_entries, self.shift, grow=True, count=True)
            self._verified.add(rect)
        self._rect = rect
        self.ws.apply(table, count=True, overwrite=overwrite)
        stamp("applied")
        if dbg:
            self.torch.cuda.synchronize()
            import sys
            print("[feed timeline ms] " + " ".join(f"{nm}={tl[0][1].elapsed_time(e):.1f}" for nm, e in tl) +
                  f" chunks={[(a, b, self._blocks(a, b)) for a, b in chunks][:3]}", file=sys.stderr, flush=True)

    def verify(self):
        """Synchronises and raises LrbError(LRB_ENOMEM) if the last partition did not fit the workspace (the lists are
        then incomplete and every apply was a no-op).  Later steps over a rectangle already seen skip the synchronising
        check so that steps stay asynchronous; a driver that re-uploads DIFFERENT reads into the same DeviceReads calls
        reset() first (or verify() at its next synchronisation point)."""
        return self.ws.check()

    def reset(self):
        """Forget which rectangles were verified (the reads behind the DeviceReads changed)."""
        self._verified.clear()
        self._rect = None

    def mirror(self, table):
        self.p.dev_mirror(table)

    def search(self, table, bin_size, bins, hist, sums, read_lo, read_hi, key_lo, key_hi):
        self._partition(read_lo, read_hi, key_lo, key_hi, count=False)   # re-used from count() when the rectangle is the same
        self.ws.apply(table, count=False, search=True, bin_size=bin_size, bins=bins, hist=hist, sums=sums)

    # -- slice-wise search (plan X pipelines the table exchange with it): slice i = bucket i of the partition count() built
    def n_slices(self, read_lo, read_hi):
        self._partition(read_lo, read_hi, 0, self.table_entries, count=False)
        return self.ws.part.n_buckets

    def slice_keys(self, i):
        return i << self.ws.part.shift, (i + 1) << self.ws.part.shift

    def search_slice(self, table, bin_size, bins, hist, sums, read_lo, read_hi, i, i_end=None):
        """slices [i, i_end) in one launch (default: slice i alone)"""
        self._partition(read_lo, read_hi, 0, self.table_entries, count=False)
        self.ws.apply(table, count=False, search=True, bin_size=bin_size, bins=bins, hist=hist, sums=sums, bucket_lo=i,
                      bucket_hi=i + 1 if i_end is None else i_end)


def _reduce_scatter(dist, out, inp, group):
    """out = this rank's chunk of sum over ranks of inp (gloo has no reduce_scatter: all_reduce + slice)."""
    if dist.get_backend(group) == "gloo":
        dist.all_reduce(inp, group=group)
        r = dist.get_rank(group)
        out.copy_(inp[r * out.shape[0]:(r + 1) * out.shape[0]])
    else:
        dist.reduce_scatter_tensor(out, inp, group=group)


def _all_reduce_canonical_half(dist, table, bit, group):
    """Sum over ranks of the entries count() can have touched: keys whose middle-base high bit is clear, i.e. the lower
    2^bit entries of every 2^(bit+1)-entry stretch — half the table, so half the bytes on NVLink.  The other half is
    still zero everywhere (mirror() runs after the exchange)."""
    canon = table.view(-1, 2, 1 << bit)[:, 0, :]
    buf = canon.contiguous()
    dist.all_reduce(buf, group=group)
    canon.copy_(buf)


def _exchange_and_search_pipelined(dist, engine, table, bit, group, bin_size, bins, hist_all, sums_all, lo, hi):
    """Plan X with the exchange hidden behind the search: the table is summed slice by slice (slice = one bucket of the
    key partition = a contiguous run of canonical rows) on a side stream while the main stream searches the slices that
    have already arrived — search(slice i) only reads table rows of slice i, and only canonical ones (no mirror needed).
    CPU tensors (gloo tests): the same order of operations, sequentially."""
    import torch
    n_slices = engine.n_slices(lo, hi)
    canon = table.view(-1, 2, 1 << bit)[:, 0, :]          # [entries / 2^(bit+1), 2^bit] canonical rows
    buf = canon.contiguous()
    rows = lambda i: tuple(k >> (bit + 1) for k in engine.slice_keys(i))
    if not table.is_cuda:
        for i in range(n_slices):
            r0, r1 = rows(i)
            dist.all_reduce(buf[r0:r1], group=group)
            canon[r0:r1].copy_(buf[r0:r1])
            if hi > lo:
                engine.search_slice(table, bin_size, bins, hist_all, sums_all, lo, hi, i)
        return
    main = torch.cuda.current_stream()
    comm = _side_stream(table.device)
    ready = torch.cuda.Event()
    ready.record(main)
    comm.wait_event(ready)
    group_of, ahead = 2, 2                                # slices per all-reduce call; exchanges enqueued ahead of the search
    starts = list(range(0, n_slices, group_of))
    events = []
    # the host alternates between the two streams so that the first search is enqueued as soon as two exchanges are
    for step in range(len(starts) + ahead):
        if step < len(starts):
            i0, i1 = starts[step], min(starts[step] + group_of, n_slices)
            r0, r1 = rows(i0)[0], rows(i1 - 1)[1]
            with torch.cuda.stream(comm):
                work = dist.all_reduce(buf[r0:r1], group=group, async_op=True)
                work.wait()                               # the side stream waits; the host does not
                canon[r0:r1].copy_(buf[r0:r1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(comm)
            events.append(ev)
        done = step - ahead
        if done >= 0:
            main.wait_event(events[done])
            if hi > lo:
                engine.search_slice(table, bin_size, bins, hist_all, sums_all, lo, hi, starts[done], min(starts[done] + group_of, n_slices))
    buf.record_stream(comm)


def exchange_schedule(n_slices, world, group_of=0):
    """Pieces and rounds of the peer-memory exchange.  Returns (pieces, rounds): pieces[g] = (first_slice, end_slice),
    consecutive and covering [0, n_slices); rounds[k] = [(g, owner), ...] with owner = g mod world — the piece that rank
    completes in step A of round k; in step B every rank fetches the round's other pieces from their owners.
    group_of = 0 picks the piece size that gives about 8 rounds."""
    if group_of <= 0:
        group_of = max(1, n_slices // (8 * world))
    pieces = [(s, min(s + group_of, n_slices)) for s in range(0, n_slices, group_of)]
    rounds = [[(g, g % world) for g in range(k * world, min((k + 1) * world, len(pieces)))]
              for k in range((len(pieces) + world - 1) // world)]
    return pieces, rounds


class PeerExchange:
    """Table exchange of plan X over NVLink peer memory, driven by the copy engines (no SM is taken from the search).

    Every rank's table lives in symmetric memory (torch symmetric memory: the same allocation mapped into every rank
    of the node).  A side stream moves rows of the canonical half between the tables with pitched device-to-device
    copies (lrb_dev_copy2d: the copy engines carry them through NVSwitch), orders the ranks with device-side barriers
    and adds pulled rows with lrb_dev_add_planes (see run()).  The main stream only waits for a round's event and
    searches its buckets, so the exchange runs ahead of the search and hides behind it; the mirror pass follows the
    search on the main stream.
    NCCL's all-reduce moves the same bytes with SM-resident kernels; pipelining it slice by slice hid only 2 of its
    6.4 ms at N = 2 and left 13 ms exposed at N = 8 (profiles/r01_bench_n2_*.json, r01_bench_n8_*.json)."""

    def __init__(self, device, bit=15, entries=TABLE_ENTRIES, group_of=0, group=None):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        self.torch, self.dist, self.lib, self.check = torch, dist, _lib.lib, _lib.check
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        self.bit, self.rows, self.cols, self.group_of = bit, entries >> (bit + 1), 1 << bit, group_of
        self.table = symm.empty(entries, dtype=torch.int32, device=device)       # THE table of this rank
        self.hdl = symm.rendezvous(self.table, group=self.group)
        self.peers = [(self.rank + d) % self.world for d in range(1, self.world)]  # rotated: no two ranks start on the same peer
        self.peer_table = {p: self.hdl.get_buffer(p, (entries,), torch.int32) for p in self.peers}
        self.stage = None
        # highest priority: k_add_planes / the mirror get SM slots ahead of the queued CTAs of the search they hide behind
        # (at default priority every 16 MiB add took 2.2 ms at N = 2, stretching the exchange over the whole search)
        self.comm = torch.cuda.Stream(device=device, priority=-1)

    def timings(self):
        """Of the last run(), after a synchronize: ms from "count done" to the first round's rows being final on this rank
        (what the search has to wait for) and to the last round (length of the whole exchange on the copy stream)."""
        if not getattr(self, "last_events", None):
            return None
        ready, first, last = self.last_events
        return {"first_round_ms": ready.elapsed_time(first), "whole_exchange_ms": ready.elapsed_time(last)}

    def run(self, engine, table, bin_size, bins, hist_all, sums_all, lo, hi):
        """table (== self.table) holds this rank's private canonical counts; on return it holds the global, mirrored table
        and hist_all / sums_all the coverage rows of the reads [lo, hi).

        Reduce-scatter + all-gather by hand, round by round.  The canonical rows are cut into pieces (a run of buckets);
        round k handles the pieces k N .. k N + N - 1, piece g owned by rank g mod N:
          A  the owner pulls the piece's rows out of every peer's table (their private counts) and adds them to its own;
             device barrier (all sums of the round are final);
          B  every rank pulls the other N - 1 finished pieces of the round from their owners over its own rows.
        Then the round's buckets are searched on the main stream while the side stream is rounds ahead.  Per rank
        2 (N-1)/N x 2 GiB come in over NVLink, every byte by copy engine."""
        import ctypes as C
        torch = self.torch
        assert table.data_ptr() == self.table.data_ptr(), "PeerExchange: the table must be the symmetric-memory one (self.table)"
        n_slices = engine.n_slices(lo, hi)
        W, me = self.world, self.rank
        rows = lambda i: tuple(k >> (self.bit + 1) for k in engine.slice_keys(i))
        pieces, rounds = exchange_schedule(n_slices, W, self.group_of)
        span = [(rows(a)[0], rows(b - 1)[1]) for a, b in pieces]      # canonical rows of every piece
        G, n_rounds = len(pieces), len(rounds)
        piece_rows = max(r1 - r0 for r0, r1 in span)
        n_peers = len(self.peers)
        if self.stage is None or self.stage.shape[1] < piece_rows:
            self.stage = torch.empty((n_peers, piece_rows, self.cols), dtype=torch.int32, device=table.device)
        main, comm = torch.cuda.current_stream(), self.comm
        st = C.c_void_p(comm.cuda_stream)
        row_bytes, pitch_bytes = 4 * self.cols, 8 * self.cols
        my_rows = lambda r0: C.c_void_p(table.data_ptr() + r0 * pitch_bytes)
        peer_rows = lambda p, r0: C.c_void_p(self.peer_table[p].data_ptr() + r0 * pitch_bytes)
        ready = torch.cuda.Event(enable_timing=True)
        ready.record(main)
        comm.wait_event(ready)
        events = []
        with torch.cuda.stream(comm):
            self.hdl.barrier()                                # every rank has counted
            for k in range(n_rounds):
                g = k * W + me
                if g < G:                                     # A: complete the sum of my piece of this round
                    r0, r1 = span[g]
                    for j, p in enumerate(self.peers):
                        self.check(self.lib.lrb_dev_copy2d(C.c_void_p(self.stage[j].data_ptr()), row_bytes, peer_rows(p, r0), pitch_bytes,
                                                           row_bytes, r1 - r0, st))
                    self.check(self.lib.lrb_dev_add_planes(my_rows(r0), 2 * self.cols, C.c_void_p(self.stage.data_ptr()),
                                                           piece_rows * self.cols, n_peers, self.cols, r1 - r0, st))
                self.hdl.barrier()                            # the sums of this round are final everywhere
                for p in self.peers:                          # B: the other pieces of the round, from their owners
                    g = k * W + p
                    if g < G:
                        r0, r1 = span[g]
                        self.check(self.lib.lrb_dev_copy2d(my_rows(r0), pitch_bytes, peer_rows(p, r0), pitch_bytes, row_bytes, r1 - r0, st))
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(comm)
                events.append(ev)
            self.hdl.barrier()                                # (the next step refills the tables only after everybody is here)
        for k, ev in enumerate(events):
            main.wait_event(ev)
            if hi > lo:                                       # the round's buckets are contiguous: one launch
                engine.search_slice(table, bin_size, bins, hist_all, sums_all, lo, hi, pieces[rounds[k][0][0]][0], pieces[rounds[k][-1][0]][1])
        main.wait_stream(comm)
        self.last_events = (ready, events[0], events[-1]) if events else None   # timings(): after a synchronize
        # after the search, not beside it: the mirror streams 4 GiB through L2 and evicts the search's resident table
        # slice (single GPU, profiles/r02_exp1_variants.jsonl: search 20.5 -> 26.2 ms with the mirror beside it)
        engine.mirror(table)


_SIDE = {}


def _side_stream(device):
    import torch
    key = (device.type, device.index)
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=device)
    return _SIDE[key]


def exchange_group(world, max_ctas=None):
    """A second NCCL communicator for the pipelined table exchange, limited to a few CTAs: the exchange only has to keep
    pace with the search it hides behind (2 GiB in ~23 ms), and every SM NCCL does not occupy keeps searching.
    Returns None when the backend cannot be configured (gloo, old torch): the default group is used then."""
    import torch.distributed as dist
    if max_ctas is None:   # measured at N = 2 (r01 notes in DESIGN.md): neither a CTA limit nor stream priority helps; off unless asked for
        max_ctas = int(os.environ.get("LRB_XCHG_CTAS", "0"))
    try:
        if dist.get_backend() != "nccl" or max_ctas <= 0:
            return None
        opts = dist.ProcessGroupNCCL.Options()
        # the search CTAs are persistent for a whole bucket: a high-priority NCCL stream gets its CTAs in at the next
        # kernel boundary instead of queueing behind every search kernel already launched
        opts.is_high_priority_stream = os.environ.get("LRB_XCHG_PRIO", "0") != "0"
        opts.config.max_ctas = max_ctas
        opts.config.min_ctas = 1
        return dist.new_group(ranks=list(range(world)), backend="nccl", pg_options=opts)
    except Exception:
        return None


def profile_distributed(engine, k, bin_size, bins, plan, table=None, group=None, comp_width=None, timers=None,
                        pipeline_exchange=True, xgroup=None, feed=None, on_comp=None, peer_exchange=None):
    """Runs the whole stage across the ranks of `group`.  Returns dict(comp, hist, sums, own=(lo, hi), table):
    comp/hist/sums hold the rows of this rank's own reads (row i <-> read own_lo + i)."""
    import torch.distributed as dist
    assert plan in PLANS, plan
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n = engine.n_reads
    c = chunk_size(n, world)
    lo, hi = own_range(n, world, rank)
    entries = engine.table_entries
    klo, khi = key_range(world, rank, entries)
    P = comp_width if comp_width is not None else {3: 32, 4: 136, 5: 512}[k]
    mark = timers.mark if timers else (lambda name: None)

    # composition: read-sharded, no exchange.  Rows are written at their global index; return the own slice.
    # feed (plan X only): [(read_lo_j, read_hi_j, wait_j)] — this rank's reads arrive in chunks; wait_j() orders the
    # current stream after chunk j's arrival.  Composition and the key partition then run chunk by chunk.
    fed = feed is not None and plan == "readshard_ar" and hasattr(engine, "count_fed") and hi > lo
    zeros_rows = getattr(engine, "zeros_rows", lambda shape, a, b: engine.zeros(shape))   # rows [lo, hi) zeroed, the rest unspecified
    comp_all = zeros_rows((n, P), lo, hi)
    if hi > lo and not fed:
        engine.composition(k, comp_all, lo, hi)
    comp = comp_all[lo:hi]
    mark("composition")

    # plan X on an engine whose count WRITES the table (every canonical slice, from one partition of all own windows): no
    # 4 GiB memset; the non-canonical half is written by the mirror
    ow = plan == "readshard_ar" and hi > lo and getattr(engine, "can_overwrite", False) and table is not None
    if table is None:
        table = engine.zeros((entries,))
    elif not ow:
        table.zero_()
    kw_ow = {"overwrite": True} if ow else {}
    pipelined = plan == "readshard_ar" and pipeline_exchange and hasattr(engine, "search_slice") and getattr(engine, "canon_bit", None) is not None
    if plan == "readshard_ar":
        if fed:
            def per_chunk(j):
                feed[j][2]()
                engine.composition(k, comp_all, feed[j][0], feed[j][1])
            engine.count_fed(table, lo, hi, [(a, b) for a, b, _ in feed], per_chunk, **kw_ow)
        elif hi > lo:
            engine.count(table, 0, entries, lo, hi, **kw_ow)
        mark("count")
        if on_comp is not None:      # the composition rows are final: the caller may start taking them home
            on_comp(comp)
        bit = getattr(engine, "canon_bit", None)
        if pipelined:
            hist_all = zeros_rows((n, bins), lo, hi)
            sums_all = zeros_rows((n,), lo, hi)
            if peer_exchange is not None:
                peer_exchange.run(engine, table, bin_size, bins, hist_all, sums_all, lo, hi)   # leaves the table mirrored
                mark("exchange_table+search+mirror")
                return {"comp": comp, "hist": hist_all[lo:hi], "sums": sums_all[lo:hi], "own": (lo, hi), "table": table}
            else:
                _exchange_and_search_pipelined(dist, engine, table, bit, xgroup if xgroup is not None else group, bin_size, bins,
                                               hist_all, sums_all, lo, hi)
            mark("exchange_table+search")
            engine.mirror(table)
            mark("mirror")
            return {"comp": comp, "hist": hist_all[lo:hi], "sums": sums_all[lo:hi], "own": (lo, hi), "table": table}
        if bit is not None:
            _all_reduce_canonical_half(dist, table, bit, group)  # 2 GiB u32 sum over NVLink
        else:
            dist.all_reduce(table, group=group)                  # whole table
        mark("exchange_table")
    else:
        engine.count(table, klo, khi, 0, n)                       # all reads, own keys: no communication
        mark("count")
        if plan == "keyshard_ag":
            dist.all_gather_into_tensor(table, table[klo:khi].clone(), group=group)   # 2^30/G entries per rank -> 4 GiB everywhere
            mark("exchange_table")

    if plan == "keyshard_rs":
        part_h = engine.zeros((world * c, bins))
        part_s = engine.zeros((world * c,))
        engine.search(table, bin_size, bins, part_h, part_s, 0, n, klo, khi)   # partial histograms over own keys
        mark("search")
        hist = engine.zeros((c, bins))
        sums = engine.zeros((c,))
        _reduce_scatter(dist, hist, part_h, group)
        _reduce_scatter(dist, sums, part_s, group)
        hist, sums = hist[:hi - lo], sums[:hi - lo]
        mark("exchange_hist")
    else:
        engine.mirror(table)
        mark("mirror")
        hist_all = zeros_rows((n, bins), lo, hi)
        sums_all = zeros_rows((n,), lo, hi)
        if hi > lo:
            engine.search(table, bin_size, bins, hist_all, sums_all, lo, hi, 0, entries)
        hist, sums = hist_all[lo:hi], sums_all[lo:hi]
        mark("search")
    return {"comp": comp, "hist": hist, "sums": sums, "own": (lo, hi), "table": table}


class _EventTimers:
    """CUDA-event phase timers on the current stream (the collectives are ordered against it by torch)."""

    def __init__(self, torch):
        self.torch, self.ev = torch, []
        self.mark("start")

    def mark(self, name):
        e = self.torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev.append((name, e))

    def phases_ms(self):
        out = {}
        for (_, a), (name, b) in zip(self.ev[:-1], self.ev[1:]):
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return out
