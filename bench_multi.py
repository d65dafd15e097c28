"""N > 1 leg of bench.py (one process per GPU, launched by torch.distributed.run).

Headline record: WEAK scaling — the global read set is `world` shards of config #2 drawn from ONE community (one global
15-mer table); every plan of lrbinner_b200/dist.py is timed, the fastest kept for the K timed steps, then the same plan
end to end from pinned host buffers.  `north_star`: BASELINE.json's multi-GPU configs at their stated TOTAL size on
these N GPUs (strong scaling): #3 (2 M reads, 10 Gbp, k=3), #4 (HiFi 7.5 Gbp, k=5), #5 (1-100 kb long tail, 10 Gbp),
plans "keyshard_rs" (north-star default: no table exchange) and "readshard_ar/p2p" timed against each other.
`verify`: every plan's outputs are reduced to content digests (position-weighted sums mod 2^64 of the composition rows,
coverage rows, row sums and the canonical half of the exchanged table), all-reduced and required to be EQUAL across the
plans (they use three different collectives); the table digest must equal that of a single-GPU count of the whole
global set by the direct kernel on rank 0; and a sample of every rank's rows is checked against the oracle.
The oracle is used here only as the checker (this file is bench support, not the product package).
"""
import os
import sys

import numpy as np

from lrbinner_b200 import dist as lrb_dist
from lrbinner_b200.dist import PLANS, TABLE_ENTRIES, CudaEngine, PeerExchange, exchange_group, own_range, profile_distributed, _EventTimers

MASK64 = (1 << 64) - 1


def _weights(torch, n, seed, device):
    """odd 64-bit weights w[i] = hash(i) (int64 arithmetic wraps mod 2^64 on the device)"""
    i = torch.arange(n, dtype=torch.int64, device=device)
    x = i * -7046029254386353131 + seed          # 0x9E3779B97F4A7C15 as int64
    x = x ^ (x >> 29)
    x = x * -4658895280553007687                 # 0xBF58476D1CE4E5B9
    x = x ^ (x >> 32)
    return x | 1


def content_digest(torch, dist, res, n_cols_hist, table=None, canon_bit=15):
    """Digests of one plan's result on this rank, all-reduced: rows are weighted by their GLOBAL read index and their
    column, so a row that lands on the wrong read, a swapped column or a lost update changes the sum."""
    lo, hi = res["own"]
    dev = res["sums"].device
    wr = _weights(torch, hi - lo, 0, dev) if hi > lo else None
    out = []
    for key, seed in (("comp", 11), ("hist", 22)):
        x = res[key].to(torch.int64) & 0xFFFFFFFF
        if hi > lo:
            wr_g = _weights(torch, hi, seed, dev)[lo:hi]                      # weight of global read index
            wc = _weights(torch, x.shape[1], seed + 1, dev)
            out.append(((x * wc[None, :]).sum(dim=1) * wr_g).sum())
        else:
            out.append(torch.zeros((), dtype=torch.int64, device=dev))
    s = res["sums"].to(torch.int64) & 0xFFFFFFFF
    out.append((s * _weights(torch, hi, 33, dev)[lo:hi]).sum() if hi > lo else torch.zeros((), dtype=torch.int64, device=dev))
    d = torch.stack(out)
    dist.all_reduce(d)                                                        # int64 sum wraps mod 2^64
    digest = {"comp": int(d[0].item()) & MASK64, "hist": int(d[1].item()) & MASK64, "sums": int(d[2].item()) & MASK64}
    if table is not None:
        digest["table"] = table_digest(torch, table, canon_bit)
    return digest


def table_digest(torch, table, canon_bit=15):
    """position-weighted sum of the canonical half (keys with bit `canon_bit` clear) — what the exchange moves"""
    canon = table.view(-1, 2, 1 << canon_bit)[:, 0, :]
    rows = canon.shape[0]
    acc = torch.zeros((), dtype=torch.int64, device=table.device)
    wc = _weights(torch, 1 << canon_bit, 55, table.device)
    step = 1024
    for r0 in range(0, rows, step):
        x = canon[r0:r0 + step].to(torch.int64) & 0xFFFFFFFF
        wr = _weights(torch, min(rows, r0 + step), 44, table.device)[r0:]
        acc = acc + ((x * wc[None, :]).sum(dim=1) * wr).sum()
    return int(acc.item()) & MASK64


def oracle_spot_check(torch, res, dr, layout, table, k, bs, bc, n_pick=64, seed=5):
    """n_pick of this rank's own reads against the oracle: composition from the read alone; coverage from the oracle's
    window keys, the counts those keys have in the exchanged device table (whose digest is checked against a single-GPU
    count of the whole set) and the oracle's bucket rule.  Returns the number of mismatching reads."""
    from oracle import oracle
    lo, hi = res["own"]
    if hi <= lo:
        return 0, 0
    rng = np.random.default_rng([seed, lo])
    pick = np.sort(rng.choice(hi - lo, size=min(n_pick, hi - lo), replace=False))
    idx = torch.from_numpy(pick).to(res["sums"].device)
    comp_h = res["comp"][idx].cpu().numpy().view(np.uint32)
    hist_h = res["hist"][idx].cpu().numpy().view(np.uint32)
    sums_h = res["sums"][idx].cpu().numpy().view(np.uint32)
    bad = 0
    for row, i in enumerate(pick):
        s = layout.unpack(int(lo + i))
        ok = np.array_equal(comp_h[row], oracle.composition(s, k)[0].astype(np.uint32))
        keys = oracle.window_keys(s)
        cnt = table[torch.from_numpy(keys.astype(np.int64)).to(table.device)].cpu().numpy().view(np.uint32)
        want = np.zeros(bc, dtype=np.uint64)
        for c in cnt:
            want[oracle.bucket(int(c), bs, bc)] += 1
        ok = ok and np.array_equal(want, hist_h[row].astype(np.uint64)) and int(sums_h[row]) == len(keys)
        bad += 0 if ok else 1
    return len(pick), bad


def h2d_ceiling(torch, dist, dev, nbytes=1 << 30, reps=3):
    """Aggregate pinned host->device bandwidth of this box with all ranks copying at once (GB/s over all ranks)."""
    src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    dst.copy_(src, non_blocking=True)
    best = 0.0
    for _ in range(reps):
        dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src, non_blocking=True)
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        best = max(best, dist.get_world_size() * nbytes / float(ms.item()) / 1e6)
    del src, dst
    return best


class _Set:
    """One global read set resident on this rank + engine; `timed(plan, steps)` runs the whole stage."""

    def __init__(self, torch, dist, dev, rank, world, cfg, n_reads, px, xg, bs, bc):
        from lrbinner_b200.synth import SynthSpec
        self.torch, self.dist, self.dev, self.rank, self.world = torch, dist, dev, rank, world
        self.k, self.bs, self.bc, self.px, self.xg = cfg["k"], bs, bc, px, xg
        self.spec = SynthSpec(n_reads, lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
        # every rank materialises the whole global set in HBM (the key-sharded plans scan all reads; plan X touches only its own)
        self.dr, self.layout = self.spec.device_reads(dev)
        self.n, self.L = self.spec.n_reads, self.spec.total_bases
        self.eng = CudaEngine(self.dr, workspace_entries=int(self.L / world * 1.25) + (1 << 20))
        self.table = px.table if px is not None else torch.zeros(TABLE_ENTRIES, dtype=torch.int32, device=dev)

    def run(self, plan, timers=None, **kw):
        return profile_distributed(self.eng, self.k, self.bs, self.bc, plan.split("/")[0], table=self.table, timers=timers,
                                   pipeline_exchange=not plan.endswith("/unpipelined"), xgroup=self.xg,
                                   peer_exchange=self.px if plan.endswith("/p2p") else None, **kw)

    def timed(self, plan, steps):
        torch, dist = self.torch, self.dist
        dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        tm = None
        for _ in range(steps):
            tm = _EventTimers(torch)
            res = self.run(plan, timers=tm)
        b.record()
        dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / steps], device=self.dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), res, tm.phases_ms()

    def close(self):
        self.eng = self.dr = self.layout = None
        self.torch.cuda.empty_cache()


def _verify(S, plans, results, single_gpu_table_digest=None, spot=True):
    """digests equal across plans (+ the table against a single-GPU count), oracle spot check of the last plan's rows"""
    torch, dist = S.torch, S.dist
    digests = {p: results[p] for p in plans}
    same = all(all(digests[p][kk] == digests[plans[0]][kk] for kk in ("comp", "hist", "sums")) for p in plans)
    tabs = {p: d["table"] for p, d in digests.items() if "table" in d}
    tab_same = len(set(tabs.values())) <= 1
    out = {"plans_compared": list(plans), "digests_equal_across_plans": bool(same and tab_same),
           "digest": {kk: f"{digests[plans[0]][kk]:016x}" for kk in ("comp", "hist", "sums")}}
    if tabs:
        out["digest"]["table_canonical_half"] = f"{next(iter(tabs.values())):016x}"
    ok = same and tab_same
    if single_gpu_table_digest is not None and tabs:
        eq = single_gpu_table_digest == next(iter(tabs.values()))
        out["table_equals_single_gpu_count_of_the_global_set"] = bool(eq)
        ok = ok and eq
    return out, ok


def bench_multi_gpu(args, cfg_name, cfg, dev, rank, world, ClockSampler, hbm_peak, peak_src, metric, bs, bc, affinity=None):
    import torch
    import torch.distributed as dist
    from lrbinner_b200 import _lib
    from lrbinner_b200.profile import COMP_WIDTH, dev_count, dev_fill_valid, dev_mirror
    from lrbinner_b200.synth import CONFIGS

    k = cfg["k"]
    n_shard = args.reads or cfg["n_reads"]
    xg = exchange_group(world)
    px = None
    try:                                                  # copy-engine exchange over peer memory (needs symmetric memory on this node)
        px = PeerExchange(dev)
    except Exception as ex:
        if rank == 0:
            print(f"[lrb] peer-memory exchange unavailable ({ex!r}); NCCL exchange only", file=sys.stderr)
    ok = torch.tensor([1 if px is not None else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if not int(ok.item()):
        px = None
    S = _Set(torch, dist, dev, rank, world, cfg, n_shard * world, px, xg, bs, bc)
    n, L, eng, dr, layout, table = S.n, S.L, S.eng, S.dr, S.layout, S.table

    all_plans = PLANS + ("readshard_ar/unpipelined",) + (("readshard_ar/p2p",) if px is not None else ())
    plan_ms, digests = {}, {}
    for plan in all_plans:
        S.timed(plan, 1)                                 # warm-up (NCCL channels, allocator)
        plan_ms[plan], res, _ = S.timed(plan, max(1, args.warmup - 1))
        full_table = plan != "keyshard_rs"               # the other plans leave the whole table on every rank
        digests[plan] = content_digest(torch, dist, res, bc, table if full_table else None)
    # the table the plans exchanged against a count of the WHOLE global set on one GPU by the direct kernel (rank 0 has
    # every read resident): an independent code path, no partition, no exchange
    ref_digest = torch.zeros(1, dtype=torch.int64, device=dev)
    if rank == 0:
        t2 = torch.zeros(TABLE_ENTRIES, dtype=torch.int32, device=dev)
        dev_count(dr, t2)
        d = table_digest(torch, t2)
        ref_digest[0] = d - (1 << 64) if d >= (1 << 63) else d
        del t2
        torch.cuda.empty_cache()
    dist.broadcast(ref_digest, 0)
    verify, v_ok = _verify(S, all_plans, digests, int(ref_digest.item()) & MASK64)
    best = min(plan_ms, key=plan_ms.get)
    valid_windows = None

    sampler = ClockSampler(dev.index)
    sampler.start()
    launches0 = int(_lib.lib.lrb_prof_launches())
    _lib.lib.lrb_prof_enable(1)
    ms_step, res, phases = S.timed(best, args.steps)
    _lib.lib.lrb_prof_enable(0)
    launches = int(_lib.lib.lrb_prof_launches()) - launches0
    prof = _lib.prof_report()
    clocks = sampler.stop()
    eng.verify()                                         # the partition lists of the timed steps fitted their workspace
    exchange_t = px.timings() if (px is not None and best.endswith("/p2p")) else None   # last timed step, rank 0
    tot = torch.stack([res["sums"].to(torch.int64).sum(), res["hist"].to(torch.int64).sum()])
    dist.all_reduce(tot)
    valid_windows = int(tot[0].item())
    assert int(tot[1].item()) == valid_windows
    # oracle spot check of the kept plan's rows on every rank (rows of the timed steps themselves)
    dr.download_into(layout)
    n_chk, n_bad = oracle_spot_check(torch, res, dr, layout, table, k, bs, bc)
    chk = torch.tensor([n_chk, n_bad], device=dev)
    dist.all_reduce(chk)
    verify["oracle_spot_check"] = {"reads": int(chk[0].item()), "mismatches": int(chk[1].item()), "plan": best}
    verify["ok"] = bool(v_ok and int(chk[1].item()) == 0)
    assert verify["ok"], f"multi-GPU verification failed: {verify}"

    # ---- e2e: every step also moves this rank's inputs host->device and its result rows device->host ------------------
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h_codes = torch.from_numpy(layout.codes.view(np.int32))   # whole global set; page-locked only if the host allowed that much
    # validity crosses PCIe as the exception list only (0 entries for pure-ACGT reads); the bitmap is rebuilt on the device
    layout.index_valid(threads=os.cpu_count() or 8)
    exc_blk, exc_word = layout.exceptions()
    h_exc = [pin(torch.from_numpy(a.view(np.int32))).copy_(torch.from_numpy(a.view(np.int32))) for a in (exc_blk, exc_word)]
    d_exc = [torch.empty(len(exc_blk), dtype=torch.int32, device=dev) for _ in range(2)]
    lo, hi = own_range(n, world, rank)
    if best.startswith("readshard_ar"):   # only the own shard's blocks are needed on this rank
        rb = layout.read_blk
        b0, b1 = int(rb[lo]), int(rb[hi])
    else:
        b0, b1 = 0, layout.n_blocks
    if best.startswith("readshard_ar") and world > 1:
        # this rank ships only its own shard: give that a page-locked buffer of its own (8 ranks x the global set would
        # ask the host for more pinned memory than it grants, and the copies would silently go through pageable staging)
        own = pin(h_codes[2 * b0:2 * b1])
        own.copy_(h_codes[2 * b0:2 * b1])
        h_own, own_w0 = own, 2 * b0
    else:
        h_own, own_w0 = h_codes, 0
    out_h = {kk: pin(res[kk]) for kk in ("comp", "hist", "sums")}

    # chunk plan of this rank's blocks (cut at read boundaries) for the pipelined plan-X step
    rb = np.asarray(layout.read_blk)
    if best.startswith("readshard_ar"):
        n_ch = 16
        cr = [lo] + [max(lo, min(hi, int(np.searchsorted(rb, b0 + (b1 - b0) * j // n_ch, side="right")) - 1)) for j in range(1, n_ch)] + [hi]
        cr = sorted(set(cr))
    else:
        cr = None
    copy_in, copy_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    marks = {}
    # Two device buffers for the packed stream (LRB_E2E_BUFFERS=1: one): the host links are the bottleneck of the e2e step
    # at N >= 4 (box ceiling measured below), so the H2D of step i+1 starts the moment the H2D of step i has finished and
    # the copy stream never idles; a buffer is free again once the key partition of the step before last is built.
    n_buf = 2 if (cr is not None and len(cr) >= 2 and os.environ.get("LRB_E2E_BUFFERS", "2") != "1") else 1
    codes_bufs = [dr.codes] + [torch.empty_like(dr.codes) for _ in range(n_buf - 1)]
    free_ev, step_no = [], [0]

    def e2e_step():
        main = torch.cuda.current_stream()
        if cr is None or len(cr) < 2:          # key-sharded plans need every read on every rank before anything starts
            dr.codes[2 * b0:2 * b1].copy_(h_codes[2 * b0:2 * b1], non_blocking=True)
            for d, h in zip(d_exc, h_exc):
                d.copy_(h, non_blocking=True)
            dev_fill_valid(dr, d_exc[0] if len(exc_blk) else None, d_exc[1] if len(exc_blk) else None)
            r = S.run(best)
            for kk in out_h:
                out_h[kk].copy_(r[kk], non_blocking=True)
            return
        # plan X: H2D in chunks on a copy stream; composition + key partition of chunk j run while chunk j+1 is on PCIe;
        # the composition rows go home on a second copy stream while the table passes run
        start = torch.cuda.Event(enable_timing=True)
        start.record(main)
        marks["start"] = start
        # the packed stream is dead once the key partition of a step is built (count and search work from the lists): the
        # H2D into a buffer starts when the last step that used THAT buffer has built its partition — BESIDE the exchange +
        # search of the steps in flight, not after them
        j_step = step_no[0]
        step_no[0] += 1
        buf = codes_bufs[j_step % n_buf]
        dr.codes = buf
        dr.view.codes = buf.data_ptr()
        copy_in.wait_event(free_ev[j_step - n_buf] if j_step >= n_buf else start)
        if "valid_built" in marks:
            copy_in.wait_event(marks["valid_built"])       # the previous step has consumed the exception lists
        copy_out.wait_event(start)
        evs = []
        with torch.cuda.stream(copy_in):
            marks["h2d_begin"] = torch.cuda.Event(enable_timing=True)
            marks["h2d_begin"].record(copy_in)
            for d, h in zip(d_exc, h_exc):
                d.copy_(h, non_blocking=True)
            ev0 = torch.cuda.Event()
            ev0.record(copy_in)
            for j in range(len(cr) - 1):
                w0, w1 = 2 * int(rb[cr[j]]), 2 * int(rb[cr[j + 1]])
                dr.codes[w0:w1].copy_(h_own[w0 - own_w0:w1 - own_w0], non_blocking=True)
                ev = torch.cuda.Event(enable_timing=(j == len(cr) - 2))
                ev.record(copy_in)
                evs.append(ev)
            marks["h2d"] = evs[-1]
        main.wait_event(ev0)
        dev_fill_valid(dr, d_exc[0] if len(exc_blk) else None, d_exc[1] if len(exc_blk) else None)
        marks["valid_built"] = torch.cuda.Event()
        marks["valid_built"].record(main)
        feed = [(cr[j], cr[j + 1], (lambda j=j: main.wait_event(evs[j]))) for j in range(len(cr) - 1)]

        def comp_home(comp):
            ready = torch.cuda.Event()
            ready.record(main)                 # composition + partition + count are enqueued: nothing later reads codes / valid
            free_ev.append(ready)
            with torch.cuda.stream(copy_out):
                copy_out.wait_event(ready)
                out_h["comp"].copy_(comp, non_blocking=True)

        marks["tm"] = _EventTimers(torch)
        r = S.run(best, timers=marks["tm"], feed=feed, on_comp=comp_home)
        marks["compute"] = torch.cuda.Event(enable_timing=True)
        marks["compute"].record(main)
        for kk in ("hist", "sums"):
            out_h[kk].copy_(r[kk], non_blocking=True)
        main.wait_stream(copy_out)
        marks["end"] = torch.cuda.Event(enable_timing=True)
        marks["end"].record(main)

    e2e_step()
    dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        e2e_step()
    b.record()
    dist.barrier()
    torch.cuda.synchronize()
    e2e_ms = torch.tensor([a.elapsed_time(b) / args.steps], device=dev)
    dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_ms.item())
    e2e_phases = {kk: marks["start"].elapsed_time(marks[kk]) for kk in ("h2d", "compute", "end")} if "end" in marks else None
    if e2e_phases is not None:
        e2e_phases["phases"] = marks["tm"].phases_ms()
        e2e_phases["h2d_copy_ms"] = marks["h2d_begin"].elapsed_time(marks["h2d"])
        e2e_phases["note"] = ("h2d = when this step's last chunk landed, relative to the step's start on the compute stream (the copy starts "
                              "during earlier steps); h2d_copy_ms = first to last chunk on the copy stream")
    # rows of the e2e step are the rows of the device-resident step, bit for bit
    e2e_same = all(torch.equal(out_h[kk].to(dev), res[kk]) for kk in out_h)
    e2e_ok = torch.tensor([1 if e2e_same else 0], device=dev)
    dist.all_reduce(e2e_ok, op=dist.ReduceOp.MIN)
    verify["e2e_rows_equal_device_resident_rows"] = bool(int(e2e_ok.item()))
    verify["ok"] = bool(verify["ok"] and int(e2e_ok.item()))
    assert verify["ok"], f"multi-GPU e2e verification failed: {verify}"
    h2d = 4 * (2 * (b1 - b0)) + 8 * len(exc_blk)
    d2h = sum(int(t.numel()) * 4 for t in out_h.values())
    del out_h, h_own, h_codes
    h2d_peak = h2d_ceiling(torch, dist, dev)

    from bench import kernel_table, load_traffic
    P = COMP_WIDTH[k]
    own_V, own_L, own_n = valid_windows / world, L / world, n / world
    kernels = kernel_table(prof, args.steps, own_L, own_V, own_n, P, bc, hbm_peak, {})
    dom = max(kernels, key=lambda nm: kernels[nm]["ms_per_step"])
    dk = kernels[dom]
    per_launch = max(dk["launches_per_step"], 1.0)
    roofline = {"kernel": dom + " (rank 0, this rank's share of the reads)", "bound": "hbm", "achieved": dk["achieved_GBps"], "peak": hbm_peak,
                "unit": "GB/s", "frac": dk["frac_of_hbm"], "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dk["algorithmic_bytes"] / per_launch, "algorithmic": dk["algorithmic"],
                "launch_ms": dk["ms_per_step"] / per_launch, "launches_per_step": dk["launches_per_step"], "alt_bound": dk.get("alt_bound")}
    line = {"metric": metric, "value": L / ms_step / 1e6, "unit": "Gbases/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": f"{world} x {cfg_name} shards of one community (one global 15-mer table)", "reads": n, "bases": L,
                       "k": k, "bin_size": bs, "bins": bc, "plan": best, "plan_ms": plan_ms, "valid_15mer_windows": valid_windows,
                       "l2_policy": "inputs larger than L2"},
            "e2e": {"value": L / e2e_ms / 1e6, "unit": "Gbases/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms, "note": "per-rank bytes; max-over-ranks time; every step ships its own inputs and results; the H2D of step "
                                                   "i+1 starts when the H2D of step i is done (%d device buffer(s) for the packed stream: it is dead once "
                                                   "a step's key partition is built), i.e. it runs beside the table exchange + search of the steps in flight" % n_buf,
                    "rank0_ms_since_step_start": e2e_phases,
                    "box_h2d_ceiling_GBps_all_ranks_copying": h2d_peak,
                    "h2d_floor_ms": h2d * world / h2d_peak / 1e6 if h2d_peak else None},
            "gpu_launches": launches, "roofline": roofline, "kernels": kernels, "verify": verify,
            "phases_ms_rank0": phases, "exchange_rank0": exchange_t, "clocks": clocks, "cpu_baseline": None, "cpu_affinity": affinity}
    S.close()
    del S, eng, dr, layout, res

    # ---- north-star configs at their stated total size on these N GPUs (strong scaling) --------------------------------
    if not args.no_north_star and not args.reads:
        line["north_star"] = []
        ns_plans = ("keyshard_rs",) + (("readshard_ar/p2p",) if px is not None else ("readshard_ar",))
        for name in ("cfg3_2M_5kb_k3", "cfg4_500k_15kb_hifi_k5", "cfg5_longtail_k3"):
            c2 = CONFIGS[name]
            torch.cuda.empty_cache()
            S2 = _Set(torch, dist, dev, rank, world, c2, c2["n_reads"], px, xg, bs, bc)
            pm, dg, ph, every = {}, {}, {}, {}
            for plan in ns_plans:
                S2.timed(plan, 1)
                # --steps steps timed one by one (barrier + synchronize around each, max over ranks); the MEDIAN is reported, so a
                # single hiccup on one of the N ranks (an allocator refill, a late NCCL channel) does not decide the plan
                runs = [S2.timed(plan, 1) for _ in range(args.steps)]
                every[plan] = [round(r[0], 3) for r in runs]
                mid = sorted(range(args.steps), key=lambda i: runs[i][0])[args.steps // 2]
                pm[plan], r2, ph[plan] = runs[mid]
                dg[plan] = content_digest(torch, dist, r2, bc, S2.table if plan != "keyshard_rs" else None)
            v2, ok2 = _verify(S2, ns_plans, dg)
            b2 = min(pm, key=pm.get)
            lo2, hi2 = own_range(S2.n, world, rank)
            rbk = S2.layout.read_blk
            own_bases = torch.tensor([float(int(rbk[hi2]) - int(rbk[lo2])) * 32.0], device=dev)
            mx = own_bases.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(own_bases)
            assert ok2, f"north-star config {name}: plans disagree: {v2}"
            line["north_star"].append({
                "workload": name, "scaling": "strong", "reads": S2.n, "bases": S2.L, "k": c2["k"], "n_gpus": world,
                "plan": b2, "plan_ms": pm, "plan_ms_every_step": every, "ms_per_step": pm[b2], "value": S2.L / pm[b2] / 1e6, "unit": "Gbases/s",
                "timing": f"median of {args.steps} single steps, each bracketed by barrier + synchronize, max over ranks",
                "phases_ms_rank0": ph[b2], "plan_phases_ms_rank0": ph, "verify": v2,
                "exchange_rank0": (px.timings() if (px is not None and b2.endswith("/p2p")) else None),
                "load_imbalance_max_over_mean_slots": float(mx.item()) / (float(own_bases.item()) / world)})
            S2.close()
            del S2, r2
    return line
