"""GPU tier (-m gpu): the CUDA path, called through the C ABI, against the oracle, the golden files
of the reference tools, and size-independent properties at BASELINE.json's full sizes.

Bar: bit-exact for every integer result (15-mer table, coverage histograms, raw composition counts)
and byte-exact for the text files; normalised values are derived from the integers by the exact %f
formatter (tests/test_host_cpu.py), so they match to the last printed digit (<= 1e-6 relative is the
stated tolerance, BASELINE.json north_star).
"""
import ctypes as C
import gzip
import os

import numpy as np
import pytest

from conftest import COV_PARAMS, GOLDEN, golden_inputs

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

from oracle import oracle  # noqa: E402
from lrbinner_b200 import _lib, runners_utils  # noqa: E402
from lrbinner_b200.profile import (COMP_WIDTH, Context, DeviceReads, PackedReads, PartitionWorkspace, dev_composition,  # noqa: E402
                                   dev_count, dev_format_composition, dev_format_coverage, dev_mirror, dev_search,
                                   dev_table15_partitioned, _ptr)
from lrbinner_b200.synth import CONFIGS, SynthSpec, write_fasta  # noqa: E402

DEV = "cuda:0"


def _gz(path):
    with gzip.open(path, "rb") as f:
        return f.read()


@pytest.fixture(scope="module")
def ctx():
    c = Context(0)
    yield c
    c.close()


def _oracle_profile(seqs, k_list, cov_params):
    table = oracle.Table()
    for s in seqs:
        table.count(s)
    comp = {k: np.stack([oracle.composition(s, k)[0] for s in seqs]).astype(np.uint32) if seqs else np.zeros((0, COMP_WIDTH[k]), np.uint32)
            for k in k_list}
    cov = {}
    for bs, bc in cov_params:
        rows = [table.coverage(s, bs, bc) for s in seqs]
        if rows:
            cov[(bs, bc)] = (np.stack([r[0] for r in rows]).astype(np.uint32), np.array([r[1] for r in rows], dtype=np.uint32))
        else:
            cov[(bs, bc)] = (np.zeros((0, bc), np.uint32), np.zeros(0, np.uint32))
    return comp, table, cov


def _assert_table_equal(got, want):
    nz = np.flatnonzero(want)
    assert np.array_equal(np.flatnonzero(got), nz)
    assert np.array_equal(got[nz], want[nz])


# ---- golden files of the reference tools, through the file-level drop-ins -------------------------------------

@pytest.mark.parametrize("name", golden_inputs())
def test_dropin_text_files_byte_identical(name, tmp_path, ctx):
    stem = name.split(".")[0]
    src = os.path.join(GOLDEN, name)
    out = str(tmp_path)
    for k in (3, 4, 5):
        runners_utils.run_kmers(src, out, k, 4)
        assert open(f"{out}/profiles/com_profs", "rb").read() == _gz(os.path.join(GOLDEN, f"{stem}.com_k{k}.txt.gz")), (name, k)
    # buffer-level table (the 4 GiB file path is exercised once below) + every coverage parameter pair
    pr = PackedReads.from_file(src, threads=2)
    gold = np.load(os.path.join(GOLDEN, f"{stem}.table.npz"))
    res = ctx.profile(pr, bin_size=COV_PARAMS[0][0], bins=COV_PARAMS[0][1], want_table=True)
    keys = gold["keys"].astype(np.int64)
    assert np.array_equal(np.flatnonzero(res["table"]), keys) and np.array_equal(res["table"][keys], gold["counts"])
    for bs, bc in COV_PARAMS:
        r = ctx.profile(pr, bin_size=bs, bins=bc, use_loaded_table=True)
        path = f"{out}/cov"
        assert _lib.lib.lrb_write_coverage_txt(path.encode(), _ptr(r["hist"]), _ptr(r["sums"]), pr.n_reads, bc, 2) == 0
        assert open(path, "rb").read() == _gz(os.path.join(GOLDEN, f"{stem}.cov_bs{bs}_bc{bc}.txt.gz")), (name, bs, bc)


def test_dropin_three_stage_sequence_and_fused(tmp_path):
    """run_kmers -> run_15mer_counts -> run_15mer_vecs exactly as pipelines.py:269-306 calls them,
    then the fused run_profile; both must leave the reference tools' bytes on disk."""
    import hashlib
    src = os.path.join(GOLDEN, "g06_community.fa")
    out = str(tmp_path / "o1")
    runners_utils.run_kmers(src, out, 3, 4)
    runners_utils.run_15mer_counts(src, out, 4)
    runners_utils.run_15mer_vecs(src, out, 32, 10, 4)
    gold = np.load(os.path.join(GOLDEN, "g06_community.table.npz"))
    tfile = f"{out}/profiles/15mers-counts"
    assert os.path.getsize(tfile) == int(gold["file_bytes"]) == 8 + 4 * 2 ** 30
    h = hashlib.sha256()
    with open(tfile, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    assert h.hexdigest() == str(gold["sha256"])          # the whole 4 GiB file, bit for bit
    assert open(f"{out}/profiles/com_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.com_k3.txt.gz"))
    assert open(f"{out}/profiles/cov_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.cov_bs32_bc10.txt.gz"))
    # resume-style: only stage 2_1 re-run with other -bs/-bc from the stored table
    runners_utils.run_15mer_vecs(src, out, 10, 8, 4)
    assert open(f"{out}/profiles/cov_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.cov_bs10_bc8.txt.gz"))
    os.remove(tfile)
    out2 = str(tmp_path / "o2")
    runners_utils.run_profile(src, out2, 5, 10, 32, 4, write_table=False, write_npy=True)
    assert open(f"{out2}/profiles/com_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.com_k5.txt.gz"))
    assert open(f"{out2}/profiles/cov_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.cov_bs10_bc32.txt.gz"))
    want = np.array([np.array(list(map(float, line.strip().split()))) for line in open(f"{out2}/profiles/cov_profs") if len(line.strip()) > 0])
    assert np.array_equal(np.load(f"{out2}/profiles/cov_profs.npy"), want)


def test_contigs_mode_seam_counts_on_reads_profiles_fragments(tmp_path):
    """Contigs mode (pipelines.py:139-175): stage 2_4 counts the 15-mers of the READS, stages 3_1 / 4_1 run count-kmers and
    search-15mers on {output}/fragments/contigs.fasta against that table.  Golden bytes: the reference tools run the same
    way by tests/golden/make_golden.py (reads g06_community.fa, fragments g10_fragments.fasta)."""
    reads = os.path.join(GOLDEN, "g06_community.fa")
    frags = os.path.join(GOLDEN, "g10_fragments.fasta")
    out = str(tmp_path)
    runners_utils.run_15mer_counts(reads, out, 4)                       # stage 2_4
    for k in (3, 4, 5):
        runners_utils.run_kmers(frags, out, k, 4)                       # stage 3_1
        assert open(f"{out}/profiles/com_profs", "rb").read() == _gz(os.path.join(GOLDEN, f"g10_contigs_mode.com_k{k}.txt.gz")), k
    for bs, bc in COV_PARAMS:
        runners_utils.run_15mer_vecs(frags, out, bs, bc, 4)             # stage 4_1
        assert open(f"{out}/profiles/cov_profs", "rb").read() == _gz(os.path.join(GOLDEN, f"g10_contigs_mode.cov_bs{bs}_bc{bc}.txt.gz")), (bs, bc)
    # the same through one context: table of the reads kept in HBM, fragments searched against it
    c = Context(0)
    c.profile(PackedReads.from_file(reads, threads=2), keep_table=True)
    fr = PackedReads.from_file(frags, threads=2)
    r = c.profile(fr, bin_size=10, bins=8, use_loaded_table=True)
    path = f"{out}/cov2"
    assert _lib.lib.lrb_write_coverage_txt(path.encode(), _ptr(r["hist"]), _ptr(r["sums"]), fr.n_reads, 8, 2) == 0
    assert open(path, "rb").read() == _gz(os.path.join(GOLDEN, "g10_contigs_mode.cov_bs10_bc8.txt.gz"))
    c.close()
    os.remove(f"{out}/profiles/15mers-counts")


def _env(**kw):
    import contextlib

    @contextlib.contextmanager
    def cm():
        old = {k: os.environ.get(k) for k in kw}
        os.environ.update({k: str(v) for k, v in kw.items()})
        try:
            yield
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    return cm()


@pytest.mark.parametrize("batch_bases", [4000, 20000])
def test_streamed_batches_equal_the_resident_run(tmp_path, batch_bases):
    """Bounded device memory (count-15mers.cpp:75-99 streams reads through a bounded queue): when the working set does not
    fit, lrb_profile_host runs in batches — table accumulated over the batches, every batch shipped again for the search.
    LRB_BATCH_BASES forces that on a small input; the files must be the reference tools' bytes all the same."""
    src = os.path.join(GOLDEN, "g06_community.fa")
    out = str(tmp_path)
    with _env(LRB_BATCH_BASES=batch_bases):
        runners_utils.run_profile(src, out, 4, 10, 8, 4, write_table=False)
        assert open(f"{out}/profiles/com_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.com_k4.txt.gz"))
        assert open(f"{out}/profiles/cov_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.cov_bs10_bc8.txt.gz"))
        # buffer level: synthetic reads with N / lowercase / edge lengths against the oracle, table included
        spec = SynthSpec(1500, seed=8, n_rate=2e-3, lowercase_frac=0.03, edge_lengths=True, scale=0.004)
        seqs = spec.host_sequences()
        pr = spec.host_packed(threads=4)
        c = Context(0)
        res = c.profile(pr, k=3, bin_size=2, bins=6, want_table=True)
        info = c.info()
        assert info["n_batches"] > 1 and info["n_devices"] == 1 and info["lists_reused"] == 0
        for path in ("direct",):
            with _env(LRB_TABLE_PATH=path):
                res_d = c.profile(pr, k=3, bin_size=2, bins=6, want_table=True)
                assert c.info()["table_path"] == 0 and c.info()["n_batches"] > 1
            for kk in ("comp", "hist", "sums", "table"):
                assert np.array_equal(res[kk], res_d[kk]), kk
        c.close()
    comp, table, cov = _oracle_profile(seqs, [3], [(2, 6)])
    _assert_table_equal(res["table"], table.array)
    assert np.array_equal(res["comp"], comp[3])
    assert np.array_equal(res["hist"], cov[(2, 6)][0]) and np.array_equal(res["sums"], cov[(2, 6)][1])
    table.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (gpurun --gpus 2)")
@pytest.mark.parametrize("n_gpus", [2, 3, 4, 8])
def test_multi_gpu_context_leaves_the_same_bytes(tmp_path, n_gpus):
    """N GPUs through the boundary (lrb_ctx_create_multi / run_profile(n_gpus=)): reads sharded over the devices, private
    tables summed over peer memory, every device searches its own reads.  Row i must still be read i
    (search-15mers.cpp:26-48) and the files the reference tools' bytes — resident and streamed, 2 consecutive calls."""
    if torch.cuda.device_count() < n_gpus:
        pytest.skip(f"{n_gpus} GPUs not available")
    import hashlib
    src = os.path.join(GOLDEN, "g06_community.fa")
    with _env(LRB_MIN_BLOCKS_PER_DEVICE=1):
        for rep, extra in enumerate(({}, {"LRB_BATCH_BASES": 9000}, {"LRB_XCHG_COPY3D": 1})):
            out = str(tmp_path / f"o{rep}")
            with _env(**extra):
                runners_utils.run_profile(src, out, 3, 32, 10, 4, write_table=(rep == 0 and n_gpus == 2), n_gpus=n_gpus)
            assert open(f"{out}/profiles/com_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.com_k3.txt.gz"))
            assert open(f"{out}/profiles/cov_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g06_community.cov_bs32_bc10.txt.gz"))
            if rep == 0 and n_gpus == 2:
                gold = np.load(os.path.join(GOLDEN, "g06_community.table.npz"))
                h = hashlib.sha256()
                with open(f"{out}/profiles/15mers-counts", "rb") as f:
                    for blk in iter(lambda: f.read(1 << 24), b""):
                        h.update(blk)
                assert h.hexdigest() == str(gold["sha256"])
                os.remove(f"{out}/profiles/15mers-counts")
        # the three separate runners with LRB_GPUS (contigs mode: table of the reads, fragments searched on N GPUs)
        out = str(tmp_path / "sep")
        with _env(LRB_GPUS=n_gpus):
            runners_utils.run_15mer_counts(src, out, 4)
            frags = os.path.join(GOLDEN, "g10_fragments.fasta")
            runners_utils.run_kmers(frags, out, 5, 4)
            runners_utils.run_15mer_vecs(frags, out, 1, 5, 4)
        assert open(f"{out}/profiles/com_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g10_contigs_mode.com_k5.txt.gz"))
        assert open(f"{out}/profiles/cov_profs", "rb").read() == _gz(os.path.join(GOLDEN, "g10_contigs_mode.cov_bs1_bc5.txt.gz"))
        os.remove(f"{out}/profiles/15mers-counts")
    # a 20k-read synthetic set (both tables well filled, every bin hit) against the single-GPU run and the oracle's rows
    spec = SynthSpec(20000, seed=77, n_rate=1e-4, lowercase_frac=0.001, edge_lengths=True, scale=0.02)
    pr = spec.host_packed(threads=8)
    one, many = Context(0), Context(list(range(n_gpus)))
    a = one.profile(pr, k=4, bin_size=8, bins=12, want_table=True)
    for step in range(2):        # twice: the second call re-zeroes tables the peers pulled from in the first
        b = many.profile(pr, k=4, bin_size=8, bins=12, want_table=True)
        info = many.info()
        assert info["n_devices"] == n_gpus and info["n_batches"] == n_gpus and info["lists_reused"] == 1
        for kk in ("comp", "hist", "sums", "table"):
            assert np.array_equal(a[kk], b[kk]), (kk, step)
    seqs = spec.host_sequences()
    table = oracle.Table()
    for s in seqs:
        table.count(s)
    for i in list(range(0, 20000, 397)) + [19999]:
        hraw, hsum, _ = table.coverage(seqs[i], 8, 12)
        assert np.array_equal(b["hist"][i], hraw.astype(np.uint32)) and b["sums"][i] == hsum, i
        assert np.array_equal(b["comp"][i], oracle.composition(seqs[i], 4)[0].astype(np.uint32)), i
    table.close()
    one.close()
    many.close()


def test_missing_input_gives_empty_outputs_like_the_tools(tmp_path):
    out = str(tmp_path)
    runners_utils.run_kmers(str(tmp_path / "nope.fa"), out, 3, 2)
    assert os.path.getsize(f"{out}/profiles/com_profs") == 0
    with pytest.raises(SystemExit):
        runners_utils.run_15mer_vecs(str(tmp_path / "nope.fa"), out, 32, 10, 2)   # no table file -> check_proc -> sys.exit


def test_bad_parameters_are_errors(ctx):
    pr = PackedReads.from_sequences([b"ACGT" * 20])
    for kw in (dict(k=6), dict(bin_size=0, bins=10), dict(bin_size=10, bins=0), dict(bin_size=10, bins=5000)):
        with pytest.raises((_lib.LrbError, KeyError)):
            ctx.profile(pr, **kw)


# ---- seeded synthetic reads vs the oracle ---------------------------------------------------------------

@pytest.mark.parametrize("seed,n,lengths,kw", [
    (1, 1500, "gamma5k", dict(n_rate=1e-3, lowercase_frac=0.01, edge_lengths=True)),
    (2, 400, "longtail", dict(n_rate=1e-4, edge_lengths=True)),
    (3, 600, "hifi15k", dict(errors="hifi")),
])
def test_synthetic_reads_bit_exact_vs_oracle(ctx, seed, n, lengths, kw):
    spec = SynthSpec(n, lengths=lengths, seed=seed, scale=0.02, **kw)
    seqs = spec.host_sequences()
    pr = spec.host_packed(threads=4)
    cov_params = [(32, 10), (10, 32), (3, 7)]
    comp, table, cov = _oracle_profile(seqs, (3, 4, 5), cov_params)
    first = True
    for k in (3, 4, 5):
        bs, bc = cov_params[0]
        res = ctx.profile(pr, k=k, bin_size=bs, bins=bc, want_table=first)
        assert np.array_equal(res["comp"], comp[k]), k
        assert np.array_equal(res["hist"], cov[(bs, bc)][0]) and np.array_equal(res["sums"], cov[(bs, bc)][1])
        if first:
            _assert_table_equal(res["table"], table.array)
        first = False
    for bs, bc in cov_params[1:]:
        res = ctx.profile(pr, bin_size=bs, bins=bc, use_loaded_table=True)
        assert np.array_equal(res["hist"], cov[(bs, bc)][0]) and np.array_equal(res["sums"], cov[(bs, bc)][1]), (bs, bc)
    table.close()


def test_empty_and_tiny_read_sets(ctx):
    for seqs in ([], [b""], [b"", b"A", b"AC"], [b"ACGTACGTACGTAC"], [b"ACGTACGTACGTACG"], [b"N" * 100], [b"acgt" * 30]):
        pr = PackedReads.from_sequences(seqs)
        res = ctx.profile(pr, k=3, bin_size=10, bins=8, want_table=True)
        comp, table, cov = _oracle_profile(seqs, (3,), [(10, 8)])
        assert np.array_equal(res["comp"], comp[3])
        assert np.array_equal(res["hist"].reshape(-1), cov[(10, 8)][0].reshape(-1)) and np.array_equal(res["sums"], cov[(10, 8)][1])
        _assert_table_equal(res["table"], table.array)
        table.close()


def test_u32_wraparound_is_modular(ctx):
    """No saturation in the reference (kmer_utils.h:139-153: +1 mod 2^32): preload a table near the top."""
    seqs = [b"ACGTTGCAAGGCTTACGATC" * 5] * 3
    pr = PackedReads.from_sequences(seqs)
    dr = DeviceReads(pr, DEV)
    table = torch.full((2 ** 30,), -2, dtype=torch.int32, device=DEV)   # 0xFFFFFFFE everywhere
    dev_count(dr, table)
    torch.cuda.synchronize()
    want = oracle.Table()
    for s in seqs:
        want.count(s)
    keys = np.flatnonzero(want.array)
    canon = keys[(keys & 0x8000) == 0]
    got = table[torch.from_numpy(canon.astype(np.int64)).to(DEV)].cpu().numpy().view(np.uint32)
    assert np.array_equal(got, (want.array[canon].astype(np.uint64) + 0xFFFFFFFE).astype(np.uint64) % (1 << 32))
    want.close()


# ---- device-level pieces -------------------------------------------------------------------------------

def test_device_synth_and_pack_match_host():
    spec = SynthSpec(3000, seed=9, n_rate=1e-3, lowercase_frac=0.02, edge_lengths=True, scale=0.02)
    host = spec.host_packed(threads=4)
    dr, layout = spec.device_reads(DEV)
    assert np.array_equal(dr.codes.cpu().numpy().view(np.uint32)[:2 * host.n_blocks + 2], host.codes)
    assert np.array_equal(dr.valid.cpu().numpy().view(np.uint32)[:host.n_blocks + 1], host.valid)
    # device packer (ASCII in HBM -> packed) against the host packer
    bases, offsets = spec.host_ascii()
    d2 = DeviceReads(layout, DEV, upload=False)
    db = torch.from_numpy(bases).to(DEV)
    do = torch.from_numpy(offsets.view(np.int64)).to(DEV)
    _lib.check(_lib.lib.lrb_dev_pack_ascii(C.byref(d2.view), C.c_void_p(db.data_ptr()), C.c_void_p(do.data_ptr()),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert np.array_equal(d2.codes.cpu().numpy().view(np.uint32)[:2 * host.n_blocks + 2], host.codes)
    assert np.array_equal(d2.valid.cpu().numpy().view(np.uint32)[:host.n_blocks + 1], host.valid)


def test_device_validity_rebuild_from_exceptions(ctx):
    """lrb_dev_fill_valid (read lengths + sparse exceptions) reproduces the host bitmap; the host path that ships
    exceptions instead of the bitmap gives the same profiles as the one that ships the bitmap."""
    from lrbinner_b200.profile import dev_fill_valid
    spec = SynthSpec(2000, seed=13, n_rate=3e-4, lowercase_frac=0.005, edge_lengths=True, scale=0.02)
    pr = spec.host_packed(threads=4)
    blk, word = pr.exceptions()
    assert 0 < len(blk) < pr.n_blocks // 16
    dr = DeviceReads(pr, DEV)
    dr.valid.fill_(0x5A5A5A5A)
    dev_fill_valid(dr, torch.from_numpy(blk.view(np.int32)).to(DEV), torch.from_numpy(word.view(np.int32)).to(DEV))
    assert np.array_equal(dr.valid.cpu().numpy().view(np.uint32)[:pr.n_blocks + 1], pr.valid)
    res_exc = ctx.profile(pr, k=4, bin_size=32, bins=10, want_table=False)
    os.environ["LRB_SHIP_VALID"] = "1"
    try:
        res_map = ctx.profile(pr, k=4, bin_size=32, bins=10, want_table=False)
    finally:
        del os.environ["LRB_SHIP_VALID"]
    for key in ("comp", "hist", "sums"):
        assert np.array_equal(res_exc[key], res_map[key]), key
    assert int(res_exc["sums"].sum()) > 0


def test_device_handoff_to_the_autoencoder_equals_the_file_path(tmp_path, ctx):
    """SURVEY 8f-4: the float32 tensors make_data_loader (ae_utils.py:19-32) builds from the text -> float() -> .npy ->
    MinMaxScaler -> .float() chain, produced on the device from the integer profiles without touching disk."""
    from sklearn.preprocessing import MinMaxScaler
    from lrbinner_b200.handoff import profile_values, vae_inputs
    spec = SynthSpec(1200, seed=17, n_rate=5e-4, lowercase_frac=0.01, edge_lengths=True, scale=0.03)
    pr = spec.host_packed(threads=4)
    k, bs, bc = 4, 32, 10
    res = ctx.profile(pr, k=k, bin_size=bs, bins=bc)
    com, cov = str(tmp_path / "com_profs"), str(tmp_path / "cov_profs")
    rl = np.array(pr.read_len, copy=True)
    assert _lib.lib.lrb_write_composition_txt(com.encode(), _ptr(res["comp"]), _ptr(rl), pr.n_reads, k, 2) == 0
    assert _lib.lib.lrb_write_coverage_txt(cov.encode(), _ptr(res["hist"]), _ptr(res["sums"]), pr.n_reads, bc, 2) == 0
    # the reference's chain (pipelines.py:315-321, ae_utils.py:21-25), literally
    comp_ref = np.array([np.array(list(map(float, line.strip().split()))) for line in open(com) if len(line.strip()) > 0])
    cov_ref = np.array([np.array(list(map(float, line.strip().split()))) for line in open(cov) if len(line.strip()) > 0])
    profs_ref = torch.from_numpy(MinMaxScaler().fit_transform(comp_ref)).float()
    covs_ref = torch.from_numpy(MinMaxScaler().fit_transform(cov_ref)).float()
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(DEV)
    comp_d, len_d, hist_d, sums_d = dev(res["comp"]), dev(rl), dev(res["hist"]), dev(res["sums"])
    assert np.array_equal(profile_values(comp_d, len_d, k).cpu().numpy(), comp_ref)
    assert np.array_equal(profile_values(hist_d, sums_d, 0).cpu().numpy(), cov_ref)
    covs, profs = vae_inputs(comp_d, len_d, hist_d, sums_d, k)
    assert covs.is_cuda and profs.dtype == torch.float32
    assert torch.equal(covs.cpu(), covs_ref) and torch.equal(profs.cpu(), profs_ref)


def test_device_text_epilogue_matches_host_writer(tmp_path, ctx):
    spec = SynthSpec(700, seed=4, n_rate=1e-3, edge_lengths=True, scale=0.02)
    pr = spec.host_packed()
    n = pr.n_reads
    for k, (bs, bc) in ((3, (32, 10)), (4, (10, 32)), (5, (1, 5))):
        res = ctx.profile(pr, k=k, bin_size=bs, bins=bc)
        P = COMP_WIDTH[k]
        rl = np.array(pr.read_len)
        path = str(tmp_path / "t")
        assert _lib.lib.lrb_write_composition_txt(path.encode(), _ptr(res["comp"]), _ptr(rl), n, k, 2) == 0
        text = torch.zeros(n * (9 * P + 1), dtype=torch.uint8, device=DEV)
        dev_format_composition(torch.from_numpy(res["comp"].view(np.int32)).to(DEV), torch.from_numpy(rl.view(np.int32)).to(DEV), n, k, text)
        assert text.cpu().numpy().tobytes() == open(path, "rb").read()
        assert _lib.lib.lrb_write_coverage_txt(path.encode(), _ptr(res["hist"]), _ptr(res["sums"]), n, bc, 2) == 0
        text = torch.zeros(n * 9 * bc, dtype=torch.uint8, device=DEV)
        dev_format_coverage(torch.from_numpy(res["hist"].view(np.int32)).to(DEV), torch.from_numpy(res["sums"].view(np.int32)).to(DEV), n, bc, text)
        assert text.cpu().numpy().tobytes() == open(path, "rb").read()


def test_key_sharded_count_and_search_sum_to_whole():
    """The multi-GPU decomposition on one device: 4 key shards counted separately and partial histograms
    summed (plan A), and read-sharded search on the merged table (plan B), both equal the single pass."""
    spec = SynthSpec(4000, seed=12, n_rate=1e-4, edge_lengths=True, scale=0.05)
    pr = spec.host_packed()
    dr = DeviceReads(pr, DEV)
    n, bs, bc = pr.n_reads, 32, 10
    whole = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, whole)
    parts = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    bounds = [0, 2 ** 28, 2 ** 29, 3 * 2 ** 28, 2 ** 30]
    hist_a = torch.zeros((n, bc), dtype=torch.int32, device=DEV)
    sums_a = torch.zeros(n, dtype=torch.int32, device=DEV)
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        dev_count(dr, parts, key_lo=lo, key_hi=hi)
        dev_search(dr, parts, bs, bc, hist_a, sums_a, key_lo=lo, key_hi=hi)      # plan A: partial histograms accumulate
    assert torch.equal(whole, parts)
    dev_mirror(whole)
    hist_w = torch.zeros((n, bc), dtype=torch.int32, device=DEV)
    sums_w = torch.zeros(n, dtype=torch.int32, device=DEV)
    dev_search(dr, whole, bs, bc, hist_w, sums_w)
    assert torch.equal(hist_w, hist_a) and torch.equal(sums_w, sums_a)
    # plan B: read shards (tile ranges) against the full table
    hist_b = torch.zeros((n, bc), dtype=torch.int32, device=DEV)
    sums_b = torch.zeros(n, dtype=torch.int32, device=DEV)
    cuts = [0, n // 3, n // 2, n]
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        tlo, thi = dr.tile_range_for_reads(lo, hi)
        dev_search(dr, whole, bs, bc, hist_b, sums_b, tile_lo=tlo, tile_hi=thi)
    assert torch.equal(hist_w, hist_b) and torch.equal(sums_w, sums_b)
    # block-range sharded count (data-parallel over the stream) also sums to the whole
    parts.zero_()
    nb = pr.n_blocks
    for lo, hi in ((0, nb // 5), (nb // 5, nb // 2 + 1), (nb // 2 + 1, nb)):
        dev_count(dr, parts, blk_lo=lo, blk_hi=hi)
    dev_mirror(parts)
    assert torch.equal(whole, parts)


def test_partitioned_l2_resident_passes_equal_direct_kernels():
    """csrc/partition.cu (key-partitioned, L2-resident count + search) against the direct kernels: fused,
    count-only, search-only, key-sharded and block-range-sharded, for several bucket sizes."""
    spec = SynthSpec(6000, seed=21, n_rate=1e-3, lowercase_frac=0.01, edge_lengths=True, scale=0.05)
    pr = spec.host_packed()
    dr = DeviceReads(pr, DEV)
    n, bs, bc = pr.n_reads, 32, 10
    z = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=DEV)
    table_d, hist_d, sums_d = z(2 ** 30), z(n, bc), z(n)
    dev_count(dr, table_d)
    dev_search(dr, table_d, bs, bc, hist_d, sums_d, key_lo=0, key_hi=2 ** 29)      # canonical-key lookups on the unmirrored table
    dev_search(dr, table_d, bs, bc, hist_d, sums_d, key_lo=2 ** 29, key_hi=2 ** 30)
    ws = PartitionWorkspace(dr)
    blk = np.array(pr.read_blk)
    assert np.array_equal(ws.blk_read.cpu().numpy().view(np.uint32)[:pr.n_blocks], np.repeat(np.arange(n, dtype=np.uint32), np.diff(blk)))
    for shift in (25, 24):
        table_p, hist_p, sums_p = z(2 ** 30), z(n, bc), z(n)
        dev_table15_partitioned(dr, ws, table_p, True, bs, bc, hist_p, sums_p, log2_bucket_keys=shift)      # fused
        assert torch.equal(table_p, table_d) and torch.equal(hist_p, hist_d) and torch.equal(sums_p, sums_d), shift
    table_p = z(2 ** 30)
    dev_table15_partitioned(dr, ws, table_p, True, log2_bucket_keys=25)                                        # count only
    assert torch.equal(table_p, table_d)
    hist_p, sums_p = z(n, bc), z(n)
    dev_table15_partitioned(dr, ws, table_d, False, 3, 7, z(n, 7), z(n))                                      # search only, other params
    dev_table15_partitioned(dr, ws, table_d, False, bs, bc, hist_p, sums_p)
    assert torch.equal(hist_p, hist_d) and torch.equal(sums_p, sums_d)
    # key shards x block shards accumulate to the whole
    table_p, hist_p, sums_p = z(2 ** 30), z(n, bc), z(n)
    nb = pr.n_blocks
    for klo, khi in ((0, 2 ** 28), (2 ** 28, 2 ** 29), (2 ** 29, 2 ** 30)):
        for blo, bhi in ((0, nb // 3), (nb // 3, nb)):
            dev_table15_partitioned(dr, ws, table_p, True, blk_lo=blo, blk_hi=bhi, key_lo=klo, key_hi=khi)
    assert torch.equal(table_p, table_d)
    for klo, khi in ((0, 2 ** 28), (2 ** 28, 2 ** 29), (2 ** 29, 2 ** 30)):
        for blo, bhi in ((0, int(blk[n // 2])), (int(blk[n // 2]), nb)):
            dev_table15_partitioned(dr, ws, table_p, False, bs, bc, hist_p, sums_p, blk_lo=blo, blk_hi=bhi, key_lo=klo, key_hi=khi)
    assert torch.equal(hist_p, hist_d) and torch.equal(sums_p, sums_d)
    # small buckets on a narrow key range (what an 8-GPU key shard looks like), then the rest of the key space
    table_p, hist_p, sums_p = z(2 ** 30), z(n, bc), z(n)
    for klo, khi, shift in ((0, 2 ** 26, 20), (2 ** 26, 2 ** 27, 21), (2 ** 27, 2 ** 30, 24)):
        dev_table15_partitioned(dr, ws, table_p, True, bs, bc, hist_p, sums_p, key_lo=klo, key_hi=khi, log2_bucket_keys=shift)
    assert torch.equal(table_p, table_d) and torch.equal(hist_p, hist_d) and torch.equal(sums_p, sums_d)
    # the shared-memory (second-level) count is the default above; the L2-atomic kernel alone, and a sub-list workspace so
    # small that every bucket overflows its share and falls back, give the same table; so does accumulating on top
    for kw in (dict(smem_count=False), dict(smem_count=True)):
        table_p = z(2 ** 30)
        dev_table15_partitioned(dr, ws, table_p, True, **kw)
        assert torch.equal(table_p, table_d), kw
    # the WRITING form of the count (apply mode bit 3: no memset by the caller): a table full of garbage comes out as the
    # counts in its canonical half — through the shared-memory path, the L2-atomic path, and a per-bucket-range apply
    garbage = lambda: torch.full((2 ** 30,), -559038737, dtype=torch.int32, device=DEV)
    canon = lambda t: t.view(-1, 2, 1 << 15)[:, 0, :]
    for kw in (dict(smem_count=True), dict(smem_count=False)):
        table_p = garbage()
        ws.build(True)
        ws.apply(table_p, count=True, overwrite=True, **kw)
        assert torch.equal(canon(table_p), canon(table_d)), kw
    table_p = garbage()
    ws.build(True, log2_bucket_keys=25)
    for lo, hi in ((0, 5), (5, 6), (6, 32)):
        ws.apply(table_p, count=True, overwrite=True, bucket_lo=lo, bucket_hi=hi)
    dev_mirror(table_p)                                    # the mirror writes every entry of the other half
    table_m = table_d.clone()
    dev_mirror(table_m)
    assert torch.equal(table_p, table_m)
    # barely enough room for the second-level lists: many (bucket, sub-slice, CTA) segments overflow and their buckets fall
    # back to the L2-atomic kernel, the others go through shared memory — one table
    tiny = PartitionWorkspace(dr, sub_capacity=int(1.6 * ws.capacity) + (1 << 20))
    table_p = torch.full((2 ** 30,), 7, dtype=torch.int32, device=DEV)
    dev_table15_partitioned(dr, tiny, table_p, True)
    dev_table15_partitioned(dr, ws, table_p, True, log2_bucket_keys=25)
    assert torch.equal(table_p, 2 * table_d + 7)
    table_p = garbage()                                    # ... and the writing form zeroes the slices of the buckets that fall back
    tiny.build(True)
    tiny.apply(table_p, count=True, overwrite=True)
    assert torch.equal(canon(table_p), canon(table_d))
    del tiny
    # workspace too small is an error, not a truncation
    small = PartitionWorkspace(dr, capacity=1000)
    t_small = z(2 ** 30)
    dev_table15_partitioned(dr, small, t_small, True)
    with pytest.raises(_lib.LrbError):
        small.check()
    assert int(t_small.count_nonzero().item()) == 0          # an overflowing chunk is dropped as a whole, never half-applied
    small.build(True, grow=True)                              # grows to the size the device reported
    small.apply(t_small, count=True)
    assert torch.equal(t_small, table_d)
    # chunked adds (as the H2D pipeline does) give the same lists' effect
    table_p, hist_p, sums_p = z(2 ** 30), z(n, bc), z(n)
    ws.begin(True)
    cuts = [0, nb // 7, nb // 2, nb - 3, nb]
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        ws.add(lo, hi)
    ws.apply(table_p, True, True, bs, bc, hist_p, sums_p)
    assert ws.check() == int(sums_d.to(torch.int64).sum().item())
    assert torch.equal(table_p, table_d) and torch.equal(hist_p, hist_d) and torch.equal(sums_p, sums_d)


_META_O2 = 2 * 64 * 64 + 65 + 2      # PartMeta (csrc/partition.cu) in u64 units: counts, offsets [64][64], chunk_base[65], needed, overflow,
                                     # then overflow2 u32[64] (32 u64), spill_n, spill_dropped


def _part_meta(ws):
    m = ws.small.cpu().numpy()
    o2 = m[_META_O2:_META_O2 + 32].view(np.uint32)[:ws.part.n_buckets].astype(bool)
    return int(o2.sum()), int(m[_META_O2 + 32]), int(m[_META_O2 + 33])   # buckets fallen back, spilled entries, spill area overflowed


def test_second_level_count_survives_key_skew():
    """Low-complexity reads (tandem repeats, homopolymers) pile thousands of windows of one 8192-entry tile into a single
    2^15-key sub-slice: k2_partition's fixed staging rows overflow into its per-tile overflow list, beyond that (or when a
    list segment is full) the entries go to the spill area and are applied by k_count_spill; only when the spill area
    fills up does a bucket fall back to k_count_keys.  Whatever the mix of paths, one table."""
    rng = np.random.default_rng(77)
    spec = SynthSpec(2500, seed=31, scale=0.05)
    seqs = spec.host_sequences()
    for _ in range(30):                                    # tandem repeats of a random unit of 6..9 bases, 2-6 kb
        unit = bytes(rng.choice(list(b"ACGT"), size=int(rng.integers(6, 10))).tolist())
        seqs.append((unit * 1200)[:int(rng.integers(2000, 6000))])
    seqs += [b"A" * 6000] * 40 + [b"T" * 5000] * 10        # homopolymers: one key, far beyond any staging row or overflow list
    order = rng.permutation(len(seqs))
    seqs = [seqs[i] for i in order]
    pr = PackedReads.from_sequences(seqs)
    dr = DeviceReads(pr, DEV)
    z = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=DEV)
    table_d = z(2 ** 30)
    dev_count(dr, table_d)
    # roomy list segments, so that a repeat read's ~1000 windows of one key overflow only the per-tile staging row
    ws = PartitionWorkspace(dr, sub_capacity=40 * pr.n_blocks * 32)
    fell_back, spilled = {}, {}
    for shift in (24, 25, 22):
        table_p = z(2 ** 30)
        if shift == 22:                                    # 64 buckets of 2^22 keys cover a quarter of the key space at a time
            for q in range(4):
                dev_table15_partitioned(dr, ws, table_p, True, key_lo=q * 2 ** 28, key_hi=(q + 1) * 2 ** 28, log2_bucket_keys=22)
        else:
            dev_table15_partitioned(dr, ws, table_p, True, log2_bucket_keys=shift)
            fell_back[shift], spilled[shift], dropped = _part_meta(ws)
            assert not dropped
        assert torch.equal(table_p, table_d), shift
        if shift != 22:                                    # the same mix of paths, writing instead of adding
            table_w = torch.full((2 ** 30,), 123456789, dtype=torch.int32, device=DEV)
            ws.build(True, log2_bucket_keys=shift)
            ws.apply(table_w, count=True, overwrite=True)
            assert torch.equal(table_w.view(-1, 2, 1 << 15)[:, 0, :], table_d.view(-1, 2, 1 << 15)[:, 0, :]), shift
            del table_w
    # the homopolymers (290 000 windows of one key) cannot fit any list segment: they went through the spill area, and no
    # bucket had to fall back
    assert fell_back[24] == 0 and fell_back[25] == 0, fell_back
    assert spilled[24] > 150000 and spilled[25] > 150000, spilled
    # a read set DOMINATED by one key overflows the spill area (1/8 of the list capacity): its bucket falls back to the
    # (aggregating) L2-atomic kernel, the other buckets still go through shared memory; adding and writing forms
    seqs2 = seqs[:600] + [b"A" * 6000] * 400
    pr2 = PackedReads.from_sequences(seqs2)
    dr2 = DeviceReads(pr2, DEV)
    table_d2 = z(2 ** 30)
    dev_count(dr2, table_d2)
    ws2 = PartitionWorkspace(dr2)
    table_p = z(2 ** 30)
    dev_table15_partitioned(dr2, ws2, table_p, True)
    fb, sp, dropped = _part_meta(ws2)
    # (once the area is full every later spill — the tandem repeats scatter hot keys over most buckets — flags its bucket)
    assert dropped and fb >= 1, (fb, sp, dropped)
    assert torch.equal(table_p, table_d2)
    table_w = torch.full((2 ** 30,), 987654321, dtype=torch.int32, device=DEV)
    ws2.build(True)
    ws2.apply(table_w, count=True, overwrite=True)
    assert torch.equal(table_w.view(-1, 2, 1 << 15)[:, 0, :], table_d2.view(-1, 2, 1 << 15)[:, 0, :])


def test_segment_capacities_follow_the_key_distribution():
    """An AT-rich genome (20 % GC) puts ~6x the mean into the AT-rich (bucket, sub-slice) cells and next to nothing into
    the GC-rich ones.  k_sample_cells / k_plan_cells size the second-level segments from a sample of the windows, so the
    whole set still goes through the shared-memory count: no bucket falls back, only a sliver passes the spill area."""
    rng = np.random.default_rng(5)
    genome = rng.choice(np.frombuffer(b"ACTG", dtype=np.uint8), size=8_000_000, p=[0.4, 0.1, 0.4, 0.1])
    comp = np.zeros(256, dtype=np.uint8)
    comp[list(b"ACGT")] = list(b"TGCA")
    seqs = []
    for _ in range(40000):
        L = int(rng.integers(2000, 8000))
        st = int(rng.integers(0, len(genome) - L))
        r = genome[st:st + L]
        seqs.append((comp[r[::-1]] if rng.random() < 0.5 else r).tobytes())
    pr = PackedReads.from_sequences(seqs, threads=8)
    dr = DeviceReads(pr, DEV)
    table_d = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, table_d)
    ws = PartitionWorkspace(dr)
    for shift in (24, 25):
        table_p = torch.full((2 ** 30,), 31337, dtype=torch.int32, device=DEV)
        ws.build(True, log2_bucket_keys=shift)
        ws.apply(table_p, count=True, overwrite=True)
        fb, spilled, dropped = _part_meta(ws)
        assert torch.equal(table_p.view(-1, 2, 1 << 15)[:, 0, :], table_d.view(-1, 2, 1 << 15)[:, 0, :]), shift
        assert fb == 0 and not dropped and spilled < 0.02 * pr.total_bases, (shift, fb, spilled, dropped)
    # the cell capacities really differ: AT-rich cells got several times the capacity of GC-rich ones
    # cell table (csrc/partition.cu, L2Layout): uint2 {offset in octets, capacity} per cell, rows permuted inside a bucket
    nsub = 1 << (ws.part.shift - 16)
    ncell = ws.part.n_buckets * nsub
    words = ws.sub.view(torch.int32)[ws.part.l2_cells0 // 2: ws.part.l2_cells0 // 2 + 2 * ncell].cpu().numpy().view(np.uint32)
    sub = np.arange(nsub)
    pos = (sub & 15) * (nsub >> 4) + (sub >> 4)
    slot = (np.arange(ws.part.n_buckets)[:, None] * nsub + pos[None, :]).reshape(-1)        # natural (bucket, sub) order -> table slot
    off, cap = words[0::2][slot].astype(np.int64), words[1::2][slot].astype(np.int64)
    assert cap.max() >= 4 * max(int(np.median(cap)), 1) and cap.min() >= 8, (cap.min(), np.median(cap), cap.max())
    assert np.array_equal(np.diff(off), (cap * ws.part.l2_ncta // 8)[:-1]) and (off[-1] + cap[-1] * ws.part.l2_ncta // 8) * 8 <= ws.part.l2_span


def test_multi_gpu_exchange_building_blocks_on_one_device():
    """The pieces of dist.PeerExchange on one GPU: two read shards counted into two private tables ("ranks"), the peer's
    canonical rows pulled piece by piece with lrb_dev_copy2d into a staging plane, added with lrb_dev_add_planes, and every
    piece's buckets searched right after its sum (lrb_dev_partition_apply_range) — equals one count + one search over
    all reads."""
    spec = SynthSpec(5000, seed=41, n_rate=1e-4, edge_lengths=True, scale=0.05)
    pr = spec.host_packed()
    dr = DeviceReads(pr, DEV)
    n, bs, bc = pr.n_reads, 32, 10
    z = lambda *shape: torch.zeros(shape, dtype=torch.int32, device=DEV)
    whole, hist_w, sums_w = z(2 ** 30), z(n, bc), z(n)
    ws = PartitionWorkspace(dr)
    dev_table15_partitioned(dr, ws, whole, True, bs, bc, hist_w, sums_w)
    blk = np.array(pr.read_blk)
    cut = n // 2
    mine, peer = z(2 ** 30), z(2 ** 30)
    dev_table15_partitioned(dr, ws, peer, True, blk_lo=int(blk[cut]), blk_hi=pr.n_blocks)        # the peer's shard
    ws.build(True, 0, int(blk[cut]))                                                             # my shard: count ...
    ws.apply(mine, count=True)
    rows, cols = 2 ** 14, 2 ** 15                                                                # canonical rows: pitch 2^16 entries
    piece = rows // 16
    stage = torch.full((1, piece, cols), -1, dtype=torch.int32, device=DEV)
    hist_p, sums_p = z(n, bc), z(n)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nb = ws.part.n_buckets
    for g in range(16):                                                                          # ... then exchange + search piece by piece
        r0 = g * piece
        _lib.check(_lib.lib.lrb_dev_copy2d(C.c_void_p(stage.data_ptr()), 4 * cols, C.c_void_p(peer.data_ptr() + r0 * 8 * cols), 8 * cols,
                                           4 * cols, piece, st))
        _lib.check(_lib.lib.lrb_dev_add_planes(C.c_void_p(mine.data_ptr() + r0 * 8 * cols), 2 * cols, C.c_void_p(stage.data_ptr()),
                                               piece * cols, 1, cols, piece, st))
        ws.apply(mine, count=False, search=True, bin_size=bs, bins=bc, hist=hist_p, sums=sums_p,
                 bucket_lo=g * nb // 16, bucket_hi=(g + 1) * nb // 16)
    assert torch.equal(mine, whole)                                                              # canonical half summed, other half still zero
    # my shard's rows are complete (the peer's reads were not in my partition): rows of reads < cut match the full search
    assert torch.equal(hist_p[:cut], hist_w[:cut]) and torch.equal(sums_p[:cut], sums_w[:cut])
    assert int(hist_p[cut:].sum().item()) == 0
    # several planes at once (N - 1 = 3 peers), odd row count
    acc = torch.arange(5 * 2 * cols, dtype=torch.int32, device=DEV).reshape(5, 2, cols).contiguous()
    planes = torch.randint(0, 2 ** 31 - 1, (3, 8, cols), dtype=torch.int32, device=DEV)          # plane stride = 8 rows, 5 used
    want = acc.clone()
    want[:, 0, :] += planes[:, :5].sum(dim=0, dtype=torch.int32)
    _lib.check(_lib.lib.lrb_dev_add_planes(C.c_void_p(acc.data_ptr()), 2 * cols, C.c_void_p(planes.data_ptr()), 8 * cols, 3, cols, 5, st))
    assert torch.equal(acc, want)


# ---- full-size properties (BASELINE.json configs) ---------------------------------------------------------

def _full_size_properties(name, subsample=200):
    torch.cuda.empty_cache()          # config #3 needs ~95 GB: start from what earlier tests have really released
    cfg = CONFIGS[name]
    spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
    dr, layout = spec.device_reads(DEV)
    n, k, bs, bc = spec.n_reads, cfg["k"], 32, 10
    P = COMP_WIDTH[k]
    lens = torch.from_numpy(spec.lengths.astype(np.int64)).to(DEV)
    comp = torch.zeros((n, P), dtype=torch.int32, device=DEV)
    dev_composition(dr, k, comp)
    assert torch.equal(comp.sum(dim=1, dtype=torch.int64), (lens - k + 1).clamp(min=0))       # every window counted once
    table = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    dev_count(dr, table)
    nwin = (lens - 14).clamp(min=0)                                                            # all-ACGT reads
    half = int((table.view(torch.int32).to(torch.int64) & 0xFFFFFFFF).sum().item())
    assert half == int(nwin.sum().item())                                                      # one increment per window (canonical half)
    dev_mirror(table)
    total = 0
    for lo in range(0, 2 ** 30, 2 ** 28):
        total += int((table[lo:lo + 2 ** 28].to(torch.int64) & 0xFFFFFFFF).sum().item())
    assert total == 2 * half                                                                   # table sum = 2 x valid windows (SURVEY 4)
    # T[x] == T[rc(x)]: mirroring again is a no-op (idempotence)
    chk = int(table[::4099].to(torch.int64).sum().item())
    dev_mirror(table)
    assert chk == int(table[::4099].to(torch.int64).sum().item())
    hist = torch.zeros((n, bc), dtype=torch.int32, device=DEV)
    sums = torch.zeros(n, dtype=torch.int32, device=DEV)
    dev_search(dr, table, bs, bc, hist, sums)
    assert torch.equal(sums.to(torch.int64), nwin) and torch.equal(hist.sum(dim=1, dtype=torch.int64), nwin)
    # the L2-resident (partitioned) passes give the same table and histograms at full size
    ws = PartitionWorkspace(dr)
    table_p = torch.zeros(2 ** 30, dtype=torch.int32, device=DEV)
    hist_p = torch.zeros((n, bc), dtype=torch.int32, device=DEV)
    sums_p = torch.zeros(n, dtype=torch.int32, device=DEV)
    dev_table15_partitioned(dr, ws, table_p, True, bs, bc, hist_p, sums_p)
    dev_mirror(table_p)
    assert torch.equal(table_p, table) and torch.equal(hist_p, hist) and torch.equal(sums_p, sums)
    del ws, table_p, hist_p, sums_p
    # spot-check reads against the oracle restricted to the sampled reads' own k-mers:
    # composition needs only the read; coverage needs global counts, looked up from the device table
    rng = np.random.default_rng(1)
    pick = np.sort(rng.choice(n, size=subsample, replace=False))
    dr.download_into(layout)
    comp_h = comp[torch.from_numpy(pick).to(DEV)].cpu().numpy().view(np.uint32)
    hist_h = hist[torch.from_numpy(pick).to(DEV)].cpu().numpy().view(np.uint32)
    for row, i in enumerate(pick):
        s = layout.unpack(int(i))
        assert np.array_equal(comp_h[row], oracle.composition(s, k)[0].astype(np.uint32)), i
        # coverage needs GLOBAL counts: take this read's window keys from the oracle's rolling code, look their
        # counts up in the device table (itself checked above by mass / symmetry and, at small sizes, bit for
        # bit against the oracle) and apply the oracle's bucket rule
        keys = oracle.window_keys(s)
        dev_counts = table[torch.from_numpy(keys.astype(np.int64)).to(DEV)].cpu().numpy().view(np.uint32)
        want = np.zeros(bc, dtype=np.uint64)
        for c in dev_counts:
            want[oracle.bucket(int(c), bs, bc)] += 1
        assert np.array_equal(want, hist_h[row].astype(np.uint64)), i
    del table, comp, hist


def test_config1_full_size_all_three_files_against_stored_digests():
    """BASELINE.json config #1 in full (100 k reads, 0.5 Gbases, -k 3 -bs 32 -bc 10): the drop-ins on the config's FASTA
    leave com_profs, cov_profs and the whole 4 GiB 15mers-counts with the size and sha256 stored in
    tests/golden/cfg1_100k_5kb_k3.files.json — fused call and the three separate calls.  make_golden.py --config1 writes
    those digests with the unmodified reference tools, or with --oracle-drivers with the oracle's file drivers, which
    tests/test_oracle_pins.py pins to the tools' files; `source` says which wrote them."""
    import hashlib
    import json
    import shutil
    import tempfile
    cfg = CONFIGS["cfg1_100k_5kb_k3"]
    with open(os.path.join(GOLDEN, "cfg1_100k_5kb_k3.files.json")) as f:
        gold = json.load(f)
    assert gold["source"] in ("reference tools (oracle/_ref)", "oracle file drivers (oracle/lrb_oracle.c)"), gold["source"]
    assert (gold["k"], gold["bin_size"], gold["bins"]) == (cfg["k"], 32, 10)
    want = gold["files"]
    assert want["com_profs"]["bytes"] == cfg["n_reads"] * (32 * 9 + 1) and want["cov_profs"]["bytes"] == cfg["n_reads"] * 90
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 12 * 2 ** 30 else None
    work = tempfile.mkdtemp(prefix="lrb_cfg1_", dir=base)
    try:
        spec = SynthSpec(cfg["n_reads"], lengths=cfg["lengths"], errors=cfg["errors"], seed=cfg["seed"])
        fasta = os.path.join(work, "cfg1.fa")
        write_fasta(fasta, spec.host_sequences())
        threads = os.cpu_count() or 8

        def digest(path):
            h = hashlib.sha256()
            with open(path, "rb") as f:
                for blk in iter(lambda: f.read(1 << 24), b""):
                    h.update(blk)
            return {"bytes": os.path.getsize(path), "sha256": h.hexdigest()}

        assert digest(fasta) == want["reads.fa"]                 # the input the golden digests were taken of
        out = os.path.join(work, "fused")
        runners_utils.run_profile(fasta, out, cfg["k"], 32, 10, threads, write_table=True)
        for name in ("com_profs", "cov_profs", "15mers-counts"):
            assert digest(f"{out}/profiles/{name}") == want[name], ("fused", name, gold["source"])
        shutil.rmtree(out)
        out = os.path.join(work, "three")
        runners_utils.run_kmers(fasta, out, cfg["k"], threads)
        runners_utils.run_15mer_counts(fasta, out, threads)
        runners_utils.run_15mer_vecs(fasta, out, 32, 10, threads)
        for name in ("com_profs", "cov_profs", "15mers-counts"):
            assert digest(f"{out}/profiles/{name}") == want[name], ("three calls", name, gold["source"])
    finally:
        shutil.rmtree(work, ignore_errors=True)


def test_full_size_properties_config1():
    _full_size_properties("cfg1_100k_5kb_k3")


def test_full_size_properties_config2_headline():
    _full_size_properties("cfg2_1M_5kb_ont_k4", subsample=100)


def test_full_size_properties_config3_10gbp():
    _full_size_properties("cfg3_2M_5kb_k3", subsample=40)


def test_full_size_properties_config4_hifi_k5():
    _full_size_properties("cfg4_500k_15kb_hifi_k5", subsample=40)


def test_full_size_properties_config5_longtail():
    _full_size_properties("cfg5_longtail_k3", subsample=40)
