"""Drop-in for the runner functions of mbcclr_utils/runners_utils.py (reference lines 78-113).

Same names, same arguments, same side effects: each call makes `{output}/profiles` if needed, blocks
until its file is complete, returns None, and on failure goes through check_proc -> logger.error x2
+ sys.exit(ret).  Instead of os.system() on the three C++/OpenMP executables the work is done by
liblrb200.so (CUDA, sm_100a) through ctypes:

    run_kmers        -> lrb_count_kmers     (count-kmers    <reads> <out> <k> <threads>)
    run_15mer_counts -> lrb_count_15mers    (count-15mers   <reads> <out> <threads>)
    run_15mer_vecs   -> lrb_search_15mers   (search-15mers  <table> <reads> <out> <bin_size> <bins> <threads>)

`threads` only sizes the host-side parser/packer/formatter pools; the profile arithmetic runs on the GPU.
A maintainer switches LRBinner over with one import line in mbcclr_utils/pipelines.py (INTEGRATION.md).
run_profile() is the fused fast path for stages 1_1 + 1_2 + 2_1 (parse once, table stays in HBM).
"""
import ctypes as C
import logging
import os
import sys

from . import _lib

logger = logging.getLogger('LRBinner')


def run_kmers(reads_path, output, k_size, threads):
    if not os.path.isdir(f"{output}/profiles"):
        os.makedirs(f"{output}/profiles")

    logger.debug(f"LIB::lrb_count_kmers \"{reads_path}\" \"{output}/profiles/com_profs\" {k_size} {threads}")
    o = _lib.lib.lrb_count_kmers(os.fsencode(reads_path), os.fsencode(f"{output}/profiles/com_profs"), int(k_size), int(threads))
    check_proc(o, "Counting Trimers")


def run_15mer_counts(reads_path, output, threads):
    if not os.path.isdir(f"{output}/profiles"):
        os.makedirs(f"{output}/profiles")

    logger.debug(f"LIB::lrb_count_15mers \"{reads_path}\" \"{output}/profiles/15mers-counts\" {threads}")
    o = _lib.lib.lrb_count_15mers(os.fsencode(reads_path), os.fsencode(f"{output}/profiles/15mers-counts"), int(threads))
    check_proc(o, "Counting 15-mers")


def run_15mer_vecs(reads_path, output, bin_size, bin_count, threads):
    if not os.path.isdir(f"{output}/profiles"):
        os.makedirs(f"{output}/profiles")

    logger.debug(f"LIB::lrb_search_15mers \"{output}/profiles/15mers-counts\" \"{reads_path}\" \"{output}/profiles/cov_profs\" {bin_size} {bin_count} {threads}")
    o = _lib.lib.lrb_search_15mers(os.fsencode(f"{output}/profiles/15mers-counts"), os.fsencode(reads_path),
                                   os.fsencode(f"{output}/profiles/cov_profs"), int(bin_size), int(bin_count), int(threads))
    check_proc(o, "Counting 15-mer profiles")


def run_15mer_vecs_settings(reads_path, output, settings, threads, write_npy=False):
    """Coverage profiles for several -bs / -bc settings at once: one load of {output}/profiles/15mers-counts and one parse
    of the reads (lrb_search_15mers_settings), writing {output}/profiles/cov_profs_bs{S}_bc{B} (and .npy with write_npy)
    for every (S, B) in `settings` (at most 8, no pair twice), each byte for byte the cov_profs that run_15mer_vecs
    writes for that setting.  cov_profs itself is never touched, so a checkpointed run stays consistent: copy the chosen
    file to cov_profs and resume from stage 3_1 (INTEGRATION.md).  No reference counterpart."""
    settings = [(int(s), int(b)) for s, b in settings]
    if not os.path.isdir(f"{output}/profiles"):
        os.makedirs(f"{output}/profiles")
    n = len(settings)
    outs = [os.fsencode(f"{output}/profiles/cov_profs_bs{s}_bc{b}") for s, b in settings]
    txts = (C.c_char_p * max(n, 1))(*outs)
    npys = (C.c_char_p * max(n, 1))(*[o + b".npy" for o in outs]) if write_npy else None
    bs = (C.c_long * max(n, 1))(*[s for s, _ in settings])
    bc = (C.c_int * max(n, 1))(*[b for _, b in settings])
    logger.debug(f"LIB::lrb_search_15mers_settings \"{output}/profiles/15mers-counts\" \"{reads_path}\" {settings} {threads}")
    o = _lib.lib.lrb_search_15mers_settings(os.fsencode(f"{output}/profiles/15mers-counts"), os.fsencode(reads_path), n, bs, bc,
                                            txts, npys, int(threads))
    check_proc(o, "Counting 15-mer profiles for several settings")


def run_15mer_vecs_samples(reads_path, output, table_paths, bin_size, bin_count, threads, write_npy=False):
    """Differential coverage: the reads against several 15mers-counts tables (typically other samples'
    {out}/profiles/15mers-counts) in one call (lrb_search_15mers_samples): each table is loaded once and the reads are
    parsed once.  Writes {output}/profiles/cov_profs_samples (and .npy with write_npy): per read, table 0's -bc values, then
    table 1's, ..., each block byte for byte the cov_profs line run_15mer_vecs writes against that table.  One (bin_size,
    bin_count) for every table, as LRBinner has one -bs / -bc.  cov_profs itself is never touched (INTEGRATION.md).  No
    reference counterpart."""
    if not os.path.isdir(f"{output}/profiles"):
        os.makedirs(f"{output}/profiles")
    n = len(table_paths)
    out = f"{output}/profiles/cov_profs_samples"
    paths = (C.c_char_p * max(n, 1))(*[os.fsencode(p) for p in table_paths])
    bs = (C.c_long * max(n, 1))(*[int(bin_size)] * n)
    bc = (C.c_int * max(n, 1))(*[int(bin_count)] * n)
    logger.debug(f"LIB::lrb_search_15mers_samples {list(table_paths)} \"{reads_path}\" \"{out}\" {bin_size} {bin_count} {threads}")
    o = _lib.lib.lrb_search_15mers_samples(paths, n, bs, bc, os.fsencode(reads_path), os.fsencode(out),
                                           os.fsencode(out + ".npy") if write_npy else None, int(threads))
    check_proc(o, "Counting 15-mer profiles against several samples")


def run_15mer_vecs_edges(reads_path, output, edges, threads, write_npy=False):
    """Coverage profiles with bins given by count edges (lrb_search_15mers_edges): a window whose 15-mer is counted c times
    in {output}/profiles/15mers-counts goes to bin searchsorted(edges, c, side="right"), for strictly increasing edges
    with the first >= 2 (geometric edges, or profile.spectrum_quantile_edges of the table's spectrum).  Writes
    {output}/profiles/cov_profs_edges (and .npy with write_npy), len(edges) + 1 values per read in the cov_profs format,
    and the edges as one line to cov_profs_edges.edges.  cov_profs itself is never touched: copy the file to cov_profs
    and resume from stage 3_1 (INTEGRATION.md).  No reference counterpart."""
    from .profile import _edges_array
    try:
        e = _edges_array(edges)
    except _lib.LrbError as err:   # refused like a library call: nothing written, the exit code of the refusal
        logger.error(f"Error in step: Counting 15-mer profiles by edges ({err})")
        sys.exit(err.code)
    if not os.path.isdir(f"{output}/profiles"):
        os.makedirs(f"{output}/profiles")
    out = f"{output}/profiles/cov_profs_edges"
    logger.debug(f"LIB::lrb_search_15mers_edges \"{output}/profiles/15mers-counts\" \"{reads_path}\" \"{out}\" {e.tolist()} {threads}")
    o = _lib.lib.lrb_search_15mers_edges(os.fsencode(f"{output}/profiles/15mers-counts"), os.fsencode(reads_path),
                                         e.ctypes.data_as(C.c_void_p), int(e.size), os.fsencode(out),
                                         os.fsencode(out + ".npy") if write_npy else None, int(threads))
    check_proc(o, "Counting 15-mer profiles by edges")
    with open(out + ".edges", "w") as f:
        f.write(" ".join(str(x) for x in e.tolist()) + "\n")


def layout_lines(table_paths, blocks):
    """The lines of cov_profs_layout.layout: one per block, "<table path>\tbs <S> bc <B>" or "<table path>\tedges <t1> <t2> ..."."""
    lines = []
    for b in blocks:
        how = f"bs {int(b.bin_size)} bc {int(b.bins)}" if b.edges is None else " ".join(["edges"] + [str(int(x)) for x in b.edges])
        lines.append(f"{table_paths[b.table]}\t{how}\n")
    return lines


def run_15mer_vecs_layout(reads_path, output, table_paths, blocks, threads, write_npy=False):
    """Mixed coverage rows (lrb_search_15mers_layout): up to 8 blocks (profile.CovBlock), block m reading the 15mers-counts
    file table_paths[blocks[m].table] and binned by its (bin_size, bins) or its edges, in one call: each table is loaded
    once and the reads are parsed once.  Writes {output}/profiles/cov_profs_layout (and .npy with write_npy): per read,
    block 0's values, then block 1's, ..., each block byte for byte the line the single-block runner (run_15mer_vecs,
    run_15mer_vecs_edges) writes against that table; and cov_profs_layout.layout, one line per block saying how it was
    made.  cov_profs itself is never touched (INTEGRATION.md).  No reference counterpart."""
    from .profile import _layout_blocks
    paths = [os.fspath(p) for p in table_paths]
    try:
        arr, _keep, _ = _layout_blocks(blocks)
        for m, b in enumerate(blocks):
            if b.table is None or not 0 <= int(b.table) < len(paths):
                raise _lib.LrbError(_lib.LRB_EINVAL, f"block {m} reads table {b.table}: a block here names its table by its index in "
                                                     f"[0, {len(paths)}) of table_paths")
        if not 1 <= len(paths) <= _lib.MAX_SAMPLE_TABLES:
            raise _lib.LrbError(_lib.LRB_EINVAL, f"the number of tables must be in [1, {_lib.MAX_SAMPLE_TABLES}] (got {len(paths)})")
    except _lib.LrbError as err:   # refused like a library call: nothing written, the exit code of the refusal
        logger.error(f"Error in step: Counting 15-mer profiles by layout ({err})")
        sys.exit(err.code)
    if not os.path.isdir(f"{output}/profiles"):
        os.makedirs(f"{output}/profiles")
    out = f"{output}/profiles/cov_profs_layout"
    n = len(paths)
    c_paths = (C.c_char_p * n)(*[os.fsencode(p) for p in paths])
    logger.debug(f"LIB::lrb_search_15mers_layout {paths} \"{reads_path}\" \"{out}\" {list(blocks)} {threads}")
    o = _lib.lib.lrb_search_15mers_layout(c_paths, n, os.fsencode(reads_path), arr, len(blocks), os.fsencode(out),
                                          os.fsencode(out + ".npy") if write_npy else None, int(threads))
    check_proc(o, "Counting 15-mer profiles by layout")
    with open(out + ".layout", "w") as f:
        f.writelines(layout_lines(paths, blocks))


def run_15mer_histo(output, threads, max_count=65536):
    """Abundance spectrum of {output}/profiles/15mers-counts as {output}/profiles/15mers-histo (jellyfish `histo`
    layout: "count n_kmers" lines of canonical 15-mers), to choose -bs / -bc from (INTEGRATION.md).  No reference
    counterpart; `threads` is accepted for symmetry with the other runners."""
    logger.debug(f"LIB::lrb_table_spectrum \"{output}/profiles/15mers-counts\" \"{output}/profiles/15mers-histo\" {max_count}")
    o = _lib.lib.lrb_table_spectrum(os.fsencode(f"{output}/profiles/15mers-counts"), os.fsencode(f"{output}/profiles/15mers-histo"),
                                    int(max_count))
    check_proc(o, "15-mer abundance spectrum")


def run_profile(reads_path, output, k_size, bin_size, bin_count, threads, write_table=True, write_npy=False, n_gpus=0):
    """Fused stages 1_1 + 1_2 + 2_1: leaves com_profs, cov_profs (and 15mers-counts unless write_table=False,
    needed by --resume with changed -bs/-bc) in {output}/profiles, byte-identical to the three separate calls.
    n_gpus > 1 shards the reads over that many GPUs of this node (0: LRB_GPUS from the environment, default 1);
    the three separate runners above honour LRB_GPUS the same way.  Same files whatever the GPU count."""
    if not os.path.isdir(f"{output}/profiles"):
        os.makedirs(f"{output}/profiles")

    logger.debug(f"LIB::lrb_profile \"{reads_path}\" \"{output}\" {k_size} {bin_size} {bin_count} {threads}")
    o = _lib.lib.lrb_profile_multi(os.fsencode(reads_path), os.fsencode(output), int(k_size), int(bin_size), int(bin_count),
                                   int(threads), int(n_gpus), 1 if write_table else 0, 1 if write_npy else 0)
    check_proc(o, "Computing profiles")


def check_proc(ret, name=""):
    if ret != 0:
        if name != "":
            logger.error(f"Error in step: {name}")
        logger.error(f"Failed due to an error. Please check the log. Good Bye! ({_lib.last_error()})")
        sys.exit(ret)
