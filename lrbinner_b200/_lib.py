"""ctypes binding of liblrb200.so (C ABI in include/lrbinner_b200.h).

There is no CPU fallback: if the shared library is missing this module raises at import, and any
compute entry point returns LRB_ECUDA when no CUDA device is present.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblrb200.so")

LRB_OK, LRB_EINVAL, LRB_EIO, LRB_ECUDA, LRB_ENOMEM, LRB_EFORMAT = range(6)
TABLE_ENTRIES = 1 << 30
TILE_BLOCKS = 256
MAX_BINS = 4096
MAX_COV_SETTINGS = 8
MAX_SAMPLE_TABLES = 8
COMPACT_ENTRIES = 1 << 29
SPECTRUM_MAX_COUNT = 1 << 24


class LrbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"liblrb200 error {code}: {msg}")
        self.code = code


class ReadsView(C.Structure):
    """lrb_reads_view: sizes + raw pointers (host or device, depending on who filled it)."""
    _fields_ = [("n_reads", C.c_uint64), ("n_blocks", C.c_uint64), ("n_tiles", C.c_uint64), ("total_bases", C.c_uint64),
                ("codes", C.c_void_p), ("valid", C.c_void_p), ("read_len", C.c_void_p), ("read_blk", C.c_void_p),
                ("tile_read", C.c_void_p), ("tile_blk", C.c_void_p)]


class Partition(C.Structure):
    """lrb_partition: caller-owned device buffers + the bucket layout filled by lrb_dev_partition_begin/add."""
    _fields_ = [("keys", C.c_void_p), ("small", C.c_void_p), ("steps", C.c_void_p), ("sub", C.c_void_p), ("capacity", C.c_uint64),
                ("sub_capacity", C.c_uint64), ("step_capacity", C.c_uint64), ("steps_used", C.c_uint64), ("n_reads", C.c_uint64),
                ("n_buckets", C.c_int), ("shift", C.c_int), ("has_rids", C.c_int), ("n_chunks", C.c_int),
                ("key_lo", C.c_uint32), ("key_hi", C.c_uint32),
                ("chunk_step0", C.c_uint32 * 64), ("chunk_nsteps", C.c_uint32 * 64),
                ("l2_enabled", C.c_int), ("l2_ncta", C.c_uint32), ("l2_C3", C.c_uint32), ("l2_seg0", C.c_uint64), ("l2_span", C.c_uint64),
                ("l2_cells0", C.c_uint64), ("l2_spill0", C.c_uint64), ("l2_spill_cap", C.c_uint32)]


PART_SMALL_U64 = 16384


class RunInfo(C.Structure):
    """lrb_run_info: how the last lrb_profile_host call ran."""
    _fields_ = [("n_devices", C.c_int), ("n_batches", C.c_int), ("table_path", C.c_int), ("lists_reused", C.c_int),
                ("wall_ms", C.c_float), ("exchange_ms", C.c_float), ("batch_bases_max", C.c_uint64),
                ("host_plan_ms", C.c_float), ("host_enqueue_ms", C.c_float)]


PROFILE_USE_LOADED_TABLE, PROFILE_KEEP_TABLE, PROFILE_ADD_TO_TABLE = 1, 2, 4


class CovBlockC(C.Structure):
    """lrb_cov_block: one block of a mixed coverage row (table -1 = the context's table, 0..7 = a sample slot)."""
    _fields_ = [("table", C.c_int), ("by_edges", C.c_int), ("bin_size", C.c_long), ("bins", C.c_int), ("edges", C.c_void_p),
                ("n_edges", C.c_int)]


class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_genomes", C.c_uint32), ("sub_thr", C.c_uint32), ("ins_thr", C.c_uint32),
                ("del_thr", C.c_uint32), ("n_thr", C.c_uint32), ("read_base", C.c_uint64)]


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
        "`make -C lrbinner_b200/csrc` (nvcc, sm_100a). lrbinner_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

_P = C.c_void_p
_SIG = {
    "lrb_version": (C.c_int, []),
    "lrb_last_error": (C.c_char_p, []),
    "lrb_reads_from_file": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(_P)]),
    "lrb_reads_from_ascii": (C.c_int, [_P, _P, C.c_uint64, C.c_int, C.POINTER(_P)]),
    "lrb_reads_from_lengths": (C.c_int, [_P, C.c_uint64, C.POINTER(_P)]),
    "lrb_reads_view_get": (C.c_int, [_P, C.POINTER(ReadsView)]),
    "lrb_reads_unpack": (C.c_int, [_P, C.c_uint64, _P, C.c_uint64]),
    "lrb_reads_slice": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.POINTER(_P)]),
    "lrb_reads_free": (None, [_P]),
    "lrb_reads_index_valid": (C.c_int, [_P, C.c_int, _P]),
    "lrb_reads_exceptions": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_uint64)]),
    "lrb_reader_open": (C.c_int, [C.c_char_p, C.c_int, C.c_uint64, C.POINTER(_P)]),
    "lrb_reader_next": (C.c_int, [_P, C.POINTER(_P)]),
    "lrb_reader_rewind": (C.c_int, [_P]),
    "lrb_reader_tell": (C.c_int, [_P, _P, _P, _P, _P]),
    "lrb_reader_close": (None, [_P]),
    "lrb_dev_fill_valid": (C.c_int, [C.POINTER(ReadsView), _P, _P, C.c_uint64, _P]),
    "lrb_dev_composition": (C.c_int, [C.POINTER(ReadsView), C.c_int, _P, C.c_uint64, C.c_uint64, _P]),
    "lrb_dev_count": (C.c_int, [C.POINTER(ReadsView), _P, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, _P]),
    "lrb_dev_mirror": (C.c_int, [_P, _P]),
    "lrb_dev_table_spectrum": (C.c_int, [_P, C.c_uint32, C.c_uint32, C.c_uint32, _P, _P]),
    "lrb_dev_compact_spectrum": (C.c_int, [_P, C.c_uint32, _P, _P]),
    "lrb_dev_copy2d": (C.c_int, [_P, C.c_uint64, _P, C.c_uint64, C.c_uint64, C.c_uint64, _P]),
    "lrb_dev_add_planes": (C.c_int, [_P, C.c_uint64, _P, C.c_uint64, C.c_int, C.c_uint32, C.c_uint32, _P]),
    "lrb_dev_search": (C.c_int, [C.POINTER(ReadsView), _P, C.c_long, C.c_int, _P, _P, C.c_uint64, C.c_uint64,
                                 C.c_uint32, C.c_uint32, _P]),
    "lrb_dev_fill_blk_read": (C.c_int, [C.POINTER(ReadsView), _P, _P]),
    "lrb_partition_step_capacity": (C.c_uint64, [C.c_uint64, C.c_int]),
    "lrb_partition_steps_words": (C.c_uint64, [C.c_uint64]),
    "lrb_dev_partition_begin": (C.c_int, [_P, C.c_int, C.c_uint32, C.c_uint32, C.c_int, _P]),
    "lrb_dev_partition_add": (C.c_int, [C.POINTER(ReadsView), _P, C.c_uint64, C.c_uint64, _P, _P]),
    "lrb_dev_partition_check": (C.c_int, [_P, _P, _P]),
    "lrb_dev_partition_build": (C.c_int, [C.POINTER(ReadsView), _P, C.c_int, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, _P, _P]),
    "lrb_dev_partition_apply": (C.c_int, [_P, C.c_int, _P, C.c_long, C.c_int, _P, _P, _P]),
    "lrb_dev_partition_apply_range": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, C.c_long, C.c_int, _P, _P, _P]),
    "lrb_dev_partition_search_settings": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P]),
    "lrb_dev_partition_search_samples": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P]),
    "lrb_dev_partition_search_edges": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P, _P]),
    "lrb_dev_partition_search_layout": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, C.c_int, _P, _P, _P]),
    "lrb_dev_table_compact": (C.c_int, [_P, _P, _P]),
    "lrb_dev_pack_ascii": (C.c_int, [C.POINTER(ReadsView), _P, _P, _P]),
    "lrb_dev_format_composition": (C.c_int, [_P, _P, C.c_uint64, C.c_int, _P, _P]),
    "lrb_dev_format_coverage": (C.c_int, [_P, _P, C.c_uint64, C.c_int, _P, _P]),
    "lrb_dev_profile_values": (C.c_int, [_P, _P, C.c_uint64, C.c_int, C.c_int, _P, _P]),
    "lrb_dev_synth": (C.c_int, [C.POINTER(ReadsView), C.POINTER(SynthParams), _P, _P, _P]),
    "lrb_synth_host": (C.c_int, [C.POINTER(SynthParams), _P, _P, _P, C.c_uint64, _P, _P]),
    "lrb_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "lrb_ctx_create_multi": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "lrb_ctx_device_count": (C.c_int, [_P]),
    "lrb_ctx_destroy": (None, [_P]),
    "lrb_ctx_last_info": (C.c_int, [_P, _P]),
    "lrb_profile_host": (C.c_int, [_P, _P, C.c_int, C.c_long, C.c_int, _P, _P, _P, _P, C.c_int]),
    "lrb_profile_host_settings": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int]),
    "lrb_profile_host_samples": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, C.c_int]),
    "lrb_profile_host_edges": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P, _P, _P, C.c_int]),
    "lrb_profile_host_layout": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P, _P, _P, C.c_int]),
    "lrb_ctx_sample_table_load": (C.c_int, [_P, C.c_int, C.c_char_p]),
    "lrb_ctx_sample_table_keep": (C.c_int, [_P, C.c_int]),
    "lrb_ctx_sample_table_free": (C.c_int, [_P, C.c_int]),
    "lrb_table_read_canonical": (C.c_int, [C.c_char_p, C.c_uint32, C.c_uint32, _P]),
    "lrb_ctx_last_timings": (C.c_int, [_P, _P]),
    "lrb_pinned_alloc": (_P, [C.c_size_t]),
    "lrb_pinned_free": (None, [_P]),
    "lrb_ctx_table_load": (C.c_int, [_P, C.c_char_p]),
    "lrb_ctx_table_save": (C.c_int, [_P, C.c_char_p]),
    "lrb_ctx_table_spectrum": (C.c_int, [_P, C.c_uint32, _P]),
    "lrb_ctx_sample_table_spectrum": (C.c_int, [_P, C.c_int, C.c_uint32, _P]),
    "lrb_prof_launches": (C.c_uint64, []),
    "lrb_prof_enable": (C.c_int, [C.c_int]),
    "lrb_prof_report": (C.c_int, [_P, C.c_size_t]),
    "lrb_fixed6": (C.c_uint32, [C.c_uint32, C.c_uint32, C.c_int]),
    "lrb_write_composition_txt": (C.c_int, [C.c_char_p, _P, _P, C.c_uint64, C.c_int, C.c_int]),
    "lrb_write_coverage_txt": (C.c_int, [C.c_char_p, _P, _P, C.c_uint64, C.c_int, C.c_int]),
    "lrb_write_composition_npy": (C.c_int, [C.c_char_p, _P, _P, C.c_uint64, C.c_int, C.c_int]),
    "lrb_write_coverage_npy": (C.c_int, [C.c_char_p, _P, _P, C.c_uint64, C.c_int, C.c_int]),
    "lrb_append_composition_txt": (C.c_int, [C.c_char_p, _P, _P, C.c_uint64, C.c_int, C.c_int, C.c_uint64]),
    "lrb_append_coverage_txt": (C.c_int, [C.c_char_p, _P, _P, C.c_uint64, C.c_int, C.c_int, C.c_uint64]),
    "lrb_append_composition_npy": (C.c_int, [C.c_char_p, _P, _P, C.c_uint64, C.c_int, C.c_int, C.c_uint64]),
    "lrb_append_coverage_npy": (C.c_int, [C.c_char_p, _P, _P, C.c_uint64, C.c_int, C.c_int, C.c_uint64]),
    "lrb_table_write_file": (C.c_int, [C.c_char_p, _P]),
    "lrb_table_read_file": (C.c_int, [C.c_char_p, _P]),
    "lrb_spectrum_bin_mass": (C.c_int, [_P, C.c_uint32, C.c_long, C.c_int, _P]),
    "lrb_spectrum_edge_mass": (C.c_int, [_P, C.c_uint32, _P, C.c_int, _P]),
    "lrb_write_spectrum_txt": (C.c_int, [C.c_char_p, _P, C.c_uint32]),
    "lrb_kmer_lut": (C.c_int, [C.c_int, _P]),
    "lrb_count_kmers": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_int]),
    "lrb_count_15mers": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int]),
    "lrb_search_15mers": (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_long, C.c_int, C.c_int]),
    "lrb_search_15mers_settings": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, _P, _P, _P, _P, C.c_int]),
    "lrb_search_15mers_samples": (C.c_int, [_P, C.c_int, _P, _P, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int]),
    "lrb_search_15mers_edges": (C.c_int, [C.c_char_p, C.c_char_p, _P, C.c_int, C.c_char_p, C.c_char_p, C.c_int]),
    "lrb_search_15mers_layout": (C.c_int, [_P, C.c_int, C.c_char_p, _P, C.c_int, C.c_char_p, C.c_char_p, C.c_int]),
    "lrb_table_spectrum": (C.c_int, [C.c_char_p, C.c_char_p, C.c_uint32]),
    "lrb_profile": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int]),
    "lrb_profile_multi": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
}

EXPORTS = tuple(_SIG)

for _name, (_res, _args) in _SIG.items():
    _fn = getattr(lib, _name)   # AttributeError here == the .so does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args


def prof_report():
    """{kernel: (launches, total_ms)} recorded since lrb_prof_enable(1); synchronise the device(s) first."""
    buf = C.create_string_buffer(1 << 16)
    check(lib.lrb_prof_report(buf, len(buf)))
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.split()
        out[name] = (int(n), float(ms))
    return out


def last_error():
    return (lib.lrb_last_error() or b"").decode("utf-8", "replace")


def check(rc):
    if rc != 0:
        raise LrbError(rc, last_error())
    return rc
