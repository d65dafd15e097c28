"""Buffer-level Python view of the profile stage (thin wrappers over the C ABI).

  PackedReads  — a read set in the packed host layout (lrb_reads*), from a FASTA/FASTQ file, from
                 ASCII bases, or layout-only from lengths.
  SegmentReader / read_segments — a FASTA/FASTQ file as consecutive read sets of bounded size (lrb_reader_*).
  Context      — one GPU: seam-to-seam `profile()` over host buffers (lrb_profile_host).
  DeviceReads / dev_* — torch-tensor plumbing for the device-pointer level (lrb_dev_*): used by the
                 device-resident benchmark and the multi-GPU driver (lrbinner_b200/dist.py), where
                 torch.distributed needs tensors over the same memory.

The arithmetic lives in the CUDA kernels; nothing here computes profiles on the CPU.
"""
import collections
import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import ReadsView, check, lib

COMP_WIDTH = {3: 32, 4: 136, 5: 512}
LRB_MAX_CHUNKS = 64


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class PackedReads:
    """Owns an lrb_reads* (host memory, page-locked when a GPU is present)."""

    def __init__(self, handle):
        self._h = handle
        self.view = ReadsView()
        check(lib.lrb_reads_view_get(self._h, C.byref(self.view)))

    # -- constructors ---------------------------------------------------------------------------
    @classmethod
    def from_file(cls, path, threads=8):
        h = C.c_void_p()
        check(lib.lrb_reads_from_file(str(path).encode(), int(threads), C.byref(h)))
        return cls(h)

    @classmethod
    def from_sequences(cls, seqs, threads=8):
        """seqs: iterable of bytes/str (one per read)."""
        bs = [s if isinstance(s, (bytes, bytearray)) else s.encode("latin-1") for s in seqs]
        offsets = np.zeros(len(bs) + 1, dtype=np.uint64)
        if bs:
            offsets[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
        bases = np.frombuffer(b"".join(bs) + b"\0", dtype=np.uint8)
        return cls.from_ascii(bases, offsets, threads)

    @classmethod
    def from_ascii(cls, bases, offsets, threads=8):
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        h = C.c_void_p()
        check(lib.lrb_reads_from_ascii(_ptr(bases), _ptr(offsets), len(offsets) - 1, int(threads), C.byref(h)))
        return cls(h)

    @classmethod
    def from_lengths(cls, lengths):
        lengths = np.ascontiguousarray(lengths, dtype=np.uint32)
        h = C.c_void_p()
        check(lib.lrb_reads_from_lengths(_ptr(lengths), len(lengths), C.byref(h)))
        return cls(h)

    def slice(self, read_lo, read_hi):
        """Reads [read_lo, read_hi) as a read set of its own (shares the packed stream with self, which it keeps alive)."""
        h = C.c_void_p()
        check(lib.lrb_reads_slice(self._h, int(read_lo), int(read_hi), C.byref(h)))
        s = PackedReads(h)
        s._parent = self
        return s

    # -- accessors ------------------------------------------------------------------------------
    n_reads = property(lambda self: int(self.view.n_reads))
    n_blocks = property(lambda self: int(self.view.n_blocks))
    n_tiles = property(lambda self: int(self.view.n_tiles))
    total_bases = property(lambda self: int(self.view.total_bases))

    def _arr(self, ptr, n):
        if n == 0:
            return np.zeros(0, dtype=np.uint32)
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint32)), shape=(n,))

    codes = property(lambda self: self._arr(self.view.codes, 2 * self.n_blocks + 2))
    valid = property(lambda self: self._arr(self.view.valid, self.n_blocks + 1))
    read_len = property(lambda self: self._arr(self.view.read_len, self.n_reads))
    read_blk = property(lambda self: self._arr(self.view.read_blk, self.n_reads + 1))
    tile_read = property(lambda self: self._arr(self.view.tile_read, self.n_tiles))
    tile_blk = property(lambda self: self._arr(self.view.tile_blk, self.n_tiles))

    def index_valid(self, threads=8):
        """(Re)build the validity-exception list from the current `valid` words; returns its length."""
        n = C.c_uint64(0)
        check(lib.lrb_reads_index_valid(self._h, int(threads), C.byref(n)))
        return int(n.value)

    def exceptions(self):
        """(blocks, words) of the validity-exception list (copies; empty when none was built)."""
        blk, word, n = C.c_void_p(), C.c_void_p(), C.c_uint64(0)
        check(lib.lrb_reads_exceptions(self._h, C.byref(blk), C.byref(word), C.byref(n)))
        if not n.value:
            return np.zeros(0, dtype=np.uint32), np.zeros(0, dtype=np.uint32)
        return (np.array(self._arr(blk, int(n.value)), copy=True), np.array(self._arr(word, int(n.value)), copy=True))

    def unpack(self, i):
        n = int(self.read_len[i])
        buf = C.create_string_buffer(max(n, 1))
        check(lib.lrb_reads_unpack(self._h, i, buf, n))
        return buf.raw[:n]

    def close(self):
        if self._h:
            lib.lrb_reads_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SegmentReader:
    """Owns an lrb_reader*: the records of a FASTA/FASTQ file (plain or gzip) as consecutive PackedReads of at most
    `segment_bases` bases each (a longer read forms a segment on its own; 0 = sized from the host's available memory).
    Concatenated, the segments are PackedReads.from_file(path)."""

    def __init__(self, path, segment_bases=0, threads=8):
        self._h = C.c_void_p()
        check(lib.lrb_reader_open(str(path).encode(), int(threads), int(segment_bases), C.byref(self._h)))

    def next(self):
        """The next segment, or None at the end of the file."""
        h = C.c_void_p()
        check(lib.lrb_reader_next(self._h, C.byref(h)))
        return PackedReads(h) if h.value else None

    def __iter__(self):
        while True:
            seg = self.next()
            if seg is None:
                return
            yield seg

    def rewind(self):
        check(lib.lrb_reader_rewind(self._h))

    def tell(self):
        """dict(reads, bases, segments) delivered since open / rewind, and at_end (no record left)."""
        v = [C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)]
        at_end = C.c_int(0)
        check(lib.lrb_reader_tell(self._h, C.byref(v[0]), C.byref(v[1]), C.byref(v[2]), C.byref(at_end)))
        return {"reads": v[0].value, "bases": v[1].value, "segments": v[2].value, "at_end": bool(at_end.value)}

    def close(self):
        if self._h:
            lib.lrb_reader_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def read_segments(path, segment_bases=0, threads=8):
    """Generator of the segments of a FASTA/FASTQ file as PackedReads (see SegmentReader); the reader lives as long as
    the generator."""
    reader = SegmentReader(path, segment_bases, threads)
    try:
        yield from reader
    finally:
        reader.close()


class Context:
    """One GPU, or several driven from this process (device = an ordinal or a list of ordinals; the first is the
    primary and ends up with the complete table).  profile() is the seam-to-seam call: host buffers in, host buffers out."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            ids = (C.c_int * len(device))(*[int(d) for d in device])
            check(lib.lrb_ctx_create_multi(ids, len(device), C.byref(self._h)))
        else:
            check(lib.lrb_ctx_create(int(device), C.byref(self._h)))
        self.device = device

    def profile(self, reads, k=None, bin_size=None, bins=None, want_table=False, use_loaded_table=False, out=None,
                keep_table=False, add_to_table=False, coverage=None, samples=None, edges=None, layout=None):
        """Returns dict(comp=[N,P] u32, hist=[N,bins] u32, sums=[N] u32, table=[2^30] u32) for the requested parts.
        `out` may carry preallocated (ideally page-locked) arrays under the same keys.  add_to_table: count these reads
        INTO the context's complete table (from an earlier count or table_load) instead of from zero; on failure the
        context holds no table.
        coverage=[(bin_size, bins), ...] (instead of bin_size / bins): up to 8 settings searched in one pass over the table
        (lrb_profile_host_settings).  hist is then [N, W], W = the sum of the bins, with each setting's columns after those of
        the settings before it; hists[m] is the [N, bins_m] view of setting m, and sums are the same for every setting.
        samples=[(slot, bin_size, bins), ...] (instead of coverage / bin_size / bins): coverage against up to 8 sample slots
        (sample_table_load / sample_table_keep) instead of the context's table (lrb_profile_host_samples); hist [N, W] holds
        table 0's bins, then table 1's, ..., hists[t] is table t's view and sums are shared.
        edges=[t_1, ..., t_{B-1}] (instead of every other coverage argument): bins given by strictly increasing count edges,
        t_1 >= 2; a window whose 15-mer is counted c times goes to bin searchsorted(edges, c, side="right") of hist [N, B]
        (lrb_profile_host_edges).
        layout=[CovBlock, ...] (instead of every other coverage argument): a mixed row of up to 8 blocks, each on the
        context's table (table=None) or a sample slot, each binned by (bin_size, bins) or by edges (lrb_profile_host_layout);
        hist [N, W] holds block 0's bins, then block 1's, ..., hists[m] is block m's view and sums are shared.  A block on
        the context's table counts it from these reads unless use_loaded_table / add_to_table; a layout of slots alone
        leaves the context's table as it was."""
        given = [arg for arg, v in (("layout=[CovBlock, ...]", layout), ("edges=[...]", edges), ("samples=[(slot, bin_size, bins), ...]", samples),
                                    ("coverage=[(bin_size, bins), ...]", coverage)) if v is not None]
        if given and len(given) + (bin_size is not None or bins is not None) > 1:
            raise _lib.LrbError(_lib.LRB_EINVAL, f"{given[0]} replaces the other coverage arguments (bin_size / bins, coverage, samples, "
                                                 "edges, layout): give one of them")
        n = reads.n_reads
        out = dict(out or {})
        comp = hist = sums = table = hists = slots = width = None
        if edges is not None:
            edges = _edges_array(edges)   # refused here, before a context is needed
            width = edges.size + 1
        if layout is not None:
            blocks, keep, widths = _layout_blocks(layout)   # refused here, before a context is needed
            width = sum(widths)
        if samples is not None:
            samples = [(int(t), int(s_), int(b)) for t, s_, b in samples]
            slots = np.array([t for t, _, _ in samples], dtype=np.int32)
            coverage = [(s_, b) for _, s_, b in samples]
        set_bs, set_bins = _settings_arrays(coverage if coverage is not None else
                                            [(bin_size if bin_size is not None else 1, bins if bins is not None else 1)])
        if bins is not None or coverage is not None:
            width = max(int(np.clip(set_bins, 1, None).sum()), 1)
            if coverage is not None and width > _lib.MAX_BINS:   # refused by the library before any work: no real buffer
                width = 1
        if k is not None:
            comp = out.get("comp")
            if comp is None:
                comp = np.zeros((n, COMP_WIDTH[k]), dtype=np.uint32)
        if width is not None:
            hist = out.get("hist")
            if hist is None:
                hist = np.zeros((n, width), dtype=np.uint32)
            sums = out.get("sums")
            if sums is None:
                sums = np.zeros(n, dtype=np.uint32)
        if want_table:
            table = out.get("table")
            if table is None:
                table = np.empty(_lib.TABLE_ENTRIES, dtype=np.uint32)
        flags = ((_lib.PROFILE_USE_LOADED_TABLE if use_loaded_table else 0) | (_lib.PROFILE_KEEP_TABLE if keep_table else 0) |
                 (_lib.PROFILE_ADD_TO_TABLE if add_to_table else 0))
        k = int(k) if k is not None else 0
        parts = (_ptr(comp) if comp is not None else None, _ptr(hist) if hist is not None else None,
                 _ptr(sums) if sums is not None else None, _ptr(table) if table is not None else None)
        if layout is not None:
            check(lib.lrb_profile_host_layout(self._h, reads._h, k, blocks, len(widths), *parts, flags))
            offs = np.concatenate([[0], np.cumsum(widths)])
            hists = [hist[:, offs[m]:offs[m + 1]] for m in range(len(widths))]
        elif edges is not None:
            check(lib.lrb_profile_host_edges(self._h, reads._h, k, _ptr(edges), int(edges.size), *parts, flags))
        elif slots is not None:
            check(lib.lrb_profile_host_samples(self._h, reads._h, k, len(set_bs), _ptr(slots), _ptr(set_bs), _ptr(set_bins), *parts, flags))
        else:
            check(lib.lrb_profile_host_settings(self._h, reads._h, k, len(set_bs), _ptr(set_bs), _ptr(set_bins), *parts, flags))
        if coverage is not None:
            offs = np.concatenate([[0], np.cumsum(set_bins)])
            hists = [hist[:, offs[m]:offs[m + 1]] for m in range(len(set_bins))]
        return {"comp": comp, "hist": hist, "hists": hists, "sums": sums, "table": table}

    def info(self):
        """How the last profile() ran: devices, batches, table path, wall / exchange milliseconds."""
        ri = _lib.RunInfo()
        check(lib.lrb_ctx_last_info(self._h, C.byref(ri)))
        return {f: getattr(ri, f) for f, _ in ri._fields_}

    def timings(self):
        ms = (C.c_float * 7)()
        check(lib.lrb_ctx_last_timings(self._h, ms))
        # phases overlap (3-stream pipeline): h2d runs beside composition+partition; "total" is the whole call
        return dict(zip(("h2d", "composition_partition", "table_passes", "mirror", "search_direct", "d2h_tail", "total"),
                        [float(x) for x in ms]))

    def table_load(self, path):
        check(lib.lrb_ctx_table_load(self._h, str(path).encode()))

    def table_save(self, path):
        check(lib.lrb_ctx_table_save(self._h, str(path).encode()))

    def sample_table_load(self, slot, path):
        """Load the canonical rows of a 15mers-counts file into sample slot `slot` on every device (2 GiB each)."""
        check(lib.lrb_ctx_sample_table_load(self._h, int(slot), os.fsencode(path)))

    def sample_table_keep(self, slot):
        """Copy the context's own complete table, in compact form, into sample slot `slot` on every device."""
        check(lib.lrb_ctx_sample_table_keep(self._h, int(slot)))

    def sample_table_free(self, slot):
        check(lib.lrb_ctx_sample_table_free(self._h, int(slot)))

    def table_spectrum(self, max_count=65536):
        """Abundance spectrum of the context's table: u64[max_count + 3] = n_c for c < max_count (canonical 15-mers
        counted c times), then keys counted >= max_count, their sum, and the largest count (lrb_dev_table_spectrum)."""
        spec = np.zeros(_spectrum_len(max_count), dtype=np.uint64)
        check(lib.lrb_ctx_table_spectrum(self._h, int(max_count), _ptr(spec)))
        return spec

    def sample_table_spectrum(self, slot, max_count=65536):
        """table_spectrum() of sample slot `slot` (lrb_ctx_sample_table_spectrum): what table_spectrum() gave for the table
        the slot was loaded from or kept, so each sample's equal-mass edges (spectrum_quantile_edges) come from its slot."""
        spec = np.zeros(_spectrum_len(max_count), dtype=np.uint64)
        check(lib.lrb_ctx_sample_table_spectrum(self._h, int(slot), int(max_count), _ptr(spec)))
        return spec

    def close(self):
        if self._h:
            lib.lrb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pinned_empty(shape, dtype=np.uint32):
    """numpy array over cudaHostAlloc memory (freed when the array's base object dies)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = lib.lrb_pinned_alloc(max(n, 16))
    if not p:
        raise _lib.LrbError(_lib.LRB_ECUDA, _lib.last_error())

    class _Owner:
        def __init__(self, p):
            self.p = p

        def __del__(self):
            lib.lrb_pinned_free(self.p)

    owner = _Owner(p)
    buf = (C.c_uint8 * max(n, 16)).from_address(p)
    buf._owner = owner
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    return arr


# ---- device-pointer level over torch tensors -------------------------------------------------------

class DeviceReads:
    """The packed read set resident in HBM as torch tensors (int32 views of the u32 words)."""

    def __init__(self, reads, device, upload=True):
        import torch
        self.torch = torch
        self.device = torch.device(device)
        self.n_reads, self.n_blocks, self.n_tiles, self.total_bases = reads.n_reads, reads.n_blocks, reads.n_tiles, reads.total_bases

        def up(a, n, fill=True):
            t = torch.zeros(max(n, 1), dtype=torch.int32, device=self.device)
            if fill and len(a):
                t[:len(a)].copy_(torch.from_numpy(a.view(np.int32)))
            return t

        self.codes = up(reads.codes, 2 * self.n_blocks + 2, upload)
        self.valid = up(reads.valid, self.n_blocks + 1, upload)
        self.read_len = up(reads.read_len, self.n_reads)
        self.read_blk = up(reads.read_blk, self.n_reads + 1)
        self.tile_read = up(reads.tile_read, self.n_tiles)
        self.tile_blk = up(reads.tile_blk, self.n_tiles)
        # int64 copy: np.searchsorted then takes any integer type without converting the whole array on every call
        # (an O(n_tiles) conversion per lookup cost 13 ms per chunk of the 4-GPU e2e step)
        self.tile_read_host = np.asarray(reads.tile_read, dtype=np.int64).copy()
        self.view = ReadsView(self.n_reads, self.n_blocks, self.n_tiles, self.total_bases, self.codes.data_ptr(),
                              self.valid.data_ptr(), self.read_len.data_ptr(), self.read_blk.data_ptr(),
                              self.tile_read.data_ptr(), self.tile_blk.data_ptr())

    def download_into(self, reads):
        """Copy the device stream back into the host buffers of `reads` (same layout)."""
        torch = self.torch
        torch.from_numpy(reads.codes.view(np.int32)).copy_(self.codes[:2 * self.n_blocks + 2])
        torch.from_numpy(reads.valid.view(np.int32)).copy_(self.valid[:self.n_blocks + 1])

    def tile_range_for_reads(self, read_lo, read_hi):
        lo = int(np.searchsorted(self.tile_read_host, np.int64(read_lo), side="left"))
        hi = int(np.searchsorted(self.tile_read_host, np.int64(read_hi), side="left"))
        return lo, hi


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dev_composition(dr, k, counts, tile_lo=0, tile_hi=None):
    check(lib.lrb_dev_composition(C.byref(dr.view), k, C.c_void_p(counts.data_ptr()), tile_lo,
                                  dr.n_tiles if tile_hi is None else tile_hi, _stream()))


def dev_count(dr, table, blk_lo=0, blk_hi=None, key_lo=0, key_hi=_lib.TABLE_ENTRIES):
    check(lib.lrb_dev_count(C.byref(dr.view), C.c_void_p(table.data_ptr()), blk_lo, dr.n_blocks if blk_hi is None else blk_hi,
                            key_lo, min(key_hi, _lib.TABLE_ENTRIES), _stream()))


def dev_fill_valid(dr, exc_blk=None, exc_word=None):
    """Rebuild dr.valid on the device from the read lengths + the exception list (torch int32 tensors or None)."""
    n = 0 if exc_blk is None else int(exc_blk.numel())
    check(lib.lrb_dev_fill_valid(C.byref(dr.view), C.c_void_p(exc_blk.data_ptr()) if n else None,
                                 C.c_void_p(exc_word.data_ptr()) if n else None, n, _stream()))


def dev_mirror(table):
    check(lib.lrb_dev_mirror(C.c_void_p(table.data_ptr()), _stream()))


def _spectrum_len(max_count):
    if not 0 <= int(max_count) < 2 ** 32:   # the C ABI takes a u32; range [2, SPECTRUM_MAX_COUNT] is checked there
        raise _lib.LrbError(_lib.LRB_EINVAL, f"max_count {max_count} out of range")
    return int(max_count) + 3


def dev_table_spectrum(table, max_count, key_lo=0, key_hi=_lib.TABLE_ENTRIES, out=None):
    """Accumulate the spectrum of the bit-15-clear keys of table[key_lo, key_hi) into `out` (int64 tensor of
    max_count + 3 words read as u64, zeroed here when not given) and return it."""
    import torch
    n = _spectrum_len(max_count)
    if out is None:
        out = torch.zeros(n, dtype=torch.int64, device=table.device)
    elif out.numel() < n or out.element_size() != 8 or not out.is_contiguous():
        raise _lib.LrbError(_lib.LRB_EINVAL, f"spectrum buffer must be {n} contiguous 8-byte words")
    check(lib.lrb_dev_table_spectrum(C.c_void_p(table.data_ptr()), int(key_lo), min(int(key_hi), _lib.TABLE_ENTRIES), int(max_count),
                                     C.c_void_p(out.data_ptr()), _stream()))
    return out


def dev_compact_spectrum(compact, max_count, out=None):
    """dev_table_spectrum of a whole compact table (dev_table_compact; lrb_dev_compact_spectrum), accumulated into `out`
    (zeroed here when not given) and returned."""
    import torch
    n = _spectrum_len(max_count)
    if out is None:
        out = torch.zeros(n, dtype=torch.int64, device=compact.device)
    elif out.numel() < n or out.element_size() != 8 or not out.is_contiguous():
        raise _lib.LrbError(_lib.LRB_EINVAL, f"spectrum buffer must be {n} contiguous 8-byte words")
    check(lib.lrb_dev_compact_spectrum(C.c_void_p(compact.data_ptr()), int(max_count), C.c_void_p(out.data_ptr()), _stream()))
    return out


def spectrum_bin_mass(spectrum, bin_size, bins):
    """Windows per coverage bin implied by a spectrum (lrb_spectrum_bin_mass): equals hist.sum(0) of a search of the
    reads the table was counted from, with the same bin_size / bins."""
    spec = np.ascontiguousarray(spectrum, dtype=np.uint64)
    if spec.size < 3:
        raise _lib.LrbError(_lib.LRB_EINVAL, "a spectrum has max_count + 3 words")
    mass = np.zeros(max(int(bins), 1), dtype=np.uint64)
    check(lib.lrb_spectrum_bin_mass(_ptr(spec), spec.size - 3, int(bin_size), int(bins), _ptr(mass)))
    return mass


def spectrum_edge_mass(spectrum, edges):
    """Windows per coverage bin implied by a spectrum for bins given by count edges (lrb_spectrum_edge_mass): equals
    hist.sum(0) of Context.profile(edges=edges) over the reads the table was counted from."""
    spec = np.ascontiguousarray(spectrum, dtype=np.uint64)
    if spec.size < 3:
        raise _lib.LrbError(_lib.LRB_EINVAL, "a spectrum has max_count + 3 words")
    e = _edges_array(edges)
    mass = np.zeros(e.size + 1, dtype=np.uint64)
    check(lib.lrb_spectrum_edge_mass(_ptr(spec), spec.size - 3, _ptr(e), int(e.size), _ptr(mass)))
    return mass


def spectrum_quantile_edges(spectrum, bins):
    """Count edges that split the windows of a spectrum (lrb_dev_table_spectrum layout) into `bins` bins of about equal
    mass, the most information per column: with M = max_count, mass(c) = c * n_c for c < M and Total = the sum of the
    masses plus the overflow keys' sum, t_i (i = 1 .. bins - 1) is the smallest c in [2, M] with
    bins * sum_{c' < c} mass(c') >= i * Total, in exact integers.  The walk stops at the first i without such a c, and
    repeated edges are dropped, so the result has at most bins - 1 strictly increasing edges: a single count holding more
    than 1 / bins of the mass (or the mass above M) gives fewer bins than asked for."""
    spec = np.ascontiguousarray(spectrum, dtype=np.uint64)
    if spec.size < 3:
        raise _lib.LrbError(_lib.LRB_EINVAL, "a spectrum has max_count + 3 words")
    B = int(bins)
    if not 1 <= B <= _lib.MAX_BINS:
        raise _lib.LrbError(_lib.LRB_EINVAL, f"bins must be in [1, {_lib.MAX_BINS}] (got {B})")
    M = spec.size - 3
    nz = [int(c) for c in np.flatnonzero(spec[:M])]
    total = sum(c * int(spec[c]) for c in nz) + int(spec[M + 1])
    # prefix(c) = sum_{c' < c} mass(c') only grows just after a counted c0, so the candidates are 2 and every c0 + 1 > 2
    steps = [(2, sum(c * int(spec[c]) for c in nz if c < 2))]
    run = steps[0][1]
    for c0 in nz:
        if c0 >= 2:
            run += c0 * int(spec[c0])
            steps.append((c0 + 1, run))
    edges, j = [], 0
    for i in range(1, B):
        while j < len(steps) and B * steps[j][1] < i * total:
            j += 1
        if j == len(steps):
            break
        if not edges or edges[-1] != steps[j][0]:
            edges.append(steps[j][0])
    return edges


def dev_search(dr, table, bin_size, bins, hist, sums, tile_lo=0, tile_hi=None, key_lo=0, key_hi=_lib.TABLE_ENTRIES):
    check(lib.lrb_dev_search(C.byref(dr.view), C.c_void_p(table.data_ptr()), bin_size, bins, C.c_void_p(hist.data_ptr()),
                             C.c_void_p(sums.data_ptr()), tile_lo, dr.n_tiles if tile_hi is None else tile_hi, key_lo,
                             min(key_hi, _lib.TABLE_ENTRIES), _stream()))


class PartitionWorkspace:
    """Scratch of the L2-resident table passes: 4-byte list entries for up to `capacity` windows, the per-step
    tables, the per-block read index, and the lrb_partition descriptor the C ABI fills."""

    def __init__(self, dr, capacity=None, max_chunks=LRB_MAX_CHUNKS, sub_capacity=None):
        torch = dr.torch
        self.dr = dr
        self.capacity = int(capacity if capacity is not None else max(dr.n_blocks * 32, 1))
        self.keys = torch.empty(self.capacity, dtype=torch.int32, device=dr.device)
        # second-level lists of the shared-memory count: 2 B per window, fixed-size segments -> 2x headroom (3x for small sets)
        self.sub_capacity = int(sub_capacity if sub_capacity is not None
                                else (2 if self.capacity >= (1 << 28) else 3) * self.capacity + (1 << 22))
        self.sub = torch.empty(self.sub_capacity, dtype=torch.int16, device=dr.device) if self.sub_capacity else None
        self.small = torch.zeros(_lib.PART_SMALL_U64, dtype=torch.int64, device=dr.device)
        self.step_capacity = int(lib.lrb_partition_step_capacity(dr.n_blocks, max_chunks))
        self.steps = torch.empty(int(lib.lrb_partition_steps_words(self.step_capacity)), dtype=torch.int32, device=dr.device)
        self.blk_read = torch.empty(max(dr.n_blocks, 1), dtype=torch.int32, device=dr.device)
        check(lib.lrb_dev_fill_blk_read(C.byref(dr.view), C.c_void_p(self.blk_read.data_ptr()), _stream()))
        self.part = _lib.Partition(keys=self.keys.data_ptr(), small=self.small.data_ptr(), steps=self.steps.data_ptr(),
                                   sub=self.sub.data_ptr() if self.sub is not None else None, capacity=self.capacity,
                                   sub_capacity=self.sub_capacity, step_capacity=self.step_capacity)

    def begin(self, with_rids=True, key_lo=0, key_hi=_lib.TABLE_ENTRIES, log2_bucket_keys=24, count=True):
        """count=False: the partition will only be searched — skip building the second-level (count) lists."""
        self.part.sub = self.sub.data_ptr() if (count and self.sub is not None) else None
        check(lib.lrb_dev_partition_begin(C.byref(self.part), 1 if with_rids else 0, key_lo, min(key_hi, _lib.TABLE_ENTRIES),
                                          log2_bucket_keys, _stream()))

    def add(self, blk_lo=0, blk_hi=None):
        check(lib.lrb_dev_partition_add(C.byref(self.dr.view), C.c_void_p(self.blk_read.data_ptr()), blk_lo,
                                        self.dr.n_blocks if blk_hi is None else blk_hi, C.byref(self.part), _stream()))

    def build(self, with_rids=True, blk_lo=0, blk_hi=None, key_lo=0, key_hi=_lib.TABLE_ENTRIES, log2_bucket_keys=24, grow=False,
              count=True):
        self.begin(with_rids, key_lo, key_hi, log2_bucket_keys, count)
        self.add(blk_lo, blk_hi)
        if grow:      # verify (synchronises); if the lists did not fit, the device told us the size: grow once and redo
            needed = C.c_uint64(0)
            rc = lib.lrb_dev_partition_check(C.byref(self.part), C.byref(needed), _stream())
            if rc == _lib.LRB_ENOMEM:
                torch = self.dr.torch
                self.keys = None
                torch.cuda.empty_cache()
                self.capacity = int(needed.value) + int(needed.value) // 64 + 1024
                self.keys = torch.empty(self.capacity, dtype=torch.int32, device=self.dr.device)
                self.part.keys, self.part.capacity = self.keys.data_ptr(), self.capacity
                if self.sub is not None and self.sub_capacity < 2 * self.capacity:
                    self.sub = None
                    torch.cuda.empty_cache()
                    self.sub_capacity = 2 * self.capacity + (1 << 22)
                    self.sub = torch.empty(self.sub_capacity, dtype=torch.int16, device=self.dr.device)
                    self.part.sub_capacity = self.sub_capacity
                self.begin(with_rids, key_lo, key_hi, log2_bucket_keys, count)
                self.add(blk_lo, blk_hi)
                rc = lib.lrb_dev_partition_check(C.byref(self.part), C.byref(needed), _stream())
            check(rc)

    def check(self):
        """Synchronises; raises LrbError(LRB_ENOMEM) if the lists overflowed `capacity`. Returns entries needed."""
        needed = C.c_uint64(0)
        check(lib.lrb_dev_partition_check(C.byref(self.part), C.byref(needed), _stream()))
        return int(needed.value)

    def apply(self, table, count=True, search=False, bin_size=1, bins=1, hist=None, sums=None, smem_count=True,
              bucket_lo=0, bucket_hi=None, overwrite=False):
        """smem_count: count through the second-level, shared-memory path (falls back per bucket on key skew).
        bucket_lo/bucket_hi: only these buckets (sums are rewritten by the call that includes the last one).
        overwrite: the count WRITES the table slices of the applied buckets (no memset by the caller; this partition must
        hold all windows of those keys)."""
        mode = (1 if count else 0) | (2 if search else 0) | (4 if (count and smem_count) else 0) | (8 if (count and overwrite) else 0)
        check(lib.lrb_dev_partition_apply_range(C.byref(self.part), mode, bucket_lo, 64 if bucket_hi is None else bucket_hi,
                                                C.c_void_p(table.data_ptr()), bin_size, bins,
                                                C.c_void_p(hist.data_ptr()) if hist is not None else None,
                                                C.c_void_p(sums.data_ptr()) if sums is not None else None, _stream()))

    def search_settings(self, table, settings, hist, sums, bucket_lo=0, bucket_hi=None):
        """Search for several (bin_size, bins) settings at once (lrb_dev_partition_search_settings): hist is [N, W] with
        W = the sum of the bins, each setting's columns after those of the settings before it; hist and sums zeroed by the
        caller as for apply(search=True)."""
        bs, bc = _settings_arrays(settings)
        check(lib.lrb_dev_partition_search_settings(C.byref(self.part), bucket_lo, 64 if bucket_hi is None else bucket_hi,
                                                    C.c_void_p(table.data_ptr()), len(bs), _ptr(bs), _ptr(bc),
                                                    C.c_void_p(hist.data_ptr()), C.c_void_p(sums.data_ptr()), _stream()))

    def search_samples(self, tables, settings, hist, sums, bucket_lo=0, bucket_hi=None):
        """Search against several compact sample tables (dev_table_compact) at once (lrb_dev_partition_search_samples):
        tables[t] is binned with settings[t] = (bin_size, bins) into its column block of hist [N, W]; hist and sums zeroed
        by the caller as for apply(search=True)."""
        bs, bc = _settings_arrays(settings)
        ptrs = (C.c_void_p * max(len(tables), 1))(*[t.data_ptr() for t in tables])
        check(lib.lrb_dev_partition_search_samples(C.byref(self.part), bucket_lo, 64 if bucket_hi is None else bucket_hi,
                                                   ptrs, len(tables), _ptr(bs), _ptr(bc), C.c_void_p(hist.data_ptr()),
                                                   C.c_void_p(sums.data_ptr()), _stream()))

    def search_edges(self, table, edges, hist, sums, bucket_lo=0, bucket_hi=None):
        """Search with bins given by count edges (lrb_dev_partition_search_edges): hist is [N, len(edges) + 1], hist and
        sums zeroed by the caller as for apply(search=True)."""
        e = _edges_array(edges)
        check(lib.lrb_dev_partition_search_edges(C.byref(self.part), bucket_lo, 64 if bucket_hi is None else bucket_hi,
                                                 C.c_void_p(table.data_ptr()), _ptr(e), int(e.size), C.c_void_p(hist.data_ptr()),
                                                 C.c_void_p(sums.data_ptr()), _stream()))


    def search_layout(self, table, compact_tables, blocks, hist, sums, bucket_lo=0, bucket_hi=None):
        """Search with a mixed row (lrb_dev_partition_search_layout): block m (a CovBlock) reads `table` (table=None) or
        compact_tables[slot] (a list, up to 8 compact tables or None, indexed by slot) into its columns of hist [N, W];
        hist and sums zeroed by the caller as for apply(search=True)."""
        arr, keep, _ = _layout_blocks(blocks)
        tables = list(compact_tables or [])
        if len(tables) > _lib.MAX_SAMPLE_TABLES:
            raise _lib.LrbError(_lib.LRB_EINVAL, f"at most {_lib.MAX_SAMPLE_TABLES} compact tables (got {len(tables)})")
        ptrs = (C.c_void_p * _lib.MAX_SAMPLE_TABLES)(*[t.data_ptr() if t is not None else None for t in tables])
        check(lib.lrb_dev_partition_search_layout(C.byref(self.part), bucket_lo, 64 if bucket_hi is None else bucket_hi,
                                                  C.c_void_p(table.data_ptr()) if table is not None else None, ptrs, arr, len(keep),
                                                  C.c_void_p(hist.data_ptr()), C.c_void_p(sums.data_ptr()), _stream()))


class CovBlock(collections.namedtuple("CovBlock", "table bin_size bins edges", defaults=(None, None, None, None))):
    """One block of a mixed coverage row: table=None reads the context's own table, table=t sample slot t (at the file
    level, runners_utils.run_15mer_vecs_layout: table_paths[t]); binned by bin_size= and bins= (-bs / -bc) or by edges=
    (strictly increasing counts, the first >= 2)."""
    __slots__ = ()


def _layout_blocks(layout):
    """(lrb_cov_block array, the edge arrays it points into, the blocks' widths) of a list of CovBlock, refused (LRB_EINVAL) as
    the library refuses it: 1 to 8 blocks, table None or a slot in [0, 8), edges or (bin_size >= 1, bins in [1, MAX_BINS]),
    no block twice, the row at most MAX_BINS wide."""
    blocks = list(layout)
    if not 1 <= len(blocks) <= _lib.MAX_COV_SETTINGS:
        raise _lib.LrbError(_lib.LRB_EINVAL, f"the number of blocks must be in [1, {_lib.MAX_COV_SETTINGS}] (got {len(blocks)})")
    arr = (_lib.CovBlockC * len(blocks))()
    keep, widths, seen = [], [], {}
    for m, b in enumerate(blocks):
        if not isinstance(b, CovBlock):
            raise _lib.LrbError(_lib.LRB_EINVAL, f"block {m} is not a CovBlock (got {b!r})")
        t = -1 if b.table is None else int(b.table)
        if b.table is not None and not 0 <= t < _lib.MAX_SAMPLE_TABLES:
            raise _lib.LrbError(_lib.LRB_EINVAL, f"table must be None (the context's table) or a slot in [0, {_lib.MAX_SAMPLE_TABLES}) "
                                                 f"(block {m}: got {b.table})")
        if b.edges is not None:
            if b.bin_size is not None or b.bins is not None:
                raise _lib.LrbError(_lib.LRB_EINVAL, f"block {m}: give edges or (bin_size, bins), not both")
            e = _edges_array(b.edges)
            keep.append(e)
            arr[m] = _lib.CovBlockC(t, 1, 1, 1, e.ctypes.data if e.size else None, int(e.size))
            key, width = (t, "edges", tuple(e.tolist())), int(e.size) + 1
        else:
            if b.bin_size is None or b.bins is None:
                raise _lib.LrbError(_lib.LRB_EINVAL, f"block {m}: give edges or both bin_size and bins")
            s_, n_ = int(b.bin_size), int(b.bins)
            if not 1 <= s_ < 2 ** (8 * C.sizeof(C.c_long) - 1):
                raise _lib.LrbError(_lib.LRB_EINVAL, f"bin_size must be >= 1 (block {m}: got {s_})")
            if not 1 <= n_ <= _lib.MAX_BINS:
                raise _lib.LrbError(_lib.LRB_EINVAL, f"bins must be in [1, {_lib.MAX_BINS}] (block {m}: got {n_})")
            keep.append(None)
            arr[m] = _lib.CovBlockC(t, 0, s_, n_, None, 0)
            key, width = (t, s_, n_), n_
        if key in seen:
            raise _lib.LrbError(_lib.LRB_EINVAL, f"block {m} repeats block {seen[key]} (same table, same binning)")
        seen[key] = m
        widths.append(width)
    if sum(widths) > _lib.MAX_BINS:
        raise _lib.LrbError(_lib.LRB_EINVAL, f"the blocks' bins add up to {sum(widths)}, more than {_lib.MAX_BINS}")
    return arr, keep, widths


def _edges_array(edges):
    """Count edges as a u32 array, refused (LRB_EINVAL) as the library refuses them: at most MAX_BINS - 1 values, strictly
    increasing, the first >= 2."""
    e = [int(x) for x in edges]
    if len(e) > _lib.MAX_BINS - 1:
        raise _lib.LrbError(_lib.LRB_EINVAL, f"the number of edges must be in [0, {_lib.MAX_BINS - 1}] (got {len(e)})")
    if e and e[0] < 2:
        raise _lib.LrbError(_lib.LRB_EINVAL, f"the first edge must be >= 2, so that counts 0 and 1 stay in bin 0 (got {e[0]})")
    for i in range(1, len(e)):
        if e[i] <= e[i - 1]:
            raise _lib.LrbError(_lib.LRB_EINVAL, f"edges must be strictly increasing (edge {i} = {e[i]} after edge {i - 1} = {e[i - 1]})")
    if e and e[-1] > 0xFFFFFFFF:
        raise _lib.LrbError(_lib.LRB_EINVAL, f"edges are u32 counts (got {e[-1]})")
    return np.array(e, dtype=np.uint32)


def dev_table_compact(table, out=None):
    """Compact form of a full-layout table (a 2^30-entry device tensor): its canonical rows, 2^29 entries
    (lrb_dev_table_compact).  Returns `out` (allocated on the table's device when None)."""
    if out is None:
        out = table.new_empty(_lib.COMPACT_ENTRIES)
    check(lib.lrb_dev_table_compact(C.c_void_p(table.data_ptr()), C.c_void_p(out.data_ptr()), _stream()))
    return out


def read_table_canonical(path, row_lo=0, row_hi=_lib.TABLE_ENTRIES >> 16):
    """Canonical rows [row_lo, row_hi) of a 15mers-counts file as u32[(row_hi - row_lo) * 2^15] (host; no device)."""
    out = np.empty((int(row_hi) - int(row_lo)) << 15, dtype=np.uint32)
    check(lib.lrb_table_read_canonical(os.fsencode(path), int(row_lo), int(row_hi), _ptr(out)))
    return out


def _settings_arrays(settings):
    """(bin_sizes as C long, bins as C int) arrays of a list of (bin_size, bins) settings"""
    settings = [(int(s), int(b)) for s, b in settings]
    return (np.array([s for s, _ in settings], dtype=np.dtype(f"i{C.sizeof(C.c_long)}")),
            np.array([b for _, b in settings], dtype=np.int32))


def dev_table15_partitioned(dr, ws, table, do_count=True, bin_size=1, bins=1, hist=None, sums=None, blk_lo=0, blk_hi=None,
                            key_lo=0, key_hi=_lib.TABLE_ENTRIES, log2_bucket_keys=24, smem_count=True):
    """One-shot: partition the windows of [blk_lo, blk_hi) x [key_lo, key_hi), then count and/or search per bucket."""
    search = hist is not None
    ws.build(search, blk_lo, blk_hi, key_lo, key_hi, log2_bucket_keys, count=do_count and smem_count)
    ws.apply(table, do_count, search, bin_size, bins, hist, sums, smem_count=smem_count)


def dev_format_composition(counts, read_len, n_reads, k, text):
    check(lib.lrb_dev_format_composition(C.c_void_p(counts.data_ptr()), C.c_void_p(read_len.data_ptr()), n_reads, k,
                                         C.c_void_p(text.data_ptr()), _stream()))


def dev_format_coverage(hist, sums, n_reads, bins, text):
    check(lib.lrb_dev_format_coverage(C.c_void_p(hist.data_ptr()), C.c_void_p(sums.data_ptr()), n_reads, bins,
                                      C.c_void_p(text.data_ptr()), _stream()))


def kmer_lut(k):
    lut = np.zeros(4 ** k, dtype=np.uint16)
    width = lib.lrb_kmer_lut(k, _ptr(lut))
    return lut, width
