/*
 * lrbinner_b200.h — C ABI of the B200-native LRBinner profile stage (liblrb200.so).
 *
 * Plain C: pointers and sizes only, no torch / C++ types.  All functions return 0 on success and a
 * non-zero LRB_E* code on failure; lrb_last_error() gives the message of the calling thread's last
 * failure.  The library is thread-compatible (one context per thread), not thread-safe.
 *
 * Reference interfaces replaced (paths relative to the LRBinner repository):
 *   lrb_count_kmers    <- `count-kmers <in> <out> <k> <threads>`        mbcclr_utils/count-kmers.cpp:189-218
 *                         launched by run_kmers()                       mbcclr_utils/runners_utils.py:78-85
 *   lrb_count_15mers   <- `count-15mers <in> <out> <threads>`           mbcclr_utils/count-15mers.cpp:97-123
 *                         launched by run_15mer_counts()                mbcclr_utils/runners_utils.py:88-95
 *   lrb_search_15mers  <- `search-15mers <tbl> <in> <out> <bs> <bc> <t>` mbcclr_utils/search-15mers.cpp:121-157
 *                         launched by run_15mer_vecs()                  mbcclr_utils/runners_utils.py:98-105
 *   lrb_profile        <- the three calls above fused (stages 1_1,1_2,2_1, mbcclr_utils/pipelines.py:269-306)
 *   lrb_reads_*        <- SeqReader / kseq_read                         mbcclr_utils/io_utils.h:133-165, kseq.h:177-218
 *   lrb_dev_composition<- count_kmers()                                 mbcclr_utils/count-kmers.cpp:66-95
 *   lrb_dev_count      <- line_to_kmer_counts()                         mbcclr_utils/kmer_utils.h:114-156
 *   lrb_dev_search     <- line_to_vec()                                 mbcclr_utils/kmer_utils.h:24-87
 *   lrb_table_*        <- writeKmerFile / readKmerFile                  mbcclr_utils/kmer_utils.h:89-112
 *   lrb_format_*       <- std::to_string(double) row emitters           count-kmers.cpp:110-118, search-15mers.cpp:35-48
 */
#ifndef LRBINNER_B200_H
#define LRBINNER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRB_OK 0
#define LRB_EINVAL 1   /* bad argument */
#define LRB_EIO 2      /* file could not be opened / written */
#define LRB_ECUDA 3    /* CUDA runtime error (also: no device) */
#define LRB_ENOMEM 4
#define LRB_EFORMAT 5  /* malformed table file */

#define LRB_TABLE_ENTRIES (1ull << 30) /* 4^15, count-15mers.cpp:99 */
#define LRB_TILE_BLOCKS 256            /* 32-slot blocks of one read per warp tile */
#define LRB_MAX_BINS 4096              /* coverage histogram width accepted by lrb_dev_search */
#define LRB_MAX_COV_SETTINGS 8         /* (bin size, bin count) settings binned in one search (*_settings calls) */
#define LRB_MAX_SAMPLE_TABLES 8        /* sample tables searched in one call (*_samples calls) and sample slots of a context */

int lrb_version(void);
const char* lrb_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * Packed read set (host side).  Layout: DESIGN.md "Data layout in HBM" / csrc/lane_core.cuh.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrb_reads lrb_reads;

typedef struct {
    uint64_t n_reads;      /* N */
    uint64_t n_blocks;     /* 32-slot blocks in the stream */
    uint64_t n_tiles;      /* warp tiles (<= LRB_TILE_BLOCKS blocks of one read each) */
    uint64_t total_bases;  /* L = sum of read lengths */
    const uint32_t* codes;     /* 2*n_blocks + 2 words, 2-bit codes, first slot in the top bit pair */
    const uint32_t* valid;     /* n_blocks + 1 words, bit s = slot s is an in-read uppercase ACGT */
    const uint32_t* read_len;  /* N */
    const uint32_t* read_blk;  /* N+1: first block of read r; read r owns floor(len/32)+1 blocks */
    const uint32_t* tile_read; /* n_tiles */
    const uint32_t* tile_blk;  /* n_tiles: first (global) block of the tile */
} lrb_reads_view;

/* Parse FASTA/FASTQ, plain or gzip, with the record semantics of kseq_read as used by SeqReader
 * (multi-line records, CR stripping, '>'/'@'/'+' leading a line ends the sequence, a bad FASTQ record
 * ends the stream silently, sequence cut at the first NUL).  A missing/unreadable file yields an EMPTY
 * read set and LRB_OK, like the tools (SURVEY.md section 4).  `threads` parallelises the 2-bit packing. */
int lrb_reads_from_file(const char* path, int threads, lrb_reads** out);
/* Concatenated ASCII bases + offsets[n_reads+1] (read r = bases[offsets[r], offsets[r+1])). */
int lrb_reads_from_ascii(const char* bases, const uint64_t* offsets, uint64_t n_reads, int threads, lrb_reads** out);
/* Layout only (no bases): builds read_blk / tile arrays for given lengths and allocates zeroed
 * codes/valid — used when the stream is produced on the device (synthetic generator). */
int lrb_reads_from_lengths(const uint32_t* lengths, uint64_t n_reads, lrb_reads** out);
int lrb_reads_view_get(const lrb_reads* r, lrb_reads_view* view);  /* host pointers */
/* Copy read i back out as ASCII from the packed form ('A','C','T','G' by code; lossy for non-ACGT). */
int lrb_reads_unpack(const lrb_reads* r, uint64_t i, char* dst, uint64_t cap);
/* (Re)build the list of validity exceptions from the current `valid` words: the blocks whose valid word is not the
 * one implied by the read length alone (every in-read slot an uppercase ACGT).  The file/ASCII constructors do this
 * while packing; call it after filling codes/valid of a lrb_reads_from_lengths layout by hand.  With the list in
 * place lrb_profile_host ships only codes + exceptions (0.25 B/base) and rebuilds `valid` on the device.
 * *n_exceptions (may be NULL) receives the list length. */
int lrb_reads_index_valid(lrb_reads* r, int threads, uint64_t* n_exceptions);
/* The current exception list (host pointers owned by `r`; *n = 0 and NULLs when none was built):
 * valid[blk[i]] == word[i] != the word implied by the read length, blk ascending. */
int lrb_reads_exceptions(const lrb_reads* r, const uint32_t** blk, const uint32_t** word, uint64_t* n);
/* Reads [read_lo, read_hi) of `r` as a read set of its own (index arrays rebased to read 0 / block 0).  The packed stream
 * is shared with `r`, which must outlive the slice.  This is how the host pipeline forms device shards and batches. */
int lrb_reads_slice(const lrb_reads* r, uint64_t read_lo, uint64_t read_hi, lrb_reads** out);
void lrb_reads_free(lrb_reads* r);

/* Segment reader: the records of a FASTA/FASTQ file (plain or gzip, same semantics as lrb_reads_from_file) as a sequence of
 * read sets of bounded size, so that host memory does not grow with the file and no read set reaches the 2^32-block limit
 * of one lrb_reads.  A SEGMENT is a contiguous run of whole records of at most `segment_bases` bases (a longer record forms
 * a segment on its own) and always below 2^32 blocks; the concatenated segments are exactly lrb_reads_from_file's read
 * set.  The file is read in chunks (plain files with pread, never mapped whole), so one segment needs its packed stream
 * (0.375 B/base) + two chunks + one record.
 * segment_bases = 0: automatic — the bases whose stream plus the rows of a fused k = 5 / 32-bin profile (2180 B per read,
 * counted as 2.18 B/base at 1 kb per read) fit half of MemAvailable at open time, capped 2^28 blocks below the block
 * limit; LRB_SEGMENT_BASES=n overrides it.  A missing or unreadable file is an empty stream.
 * lrb_reader_next: the next segment as an ordinary read set (exception list built; free with lrb_reads_free), or *out =
 * NULL at the end.  lrb_reader_rewind: start again from the first record.  lrb_reader_tell: reads, bases and segments
 * delivered since open / rewind; *at_end = 1 once no record is left (any argument may be NULL). */
typedef struct lrb_reader lrb_reader;
int lrb_reader_open(const char* path, int threads, uint64_t segment_bases, lrb_reader** out);
int lrb_reader_next(lrb_reader* reader, lrb_reads** out);
int lrb_reader_rewind(lrb_reader* reader);
int lrb_reader_tell(const lrb_reader* reader, uint64_t* reads, uint64_t* bases, uint64_t* segments, int* at_end);
void lrb_reader_close(lrb_reader* reader);

/* ------------------------------------------------------------------------------------------------
 * Device-pointer level (the kernels).  All pointers are DEVICE pointers; `stream` is a cudaStream_t
 * passed as void* (NULL = default stream).  Calls are asynchronous on that stream.
 * ---------------------------------------------------------------------------------------------- */

/* count_kmers (count-kmers.cpp:66-95): counts[N*P] += raw canonical k-mer counts, P = 32/136/512 for
 * k = 3/4/5.  counts must be zeroed by the caller (the call accumulates). EVERY byte of a read takes part
 * (no ACGT check), total windows per read = max(0, len-k+1). Restricted to tiles [tile_lo, tile_hi). */
int lrb_dev_composition(const lrb_reads_view* dev, int k, uint32_t* counts, uint64_t tile_lo, uint64_t tile_hi,
                        void* stream);

/* line_to_kmer_counts (kmer_utils.h:114-156) over blocks [blk_lo, blk_hi): for every valid 15-mer
 * window increments table[c] where c is the member of {val, revcomp(val)} with bit 15 clear, if
 * key_lo <= c < key_hi (key-space shard; pass 0, 2^30 for everything).  lrb_dev_mirror then makes
 * table[x] = table[revcomp(x)] for every x with bit 15 set in [0, 2^30), which yields exactly the
 * reference table (both strands incremented per window => T[x] == T[rc(x)]).  u32 wrap-around. */
int lrb_dev_count(const lrb_reads_view* dev, uint32_t* table, uint64_t blk_lo, uint64_t blk_hi,
                  uint32_t key_lo, uint32_t key_hi, void* stream);
int lrb_dev_mirror(uint32_t* table, void* stream);

/* Abundance spectrum of the table (the reference has no counterpart: it never reads the table as a distribution).
 * Reads only the bit-15-clear keys in [key_lo, key_hi) — one key per {x, revcomp(x)} pair, 2 GiB for the whole table —
 * so neither a mirror nor a complete key space is needed (a key-sharded table works as it is).  Accumulates into
 * spectrum[max_count + 3] u64 (device; the caller zeroes it once):
 *   spectrum[c]   += keys with T == c, c < max_count     spectrum[max_count]     += keys with T >= max_count
 *   spectrum[max_count + 1] += sum of T over those keys  spectrum[max_count + 2]  = max(itself, largest T in the range)
 * so spectra of disjoint key ranges added into one buffer equal the spectrum of their union.  The table is not written.
 * 2 <= max_count <= LRB_SPECTRUM_MAX_COUNT; an empty key range does nothing. */
#define LRB_SPECTRUM_MAX_COUNT (1u << 24)
int lrb_dev_table_spectrum(const uint32_t* table, uint32_t key_lo, uint32_t key_hi, uint32_t max_count, uint64_t* spectrum,
                           void* stream);
/* Compact form of a sample table: only its canonical (bit-15-clear) half, 2^29 u32 = 2 GiB, entry i holding
 * table[((i >> 15) << 16) | (i & 0x7FFF)].  The multi-table search reads sample tables only at bit-15-clear keys, so it
 * takes them in this form.  `table` is a full-layout 2^30-entry table (the other half need not be mirrored). */
#define LRB_COMPACT_ENTRIES (1ull << 29)
int lrb_dev_table_compact(const uint32_t* table, uint32_t* compact, void* stream);
/* lrb_dev_table_spectrum of a whole compact table (lrb_dev_table_compact): entry i of the compact table is read where the
 * full form reads canonical key i, so the spectrum equals that of the full-layout table it was taken from.  Same layout,
 * accumulate-into contract and max_count range as lrb_dev_table_spectrum; `compact` must be 16-byte aligned. */
int lrb_dev_compact_spectrum(const uint32_t* compact, uint32_t max_count, uint64_t* spectrum, void* stream);

/* Multi-GPU table exchange helpers (the reference has no counterpart: it is single-process; SURVEY.md 8e).
 * lrb_dev_copy2d: pitched device-to-device copy on the copy engines; src may be a peer GPU's table mapped into this
 * process (rows of 2^15 bit-15-clear entries, pitch 2^16 entries).  lrb_dev_add_planes: dst rows (pitched) += the sum of
 * n_planes staged copies of those rows (contiguous planes of rows x width_words); 16-byte aligned. */
int lrb_dev_copy2d(void* dst, uint64_t dpitch, const void* src, uint64_t spitch, uint64_t width_bytes, uint64_t height, void* stream);
int lrb_dev_add_planes(uint32_t* dst, uint64_t dst_pitch_words, const uint32_t* src, uint64_t plane_words, int n_planes,
                       uint32_t width_words, uint32_t rows, void* stream);

/* valid[] of `dev` from the read lengths alone (all in-read slots valid, padding slots invalid), then
 * valid[exc_blk[i]] = exc_valid[i] for the n_exc exception blocks (device arrays; may be NULL when n_exc == 0). */
int lrb_dev_fill_valid(const lrb_reads_view* dev, const uint32_t* exc_blk, const uint32_t* exc_valid, uint64_t n_exc,
                       void* stream);

/* line_to_vec (kmer_utils.h:24-87): hist[N*bins] += bucket counts, sums[N] += valid windows, for the
 * reads of tiles [tile_lo, tile_hi).  With key range [0, 2^30) every valid window looks up table[val]
 * (forward key; the table must be mirrored).  With a narrower range (key-sharded search) only windows
 * whose bit-15-clear key c lies in [key_lo, key_hi) are bucketed, through table[c] (no mirror needed);
 * summing hist/sums over a partition of the key space gives the full result.
 * hist/sums must be zeroed by the caller. */
int lrb_dev_search(const lrb_reads_view* dev, const uint32_t* table, long bin_size, int bins, uint32_t* hist,
                   uint32_t* sums, uint64_t tile_lo, uint64_t tile_hi, uint32_t key_lo, uint32_t key_hi, void* stream);

/* L2-resident variant of count and search (csrc/partition.cu).  The valid windows whose bit-15-clear key lies
 * in [key_lo, key_hi) are partitioned ONCE by key >> log2_bucket_keys into at most 64 buckets (key range
 * bucket-aligned, 20 <= log2_bucket_keys <= 25) as lists of 4-byte entries (key inside the bucket + read index
 * relative to the entry's 8192-slot step); lrb_dev_partition_apply then walks the buckets and applies each list to
 * the table slice while that slice is resident in L2:
 *   mode 1  count : table[key] += 1                    (== lrb_dev_count; mirror separately)
 *   mode 2  search: hist/sums through table[key]       (== lrb_dev_search on bit-15-clear keys; no mirror needed);
 *                   sums[r] is rewritten as the sum of hist row r for r < n_reads (hist and sums must have been
 *                   zeroed together and only ever updated by lrb_dev_search / this call)
 *   mode 3  both  : per bucket count, then search      (single-GPU fused path)
 *   mode bit 2 (4): count through shared memory.  When `sub` is given (sub_capacity u16 entries, >= ~1.3 x capacity; 2 x is
 *                   comfortable) add() also splits every bucket list of the chunk into 2-byte lists per 2^15-key
 *                   sub-slice, whose counters then live in one SM's shared memory.  Entries that find their list's fixed share
 *                   full (hot keys of low-complexity reads) go to a spill area (1/8 of the capacity) and are applied with
 *                   warp-aggregated REDs; only if that fills up does a bucket fall back to the L2-atomic kernel.  Same table
 *                   either way.  Ignored without `sub`.
 *   mode bit 3 (8): count WRITES: the table slices of the applied buckets need not be zeroed by the caller (the shared-memory
 *                   path stores its counters instead of adding them — no 4 GiB memset, no read of the slice; the L2-atomic path
 *                   zeroes the slices itself first).  Only for a partition that holds ALL windows of those keys (one apply per
 *                   table); accumulating several partitions into one table (batches, chunks applied apart) needs the adding form.
 * begin() resets the lists; add() appends the windows of blocks [blk_lo, blk_hi) as one chunk (up to 64 chunks,
 * e.g. one per host-to-device copy so partitioning overlaps the transfer); build() = begin + one add.  A
 * partition can be applied several times (count, exchange tables between GPUs, then search).  Everything is
 * asynchronous on `stream`; sizes are computed on the device and the list layout is deterministic.  If the lists
 * would exceed `capacity` the chunk is dropped and a device flag is raised: apply then does nothing and
 * lrb_dev_partition_check (synchronises) returns LRB_ENOMEM and the number of entries needed.
 * capacity >= total number of slots can never overflow.
 * blk_read[n_blocks] = read index of every block (lrb_dev_fill_blk_read).  The caller owns the device buffers and
 * fills keys/small/steps/capacity/step_capacity; the library fills the rest.  `steps` holds the per-step tables:
 * lrb_partition_steps_words(step_capacity) u32 words, step_capacity >= lrb_partition_step_capacity(n_blocks,
 * number of add() calls).  Bit-identical to the direct kernels. */
#define LRB_PART_MAX_BUCKETS 64
#define LRB_PART_MAX_CHUNKS 64
#define LRB_PART_MAX_GROUPS 8192
#define LRB_PART_SMALL_U64 16384
typedef struct {
    uint32_t* keys;                /* device, capacity entries */
    unsigned long long* small;     /* device scratch, LRB_PART_SMALL_U64 u64 */
    uint32_t* steps;               /* device, lrb_partition_steps_words(step_capacity) u32 */
    uint16_t* sub;                 /* device, sub_capacity u16 (optional: second-level lists of the shared-memory count) */
    uint64_t capacity;
    uint64_t sub_capacity;
    uint64_t step_capacity;
    uint64_t steps_used, n_reads;
    int n_buckets, shift, has_rids, n_chunks;
    uint32_t key_lo, key_hi;
    uint32_t chunk_step0[LRB_PART_MAX_CHUNKS], chunk_nsteps[LRB_PART_MAX_CHUNKS];
    int l2_enabled;                /* second-level lists are being built (filled by begin()) */
    uint32_t l2_ncta, l2_C3;
    uint64_t l2_seg0, l2_span;
    uint64_t l2_cells0;            /* per-(bucket, sub-slice) segment table (offsets, capacities, sampled histogram), u16 offset in `sub` */
    uint64_t l2_spill0;            /* spill area of the second level (hot keys), u16 offset in `sub` */
    uint32_t l2_spill_cap;         /* ... and its capacity in entries */
} lrb_partition;
uint64_t lrb_partition_step_capacity(uint64_t n_blocks, int max_chunks);
uint64_t lrb_partition_steps_words(uint64_t step_capacity);
int lrb_dev_fill_blk_read(const lrb_reads_view* dev, uint32_t* blk_read, void* stream);
int lrb_dev_partition_begin(lrb_partition* part, int with_rids, uint32_t key_lo, uint32_t key_hi, int log2_bucket_keys,
                            void* stream);
int lrb_dev_partition_add(const lrb_reads_view* dev, const uint32_t* blk_read, uint64_t blk_lo, uint64_t blk_hi,
                          lrb_partition* part, void* stream);
int lrb_dev_partition_build(const lrb_reads_view* dev, const uint32_t* blk_read, int with_rids, uint64_t blk_lo,
                            uint64_t blk_hi, uint32_t key_lo, uint32_t key_hi, int log2_bucket_keys, lrb_partition* part,
                            void* stream);
int lrb_dev_partition_check(const lrb_partition* part, uint64_t* needed, void* stream);
int lrb_dev_partition_apply(const lrb_partition* part, int mode, uint32_t* table, long bin_size, int bins, uint32_t* hist,
                            uint32_t* sums, void* stream);
/* The same for the buckets [bucket_lo, bucket_hi) only (clamped): a multi-GPU driver exchanges the table slice of
 * bucket b+1 (keys [key_lo + (b+1) << log2_bucket_keys, ...)) while bucket b is searched.  sums are rewritten by the call
 * that includes the last bucket. */
int lrb_dev_partition_apply_range(const lrb_partition* part, int mode, int bucket_lo, int bucket_hi, uint32_t* table,
                                  long bin_size, int bins, uint32_t* hist, uint32_t* sums, void* stream);
/* Search for n coverage settings at once (no reference counterpart: the reference runs search-15mers once per -bs/-bc).
 * Every window's count is gathered once and binned by each setting (bin_sizes[m], bins[m]) into rows of W = sum of bins[m]
 * words: setting 0's bins, then setting 1's, ...  Row r of setting m is hist[r*W + sum_{j<m} bins[j] + b]; sums[r] (the
 * read's valid windows, the same for every setting) is rewritten by the call that includes the last bucket, as in mode 2.
 * LRB_EINVAL unless 1 <= n <= LRB_MAX_COV_SETTINGS, every bin_size >= 1, every bins in [1, LRB_MAX_BINS], W <= LRB_MAX_BINS
 * and no (bin_size, bins) pair repeats.  n = 1 is mode 2 of lrb_dev_partition_apply_range, row for row. */
int lrb_dev_partition_search_settings(const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* table, int n,
                                      const long* bin_sizes, const int* bins, uint32_t* hist, uint32_t* sums, void* stream);
/* Search the partition's reads against n compact sample tables at once (differential coverage; no reference counterpart:
 * the reference runs search-15mers once per table).  compact_tables is a HOST array of n device pointers to
 * lrb_dev_table_compact tables; table t is binned with (bin_sizes[t], bins[t]) into rows of W = sum of bins[t] words:
 * table 0's bins, then table 1's, ...  Row r of table t is hist[r*W + sum_{j<t} bins[j] + b] and equals row r of a
 * single-table search with that table's full layout, for every table that is symmetric (T[x] == T[revcomp x], as every
 * counted table is): like every partitioned search, only the bit-15-clear member of each {x, revcomp x} pair is read.
 * sums[r] (the read's valid windows, the same for every table) is rewritten by the call that includes the last bucket.
 * One walk over the lists per table.  LRB_EINVAL unless 1 <= n <= LRB_MAX_SAMPLE_TABLES, every bin_size >= 1, every
 * bins in [1, LRB_MAX_BINS], W <= LRB_MAX_BINS, no (table pointer, bin_size, bins) repeats, the partition has read ids
 * and starts at a bucket boundary. */
int lrb_dev_partition_search_samples(const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* const* compact_tables,
                                     int n, const long* bin_sizes, const int* bins, uint32_t* hist, uint32_t* sums, void* stream);
/* Search with coverage bins given by count edges (no reference counterpart): edges is a HOST array of n_edges strictly
 * increasing thresholds t_0 < ... < t_{n-1}, t_0 >= 2, and a window whose 15-mer is counted c times goes to bin
 * #{i : t_i <= c} (searchsorted(edges, c, side="right")) of rows of B = n_edges + 1 words.  Counts 0 and 1 always go to
 * bin 0, as in the reference's rule; edges {2, 3, ..., B} equal -bs 1 -bc B and no edges equal -bc 1.  Bucket range and
 * sums as in lrb_dev_partition_search_settings.  LRB_EINVAL unless 0 <= n_edges <= LRB_MAX_BINS - 1, edges is non-NULL
 * when n_edges > 0, the edges are strictly increasing and t_0 >= 2, and the partition has read ids. */
int lrb_dev_partition_search_edges(const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* table,
                                   const uint32_t* edges, int n_edges, uint32_t* hist, uint32_t* sums, void* stream);
/* One block of a mixed coverage row: the table it reads and how it bins the count.  table -1 is the full-layout table
 * (the context's own table); 0..7 is compact table / sample slot t (at the file level: table_paths[t]).  by_edges 0 bins by
 * (bin_size, bins) as -bs / -bc do; by_edges 1 bins by edges[n_edges] as lrb_dev_partition_search_edges does (n_edges = 0
 * is one bin). */
typedef struct {
    int table;
    int by_edges;
    long bin_size;
    int bins;
    const uint32_t* edges;
    int n_edges;
} lrb_cov_block;
/* Search with a mixed coverage row (no reference counterpart): up to LRB_MAX_COV_SETTINGS blocks, each on the full-layout
 * `table` or on compact_tables[t] (a HOST array of LRB_MAX_SAMPLE_TABLES device pointers, NULL where unused; may be NULL
 * when no block reads a slot), each binned by (bin_size, bins) or by edges (HOST arrays).  Rows of W = the blocks' bins
 * together, block 0's bins first, in the caller's order; block m of row r equals row r of the single-block search of its
 * table and binning (for compact tables: of every symmetric table, as in lrb_dev_partition_search_samples).  The lists are
 * walked once per distinct table, and every block of that table is binned from the one gather.  A layout the settings,
 * samples or edges search could take runs exactly as that search does.  Bucket range and sums as in
 * lrb_dev_partition_search_settings.  LRB_EINVAL unless 1 <= n <= LRB_MAX_COV_SETTINGS, every table is -1 or in
 * [0, LRB_MAX_SAMPLE_TABLES), every block passes the checks of its binning, W <= LRB_MAX_BINS, no block repeats (same table
 * and binning), the tables the blocks read are non-NULL, the partition has read ids and, when a block reads a compact
 * table, starts at a bucket boundary. */
int lrb_dev_partition_search_layout(const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* table,
                                    const uint32_t* const* compact_tables, const lrb_cov_block* blocks, int n, uint32_t* hist,
                                    uint32_t* sums, void* stream);

/* Pack ASCII on the device: bases[] (device, concatenated) -> codes/valid of `dev` (layout prebuilt). */
int lrb_dev_pack_ascii(const lrb_reads_view* dev, const char* bases, const uint64_t* offsets, void* stream);

/* Text epilogue on the device: fixed-width "%f" rows, byte-identical to the tools' output.
 *   composition: N rows of P values "d.dddddd " then '\n'            (count-kmers.cpp:110-118)
 *   coverage   : N rows of B values separated by ' ', then '\n'      (search-15mers.cpp:35-48)
 * value = count/max(1,total) resp. count/sum with the <1e-4 -> 0 rule (kmer_utils.h:75-84). */
int lrb_dev_format_composition(const uint32_t* counts, const uint32_t* read_len, uint64_t n_reads, int k, char* text,
                               void* stream);
/* The same values as float64 on the device — out[N*width] = float("%f" text of count/denominator), i.e. exactly what
 * stage 3_1 (pipelines.py:310-330) parses back out of com_profs / cov_profs and ae_utils.make_data_loader
 * (ae_utils.py:19-32) consumes.  k = 3/4/5: composition (denom = read_len, width = 32/136/512);
 * k = 0: coverage (denom = sums, width = bins, `< 1e-4 -> 0` rule). */
int lrb_dev_profile_values(const uint32_t* counts, const uint32_t* denom, uint64_t n_reads, int width, int k, double* out,
                           void* stream);
int lrb_dev_format_coverage(const uint32_t* hist, const uint32_t* sums, uint64_t n_reads, int bins, char* text,
                            void* stream);

/* Synthetic ONT/HiFi-like reads generated directly into the packed stream (bench/test input only).
 * meta[4*r+0..3] = genome id, start, flags (bit0 reverse strand, bit1 lowercase read), reserved.
 * genome g has glen[g] bases, base i = hash(seed,g,i).  thresholds are u32 fractions of 2^32. */
typedef struct {
    uint64_t seed;
    uint32_t n_genomes;
    uint32_t sub_thr, ins_thr, del_thr, n_thr;
    uint64_t read_base;   /* global index of read 0 (lets shards of one community be generated apart) */
} lrb_synth_params;
int lrb_dev_synth(const lrb_reads_view* dev, const lrb_synth_params* p, const uint32_t* glen, const uint32_t* meta,
                  void* stream);
/* The same generator on the host, writing ASCII (tests feed this to the oracle). */
int lrb_synth_host(const lrb_synth_params* p, const uint32_t* glen, const uint32_t* meta, const uint32_t* lengths,
                   uint64_t n_reads, const uint64_t* offsets, char* bases);

/* ------------------------------------------------------------------------------------------------
 * Host-buffer level: owns device memory, streams and the H2D/D2H pipeline on one GPU.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lrb_ctx lrb_ctx;
int lrb_ctx_create(int device, lrb_ctx** out);
/* One context driving n_devices GPUs from this process (devices[] = CUDA ordinals, NULL = 0..n-1).  devices[0] is
 * the primary: it ends up with the complete table (lrb_ctx_table_save / _load act on it).  lrb_profile_host then shards
 * the reads over the devices (contiguous ranges, so row i is still read i), every device counts its own reads into a
 * private table, the tables are summed over NVLink peer memory by the copy engines, and every device searches its own
 * reads: SURVEY.md 8(e) plan "read-sharded" — the one that won the three-way measurement (DESIGN.md section 6). */
int lrb_ctx_create_multi(const int* devices, int n_devices, lrb_ctx** out);
int lrb_ctx_device_count(const lrb_ctx* ctx);
void lrb_ctx_destroy(lrb_ctx* ctx);

/* Whole profile stage for one read set held in (pinned) HOST memory:
 *   H2D(packed reads, chunked) || composition + key partition per chunk -> count + search per bucket (L2-resident)
 *   -> mirror -> D2H(results; composition rows return while the table passes run).
 * comp_counts[N*P] (P from k), cov_hist[N*bins], cov_sums[N] are HOST buffers (may be NULL to skip the
 * corresponding phase).  If table_host != NULL the 4 GiB table is copied back as well.
 * flags: LRB_PROFILE_USE_LOADED_TABLE — skip the count phase and search the table already in the context;
 *        LRB_PROFILE_KEEP_TABLE — count even when neither the search nor table_host asks for it (lrb_ctx_table_save follows);
 *        LRB_PROFILE_ADD_TO_TABLE — count, ADDING this read set's windows to the complete table already in the context
 *        (after a count or lrb_ctx_table_load) instead of starting from zero: tables of read sets profiled one after another
 *        this way equal the table of their union (segments of one file, lrb_reader_*).  Needs a table; on any error the
 *        context holds no table afterwards (it may be partly added to).
 * Bounded device memory: a read set whose working set (8.6 B per base of lists beside the 4 GiB table) does not fit is
 * processed in BATCHES — the table accumulates over the batches, then every batch is shipped and partitioned again for
 * the search — with a one-line notice on stderr; results are identical (tests force this with LRB_BATCH_BASES).  This
 * is the reference's constant-memory behaviour (count-15mers.cpp:75-99: reads stream through a bounded queue). */
#define LRB_PROFILE_USE_LOADED_TABLE 1
#define LRB_PROFILE_KEEP_TABLE 2
#define LRB_PROFILE_ADD_TO_TABLE 4
int lrb_profile_host(lrb_ctx* ctx, const lrb_reads* reads, int k, long bin_size, int bins, uint32_t* comp_counts,
                     uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags);
/* The same with n coverage settings searched in one pass over the table (lrb_dev_partition_search_settings): cov_hist[N*W],
 * W = sum of bins[m], holds for every read setting 0's bins, then setting 1's, ...; cov_sums[N] is shared by all settings.
 * Every flag and part of lrb_profile_host works alongside (composition, count, KEEP / ADD_TO / USE_LOADED_TABLE, batches,
 * several devices); lrb_profile_host is its n = 1 case.  The settings are checked as in lrb_dev_partition_search_settings
 * when coverage is asked for, before any device work; n > 1 under LRB_TABLE_PATH=direct is refused (LRB_EINVAL). */
int lrb_profile_host_settings(lrb_ctx* ctx, const lrb_reads* reads, int k, int n, const long* bin_sizes, const int* bins,
                              uint32_t* comp_counts, uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags);
/* Sample slots: a context holds up to LRB_MAX_SAMPLE_TABLES sample tables beside its own table, each in compact form
 * (lrb_dev_table_compact, 2 GiB) on EVERY device of the context (the multi-device search shards reads, so every device
 * needs every table).  Loading or keeping into a slot replaces what it held; neither touches the context's own table.
 * lrb_ctx_sample_table_load reads only the canonical rows of a 15mers-counts file (2^14 rows of 128 KiB at a 256 KiB
 * stride: 2 GiB of the 4 GiB); the header and the file size are checked first: missing file LRB_EIO, bad header or size
 * LRB_EFORMAT.  lrb_ctx_sample_table_keep compacts the context's own complete table into the slot (LRB_EINVAL when the
 * context holds none).  lrb_ctx_sample_table_free releases the slot's memory. */
int lrb_ctx_sample_table_load(lrb_ctx* ctx, int slot, const char* path);
int lrb_ctx_sample_table_keep(lrb_ctx* ctx, int slot);
int lrb_ctx_sample_table_free(lrb_ctx* ctx, int slot);
/* Host side of lrb_ctx_sample_table_load: canonical rows [row_lo, row_hi) (row j = entries j 2^16 .. j 2^16 + 2^15 - 1)
 * of a 15mers-counts file into compact[(row_hi - row_lo) 2^15], after the same header and size checks. */
int lrb_table_read_canonical(const char* path, uint32_t row_lo, uint32_t row_hi, uint32_t* compact);
/* lrb_profile_host_settings with coverage against n sample slots instead of the context's table: slot slots[t] binned with
 * (bin_sizes[t], bins[t]) into cov_hist[N*W], W = sum of bins[t], table 0's bins first (lrb_dev_partition_search_samples).
 * The context's own table is not searched (keep it into a slot to search it).  Composition, the count flags
 * (KEEP_TABLE, ADD_TO_TABLE, table_host), batches and several devices work alongside; coverage itself needs no count.
 * LRB_EINVAL before any device work for an empty or out-of-range slot, bad settings, the same (slot, bin_size, bins)
 * twice, and LRB_TABLE_PATH=direct (the direct kernels read only the full-layout table). */
int lrb_profile_host_samples(lrb_ctx* ctx, const lrb_reads* reads, int k, int n, const int* slots, const long* bin_sizes,
                             const int* bins, uint32_t* comp_counts, uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host,
                             int flags);
/* lrb_profile_host with coverage bins given by count edges (lrb_dev_partition_search_edges): cov_hist[N*(n_edges + 1)].
 * Every flag and part of lrb_profile_host works alongside (composition, count, KEEP / ADD_TO / USE_LOADED_TABLE, batches,
 * several devices).  The edges are checked as in lrb_dev_partition_search_edges when coverage is asked for, before any
 * device work; LRB_TABLE_PATH=direct is refused (LRB_EINVAL). */
int lrb_profile_host_edges(lrb_ctx* ctx, const lrb_reads* reads, int k, const uint32_t* edges, int n_edges, uint32_t* comp_counts,
                           uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags);
/* lrb_profile_host with a mixed coverage row (lrb_dev_partition_search_layout): cov_hist[N*W], block 0's bins first; a
 * block reads the context's own table (table -1) or sample slot t.  A block on the context's table needs it counted from
 * these reads, or loaded (USE_LOADED_TABLE / ADD_TO_TABLE), as lrb_profile_host does; a layout of slots alone searches no
 * count and leaves the context's table as it was.  Every flag and part works alongside (composition, count, KEEP / ADD_TO /
 * USE_LOADED_TABLE, batches, several devices).  The blocks are checked as in lrb_dev_partition_search_layout before any
 * device work; an empty slot, a slot block without cov_hist / cov_sums and LRB_TABLE_PATH=direct (unless the layout is one
 * (bin_size, bins) block on the context's table) are refused with LRB_EINVAL. */
int lrb_profile_host_layout(lrb_ctx* ctx, const lrb_reads* reads, int k, const lrb_cov_block* blocks, int n, uint32_t* comp_counts,
                            uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags);
/* How the last lrb_profile_host call ran. */
typedef struct {
    int n_devices;            /* GPUs that took part */
    int n_batches;            /* batches over all devices; == n_devices when everything stayed resident */
    int table_path;           /* 0 direct kernels (LRB_TABLE_PATH=direct), 1 key-partitioned + L2 atomics, 2 + shared-memory count */
    int lists_reused;         /* 1: the search re-used the lists the count built (single batch per device) */
    float wall_ms;            /* host wall clock of the call */
    float exchange_ms;        /* device 0: first to last operation of the table exchange (0 on one GPU) */
    uint64_t batch_bases_max; /* slots of the largest batch */
    float host_plan_ms;       /* host: entry -> devices, tables and batches planned */
    float host_enqueue_ms;    /* host: entry -> device 0's last operation enqueued (the rest of wall_ms is waiting for the device) */
} lrb_run_info;
int lrb_ctx_last_info(const lrb_ctx* ctx, lrb_run_info* info);
/* Device milliseconds (CUDA events) of the last lrb_profile_host call.  The call is a 3-stream pipeline, so the
 * phases overlap: [0] H2D of the packed reads (copy stream) [1] composition + partition until the last chunk is
 * processed (runs beside [0]) [2] table passes (count + search per bucket) [3] mirror [4] direct search (only
 * on the LRB_TABLE_PATH=direct path) [5] result D2H tail [6] the whole call */
int lrb_ctx_last_timings(const lrb_ctx* ctx, float* ms7);
/* page-locked host memory for result buffers of lrb_profile_host (NULL + lrb_last_error on failure) */
void* lrb_pinned_alloc(size_t bytes);
void lrb_pinned_free(void* p);
int lrb_ctx_table_load(lrb_ctx* ctx, const char* path);          /* readKmerFile -> HBM */
int lrb_ctx_table_save(lrb_ctx* ctx, const char* path);          /* HBM -> writeKmerFile format */
/* lrb_dev_table_spectrum over the whole table of the primary device (complete after lrb_profile_host with a count, a
 * multi-device call included, or lrb_ctx_table_load) into spectrum_host[max_count + 3]; synchronous.  LRB_EINVAL when the
 * context holds no table.  The table is left as it is.  No reference counterpart. */
int lrb_ctx_table_spectrum(lrb_ctx* ctx, uint32_t max_count, uint64_t* spectrum_host);
/* The same for sample slot `slot` of the context (lrb_dev_compact_spectrum on the primary device).  LRB_EINVAL for a slot
 * outside [0, LRB_MAX_SAMPLE_TABLES) or an empty slot.  No reference counterpart. */
int lrb_ctx_sample_table_spectrum(lrb_ctx* ctx, int slot, uint32_t max_count, uint64_t* spectrum_host);

/* Launch accounting (csrc/prof.cu).  lrb_prof_launches: kernels this library has launched since it was loaded (always
 * counted; bench.py's gpu_launches).  lrb_prof_enable(1) additionally brackets every launch with CUDA events on the stream
 * it is launched on (and forgets earlier records); after synchronising, lrb_prof_report writes one line per kernel,
 * "name launches total_ms".  This is how bench.py quotes single-kernel durations inside its timed region without a
 * profiler attached.  Returns the previous state. */
uint64_t lrb_prof_launches(void);
int lrb_prof_enable(int on);
int lrb_prof_report(char* buf, size_t cap);

/* ------------------------------------------------------------------------------------------------
 * Host text / file epilogue (multi-threaded, exact "%f").
 * ---------------------------------------------------------------------------------------------- */
/* q = the 6 decimals printf("%f") prints for double(num)/double(den), as an integer in [0, 10^6]
 * (den == 0 is treated as 1: max(1.0,total), count-kmers.cpp:91).  coverage != 0 applies the
 * `< 1e-4 -> 0` rule first (kmer_utils.h:80-83). */
uint32_t lrb_fixed6(uint32_t num, uint32_t den, int coverage);
int lrb_write_composition_txt(const char* path, const uint32_t* counts, const uint32_t* read_len, uint64_t n_reads,
                              int k, int threads);
int lrb_write_coverage_txt(const char* path, const uint32_t* hist, const uint32_t* sums, uint64_t n_reads, int bins,
                           int threads);
/* .npy (float64, C order) holding float(text) for every value: what pipelines.py:313-324 would produce. */
int lrb_write_composition_npy(const char* path, const uint32_t* counts, const uint32_t* read_len, uint64_t n_reads,
                              int k, int threads);
int lrb_write_coverage_npy(const char* path, const uint32_t* hist, const uint32_t* sums, uint64_t n_reads, int bins,
                           int threads);
/* The same four writers for a file written in parts (one segment of rows at a time): the rows go after the `row0` rows
 * already in the file; row0 = 0 creates / truncates it.  The .npy forms rewrite the header with row0 + n_reads rows each
 * time (its size, 128 bytes, does not depend on the shape), so after the last part the file is the one-shot writer's,
 * byte for byte, and so are the text files. */
int lrb_append_composition_txt(const char* path, const uint32_t* counts, const uint32_t* read_len, uint64_t n_reads, int k,
                               int threads, uint64_t row0);
int lrb_append_coverage_txt(const char* path, const uint32_t* hist, const uint32_t* sums, uint64_t n_reads, int bins,
                            int threads, uint64_t row0);
int lrb_append_composition_npy(const char* path, const uint32_t* counts, const uint32_t* read_len, uint64_t n_reads, int k,
                               int threads, uint64_t row0);
int lrb_append_coverage_npy(const char* path, const uint32_t* hist, const uint32_t* sums, uint64_t n_reads, int bins,
                            int threads, uint64_t row0);
int lrb_table_write_file(const char* path, const uint32_t* table);  /* u64 2^30, then 2^30 u32 */
int lrb_table_read_file(const char* path, uint32_t* table);
/* What a spectrum (lrb_dev_table_spectrum layout) implies for the coverage profile with -bs bin_size -bc bins:
 * mass[b] = sum over c of c * n_c * [coverage bin of c == b], i.e. the number of windows that land in bin b summed over
 * all reads, when the table was counted from the same reads that are searched (each canonical pair counted c times
 * is met by c windows, all binned by c).  Keys at or above max_count add their sum to the last bin.  LRB_EINVAL for
 * bin_size < 1 or bins outside [1, LRB_MAX_BINS], and when keys at or above max_count exist but
 * max_count < bin_size * (bins + 1): their bin is then not determined by the spectrum.  No reference counterpart. */
int lrb_spectrum_bin_mass(const uint64_t* spectrum, uint32_t max_count, long bin_size, int bins, uint64_t* mass);
/* The same for coverage bins given by count edges (lrb_dev_partition_search_edges): mass[n_edges + 1], mass[b] = sum over c
 * of c * n_c * [#{i : edges[i] <= c} == b].  Keys at or above max_count add their sum to the last bin.  LRB_EINVAL for
 * edges lrb_dev_partition_search_edges refuses, and when keys at or above max_count exist but max_count is below the last
 * edge: their bin is then not determined by the spectrum.  No reference counterpart. */
int lrb_spectrum_edge_mass(const uint64_t* spectrum, uint32_t max_count, const uint32_t* edges, int n_edges, uint64_t* mass);
/* jellyfish `histo` text of a spectrum: "c n_c\n" for every c in [1, max_count) with n_c > 0, ascending, then
 * "max_count n_over\n" when keys at or above max_count exist.  Counts are of canonical 15-mers (each {x, revcomp(x)}
 * pair once).  No reference counterpart. */
int lrb_write_spectrum_txt(const char* path, const uint64_t* spectrum, uint32_t max_count);

/* canonical k-mer index table of count-kmers (compute_kmer_inds, count-kmers.cpp:38-64); returns P. */
int lrb_kmer_lut(int k, uint16_t* lut /* 4^k */);

/* ------------------------------------------------------------------------------------------------
 * File level: the drop-ins for the three tools (same argument meaning; exit code -> return value).
 * ---------------------------------------------------------------------------------------------- */
int lrb_count_kmers(const char* reads_path, const char* out_txt, int k, int threads);
int lrb_count_15mers(const char* reads_path, const char* out_table, int threads);
int lrb_search_15mers(const char* table_path, const char* reads_path, const char* out_txt, long bin_size, int bins,
                      int threads);
/* lrb_search_15mers for n settings with one table load and one parse: out_txts[m] receives the coverage text of
 * (bin_sizes[m], bins[m]), byte for byte the file lrb_search_15mers writes for that setting; out_npys (may be NULL, or
 * hold NULLs) the matching .npy.  Input larger than one segment is read segment by segment (rows of 4 (W + 1) bytes per
 * read) and every file gets its rows appended in file order.  The arguments are checked before any file or device is
 * touched (LRB_EINVAL as for lrb_profile_host_settings; a NULL path too).  No reference counterpart. */
int lrb_search_15mers_settings(const char* table_path, const char* reads_path, int n, const long* bin_sizes, const int* bins,
                               const char* const* out_txts, const char* const* out_npys, int threads);
/* Differential coverage: the reads against n 15mers-counts files at once, each loaded once into a sample slot (canonical
 * rows only) and the reads parsed once.  Line r of out_txt holds table 0's bins, then table 1's, ... (W = sum of bins[t]
 * values): block t is, byte for byte, line r of lrb_search_15mers(table_paths[t], reads, bin_sizes[t], bins[t]) for every
 * symmetric (counted) table, and the blocks are joined by one space.  out_npy (may be NULL) gets the [N, W] float rows.
 * Input larger than one segment is read segment by segment (rows of 4 (W + 1) bytes per read).  LRB_GPUS is honoured.
 * Arguments are checked before any file or device work (LRB_EINVAL: a NULL path, n, the settings, the same (path, bin_size,
 * bins) twice).  No reference counterpart. */
int lrb_search_15mers_samples(const char* const* table_paths, int n, const long* bin_sizes, const int* bins, const char* reads_path,
                              const char* out_txt, const char* out_npy, int threads);
/* lrb_search_15mers with coverage bins given by count edges (lrb_dev_partition_search_edges): one table load and one parse;
 * out_txt gets rows of n_edges + 1 values written exactly as lrb_search_15mers writes its rows (edges {2, ..., B} give its
 * -bs 1 -bc B file byte for byte), out_npy (may be NULL) the [N, n_edges + 1] float rows.  Input larger than one segment
 * is read segment by segment and the rows are appended in file order.  The arguments are checked before any file or
 * device is touched (LRB_EINVAL as for lrb_profile_host_edges; a NULL path too).  No reference counterpart. */
int lrb_search_15mers_edges(const char* table_path, const char* reads_path, const uint32_t* edges, int n_edges, const char* out_txt,
                            const char* out_npy, int threads);
/* Mixed coverage rows from files: the reads against n_tables 15mers-counts files (1 <= n_tables <= LRB_MAX_SAMPLE_TABLES),
 * each loaded once into a sample slot (canonical rows only; a path listed twice is loaded once), the reads parsed once.
 * Block m reads table_paths[blocks[m].table] (table -1 is refused: there is no context table here) and line r of out_txt
 * is, block after block joined by one space, the line the single-block call (lrb_search_15mers, or
 * lrb_search_15mers_edges) writes for that table and binning, for every symmetric (counted) table.  out_npy (may be NULL)
 * gets the [N, W] float rows.  Input larger than one segment is read segment by segment.  LRB_GPUS is honoured.  Arguments
 * are checked before any file or device work (LRB_EINVAL: a NULL path, n_tables, a table index, the checks of
 * lrb_dev_partition_search_layout, the same (path, binning) twice).  No reference counterpart. */
int lrb_search_15mers_layout(const char* const* table_paths, int n_tables, const char* reads_path, const lrb_cov_block* blocks, int n,
                             const char* out_txt, const char* out_npy, int threads);
/* Abundance spectrum of a 15mers-counts file as lrb_write_spectrum_txt text (loaded on device LRB_DEVICE).  Missing or
 * malformed table file: LRB_EIO / LRB_EFORMAT; no device: LRB_ECUDA.  No reference counterpart. */
int lrb_table_spectrum(const char* table_path, const char* out_txt, uint32_t max_count);
/* Fused stage: parse once, keep reads + table in HBM, write com_profs, cov_profs (and 15mers-counts if
 * write_table) into out_dir/profiles/; write_npy additionally emits com_profs.npy / cov_profs.npy.
 * Input larger than one segment (lrb_reader_open with the budget of the call's rows; a plain file no larger in bytes than
 * the budget is read whole as before): the file-level calls above and below go segment by segment and append the rows —
 * count: one pass adding each segment to the table; search: one pass against the loaded table; fused: pass 1 writes the
 * composition rows and counts, pass 2 reads the file again and writes the coverage rows.  The files are those of a
 * one-segment run, byte for byte; one line on stderr gives the number of segments and passes. */
int lrb_profile(const char* reads_path, const char* out_dir, int k, long bin_size, int bins, int threads,
                int write_table, int write_npy);
/* The same on n_gpus GPUs of this node (devices LRB_DEVICE.. ; n_gpus <= 0: LRB_GPUS from the environment, default 1),
 * byte-identical files.  The three tool drop-ins above and lrb_profile honour LRB_GPUS the same way. */
int lrb_profile_multi(const char* reads_path, const char* out_dir, int k, long bin_size, int bins, int threads, int n_gpus,
                      int write_table, int write_npy);

#ifdef __cplusplus
}
#endif
#endif
