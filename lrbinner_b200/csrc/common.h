// common.h — error plumbing shared by the translation units of liblrb200.so
#pragma once
#include <stdint.h>

#include "../../include/lrbinner_b200.h"

// Records `msg` (printf-style) as the calling thread's last error and returns `code`.
int lrb_set_error(int code, const char* fmt, ...);

#ifdef __CUDACC__
#define LRB_CUDA(expr)                                                                                      \
    do {                                                                                                    \
        cudaError_t lrb_e_ = (expr);                                                                        \
        if (lrb_e_ != cudaSuccess)                                                                          \
            return lrb_set_error(LRB_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(lrb_e_),     \
                                 __FILE__, __LINE__);                                                       \
    } while (0)
#endif

// One kernel launch: always counted, timed with CUDA events on its own stream when lrb_prof_enable(1) (csrc/prof.cu).
class ProfScope {
public:
    ProfScope(const char* name, void* stream);
    ~ProfScope();
    ProfScope(const ProfScope&) = delete;
    ProfScope& operator=(const ProfScope&) = delete;
private:
    const char* name_;
    void* stream_;
    void* a_;
};
#define LRB_LAUNCH(name, stream, ...)            \
    do {                                         \
        ProfScope lrb_ps_(name, (void*)(stream)); \
        __VA_ARGS__;                             \
    } while (0)

// host-side internals shared between ingest.cpp / format.cpp / api.cu
struct lrb_reads {
    uint64_t n_reads = 0, n_blocks = 0, n_tiles = 0, total_bases = 0;
    uint32_t* codes = nullptr;      // 2*n_blocks + 2
    uint32_t* valid = nullptr;      // n_blocks + 1
    uint32_t* read_len = nullptr;   // n_reads
    uint32_t* read_blk = nullptr;   // n_reads + 1
    uint32_t* tile_read = nullptr;  // n_tiles
    uint32_t* tile_blk = nullptr;   // n_tiles
    bool pinned = false;            // buffers came from cudaHostAlloc
    bool borrowed = false;          // codes/valid point into another lrb_reads (lrb_reads_slice): not freed here
    // validity exceptions: blocks whose valid word differs from the one implied by the read length (all in-read
    // slots valid).  Lets the host path ship 0.25 B/base instead of 0.375: the device rebuilds `valid` from
    // read_len and patches these blocks (lrb_dev_fill_valid).
    uint64_t n_exc = 0;
    uint32_t* exc_blk = nullptr;    // n_exc, ascending
    uint32_t* exc_valid = nullptr;  // n_exc
    bool exc_pinned = false, exc_ready = false;
};

// page-locked when asked for and a CUDA device is usable, plain aligned memory otherwise (host-only unit tests)
void* lrb_host_alloc(size_t bytes, bool* pinned, bool want_pinned = true);
void lrb_host_free(void* p, bool pinned);

// bases per segment of the segment reader for result rows of `row_bytes_per_read` (lrb_reader_open: segment_bases = 0)
uint64_t lrb_segment_budget(uint64_t row_bytes_per_read);

// ---- the coverage row of one search --------------------------------------------------------------------------------
// A row is up to 8 column blocks side by side.  Each block bins the count of one table, the full-layout table or compact
// table (sample slot) `table`, either by (bin_size, bins) or by count edges.  The settings, samples and edges calls build
// three shapes (n (bin_size, bins) blocks on the full table, n such blocks on compact tables, one edge block on the full
// table); the layout calls take any blocks (lrb_cov_block).
static_assert(LRB_MAX_COV_SETTINGS == LRB_MAX_SAMPLE_TABLES, "one block per setting or per sample table");

struct CovBlock {
    int table = -1;                    // -1: the full-layout table; t >= 0: compact table t
    long bin_size = 1;                 // bins by (bin_size, bins), unless by_edges:
    int bins = 1;
    bool by_edges = false;             // bins by edges[n_edges] (the caller's array): a count c goes to #{i : edges[i] <= c}
    const uint32_t* edges = nullptr;
    int n_edges = 0;
    uint32_t width() const { return by_edges ? (uint32_t)n_edges + 1u : (uint32_t)bins; }
};

// which public call built a layout: the words its refusals use ("setting", "sample table", "block")
enum class CovKind { settings, samples, edges, blocks };

struct CovLayout {
    int n = 1;                         // blocks as asked for: lrb_check_cov_layout refuses n outside [1, 8]
    CovKind kind = CovKind::settings;
    bool null_settings = false;        // bin_sizes / bins (or the blocks) were NULL: the blocks were left unset
    CovBlock b[LRB_MAX_COV_SETTINGS];
    uint32_t W = 1;                    // row width, the blocks' bins together (lrb_check_cov_layout)
    bool single() const { return n == 1 && b[0].table < 0 && !b[0].by_edges; }   // what the direct search and k_search_keys take
    // some block reads the full-layout table (it must be counted or loaded, on every device) / some block reads a slot
    bool reads_full() const { for (int m = 0; m < n && m < LRB_MAX_COV_SETTINGS; ++m) if (b[m].table < 0) return true; return false; }
    bool reads_slots() const { for (int m = 0; m < n && m < LRB_MAX_COV_SETTINGS; ++m) if (b[m].table >= 0) return true; return false; }
};

// n (bin_sizes[m], bins[m]) blocks, on the full table (slots NULL) or on compact table slots[m].  Reads the arrays only as
// far as lrb_check_cov_layout can then refuse them: not when one is NULL, never past LRB_MAX_COV_SETTINGS blocks.
CovLayout lrb_cov_settings(int n, const long* bin_sizes, const int* bins, const int* slots = nullptr);
// one block on the full table binned by count edges (the array is kept, not copied)
CovLayout lrb_cov_edges(const uint32_t* edges, int n_edges);
// the n public blocks as they are (edge arrays kept, not copied); read as far as lrb_cov_settings reads its arrays
CovLayout lrb_cov_layout(const lrb_cov_block* blocks, int n);

// Checks a layout and fills L->W; LRB_EINVAL naming `who` and the bad value.  Blocks: 1 <= n <= 8, compact tables in
// [0, 8) (and -1, the full table, in a layout of lrb_cov_block), bin_size >= 1, bins in [1, LRB_MAX_BINS]; edges: at most
// LRB_MAX_BINS - 1, non-NULL when there are any, strictly increasing, the first >= 2 (counts 0 and 1 stay in bin 0, as in
// the reference's rule); no block twice (same table, same binning); the row at most LRB_MAX_BINS wide.
int lrb_check_cov_layout(const char* who, CovLayout* L);

// The partitioned search of the buckets [bucket_lo, bucket_hi) for a checked layout: a block reads `table`, or
// compact[b[m].table] when b[m].table >= 0.  sums are rewritten by the call that includes the last bucket (partition.cu).
int lrb_partition_search(const char* who, const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* table,
                         const uint32_t* const* compact, const CovLayout& L, uint32_t* hist, uint32_t* sums, void* stream);
