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

// n coverage settings (bin_sizes[m], bins[m]) of one search: 1 <= n <= LRB_MAX_COV_SETTINGS, bin_size >= 1, bins in
// [1, LRB_MAX_BINS], no pair twice, row width W = sum of bins <= LRB_MAX_BINS (into *width).  LRB_EINVAL naming `who`.
int lrb_check_cov_settings(const char* who, int n, const long* bin_sizes, const int* bins, uint32_t* width);

// The same for n sample tables with one setting each (LRB_MAX_SAMPLE_TABLES at most): ids[t] says which table t is, and only
// the same (table, bin_size, bins) twice is refused.
int lrb_check_table_settings(const char* who, int n, const uint64_t* ids, const long* bin_sizes, const int* bins, uint32_t* width);

// Coverage bins given by n count edges: 0 <= n <= LRB_MAX_BINS - 1, edges non-NULL when n > 0, strictly increasing, the
// first >= 2 (counts 0 and 1 stay in bin 0, as in the reference's rule).  LRB_EINVAL naming `who` and the bad value.
int lrb_check_cov_edges(const char* who, const uint32_t* edges, int n);
