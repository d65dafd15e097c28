// format.cpp — host epilogue: exact "%f" text rows, .npy arrays, the 15mers-counts table file,
// plus the small host utilities shared by the library (error string, canonical k-mer LUT).
//
// Replaces the serial std::to_string loops of the tools (count-kmers.cpp:110-118,
// search-15mers.cpp:35-48) and writeKmerFile/readKmerFile (kmer_utils.h:89-112).
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include "common.h"
#include "fixed6.h"
#include "lane_core.cuh"

// ---- error plumbing ----------------------------------------------------------------------------
static thread_local char t_err[512] = "";

int lrb_set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof t_err, fmt, ap);
    va_end(ap);
    return code;
}

extern "C" const char* lrb_last_error(void) { return t_err; }
extern "C" int lrb_version(void) { return 100; }

// ---- canonical k-mer index (compute_kmer_inds, count-kmers.cpp:38-64) ---------------------------
// index = rank of min(x, rc(x)) among the canonical values in ascending order; a k-mer met after its
// reverse complement shares that one's index.
extern "C" int lrb_kmer_lut(int k, uint16_t* lut) {
    if (k < 1 || k > 5 || !lut) return -1;
    const uint32_t n = 1u << (2 * k);
    uint32_t next = 0;
    for (uint32_t x = 0; x < n; ++x) {
        uint32_t rc = 0, t = x;
        for (int i = 0; i < k; ++i) { rc = (rc << 2) | ((t & 3u) ^ 2u); t >>= 2; }
        lut[x] = (rc < x) ? lut[rc] : (uint16_t)next++;
    }
    return (int)next;
}

// ---- "%f" of count/total -----------------------------------------------------------------------
extern "C" uint32_t lrb_fixed6(uint32_t num, uint32_t den, int coverage) { return lrb::fixed6(num, den, coverage != 0); }

namespace {

// two decimal digits at a time
struct Digits2 {
    char d[100][2];
    Digits2() { for (int i = 0; i < 100; ++i) { d[i][0] = (char)('0' + i / 10); d[i][1] = (char)('0' + i % 10); } }
};
const Digits2 kDigits2;

inline void put_fixed6(char* dst, uint32_t q) {  // 8 chars "d.dddddd"
    if (q == 0) { memcpy(dst, "0.000000", 8); return; }   // most composition / coverage cells
    const uint32_t ip = q / 1000000u, f = q - ip * 1000000u;
    const uint32_t a = f / 10000u, r = f - a * 10000u, b2 = r / 100u, c2 = r - b2 * 100u;
    dst[0] = (char)('0' + ip);
    dst[1] = '.';
    memcpy(dst + 2, kDigits2.d[a], 2);
    memcpy(dst + 4, kDigits2.d[b2], 2);
    memcpy(dst + 6, kDigits2.d[c2], 2);
}

int comp_width(int k) { return k == 3 ? 32 : k == 4 ? 136 : k == 5 ? 512 : 0; }

bool pwrite_all(int fd, const char* p, size_t n, uint64_t off) {
    while (n) {
        const ssize_t w = pwrite(fd, p, n, (off_t)off);
        if (w <= 0) return false;
        p += w;
        n -= (size_t)w;
        off += (uint64_t)w;
    }
    return true;
}

// Fixed-width rows: every thread formats blocks of its share of the rows into a private buffer and writes them at their
// final offset (pwrite), so neither the text nor the file copy is ever serial and nothing of file size sits in memory.
// row(i, dst) fills row i (row_bytes bytes).  The rows go after `row0` rows already in the file (row0 = 0: a new file); the
// head, if any, is (re)written at offset 0.
template <class RowFn>
int write_fixed_rows(const char* path, const void* head, size_t head_bytes, uint64_t n_rows, size_t row_bytes, int threads, RowFn row,
                     uint64_t row0) {
    const int fd = open(path, O_WRONLY | O_CREAT | (row0 ? 0 : O_TRUNC), 0644);
    if (fd < 0) return lrb_set_error(LRB_EIO, "cannot open %s for writing", path);
    bool ok = !head_bytes || pwrite_all(fd, (const char*)head, head_bytes, 0);
    if (threads < 1) threads = 1;
    if (threads > 64) threads = 64;
    if (n_rows < 256) threads = 1;
    const uint64_t block_rows = std::max<uint64_t>(1, (2ull << 20) / std::max<size_t>(row_bytes, 1));
    std::vector<char> failed((size_t)threads, 0);
    auto work = [&](int t) {
        const uint64_t a = n_rows * (uint64_t)t / (uint64_t)threads, b = n_rows * (uint64_t)(t + 1) / (uint64_t)threads;
        std::vector<char> buf((size_t)std::min<uint64_t>(block_rows, std::max<uint64_t>(b - a, 1)) * row_bytes);
        for (uint64_t lo = a; lo < b; lo += block_rows) {
            const uint64_t hi = std::min(b, lo + block_rows);
            for (uint64_t i = lo; i < hi; ++i) row(i, buf.data() + (size_t)(i - lo) * row_bytes);
            if (!pwrite_all(fd, buf.data(), (size_t)(hi - lo) * row_bytes, head_bytes + (row0 + lo) * row_bytes)) { failed[(size_t)t] = 1; return; }
        }
    };
    if (ok && n_rows) {
        if (threads == 1) work(0);
        else {
            std::vector<std::thread> pool;
            for (int t = 0; t < threads; ++t) pool.emplace_back(work, t);
            for (auto& th : pool) th.join();
        }
        for (char f : failed) ok = ok && !f;
    }
    if (close(fd) != 0) ok = false;
    if (!ok) return lrb_set_error(LRB_EIO, "short write to %s", path);
    return LRB_OK;
}

template <class RowFn>
int write_rows(const char* path, uint64_t n_rows, size_t row_bytes, int threads, RowFn row, uint64_t row0) {
    return write_fixed_rows(path, nullptr, 0, n_rows, row_bytes, threads, row, row0);
}

// 10 + len("{'descr': '<f8', 'fortran_order': False, 'shape': (R, C), }\n") = 69 + digits(R) + digits(C) <= 128 for any
// u64 R and C < 10^39, so the header is 128 bytes for every shape: a file written in parts can take the final row count
// in place.
std::string npy_header(uint64_t rows, uint64_t cols) {
    char dict[160];
    snprintf(dict, sizeof dict, "{'descr': '<f8', 'fortran_order': False, 'shape': (%llu, %llu), }",
             (unsigned long long)rows, (unsigned long long)cols);
    std::string h("\x93NUMPY\x01\x00", 8);
    size_t len = strlen(dict) + 1;              // + '\n'
    size_t total = 10 + len;
    size_t pad = (64 - total % 64) % 64;
    uint16_t hlen = (uint16_t)(len + pad);
    h.push_back((char)(hlen & 0xFF));
    h.push_back((char)(hlen >> 8));
    h += dict;
    h.append(pad, ' ');
    h.push_back('\n');
    return h;
}

template <class RowFn>
int write_npy(const char* path, uint64_t n_rows, uint64_t cols, int threads, RowFn row, uint64_t row0) {
    const std::string h = npy_header(row0 + n_rows, cols);
    if (h.size() != 128) return lrb_set_error(LRB_EINVAL, "npy header of %zu bytes", h.size());
    return write_fixed_rows(path, h.data(), h.size(), n_rows, (size_t)cols * 8, threads,
                            [&](uint64_t i, char* dst) { row(i, reinterpret_cast<double*>(dst)); }, row0);
}

inline uint32_t comp_total(uint32_t len, int k) { return len >= (uint32_t)k ? len - (uint32_t)k + 1u : 0u; }

}  // namespace

extern "C" int lrb_append_composition_txt(const char* path, const uint32_t* counts, const uint32_t* read_len,
                                         uint64_t n_reads, int k, int threads, uint64_t row0) {
    const int P = comp_width(k);
    if (!path || !P || (n_reads && (!counts || !read_len))) return lrb_set_error(LRB_EINVAL, "lrb_append_composition_txt: bad argument");
    const size_t row_bytes = (size_t)P * 9 + 1;  // "d.dddddd " x P, then '\n'  (count-kmers.cpp:110-118)
    return write_rows(path, n_reads, row_bytes, threads, [=](uint64_t i, char* dst) {
        const uint32_t total = comp_total(read_len[i], k);
        const uint32_t* c = counts + (size_t)i * P;
        for (int j = 0; j < P; ++j) {
            put_fixed6(dst + (size_t)j * 9, lrb::fixed6(c[j], total, false));
            dst[(size_t)j * 9 + 8] = ' ';
        }
        dst[row_bytes - 1] = '\n';
    }, row0);
}

extern "C" int lrb_write_composition_txt(const char* path, const uint32_t* counts, const uint32_t* read_len,
                                         uint64_t n_reads, int k, int threads) {
    return lrb_append_composition_txt(path, counts, read_len, n_reads, k, threads, 0);
}

extern "C" int lrb_append_coverage_txt(const char* path, const uint32_t* hist, const uint32_t* sums, uint64_t n_reads,
                                      int bins, int threads, uint64_t row0) {
    if (!path || bins <= 0 || (n_reads && (!hist || !sums))) return lrb_set_error(LRB_EINVAL, "lrb_append_coverage_txt: bad argument");
    const size_t row_bytes = (size_t)bins * 9;  // values separated by ' ', '\n' after the last (search-15mers.cpp:35-48)
    return write_rows(path, n_reads, row_bytes, threads, [=](uint64_t i, char* dst) {
        const uint32_t* c = hist + (size_t)i * bins;
        for (int j = 0; j < bins; ++j) {
            put_fixed6(dst + (size_t)j * 9, lrb::fixed6(c[j], sums[i], true));
            dst[(size_t)j * 9 + 8] = (j == bins - 1) ? '\n' : ' ';
        }
    }, row0);
}

extern "C" int lrb_write_coverage_txt(const char* path, const uint32_t* hist, const uint32_t* sums, uint64_t n_reads,
                                      int bins, int threads) {
    return lrb_append_coverage_txt(path, hist, sums, n_reads, bins, threads, 0);
}

extern "C" int lrb_append_composition_npy(const char* path, const uint32_t* counts, const uint32_t* read_len,
                                         uint64_t n_reads, int k, int threads, uint64_t row0) {
    const int P = comp_width(k);
    if (!path || !P || (n_reads && (!counts || !read_len))) return lrb_set_error(LRB_EINVAL, "lrb_append_composition_npy: bad argument");
    return write_npy(path, n_reads, (uint64_t)P, threads, [=](uint64_t i, double* dst) {
        const uint32_t total = comp_total(read_len[i], k);
        const uint32_t* c = counts + (size_t)i * P;
        for (int j = 0; j < P; ++j) dst[j] = (double)lrb::fixed6(c[j], total, false) / 1e6;  // == float("%f" text)
    }, row0);
}

extern "C" int lrb_write_composition_npy(const char* path, const uint32_t* counts, const uint32_t* read_len,
                                         uint64_t n_reads, int k, int threads) {
    return lrb_append_composition_npy(path, counts, read_len, n_reads, k, threads, 0);
}

extern "C" int lrb_append_coverage_npy(const char* path, const uint32_t* hist, const uint32_t* sums, uint64_t n_reads,
                                      int bins, int threads, uint64_t row0) {
    if (!path || bins <= 0 || (n_reads && (!hist || !sums))) return lrb_set_error(LRB_EINVAL, "lrb_append_coverage_npy: bad argument");
    return write_npy(path, n_reads, (uint64_t)bins, threads, [=](uint64_t i, double* dst) {
        const uint32_t* c = hist + (size_t)i * bins;
        for (int j = 0; j < bins; ++j) dst[j] = (double)lrb::fixed6(c[j], sums[i], true) / 1e6;
    }, row0);
}

extern "C" int lrb_write_coverage_npy(const char* path, const uint32_t* hist, const uint32_t* sums, uint64_t n_reads,
                                      int bins, int threads) {
    return lrb_append_coverage_npy(path, hist, sums, n_reads, bins, threads, 0);
}

// ---- 15mers-counts file (kmer_utils.h:89-112): u64 size (= 2^30), then size little-endian u32 -----
extern "C" int lrb_table_write_file(const char* path, const uint32_t* table) {
    if (!path || !table) return lrb_set_error(LRB_EINVAL, "lrb_table_write_file: null argument");
    int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return lrb_set_error(LRB_EIO, "cannot open %s for writing", path);
    const uint64_t size = LRB_TABLE_ENTRIES;
    if (write(fd, &size, sizeof size) != (ssize_t)sizeof size) { close(fd); return lrb_set_error(LRB_EIO, "short write to %s", path); }
    const char* p = (const char*)table;
    size_t left = (size_t)size * 4;
    while (left) {
        const ssize_t w = write(fd, p, std::min<size_t>(left, 1u << 30));
        if (w <= 0) { close(fd); return lrb_set_error(LRB_EIO, "short write to %s", path); }
        p += w;
        left -= (size_t)w;
    }
    if (close(fd) != 0) return lrb_set_error(LRB_EIO, "close failed for %s", path);
    return LRB_OK;
}

extern "C" int lrb_table_read_file(const char* path, uint32_t* table) {
    if (!path || !table) return lrb_set_error(LRB_EINVAL, "lrb_table_read_file: null argument");
    int fd = open(path, O_RDONLY);
    if (fd < 0) return lrb_set_error(LRB_EIO, "cannot open table file %s", path);
    uint64_t size = 0;
    if (read(fd, &size, sizeof size) != (ssize_t)sizeof size || size != LRB_TABLE_ENTRIES) {
        close(fd);
        return lrb_set_error(LRB_EFORMAT, "%s is not a 4^15-entry 15mers-counts file", path);
    }
    char* p = (char*)table;
    size_t left = (size_t)size * 4;
    while (left) {
        const ssize_t r = read(fd, p, std::min<size_t>(left, 1u << 30));
        if (r <= 0) { close(fd); return lrb_set_error(LRB_EFORMAT, "%s is truncated", path); }
        p += r;
        left -= (size_t)r;
    }
    close(fd);
    return LRB_OK;
}

// ---- the coverage row of a search (common.h) ---------------------------------------------------------------------
CovLayout lrb_cov_settings(int n, const long* bin_sizes, const int* bins, const int* slots) {
    CovLayout L;
    L.n = n;
    L.kind = slots ? CovKind::samples : CovKind::settings;
    L.null_settings = !bin_sizes || !bins;
    for (int m = 0; m < n && m < LRB_MAX_COV_SETTINGS && !L.null_settings; ++m) {
        L.b[m].table = slots ? slots[m] : -1;
        L.b[m].bin_size = bin_sizes[m];
        L.b[m].bins = bins[m];
    }
    return L;
}

CovLayout lrb_cov_edges(const uint32_t* edges, int n_edges) {
    CovLayout L;
    L.kind = CovKind::edges;
    L.b[0].by_edges = true;
    L.b[0].edges = edges;
    L.b[0].n_edges = n_edges;
    return L;
}

CovLayout lrb_cov_layout(const lrb_cov_block* blocks, int n) {
    CovLayout L;
    L.n = n;
    L.kind = CovKind::blocks;
    L.null_settings = !blocks;
    for (int m = 0; m < n && m < LRB_MAX_COV_SETTINGS && blocks; ++m) {
        CovBlock& b = L.b[m];
        b.table = blocks[m].table;
        b.by_edges = blocks[m].by_edges != 0;
        b.bin_size = b.by_edges ? 1 : blocks[m].bin_size;
        b.bins = b.by_edges ? 1 : blocks[m].bins;
        b.edges = b.by_edges ? blocks[m].edges : nullptr;
        b.n_edges = b.by_edges ? blocks[m].n_edges : 0;
    }
    return L;
}

static int check_edges(const char* who, const uint32_t* edges, int n) {
    if (n < 0 || n > LRB_MAX_BINS - 1) return lrb_set_error(LRB_EINVAL, "%s: the number of edges must be in [0, %d] (got %d)", who, LRB_MAX_BINS - 1, n);
    if (n > 0 && !edges) return lrb_set_error(LRB_EINVAL, "%s: null edges (%d edges)", who, n);
    if (n > 0 && edges[0] < 2)
        return lrb_set_error(LRB_EINVAL, "%s: the first edge must be >= 2, so that counts 0 and 1 stay in bin 0 (got %u)", who, edges[0]);
    for (int i = 1; i < n; ++i)
        if (edges[i] <= edges[i - 1])
            return lrb_set_error(LRB_EINVAL, "%s: edges must be strictly increasing (edge %d = %u after edge %d = %u)", who, i, edges[i], i - 1, edges[i - 1]);
    return LRB_OK;
}

static bool same_binning(const CovBlock& a, const CovBlock& b) {
    if (a.table != b.table || a.by_edges != b.by_edges) return false;
    if (!a.by_edges) return a.bin_size == b.bin_size && a.bins == b.bins;
    return a.n_edges == b.n_edges && std::equal(a.edges, a.edges + a.n_edges, b.edges);
}

int lrb_check_cov_layout(const char* who, CovLayout* L) {
    const bool samples = L->kind == CovKind::samples, blocks = L->kind == CovKind::blocks;
    const char* what = blocks ? "block" : samples ? "table" : "setting";
    if (L->n < 1 || L->n > LRB_MAX_COV_SETTINGS)
        return lrb_set_error(LRB_EINVAL, "%s: the number of %ss must be in [1, %d] (got %d)", who, blocks ? "block" : samples ? "sample table" : "setting",
                             LRB_MAX_COV_SETTINGS, L->n);
    if (L->null_settings) return lrb_set_error(LRB_EINVAL, blocks ? "%s: null blocks" : "%s: null bin_sizes / bins", who);
    uint64_t W = 0;
    for (int m = 0; m < L->n; ++m) {
        const CovBlock& b = L->b[m];
        if (blocks && (b.table < -1 || b.table >= LRB_MAX_SAMPLE_TABLES))
            return lrb_set_error(LRB_EINVAL, "%s: table must be -1 (the full-layout table) or a slot in [0, %d) (block %d: got %d)", who,
                                 LRB_MAX_SAMPLE_TABLES, m, b.table);
        if (b.by_edges) {
            char at[160];   // a block of a layout is named in the message
            if (blocks) snprintf(at, sizeof at, "%s: block %d", who, m);
            const int rc = check_edges(blocks ? at : who, b.edges, b.n_edges);
            if (rc) return rc;
        } else {
            if (samples && (b.table < 0 || b.table >= LRB_MAX_SAMPLE_TABLES))
                return lrb_set_error(LRB_EINVAL, "%s: slot must be in [0, %d) (table %d: got %d)", who, LRB_MAX_SAMPLE_TABLES, m, b.table);
            if (b.bin_size < 1) return lrb_set_error(LRB_EINVAL, "%s: bin_size must be >= 1 (%s %d: got %ld)", who, what, m, b.bin_size);
            if (b.bins < 1 || b.bins > LRB_MAX_BINS) return lrb_set_error(LRB_EINVAL, "%s: bins must be in [1, %d] (%s %d: got %d)", who, LRB_MAX_BINS, what, m, b.bins);
        }
        for (int j = 0; j < m; ++j) {
            if (!same_binning(L->b[j], b)) continue;
            if (b.by_edges)
                return lrb_set_error(LRB_EINVAL, "%s: block %d repeats block %d (same table, the same %d edges)", who, m, j, b.n_edges);
            return lrb_set_error(LRB_EINVAL, "%s: %s %d repeats %s %d (%sbin_size %ld, bins %d)", who, what, m, what, j,
                                 samples || blocks ? "same table, " : "", b.bin_size, b.bins);
        }
        W += b.width();
    }
    if (W > LRB_MAX_BINS) return lrb_set_error(LRB_EINVAL, "%s: the %ss' bins add up to %llu, more than %d", who, what, (unsigned long long)W, LRB_MAX_BINS);
    L->W = (uint32_t)W;
    return LRB_OK;
}

// ---- abundance spectrum of the table (lrb_dev_table_spectrum layout: n_c for c < M, then n_over, sum_over, max) ----
extern "C" int lrb_spectrum_bin_mass(const uint64_t* spectrum, uint32_t max_count, long bin_size, int bins, uint64_t* mass) {
    if (!spectrum || !mass) return lrb_set_error(LRB_EINVAL, "lrb_spectrum_bin_mass: null argument");
    if (bin_size < 1) return lrb_set_error(LRB_EINVAL, "lrb_spectrum_bin_mass: bin_size must be >= 1");
    if (bins < 1 || bins > LRB_MAX_BINS) return lrb_set_error(LRB_EINVAL, "lrb_spectrum_bin_mass: bins must be in [1, %d]", LRB_MAX_BINS);
    const uint64_t M = max_count;
    // every count >= S * (B + 1) lands in the last bin; below that the spectrum must resolve the count itself
    const bool over_determined = bin_size < (long)M && M >= (uint64_t)bin_size * (uint64_t)(bins + 1);
    if (spectrum[M] > 0 && !over_determined)
        return lrb_set_error(LRB_EINVAL, "lrb_spectrum_bin_mass: %llu keys counted >= max_count %u, which is below bin_size * (bins + 1) = %lld",
                             (unsigned long long)spectrum[M], max_count, (long long)bin_size * (bins + 1));
    const uint32_t S32 = bin_size > 0xFFFFFFFFl ? 0xFFFFFFFFu : (uint32_t)bin_size;
    const uint64_t magic = lrb::coverage_magic(S32);
    std::fill(mass, mass + bins, 0ull);
    for (uint64_t c = 0; c < M; ++c)
        if (spectrum[c]) mass[lrb::coverage_bin((uint32_t)c, S32, magic, (uint32_t)bins)] += c * spectrum[c];
    mass[bins - 1] += spectrum[M + 1];
    return LRB_OK;
}

extern "C" int lrb_spectrum_edge_mass(const uint64_t* spectrum, uint32_t max_count, const uint32_t* edges, int n_edges, uint64_t* mass) {
    static const char* who = "lrb_spectrum_edge_mass";
    if (!spectrum || !mass) return lrb_set_error(LRB_EINVAL, "%s: null argument", who);
    CovLayout L = lrb_cov_edges(edges, n_edges);
    const int rc = lrb_check_cov_layout(who, &L);
    if (rc) return rc;
    const uint64_t M = max_count;
    // every count >= the last edge lands in the last bin; below it the spectrum must resolve the count itself
    if (spectrum[M] > 0 && n_edges > 0 && M < edges[n_edges - 1])
        return lrb_set_error(LRB_EINVAL, "%s: %llu keys counted >= max_count %u, which is below the last edge %u", who,
                             (unsigned long long)spectrum[M], max_count, edges[n_edges - 1]);
    std::fill(mass, mass + n_edges + 1, 0ull);
    int b = 0;   // bin of count c: the edges are increasing, so it only moves forward
    for (uint64_t c = 0; c < M; ++c) {
        while (b < n_edges && edges[b] <= c) ++b;
        mass[b] += c * spectrum[c];
    }
    mass[n_edges] += spectrum[M + 1];
    return LRB_OK;
}

extern "C" int lrb_write_spectrum_txt(const char* path, const uint64_t* spectrum, uint32_t max_count) {
    if (!path || !spectrum) return lrb_set_error(LRB_EINVAL, "lrb_write_spectrum_txt: null argument");
    FILE* f = fopen(path, "w");
    if (!f) return lrb_set_error(LRB_EIO, "cannot open %s for writing", path);
    bool ok = true;
    for (uint32_t c = 1; c < max_count && ok; ++c)
        if (spectrum[c]) ok = fprintf(f, "%u %llu\n", c, (unsigned long long)spectrum[c]) > 0;
    if (ok && spectrum[max_count]) ok = fprintf(f, "%u %llu\n", max_count, (unsigned long long)spectrum[max_count]) > 0;
    if (fclose(f) != 0) ok = false;
    if (!ok) return lrb_set_error(LRB_EIO, "short write to %s", path);
    return LRB_OK;
}
