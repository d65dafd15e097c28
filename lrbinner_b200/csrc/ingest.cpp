// ingest.cpp — host side of the read stream: FASTA/FASTQ(+gzip) records -> 2-bit packed blocks.
//
// Replaces SeqReader (mbcclr_utils/io_utils.h:133-165) + kseq_read (mbcclr_utils/kseq.h:177-218).
// The file is parsed ONCE; the three tools of the reference each re-parse it.  Record semantics are the
// ones the tools observe (see parse_records below); packing follows csrc/lane_core.cuh.
#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "common.h"
#include "lane_core.cuh"

namespace {

// ---- record scanner --------------------------------------------------------------------------
// Works on the whole (decompressed) file image.  Rules, as exercised by the tools:
//  * with no pending header char, skip forward to the next '>' or '@' ANYWHERE (kseq.h:181-185);
//  * the name runs to the first isspace(); unless that was '\n' the rest of the line is a comment;
//    end of data right after the header char ends the stream without a record (kseq.h:187);
//  * sequence lines follow until a line STARTS with '>', '@' or '+'; empty lines are skipped; after a
//    line is appended a single trailing '\r' is dropped when the accumulated sequence is longer than
//    one byte (kseq.h:141,193-197) — not when the line was cut short by end of data with nothing read;
//  * '+' starts a FASTQ quality block: rest of that line ignored; quality lines are appended (same CR
//    rule) while shorter than the sequence; then the next header is searched afresh.  Missing '\n'
//    after '+' or a length mismatch ends the stream WITHOUT emitting the record (kseq.h:209-214);
//  * the tools copy the sequence as a C string (io_utils.h:159): it is cut at the first NUL byte.
struct Record {
    uint64_t off;    // into the file image (in_pool == 0) or into the parsing thread's pool
    uint32_t len;
    uint32_t in_pool;
};

static inline bool is_space(unsigned char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }

struct Parsed {
    std::string pool;  // sequences that span several lines, concatenated (single-line ones stay in the file image)
    std::vector<Record> recs;
    // streaming (gzip) mode: where every record's header starts, and where the record begins that was being parsed when the
    // data ran out (== n when none was): the reader keeps everything from there on for the next round
    bool want_hdr = false;
    std::vector<uint64_t> hdr;
    size_t open_hdr = 0;
    bool tail_open = false;    // the last record's parse ran into the end of the data (it may continue in the next chunk)
    bool end_touched = false;  // the stream "ended" because the data ran out, not because of a malformed record
};

// Parses the records whose header character lies in [pos, limit).  `pos` is either 0 (the start of the stream) or
// the position of a header character.  Returns the position of the first header character at or beyond `limit`
// (where the next range starts) or n; *ended is set when the stream ends here for good (end of data, or a FASTQ
// record without its quality block / with a length mismatch, which makes kseq stop silently).
static size_t parse_range(const unsigned char* buf, size_t n, size_t pos, size_t limit, Parsed& out, bool* ended) {
    int pending = 0;  // header char already consumed
    std::string qual;
    bool reserved = false;
    *ended = false;
    out.open_hdr = n;
    while (true) {
        size_t hdr;
        if (!pending) {
            while (pos < n && buf[pos] != '>' && buf[pos] != '@') ++pos;
            if (pos >= n) { *ended = true; out.end_touched = true; return n; }
            hdr = pos;
            pending = buf[pos++];
        } else {
            hdr = pos - 1;
        }
        if (hdr >= limit) return hdr;
        out.open_hdr = hdr;   // the record being parsed from here on is complete only once the next header (or EOF) is seen
        if (pos >= n) { *ended = true; out.end_touched = true; return n; }  // nothing after the header char
        bool touched = false;  // some step of this record's parse ran into the end of the data
        // name
        size_t i = pos;
        while (i < n && !is_space(buf[i])) ++i;
        int delim = 0;
        if (i < n) { delim = buf[i]; pos = i + 1; } else { pos = n; touched = true; }
        if (delim != '\n') {  // comment to end of line
            const void* nl = pos < n ? memchr(buf + pos, '\n', n - pos) : nullptr;
            if (!nl) touched = true;
            pos = nl ? (size_t)((const unsigned char*)nl - buf) + 1 : n;
        }
        // sequence: the first line stays where it is; a second line moves the record into the pool
        const size_t pool_off = out.pool.size();
        size_t first_off = 0, acc = 0;  // acc = accumulated length
        bool multi = false;
        int c = -1;
        while (true) {
            if (pos >= n) { c = -1; touched = true; break; }
            c = buf[pos++];
            if (c == '>' || c == '+' || c == '@') break;
            if (c == '\n') continue;
            const size_t ls = pos - 1;  // line start (the char just read belongs to the sequence)
            size_t le = pos;
            if (pos < n) {
                const void* nl = memchr(buf + pos, '\n', n - pos);
                if (!nl) touched = true;
                le = nl ? (size_t)((const unsigned char*)nl - buf) : n;
                pos = nl ? le + 1 : n;
            } else {
                touched = true;
            }
            // kseq appends the first char, then the rest of the line, then drops one trailing CR if more than one byte
            // has been accumulated — except when the line was cut by end of data right after its first char
            const bool appended_rest = ls + 1 < n;
            size_t len = le - ls;
            if (acc == 0 && !multi) {
                first_off = ls;
                acc = len;
                if (appended_rest && acc > 1 && buf[ls + acc - 1] == '\r') --acc;
            } else {
                if (!multi) {
                    // first multi-line record of this range: the pool can never need more than the rest of the range, and
                    // reserving that once (address space only) avoids the copy-on-grow of a 10^8-byte string
                    // (0.43 -> 0.15 s per 200 MB of 80-column FASTA)
                    if (!reserved) { out.pool.reserve(out.pool.size() + (std::min(limit, n) > hdr ? std::min(limit, n) - hdr : 0)); reserved = true; }
                    out.pool.append((const char*)buf + first_off, acc);
                    multi = true;
                }
                out.pool.append((const char*)buf + ls, len);
                acc += len;
                if (appended_rest && acc > 1 && out.pool.back() == '\r') { out.pool.pop_back(); --acc; }
            }
        }
        if (c == '>' || c == '@') pending = c;
        size_t seq_len = acc;
        if (c == '+') {
            const void* nl = pos < n ? memchr(buf + pos, '\n', n - pos) : nullptr;
            if (!nl) { out.pool.resize(pool_off); *ended = true; out.end_touched = true; return n; }  // no quality block: stream ends, record dropped
            pos = (size_t)((const unsigned char*)nl - buf) + 1;
            qual.clear();
            while (pos < n) {
                const void* q = memchr(buf + pos, '\n', n - pos);
                if (!q) touched = true;
                const size_t e = q ? (size_t)((const unsigned char*)q - buf) : n;
                qual.append((const char*)buf + pos, e - pos);
                pos = q ? e + 1 : n;
                if (qual.size() > 1 && qual.back() == '\r') qual.pop_back();
                if (!(qual.size() < seq_len)) break;
            }
            if (pos >= n) touched = true;   // the data ran out inside (or right behind) the quality block: kseq reads at least one
                                            // quality line when there is one, and goes on while the block is shorter than the sequence
            pending = 0;
            if (qual.size() != seq_len) { out.pool.resize(pool_off); *ended = true; out.end_touched = touched; return n; }
        }
        // C-string copy: cut at the first NUL
        const unsigned char* sp = multi ? (const unsigned char*)out.pool.data() + pool_off : buf + first_off;
        if (seq_len) {
            const void* z = memchr(sp, 0, seq_len);
            if (z) {
                seq_len = (size_t)((const unsigned char*)z - sp);
                if (multi) out.pool.resize(pool_off + seq_len);
            }
        }
        if (seq_len > 0xFFFFFFFFull) { out.pool.resize(pool_off); *ended = true; return n; }  // > 4 Gbase record: not representable
        out.recs.push_back(Record{multi ? (uint64_t)pool_off : (uint64_t)first_off, (uint32_t)seq_len, multi ? 1u : 0u});
        if (out.want_hdr) out.hdr.push_back(hdr);
        if (touched) out.tail_open = true;
        if (!pending) out.open_hdr = pos;   // a complete FASTQ record: whatever follows starts here
    }
}

// Candidate start of a range: the first header-looking line start at or after `from` ('\n' then '>' or '@'; for '@'
// the line after next must start with '+', which rules out nearly every quality line that happens to begin with '@').
// Only a guess — parse_all checks it against the parse of the preceding range.
static size_t find_candidate(const unsigned char* buf, size_t n, size_t from) {
    size_t p = from ? from : 1;
    while (p < n) {
        const void* nl = memchr(buf + p - 1, '\n', n - (p - 1));
        if (!nl) return n;
        p = (size_t)((const unsigned char*)nl - buf) + 1;
        if (p >= n) return n;
        if (buf[p] == '>') return p;
        if (buf[p] == '@') {
            const void* l1 = memchr(buf + p, '\n', n - p);
            const void* l2 = l1 ? memchr((const unsigned char*)l1 + 1, '\n', n - ((const unsigned char*)l1 + 1 - buf)) : nullptr;
            if (!l2 || (size_t)((const unsigned char*)l2 + 1 - buf) >= n || ((const unsigned char*)l2)[1] == '+') return p;
        }
        ++p;
    }
    return n;
}

// Whole-stream parse on `threads` threads: ranges start at guessed record boundaries and are parsed speculatively;
// a sequential pass then keeps a range's result only if the preceding range really ended on its start, and
// re-parses it from the true boundary otherwise.  The outcome equals parse_range(0, n) by construction.
// *stream_ended (optional): the stream ended for good inside this buffer (parts.back() says whether because the data ran out)
static void parse_all(const unsigned char* buf, size_t n, int threads, size_t min_chunk, std::vector<Parsed>& parts,
                      bool want_hdr = false, bool* stream_ended = nullptr) {
    parts.clear();
    size_t nr = std::max<size_t>(1, std::min<size_t>((size_t)std::max(1, threads), n / std::max<size_t>(min_chunk, 1)));
    if (stream_ended) *stream_ended = false;
    if (nr == 1) {
        parts.resize(1);
        parts[0].want_hdr = want_hdr;
        bool ended;
        parse_range(buf, n, 0, n, parts[0], &ended);
        if (stream_ended) *stream_ended = ended;
        return;
    }
    std::vector<size_t> start(nr + 1);
    start[0] = 0;
    for (size_t t = 1; t < nr; ++t) start[t] = std::max(start[t - 1], find_candidate(buf, n, n / nr * t));
    start[nr] = n;
    std::vector<Parsed> spec(nr);
    for (auto& sp : spec) sp.want_hdr = want_hdr;
    std::vector<size_t> next(nr);
    std::vector<char> ended(nr);
    {
        std::vector<std::thread> pool;
        for (size_t t = 0; t < nr; ++t)
            pool.emplace_back([&, t]() {
                bool e = false;
                next[t] = start[t] < start[t + 1] ? parse_range(buf, n, start[t], start[t + 1], spec[t], &e) : start[t];
                ended[t] = e;
            });
        for (auto& th : pool) th.join();
    }
    size_t cur = next[0];
    bool done = ended[0];
    parts.push_back(std::move(spec[0]));
    for (size_t t = 1; t < nr && !done; ++t) {
        if (start[t] >= start[t + 1]) continue;   // empty range
        if (cur >= start[t + 1]) continue;        // the previous record runs past this whole range
        if (cur == start[t]) {
            cur = next[t];
            done = ended[t];
            parts.push_back(std::move(spec[t]));
        } else {                                   // the guess was not a record boundary: parse from the real one
            Parsed fix;
            fix.want_hdr = want_hdr;
            bool e = false;
            cur = parse_range(buf, n, cur, start[t + 1], fix, &e);
            done = e;
            parts.push_back(std::move(fix));
        }
    }
    if (stream_ended) *stream_ended = done;
}

// The decompressed file image: a private mapping for plain files, a heap buffer for gzip (zlib's gzread, like
// io_utils.h:143; a plain file passes through gzread unchanged, so mapping it is equivalent).
struct FileImage {
    const unsigned char* data = nullptr;
    size_t size = 0;
    void* map = nullptr;
    size_t map_len = 0;
    std::vector<unsigned char> heap;
    ~FileImage() { if (map) munmap(map, map_len); }
};

static bool read_gz(const char* path, std::vector<unsigned char>& data, uint64_t size_hint) {
    gzFile f = gzopen(path, "rb");
    if (!f) return false;
    gzbuffer(f, 1 << 20);
    size_t n = 0;
    // size_hint: ISIZE of the (last) gzip member = its uncompressed size mod 2^32 — right for the usual single-member
    // file below 4 GiB, and only a starting size otherwise (the buffer still doubles when it runs out)
    data.resize(std::max<uint64_t>(size_hint + (1u << 20) + 1, 1u << 22));
    for (;;) {
        if (data.size() - n < (1 << 20)) data.resize(data.size() * 2);
        const size_t room = std::min<size_t>(data.size() - n, 1u << 30);
        const int got = gzread(f, data.data() + n, (unsigned)room);
        if (got <= 0) break;  // EOF or a damaged stream: the tools stop quietly at that point too
        n += (size_t)got;
    }
    gzclose(f);
    data.resize(n);
    return true;
}

static void load_file(const char* path, FileImage& img) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return;  // unreadable file == empty stream (tools: exit 0, empty outputs)
    struct stat st;
    unsigned char magic[2] = {0, 0};
    const bool regular = fstat(fd, &st) == 0 && S_ISREG(st.st_mode);
    const bool gz = regular && st.st_size >= 2 && pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
    if (regular && !gz && st.st_size > 0) {
        void* m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m != MAP_FAILED) {
            madvise(m, (size_t)st.st_size, MADV_WILLNEED);
            img.map = m;
            img.map_len = img.size = (size_t)st.st_size;
            img.data = (const unsigned char*)m;
            close(fd);
            return;
        }
    }
    uint64_t hint = 0;
    if (gz && st.st_size >= 18) {
        unsigned char isize[4];
        if (pread(fd, isize, 4, st.st_size - 4) == 4)
            hint = (uint64_t)isize[0] | (uint64_t)isize[1] << 8 | (uint64_t)isize[2] << 16 | (uint64_t)isize[3] << 24;
        if (hint < (uint64_t)st.st_size) hint = 0;   // wrapped around 2^32 (or not a plain single member): no use as a size
    }
    close(fd);
    if (read_gz(path, img.heap, hint)) {
        img.data = img.heap.data();
        img.size = img.heap.size();
    }
}

// ---- packing -----------------------------------------------------------------------------------
struct PackLut {
    uint8_t code[256];
    uint8_t ok[256];
    PackLut() {
        for (int c = 0; c < 256; ++c) {
            code[c] = (uint8_t)((c >> 1) & 3);  // count-kmers.cpp:77, kmer_utils.h:47
            ok[c] = (c == 'A' || c == 'C' || c == 'G' || c == 'T') ? 1 : 0;  // kmer_utils.h:38
        }
    }
};
static const PackLut g_pack;

static void pack_tail(const unsigned char* p, uint32_t rem, uint32_t* codes2, uint32_t* valid1) {
    uint32_t w0 = 0, w1 = 0, v = 0;
    for (uint32_t j = 0; j < rem; ++j) {
        const uint32_t code = g_pack.code[p[j]];
        if (j < 16) w0 |= code << (30 - 2 * j); else w1 |= code << (62 - 2 * j);
        v |= (uint32_t)g_pack.ok[p[j]] << j;
    }
    codes2[0] = w0;
    codes2[1] = w1;
    *valid1 = v;
}

static void pack_read_scalar(const unsigned char* s, uint32_t len, uint32_t* codes, uint32_t* valid) {
    // codes/valid point at the read's first block; the read owns len/32 + 1 blocks, every one of which is written
    const uint32_t full = len / 32;
    for (uint32_t b = 0; b < full; ++b) {
        const unsigned char* p = s + (size_t)b * 32;
        uint32_t w0 = 0, w1 = 0, v = 0;
        for (int j = 0; j < 16; ++j) {
            w0 = (w0 << 2) | g_pack.code[p[j]];
            w1 = (w1 << 2) | g_pack.code[p[16 + j]];
            v |= (uint32_t)g_pack.ok[p[j]] << j;
            v |= (uint32_t)g_pack.ok[p[16 + j]] << (16 + j);
        }
        codes[2 * (size_t)b] = w0;
        codes[2 * (size_t)b + 1] = w1;
        valid[b] = v;
    }
    pack_tail(s + (size_t)full * 32, len - full * 32, codes + 2 * (size_t)full, valid + full);
}

#if defined(__x86_64__)
#include <immintrin.h>
// 32 bases per step: the two code bits of every byte (bits 1-2) are gathered with PEXT after a byte swap (first base
// -> most significant pair), validity = four byte compares + MOVEMASK (bit j <-> byte j, the layout of `valid`).
__attribute__((target("avx2,bmi2"))) static void pack_read_avx2(const unsigned char* s, uint32_t len, uint32_t* codes, uint32_t* valid) {
    const uint32_t full = len / 32;
    const __m256i cA = _mm256_set1_epi8('A'), cC = _mm256_set1_epi8('C'), cG = _mm256_set1_epi8('G'), cT = _mm256_set1_epi8('T');
    for (uint32_t b = 0; b < full; ++b) {
        const unsigned char* p = s + (size_t)b * 32;
        uint64_t q0, q1, q2, q3;
        memcpy(&q0, p, 8); memcpy(&q1, p + 8, 8); memcpy(&q2, p + 16, 8); memcpy(&q3, p + 24, 8);
        const uint64_t m = 0x0606060606060606ull;
        const uint32_t w0 = (uint32_t)(_pext_u64(__builtin_bswap64(q0), m) << 16 | _pext_u64(__builtin_bswap64(q1), m));
        const uint32_t w1 = (uint32_t)(_pext_u64(__builtin_bswap64(q2), m) << 16 | _pext_u64(__builtin_bswap64(q3), m));
        const __m256i x = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(p));
        const __m256i ok = _mm256_or_si256(_mm256_or_si256(_mm256_cmpeq_epi8(x, cA), _mm256_cmpeq_epi8(x, cC)),
                                           _mm256_or_si256(_mm256_cmpeq_epi8(x, cG), _mm256_cmpeq_epi8(x, cT)));
        codes[2 * (size_t)b] = w0;
        codes[2 * (size_t)b + 1] = w1;
        valid[b] = (uint32_t)_mm256_movemask_epi8(ok);
    }
    pack_tail(s + (size_t)full * 32, len - full * 32, codes + 2 * (size_t)full, valid + full);
}
static const bool g_have_avx2 = __builtin_cpu_supports("avx2") && __builtin_cpu_supports("bmi2");
#else
static const bool g_have_avx2 = false;
static void pack_read_avx2(const unsigned char* s, uint32_t len, uint32_t* codes, uint32_t* valid) { pack_read_scalar(s, len, codes, valid); }
#endif

static void pack_read(const unsigned char* s, uint32_t len, uint32_t* codes, uint32_t* valid) {
    static const bool force_scalar = getenv("LRB_PACK_SCALAR") != nullptr;
    if (g_have_avx2 && !force_scalar) pack_read_avx2(s, len, codes, valid);
    else pack_read_scalar(s, len, codes, valid);
}

static void free_reads(lrb_reads* r) {
    if (!r) return;
    if (!r->borrowed) {
        lrb_host_free(r->codes, r->pinned);
        lrb_host_free(r->valid, r->pinned);
    }
    free(r->read_len);
    free(r->read_blk);
    free(r->tile_read);
    free(r->tile_blk);
    lrb_host_free(r->exc_blk, r->exc_pinned);
    lrb_host_free(r->exc_valid, r->exc_pinned);
    delete r;
}

// builds read_blk / tiles from read_len and allocates codes/valid — zeroed only on request: the packers write every
// word of every block themselves (in parallel, which also spreads the first-touch page faults over the threads)
// Page-locking costs ~0.5 s per GB (measured, profiles/r01_ingest_timing.log) — more than a one-shot pageable copy of
// the same bytes — so the file / ASCII constructors use plain memory unless LRB_PIN_READS=1; the layout-only
// constructor (streams that are filled once and profiled many times) pins.
static bool pin_reads_default() {
    const char* e = getenv("LRB_PIN_READS");
    return e && atoi(e) > 0;
}

static int build_layout(lrb_reads* r, bool zero = false, bool want_pinned = true, bool alloc_stream = true) {
    const uint64_t n = r->n_reads;
    r->read_blk = (uint32_t*)malloc(sizeof(uint32_t) * (n + 1));
    if (!r->read_blk) return lrb_set_error(LRB_ENOMEM, "out of memory (read_blk)");
    uint64_t blk = 0, tiles = 0, bases = 0;
    for (uint64_t i = 0; i < n; ++i) {
        r->read_blk[i] = (uint32_t)blk;
        const uint64_t nb = (uint64_t)r->read_len[i] / 32 + 1;
        blk += nb;
        tiles += (nb + LRB_TILE_BLOCKS - 1) / LRB_TILE_BLOCKS;
        bases += r->read_len[i];
        if (blk > 0xFFFFFFF0ull) return lrb_set_error(LRB_EINVAL, "read set too large: more than 2^32 blocks (137 Gbases)");
    }
    r->read_blk[n] = (uint32_t)blk;
    r->n_blocks = blk;
    r->n_tiles = tiles;
    r->total_bases = bases;
    r->tile_read = (uint32_t*)malloc(sizeof(uint32_t) * (tiles + 1));
    r->tile_blk = (uint32_t*)malloc(sizeof(uint32_t) * (tiles + 1));
    if (!r->tile_read || !r->tile_blk) return lrb_set_error(LRB_ENOMEM, "out of memory (tiles)");
    uint64_t t = 0;
    for (uint64_t i = 0; i < n; ++i) {
        for (uint32_t b = r->read_blk[i]; b < r->read_blk[i + 1]; b += LRB_TILE_BLOCKS) {
            r->tile_read[t] = (uint32_t)i;
            r->tile_blk[t] = b;
            ++t;
        }
    }
    if (!alloc_stream) {   // the caller packed while reading (streamed gzip): codes / valid are in place and large enough
        r->codes[2 * blk] = r->codes[2 * blk + 1] = 0;
        r->valid[blk] = 0;
        return LRB_OK;
    }
    r->codes = (uint32_t*)lrb_host_alloc(sizeof(uint32_t) * (2 * blk + 2), &r->pinned, want_pinned);
    bool pinned2 = r->pinned;
    r->valid = r->codes ? (uint32_t*)lrb_host_alloc(sizeof(uint32_t) * (blk + 1), &pinned2, want_pinned) : nullptr;
    if (!r->codes || !r->valid) return lrb_set_error(LRB_ENOMEM, "out of memory (packed stream, %llu blocks)", (unsigned long long)blk);
    if (pinned2 != r->pinned) {  // keep one allocation kind for both
        lrb_host_free(r->valid, pinned2);
        lrb_host_free(r->codes, r->pinned);
        r->pinned = false;
        r->codes = (uint32_t*)calloc(2 * blk + 2, 4);
        r->valid = (uint32_t*)calloc(blk + 1, 4);
        if (!r->codes || !r->valid) return lrb_set_error(LRB_ENOMEM, "out of memory (packed stream)");
    } else if (zero) {
        memset(r->codes, 0, sizeof(uint32_t) * (2 * blk + 2));
        memset(r->valid, 0, sizeof(uint32_t) * (blk + 1));
    }
    r->codes[2 * blk] = r->codes[2 * blk + 1] = 0;  // the words after the stream
    r->valid[blk] = 0;
    return LRB_OK;
}

template <class GetSeq>
static void pack_all(lrb_reads* r, int threads, GetSeq get) {
    const uint64_t n = r->n_reads;
    threads = std::max(1, std::min(threads, 64));
    if (n < 64) threads = 1;
    auto work = [&](uint64_t lo, uint64_t hi) {
        for (uint64_t i = lo; i < hi; ++i)
            pack_read(get(i), r->read_len[i], r->codes + 2 * (size_t)r->read_blk[i], r->valid + r->read_blk[i]);
    };
    if (threads == 1) { work(0, n); return; }
    // split by blocks so threads get even byte counts
    std::vector<std::thread> pool;
    uint64_t lo = 0;
    for (int t = 0; t < threads; ++t) {
        const uint64_t target = r->n_blocks * (uint64_t)(t + 1) / threads;
        uint64_t hi = (t == threads - 1) ? n : (uint64_t)(std::upper_bound(r->read_blk, r->read_blk + n, (uint32_t)target) - r->read_blk);
        if (hi < lo) hi = lo;
        if (hi > n) hi = n;
        pool.emplace_back(work, lo, hi);
        lo = hi;
    }
    for (auto& th : pool) th.join();
}

// exception list = blocks whose valid word differs from default_valid (threads scan disjoint read ranges, in order)
static int index_valid(lrb_reads* r, int threads) {
    lrb_host_free(r->exc_blk, r->exc_pinned);
    lrb_host_free(r->exc_valid, r->exc_pinned);
    r->exc_blk = r->exc_valid = nullptr;
    r->n_exc = 0;
    r->exc_ready = false;
    const uint64_t n = r->n_reads;
    threads = std::max(1, std::min(threads, 64));
    if (n < 64) threads = 1;
    std::vector<std::vector<uint32_t>> found(threads);  // (block, word) pairs
    auto work = [&](int t, uint64_t lo, uint64_t hi) {
        std::vector<uint32_t>& f = found[t];
        for (uint64_t i = lo; i < hi; ++i) {
            const uint32_t b0 = r->read_blk[i], b1 = r->read_blk[i + 1], len = r->read_len[i];
            for (uint32_t b = b0; b < b1; ++b) {
                const uint32_t v = r->valid[b];
                if (v != lrb::default_valid_word(len, (uint64_t)(b - b0) * 32)) { f.push_back(b); f.push_back(v); }
            }
        }
    };
    if (threads == 1) work(0, 0, n);
    else {
        std::vector<std::thread> pool;
        uint64_t lo = 0;
        for (int t = 0; t < threads; ++t) {
            const uint64_t target = r->n_blocks * (uint64_t)(t + 1) / threads;
            uint64_t hi = (t == threads - 1) ? n : (uint64_t)(std::upper_bound(r->read_blk, r->read_blk + n, (uint32_t)target) - r->read_blk);
            hi = std::min(std::max(hi, lo), n);
            pool.emplace_back(work, t, lo, hi);
            lo = hi;
        }
        for (auto& th : pool) th.join();
    }
    uint64_t total = 0;
    for (auto& f : found) total += f.size() / 2;
    bool p1 = false, p2 = false;
    r->exc_blk = (uint32_t*)lrb_host_alloc(sizeof(uint32_t) * (total + 1), &p1, r->pinned);
    r->exc_valid = (uint32_t*)lrb_host_alloc(sizeof(uint32_t) * (total + 1), &p2, r->pinned);
    if (!r->exc_blk || !r->exc_valid || p1 != p2) {
        lrb_host_free(r->exc_blk, p1);
        lrb_host_free(r->exc_valid, p2);
        r->exc_blk = r->exc_valid = nullptr;
        return lrb_set_error(LRB_ENOMEM, "out of memory (validity exceptions)");
    }
    r->exc_pinned = p1;
    uint64_t k = 0;
    for (auto& f : found)
        for (size_t j = 0; j < f.size(); j += 2) { r->exc_blk[k] = f[j]; r->exc_valid[k] = f[j + 1]; ++k; }
    r->n_exc = total;
    r->exc_ready = true;
    return LRB_OK;
}

}  // namespace

// ---- segment reader: the read stream in chunks, delivered as read sets of bounded size -----------------------------------
// The file is read in chunks (gzip: inflated by zlib; plain: pread windows, never mapped whole) by a producer thread while
// the previous chunk is parsed (all `threads` ranges) and packed; a record whose parse ran into the end of the data read so
// far is kept back, with everything after it, for the next round.  Records go into the current SEGMENT until the next one
// would take it past its budget of bases or past kSegmentMaxBlocks; that record then starts the next segment (parsed again
// from its header), and a record longer than the budget forms a segment on its own.  Host memory: one segment's packed
// stream (0.375 B/base) + two chunks + one record, whatever the file's size.  Record semantics are parse_range's, so the
// concatenated segments equal the whole-image parse (tests: every fixture and the fuzz files, plain and gzip, with chunks
// and budgets down to 1 byte / 1 base, against the oracle reader).
namespace {

// A read set indexes its blocks with u32 (2^32 - 16 at most, build_layout); segments stay 2^28 blocks (8.6 Gbases) below.
constexpr uint64_t kSegmentMaxBlocks = 0xF0000000ull;
constexpr uint64_t kSegmentMaxBases = kSegmentMaxBlocks * 32;
// lrb_reader_open(.., 0, ..) sizes segments for the largest rows of a fused call: k = 5 composition + 32 coverage bins + sum
constexpr uint64_t kDefaultRowBytes = 4 * (512 + 32 + 1);
// the per-read estimate that turns result rows into bytes per base: long reads (ONT / HiFi) are several kb, so 1 kb is
// conservative for them; a read set of much shorter reads holds proportionally more rows per segment
constexpr uint64_t kReadLenEstimate = 1000;

struct GrowWords {
    uint32_t* p = nullptr;
    size_t cap = 0;  // words
    bool need(size_t words) {
        if (words <= cap) return true;
        size_t nc = std::max<size_t>(std::max<size_t>(words, cap + cap / 2), 1u << 16);
        void* q = realloc(p, nc * sizeof(uint32_t));
        if (!q) return false;
        p = (uint32_t*)q;
        cap = nc;
        return true;
    }
};

uint64_t mem_available_bytes() {
    if (FILE* f = fopen("/proc/meminfo", "r")) {
        char line[256];
        unsigned long long kb = 0;
        bool found = false;
        while (!found && fgets(line, sizeof line, f)) found = sscanf(line, "MemAvailable: %llu kB", &kb) == 1;
        fclose(f);
        if (found) return (uint64_t)kb << 10;
    }
    return (uint64_t)sysconf(_SC_AVPHYS_PAGES) * (uint64_t)sysconf(_SC_PAGESIZE);
}

}  // namespace

uint64_t lrb_segment_budget(uint64_t row_bytes_per_read) {
    const char* e = getenv("LRB_SEGMENT_BASES");   // tests: segments of a few bases
    if (e && atoll(e) > 0) return std::min<uint64_t>((uint64_t)atoll(e), kSegmentMaxBases);
    // half of MemAvailable for the stream (0.375 B/base) + the rows (row_bytes per kReadLenEstimate bases)
    const double per_base = 0.375 + (double)row_bytes_per_read / (double)kReadLenEstimate;
    const double bases = (double)(mem_available_bytes() / 2) / per_base;
    return (uint64_t)std::max(1.0, std::min(bases, (double)kSegmentMaxBases));
}

struct lrb_reader {
    std::string path;
    int threads = 1;
    uint64_t budget = kSegmentMaxBases;     // bases per segment
    uint64_t max_blocks = kSegmentMaxBlocks;
    bool whole = false;                      // one read set of the whole stream: passing max_blocks is an error, not a cut
    size_t chunk = 64u << 20;   // measured (200 MB FASTA, 8 threads): 64 MiB chunks 1.16 s, one 256 MiB chunk 1.52 s, whole image 1.19 s
    size_t min_chunk = 8u << 20;
    bool gz = false;
    gzFile f = nullptr;
    int fd = -1;
    uint64_t file_off = 0;
    std::vector<unsigned char> work, next;
    size_t next_n = 0;
    bool next_eof = false;
    bool pending = false;   // `work` holds complete records not delivered yet: the last segment was cut inside it
    bool done = false;
    uint64_t reads_out = 0, bases_out = 0, segments_out = 0;

    ~lrb_reader() {
        if (f) gzclose(f);
        if (fd >= 0) close(fd);
    }
    // fills `next`; a short read is the end of the stream (or of a damaged one: the tools stop quietly there too)
    void fill_next() {
        next_n = 0;
        next_eof = false;
        while (next_n < chunk) {
            const size_t want = std::min<size_t>(chunk - next_n, 1u << 30);
            const long got = gz ? (long)gzread(f, next.data() + next_n, (unsigned)want) : (long)pread(fd, next.data() + next_n, want, (off_t)file_off);
            if (got <= 0) { next_eof = true; break; }
            if (!gz) file_off += (uint64_t)got;
            next_n += (size_t)got;
        }
    }
    void start() {
        work.clear();
        pending = false;
        done = !f && fd < 0;   // unreadable file == empty stream, like the tools
        reads_out = bases_out = segments_out = 0;
        next_n = 0;
        next_eof = true;
        if (!done) fill_next();
    }
};

namespace {

int reader_open(const char* path, int threads, uint64_t segment_bases, bool whole, lrb_reader** out) {
    lrb_reader* rd = new lrb_reader();
    rd->path = path;
    rd->threads = std::max(1, std::min(threads, 64));
    rd->whole = whole;
    if (whole) { rd->budget = UINT64_MAX; rd->max_blocks = 0xFFFFFFF0ull; }
    else rd->budget = std::min<uint64_t>(segment_bases ? segment_bases : lrb_segment_budget(kDefaultRowBytes), kSegmentMaxBases);
    {
        const char* e = getenv("LRB_GZ_CHUNK");   // tests: chunks of a few bytes (plain files too)
        if (e && atoll(e) > 0) rd->chunk = (size_t)atoll(e);
        e = getenv("LRB_PARSE_CHUNK");
        if (e && atoll(e) > 0) rd->min_chunk = (size_t)atoll(e);
    }
    // a regular plain file is read with pread; gzip (and anything that is not a regular file) goes through zlib, which passes
    // plain data through unchanged (io_utils.h:143)
    const int fd = open(path, O_RDONLY);
    struct stat st;
    unsigned char magic[2] = {0, 0};
    const bool regular = fd >= 0 && fstat(fd, &st) == 0 && S_ISREG(st.st_mode);
    rd->gz = !regular || (pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b);
    if (rd->gz) {
        if (fd >= 0) close(fd);
        if (fd >= 0 && (rd->f = gzopen(path, "rb"))) gzbuffer(rd->f, 1 << 20);
    } else {
        rd->fd = fd;
    }
    rd->next.resize(rd->chunk);
    rd->start();
    *out = rd;
    return LRB_OK;
}

// The next segment (NULL once the stream is exhausted).
int reader_next(lrb_reader* rd, lrb_reads** out) {
    *out = nullptr;
    std::vector<uint32_t> lens;
    GrowWords codes, valid;
    uint64_t blk = 0, bases = 0;
    int rc = LRB_OK;
    bool full = false;
    struct Item { const unsigned char* s; uint32_t len; uint64_t blk; };
    std::vector<Item> items;
    std::vector<Parsed> parts;
    std::vector<unsigned char>& work = rd->work;
    const int threads = rd->threads;
    while (!full && !rd->done && rc == LRB_OK) {
        bool eof;   // nothing follows `work` in the stream
        std::thread producer;
        if (!rd->pending) {
            work.insert(work.end(), rd->next.begin(), rd->next.begin() + (ptrdiff_t)rd->next_n);
            rd->next_n = 0;
            eof = rd->next_eof;
            if (!eof) producer = std::thread([rd]() { rd->fill_next(); });   // the next chunk is read while this one is parsed and packed
        } else {
            eof = rd->next_eof && rd->next_n == 0;
        }
        bool ended = false;
        parse_all(work.data(), work.size(), threads, rd->min_chunk, parts, true, &ended);
        size_t carry_from = work.size();
        bool stop = eof;   // the stream ends for good behind this round's records
        if (!eof) {
            Parsed& last = parts.back();
            if (ended && !last.end_touched) stop = true;            // a malformed record ends the stream for good (kseq.h:209-214)
            else if (last.tail_open && !last.recs.empty()) {        // the last record may go on in the next chunk: parse it again then
                carry_from = (size_t)last.hdr.back();
                last.recs.pop_back();
                last.hdr.pop_back();
            } else carry_from = last.open_hdr;
        }
        items.clear();
        for (size_t pi = 0; pi < parts.size() && !full && rc == LRB_OK; ++pi) {
            Parsed& p = parts[pi];
            for (size_t j = 0; j < p.recs.size(); ++j) {
                const Record& rec = p.recs[j];
                const uint64_t nb = (uint64_t)rec.len / 32 + 1;
                if (blk + nb > rd->max_blocks && rd->whole) { rc = lrb_set_error(LRB_EINVAL, "read set too large: more than 2^32 blocks (137 Gbases)"); break; }
                if (!lens.empty() && (bases + rec.len > rd->budget || blk + nb > rd->max_blocks)) {   // starts the next segment
                    carry_from = (size_t)p.hdr[j];
                    full = true;
                    break;
                }
                items.push_back({rec.in_pool ? (const unsigned char*)p.pool.data() + rec.off : work.data() + rec.off, rec.len, blk});
                blk += nb;
                bases += rec.len;
                lens.push_back(rec.len);
            }
        }
        if (rc == LRB_OK && (!codes.need(2 * blk + 2) || !valid.need(blk + 1)))
            rc = lrb_set_error(LRB_ENOMEM, "out of memory (packed stream, %llu blocks)", (unsigned long long)blk);
        if (rc == LRB_OK && !items.empty()) {
            const int T = items.size() < 64 ? 1 : threads;
            auto work_fn = [&](size_t lo, size_t hi) {
                for (size_t i = lo; i < hi; ++i) pack_read(items[i].s, items[i].len, codes.p + 2 * items[i].blk, valid.p + items[i].blk);
            };
            if (T == 1) work_fn(0, items.size());
            else {
                std::vector<std::thread> pool;
                const uint64_t b_lo = items.front().blk, b_span = blk - b_lo;
                size_t lo = 0;
                for (int t = 0; t < T; ++t) {
                    size_t hi = items.size();
                    if (t + 1 < T) {
                        const uint64_t target = b_lo + b_span * (uint64_t)(t + 1) / (uint64_t)T;
                        hi = (size_t)(std::lower_bound(items.begin() + (ptrdiff_t)lo, items.end(), target, [](const Item& it, uint64_t v) { return it.blk < v; }) - items.begin());
                    }
                    pool.emplace_back(work_fn, lo, hi);
                    lo = hi;
                }
                for (auto& th : pool) th.join();
            }
        }
        if (producer.joinable()) producer.join();
        rd->pending = full;
        if (full || !stop) work.erase(work.begin(), work.begin() + (ptrdiff_t)carry_from);
        else { rd->done = true; work.clear(); }
    }
    if (rc) { free(codes.p); free(valid.p); rd->done = true; return rc; }
    if (lens.empty() && !rd->whole) { free(codes.p); free(valid.p); return LRB_OK; }
    lrb_reads* r = new lrb_reads();
    r->n_reads = lens.size();
    r->read_len = (uint32_t*)malloc(sizeof(uint32_t) * (lens.size() + 1));
    if (!r->read_len || !codes.need(2 * blk + 2) || !valid.need(blk + 1)) { free(codes.p); free(valid.p); free_reads(r); return lrb_set_error(LRB_ENOMEM, "out of memory (read_len)"); }
    if (!lens.empty()) memcpy(r->read_len, lens.data(), sizeof(uint32_t) * lens.size());
    r->codes = codes.p;
    r->valid = valid.p;
    r->pinned = false;
    if ((rc = build_layout(r, false, false, /*alloc_stream=*/false)) || (rc = index_valid(r, threads))) { free_reads(r); return rc; }
    rd->reads_out += r->n_reads;
    rd->bases_out += r->total_bases;
    rd->segments_out += 1;
    *out = r;
    return LRB_OK;
}

// gzip input of lrb_reads_from_file: the whole stream as one read set, read in chunks (round 1 inflated the whole file:
// a 100 Gbase .gz needed 100 GB of RAM; this needs the packed stream + two chunks + one record)
int reads_from_gz_stream(const char* path, int threads, lrb_reads** out) {
    lrb_reader* rd = nullptr;
    reader_open(path, threads, 0, /*whole=*/true, &rd);
    const int rc = reader_next(rd, out);
    delete rd;
    return rc;
}

}  // namespace

extern "C" int lrb_reader_open(const char* path, int threads, uint64_t segment_bases, lrb_reader** out) {
    if (!path || !out) return lrb_set_error(LRB_EINVAL, "lrb_reader_open: null argument");
    return reader_open(path, threads, segment_bases, /*whole=*/false, out);
}

extern "C" int lrb_reader_next(lrb_reader* rd, lrb_reads** out) {
    if (!rd || !out) return lrb_set_error(LRB_EINVAL, "lrb_reader_next: null argument");
    return reader_next(rd, out);
}

extern "C" int lrb_reader_rewind(lrb_reader* rd) {
    if (!rd) return lrb_set_error(LRB_EINVAL, "lrb_reader_rewind: null argument");
    if (rd->f && gzrewind(rd->f) != 0) return lrb_set_error(LRB_EIO, "cannot rewind %s", rd->path.c_str());
    rd->file_off = 0;
    rd->start();
    return LRB_OK;
}

extern "C" int lrb_reader_tell(const lrb_reader* rd, uint64_t* reads, uint64_t* bases, uint64_t* segments, int* at_end) {
    if (!rd) return lrb_set_error(LRB_EINVAL, "lrb_reader_tell: null argument");
    if (reads) *reads = rd->reads_out;
    if (bases) *bases = rd->bases_out;
    if (segments) *segments = rd->segments_out;
    if (at_end) *at_end = rd->done ? 1 : 0;
    return LRB_OK;
}

extern "C" void lrb_reader_close(lrb_reader* rd) { delete rd; }

extern "C" int lrb_reads_index_valid(lrb_reads* r, int threads, uint64_t* n_exceptions) {
    if (!r) return lrb_set_error(LRB_EINVAL, "lrb_reads_index_valid: null argument");
    const int rc = index_valid(r, threads);
    if (!rc && n_exceptions) *n_exceptions = r->n_exc;
    return rc;
}

extern "C" int lrb_reads_exceptions(const lrb_reads* r, const uint32_t** blk, const uint32_t** word, uint64_t* n) {
    if (!r || !blk || !word || !n) return lrb_set_error(LRB_EINVAL, "lrb_reads_exceptions: null argument");
    *blk = r->exc_ready ? r->exc_blk : nullptr;
    *word = r->exc_ready ? r->exc_valid : nullptr;
    *n = r->exc_ready ? r->n_exc : 0;
    return LRB_OK;
}

extern "C" int lrb_reads_from_file(const char* path, int threads, lrb_reads** out) {
    if (!path || !out) return lrb_set_error(LRB_EINVAL, "lrb_reads_from_file: null argument");
    *out = nullptr;
    const bool trace = getenv("LRB_INGEST_TRACE") != nullptr;
    auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    {   // gzip input: streamed (bounded host memory, inflate beside parse) unless LRB_GZ_WHOLE=1 asks for the whole image
        unsigned char magic[2] = {0, 0};
        const int fd = open(path, O_RDONLY);
        const bool gz = fd >= 0 && pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
        if (fd >= 0) close(fd);
        const char* whole = getenv("LRB_GZ_WHOLE");
        if (gz && !(whole && atoi(whole) > 0)) return reads_from_gz_stream(path, threads, out);
    }
    FileImage img;
    load_file(path, img);
    const double t1 = now();
    size_t min_chunk = 8u << 20;  // below this a range is not worth a thread
    {
        const char* e = getenv("LRB_PARSE_CHUNK");  // tests force tiny ranges to exercise the boundary logic
        if (e && atoll(e) > 0) min_chunk = (size_t)atoll(e);
    }
    std::vector<Parsed> parts;
    parse_all(img.data, img.size, threads, min_chunk, parts);
    const double t2 = now();
    uint64_t n_reads = 0;
    for (auto& p : parts) n_reads += p.recs.size();
    lrb_reads* r = new lrb_reads();
    r->n_reads = n_reads;
    r->read_len = (uint32_t*)malloc(sizeof(uint32_t) * (n_reads + 1));
    if (!r->read_len) { free_reads(r); return lrb_set_error(LRB_ENOMEM, "out of memory (read_len)"); }
    std::vector<const unsigned char*> ptr(n_reads + 1);
    {
        uint64_t i = 0;
        for (auto& p : parts)
            for (const Record& rec : p.recs) {
                r->read_len[i] = rec.len;
                ptr[i] = rec.in_pool ? (const unsigned char*)p.pool.data() + rec.off : img.data + rec.off;
                ++i;
            }
    }
    int rc = build_layout(r, false, pin_reads_default());
    if (rc) { free_reads(r); return rc; }
    const double t3 = now();
    pack_all(r, threads, [&](uint64_t i) { return ptr[i]; });
    const double t4 = now();
    if ((rc = index_valid(r, threads))) { free_reads(r); return rc; }
    if (trace)
        fprintf(stderr, "[lrb ingest] %zu bytes, %llu reads: load %.3f s, parse %.3f s (%zu ranges), layout+alloc %.3f s, pack %.3f s, index %.3f s\n",
                img.size, (unsigned long long)n_reads, t1 - t0, t2 - t1, parts.size(), t3 - t2, t4 - t3, now() - t4);
    *out = r;
    return LRB_OK;
}

extern "C" int lrb_reads_from_ascii(const char* bases, const uint64_t* offsets, uint64_t n_reads, int threads,
                                    lrb_reads** out) {
    if (!out || (n_reads && (!bases || !offsets))) return lrb_set_error(LRB_EINVAL, "lrb_reads_from_ascii: null argument");
    *out = nullptr;
    lrb_reads* r = new lrb_reads();
    r->n_reads = n_reads;
    r->read_len = (uint32_t*)malloc(sizeof(uint32_t) * (n_reads + 1));
    if (!r->read_len) { free_reads(r); return lrb_set_error(LRB_ENOMEM, "out of memory (read_len)"); }
    for (uint64_t i = 0; i < n_reads; ++i) {
        const uint64_t l = offsets[i + 1] - offsets[i];
        if (offsets[i + 1] < offsets[i] || l > 0xFFFFFFFFull) { free_reads(r); return lrb_set_error(LRB_EINVAL, "lrb_reads_from_ascii: bad offsets at read %llu", (unsigned long long)i); }
        r->read_len[i] = (uint32_t)l;
    }
    int rc = build_layout(r, false, pin_reads_default());
    if (rc) { free_reads(r); return rc; }
    pack_all(r, threads, [&](uint64_t i) { return (const unsigned char*)bases + offsets[i]; });
    if ((rc = index_valid(r, threads))) { free_reads(r); return rc; }
    *out = r;
    return LRB_OK;
}

extern "C" int lrb_reads_from_lengths(const uint32_t* lengths, uint64_t n_reads, lrb_reads** out) {
    if (!out || (n_reads && !lengths)) return lrb_set_error(LRB_EINVAL, "lrb_reads_from_lengths: null argument");
    *out = nullptr;
    lrb_reads* r = new lrb_reads();
    r->n_reads = n_reads;
    r->read_len = (uint32_t*)malloc(sizeof(uint32_t) * (n_reads + 1));
    if (!r->read_len) { free_reads(r); return lrb_set_error(LRB_ENOMEM, "out of memory (read_len)"); }
    if (n_reads) memcpy(r->read_len, lengths, sizeof(uint32_t) * n_reads);
    int rc = build_layout(r, true);
    if (rc) { free_reads(r); return rc; }
    *out = r;
    return LRB_OK;
}

// A contiguous run of reads as a read set of its own: index arrays rebased to block 0 / read 0, the packed stream
// shared with the parent (a read always starts on a block boundary, so the sub-stream is a plain sub-array).
extern "C" int lrb_reads_slice(const lrb_reads* p, uint64_t read_lo, uint64_t read_hi, lrb_reads** out) {
    if (!p || !out) return lrb_set_error(LRB_EINVAL, "lrb_reads_slice: null argument");
    *out = nullptr;
    if (read_hi > p->n_reads) read_hi = p->n_reads;
    if (read_lo > read_hi) read_lo = read_hi;
    const uint64_t n = read_hi - read_lo;
    const uint32_t b0 = p->read_blk[read_lo], b1 = p->read_blk[read_hi];
    const uint64_t t0 = (uint64_t)(std::lower_bound(p->tile_read, p->tile_read + p->n_tiles, (uint32_t)read_lo) - p->tile_read);
    const uint64_t t1 = (uint64_t)(std::lower_bound(p->tile_read, p->tile_read + p->n_tiles, (uint32_t)read_hi) - p->tile_read);
    lrb_reads* r = new lrb_reads();
    r->borrowed = true;
    r->pinned = p->pinned;
    r->n_reads = n;
    r->n_blocks = b1 - b0;
    r->n_tiles = t1 - t0;
    r->codes = p->codes + 2 * (size_t)b0;
    r->valid = p->valid + b0;
    r->read_len = (uint32_t*)malloc(sizeof(uint32_t) * (n + 1));
    r->read_blk = (uint32_t*)malloc(sizeof(uint32_t) * (n + 1));
    r->tile_read = (uint32_t*)malloc(sizeof(uint32_t) * (r->n_tiles + 1));
    r->tile_blk = (uint32_t*)malloc(sizeof(uint32_t) * (r->n_tiles + 1));
    if (!r->read_len || !r->read_blk || !r->tile_read || !r->tile_blk) { free_reads(r); return lrb_set_error(LRB_ENOMEM, "out of memory (slice index)"); }
    uint64_t bases = 0;
    for (uint64_t i = 0; i < n; ++i) {
        r->read_len[i] = p->read_len[read_lo + i];
        r->read_blk[i] = p->read_blk[read_lo + i] - b0;
        bases += r->read_len[i];
    }
    r->read_blk[n] = b1 - b0;
    r->total_bases = bases;
    for (uint64_t t = 0; t < r->n_tiles; ++t) {
        r->tile_read[t] = p->tile_read[t0 + t] - (uint32_t)read_lo;
        r->tile_blk[t] = p->tile_blk[t0 + t] - b0;
    }
    if (p->exc_ready) {  // the parent's exception list is ascending by block: the slice owns a contiguous stretch of it
        const uint32_t* e0 = std::lower_bound(p->exc_blk, p->exc_blk + p->n_exc, b0);
        const uint32_t* e1 = std::lower_bound(p->exc_blk, p->exc_blk + p->n_exc, b1);
        const uint64_t ne = (uint64_t)(e1 - e0);
        bool p1 = false, p2 = false;
        r->exc_blk = (uint32_t*)lrb_host_alloc(sizeof(uint32_t) * (ne + 1), &p1, false);
        r->exc_valid = (uint32_t*)lrb_host_alloc(sizeof(uint32_t) * (ne + 1), &p2, false);
        if (!r->exc_blk || !r->exc_valid) { free_reads(r); return lrb_set_error(LRB_ENOMEM, "out of memory (slice exceptions)"); }
        for (uint64_t i = 0; i < ne; ++i) {
            r->exc_blk[i] = e0[i] - b0;
            r->exc_valid[i] = p->exc_valid[(e0 - p->exc_blk) + i];
        }
        r->n_exc = ne;
        r->exc_pinned = false;
        r->exc_ready = true;
    }
    *out = r;
    return LRB_OK;
}

extern "C" int lrb_reads_view_get(const lrb_reads* r, lrb_reads_view* v) {
    if (!r || !v) return lrb_set_error(LRB_EINVAL, "lrb_reads_view_get: null argument");
    v->n_reads = r->n_reads;
    v->n_blocks = r->n_blocks;
    v->n_tiles = r->n_tiles;
    v->total_bases = r->total_bases;
    v->codes = r->codes;
    v->valid = r->valid;
    v->read_len = r->read_len;
    v->read_blk = r->read_blk;
    v->tile_read = r->tile_read;
    v->tile_blk = r->tile_blk;
    return LRB_OK;
}

extern "C" int lrb_reads_unpack(const lrb_reads* r, uint64_t i, char* dst, uint64_t cap) {
    if (!r || !dst || i >= r->n_reads) return lrb_set_error(LRB_EINVAL, "lrb_reads_unpack: bad argument");
    const uint32_t len = r->read_len[i];
    if (cap < len) return lrb_set_error(LRB_EINVAL, "lrb_reads_unpack: buffer too small");
    static const char letters[4] = {'A', 'C', 'T', 'G'};
    const uint32_t* codes = r->codes + 2 * (size_t)r->read_blk[i];
    for (uint32_t p = 0; p < len; ++p) dst[p] = letters[(codes[p >> 4] >> (30 - 2 * (p & 15))) & 3u];
    return LRB_OK;
}

extern "C" void lrb_reads_free(lrb_reads* r) { free_reads(r); }
