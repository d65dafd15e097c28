// api.cu — context / host-buffer / file level of the C ABI (see include/lrbinner_b200.h).
//
// lrb_ctx owns the device copy of one read set, the 4 GiB 15-mer table, the result buffers and the
// stream they are driven on.  lrb_profile_host is the seam-to-seam path: packed reads in (pinned) host
// memory -> H2D -> composition -> count -> mirror -> search -> D2H.  The file-level functions are the
// drop-ins for the reference's three executables (argv contracts in the header).
#include <cuda_runtime.h>
#include <errno.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "common.h"
#include "lane_core.cuh"
#include "synth_core.h"

using namespace lrb;

// ---- host allocation -------------------------------------------------------------------------
void* lrb_host_alloc(size_t bytes, bool* pinned, bool want_pinned) {
    void* p = nullptr;
    if (bytes == 0) bytes = 16;
    if (want_pinned) {
        if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) == cudaSuccess) {
            *pinned = true;
            return p;
        }
        cudaGetLastError();  // no device (host-only tests): plain memory; any later device call reports the real error
    }
    *pinned = false;
    if (posix_memalign(&p, 4096, bytes) != 0) return nullptr;
    return p;
}

void lrb_host_free(void* p, bool pinned) {
    if (!p) return;
    if (pinned) cudaFreeHost(p);
    else free(p);
}

extern "C" void* lrb_pinned_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocPortable) != cudaSuccess) {
        lrb_set_error(LRB_ECUDA, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}
extern "C" void lrb_pinned_free(void* p) { if (p) cudaFreeHost(p); }

// ---- context -----------------------------------------------------------------------------------
// dry run of the reserve() calls of a batch: "do the buffers of earlier calls already hold this batch?" (thread-local: every
// device plans on its own host thread)
static thread_local bool t_reserve_dry = false;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return LRB_OK;
        if (t_reserve_dry) return LRB_ENOMEM;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return lrb_set_error(LRB_ECUDA, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        cap = bytes;
        return LRB_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

constexpr int kMaxDevices = 16;
constexpr int kMaxRounds = LRB_PART_MAX_BUCKETS;

struct lrb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr, copy_in = nullptr, copy_out = nullptr, xchg = nullptr;
    cudaEvent_t ev[8] = {};
    cudaEvent_t sync_ev[LRB_PART_MAX_CHUNKS + 2] = {};  // [0] index arrays, [1..] H2D chunks, [last] composition D2H
    cudaEvent_t counted = nullptr;                       // this device's private counts are complete
    cudaEvent_t sum_ev[kMaxRounds] = {}, round_ev[kMaxRounds] = {};  // exchange: my piece of round k is summed / round k has arrived here
    cudaEvent_t xev[2] = {};                             // exchange start / end (timed)
    DevBuf codes, valid, read_len, read_blk, tile_read, tile_blk;
    DevBuf table, comp, hist, sums, text;
    DevBuf part_keys, part_small, part_steps, part_sub, blk_read;  // L2-resident (partitioned) table passes
    DevBuf exc_blk, exc_valid;                            // validity exceptions (lrb_dev_fill_valid)
    DevBuf stage;                                         // multi-GPU exchange: rows pulled from the peers
    lrb_partition part = {};
    bool table_ready = false;  // holds a complete (mirrored) table
    DevBuf sample[LRB_MAX_SAMPLE_TABLES];               // sample slots: compact tables (lrb_dev_table_compact), 2 GiB each
    bool sample_ready[LRB_MAX_SAMPLE_TABLES] = {};
    lrb_reads_view dview = {};
    float ms[7] = {0, 0, 0, 0, 0, 0, 0};
    std::vector<lrb_ctx*> peers;   // devices 1.. of a multi-GPU context (owned by the context of devices[0])
    bool peer_access = false;      // every pair of devices maps the other's memory (copies go GPU to GPU over NVLink)
    lrb_run_info info = {};
    // composition rows whose host destination is pageable: copied at the end of the call (a pageable D2H blocks the host
    // thread until everything enqueued before it has run, which would serialise the table passes behind it)
    uint32_t* comp_late_dst = nullptr;
    size_t comp_late_bytes = 0;
};

#define CTX_CUDA(expr)                                                                                    \
    do {                                                                                                  \
        cudaError_t e_ = (expr);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return lrb_set_error(LRB_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// The exchange stream runs at the highest priority: its small kernels (lrb_dev_add_planes, the mirror) then get SM slots
// ahead of the queued CTAs of the search they hide behind, instead of being stretched over the whole search
// (measured at N = 2: k_add_planes 2.2 ms per 16 MiB piece at default priority).
static cudaError_t create_xchg_stream(cudaStream_t* s) {
    int lo = 0, hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) return cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
    return cudaStreamCreateWithPriority(s, cudaStreamNonBlocking, hi);
}

static int ctx_create_one(int device, lrb_ctx** out) {
    CTX_CUDA(cudaSetDevice(device));
    lrb_ctx* c = new lrb_ctx();
    c->device = device;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->copy_in, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->copy_out, cudaStreamNonBlocking) != cudaSuccess ||
        create_xchg_stream(&c->xchg) != cudaSuccess) {
        const int rc = lrb_set_error(LRB_ECUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
        lrb_ctx_destroy(c);
        return rc;
    }
    for (auto& ev : c->ev) cudaEventCreate(&ev);
    for (auto& ev : c->xev) cudaEventCreate(&ev);
    for (auto& ev : c->sync_ev) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->counted, cudaEventDisableTiming);
    for (auto& ev : c->sum_ev) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    for (auto& ev : c->round_ev) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    *out = c;
    return LRB_OK;
}

extern "C" int lrb_ctx_create_multi(const int* devices, int n_devices, lrb_ctx** out) {
    if (!out) return lrb_set_error(LRB_EINVAL, "lrb_ctx_create: null out");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return lrb_set_error(LRB_ECUDA, "no CUDA device available (%s): liblrb200 has no CPU path", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (n_devices < 1 || n_devices > kMaxDevices) return lrb_set_error(LRB_EINVAL, "n_devices must be in [1, %d] (got %d)", kMaxDevices, n_devices);
    if (n_devices > n) return lrb_set_error(LRB_EINVAL, "%d GPUs asked for, %d visible", n_devices, n);
    int ids[kMaxDevices];
    for (int i = 0; i < n_devices; ++i) {
        ids[i] = devices ? devices[i] : i;
        if (ids[i] < 0 || ids[i] >= n) return lrb_set_error(LRB_EINVAL, "device %d out of range (have %d)", ids[i], n);
        for (int j = 0; j < i; ++j)
            if (ids[j] == ids[i]) return lrb_set_error(LRB_EINVAL, "device %d listed twice", ids[i]);
    }
    lrb_ctx* c = nullptr;
    int rc = ctx_create_one(ids[0], &c);
    if (rc) return rc;
    for (int i = 1; i < n_devices; ++i) {
        lrb_ctx* p = nullptr;
        if ((rc = ctx_create_one(ids[i], &p))) { lrb_ctx_destroy(c); return rc; }
        c->peers.push_back(p);
    }
    // peer mappings: with them the table exchange is GPU-to-GPU over NVLink; without, the driver stages the copies
    c->peer_access = n_devices > 1;
    for (int i = 0; i < n_devices && n_devices > 1; ++i)
        for (int j = 0; j < n_devices; ++j) {
            if (i == j) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, ids[i], ids[j]);
            if (!can) { c->peer_access = false; continue; }
            cudaSetDevice(ids[i]);
            const cudaError_t pe = cudaDeviceEnablePeerAccess(ids[j], 0);
            if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) c->peer_access = false;
            cudaGetLastError();
        }
    cudaSetDevice(ids[0]);
    *out = c;
    return LRB_OK;
}

extern "C" int lrb_ctx_create(int device, lrb_ctx** out) { return lrb_ctx_create_multi(&device, 1, out); }

extern "C" int lrb_ctx_device_count(const lrb_ctx* c) { return c ? 1 + (int)c->peers.size() : 0; }

extern "C" void lrb_ctx_destroy(lrb_ctx* c) {
    if (!c) return;
    for (lrb_ctx* p : c->peers) lrb_ctx_destroy(p);
    c->peers.clear();
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->xchg) cudaStreamSynchronize(c->xchg);
    for (DevBuf* b : {&c->codes, &c->valid, &c->read_len, &c->read_blk, &c->tile_read, &c->tile_blk, &c->table, &c->comp,
                      &c->hist, &c->sums, &c->text, &c->part_keys, &c->part_small, &c->part_steps, &c->part_sub, &c->blk_read, &c->exc_blk, &c->exc_valid, &c->stage})
        b->release();
    for (DevBuf& b : c->sample) b.release();
    for (auto& ev : c->ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : c->xev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : c->sync_ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : c->sum_ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : c->round_ev) if (ev) cudaEventDestroy(ev);
    if (c->counted) cudaEventDestroy(c->counted);
    if (c->copy_in) cudaStreamDestroy(c->copy_in);
    if (c->copy_out) cudaStreamDestroy(c->copy_out);
    if (c->xchg) cudaStreamDestroy(c->xchg);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

static int comp_width(int k) { return k == 3 ? 32 : k == 4 ? 136 : k == 5 ? 512 : 0; }

// ---- the profile stage over host buffers: batches x devices -------------------------------------------------------
//
// One call = two passes over the read set with the 15-mer table between them:
//   pass 1  per batch: H2D (chunked) || composition + key partition per chunk -> count into the device's table
//   exchange (n devices > 1): the devices' private tables are summed over NVLink peer memory, round by round
//   pass 2  per batch: search against the finished table -> coverage rows -> D2H
// A BATCH is a contiguous run of reads whose working set (packed stream + 8 B per slot of partition lists + result rows)
// fits the device beside the 4 GiB table; a batch is a read set of its own (lrb_reads_slice).  When a device's share is
// ONE batch — every BASELINE config on a 180 GB B200 — everything stays resident, the search re-uses the lists the count
// built, and the call is the 3-stream pipeline described in DESIGN.md section 5.  Larger inputs run in several batches:
// the table accumulates over pass 1 (u32 sums are associative), and pass 2 ships every batch again and partitions it
// once more (with read ids) for the search — the reference's constant-memory behaviour (count-15mers.cpp:75-99,
// search-15mers.cpp:99-119: reads stream through a bounded queue twice) instead of a failure or a silent slow path.
// Devices own contiguous read ranges (balanced by blocks), so row i of every output is read i of the input.
namespace {

struct Job {
    const lrb_reads* reads = nullptr;
    int k = 0, P = 0;
    CovLayout cov;                    // the coverage row (checked); a block with b[m].table >= 0 reads that sample slot
    uint32_t *comp = nullptr, *hist = nullptr, *sums = nullptr, *table_host = nullptr;
    bool do_comp = false, do_search = false, do_count = false, use_loaded = false, add_to_table = false;
    bool use_part = true, want_smem_env = false, force_l2 = false, comp_pinned = false;
    int bucket_shift = 24;
    bool force_ship_valid = false;
};

struct Batch { uint64_t r0, r1; };

struct DevPlan {
    lrb_ctx* c = nullptr;
    uint64_t r0 = 0, r1 = 0;          // this device's reads
    std::vector<Batch> batches;
    lrb_reads* kept = nullptr;        // single batch: the slice (or the parent itself) stays for pass 2
    bool kept_owned = false;
    int rc = LRB_OK;
    std::string err;
};

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return (e && *e) ? atoi(e) : dflt;
}

bool host_ptr_is_pinned(const void* p) {
    if (!p) return true;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// bytes of device memory a batch of `blocks` blocks / `reads` reads needs beside the table and the sample slots (both are
// allocated before the batches are planned, so the free memory the plan starts from already leaves them out)
uint64_t batch_bytes(const Job& J, uint64_t blocks, uint64_t reads, uint64_t tiles) {
    uint64_t b = blocks * 12 + 64;                                        // codes + valid
    b += reads * 8 + tiles * 8 + 64;                                      // read_len, read_blk, tiles
    if (J.do_comp) b += reads * 4ull * J.P;
    if (J.do_search) b += reads * 4ull * (J.cov.W + 1);
    if (J.use_part && (J.do_count || J.do_search)) {
        b += blocks * 128 + blocks * 4;                                   // 4 B per slot of list entries, blk_read
        b += 4ull * lrb_partition_steps_words(lrb_partition_step_capacity(blocks, LRB_PART_MAX_CHUNKS));
        if (J.do_count && !J.force_l2 && blocks >= (1u << 19)) b += blocks * 128 + (8u << 20);   // second-level lists (2 x 2 B per slot)
    }
    return b + (64u << 20);                                               // allocator granularity, small scratch
}

int reserve_batch(lrb_ctx* c, const lrb_reads* r, const Job& J, bool want_count_lists) {
    const uint64_t n = r->n_reads, nb = r->n_blocks, nt = r->n_tiles;
    int rc;
    if ((rc = c->codes.reserve(sizeof(uint32_t) * (2 * nb + 2)))) return rc;
    if ((rc = c->valid.reserve(sizeof(uint32_t) * (nb + 1)))) return rc;
    if ((rc = c->read_len.reserve(sizeof(uint32_t) * (n + 1)))) return rc;
    if ((rc = c->read_blk.reserve(sizeof(uint32_t) * (n + 1)))) return rc;
    if ((rc = c->tile_read.reserve(sizeof(uint32_t) * (nt + 1)))) return rc;
    if ((rc = c->tile_blk.reserve(sizeof(uint32_t) * (nt + 1)))) return rc;
    if (J.do_comp && (rc = c->comp.reserve(std::max<size_t>(16, sizeof(uint32_t) * n * J.P)))) return rc;
    if (J.do_search) {
        if ((rc = c->hist.reserve(std::max<size_t>(16, sizeof(uint32_t) * n * (size_t)J.cov.W)))) return rc;
        if ((rc = c->sums.reserve(std::max<size_t>(16, sizeof(uint32_t) * n)))) return rc;
    }
    if ((rc = c->exc_blk.reserve(sizeof(uint32_t) * (r->n_exc + 1)))) return rc;
    if ((rc = c->exc_valid.reserve(sizeof(uint32_t) * (r->n_exc + 1)))) return rc;
    if (J.use_part && (J.do_count || J.do_search) && nb > 0) {
        const size_t cap = std::max<uint64_t>(nb * 32, 1);  // >= number of slots: the lists can never overflow
        const uint64_t step_cap = lrb_partition_step_capacity(nb, LRB_PART_MAX_CHUNKS);
        if ((rc = c->part_keys.reserve(sizeof(uint32_t) * cap))) return rc;
        if ((rc = c->part_steps.reserve(sizeof(uint32_t) * lrb_partition_steps_words(step_cap)))) return rc;
        if ((rc = c->part_small.reserve(sizeof(unsigned long long) * LRB_PART_SMALL_U64))) return rc;
        if ((rc = c->blk_read.reserve(sizeof(uint32_t) * (nb + 1)))) return rc;
        c->part.keys = (uint32_t*)c->part_keys.p;
        c->part.steps = (uint32_t*)c->part_steps.p;
        c->part.small = (unsigned long long*)c->part_small.p;
        c->part.capacity = cap;
        c->part.step_capacity = step_cap;
        // second-level lists for the shared-memory count: worth it once the batch is large
        c->part.sub = nullptr;
        c->part.sub_capacity = 0;
        const bool want_smem = J.want_smem_env || nb >= (1u << 19);
        if (want_count_lists && want_smem && !J.force_l2) {
            const size_t sub_cap = 2 * cap + (1u << 22);  // 2-byte entries in fixed-size segments: 2x headroom + fill counters and dump areas
            if ((rc = c->part_sub.reserve(sizeof(uint16_t) * sub_cap))) return rc;
            c->part.sub = (uint16_t*)c->part_sub.p;
            c->part.sub_capacity = sub_cap;
        }
    }
    lrb_reads_view& v = c->dview;
    v.n_reads = n; v.n_blocks = nb; v.n_tiles = nt; v.total_bases = r->total_bases;
    v.codes = (const uint32_t*)c->codes.p; v.valid = (const uint32_t*)c->valid.p;
    v.read_len = (const uint32_t*)c->read_len.p; v.read_blk = (const uint32_t*)c->read_blk.p;
    v.tile_read = (const uint32_t*)c->tile_read.p; v.tile_blk = (const uint32_t*)c->tile_blk.p;
    return LRB_OK;
}

struct ChunkPlan {
    int n = 1;
    std::vector<uint64_t> cr, cb, ct;  // read / block / tile cut points
};

ChunkPlan plan_chunks(const lrb_reads* r, int want) {
    ChunkPlan p;
    const uint64_t n = r->n_reads, nb = r->n_blocks, nt = r->n_tiles;
    p.n = (int)std::min<uint64_t>((uint64_t)std::min(want, LRB_PART_MAX_CHUNKS), std::max<uint64_t>(1, nb >> 16));
    p.cr.assign(p.n + 1, 0); p.cb.assign(p.n + 1, 0); p.ct.assign(p.n + 1, 0);
    for (int i = 1; i < p.n; ++i) {
        const uint32_t target = (uint32_t)(nb * (uint64_t)i / p.n);
        uint64_t ri = (uint64_t)(std::upper_bound(r->read_blk, r->read_blk + n, target) - r->read_blk);
        if (ri > 0) --ri;
        ri = std::max(ri, p.cr[i - 1]);
        p.cr[i] = ri;
        p.cb[i] = r->read_blk[ri];
        p.ct[i] = (uint64_t)(std::lower_bound(r->tile_read, r->tile_read + nt, (uint32_t)ri) - r->tile_read);
    }
    p.cr[p.n] = n; p.cb[p.n] = nb; p.ct[p.n] = nt;
    return p;
}

// H2D of one batch on copy_in (index arrays, validity exceptions or bitmap, codes in chunks cut at read boundaries); the
// compute stream picks the chunks up through sync_ev[1 + i].  Returns whether the validity bitmap was shipped.
int enqueue_upload(lrb_ctx* c, const lrb_reads* r, const Job& J, const ChunkPlan& ch, bool* shipped_valid) {
    const uint64_t n = r->n_reads, nb = r->n_blocks, nt = r->n_tiles;
    cudaStream_t sin = c->copy_in;
    // validity bitmap: when the reads carry their exception list (blocks whose valid word is not implied by the read
    // length) and it is short, only codes + exceptions cross PCIe (0.25 instead of 0.375 B/base) and the bitmap is
    // rebuilt on the device; LRB_SHIP_VALID=1 forces the plain copy.
    const bool ship_valid = J.force_ship_valid || !(r->exc_ready && r->n_exc <= nb / 16);
    *shipped_valid = ship_valid;
    if (n) CTX_CUDA(cudaMemcpyAsync(c->read_len.p, r->read_len, sizeof(uint32_t) * n, cudaMemcpyHostToDevice, sin));
    CTX_CUDA(cudaMemcpyAsync(c->read_blk.p, r->read_blk, sizeof(uint32_t) * (n + 1), cudaMemcpyHostToDevice, sin));
    if (nt) {
        CTX_CUDA(cudaMemcpyAsync(c->tile_read.p, r->tile_read, sizeof(uint32_t) * nt, cudaMemcpyHostToDevice, sin));
        CTX_CUDA(cudaMemcpyAsync(c->tile_blk.p, r->tile_blk, sizeof(uint32_t) * nt, cudaMemcpyHostToDevice, sin));
    }
    if (!ship_valid && r->n_exc) {
        CTX_CUDA(cudaMemcpyAsync(c->exc_blk.p, r->exc_blk, sizeof(uint32_t) * r->n_exc, cudaMemcpyHostToDevice, sin));
        CTX_CUDA(cudaMemcpyAsync(c->exc_valid.p, r->exc_valid, sizeof(uint32_t) * r->n_exc, cudaMemcpyHostToDevice, sin));
    }
    // the two code words / one validity word after the stream are never part of a window; a slice's host copy of them
    // belongs to the next read, so they are zeroed here instead of shipped
    CTX_CUDA(cudaMemsetAsync((uint32_t*)c->codes.p + 2 * nb, 0, 2 * sizeof(uint32_t), sin));
    CTX_CUDA(cudaMemsetAsync((uint32_t*)c->valid.p + nb, 0, sizeof(uint32_t), sin));
    CTX_CUDA(cudaEventRecord(c->sync_ev[0], sin));
    for (int i = 0; i < ch.n; ++i) {
        const uint64_t b0 = ch.cb[i], b1 = ch.cb[i + 1];
        if (b1 > b0) {
            CTX_CUDA(cudaMemcpyAsync((uint32_t*)c->codes.p + 2 * b0, r->codes + 2 * b0, sizeof(uint32_t) * 2 * (b1 - b0), cudaMemcpyHostToDevice, sin));
            if (ship_valid)
                CTX_CUDA(cudaMemcpyAsync((uint32_t*)c->valid.p + b0, r->valid + b0, sizeof(uint32_t) * (b1 - b0), cudaMemcpyHostToDevice, sin));
        }
        CTX_CUDA(cudaEventRecord(c->sync_ev[1 + i], sin));
    }
    return LRB_OK;
}

// Pass 1 of one batch.  row0 = index of the batch's first read in the caller's output arrays.  with_rids: the lists will
// also serve the search (single-batch mode).  timed: record the phase events of lrb_ctx_last_timings.  add_into_table: the
// device's table is complete already (LRB_PROFILE_ADD_TO_TABLE on the primary device): the count adds to it, never zeroes
// or writes it.
int stage_front(lrb_ctx* c, const lrb_reads* r, const Job& J, uint64_t row0, bool with_rids, bool defer_comp, bool timed,
                bool first_batch = false, bool only_batch = false, bool add_into_table = false) {
    CTX_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = c->stream, sin = c->copy_in, sout = c->copy_out;
    const uint64_t n = r->n_reads, nb = r->n_blocks;
    const bool lists = J.use_part && nb > 0 && (J.do_count || (with_rids && J.do_search));
    int rc;
    if ((rc = reserve_batch(c, r, J, J.do_count))) {
        // buffers left over from a differently shaped earlier call can add up to more than the device has (the plan counts
        // them as reusable): give everything back and allocate this batch afresh before calling it an error
        for (DevBuf* b : {&c->codes, &c->valid, &c->read_len, &c->read_blk, &c->tile_read, &c->tile_blk, &c->comp, &c->hist, &c->sums,
                          &c->part_keys, &c->part_steps, &c->part_sub, &c->blk_read, &c->exc_blk, &c->exc_valid, &c->text})
            b->release();
        cudaGetLastError();
        if ((rc = reserve_batch(c, r, J, J.do_count))) return rc;
    }
    const ChunkPlan ch = plan_chunks(r, 16);
    if (timed) CTX_CUDA(cudaEventRecord(c->ev[0], st));
    else CTX_CUDA(cudaEventRecord(c->sync_ev[LRB_PART_MAX_CHUNKS + 1], st));
    CTX_CUDA(cudaStreamWaitEvent(sin, timed ? c->ev[0] : c->sync_ev[LRB_PART_MAX_CHUNKS + 1], 0));   // earlier work is done with the buffers
    CTX_CUDA(cudaStreamWaitEvent(sout, timed ? c->ev[0] : c->sync_ev[LRB_PART_MAX_CHUNKS + 1], 0));
    bool ship_valid = false;
    if ((rc = enqueue_upload(c, r, J, ch, &ship_valid))) return rc;
    if (timed) CTX_CUDA(cudaEventRecord(c->ev[1], sin));  // H2D done
    lrb_reads_view& v = c->dview;
    // compute stream: zero the outputs while the first chunk is in flight.  The table is zeroed only when counts will be
    // ADDED to it (several batches, or no lists): a device's only batch WRITES its table slices (apply mode bit 3).
    const bool count_writes = J.do_count && lists && only_batch && !add_into_table;
    if (J.do_count && first_batch && !count_writes && !add_into_table)
        CTX_CUDA(cudaMemsetAsync(c->table.p, 0, sizeof(uint32_t) * (size_t)kTableEntries, st));
    if (J.do_comp && n) CTX_CUDA(cudaMemsetAsync(c->comp.p, 0, sizeof(uint32_t) * n * J.P, st));
    CTX_CUDA(cudaStreamWaitEvent(st, c->sync_ev[0], 0));  // index arrays (and validity exceptions) are on the device
    if (!ship_valid && (rc = lrb_dev_fill_valid(&v, (const uint32_t*)c->exc_blk.p, (const uint32_t*)c->exc_valid.p, r->n_exc, st))) return rc;
    if (lists) {
        if (with_rids && (rc = lrb_dev_fill_blk_read(&v, (uint32_t*)c->blk_read.p, st))) return rc;
        if ((rc = lrb_dev_partition_begin(&c->part, with_rids ? 1 : 0, 0, kTableEntries, J.bucket_shift, st))) return rc;
    }
    for (int i = 0; i < ch.n; ++i) {
        CTX_CUDA(cudaStreamWaitEvent(st, c->sync_ev[1 + i], 0));
        if (J.do_comp && n && (rc = lrb_dev_composition(&v, J.k, (uint32_t*)c->comp.p, ch.ct[i], ch.ct[i + 1], st))) return rc;
        if (lists) {
            if ((rc = lrb_dev_partition_add(&v, (const uint32_t*)c->blk_read.p, ch.cb[i], ch.cb[i + 1], &c->part, st))) return rc;
        } else if (J.do_count && !J.use_part) {
            if ((rc = lrb_dev_count(&v, (uint32_t*)c->table.p, ch.cb[i], ch.cb[i + 1], 0, kTableEntries, st))) return rc;
        }
    }
    if (timed) CTX_CUDA(cudaEventRecord(c->ev[2], st));  // composition (+ partition) of every chunk done
    c->comp_late_dst = nullptr;
    if (J.do_comp && n) {
        uint32_t* dst = J.comp + (size_t)row0 * J.P;
        const size_t bytes = sizeof(uint32_t) * n * J.P;
        if (defer_comp) {                          // pageable destination: goes home at the end of the call
            c->comp_late_dst = dst;
            c->comp_late_bytes = bytes;
        } else {                                   // composition rows go home while the table passes run
            CTX_CUDA(cudaEventRecord(c->sync_ev[LRB_PART_MAX_CHUNKS + 1], st));
            CTX_CUDA(cudaStreamWaitEvent(sout, c->sync_ev[LRB_PART_MAX_CHUNKS + 1], 0));
            CTX_CUDA(cudaMemcpyAsync(dst, c->comp.p, bytes, cudaMemcpyDeviceToHost, sout));
        }
    }
    CTX_CUDA(cudaEventRecord(c->sync_ev[LRB_PART_MAX_CHUNKS + 1], sout));
    if (J.do_count && lists) {
        // ONE launch over all buckets when the second-level lists exist (no per-bucket tails), else RED.ADD per bucket
        const int mode = (c->part.sub ? (1 | 4) : 1) | (count_writes ? 8 : 0);
        if ((rc = lrb_dev_partition_apply(&c->part, mode, (uint32_t*)c->table.p, 1, 1, nullptr, nullptr, st))) return rc;
    }
    return LRB_OK;
}

// Pass 2: coverage rows of the batch's reads against the device's (finished) table, buckets [b_lo, b_hi) of the lists.
int search_lists(lrb_ctx* c, const Job& J, uint64_t n, int b_lo, int b_hi) {
    if (!n) return LRB_OK;
    const uint32_t* slots[LRB_MAX_SAMPLE_TABLES];
    for (int t = 0; t < LRB_MAX_SAMPLE_TABLES; ++t) slots[t] = (const uint32_t*)c->sample[t].p;
    return lrb_partition_search("lrb_profile_host", &c->part, b_lo, b_hi, (const uint32_t*)c->table.p, slots, J.cov, (uint32_t*)c->hist.p,
                                (uint32_t*)c->sums.p, c->stream);
}

int rows_home(lrb_ctx* c, const Job& J, uint64_t n, uint64_t row0) {
    cudaStream_t st = c->stream;
    if (J.do_search && n) {
        CTX_CUDA(cudaMemcpyAsync(J.hist + (size_t)row0 * J.cov.W, c->hist.p, sizeof(uint32_t) * n * (size_t)J.cov.W, cudaMemcpyDeviceToHost, st));
        CTX_CUDA(cudaMemcpyAsync(J.sums + row0, c->sums.p, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, st));
    }
    CTX_CUDA(cudaStreamWaitEvent(st, c->sync_ev[LRB_PART_MAX_CHUNKS + 1], 0));  // join the copy_out stream (early composition D2H)
    if (c->comp_late_dst) {
        CTX_CUDA(cudaMemcpyAsync(c->comp_late_dst, c->comp.p, c->comp_late_bytes, cudaMemcpyDeviceToHost, st));
        c->comp_late_dst = nullptr;
    }
    return LRB_OK;
}

int sync_ctx(lrb_ctx* c) {
    CTX_CUDA(cudaSetDevice(c->device));
    CTX_CUDA(cudaStreamSynchronize(c->stream));
    CTX_CUDA(cudaStreamSynchronize(c->copy_in));
    CTX_CUDA(cudaStreamSynchronize(c->copy_out));
    CTX_CUDA(cudaStreamSynchronize(c->xchg));
    CTX_CUDA(cudaGetLastError());
    return LRB_OK;
}

// f(plan) on every device, one host thread per device beyond the first; the first failure becomes the caller's error
template <class F>
int on_devices(std::vector<DevPlan>& plans, F f) {
    auto run = [&](DevPlan& p) {
        p.rc = f(p);
        if (p.rc) p.err = lrb_last_error();
    };
    if (plans.size() == 1) run(plans[0]);
    else {
        std::vector<std::thread> pool;
        for (size_t i = 1; i < plans.size(); ++i) pool.emplace_back([&, i] { run(plans[i]); });
        run(plans[0]);
        for (auto& t : pool) t.join();
    }
    for (auto& p : plans)
        if (p.rc) return lrb_set_error(p.rc, "%s (device %d)", p.err.c_str(), p.c->device);
    return LRB_OK;
}

// pitched rows between two devices' tables (or a table and a staging plane)
int copy_rows(lrb_ctx* dst_ctx, void* dst, uint64_t dpitch, const lrb_ctx* src_ctx, const void* src, uint64_t spitch, uint64_t width,
              uint64_t rows, bool peer_access, cudaStream_t st) {
    if (!rows) return LRB_OK;
    if (peer_access) {
        CTX_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, cudaMemcpyDeviceToDevice, st));
    } else {
        cudaMemcpy3DPeerParms p;
        memset(&p, 0, sizeof p);
        p.srcDevice = src_ctx->device;
        p.dstDevice = dst_ctx->device;
        p.srcPtr = make_cudaPitchedPtr(const_cast<void*>(src), spitch, width, rows);
        p.dstPtr = make_cudaPitchedPtr(dst, dpitch, width, rows);
        p.extent = make_cudaExtent(width, rows, 1);
        CTX_CUDA(cudaMemcpy3DPeerAsync(&p, st));
    }
    return LRB_OK;
}

// Sum of the devices' private tables, left in every device's table (canonical half only: count touches nothing else).
// Reduce-scatter + all-gather by hand over peer memory, moved by the copy engines, in rounds so that the search of a
// round's buckets can start while later rounds are still on NVLink.  The canonical rows (2^14 rows of 2^15 entries, pitch
// 2^16) are cut into pieces of `g` buckets; round k handles the pieces k D .. k D + D - 1, piece q owned by device q mod D:
//   A  the owner pulls the piece's rows out of every peer's table into staging planes and adds them to its own rows
//      (lrb_dev_add_planes); sum_ev[k] says the piece is final;
//   B  every device pulls the round's other pieces from their owners (after their sum_ev[k]) over its own rows; round_ev[k].
// A device never writes rows a peer may still be reading: B overwrites piece q only after the owner of q has summed it,
// i.e. has finished reading everybody's private rows of q.
struct XchgSchedule {
    int n_rounds = 0, buckets_per_piece = 1, n_pieces = 0;
    int round_bucket_lo(int k, int D) const { return std::min(n_pieces, k * D) * buckets_per_piece; }
};

int enqueue_exchange(std::vector<DevPlan>& plans, int n_buckets, int shift, bool peer_access, XchgSchedule* sched) {
    const int D = (int)plans.size();
    const int g = std::max(1, n_buckets / (8 * D));                 // about 8 rounds
    const int G = (n_buckets + g - 1) / g;
    const int n_rounds = (G + D - 1) / D;
    sched->n_rounds = n_rounds; sched->buckets_per_piece = g; sched->n_pieces = G;
    const uint64_t rows_per_bucket = (1ull << shift) >> 16;         // table rows (2^16 entries) per bucket
    const uint64_t row_bytes = 4ull << 15, pitch_bytes = 4ull << 16;
    const uint64_t piece_rows = rows_per_bucket * g;
    auto piece_span = [&](int q, uint64_t* r0, uint64_t* r1) {
        *r0 = (uint64_t)q * piece_rows;
        *r1 = std::min<uint64_t>((uint64_t)n_buckets * rows_per_bucket, *r0 + piece_rows);
    };
    int rc;
    for (int d = 0; d < D; ++d) {
        lrb_ctx* c = plans[d].c;
        CTX_CUDA(cudaSetDevice(c->device));
        if ((rc = c->stage.reserve((size_t)(D - 1) * piece_rows * row_bytes))) return rc;
        CTX_CUDA(cudaEventRecord(c->counted, c->stream));
    }
    for (int d = 0; d < D; ++d) {
        lrb_ctx* c = plans[d].c;
        CTX_CUDA(cudaSetDevice(c->device));
        for (int p = 0; p < D; ++p) CTX_CUDA(cudaStreamWaitEvent(c->xchg, plans[p].c->counted, 0));
        CTX_CUDA(cudaEventRecord(c->xev[0], c->xchg));
    }
    for (int k = 0; k < n_rounds; ++k) {
        for (int d = 0; d < D; ++d) {   // A
            lrb_ctx* c = plans[d].c;
            CTX_CUDA(cudaSetDevice(c->device));
            const int q = k * D + d;
            if (q < G) {
                uint64_t r0, r1;
                piece_span(q, &r0, &r1);
                for (int j = 1; j < D; ++j) {   // rotated: no two devices start on the same peer
                    const lrb_ctx* s = plans[(d + j) % D].c;
                    if ((rc = copy_rows(c, (char*)c->stage.p + (size_t)(j - 1) * piece_rows * row_bytes, row_bytes, s,
                                        (const char*)s->table.p + r0 * pitch_bytes, pitch_bytes, row_bytes, r1 - r0, peer_access, c->xchg)))
                        return rc;
                }
                if ((rc = lrb_dev_add_planes((uint32_t*)((char*)c->table.p + r0 * pitch_bytes), pitch_bytes / 4, (const uint32_t*)c->stage.p,
                                             piece_rows * row_bytes / 4, D - 1, (uint32_t)(row_bytes / 4), (uint32_t)(r1 - r0), c->xchg)))
                    return rc;
            }
            CTX_CUDA(cudaEventRecord(c->sum_ev[k], c->xchg));
        }
        for (int d = 0; d < D; ++d) {   // B
            lrb_ctx* c = plans[d].c;
            CTX_CUDA(cudaSetDevice(c->device));
            for (int j = 1; j < D; ++j) {
                const int o = (d + j) % D, q = k * D + o;
                if (q >= G) continue;
                const lrb_ctx* s = plans[o].c;
                uint64_t r0, r1;
                piece_span(q, &r0, &r1);
                CTX_CUDA(cudaStreamWaitEvent(c->xchg, s->sum_ev[k], 0));
                if ((rc = copy_rows(c, (char*)c->table.p + r0 * pitch_bytes, pitch_bytes, s, (const char*)s->table.p + r0 * pitch_bytes, pitch_bytes,
                                    row_bytes, r1 - r0, peer_access, c->xchg)))
                    return rc;
            }
            CTX_CUDA(cudaEventRecord(c->round_ev[k], c->xchg));
        }
    }
    for (int d = 0; d < D; ++d) {
        lrb_ctx* c = plans[d].c;
        CTX_CUDA(cudaSetDevice(c->device));
        CTX_CUDA(cudaEventRecord(c->xev[1], c->xchg));
    }
    return LRB_OK;
}

}  // namespace

// Seam-to-seam pipeline (see the block comment above).  Phase timings of device 0's first batch
// (lrb_ctx_last_timings) overlap; [6] is the whole call on device 0's stream; lrb_ctx_last_info has the wall clock.
static bool direct_table_path() {   // one random HBM access per window (kernels.cu): experiments only
    const char* e = getenv("LRB_TABLE_PATH");
    return e && !strcmp(e, "direct");
}

// The direct search takes one (bin_size, bins) block of the full-layout table.
static int refuse_direct(const char* who, const CovLayout& cov) {
    if (cov.single() || !direct_table_path()) return LRB_OK;
    char what[32];
    if (cov.kind == CovKind::blocks) snprintf(what, sizeof what, "a layout of %d blocks", cov.n);
    else if (cov.kind == CovKind::samples) snprintf(what, sizeof what, "sample tables");
    else if (cov.b[0].by_edges) snprintf(what, sizeof what, "count edges");
    else snprintf(what, sizeof what, "%d settings", cov.n);
    return lrb_set_error(LRB_EINVAL, "%s: LRB_TABLE_PATH=direct searches the full-layout table with one (bin_size, bins) setting per call, not %s",
                         who, what);
}

// cov: checked (lrb_check_cov_layout); a block with b[m].table >= 0 searches that sample slot instead of the context's table
static int profile_host(const char* who, lrb_ctx* c, const lrb_reads* r, int k, const CovLayout& cov, uint32_t* comp_counts,
                        uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags) {
    Job J;
    J.reads = r; J.k = k; J.P = comp_width(k);
    J.comp = comp_counts; J.hist = cov_hist; J.sums = cov_sums; J.table_host = table_host;
    J.cov = cov;
    J.do_comp = comp_counts != nullptr;
    if (J.do_comp && !J.P) return lrb_set_error(LRB_EINVAL, "k must be 3, 4 or 5 (got %d)", k);
    J.do_search = cov_hist || cov_sums;
    if (J.do_search && (!cov_hist || !cov_sums)) return lrb_set_error(LRB_EINVAL, "cov_hist and cov_sums go together");
    if (cov.reads_slots() && !J.do_search) return lrb_set_error(LRB_EINVAL, "%s: sample tables need cov_hist and cov_sums", who);
    for (int t = 0; t < cov.n; ++t)
        if (cov.b[t].table >= 0 && !c->sample_ready[cov.b[t].table])
            return lrb_set_error(LRB_EINVAL, "%s: sample slot %d is empty (%s %d)", who, cov.b[t].table, cov.kind == CovKind::blocks ? "block" : "table", t);
    int rc;
    if (J.do_search && (rc = refuse_direct(who, cov))) return rc;
    J.use_loaded = (flags & LRB_PROFILE_USE_LOADED_TABLE) != 0;
    J.add_to_table = (flags & LRB_PROFILE_ADD_TO_TABLE) != 0;
    if (J.use_loaded && J.add_to_table) return lrb_set_error(LRB_EINVAL, "LRB_PROFILE_USE_LOADED_TABLE and LRB_PROFILE_ADD_TO_TABLE exclude each other");
    if ((J.use_loaded || J.add_to_table) && !c->table_ready) return lrb_set_error(LRB_EINVAL, "no table loaded in this context");
    J.do_count = !J.use_loaded && ((J.do_search && cov.reads_full()) || table_host || (flags & (LRB_PROFILE_KEEP_TABLE | LRB_PROFILE_ADD_TO_TABLE)));
    {
        if (direct_table_path()) J.use_part = false;
        const char* e = getenv("LRB_COUNT_PATH");
        J.want_smem_env = e && !strcmp(e, "smem");
        J.force_l2 = e && !strcmp(e, "l2");
        const int bl = env_int("LRB_BUCKET_LOG2", 24);
        if (bl >= 24 && bl <= 25) J.bucket_shift = bl;
        J.force_ship_valid = env_int("LRB_SHIP_VALID", 0) > 0;
    }
    J.comp_pinned = host_ptr_is_pinned(comp_counts);
    const auto wall0 = std::chrono::steady_clock::now();
    const uint64_t n = r->n_reads, nb = r->n_blocks;
    const bool need_table = J.do_count || (J.do_search && cov.reads_full());   // sample slots are allocated already

    // ---- devices and their read ranges (contiguous, balanced by blocks) ------------------------------------------
    std::vector<DevPlan> plans;
    {
        std::vector<lrb_ctx*> devs{c};
        for (lrb_ctx* p : c->peers) devs.push_back(p);
        const uint64_t min_blocks = (uint64_t)std::max(1, env_int("LRB_MIN_BLOCKS_PER_DEVICE", 1 << 12));   // tests lower it
        while (devs.size() > 1 && nb < devs.size() * min_blocks) devs.pop_back();   // tiny input: fewer devices
        const int D = (int)devs.size();
        uint64_t lo = 0;
        for (int d = 0; d < D; ++d) {
            DevPlan p;
            p.c = devs[d];
            p.r0 = lo;
            if (d == D - 1) p.r1 = n;
            else {
                const uint32_t target = (uint32_t)(nb * (uint64_t)(d + 1) / D);
                uint64_t hi = (uint64_t)(std::upper_bound(r->read_blk, r->read_blk + n, target) - r->read_blk);
                if (hi > 0) --hi;
                p.r1 = std::min(std::max(hi, lo), n);
            }
            lo = p.r1;
            plans.push_back(p);
        }
    }
    const int D = (int)plans.size();
    const bool multi = D > 1;

    // ---- tables first, then size the batches against what is left --------------------------------------------------
    rc = on_devices(plans, [&](DevPlan& p) -> int {
        CTX_CUDA(cudaSetDevice(p.c->device));
        int rc2;
        if (need_table && (rc2 = p.c->table.reserve(sizeof(uint32_t) * (size_t)kTableEntries))) return rc2;
        const uint64_t b0 = r->read_blk[p.r0], b1 = r->read_blk[p.r1];
        const uint64_t t0 = (uint64_t)(std::lower_bound(r->tile_read, r->tile_read + r->n_tiles, (uint32_t)p.r0) - r->tile_read);
        const uint64_t t1 = (uint64_t)(std::lower_bound(r->tile_read, r->tile_read + r->n_tiles, (uint32_t)p.r1) - r->tile_read);
        const long long cap_bases = atoll(getenv("LRB_BATCH_BASES") ? getenv("LRB_BATCH_BASES") : "0");   // tests: force small batches
        if (cap_bases <= 0) {
            // steady state (a context profiling read sets of one size again and again): the buffers of the previous call hold
            // this device's whole share -> one batch, and no cudaMemGetInfo (it costs up to ~10 ms beside a busy allocator)
            lrb_reads shape;
            shape.n_reads = p.r1 - p.r0; shape.n_blocks = b1 - b0; shape.n_tiles = t1 - t0; shape.n_exc = r->n_exc;
            t_reserve_dry = true;
            const int fits = reserve_batch(p.c, &shape, J, J.do_count);
            t_reserve_dry = false;
            if (fits == LRB_OK) { p.batches.push_back({p.r0, p.r1}); return LRB_OK; }
        }
        size_t free_b = 0, total_b = 0;
        CTX_CUDA(cudaMemGetInfo(&free_b, &total_b));
        uint64_t avail = free_b;
        for (DevBuf* b : {&p.c->codes, &p.c->valid, &p.c->read_len, &p.c->read_blk, &p.c->tile_read, &p.c->tile_blk, &p.c->comp, &p.c->hist,
                          &p.c->sums, &p.c->part_keys, &p.c->part_steps, &p.c->part_sub, &p.c->blk_read, &p.c->exc_blk, &p.c->exc_valid})
            avail += b->cap;   // cached buffers of earlier calls are re-used or released by reserve()
        if (multi) avail = avail > (2ull << 30) / 4 ? avail - (2ull << 30) / 4 : 0;   // exchange staging
        const uint64_t budget = (uint64_t)((double)avail * 0.92);
        const uint64_t need = batch_bytes(J, b1 - b0, p.r1 - p.r0, t1 - t0);
        uint64_t nbat = std::max<uint64_t>(1, (need + budget - 1) / std::max<uint64_t>(budget, 1));
        if (cap_bases > 0) nbat = std::max<uint64_t>(nbat, ((b1 - b0) * 32 + (uint64_t)cap_bases - 1) / (uint64_t)cap_bases);
        nbat = std::min<uint64_t>(nbat, std::max<uint64_t>(1, p.r1 - p.r0));
        uint64_t lo = p.r0;
        for (uint64_t i = 0; i < nbat; ++i) {
            uint64_t hi = p.r1;
            if (i + 1 < nbat) {
                const uint32_t target = (uint32_t)(b0 + (b1 - b0) * (i + 1) / nbat);
                hi = (uint64_t)(std::upper_bound(r->read_blk + p.r0, r->read_blk + p.r1, target) - r->read_blk);
                hi = std::min(std::max(hi, lo + 1), p.r1);
            }
            if (hi > lo || nbat == 1) p.batches.push_back({lo, hi});
            lo = hi;
        }
        if (p.batches.empty()) p.batches.push_back({p.r0, p.r1});
        return LRB_OK;
    });
    if (rc) return rc;
    lrb_run_info& info = c->info;
    memset(&info, 0, sizeof info);
    info.n_devices = D;
    for (auto& p : plans) {
        info.n_batches += (int)p.batches.size();
        for (auto& b : p.batches) info.batch_bases_max = std::max<uint64_t>(info.batch_bases_max, ((uint64_t)r->read_blk[b.r1] - r->read_blk[b.r0]) * 32);
    }
    info.table_path = !J.use_part ? 0 : 1;
    const bool streamed = info.n_batches > D;
    if (streamed || env_int("LRB_VERBOSE", 0) > 0)
        fprintf(stderr, "[lrb] profile: %llu reads / %llu bases on %d GPU(s) in %d batch(es)%s; table passes: %s\n", (unsigned long long)n,
                (unsigned long long)r->total_bases, D, info.n_batches,
                streamed ? " (working set larger than device memory: reads are shipped and partitioned once per pass)" : "",
                J.use_part ? "key-partitioned, L2-resident" : "direct (LRB_TABLE_PATH=direct)");

    auto since0 = [&]() { return (float)std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count(); };
    info.host_plan_ms = since0();

    // ---- pass 1 -----------------------------------------------------------------------------------------------------
    // Adding to the table: device 0 counts into its complete table, every other device into a private table from zero, so
    // that after the exchange  sum over devices of the canonical halves = previous table + this read set;  the mirror then
    // rebuilds the other half on device 0 as for any count.
    c->table_ready = (J.use_loaded || (!cov.reads_full() && !J.do_count)) ? c->table_ready : false;   // a search of sample slots leaves it
    if (J.use_loaded && multi) {   // the loaded table lives on device 0: hand it to the others
        CTX_CUDA(cudaSetDevice(c->device));
        CTX_CUDA(cudaEventRecord(c->counted, c->stream));
        for (int d = 1; d < D; ++d) {
            lrb_ctx* p = plans[d].c;
            CTX_CUDA(cudaSetDevice(p->device));
            CTX_CUDA(cudaStreamWaitEvent(p->stream, c->counted, 0));
            CTX_CUDA(cudaMemcpyPeerAsync(p->table.p, p->device, c->table.p, c->device, sizeof(uint32_t) * (size_t)kTableEntries, p->stream));
        }
    }
    rc = on_devices(plans, [&](DevPlan& p) -> int {
        lrb_ctx* x = p.c;
        CTX_CUDA(cudaSetDevice(x->device));
        const bool single = p.batches.size() == 1;
        int rc2 = LRB_OK;
        for (size_t i = 0; i < p.batches.size() && !rc2; ++i) {
            const Batch& b = p.batches[i];
            lrb_reads* s = nullptr;
            bool owned = false;
            if (b.r0 == 0 && b.r1 == n) s = const_cast<lrb_reads*>(r);
            else { if ((rc2 = lrb_reads_slice(r, b.r0, b.r1, &s))) break; owned = true; }
            rc2 = stage_front(x, s, J, b.r0, /*with_rids=*/single && J.do_search, /*defer_comp=*/single && !J.comp_pinned, /*timed=*/x == c && i == 0,
                              /*first_batch=*/i == 0, /*only_batch=*/single, /*add_into_table=*/J.add_to_table && x == c);
            if (single && !rc2) { p.kept = s; p.kept_owned = owned; break; }
            if (!rc2) rc2 = sync_ctx(x);   // the buffers are re-used by the next batch
            if (owned) lrb_reads_free(s);
        }
        return rc2;
    });
    auto cleanup = [&]() {
        for (auto& p : plans) { if (p.kept_owned) lrb_reads_free(p.kept); p.kept = nullptr; p.kept_owned = false; }
    };
    if (rc) { cleanup(); for (auto& p : plans) sync_ctx(p.c); cudaGetLastError(); return rc; }
    if (c->part.sub && J.use_part) info.table_path = 2;

    // ---- exchange ---------------------------------------------------------------------------------------------------
    XchgSchedule sched;
    const int n_buckets = (int)(kTableEntries >> J.bucket_shift);
    if (multi && J.do_count) {
        if ((rc = enqueue_exchange(plans, n_buckets, J.bucket_shift, c->peer_access && env_int("LRB_XCHG_COPY3D", 0) == 0, &sched))) {
            cleanup(); for (auto& p : plans) sync_ctx(p.c); cudaGetLastError(); return rc;
        }
    }

    // ---- pass 2 -----------------------------------------------------------------------------------------------------
    rc = on_devices(plans, [&](DevPlan& p) -> int {
        lrb_ctx* x = p.c;
        CTX_CUDA(cudaSetDevice(x->device));
        cudaStream_t st = x->stream;
        const bool single = p.batches.size() == 1;
        const bool exchanged = multi && J.do_count;
        int rc2 = LRB_OK;
        auto wait_rounds = [&]() -> int {
            for (int kx = 0; exchanged && kx < sched.n_rounds; ++kx) CTX_CUDA(cudaStreamWaitEvent(st, x->round_ev[kx], 0));
            return LRB_OK;
        };
        if (single) {
            const uint64_t nr = p.kept->n_reads;
            // The mirror writes only the half of the table the list-driven search never reads, yet it runs after the search:
            // beside it (measured, profiles/r02_exp1_variants.jsonl) the 4 GiB it streams through L2 evict the search's
            // resident table slice — the search goes from 20.5 to 26.2 ms to hide a 1.26 ms pass.
            const bool mirror_here = J.do_count && (x == c || !J.use_part);
            if (J.do_search && nr) {
                CTX_CUDA(cudaMemsetAsync(x->hist.p, 0, sizeof(uint32_t) * nr * (size_t)J.cov.W, st));
                CTX_CUDA(cudaMemsetAsync(x->sums.p, 0, sizeof(uint32_t) * nr, st));
            }
            if (J.do_search && J.use_part && p.kept->n_blocks) {
                if (exchanged) {   // the round's buckets as soon as they have arrived
                    for (int kx = 0; kx < sched.n_rounds && !rc2; ++kx) {
                        CTX_CUDA(cudaStreamWaitEvent(st, x->round_ev[kx], 0));
                        rc2 = search_lists(x, J, nr, sched.round_bucket_lo(kx, D), kx + 1 == sched.n_rounds ? n_buckets : sched.round_bucket_lo(kx + 1, D));
                    }
                } else {
                    rc2 = search_lists(x, J, nr, 0, n_buckets);
                }
            } else if ((rc2 = wait_rounds())) {
                return rc2;
            }
            if (rc2) return rc2;
            if (x == c) CTX_CUDA(cudaEventRecord(c->ev[3], st));  // table passes done
            // the full table (both strands) is needed on device 0 (lrb_ctx_table_save, table_host) and by the direct search
            if (mirror_here && (rc2 = lrb_dev_mirror((uint32_t*)x->table.p, st))) return rc2;
            if (x == c) CTX_CUDA(cudaEventRecord(c->ev[4], st));
            if (!J.use_part && J.do_search && nr &&
                (rc2 = lrb_dev_search(&x->dview, (const uint32_t*)x->table.p, J.cov.b[0].bin_size, J.cov.W, (uint32_t*)x->hist.p, (uint32_t*)x->sums.p, 0,
                                      p.kept->n_tiles, 0, kTableEntries, st)))
                return rc2;
            if (x == c) CTX_CUDA(cudaEventRecord(c->ev[5], st));
            if ((rc2 = rows_home(x, J, nr, p.batches[0].r0))) return rc2;
        } else {
            if ((rc2 = wait_rounds())) return rc2;
            if (x == c) CTX_CUDA(cudaEventRecord(c->ev[3], st));
            if (J.do_count && (x == c || !J.use_part) && (rc2 = lrb_dev_mirror((uint32_t*)x->table.p, st))) return rc2;
            if (x == c) { CTX_CUDA(cudaEventRecord(c->ev[4], st)); CTX_CUDA(cudaEventRecord(c->ev[5], st)); }
            Job S = J;          // pass 2 of a streamed run: ship the batch again, lists with read ids, search
            S.do_comp = false;
            S.do_count = false;
            for (size_t i = 0; i < p.batches.size() && J.do_search && !rc2; ++i) {
                const Batch& b = p.batches[i];
                lrb_reads* s = nullptr;
                if ((rc2 = lrb_reads_slice(r, b.r0, b.r1, &s))) break;
                const uint64_t nr = s->n_reads;
                rc2 = stage_front(x, s, S, b.r0, /*with_rids=*/true, false, false);
                if (!rc2 && nr) {
                    cudaMemsetAsync(x->hist.p, 0, sizeof(uint32_t) * nr * (size_t)J.cov.W, st);
                    cudaMemsetAsync(x->sums.p, 0, sizeof(uint32_t) * nr, st);
                    if (J.use_part && s->n_blocks) rc2 = search_lists(x, J, nr, 0, n_buckets);
                    else if (!J.use_part)
                        rc2 = lrb_dev_search(&x->dview, (const uint32_t*)x->table.p, J.cov.b[0].bin_size, J.cov.W, (uint32_t*)x->hist.p, (uint32_t*)x->sums.p, 0,
                                             s->n_tiles, 0, kTableEntries, st);
                }
                if (!rc2) rc2 = rows_home(x, J, nr, b.r0) || sync_ctx(x);
                lrb_reads_free(s);
            }
            if (rc2) return rc2;
        }
        if (x == c && table_host)
            CTX_CUDA(cudaMemcpyAsync(table_host, c->table.p, sizeof(uint32_t) * (size_t)kTableEntries, cudaMemcpyDeviceToHost, st));
        if (x == c) CTX_CUDA(cudaEventRecord(c->ev[6], st));
        if (x == c) info.host_enqueue_ms = since0();   // everything is enqueued (single batch); what follows is waiting for the device
        return sync_ctx(x);
    });
    cleanup();
    if (rc) { for (auto& p : plans) sync_ctx(p.c); cudaGetLastError(); return rc; }
    if (J.do_count) c->table_ready = true;   // only now: every pass has run to completion without an error
    // [0] h2d (copy stream) [1] composition+partition (until the last chunk is processed) [2] table passes
    // [3] mirror [4] direct search [5] result D2H tail [6] whole call  — device 0, first batch
    CTX_CUDA(cudaSetDevice(c->device));
    if (plans[0].batches.size() == 1) {
        cudaEventElapsedTime(&c->ms[0], c->ev[0], c->ev[1]);
        cudaEventElapsedTime(&c->ms[1], c->ev[0], c->ev[2]);
        for (int i = 2; i < 6; ++i) cudaEventElapsedTime(&c->ms[i], c->ev[i], c->ev[i + 1]);
    } else {
        for (int i = 0; i < 6; ++i) c->ms[i] = 0.f;
    }
    cudaEventElapsedTime(&c->ms[6], c->ev[0], c->ev[6]);
    if (multi && J.do_count) cudaEventElapsedTime(&info.exchange_ms, c->xev[0], c->xev[1]);
    cudaGetLastError();
    info.lists_reused = !streamed && J.use_part && J.do_count && J.do_search;
    info.wall_ms = (float)std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
    return LRB_OK;
}

// The public profile calls: the coverage layout is checked before the context, so that no device is needed to refuse it,
// and a failed LRB_PROFILE_ADD_TO_TABLE call leaves the context without a table (it may hold part of the read set).
static int profile_call(const char* who, lrb_ctx* c, const lrb_reads* r, int k, CovLayout cov, uint32_t* comp_counts, uint32_t* cov_hist,
                        uint32_t* cov_sums, uint32_t* table_host, int flags) {
    if (!r) return lrb_set_error(LRB_EINVAL, "%s: null argument", who);
    int rc = lrb_check_cov_layout(who, &cov);
    if (!rc && !c) return lrb_set_error(LRB_EINVAL, "%s: null context", who);
    if (!rc) rc = profile_host(who, c, r, k, cov, comp_counts, cov_hist, cov_sums, table_host, flags);
    if (rc && c && (flags & LRB_PROFILE_ADD_TO_TABLE)) c->table_ready = false;
    return rc;
}

extern "C" int lrb_profile_host_settings(lrb_ctx* c, const lrb_reads* r, int k, int n, const long* bin_sizes, const int* bins,
                                         uint32_t* comp_counts, uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags) {
    // without coverage rows the settings are not used, and not checked
    const CovLayout cov = cov_hist || cov_sums ? lrb_cov_settings(n, bin_sizes, bins) : CovLayout{};
    return profile_call("lrb_profile_host", c, r, k, cov, comp_counts, cov_hist, cov_sums, table_host, flags);
}

extern "C" int lrb_profile_host_samples(lrb_ctx* c, const lrb_reads* r, int k, int n, const int* slots, const long* bin_sizes,
                                        const int* bins, uint32_t* comp_counts, uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host,
                                        int flags) {
    if (!slots) return lrb_set_error(LRB_EINVAL, "lrb_profile_host_samples: null argument");
    return profile_call("lrb_profile_host_samples", c, r, k, lrb_cov_settings(n, bin_sizes, bins, slots), comp_counts, cov_hist, cov_sums,
                        table_host, flags);
}

extern "C" int lrb_profile_host_edges(lrb_ctx* c, const lrb_reads* r, int k, const uint32_t* edges, int n_edges, uint32_t* comp_counts,
                                      uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags) {
    return profile_call("lrb_profile_host_edges", c, r, k, lrb_cov_edges(edges, n_edges), comp_counts, cov_hist, cov_sums, table_host, flags);
}

extern "C" int lrb_profile_host_layout(lrb_ctx* c, const lrb_reads* r, int k, const lrb_cov_block* blocks, int n, uint32_t* comp_counts,
                                       uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags) {
    return profile_call("lrb_profile_host_layout", c, r, k, lrb_cov_layout(blocks, n), comp_counts, cov_hist, cov_sums, table_host, flags);
}

extern "C" int lrb_profile_host(lrb_ctx* c, const lrb_reads* r, int k, long bin_size, int bins, uint32_t* comp_counts,
                                uint32_t* cov_hist, uint32_t* cov_sums, uint32_t* table_host, int flags) {
    return lrb_profile_host_settings(c, r, k, 1, &bin_size, &bins, comp_counts, cov_hist, cov_sums, table_host, flags);
}

extern "C" int lrb_ctx_last_timings(const lrb_ctx* c, float* ms7) {
    if (!c || !ms7) return lrb_set_error(LRB_EINVAL, "lrb_ctx_last_timings: null argument");
    memcpy(ms7, c->ms, sizeof c->ms);
    return LRB_OK;
}

extern "C" int lrb_ctx_last_info(const lrb_ctx* c, lrb_run_info* info) {
    if (!c || !info) return lrb_set_error(LRB_EINVAL, "lrb_ctx_last_info: null argument");
    *info = c->info;
    return LRB_OK;
}

// table <-> file through a pair of pinned staging buffers (the 4 GiB never sits in host RAM as a whole).  The file side
// of every staged chunk is split over a few threads (pwrite / pread at disjoint offsets): one thread moves ~2-3 GB/s
// through the page cache, which made the table file the whole cost of the three-call drop-in sequence.
namespace {

constexpr size_t kTableChunk = 64u << 20;

int io_threads() { return std::max(1, std::min(8, (int)std::thread::hardware_concurrency())); }

// fn(fd, buf + a, len, file_off + a) over disjoint parts of [0, n) in parallel; returns false if any part failed
template <class F>
bool split_io(char* buf, size_t n, off_t file_off, F fn) {
    const int T = io_threads();
    const size_t part = ((n + T - 1) / T + 4095) & ~(size_t)4095;
    std::vector<char> ok((size_t)T, 1);
    std::vector<std::thread> pool;
    for (int t = 0; t < T; ++t) {
        const size_t a = (size_t)t * part;
        if (a >= n) break;
        const size_t len = std::min(part, n - a);
        pool.emplace_back([&, t, a, len] { ok[t] = fn(buf + a, len, file_off + (off_t)a) ? 1 : 0; });
    }
    for (auto& th : pool) th.join();
    for (char c : ok) if (!c) return false;
    return true;
}

}  // namespace

extern "C" int lrb_ctx_table_save(lrb_ctx* c, const char* path) {
    if (!c || !path) return lrb_set_error(LRB_EINVAL, "lrb_ctx_table_save: null argument");
    if (!c->table_ready) return lrb_set_error(LRB_EINVAL, "lrb_ctx_table_save: no table in this context");
    CTX_CUDA(cudaSetDevice(c->device));
    const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return lrb_set_error(LRB_EIO, "cannot open %s for writing", path);
    const uint64_t size = kTableEntries;
    if (pwrite(fd, &size, sizeof size, 0) != (ssize_t)sizeof size) { close(fd); return lrb_set_error(LRB_EIO, "short write to %s", path); }
    bool pin = false, pin2 = false;
    char* stage[2] = {(char*)lrb_host_alloc(kTableChunk, &pin), (char*)lrb_host_alloc(kTableChunk, &pin2)};
    int rc = LRB_OK;
    const size_t total = (size_t)size * 4;
    const char* dsrc = (const char*)c->table.p;
    size_t off = 0;
    int cur = 0;
    auto put = [fd](char* p, size_t len, off_t at) {
        while (len) {
            const ssize_t w = pwrite(fd, p, len, at);
            if (w <= 0) return false;
            p += w; len -= (size_t)w; at += w;
        }
        return true;
    };
    if (!stage[0] || !stage[1]) rc = lrb_set_error(LRB_ENOMEM, "out of memory (staging)");
    if (!rc && cudaMemcpyAsync(stage[0], dsrc, std::min(kTableChunk, total), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) rc = lrb_set_error(LRB_ECUDA, "D2H failed");
    while (!rc && off < total) {
        const size_t nbytes = std::min(kTableChunk, total - off);
        if (cudaStreamSynchronize(c->stream) != cudaSuccess) { rc = lrb_set_error(LRB_ECUDA, "D2H failed: %s", cudaGetErrorString(cudaGetLastError())); break; }
        const size_t next = off + nbytes;
        if (next < total && cudaMemcpyAsync(stage[cur ^ 1], dsrc + next, std::min(kTableChunk, total - next), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) { rc = lrb_set_error(LRB_ECUDA, "D2H failed"); break; }
        if (!split_io(stage[cur], nbytes, (off_t)(sizeof size + off), put)) { rc = lrb_set_error(LRB_EIO, "short write to %s", path); break; }
        off = next;
        cur ^= 1;
    }
    cudaStreamSynchronize(c->stream);
    lrb_host_free(stage[0], pin);
    lrb_host_free(stage[1], pin2);
    if (close(fd) != 0 && !rc) rc = lrb_set_error(LRB_EIO, "close failed for %s", path);
    return rc;
}

extern "C" int lrb_ctx_table_load(lrb_ctx* c, const char* path) {
    if (!c || !path) return lrb_set_error(LRB_EINVAL, "lrb_ctx_table_load: null argument");
    CTX_CUDA(cudaSetDevice(c->device));
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return lrb_set_error(LRB_EIO, "cannot open table file %s", path);
    uint64_t size = 0;
    if (pread(fd, &size, sizeof size, 0) != (ssize_t)sizeof size || size != kTableEntries) {
        close(fd);
        return lrb_set_error(LRB_EFORMAT, "%s is not a 4^15-entry 15mers-counts file", path);
    }
    int rc = c->table.reserve(sizeof(uint32_t) * (size_t)kTableEntries);
    if (rc) { close(fd); return rc; }
    c->table_ready = false;
    bool pin = false, pin2 = false;
    char* stage[2] = {(char*)lrb_host_alloc(kTableChunk, &pin), (char*)lrb_host_alloc(kTableChunk, &pin2)};
    if (!stage[0] || !stage[1]) rc = lrb_set_error(LRB_ENOMEM, "out of memory (staging)");
    const size_t total = (size_t)size * 4;
    size_t off = 0;
    int cur = 0;
    cudaEvent_t done[2];
    cudaEventCreate(&done[0]);
    cudaEventCreate(&done[1]);
    bool used[2] = {false, false};
    auto get = [fd](char* p, size_t len, off_t at) {
        while (len) {
            const ssize_t r = pread(fd, p, len, at);
            if (r <= 0) return false;
            p += r; len -= (size_t)r; at += r;
        }
        return true;
    };
    while (!rc && off < total) {
        const size_t nbytes = std::min(kTableChunk, total - off);
        if (used[cur]) cudaEventSynchronize(done[cur]);
        if (!split_io(stage[cur], nbytes, (off_t)(sizeof size + off), get)) { rc = lrb_set_error(LRB_EFORMAT, "%s is truncated", path); break; }
        if (cudaMemcpyAsync((char*)c->table.p + off, stage[cur], nbytes, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) { rc = lrb_set_error(LRB_ECUDA, "H2D failed"); break; }
        cudaEventRecord(done[cur], c->stream);
        used[cur] = true;
        off += nbytes;
        cur ^= 1;
    }
    if (cudaStreamSynchronize(c->stream) != cudaSuccess && !rc) rc = lrb_set_error(LRB_ECUDA, "H2D failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaEventDestroy(done[0]);
    cudaEventDestroy(done[1]);
    lrb_host_free(stage[0], pin);
    lrb_host_free(stage[1], pin2);
    close(fd);
    if (!rc) c->table_ready = true;
    return rc;
}

// ---- sample slots: compact tables (canonical halves) on every device of the context ----------------------------------
namespace {

constexpr uint64_t kCanonRows = (uint64_t)kTableEntries >> 16;   // 2^14 rows of 2^16 entries; the first 2^15 of each are canonical
constexpr size_t kCanonRowBytes = 4u << 15;                       // 128 KiB of a row read, at a stride of 256 KiB
constexpr size_t kCompactBytes = sizeof(uint32_t) * (size_t)LRB_COMPACT_ENTRIES;

// open a 15mers-counts file after checking its header and its size (reading only canonical rows would not notice a file
// cut short by less than one row)
int open_table_file(const char* path, int* fd_out) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return lrb_set_error(LRB_EIO, "cannot open table file %s", path);
    uint64_t size = 0;
    struct stat st;
    if (pread(fd, &size, sizeof size, 0) != (ssize_t)sizeof size || size != kTableEntries || fstat(fd, &st) != 0 ||
        (uint64_t)st.st_size != sizeof size + 4ull * kTableEntries) {
        close(fd);
        return lrb_set_error(LRB_EFORMAT, "%s is not a 4^15-entry 15mers-counts file (header or size)", path);
    }
    *fd_out = fd;
    return LRB_OK;
}

// canonical rows [row_lo, row_hi) of the open table file side by side into dst (split over threads like the table load)
bool read_canonical_rows(int fd, uint64_t row_lo, uint64_t row_hi, char* dst) {
    return split_io(dst, (size_t)(row_hi - row_lo) * kCanonRowBytes, 0, [&](char* p, size_t len, off_t at) {
        while (len) {   // `at` is the byte offset in dst; its row and the place inside the row give the file offset
            const uint64_t row = row_lo + (uint64_t)at / kCanonRowBytes, in_row = (uint64_t)at % kCanonRowBytes;
            size_t want = std::min<size_t>(len, kCanonRowBytes - in_row);
            const ssize_t r = pread(fd, p, want, (off_t)(sizeof(uint64_t) + row * 2 * kCanonRowBytes + in_row));
            if (r <= 0) return false;
            p += r; len -= (size_t)r; at += r;
        }
        return true;
    });
}

int check_slot(const lrb_ctx* c, int slot, const char* who) {
    if (!c) return lrb_set_error(LRB_EINVAL, "%s: null context", who);
    if (slot < 0 || slot >= LRB_MAX_SAMPLE_TABLES) return lrb_set_error(LRB_EINVAL, "%s: slot must be in [0, %d) (got %d)", who, LRB_MAX_SAMPLE_TABLES, slot);
    return LRB_OK;
}

std::vector<lrb_ctx*> ctx_devices(lrb_ctx* c) {
    std::vector<lrb_ctx*> d{c};
    for (lrb_ctx* p : c->peers) d.push_back(p);
    return d;
}

// the slot's buffer on every device, marked empty until it is filled
int reserve_slot(lrb_ctx* c, int slot) {
    for (lrb_ctx* x : ctx_devices(c)) {
        x->sample_ready[slot] = false;
        CTX_CUDA(cudaSetDevice(x->device));
        int rc;
        if ((rc = x->sample[slot].reserve(kCompactBytes))) return rc;
    }
    CTX_CUDA(cudaSetDevice(c->device));
    return LRB_OK;
}

// device 0's slot to the other devices (after the work already on device 0's stream), then wait; all slots ready
int broadcast_slot(lrb_ctx* c, int slot) {
    CTX_CUDA(cudaSetDevice(c->device));
    for (lrb_ctx* p : c->peers)
        CTX_CUDA(cudaMemcpyPeerAsync(p->sample[slot].p, p->device, c->sample[slot].p, c->device, kCompactBytes, c->stream));
    CTX_CUDA(cudaStreamSynchronize(c->stream));
    for (lrb_ctx* x : ctx_devices(c)) x->sample_ready[slot] = true;
    return LRB_OK;
}

}  // namespace

extern "C" int lrb_table_read_canonical(const char* path, uint32_t row_lo, uint32_t row_hi, uint32_t* compact) {
    if (!path || !compact) return lrb_set_error(LRB_EINVAL, "lrb_table_read_canonical: null argument");
    if (row_lo > row_hi || row_hi > kCanonRows)
        return lrb_set_error(LRB_EINVAL, "lrb_table_read_canonical: rows [%u, %u) outside [0, %llu)", row_lo, row_hi, (unsigned long long)kCanonRows);
    int fd = -1, rc;
    if ((rc = open_table_file(path, &fd))) return rc;
    const bool ok = read_canonical_rows(fd, row_lo, row_hi, (char*)compact);
    close(fd);
    return ok ? LRB_OK : lrb_set_error(LRB_EFORMAT, "%s is truncated", path);
}

extern "C" int lrb_ctx_sample_table_load(lrb_ctx* c, int slot, const char* path) {
    int rc;
    if ((rc = check_slot(c, slot, "lrb_ctx_sample_table_load"))) return rc;
    if (!path) return lrb_set_error(LRB_EINVAL, "lrb_ctx_sample_table_load: null path");
    int fd = -1;
    if ((rc = open_table_file(path, &fd))) return rc;
    if ((rc = reserve_slot(c, slot))) { close(fd); return rc; }
    // the rows of a 64 MiB staging buffer are read while the other one is on its way to device 0
    bool pin = false, pin2 = false;
    char* stage[2] = {(char*)lrb_host_alloc(kTableChunk, &pin), (char*)lrb_host_alloc(kTableChunk, &pin2)};
    if (!stage[0] || !stage[1]) rc = lrb_set_error(LRB_ENOMEM, "out of memory (staging)");
    const uint64_t rows_per_chunk = kTableChunk / kCanonRowBytes;
    cudaEvent_t done[2];
    cudaEventCreate(&done[0]);
    cudaEventCreate(&done[1]);
    bool used[2] = {false, false};
    int cur = 0;
    for (uint64_t row = 0; !rc && row < kCanonRows; row += rows_per_chunk, cur ^= 1) {
        const uint64_t row_hi = std::min(kCanonRows, row + rows_per_chunk);
        if (used[cur]) cudaEventSynchronize(done[cur]);
        if (!read_canonical_rows(fd, row, row_hi, stage[cur])) { rc = lrb_set_error(LRB_EFORMAT, "%s is truncated", path); break; }
        if (cudaMemcpyAsync((char*)c->sample[slot].p + row * kCanonRowBytes, stage[cur], (row_hi - row) * kCanonRowBytes, cudaMemcpyHostToDevice,
                            c->stream) != cudaSuccess) { rc = lrb_set_error(LRB_ECUDA, "H2D failed"); break; }
        cudaEventRecord(done[cur], c->stream);
        used[cur] = true;
    }
    if (cudaStreamSynchronize(c->stream) != cudaSuccess && !rc) rc = lrb_set_error(LRB_ECUDA, "H2D failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaEventDestroy(done[0]);
    cudaEventDestroy(done[1]);
    lrb_host_free(stage[0], pin);
    lrb_host_free(stage[1], pin2);
    close(fd);
    return rc ? rc : broadcast_slot(c, slot);
}

extern "C" int lrb_ctx_sample_table_keep(lrb_ctx* c, int slot) {
    int rc;
    if ((rc = check_slot(c, slot, "lrb_ctx_sample_table_keep"))) return rc;
    if (!c->table_ready) return lrb_set_error(LRB_EINVAL, "lrb_ctx_sample_table_keep: no table in this context");
    if ((rc = reserve_slot(c, slot))) return rc;
    if ((rc = lrb_dev_table_compact((const uint32_t*)c->table.p, (uint32_t*)c->sample[slot].p, c->stream))) return rc;
    return broadcast_slot(c, slot);
}

extern "C" int lrb_ctx_sample_table_free(lrb_ctx* c, int slot) {
    int rc;
    if ((rc = check_slot(c, slot, "lrb_ctx_sample_table_free"))) return rc;
    for (lrb_ctx* x : ctx_devices(c)) {
        CTX_CUDA(cudaSetDevice(x->device));
        x->sample_ready[slot] = false;
        x->sample[slot].release();
    }
    CTX_CUDA(cudaSetDevice(c->device));
    return LRB_OK;
}

extern "C" int lrb_ctx_table_spectrum(lrb_ctx* c, uint32_t max_count, uint64_t* spectrum_host) {
    if (!c || !spectrum_host) return lrb_set_error(LRB_EINVAL, "lrb_ctx_table_spectrum: null argument");
    if (max_count < 2 || max_count > LRB_SPECTRUM_MAX_COUNT)
        return lrb_set_error(LRB_EINVAL, "lrb_ctx_table_spectrum: max_count must be in [2, %u] (got %u)", LRB_SPECTRUM_MAX_COUNT, max_count);
    if (!c->table_ready) return lrb_set_error(LRB_EINVAL, "lrb_ctx_table_spectrum: no table in this context");
    CTX_CUDA(cudaSetDevice(c->device));
    const size_t bytes = sizeof(uint64_t) * ((size_t)max_count + 3);
    DevBuf spec;
    int rc = spec.reserve(bytes);
    if (!rc && cudaMemsetAsync(spec.p, 0, bytes, c->stream) != cudaSuccess) rc = lrb_set_error(LRB_ECUDA, "cudaMemsetAsync failed");
    if (!rc) rc = lrb_dev_table_spectrum((const uint32_t*)c->table.p, 0, (uint32_t)kTableEntries, max_count, (uint64_t*)spec.p, c->stream);
    if (!rc && cudaMemcpyAsync(spectrum_host, spec.p, bytes, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) rc = lrb_set_error(LRB_ECUDA, "D2H failed");
    if (cudaStreamSynchronize(c->stream) != cudaSuccess && !rc) rc = lrb_set_error(LRB_ECUDA, "spectrum failed: %s", cudaGetErrorString(cudaGetLastError()));
    spec.release();
    return rc;
}

extern "C" int lrb_ctx_sample_table_spectrum(lrb_ctx* c, int slot, uint32_t max_count, uint64_t* spectrum_host) {
    static const char* who = "lrb_ctx_sample_table_spectrum";
    int rc;
    if ((rc = check_slot(c, slot, who))) return rc;
    if (!spectrum_host) return lrb_set_error(LRB_EINVAL, "%s: null argument", who);
    if (max_count < 2 || max_count > LRB_SPECTRUM_MAX_COUNT)
        return lrb_set_error(LRB_EINVAL, "%s: max_count must be in [2, %u] (got %u)", who, LRB_SPECTRUM_MAX_COUNT, max_count);
    if (!c->sample_ready[slot]) return lrb_set_error(LRB_EINVAL, "%s: sample slot %d is empty", who, slot);
    CTX_CUDA(cudaSetDevice(c->device));
    const size_t bytes = sizeof(uint64_t) * ((size_t)max_count + 3);
    DevBuf spec;
    rc = spec.reserve(bytes);
    if (!rc && cudaMemsetAsync(spec.p, 0, bytes, c->stream) != cudaSuccess) rc = lrb_set_error(LRB_ECUDA, "cudaMemsetAsync failed");
    if (!rc) rc = lrb_dev_compact_spectrum((const uint32_t*)c->sample[slot].p, max_count, (uint64_t*)spec.p, c->stream);
    if (!rc && cudaMemcpyAsync(spectrum_host, spec.p, bytes, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) rc = lrb_set_error(LRB_ECUDA, "D2H failed");
    if (cudaStreamSynchronize(c->stream) != cudaSuccess && !rc) rc = lrb_set_error(LRB_ECUDA, "spectrum failed: %s", cudaGetErrorString(cudaGetLastError()));
    spec.release();
    return rc;
}

// ---- synthetic reads ---------------------------------------------------------------------------
namespace {

struct DevEmit {
    uint32_t* codes;  // first code word of the read
    uint32_t* valid;
    uint32_t w0 = 0, w1 = 0, v = 0;
    __device__ void operator()(uint32_t pos, char c) {
        const uint32_t j = pos & 31u;
        const uint32_t code = ((unsigned char)c >> 1) & 3u;
        if (j < 16) w0 |= code << (30 - 2 * j); else w1 |= code << (62 - 2 * j);
        if (c == 'A' || c == 'C' || c == 'G' || c == 'T') v |= 1u << j;
        if (j == 31u) {
            const uint32_t b = pos >> 5;
            codes[2 * (size_t)b] = w0; codes[2 * (size_t)b + 1] = w1; valid[b] = v;
            w0 = w1 = v = 0;
        }
    }
};

__global__ void __launch_bounds__(128)
k_synth(lrb_reads_view R, lrb_synth_params p, const uint32_t* __restrict__ glen, const uint32_t* __restrict__ meta,
        uint32_t* __restrict__ codes, uint32_t* __restrict__ valid) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R.n_reads) return;
    const uint32_t len = R.read_len[r], b0 = R.read_blk[r];
    DevEmit e{codes + 2 * (size_t)b0, valid + b0};
    synth_read(p, glen, r, meta[4 * r] % p.n_genomes, meta[4 * r + 1], meta[4 * r + 2], len, [&](uint32_t pos, char c) { e(pos, c); });
    const uint32_t b = len >> 5;  // trailing (partial or empty) block
    e.codes[2 * (size_t)b] = e.w0; e.codes[2 * (size_t)b + 1] = e.w1; e.valid[b] = e.v;
}

}  // namespace

extern "C" int lrb_dev_synth(const lrb_reads_view* dev, const lrb_synth_params* p, const uint32_t* glen,
                             const uint32_t* meta, void* stream) {
    if (!dev || !p || !glen || !meta || p->n_genomes == 0) return lrb_set_error(LRB_EINVAL, "lrb_dev_synth: bad argument");
    if (dev->n_reads == 0) return LRB_OK;
    const unsigned grid = (unsigned)((dev->n_reads + 127) / 128);
    LRB_LAUNCH("k_synth", (cudaStream_t)stream, k_synth<<<grid, 128, 0, (cudaStream_t)stream>>>(*dev, *p, glen, meta, const_cast<uint32_t*>(dev->codes), const_cast<uint32_t*>(dev->valid)));
    CTX_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_synth_host(const lrb_synth_params* p, const uint32_t* glen, const uint32_t* meta,
                              const uint32_t* lengths, uint64_t n_reads, const uint64_t* offsets, char* bases) {
    if (!p || !glen || !meta || !lengths || !offsets || !bases || p->n_genomes == 0) return lrb_set_error(LRB_EINVAL, "lrb_synth_host: bad argument");
    for (uint64_t r = 0; r < n_reads; ++r) {
        char* dst = bases + offsets[r];
        synth_read(*p, glen, r, meta[4 * r] % p->n_genomes, meta[4 * r + 1], meta[4 * r + 2], lengths[r],
                   [&](uint32_t pos, char c) { dst[pos] = c; });
    }
    return LRB_OK;
}

// ---- file level (the three tools + the fused stage) ----------------------------------------------
namespace {

struct CtxGuard {
    lrb_ctx* c = nullptr;
    ~CtxGuard() { lrb_ctx_destroy(c); }
};

int default_device() {
    const char* e = getenv("LRB_DEVICE");
    if (e && *e) return atoi(e);
    const char* lr = getenv("LOCAL_RANK");
    if (lr && *lr) return atoi(lr);
    return 0;
}

// GPUs a file-level call drives: n_gpus > 0 as given, else LRB_GPUS (default 1).  Devices default_device() .. +n-1.
int create_ctx(int n_gpus, lrb_ctx** out) {
    if (n_gpus <= 0) n_gpus = std::max(1, env_int("LRB_GPUS", 1));
    if (n_gpus > kMaxDevices) return lrb_set_error(LRB_EINVAL, "at most %d GPUs (got %d)", kMaxDevices, n_gpus);
    int ids[kMaxDevices];
    for (int i = 0; i < n_gpus; ++i) ids[i] = default_device() + i;
    return lrb_ctx_create_multi(ids, n_gpus, out);
}

int truncate_file(const char* path) {  // the tools create/truncate their output before reading (count-kmers.cpp:210)
    FILE* f = fopen(path, "wb");
    if (!f) return lrb_set_error(LRB_EIO, "cannot open %s for writing", path);
    fclose(f);
    return LRB_OK;
}

int make_dir(const char* path) {
    if (mkdir(path, 0755) == 0 || errno == EEXIST) return LRB_OK;
    return lrb_set_error(LRB_EIO, "cannot create directory %s: %s", path, strerror(errno));
}

// The reads of a file-level call: one read set (lrb_reads_from_file) when the input fits one segment, else the segment
// reader positioned after its first segment.  Host memory then holds one segment's packed stream and result rows, whatever
// the size of the file, and no read set reaches the 2^32-block limit.
struct Input {
    lrb_reads* whole = nullptr;   // the input as one read set, or
    lrb_reader* rd = nullptr;     // its reader, with the current segment in `seg`
    lrb_reads* seg = nullptr;
    ~Input() { lrb_reads_free(whole); lrb_reads_free(seg); lrb_reader_close(rd); }
};

bool is_gzip(const char* path) {
    unsigned char magic[2] = {0, 0};
    const int fd = open(path, O_RDONLY);
    const bool gz = fd >= 0 && pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
    if (fd >= 0) close(fd);
    return gz;
}

// row_bytes: host bytes of result rows per read.  A missing file, or a plain file no larger in bytes than the segment budget,
// is read whole as before; otherwise the reader decides, and a first segment that is the whole stream is used as one read set.
int open_input(const char* path, int threads, uint64_t row_bytes, Input& in) {
    const uint64_t budget = lrb_segment_budget(row_bytes + 16);   // + read_len, read_blk and >= 1 tile per read
    struct stat st;
    if (stat(path, &st) != 0 || (S_ISREG(st.st_mode) && (uint64_t)st.st_size <= budget && !is_gzip(path)))
        return lrb_reads_from_file(path, threads, &in.whole);
    int rc, at_end = 0;
    if ((rc = lrb_reader_open(path, threads, budget, &in.rd)) || (rc = lrb_reader_next(in.rd, &in.seg))) return rc;
    lrb_reader_tell(in.rd, nullptr, nullptr, nullptr, &at_end);
    if (!at_end) return LRB_OK;
    std::swap(in.whole, in.seg);
    return in.whole ? LRB_OK : lrb_reads_from_lengths(nullptr, 0, &in.whole);   // no record at all: an empty read set
}

// f(segment, index of its first read) for every segment from the current one on; rewind: from the first record again
template <class F>
int each_segment(Input& in, bool rewind, F f) {
    int rc;
    if (rewind) {
        lrb_reads_free(in.seg);
        in.seg = nullptr;
        if ((rc = lrb_reader_rewind(in.rd)) || (rc = lrb_reader_next(in.rd, &in.seg))) return rc;
    }
    for (uint64_t row0 = 0; in.seg;) {
        if ((rc = f(in.seg, row0))) return rc;
        row0 += in.seg->n_reads;
        lrb_reads_free(in.seg);
        in.seg = nullptr;
        if ((rc = lrb_reader_next(in.rd, &in.seg))) return rc;
    }
    return LRB_OK;
}

void segments_notice(const Input& in, int passes) {
    uint64_t reads = 0, bases = 0, segs = 0;
    lrb_reader_tell(in.rd, &reads, &bases, &segs, nullptr);
    fprintf(stderr, "[lrb] input: %llu reads / %llu bases in %llu segments (larger than one segment of host memory); %d pass%s over the file\n",
            (unsigned long long)reads, (unsigned long long)bases, (unsigned long long)segs, passes, passes == 1 ? "" : "es");
}

}  // namespace

extern "C" int lrb_count_kmers(const char* reads_path, const char* out_txt, int k, int threads) {
    if (!reads_path || !out_txt) return lrb_set_error(LRB_EINVAL, "lrb_count_kmers: null path");
    const int P = comp_width(k);
    if (!P) return lrb_set_error(LRB_EINVAL, "k must be 3, 4 or 5 (got %d)", k);
    int rc;
    if ((rc = truncate_file(out_txt))) return rc;
    CtxGuard cg;
    if ((rc = create_ctx(0, &cg.c))) return rc;
    Input in;
    if ((rc = open_input(reads_path, threads, 4ull * P, in))) return rc;
    if (in.whole) {
        std::vector<uint32_t> counts((size_t)in.whole->n_reads * P + 1);
        if ((rc = lrb_profile_host(cg.c, in.whole, k, 1, 1, counts.data(), nullptr, nullptr, nullptr, 0))) return rc;
        return lrb_write_composition_txt(out_txt, counts.data(), in.whole->read_len, in.whole->n_reads, k, threads);
    }
    rc = each_segment(in, false, [&](const lrb_reads* s, uint64_t row0) -> int {
        std::vector<uint32_t> counts((size_t)s->n_reads * P + 1);
        const int rc2 = lrb_profile_host(cg.c, s, k, 1, 1, counts.data(), nullptr, nullptr, nullptr, 0);
        return rc2 ? rc2 : lrb_append_composition_txt(out_txt, counts.data(), s->read_len, s->n_reads, k, threads, row0);
    });
    if (!rc) segments_notice(in, 1);
    return rc;
}

extern "C" int lrb_count_15mers(const char* reads_path, const char* out_table, int threads) {
    if (!reads_path || !out_table) return lrb_set_error(LRB_EINVAL, "lrb_count_15mers: null path");
    int rc;
    CtxGuard cg;
    if ((rc = create_ctx(0, &cg.c))) return rc;
    Input in;
    if ((rc = open_input(reads_path, threads, 0, in))) return rc;
    // the same key-partitioned count as the fused stage; the table stays in the context and is streamed to the file
    if (in.whole) rc = lrb_profile_host(cg.c, in.whole, 0, 1, 1, nullptr, nullptr, nullptr, nullptr, LRB_PROFILE_KEEP_TABLE);
    else rc = each_segment(in, false, [&](const lrb_reads* s, uint64_t row0) -> int {
        return lrb_profile_host(cg.c, s, 0, 1, 1, nullptr, nullptr, nullptr, nullptr, row0 ? LRB_PROFILE_ADD_TO_TABLE : LRB_PROFILE_KEEP_TABLE);
    });
    if (rc) return rc;
    if (!in.whole) segments_notice(in, 1);
    return lrb_ctx_table_save(cg.c, out_table);
}

namespace {

// The file-level searches: the coverage rows of every read of reads_path against the table(s) load(context) brings into a
// new context, segment by segment; write(hist, sums, n_reads, row0) appends a segment's rows to the outputs, the n_outs
// files of outs truncated first.  cov is checked; its blocks on slots read the sample slots load() fills.
template <class Load, class Write>
int search_file(const char* who, const CovLayout& cov, const char* reads_path, const char* const* outs, int n_outs, int threads, Load load,
                Write write) {
    int rc = refuse_direct(who, cov);   // before any file or device work
    if (rc) return rc;
    CtxGuard cg;
    if ((rc = create_ctx(0, &cg.c)) || (rc = load(cg.c))) return rc;
    for (int i = 0; i < n_outs; ++i)
        if ((rc = truncate_file(outs[i]))) return rc;
    Input in;
    if ((rc = open_input(reads_path, threads, 4ull * ((uint64_t)cov.W + 1), in))) return rc;
    auto search = [&](const lrb_reads* s, uint64_t row0) -> int {
        const uint64_t n = s->n_reads;
        std::vector<uint32_t> hist((size_t)n * cov.W + 1), sums(n + 1);
        const int rc2 = profile_call(who, cg.c, s, 0, cov, nullptr, hist.data(), sums.data(), nullptr, cov.reads_full() ? LRB_PROFILE_USE_LOADED_TABLE : 0);
        return rc2 ? rc2 : write(hist.data(), sums.data(), n, row0);
    };
    if (in.whole) return search(in.whole, 0);
    if ((rc = each_segment(in, false, search))) return rc;
    segments_notice(in, 1);
    return LRB_OK;
}

// writer of search_file: rows whole, as "%f" text and, when out_npy is given, .npy
auto whole_rows(const char* out_txt, const char* out_npy, uint32_t W, int threads) {
    return [=](const uint32_t* hist, const uint32_t* sums, uint64_t n, uint64_t row0) -> int {
        int rc = lrb_append_coverage_txt(out_txt, hist, sums, n, (int)W, threads, row0);
        if (!rc && out_npy) rc = lrb_append_coverage_npy(out_npy, hist, sums, n, (int)W, threads, row0);
        return rc;
    };
}

}  // namespace

extern "C" int lrb_search_15mers(const char* table_path, const char* reads_path, const char* out_txt, long bin_size,
                                 int bins, int threads) {
    static const char* who = "lrb_search_15mers";
    if (!table_path || !reads_path || !out_txt) return lrb_set_error(LRB_EINVAL, "%s: null path", who);
    CovLayout cov = lrb_cov_settings(1, &bin_size, &bins);
    const int rc = lrb_check_cov_layout(who, &cov);
    if (rc) return rc;
    return search_file(who, cov, reads_path, &out_txt, 1, threads, [&](lrb_ctx* c) { return lrb_ctx_table_load(c, table_path); },
                       whole_rows(out_txt, nullptr, cov.W, threads));
}

extern "C" int lrb_search_15mers_settings(const char* table_path, const char* reads_path, int n, const long* bin_sizes, const int* bins,
                                          const char* const* out_txts, const char* const* out_npys, int threads) {
    static const char* who = "lrb_search_15mers_settings";
    if (!table_path || !reads_path || !out_txts) return lrb_set_error(LRB_EINVAL, "%s: null path", who);
    CovLayout cov = lrb_cov_settings(n, bin_sizes, bins);
    const int rc = lrb_check_cov_layout(who, &cov);
    if (rc) return rc;
    for (int m = 0; m < n; ++m)
        if (!out_txts[m]) return lrb_set_error(LRB_EINVAL, "%s: null output path (setting %d)", who, m);
    // rows of W words come back; each file gets its setting's columns, so the writers are those of lrb_search_15mers
    std::vector<uint32_t> one;
    auto split = [&](const uint32_t* hist, const uint32_t* sums, uint64_t nr, uint64_t row0) -> int {
        int rc2 = LRB_OK;
        for (int m = 0, off = 0; m < n && !rc2; off += bins[m], ++m) {
            const size_t B = (size_t)bins[m];
            one.resize(nr * B + 1);
            for (uint64_t r = 0; r < nr; ++r) std::copy_n(hist + r * cov.W + off, B, one.data() + r * B);
            rc2 = lrb_append_coverage_txt(out_txts[m], one.data(), sums, nr, bins[m], threads, row0);
            if (!rc2 && out_npys && out_npys[m]) rc2 = lrb_append_coverage_npy(out_npys[m], one.data(), sums, nr, bins[m], threads, row0);
        }
        return rc2;
    };
    return search_file(who, cov, reads_path, out_txts, n, threads, [&](lrb_ctx* c) { return lrb_ctx_table_load(c, table_path); }, split);
}

extern "C" int lrb_search_15mers_samples(const char* const* table_paths, int n, const long* bin_sizes, const int* bins, const char* reads_path,
                                         const char* out_txt, const char* out_npy, int threads) {
    static const char* who = "lrb_search_15mers_samples";
    if (!table_paths || !reads_path || !out_txt) return lrb_set_error(LRB_EINVAL, "%s: null path", who);
    // slot of each table, numbered in order of first appearance: a table listed twice (the same path string) is loaded once
    int slots[LRB_MAX_SAMPLE_TABLES] = {}, n_slots = 0;
    for (int t = 0; t < n && t < LRB_MAX_SAMPLE_TABLES; ++t) {
        if (!table_paths[t]) return lrb_set_error(LRB_EINVAL, "%s: null table path (table %d)", who, t);
        int j = 0;
        while (j < t && strcmp(table_paths[j], table_paths[t])) ++j;
        slots[t] = j == t ? n_slots++ : slots[j];
    }
    CovLayout cov = lrb_cov_settings(n, bin_sizes, bins, slots);
    const int rc = lrb_check_cov_layout(who, &cov);
    if (rc) return rc;
    auto load = [&](lrb_ctx* c) -> int {
        for (int t = 0, next = 0; t < n; ++t)
            if (slots[t] == next) {
                const int rc2 = lrb_ctx_sample_table_load(c, next++, table_paths[t]);
                if (rc2) return rc2;
            }
        return LRB_OK;
    };
    // every block of a row is normalised by the same sums (the read's valid windows), so the writers of one table apply at
    // width W and the line is the n single-table lines joined by one space
    return search_file(who, cov, reads_path, &out_txt, 1, threads, load, whole_rows(out_txt, out_npy, cov.W, threads));
}

extern "C" int lrb_search_15mers_edges(const char* table_path, const char* reads_path, const uint32_t* edges, int n_edges,
                                       const char* out_txt, const char* out_npy, int threads) {
    static const char* who = "lrb_search_15mers_edges";
    if (!table_path || !reads_path || !out_txt) return lrb_set_error(LRB_EINVAL, "%s: null path", who);
    CovLayout cov = lrb_cov_edges(edges, n_edges);
    const int rc = lrb_check_cov_layout(who, &cov);
    if (rc) return rc;
    return search_file(who, cov, reads_path, &out_txt, 1, threads, [&](lrb_ctx* c) { return lrb_ctx_table_load(c, table_path); },
                       whole_rows(out_txt, out_npy, cov.W, threads));
}

extern "C" int lrb_search_15mers_layout(const char* const* table_paths, int n_tables, const char* reads_path, const lrb_cov_block* blocks, int n,
                                        const char* out_txt, const char* out_npy, int threads) {
    static const char* who = "lrb_search_15mers_layout";
    if (!table_paths || !reads_path || !out_txt) return lrb_set_error(LRB_EINVAL, "%s: null path", who);
    if (n_tables < 1 || n_tables > LRB_MAX_SAMPLE_TABLES)
        return lrb_set_error(LRB_EINVAL, "%s: the number of tables must be in [1, %d] (got %d)", who, LRB_MAX_SAMPLE_TABLES, n_tables);
    CovLayout cov = lrb_cov_layout(blocks, n);
    int rc = lrb_check_cov_layout(who, &cov);
    if (rc) return rc;
    // slot of each table, numbered in order of first appearance: a path listed twice (the same string) is loaded once
    int slot_of[LRB_MAX_SAMPLE_TABLES] = {}, n_slots = 0;
    const char* slot_path[LRB_MAX_SAMPLE_TABLES] = {};
    for (int t = 0; t < n_tables; ++t) {
        if (!table_paths[t]) return lrb_set_error(LRB_EINVAL, "%s: null table path (table %d)", who, t);
        int j = 0;
        while (j < t && strcmp(table_paths[j], table_paths[t])) ++j;
        slot_of[t] = j == t ? n_slots++ : slot_of[j];
        slot_path[slot_of[t]] = table_paths[j];
    }
    for (int m = 0; m < cov.n; ++m) {
        const int t = cov.b[m].table;
        if (t < 0 || t >= n_tables)
            return lrb_set_error(LRB_EINVAL, "%s: block %d reads table %d; a block of a file-level layout names its table by its index in [0, %d) "
                                 "of table_paths", who, m, t, n_tables);
        cov.b[m].table = slot_of[t];
    }
    if ((rc = lrb_check_cov_layout(who, &cov))) return rc;   // the same path and binning twice
    bool used[LRB_MAX_SAMPLE_TABLES] = {};
    for (int m = 0; m < cov.n; ++m) used[cov.b[m].table] = true;
    auto load = [&](lrb_ctx* c) -> int {   // the tables some block reads
        for (int t = 0; t < n_slots; ++t) {
            const int rc2 = used[t] ? lrb_ctx_sample_table_load(c, t, slot_path[t]) : LRB_OK;
            if (rc2) return rc2;
        }
        return LRB_OK;
    };
    // every block of a row is normalised by the same sums (the read's valid windows), so the writers of one block apply at
    // width W and the line is the n single-block lines joined by one space
    return search_file(who, cov, reads_path, &out_txt, 1, threads, load, whole_rows(out_txt, out_npy, cov.W, threads));
}

extern "C" int lrb_table_spectrum(const char* table_path, const char* out_txt, uint32_t max_count) {
    if (!table_path || !out_txt) return lrb_set_error(LRB_EINVAL, "lrb_table_spectrum: null path");
    if (max_count < 2 || max_count > LRB_SPECTRUM_MAX_COUNT)
        return lrb_set_error(LRB_EINVAL, "max_count must be in [2, %u] (got %u)", LRB_SPECTRUM_MAX_COUNT, max_count);
    int rc;
    CtxGuard cg;
    if ((rc = create_ctx(1, &cg.c))) return rc;
    if ((rc = lrb_ctx_table_load(cg.c, table_path))) return rc;
    std::vector<uint64_t> spec((size_t)max_count + 3);
    if ((rc = lrb_ctx_table_spectrum(cg.c, max_count, spec.data()))) return rc;
    return lrb_write_spectrum_txt(out_txt, spec.data(), max_count);
}

extern "C" int lrb_profile_multi(const char* reads_path, const char* out_dir, int k, long bin_size, int bins, int threads,
                                 int n_gpus, int write_table, int write_npy) {
    if (!reads_path || !out_dir) return lrb_set_error(LRB_EINVAL, "lrb_profile: null path");
    const int P = comp_width(k);
    if (!P) return lrb_set_error(LRB_EINVAL, "k must be 3, 4 or 5 (got %d)", k);
    if (bin_size <= 0) return lrb_set_error(LRB_EINVAL, "bin_size must be >= 1 (the reference divides by it)");
    if (bins <= 0 || bins > LRB_MAX_BINS) return lrb_set_error(LRB_EINVAL, "bins must be in [1, %d]", LRB_MAX_BINS);
    const std::string prof = std::string(out_dir) + "/profiles";
    int rc;
    if ((rc = make_dir(out_dir)) || (rc = make_dir(prof.c_str()))) return rc;
    CtxGuard cg;
    if ((rc = create_ctx(n_gpus, &cg.c))) return rc;
    Input in;
    if ((rc = open_input(reads_path, threads, 4ull * ((uint64_t)P + bins + 1), in))) return rc;
    const std::string com = prof + "/com_profs", cov = prof + "/cov_profs", com_npy = com + ".npy", cov_npy = cov + ".npy";
    if (in.whole) {
        const lrb_reads* r = in.whole;
        const uint64_t n = r->n_reads;
        std::vector<uint32_t> counts((size_t)n * P + 1), hist((size_t)n * bins + 1), sums(n + 1);
        if ((rc = lrb_profile_host(cg.c, r, k, bin_size, bins, counts.data(), hist.data(), sums.data(), nullptr, 0))) return rc;
        if ((rc = lrb_write_composition_txt(com.c_str(), counts.data(), r->read_len, n, k, threads))) return rc;
        if ((rc = lrb_write_coverage_txt(cov.c_str(), hist.data(), sums.data(), n, bins, threads))) return rc;
        if (write_npy) {
            if ((rc = lrb_write_composition_npy(com_npy.c_str(), counts.data(), r->read_len, n, k, threads))) return rc;
            if ((rc = lrb_write_coverage_npy(cov_npy.c_str(), hist.data(), sums.data(), n, bins, threads))) return rc;
        }
    } else {
        // pass 1: composition rows, and every segment counted into the one table
        rc = each_segment(in, false, [&](const lrb_reads* s, uint64_t row0) -> int {
            const uint64_t n = s->n_reads;
            std::vector<uint32_t> counts((size_t)n * P + 1);
            int rc2 = lrb_profile_host(cg.c, s, k, bin_size, bins, counts.data(), nullptr, nullptr, nullptr,
                                       row0 ? LRB_PROFILE_ADD_TO_TABLE : LRB_PROFILE_KEEP_TABLE);
            if (!rc2) rc2 = lrb_append_composition_txt(com.c_str(), counts.data(), s->read_len, n, k, threads, row0);
            if (!rc2 && write_npy) rc2 = lrb_append_composition_npy(com_npy.c_str(), counts.data(), s->read_len, n, k, threads, row0);
            return rc2;
        });
        if (rc) return rc;
        // pass 2: the file again, every segment searched against the finished table
        rc = each_segment(in, true, [&](const lrb_reads* s, uint64_t row0) -> int {
            const uint64_t n = s->n_reads;
            std::vector<uint32_t> hist((size_t)n * bins + 1), sums(n + 1);
            int rc2 = lrb_profile_host(cg.c, s, k, bin_size, bins, nullptr, hist.data(), sums.data(), nullptr, LRB_PROFILE_USE_LOADED_TABLE);
            if (!rc2) rc2 = lrb_append_coverage_txt(cov.c_str(), hist.data(), sums.data(), n, bins, threads, row0);
            if (!rc2 && write_npy) rc2 = lrb_append_coverage_npy(cov_npy.c_str(), hist.data(), sums.data(), n, bins, threads, row0);
            return rc2;
        });
        if (rc) return rc;
        segments_notice(in, 2);
    }
    if (write_table && (rc = lrb_ctx_table_save(cg.c, (prof + "/15mers-counts").c_str()))) return rc;
    return LRB_OK;
}

extern "C" int lrb_profile(const char* reads_path, const char* out_dir, int k, long bin_size, int bins, int threads,
                           int write_table, int write_npy) {
    return lrb_profile_multi(reads_path, out_dir, k, bin_size, bins, threads, 0, write_table, write_npy);
}
