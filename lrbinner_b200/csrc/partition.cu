// partition.cu — L2-resident 15-mer table passes (count and search) via one key-partition of the windows.
//
// Why (measured on this pool's B200, profiles/r01_ubench_roofline.jsonl): uniform-random RED.ADD.U32 runs at
// 20 G/s over a 4 GiB table (every update misses L2: a sector pair in, a sector out) but at ~190 G/s when
// the touched slice is <= 64 MiB; random 4 B gathers: 38-48 G/s vs 288 G/s.  The direct kernels
// (kernels.cu: k_count15 / k_search15) sit exactly on the DRAM-random numbers (profiles/r01_bench_n1_v0_*).
// Here the valid windows are first partitioned by the high bits of their bit-15-clear key into buckets whose
// table slice (2^24 keys = 64 MiB of addresses, 32 MiB touched because bit 15 is clear) fits the 126 MB L2
// together with the histogram rows; then, bucket by bucket, the lists are streamed back (coalesced) and
// applied to the resident slice.
//
// Layout of the lists (deterministic, no global cursors).  A STEP is 256 consecutive blocks (8192 slots) of a
// chunk of the stream.  The windows of step s that fall into bucket b form a RUN; bucket b's region of the
// chunk is the concatenation of its runs in step order.  One list entry is 4 bytes:
//     entry = compact(key inside the bucket) | (read index - read index of the step's first block) << (shift-1)
// compact() drops bit 15 (always 0 for the bit-15-clear key); a step spans at most 256 reads (every read owns at
// least one block), so the read delta needs 8 bits and shift <= 25.
//
//   k_step_hist     one scan of the chunk: windows per (step, bucket) -> step_cnt (u16), per-group totals
//   k_group_scan    per bucket: exclusive scan of the group totals, bucket total; its last CTA also computes the region
//                   offsets of the chunk (exclusive scan over buckets) and guards the capacity
//   k_partition     second scan: each CTA walks the steps of its group in order; the entries of a step are ranked
//                   and placed in shared memory in ONE pass (the staging offsets are known from step_cnt), then
//                   copied out run by run (contiguous on both sides); writes step_off[bucket][step]
//   k_count_keys    per bucket: RED.ADD.U32 table[key]                              (L2-resident atomics)
//   k_search_keys   per bucket, warp per run: count = table[key] (an L2 hit), bucket rule, aggregation of equal
//                   (read, bin) entries of the warp, RED into hist[read][bin]
//   k_search_settings  the same walk, the gathered count binned by up to 8 (bin size, bin count) settings into one
//                   row of their concatenated bins (lrb_dev_partition_search_settings)
//   k_search_samples  the same walk over compact sample tables, one or two per launch: each table's count binned by
//                   its own setting into its column block of one row (lrb_dev_partition_search_samples)
//   k_search_edges  the same walk, the gathered count binned by caller-given count edges: bin = #{i : t_i <= count}
//                   (lrb_dev_partition_search_edges)
//   k_search_layout  the same walk, once per distinct table of a mixed row: the gathered count binned by every block of
//                   that table, (bin size, bin count) or count edges, into the block's columns (lrb_dev_partition_search_layout)
//   k_row_sums      sums[read] = sum of hist[read][*]  (every window lands in exactly one bin of each setting)
//
// The stream can be added in several chunks (lrb_dev_partition_add), each with its own regions, so the
// partition of chunk i overlaps the host-to-device copy of chunk i+1; everything is asynchronous on the
// caller's stream.  Results are bit-identical to the direct kernels: same windows, same keys, integer sums.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <algorithm>

#include "../../include/lrbinner_b200.h"
#include "common.h"
#include "lane_core.cuh"

using namespace lrb;

namespace {

constexpr int kPartThreads = 256;          // one 32-slot block per thread -> 8192 slots per step
constexpr int kStepSlots = kPartThreads * 32;
constexpr int kMaxBuckets = LRB_PART_MAX_BUCKETS;
constexpr int kMaxChunks = LRB_PART_MAX_CHUNKS;
constexpr int kMaxGroups = LRB_PART_MAX_GROUPS;
constexpr int kSubBits = 15;               // a sub-slice = 2^15 bit-15-clear keys = 128 KB of u32 counters in shared memory
constexpr int kMaxSubs = 1 << (25 - 16);   // sub-slices per bucket at the largest bucket size (shift 25)
constexpr uint64_t kMaxChunkBlocks = 1ull << 26;  // 2^31 slots: run offsets inside a chunk's bucket region fit u32
typedef unsigned long long ull;

// device-side bookkeeping, lives in lrb_partition.small (LRB_PART_SMALL_U64 u64)
struct PartMeta {
    ull counts[kMaxChunks][kMaxBuckets];   // entries of (chunk, bucket)
    ull offsets[kMaxChunks][kMaxBuckets];  // first entry of (chunk, bucket) in keys[]
    ull chunk_base[kMaxChunks + 1];        // first entry of each chunk's region
    ull needed;                            // entries the chunks added so far need in total
    ull overflow;                          // != 0: capacity exceeded, lists are incomplete (apply does nothing)
    uint32_t overflow2[kMaxBuckets];       // second level: bucket b could not be listed (spill area full) -> k_count_keys counts b
    ull spill_n;                           // entries in the spill area (second level: rows / segments that overflowed)
    ull spill_dropped;                     // != 0: the spill area itself overflowed (its buckets are flagged in overflow2)
    uint32_t scan_ticket;                  // k_group_scan: CTAs that have finished their bucket (the last one scans the chunk)
};
static_assert(sizeof(PartMeta) <= sizeof(ull) * LRB_PART_SMALL_U64, "lrb_partition.small too small");

// views into lrb_partition.steps (u32 words)
struct StepTables {
    uint32_t* grp_tot;    // [kMaxGroups][64]  windows of (group, bucket)                (re-used by every chunk)
    uint32_t* grp_off;    // [kMaxGroups][64]  exclusive scan over groups
    uint32_t* rid0;       // [cap]             read index of the step's first block
    uint16_t* cnt;        // [cap][64]         windows of (step, bucket)
    uint32_t* off;        // [64][cap]         first entry of run (bucket, step) inside the chunk's bucket region
    uint64_t cap;
};

__host__ __device__ inline StepTables step_tables(uint32_t* steps, uint64_t cap) {
    StepTables t;
    t.cap = cap;
    t.grp_tot = steps;
    t.grp_off = t.grp_tot + (size_t)kMaxGroups * kMaxBuckets;
    t.rid0 = t.grp_off + (size_t)kMaxGroups * kMaxBuckets;
    t.cnt = reinterpret_cast<uint16_t*>(t.rid0 + cap);
    t.off = t.rid0 + cap + cap * (kMaxBuckets / 2);
    return t;
}

struct ChunkList {  // by-value kernel argument of the apply kernels
    uint32_t step0[kMaxChunks];
    uint32_t nsteps[kMaxChunks];
    uint32_t task0[kMaxChunks + 1];  // first search task of each chunk (k_search_keys)
};

__global__ void __launch_bounds__(256) k_fill_blk_read(lrb_reads_view R, uint32_t* __restrict__ blk_read) {
    const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= R.n_reads) return;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t b1 = R.read_blk[r + 1];
    for (uint32_t b = R.read_blk[r] + lane; b < b1; b += 32) blk_read[b] = (uint32_t)r;
}

struct BlockWindows {
    uint32_t m, pw, w0, w1;
};

__device__ __forceinline__ BlockWindows load_block(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ valid,
                                                   uint64_t gb) {
    BlockWindows b;
    const uint32_t v = __ldg(valid + gb);
    const uint32_t pv = gb ? __ldg(valid + gb - 1) : 0u;
    b.m = window15_mask(pv, v);
    b.pw = b.w0 = b.w1 = 0;
    if (b.m) {
        const uint2 w = __ldg(reinterpret_cast<const uint2*>(codes) + gb);
        b.w0 = w.x;
        b.w1 = w.y;
        b.pw = gb ? __ldg(codes + 2 * gb - 1) : 0u;
    }
    return b;
}

// f(key) for every window of the block whose bit-15-clear key lies in the partition's key range.  The common case
// (every lane of the warp holds an interior block of a read, whole key space) runs without any predicate.
template <bool FULL, class F>
__device__ __forceinline__ void for_each_key(const BlockWindows& b, uint32_t key_lo, uint32_t key_hi, F f) {
    const uint32_t r0 = rc16(b.w1), r1 = rc16(b.w0), r2 = rc16(b.pw);
    if (FULL && __all_sync(0xFFFFFFFFu, b.m == 0xFFFFFFFFu)) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f(canonical15(kmer_ending_at<15>(b.pw, b.w0, b.w1, j), rc15_ending_at(r0, r1, r2, j)));
    } else if (__any_sync(0xFFFFFFFFu, b.m != 0u)) {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            if ((b.m >> j) & 1u) {
                const uint32_t kk = canonical15(kmer_ending_at<15>(b.pw, b.w0, b.w1, j), rc15_ending_at(r0, r1, r2, j));
                if (FULL || (kk >= key_lo && kk < key_hi)) f(kk);
            }
        }
    }
}

// ---- pass 1: windows per (step, bucket) --------------------------------------------------------------------
// CTA g walks the steps [g*G, (g+1)*G) of the chunk.  s_cnt is double-buffered so one barrier per step suffices.
template <bool FULL>
__global__ void __launch_bounds__(kPartThreads)
k_step_hist(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ valid, const uint32_t* __restrict__ blk_read,
            uint64_t blk_lo, uint64_t blk_hi, uint32_t key_lo, uint32_t key_hi, int shift, uint32_t n_steps, uint32_t G,
            uint32_t step0, StepTables T) {
    __shared__ uint32_t s_cnt[2][kMaxBuckets];
    const int tid = threadIdx.x;
    if (tid < 2 * kMaxBuckets) (&s_cnt[0][0])[tid] = 0;
    __syncthreads();
    const uint32_t bucket0 = key_lo >> shift;
    const uint32_t s_beg = blockIdx.x * G, s_end = min(n_steps, s_beg + G);
    uint32_t run = 0;  // thread b < 64: windows of (this group, bucket b) so far
    for (uint32_t s = s_beg; s < s_end; ++s) {
        uint32_t* cnt = s_cnt[s & 1u];
        const uint64_t gb = blk_lo + (uint64_t)s * kPartThreads + tid;
        BlockWindows b;
        b.m = b.pw = b.w0 = b.w1 = 0;
        if (gb < blk_hi) b = load_block(codes, valid, gb);
        for_each_key<FULL>(b, key_lo, key_hi, [&](uint32_t kk) { atomicAdd(&cnt[(kk >> shift) - bucket0], 1u); });
        __syncthreads();
        if (tid < kMaxBuckets) {
            const uint32_t c = cnt[tid];
            cnt[tid] = 0;  // next used at step s+2, after another barrier
            T.cnt[(size_t)(step0 + s) * kMaxBuckets + tid] = (uint16_t)c;
            run += c;
        }
        if (tid == kMaxBuckets && blk_read) T.rid0[step0 + s] = __ldg(blk_read + blk_lo + (uint64_t)s * kPartThreads);
    }
    if (tid < kMaxBuckets) T.grp_tot[(size_t)blockIdx.x * kMaxBuckets + tid] = run;
}

__device__ void chunk_scan_warp(PartMeta* __restrict__ m, int c, int nb, ull capacity);

// CTA b: grp_off[g][b] = exclusive scan over groups of grp_tot[g][b]; counts[c][b] = total.  The CTA that finishes last
// also computes the chunk's region offsets (chunk_scan_warp): a second launch for that one warp cost 30 us per chunk in the
// dependency chain of the host pipeline's 16 chunks.
__global__ void __launch_bounds__(256) k_group_scan(StepTables T, uint32_t n_groups, PartMeta* __restrict__ meta, int c, int nb, ull capacity) {
    __shared__ uint32_t s_last;
    __shared__ ull s_part[256];
    const uint32_t b = blockIdx.x, tid = threadIdx.x;
    const uint32_t span = (n_groups + 255u) / 256u;
    const uint32_t g0 = min(n_groups, tid * span), g1 = min(n_groups, g0 + span);
    ull sum = 0;
    for (uint32_t g = g0; g < g1; ++g) sum += T.grp_tot[(size_t)g * kMaxBuckets + b];
    s_part[tid] = sum;
    __syncthreads();
    for (int d = 1; d < 256; d <<= 1) {  // Hillis-Steele inclusive scan
        const ull v = (tid >= (uint32_t)d) ? s_part[tid - d] : 0ull;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    ull acc = s_part[tid] - sum;
    for (uint32_t g = g0; g < g1; ++g) {
        T.grp_off[(size_t)g * kMaxBuckets + b] = (uint32_t)acc;  // < 2^31: a chunk has at most 2^31 slots
        acc += T.grp_tot[(size_t)g * kMaxBuckets + b];
    }
    if (tid == 255) {
        meta->counts[c][b] = s_part[255];
        __threadfence();
        const uint32_t ticket = atomicAdd(&meta->scan_ticket, 1u);
        s_last = (ticket == gridDim.x - 1u) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last && tid < 32) {
        __threadfence();   // the other CTAs' counts are visible
        chunk_scan_warp(meta, c, nb, capacity);
        if (tid == 0) meta->scan_ticket = 0;   // for the next chunk
    }
}

// one warp: offsets of chunk c = chunk_base[c] + exclusive scan of its bucket counts; guards the capacity
__device__ void chunk_scan_warp(PartMeta* __restrict__ m, int c, int nb, ull capacity) {
    const int lane = threadIdx.x & 31;
    const ull c0 = (lane < nb) ? m->counts[c][lane] : 0ull;
    const ull c1 = (lane + 32 < nb) ? m->counts[c][lane + 32] : 0ull;
    ull x0 = c0, x1 = c1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const ull y0 = __shfl_up_sync(0xFFFFFFFFu, x0, d), y1 = __shfl_up_sync(0xFFFFFFFFu, x1, d);
        if (lane >= d) { x0 += y0; x1 += y1; }
    }
    const ull tot0 = __shfl_sync(0xFFFFFFFFu, x0, 31);
    const ull total = tot0 + __shfl_sync(0xFFFFFFFFu, x1, 31);
    const ull base = m->chunk_base[c];
    const bool fits = (m->overflow == 0) && (base + total <= capacity);
    __syncwarp();
    m->offsets[c][lane] = base + x0 - c0;
    m->offsets[c][lane + 32] = base + tot0 + x1 - c1;
    if (!fits) {  // keep the lists consistent (this chunk contributes nothing) and remember how much was needed
        m->counts[c][lane] = 0;
        m->counts[c][lane + 32] = 0;
    }
    if (lane == 0) {
        m->needed += total;
        m->chunk_base[c + 1] = fits ? base + total : base;
        if (!fits) m->overflow = 1;
    }
}

// ---- pass 2: entries -> bucket regions ---------------------------------------------------------------------
// Per step: (prelude, warp 0) staging layout from the step's known bucket counts; (rank + place) every window takes
// the next staging slot of its bucket with one shared-memory atomic and drops its entry there; (copy-out) each warp
// copies whole runs, contiguous on both sides.  The next step's block and prelude are fetched while the current one
// is copied out; two barriers per step.  The kernel is bound by shared-memory wavefronts (the scattered staging
// store and the ranking atomic), so nothing else is staged.
template <bool WITH_RID, bool FULL>
__global__ void __launch_bounds__(kPartThreads)
k_partition(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ valid, const uint32_t* __restrict__ blk_read,
            uint64_t blk_lo, uint64_t blk_hi, uint32_t key_lo, uint32_t key_hi, int shift, int nb, uint32_t n_steps, uint32_t G,
            uint32_t step0, StepTables T, const PartMeta* __restrict__ meta, int c, uint32_t* __restrict__ ent_out) {
    __shared__ uint32_t s_ent[kStepSlots];                          // staged entries, grouped by bucket
    __shared__ uint32_t s_cur[2][kMaxBuckets];                      // staging cursor of each bucket
    __shared__ uint32_t s_beg[2][kMaxBuckets], s_n[2][kMaxBuckets]; // staged run of each bucket
    __shared__ uint32_t* s_dst[2][kMaxBuckets];                     // where the run goes in ent_out
    if (meta->overflow) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t bucket0 = key_lo >> shift;
    const uint32_t lo15 = 0x7FFFu, hi_mask = ((1u << (shift - 1)) - 1u) & ~lo15;
    const uint32_t s_first = blockIdx.x * G, s_end = min(n_steps, s_first + G);
    // lane l of warp 0 keeps the running offsets of buckets l and l+32 inside their regions
    uint32_t run0 = 0, run1 = 0;
    ull reg0 = 0, reg1 = 0;
    if (warp == 0) {
        if (lane < nb) { run0 = T.grp_off[(size_t)blockIdx.x * kMaxBuckets + lane]; reg0 = meta->offsets[c][lane]; }
        if (lane + 32 < nb) { run1 = T.grp_off[(size_t)blockIdx.x * kMaxBuckets + lane + 32]; reg1 = meta->offsets[c][lane + 32]; }
    }
    auto prelude = [&](uint32_t s, int buf) {  // warp 0 only
        const uint16_t* cs = T.cnt + (size_t)(step0 + s) * kMaxBuckets;
        const uint32_t c0 = (lane < nb) ? cs[lane] : 0u;
        const uint32_t c1 = (lane + 32 < nb) ? cs[lane + 32] : 0u;
        uint32_t x0 = c0, x1 = c1;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y0 = __shfl_up_sync(0xFFFFFFFFu, x0, d), y1 = __shfl_up_sync(0xFFFFFFFFu, x1, d);
            if (lane >= d) { x0 += y0; x1 += y1; }
        }
        const uint32_t tot0 = __shfl_sync(0xFFFFFFFFu, x0, 31);
        const uint32_t e0 = x0 - c0, e1 = tot0 + x1 - c1;  // exclusive staging offsets
        s_cur[buf][lane] = s_beg[buf][lane] = e0;
        s_cur[buf][lane + 32] = s_beg[buf][lane + 32] = e1;
        s_n[buf][lane] = c0;
        s_n[buf][lane + 32] = c1;
        s_dst[buf][lane] = ent_out + (reg0 + run0);
        s_dst[buf][lane + 32] = ent_out + (reg1 + run1);
        if (lane < nb) T.off[(size_t)lane * T.cap + step0 + s] = run0;
        if (lane + 32 < nb) T.off[(size_t)(lane + 32) * T.cap + step0 + s] = run1;
        run0 += c0;
        run1 += c1;
    };
    // all loads of a block are issued back to back (no load depends on another), so a prefetch never stalls
    auto fetch = [&](uint32_t s, uint32_t& v, uint32_t& pv, BlockWindows& b, uint32_t& rd, uint32_t& r0v) {
        const uint64_t gb = blk_lo + (uint64_t)s * kPartThreads + tid;
        v = pv = b.pw = b.w0 = b.w1 = rd = r0v = 0;
        if (gb < blk_hi) {
            v = __ldg(valid + gb);
            pv = gb ? __ldg(valid + gb - 1) : 0u;
            const uint2 w = __ldg(reinterpret_cast<const uint2*>(codes) + gb);
            b.w0 = w.x;
            b.w1 = w.y;
            b.pw = gb ? __ldg(codes + 2 * gb - 1) : 0u;
            if (WITH_RID) { rd = __ldg(blk_read + gb); r0v = __ldg(T.rid0 + step0 + s); }
        }
    };
    BlockWindows b;
    uint32_t v, pv, rd, r0v;
    if (s_first < s_end) {
        fetch(s_first, v, pv, b, rd, r0v);
        if (warp == 0) prelude(s_first, 0);
    }
    __syncthreads();
    for (uint32_t s = s_first; s < s_end; ++s) {
        const int buf = (int)((s - s_first) & 1u);
        uint32_t* cur = s_cur[buf];
        b.m = window15_mask(pv, v);
        const uint32_t rds = (rd - r0v) << (shift - 1);
        for_each_key<FULL>(b, key_lo, key_hi, [&](uint32_t kk) {
            const uint32_t idx = atomicAdd(&cur[(kk >> shift) - bucket0], 1u);
            s_ent[idx] = (kk & lo15) | ((kk >> 1) & hi_mask) | rds;
        });
        __syncthreads();
        if (s + 1 < s_end) {  // next step's inputs travel while this one is copied out
            fetch(s + 1, v, pv, b, rd, r0v);
            if (warp == 0) prelude(s + 1, buf ^ 1);
        }
        for (int bk = warp; bk < nb; bk += kPartThreads / 32) {  // each warp copies whole runs: contiguous both sides
            const uint32_t n = s_n[buf][bk];
            const uint32_t* src = s_ent + s_beg[buf][bk];
            uint32_t* dst = s_dst[buf][bk];
#pragma unroll 2
            for (uint32_t i = lane; i < n; i += 32) __stcs(dst + i, src[i]);
        }
        __syncthreads();
    }
    // terminal offsets (run lengths are differences of consecutive step_off entries)
    if (warp == 0 && s_end == n_steps && s_first < s_end) {
        if (lane < nb) T.off[(size_t)lane * T.cap + step0 + n_steps] = run0;
        if (lane + 32 < nb) T.off[(size_t)(lane + 32) * T.cap + step0 + n_steps] = run1;
    }
}

// list entry -> table index (bucket_base = first key of the bucket)
__device__ __forceinline__ uint32_t entry_key(uint32_t e, uint32_t bucket_base, uint32_t hi_mask2) {
    return bucket_base | (e & 0x7FFFu) | ((e << 1) & hi_mask2);
}

// one RED per distinct key of the warp's 32 entries: equal keys come in runs when a read is a homopolymer or a tandem
// repeat, and same-address atomics serialise (profiles/r02_exp_skew_*.jsonl)
__device__ __forceinline__ void red_aggregated(uint32_t* __restrict__ table, uint32_t key, bool active) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, active ? key : (0xFFFFFFE0u | lane));   // inactive lanes match nobody (keys are < 2^30)
    if (active && (uint32_t)__ffs(peers) - 1u == lane) atomicAdd(table + key, (uint32_t)__popc(peers));
}

__global__ void __launch_bounds__(256)
k_count_keys(const uint32_t* __restrict__ ents, const PartMeta* __restrict__ meta, int bucket0, int n_chunks, uint32_t bucket_base0,
             int shift, uint32_t hi_mask2, uint32_t* __restrict__ table, int fallback_only) {
    const int bucket = bucket0 + (int)blockIdx.y;   // one launch may cover several buckets (gridDim.y)
    const uint32_t bucket_base = bucket_base0 + ((uint32_t)blockIdx.y << shift);
    if (meta->overflow) return;
    if (fallback_only && !meta->overflow2[bucket]) return;  // the shared-memory path counted this bucket
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    if (fallback_only) {   // a bucket that could not be listed is a key-skewed one: aggregate equal keys (warp-uniform loop)
        for (int c = 0; c < n_chunks; ++c) {
            const uint64_t n = meta->counts[c][bucket];
            const uint32_t* __restrict__ ee = ents + meta->offsets[c][bucket];
            for (uint64_t i0 = ((uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)); i0 < n; i0 += stride) {
                const uint64_t i = i0 + (threadIdx.x & 31u);
                const bool act = i < n;
                red_aggregated(table, act ? entry_key(__ldcs(ee + i), bucket_base, hi_mask2) : 0u, act);
            }
        }
        return;
    }
    for (int c = 0; c < n_chunks; ++c) {
        const uint64_t n = meta->counts[c][bucket];
        const uint32_t* __restrict__ ee = ents + meta->offsets[c][bucket];
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        for (; i + 3 * stride < n; i += 4 * stride) {
            const uint32_t e0 = __ldcs(ee + i), e1 = __ldcs(ee + i + stride), e2 = __ldcs(ee + i + 2 * stride),
                           e3 = __ldcs(ee + i + 3 * stride);
            atomicAdd(table + entry_key(e0, bucket_base, hi_mask2), 1u);
            atomicAdd(table + entry_key(e1, bucket_base, hi_mask2), 1u);
            atomicAdd(table + entry_key(e2, bucket_base, hi_mask2), 1u);
            atomicAdd(table + entry_key(e3, bucket_base, hi_mask2), 1u);
        }
        for (; i < n; i += stride) atomicAdd(table + entry_key(__ldcs(ee + i), bucket_base, hi_mask2), 1u);
    }
}

// ---- second level (count only): bucket lists -> 2-byte lists per 2^15-key sub-slice -> shared-memory counting ------
// RED.ADD into an L2-resident slice tops out near 1.3 cycles per lane per SM (~196 G/s on this part,
// profiles/r01_ubench_roofline.jsonl); shared-memory atomics run ~8x faster.  So for counting, every bucket's list is
// partitioned once more by the next key bits into sub-slices of 2^15 keys whose counters fit one SM's shared memory.
//
// k2_partition runs once per chunk, right after k_partition (so in the host pipeline it sits in the shadow of the
// host-to-device copy of the next chunk): persistent CTAs take tiles of 8192 entries of the chunk's bucket regions,
// kL2Run consecutive tiles of one bucket at a time (schedule in the kernel).  Every entry is touched ONCE: it arrives in a register (the next tile's entries are fetched while the
// current ones are swept), takes the next slot of its sub-slice's staging row with one returning shared-memory atomic
// and drops its low 15 key bits there (2-byte staging, kL2Stage slots = 4x the expected share per sub-slice, so no
// count pass and no scan are needed); after one barrier each warp sweeps the rows of the sub-slices it owns into the
// lists (each row is staged at its destination's position modulo 8, so it is copied as 16-byte words after a short
// head).  The few entries that find their row full go through a small overflow list that
// the owning warp appends after the row.  Every CTA appends to its OWN segment of every (bucket, sub-slice) list
// ([bucket][sub][cta][C3] entries; fill counters in a private global row, read and written only by the owning lane),
// so there is no reservation between CTAs and no ordering; list order is irrelevant for counting.  Segments have a
// fixed capacity (a multiple of the expected fill); a bucket whose keys are skewed enough to overflow a segment (or
// the per-tile overflow list) raises overflow2[bucket] and is counted by k_count_keys instead (both count kernels look
// at the flag).  Workspace (u16 units): fill[n_cta][n_buckets * nsub] as u32, then per bucket its segments.
constexpr int kL2Threads = 512;   // 16 entries per thread
constexpr int kL2Warps = kL2Threads / 32;
constexpr int kL2PerThread = kStepSlots / kL2Threads;
constexpr int kL2Stage = 32768;   // u16 staging slots (64 KB): rows of kL2Stage / nsub slots
constexpr int kL2Ovl = 1536;      // entries of a tile that may miss their staging row before the bucket falls back
constexpr uint32_t kL2Run = 8;    // consecutive tiles of one bucket a CTA takes at a time
constexpr int kL2CtasPerSm = 2;   // measured: a third CTA per SM (fits: 40 registers, 74 KB) makes the kernel 40 % slower (l1tex is already 80 % busy)

struct L2Layout {
    uint32_t nsub, n_cta, C3, nb;   // sub-slices per bucket, CTAs of k2_partition, UNIFORM entries per segment (small inputs), buckets
    // position of a sub-slice's counter in a fill row: the sub-slices warp + 16 j that one k2_partition warp owns sit next to
    // each other, so its lanes read and write one 64-byte stretch instead of 16 sectors
    __host__ __device__ uint32_t fill_pos(uint32_t sub) const { return (sub & 15u) * (nsub >> 4) + (sub >> 4); }
    // Segments.  A CELL is one (bucket, sub-slice) pair, cell = bucket * nsub + sub; its n_cta segments of cell_cap[cell]
    // entries each lie back to back ([cta][cap]) at seg0 + 8 * cell_off[cell] (u16 units; offsets are kept in octets so
    // that 32 bits reach 64 GB).  Capacities FOLLOW THE KEY DISTRIBUTION: k_sample_cells histograms the cells of a
    // sample of the first chunk's blocks, k_plan_cells hands every cell its share of the segment space (plus a floor), so a
    // GC-skewed community fills its segments as evenly as a uniform one (round 1 / early round 2 gave every cell the same
    // capacity and leaned on the fallback / spill area).  Too small a sample -> the uniform C3.
    uint64_t seg0, seg_units;       // first segment; u16 units available for segments
    // cell table (u16 offset cells0): uint2 info[ncell] = {offset in octets, capacity}, u32 hist[ncell], u32 run_len[nb].
    // info of cell (b, sub) sits at b * nsub + fill_pos(sub): the permutation of the fill rows, so that the 16 rows a
    // k2_partition warp owns are one 128-byte load (in natural order they are 16 sectors: +25 % l1tex wavefronts per tile)
    uint64_t cells0;
    uint64_t windows_est;           // upper estimate of the windows the whole partition will hold (its list capacity)
    __host__ __device__ uint32_t ncell() const { return nb * nsub; }
    __device__ const uint2* cell_info(const uint16_t* ws) const { return reinterpret_cast<const uint2*>(ws + cells0); }
    __device__ uint32_t* cell_hist(uint16_t* ws) const { return reinterpret_cast<uint32_t*>(ws + cells0) + 2 * ncell(); }
    // tiles of bucket b a k2_partition CTA takes per visit (<= kL2Run; shorter for small buckets, so that every CTA still
    // gets its share of the bucket and no (cell, CTA) segment sees much more than the mean)
    __device__ const uint32_t* run_len(const uint16_t* ws) const { return reinterpret_cast<const uint32_t*>(ws + cells0) + 3 * ncell(); }
    // spill area: full table keys (u32) of the entries that found their staging row, the tile's overflow list or their
    // segment full (hot keys: low-complexity reads put thousands of equal windows into one tile); applied with warp-
    // aggregated REDs by k_count_spill after the shared-memory count
    uint64_t spill0;                // u16 offset of the area in the workspace
    uint32_t spill_cap;             // entries
    uint32_t key_lo;                // first key of bucket 0
    int shift;
    __host__ __device__ uint32_t key_of(uint32_t bucket, uint32_t sub, uint32_t low15) const {
        return key_lo + (bucket << shift) + (sub << 16) + low15;
    }
};

constexpr uint32_t kCellFloor = 16;   // entries every segment gets whatever the sample says

// cells of a sample of the chunk's blocks (every `stride`-th block, one thread per sampled block)
template <bool FULL>
__global__ void __launch_bounds__(256)
k_sample_cells(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ valid, uint64_t blk_lo, uint64_t blk_hi, uint64_t stride,
               uint32_t key_lo, uint32_t key_hi, uint16_t* __restrict__ ws, L2Layout Y) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t gb = blk_lo + i * stride;
    BlockWindows b;
    b.m = b.pw = b.w0 = b.w1 = 0;
    if (gb < blk_hi) b = load_block(codes, valid, gb);
    uint32_t* __restrict__ hist = Y.cell_hist(ws);
    for_each_key<FULL>(b, key_lo, key_hi, [&](uint32_t kk) { atomicAdd(hist + ((kk - key_lo) >> 16), 1u); });
}

// one CTA: run lengths, capacities and offsets of all cells from the sampled histogram.
// A CTA of k2_partition receives bucket b in RUNS of run_len[b] tiles, cyclically over the CTAs, so over the whole input a
// (cell, CTA) segment gets the cell's mean share per CTA give or take ONE run.  Capacity of a cell's segments therefore =
// floor + its share of the space that is left + one run's worth of the cell (run_len[b] * 8192 * share inside b).
__global__ void __launch_bounds__(1024) k_plan_cells(uint16_t* __restrict__ ws, L2Layout Y) {
    __shared__ ull s_red[1024];
    __shared__ ull s_scan[1024];
    __shared__ ull s_bsum[kMaxBuckets];
    __shared__ uint32_t s_rl[kMaxBuckets];
    __shared__ ull s_slack;
    const uint32_t tid = threadIdx.x, ncell = Y.ncell();
    uint2* info = const_cast<uint2*>(Y.cell_info(ws));
    uint32_t* rl = const_cast<uint32_t*>(Y.run_len(ws));
    auto slot = [&](uint32_t c) { return (c / Y.nsub) * Y.nsub + Y.fill_pos(c % Y.nsub); };
    const uint32_t* hist = Y.cell_hist(ws);
    if (tid < (uint32_t)kMaxBuckets) s_bsum[tid] = 0;
    __syncthreads();
    ull sum = 0;
    for (uint32_t c = tid; c < ncell; c += 1024) {
        sum += hist[c];
        atomicAdd(&s_bsum[c / Y.nsub], (ull)hist[c]);
    }
    s_red[tid] = sum;
    __syncthreads();
    for (int d = 512; d > 0; d >>= 1) {
        if (tid < (uint32_t)d) s_red[tid] += s_red[tid + d];
        __syncthreads();
    }
    const ull total = s_red[0];
    const ull per_cta = Y.seg_units / Y.n_cta;   // entries a CTA can be given over all cells
    const ull floor_all = (ull)ncell * kCellFloor;
    bool uniform = total < 32ull * ncell || per_cta <= floor_all;
    if (tid == 0) {
        ull slack = 0;
        for (uint32_t bkt = 0; bkt < Y.nb; ++bkt) {
            // tiles the bucket will hold in the end; at least 4 runs per CTA when the bucket is big enough
            const ull tiles = uniform ? ~0ull : (ull)((double)s_bsum[bkt] / (double)total * (double)Y.windows_est / kStepSlots);
            const uint32_t r = (uint32_t)min((ull)kL2Run, max(1ull, tiles / (4ull * Y.n_cta)));
            s_rl[bkt] = r;
            slack += (ull)r * kStepSlots;
        }
        s_slack = slack;
    }
    __syncthreads();
    if (per_cta <= floor_all + s_slack + (per_cta >> 2)) uniform = true;   // no room for the scheme: one capacity, full runs
    if (tid < Y.nb) rl[tid] = uniform ? kL2Run : s_rl[tid];
    const ull avail = uniform ? 0ull : per_cta - floor_all - s_slack;
    const double share_scale = uniform ? 0.0 : (double)avail / (double)total * 0.999;   // 0.999: rounding never hands out more than there is
    const ull clamp = ((1ull << 32) - 8 - kStepSlots) / ((ull)Y.nsub * Y.n_cta);   // a bucket's segments stay below 2^32 u16 units
    // contiguous stretch of cells per thread, so that one scan over the threads' totals gives every cell its offset
    const uint32_t per = (ncell + 1023u) / 1024u;
    const uint32_t c0 = min(ncell, tid * per), c1 = min(ncell, c0 + per);
    ull mine = 0;
    for (uint32_t c = c0; c < c1; ++c) {
        ull w;
        if (uniform) w = Y.C3;
        else {
            const uint32_t bkt = c / Y.nsub;
            const double h = (double)hist[c];   // doubles: 16 K 64-bit divisions in one CTA would be most of this kernel's time
            const double one_run = s_bsum[bkt] ? (double)s_rl[bkt] * kStepSlots * h / (double)s_bsum[bkt] : 0.0;
            w = kCellFloor + (ull)(h * share_scale) + (ull)one_run;
        }
        w = min(w, clamp) & ~7ull;
        info[slot(c)].y = (uint32_t)w;
        mine += w * Y.n_cta / 8;   // octets
    }
    s_scan[tid] = mine;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const ull v = tid >= (uint32_t)d ? s_scan[tid - d] : 0ull;
        __syncthreads();
        s_scan[tid] += v;
        __syncthreads();
    }
    ull acc = s_scan[tid] - mine;
    for (uint32_t c = c0; c < c1; ++c) {   // natural order: cell (b, 0) has the lowest offset of bucket b
        info[slot(c)].x = (uint32_t)acc;
        acc += (ull)info[slot(c)].y * Y.n_cta / 8;
    }
}

template <int LOG2_NSUB>
__global__ void __launch_bounds__(kL2Threads, kL2CtasPerSm)
k2_partition(const uint32_t* __restrict__ ents, PartMeta* __restrict__ meta, int c, uint16_t* __restrict__ ws, L2Layout Y) {
    extern __shared__ uint32_t s_dyn[];
    uint16_t* s_stage = reinterpret_cast<uint16_t*>(s_dyn);  // [nsub][cap] low 15 key bits
    __shared__ uint32_t s_cnt[kMaxSubs];           // entries of the tile per sub-slice (zero between tiles)
    __shared__ uint32_t s_ovl[kL2Ovl];             // (sub << 15) | low key bits of the entries that found their row full
    __shared__ uint32_t s_novl[2];                 // length of s_ovl, by tile parity
    __shared__ uint32_t s_sp2[kMaxSubs];           // entries of the tile per sub-slice that went straight to the spill area (rare)
    __shared__ uint32_t s_tiles[kMaxBuckets], s_runs[kMaxBuckets], s_start[kMaxBuckets], s_runs0[kMaxBuckets], s_rl[kMaxBuckets];  // tile schedule (below)
    __shared__ ull s_reg_n[kMaxBuckets], s_reg_off[kMaxBuckets];
    __shared__ uint32_t s_ovf[kMaxBuckets];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    constexpr uint32_t nsub = 1u << LOG2_NSUB, sub_mask = nsub - 1u;   // == Y.nsub
    constexpr uint32_t cap = (uint32_t)kL2Stage / nsub, cap_shift = 15u - LOG2_NSUB;
    constexpr uint32_t spw = nsub / kL2Warps;      // sub-slices (staging rows) owned by a warp (nsub >= 16)
    if (meta->overflow) return;  // lists incomplete: nothing is applied anywhere
    uint32_t* __restrict__ fill = reinterpret_cast<uint32_t*>(ws) + (size_t)blockIdx.x * Y.nb * nsub;  // this CTA's row
    for (uint32_t i = tid; i < (uint32_t)kMaxSubs; i += kL2Threads) { s_cnt[i] = 0; s_sp2[i] = 0; }
    const uint32_t n_cta = gridDim.x;
    if (tid < (uint32_t)kMaxBuckets) {
        s_ovf[tid] = 0;
        const ull n_reg = tid < Y.nb ? meta->counts[c][tid] : 0ull;
        s_reg_n[tid] = n_reg;
        s_reg_off[tid] = tid < Y.nb ? meta->offsets[c][tid] : 0ull;
        const uint32_t tiles = (uint32_t)((n_reg + kStepSlots - 1) / kStepSlots);
        s_tiles[tid] = tiles;
        const uint32_t rlen = tid < Y.nb ? max(1u, min((uint32_t)kL2Run, __ldg(Y.run_len(ws) + tid))) : (uint32_t)kL2Run;
        s_rl[tid] = rlen;
        s_runs[tid] = (tiles + rlen - 1u) / rlen;
        // runs of this bucket in the earlier chunks, and in chunk 0 (the base spread of the buckets over the CTAs)
        uint32_t before = 0, runs0 = 0;
        if (tid < Y.nb) {
            for (int cc = 0; cc < c; ++cc) {
                const uint32_t rr = (uint32_t)(((meta->counts[cc][tid] + kStepSlots - 1) / kStepSlots + rlen - 1u) / rlen);
                before += rr;
                if (cc == 0) runs0 = rr;
            }
            if (c == 0) runs0 = s_runs[tid];
        }
        s_start[tid] = before;
        s_runs0[tid] = runs0;
    }
    if (tid < 2) s_novl[tid] = 0;
    __syncthreads();
    if (tid == 0) {
        uint32_t acc = 0;
        for (uint32_t b = 0; b < Y.nb; ++b) {
            s_start[b] = (s_start[b] + acc) % n_cta;
            acc += s_runs0[b];
        }
    }
    __syncthreads();
    // Tile schedule.  A RUN is kL2Run consecutive tiles of one bucket region; run r of bucket b belongs to CTA
    // (start[b] + r) mod n_cta, where start[b] continues from chunk to chunk (runs of b in the earlier chunks) on top of
    // chunk 0's global run numbering.  So (1) a CTA appends kL2Run tiles' worth to a segment while its frontier sectors
    // are hot in L2 (with one tile per visit, as a chunked build would give, every append re-fetches a partial sector),
    // (2) every (bucket, CTA) pair receives the same share of the bucket whatever the chunking (the segments have a fixed
    // capacity), (3) the 64 windows of a launch tile the ring of CTAs evenly.
    uint32_t gb = 0, gr = 0, gt = 0;  // generator state: bucket, run (of this CTA) in it, tile in the run
    auto seek = [&]() {               // first run of this CTA in bucket gb or a later one
        for (; gb < Y.nb; ++gb) {
            gr = (blockIdx.x + n_cta - s_start[gb]) % n_cta;
            if (gr < s_runs[gb]) { gt = 0; return true; }
        }
        return false;
    };
    auto advance = [&]() {
        if (++gt < s_rl[gb] && gr * s_rl[gb] + gt < s_tiles[gb]) return true;
        gt = 0;
        gr += n_cta;
        if (gr < s_runs[gb]) return true;
        ++gb;
        return seek();
    };
    auto fetch = [&](uint32_t (&e)[kL2PerThread], uint32_t& b, uint32_t& n_tile) {  // the generator's current tile
        b = gb;
        const uint32_t t = gr * s_rl[b] + gt;
        n_tile = (uint32_t)min((ull)kStepSlots, s_reg_n[b] - (ull)t * kStepSlots);
        const uint32_t* __restrict__ src = ents + s_reg_off[b] + (ull)t * kStepSlots;
        if (n_tile == (uint32_t)kStepSlots) {
#pragma unroll
            for (int j = 0; j < kL2PerThread; ++j) e[j] = __ldcs(src + j * kL2Threads + tid);
        } else {
#pragma unroll
            for (int j = 0; j < kL2PerThread; ++j) e[j] = (j * kL2Threads + tid < n_tile) ? __ldcs(src + j * kL2Threads + tid) : 0u;
        }
    };
    const uint32_t stage_mask = (nsub << kSubBits) - 1u;  // sub-slice index + low key bits, as they sit in the entry
    uint32_t* __restrict__ spill_keys = reinterpret_cast<uint32_t*>(ws + Y.spill0);
    const uint2* __restrict__ c_info = Y.cell_info(ws);
    // n keys of this warp into the spill area: one reservation per call (warp-aggregated), keys produced by key_at(i).
    // When the area is full the remaining keys are dropped and the bucket is flagged: k_count_keys then counts the whole
    // bucket from the first-level list and both other count kernels skip it.
    auto spill_warp = [&](uint32_t n, uint32_t bucket, auto key_at) {   // called by all lanes of a warp with equal arguments
        ull base = 0;
        if (lane == 0) base = atomicAdd(&meta->spill_n, (ull)n);
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (base + n > (ull)Y.spill_cap) {
            if (lane == 0) { s_ovf[bucket] = 1u; meta->spill_dropped = 1ull; }
            if (base >= (ull)Y.spill_cap) return;
            n = (uint32_t)((ull)Y.spill_cap - base);
        }
        for (uint32_t i = lane; i < n; i += 32) spill_keys[base + i] = key_at(i);
    };
    // lane j < spw of a warp looks after row / fill counter j of the warp's sub-slices.  The warp owns sub-slices
    // warp + 16 j — measured 2 ms faster per step than the blocked ownership 16 warp + j
    const uint32_t my_sub = warp + (uint32_t)kL2Warps * lane;
    const uint32_t my_pos = Y.fill_pos(my_sub);   // its counter in the fill row
    constexpr uint32_t cm = cap - 1u;
    // Staging rows are rings ALIGNED WITH THEIR DESTINATION: the entry bound for list position d (u16 units from the
    // bucket's first segment) is staged in slot (d + 8 sub) mod cap of row sub.  Segments start on 16-byte boundaries and
    // cap is a multiple of 8, so every aligned 8-entry word of a segment is one aligned 16-byte word of the row and the
    // sweep copies rows as uint4.  The rank-0 slot moves with the row's fill, which spreads rows over the banks as the
    // former fixed rotation by 2 sub did; + 8 sub keeps rows apart when their fills agree modulo 64 (first tiles).
    // s_cnt[sub] = (slot of rank 0) << 16 | entries ranked so far: the returning atomic of the place phase yields both.
    uint32_t f_my = 0, cap_my = 0, rel_my = 0, boff0 = 0;   // the lane's row in the current bucket (b_cur)
    auto rank0 = [&]() { return ((rel_my + f_my + 8u * my_sub) & cm) << 16; };
    uint32_t e[kL2PerThread];
    uint32_t n_cur = 0, n_next = 0, b_cur = 0, b_next = 0;
    bool have = seek();
    if (have) {
        fetch(e, b_cur, n_cur);
        const uint32_t cell0 = b_cur * nsub;
        const uint2 ci = lane < spw ? __ldg(c_info + cell0 + my_pos) : make_uint2(0u, 0u);
        boff0 = __ldg(&c_info[cell0].x);
        f_my = lane < spw ? fill[(size_t)cell0 + my_pos] : 0u;
        cap_my = ci.y;
        rel_my = (ci.x - boff0) * 8u + blockIdx.x * cap_my;
        if (lane < spw) s_cnt[my_sub] = rank0();
    }
    __syncthreads();
    for (uint32_t it = 0; have; ++it) {
        const uint32_t par = it & 1u;
        uint32_t* frow = fill + (size_t)b_cur * nsub;
        // place: one returning atomic + one predicated 2-byte store per entry (the staged half-word keeps entry bit 15, a
        // sub-slice bit: k_count_smem masks it off); entries that find their row full are remembered in a bit mask and go
        // to the overflow list afterwards
        uint32_t spill = 0;
        auto place = [&](int j) {
            const uint32_t sub = (e[j] >> kSubBits) & sub_mask;
            const uint32_t r = atomicAdd(&s_cnt[sub], 1u);
            if ((r & 0xFFFFu) < cap) s_stage[(sub << cap_shift) + ((r + (r >> 16)) & cm)] = (uint16_t)e[j];
            else spill |= 1u << j;
        };
        if (n_cur == (uint32_t)kStepSlots) {
#pragma unroll
            for (int j = 0; j < kL2PerThread; ++j) place(j);
        } else {
#pragma unroll
            for (int j = 0; j < kL2PerThread; ++j)
                if (j * kL2Threads + tid < n_cur) place(j);
        }
        uint32_t spill2 = 0;   // entries that missed the overflow list as well: straight to the spill area
        if (spill) {   // one reservation per thread (the list counter is a single address: hot cells would serialise on it)
            uint32_t o = atomicAdd(&s_novl[par], (uint32_t)__popc(spill));
#pragma unroll
            for (int j = 0; j < kL2PerThread; ++j) {
                if ((spill >> j) & 1u) {
                    if (o < (uint32_t)kL2Ovl) s_ovl[o] = e[j] & stage_mask;
                    else spill2 |= 1u << j;
                    ++o;
                }
            }
        }
        if (__any_sync(0xFFFFFFFFu, spill2 != 0u)) {   // rare: a hot key filled row + overflow list of this tile
            const uint32_t mine = (uint32_t)__popc(spill2);
            uint32_t incl = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, incl, d);
                if (lane >= (uint32_t)d) incl += y;
            }
            const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
            ull base = 0;
            if (lane == 0) base = atomicAdd(&meta->spill_n, (ull)total);
            base = __shfl_sync(0xFFFFFFFFu, base, 0) + (incl - mine);
            if (base + mine > (ull)Y.spill_cap) { s_ovf[b_cur] = 1u; meta->spill_dropped = 1ull; }
#pragma unroll
            for (int j = 0; j < kL2PerThread; ++j) {
                if ((spill2 >> j) & 1u) {
                    const uint32_t sub = (e[j] >> kSubBits) & sub_mask;
                    if (base < (ull)Y.spill_cap) spill_keys[base] = Y.key_of(b_cur, sub, e[j] & 0x7FFFu);
                    ++base;
                    atomicAdd(&s_sp2[sub], 1u);   // the row's list entry count excludes these
                }
            }
        }
        // the next tile's entries travel during the sweep, into the registers the placed ones just left (a fetch issued
        // BEFORE the place phase would share its scoreboard with the loads the place phase waits for, and stall it)
        have = advance();
        if (have) fetch(e, b_next, n_next);
        __syncthreads();
        // the next tile's bucket when it is another one: where the lane's row goes there (read now, used after the sweep)
        const bool switch_b = have && b_next != b_cur;
        uint2 ci_nx = make_uint2(0u, 0u);
        uint32_t boff_nx = 0, f_nx = 0;
        if (switch_b) {
            const uint32_t cell0 = b_next * nsub;
            if (lane < spw) { ci_nx = __ldg(c_info + cell0 + my_pos); f_nx = fill[(size_t)cell0 + my_pos]; }
            boff_nx = __ldg(&c_info[cell0].x);
        }
        // sweep: the rows of this warp's sub-slices go to this CTA's segments.  The owning lane works out where its row
        // goes (a 32-bit position inside the bucket's span) and how much of it; the copy is then one 16-byte word per
        // lane, eight lanes (one 128-byte shared-memory wavefront) per row, plus the entries in front of the row's first
        // aligned word (the expected row holds 8192 / nsub = cap / 4 entries)
        const uint32_t novl_raw = s_novl[par];
        uint32_t n_my = lane < spw ? s_cnt[my_sub] & 0xFFFFu : 0u;   // entries of the tile ranked into this row ...
        if (novl_raw > (uint32_t)kL2Ovl && lane < spw) {   // ... minus those that left through the spill area (warp-uniform test)
            const uint32_t gone = s_sp2[my_sub];
            if (gone) { n_my -= gone; s_sp2[my_sub] = 0; }
        }
        const bool ok_my = f_my + n_my <= cap_my;   // a full segment takes nothing more: the row goes to the spill area
        const uint32_t off_my = rel_my + f_my;      // list position of the row's rank 0 (< 2^32: k_plan_cells clamps the capacities)
        uint32_t ns_my = 0;
        if (lane < spw && n_my && ok_my) {
            frow[my_pos] = f_my + n_my;
            ns_my = min(n_my, cap);
        }
        if (tid == 0) s_novl[par ^ 1u] = 0;  // the next tile's list; last read before the previous tile's closing barrier
        // rows whose segment is full (a hot sub-slice: more than C3 entries from this CTA): staged part and overflow-list
        // part go to the spill area
        const uint32_t full_rows = __ballot_sync(0xFFFFFFFFu, lane < spw && n_my != 0u && !ok_my);
        for (uint32_t rest = full_rows; rest; rest &= rest - 1u) {
            const uint32_t jj = (uint32_t)__ffs(rest) - 1u;
            const uint32_t n = __shfl_sync(0xFFFFFFFFu, n_my, jj), off = __shfl_sync(0xFFFFFFFFu, off_my, jj);
            const uint32_t sub = warp + (uint32_t)kL2Warps * jj;
            const uint16_t* src = s_stage + (sub << cap_shift);
            const uint32_t bkt = b_cur;
            spill_warp(min(n, cap), bkt, [&](uint32_t i) { return Y.key_of(bkt, sub, src[(off + i + 8u * sub) & cm] & 0x7FFFu); });
            if (n > cap) {
                const uint32_t novl = min(novl_raw, (uint32_t)kL2Ovl);
                for (uint32_t i0 = 0; i0 < novl; i0 += 32) {
                    const uint32_t i = i0 + lane;
                    const uint32_t r = i < novl ? s_ovl[i] : 0xFFFFFFFFu;
                    const bool mine = i < novl && (r >> kSubBits) == sub;
                    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, mine);
                    if (!bal) continue;
                    const uint32_t cnt = (uint32_t)__popc(bal), pos = (uint32_t)__popc(bal & ((1u << lane) - 1u));
                    ull base = 0;
                    if (lane == 0) base = atomicAdd(&meta->spill_n, (ull)cnt);
                    base = __shfl_sync(0xFFFFFFFFu, base, 0);
                    if (base + cnt > (ull)Y.spill_cap && lane == 0) { s_ovf[bkt] = 1u; meta->spill_dropped = 1ull; }
                    if (mine && base + pos < (ull)Y.spill_cap) spill_keys[base + pos] = Y.key_of(bkt, sub, r & 0x7FFFu);
                }
            }
        }
        uint16_t* __restrict__ lists = ws + Y.seg0 + 8ull * boff0;
        // Row jj = g + lane / 8 of the warp, lane q = lane % 8 of its group.  Head: list positions [off, next multiple of
        // 8), entry by entry.  Then the aligned words from there up to the word holding the last entry, whole: the entries
        // of that word past the row are past the segment's fill (k_count_smem reads only up to the fill, and the next tile
        // of this row overwrites them), and the word ends inside the segment (segments are whole words).  One word per
        // lane covers rows of up to 64 entries; the groups are independent, so their loads and stores overlap.  Longer
        // rows (the mean row is 8192 / nsub entries: rare from 256 sub-slices per bucket up) take more words in a second loop.
        const uint32_t q = lane & 7u;
        auto row_of = [&](uint32_t g, uint32_t& ns, uint32_t& off, uint32_t& sub) {
            const uint32_t jj = g + (lane >> 3);
            ns = __shfl_sync(0xFFFFFFFFu, ns_my, jj & 31u);
            off = __shfl_sync(0xFFFFFFFFu, off_my, jj & 31u);
            if (jj >= spw) ns = 0;
            sub = warp + (uint32_t)kL2Warps * jj;
        };
        auto copy_word = [&](uint32_t sub, uint32_t dw) {   // list word at dw (a multiple of 8) from its ring word
            const uint16_t* src = s_stage + (sub << cap_shift);
            *reinterpret_cast<uint4*>(lists + dw) = *reinterpret_cast<const uint4*>(src + ((dw + 8u * sub) & cm));
        };
        bool longer = false;
#pragma unroll
        for (uint32_t g = 0; g < spw; g += 4) {
            uint32_t ns, off, sub;
            row_of(g, ns, off, sub);
            const uint32_t w0 = (off + 7u) >> 3, w1 = (off + ns + 7u) >> 3;   // first whole word, end of the row's words
            const uint32_t d = (off & ~7u) + q;
            if (d >= off && d < off + ns && d < w0 * 8u) lists[d] = s_stage[(sub << cap_shift) + ((d + 8u * sub) & cm)];
            const uint32_t nw = (ns && w1 > w0) ? w1 - w0 : 0u;
            if (q < nw) copy_word(sub, (w0 + q) * 8u);
            longer |= nw > 8u;
        }
        if (__any_sync(0xFFFFFFFFu, longer)) {
#pragma unroll 1
            for (uint32_t g = 0; g < spw; g += 4) {
                uint32_t ns, off, sub;
                row_of(g, ns, off, sub);
                const uint32_t w0 = (off + 7u) >> 3, w1 = (off + ns + 7u) >> 3;
                const uint32_t nw = (ns && w1 > w0) ? w1 - w0 : 0u;
                for (uint32_t i = q + 8u; i < nw; i += 8) copy_word(sub, (w0 + i) * 8u);
            }
        }
        const uint32_t ovl_rows = __ballot_sync(0xFFFFFFFFu, ok_my && n_my > cap);
        if (ovl_rows) __syncwarp();   // the overflow-list entries land after (and over the tail of) the row's last word
        for (uint32_t rest = ovl_rows; rest; rest &= rest - 1u) {  // rare: rows that spilled into the overflow list
            const uint32_t jj = (uint32_t)__ffs(rest) - 1u;
            const uint32_t n = __shfl_sync(0xFFFFFFFFu, n_my, jj);
            const uint32_t sub = warp + (uint32_t)kL2Warps * jj;
            uint16_t* __restrict__ dst = lists + __shfl_sync(0xFFFFFFFFu, off_my, jj);
            const uint32_t novl = min(novl_raw, (uint32_t)kL2Ovl);
            uint32_t base = cap;
            for (uint32_t i0 = 0; i0 < novl; i0 += 32) {
                const uint32_t i = i0 + lane;
                const uint32_t r = i < novl ? s_ovl[i] : 0xFFFFFFFFu;
                const bool mine = i < novl && (r >> kSubBits) == sub;
                const uint32_t bal = __ballot_sync(0xFFFFFFFFu, mine);
                const uint32_t at = base + (uint32_t)__popc(bal & ((1u << lane) - 1u));
                if (mine && at < n) dst[at] = (uint16_t)(r & 0x7FFFu);
                base += (uint32_t)__popc(bal);
            }
        }
        // the next tile's rows: rank counters reset, rank-0 slots where its entries will go
        if (ok_my) f_my += n_my;
        if (switch_b) {
            boff0 = boff_nx;
            f_my = f_nx;
            cap_my = ci_nx.y;
            rel_my = (ci_nx.x - boff0) * 8u + blockIdx.x * cap_my;
        }
        if (have && lane < spw) s_cnt[my_sub] = rank0();
        __syncthreads();
        n_cur = n_next;
        b_cur = b_next;
    }
    __syncthreads();
    if (tid < Y.nb && s_ovf[tid]) meta->overflow2[tid] = 1u;
}

// the spill area of k2_partition: full table keys of hot rows -> warp-aggregated REDs, after the shared-memory count has
// written / added its slices.  Keys of buckets [bucket_lo, bucket_hi) only; buckets counted by k_count_keys are skipped.
__global__ void __launch_bounds__(256)
k_count_spill(const uint16_t* __restrict__ ws, const PartMeta* __restrict__ meta, L2Layout Y, int bucket_lo, int bucket_hi,
              uint32_t* __restrict__ table) {
    if (meta->overflow) return;
    const uint64_t n = min(meta->spill_n, (ull)Y.spill_cap);
    const uint32_t* __restrict__ spill = reinterpret_cast<const uint32_t*>(ws + Y.spill0);
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i0 = ((uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)); i0 < n; i0 += stride) {
        const uint64_t i = i0 + (threadIdx.x & 31u);
        bool act = i < n;
        uint32_t key = 0;
        if (act) {
            key = __ldcs(spill + i);
            const int b = (int)((key - Y.key_lo) >> Y.shift);
            act = b >= bucket_lo && b < bucket_hi && !meta->overflow2[b];
        }
        red_aggregated(table, key, act);
    }
}

// one CTA per sub-slice: its segments -> 2^15 counters in shared memory -> added to the table slice (128 KB, contiguous)
// OVERWRITE: the slice is WRITTEN (counts, or zeros for a bucket that falls back to k_count_keys) instead of added to, so
// the caller needs no memset of the table and the slice is not read: -4 GiB of memset writes and -2 GiB of reads per step.
template <bool OVERWRITE>
__global__ void __launch_bounds__(1024)
k_count_smem(const uint16_t* __restrict__ ws, const PartMeta* __restrict__ meta, int bucket0, L2Layout Y, uint32_t bucket_base0, int shift,
             uint32_t* __restrict__ table) {
    extern __shared__ uint32_t s_tab[];  // 2^15
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5, sub = blockIdx.x;
    const int bucket = bucket0 + (int)blockIdx.y;   // one launch may cover several buckets (gridDim.y): no 1.7-wave tail per bucket
    const uint32_t bucket_base = bucket_base0 + ((uint32_t)blockIdx.y << shift);
    if (meta->overflow) return;
    if (meta->overflow2[bucket]) {
        if (OVERWRITE) {  // k_count_keys adds this bucket's windows to a zeroed slice
            uint4* z4 = reinterpret_cast<uint4*>(table + bucket_base + (sub << 16));
            for (uint32_t i = tid; i < (1u << kSubBits) / 4; i += 1024) z4[i] = make_uint4(0, 0, 0, 0);
        }
        return;
    }
    const uint32_t* __restrict__ fill = reinterpret_cast<const uint32_t*>(ws) + (size_t)bucket * Y.nsub + Y.fill_pos(sub);  // + cta * nb * nsub
    const size_t fill_stride = (size_t)Y.nb * Y.nsub;
    const uint2 ci = __ldg(Y.cell_info(ws) + (uint32_t)bucket * Y.nsub + Y.fill_pos(sub));
    const uint32_t seg_cap = ci.y;
    const uint16_t* __restrict__ lists = ws + Y.seg0 + 8ull * ci.x;   // this cell's n_cta segments
    uint4* tab4 = reinterpret_cast<uint4*>(s_tab);
    for (uint32_t i = tid; i < (1u << kSubBits) / 4; i += 1024) tab4[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    auto bump8 = [&](const uint4& v) {  // list entries are 16 bits wide; bit 15 is not part of the key inside the sub-slice
        atomicAdd(&s_tab[v.x & 0x7FFFu], 1u); atomicAdd(&s_tab[(v.x >> 16) & 0x7FFFu], 1u);
        atomicAdd(&s_tab[v.y & 0x7FFFu], 1u); atomicAdd(&s_tab[(v.y >> 16) & 0x7FFFu], 1u);
        atomicAdd(&s_tab[v.z & 0x7FFFu], 1u); atomicAdd(&s_tab[(v.z >> 16) & 0x7FFFu], 1u);
        atomicAdd(&s_tab[v.w & 0x7FFFu], 1u); atomicAdd(&s_tab[(v.w >> 16) & 0x7FFFu], 1u);
    };
    // a warp per segment (a few KB each), 16 B vectors.  The lengths of the warp's segments are fetched in one go and
    // the first four vectors of the next segment travel while the current one is counted.
    const uint32_t my_cta = warp + 32u * lane;                     // lane l holds the length of the warp's l-th segment
    const uint32_t my_len = my_cta < Y.n_cta ? __ldg(fill + my_cta * fill_stride) : 0u;
    const uint32_t n_seg = (Y.n_cta > warp) ? (Y.n_cta - warp + 31u) / 32u : 0u;   // segments of this warp (n_cta <= 1024)
    bool any = __any_sync(0xFFFFFFFFu, my_len != 0u);
    auto seg_ptr = [&](uint32_t k) { return lists + (size_t)(warp + 32u * k) * seg_cap; };
    auto fetch4 = [&](uint32_t k, uint32_t n, uint4* v) {
        const uint4* __restrict__ src4 = reinterpret_cast<const uint4*>(seg_ptr(k));
        const uint32_t n8 = n / 8;
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = (lane + 32u * u < n8) ? __ldcs(src4 + lane + 32u * u) : make_uint4(0, 0, 0, 0);
    };
    const uint32_t rounds = min(n_seg, 32u);
    uint4 cur[4], nxt[4];
    uint32_t n = rounds ? __shfl_sync(0xFFFFFFFFu, my_len, 0) : 0u;
    if (rounds) fetch4(0, n, cur);
    for (uint32_t k = 0; k < rounds; ++k) {
        const uint32_t n_next = (k + 1 < rounds) ? __shfl_sync(0xFFFFFFFFu, my_len, (k + 1) & 31u) : 0u;
        if (k + 1 < rounds) fetch4(k + 1, n_next, nxt);
        const uint32_t n8 = n / 8;
        const uint16_t* __restrict__ src = seg_ptr(k);
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (lane + 32u * u < n8) bump8(cur[u]);
        const uint4* __restrict__ src4 = reinterpret_cast<const uint4*>(src);
        for (uint32_t i = lane + 128u; i < n8; i += 32) bump8(__ldcs(src4 + i));      // long segments: the rest
        for (uint32_t i = n8 * 8 + lane; i < n; i += 32) atomicAdd(&s_tab[src[i] & 0x7FFFu], 1u);
#pragma unroll
        for (int u = 0; u < 4; ++u) cur[u] = nxt[u];
        n = n_next;
    }
    uint4* slice4 = reinterpret_cast<uint4*>(table + bucket_base + (sub << 16));
    if (OVERWRITE) {
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 8; ++u) slice4[tid + 1024 * u] = tab4[tid + 1024 * u];
        return;
    }
    if (!__syncthreads_or(any)) return;  // empty sub-slice: the table slice stays as it is
    uint4 t4[8];  // 8192 uint4 per slice, eight per thread: all loads first
#pragma unroll
    for (int u = 0; u < 8; ++u) t4[u] = slice4[tid + 1024 * u];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const uint4 a = tab4[tid + 1024 * u];
        t4[u].x += a.x; t4[u].y += a.y; t4[u].z += a.z; t4[u].w += a.w;
        slice4[tid + 1024 * u] = t4[u];
    }
}

// entries of one bucket: hist[read][bin(table[key])] += 1.  A warp task is kTaskRuns consecutive runs of one chunk —
// one contiguous span of the bucket's region — streamed 128 entries per step (four gathers in flight per lane; the
// kernel is bound by the latency of the dependent stream-load -> gather chain otherwise).  The run boundaries and
// first-read indices of the span sit in shared memory; each lane walks them monotonically to recover the read of
// its entries.  Equal (read, bin) entries of a warp share one RED.  Tasks are numbered across all chunks
// (L.task0 = prefix of tasks per chunk) so small chunks still fill the machine.
constexpr uint32_t kTaskRuns = 16;
constexpr int kSearchUnroll = 8;   // gathers in flight per lane in the walk's full steps: 8 (22.3 ms at config #2) beats 4 (23.7 ms)

// The walk over the entries of one bucket, shared by the single-setting search, the multi-setting one and the multi-table
// one: load(e) gathers what entry e needs from the table(s) (a count, or one count per table); put(hbase, cnt,
// act, lane, seek, row) bins the gathered `cnt` of an entry and adds it to the histogram row row() (relative to
// hbase, whose rows are `pitch` words apart) after seek(); both only where act (the lane has an entry).  put is called by
// every lane of the warp together, so it may use warp-wide primitives.  One launch may cover several buckets (gridDim.y):
// CTAs are dispatched x-fastest, so the buckets are still worked on one after the other (their slices take turns in L2)
// but the tail of one overlaps the head of the next.
template <class Load, class Put>
__device__ __forceinline__ void search_keys_body(const uint32_t* __restrict__ ents, const PartMeta* __restrict__ meta, int bucket,
                                                 int n_chunks, const ChunkList& L, const StepTables& T, int shift,
                                                 uint32_t* __restrict__ hist, uint32_t pitch, uint32_t (*s_bnd)[kTaskRuns + 1],
                                                 uint32_t (*s_r0)[kTaskRuns], Load load, Put put) {
    using Count = decltype(load(0u));
    const uint32_t lane = threadIdx.x & 31u, wl = threadIdx.x >> 5;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t* __restrict__ off_row = T.off + (size_t)bucket * T.cap;
    uint32_t* bnd = s_bnd[wl];
    uint32_t* r0 = s_r0[wl];
    const uint32_t n_tasks = L.task0[n_chunks];
    const int rsh = shift - 1;
    int c = 0;
    for (uint32_t task = warp; task < n_tasks; task += n_warps) {
        while (task >= L.task0[c + 1]) ++c;  // tasks ascend: the chunk index only moves forward
        const uint32_t s0 = L.step0[c], ns = L.nsteps[c];
        const uint32_t sb = (task - L.task0[c]) * kTaskRuns;
        const uint32_t* __restrict__ region = ents + meta->offsets[c][bucket];
        __syncwarp();
        if (lane <= kTaskRuns) bnd[lane] = __ldg(off_row + s0 + min(sb + lane, ns));  // off_row[s0 + ns] is the terminal offset
        const uint32_t my_r0 = __ldg(T.rid0 + s0 + min(sb + min(lane, kTaskRuns - 1u), ns - 1u));
        const uint32_t rbase = __shfl_sync(0xFFFFFFFFu, my_r0, 0);
        if (lane < kTaskRuns) r0[lane] = my_r0 - rbase;
        __syncwarp();
        const uint32_t span_beg = bnd[0], span_end = bnd[kTaskRuns];
        uint32_t* __restrict__ hbase = hist + (size_t)rbase * pitch;
        uint32_t cur = 0, nxt = bnd[1], rr = 0;  // run of this lane's current entry, its end, its relative read base
        auto emit = [&](uint32_t e, const Count& cnt, uint32_t i, bool act) {
            // seek(): move to the run of entry i (active lanes only); row(): then the entry's read, relative to hbase
            auto seek = [&]() { while (i >= nxt) { ++cur; nxt = bnd[cur + 1]; rr = r0[cur]; } };  // runs may be empty; i < bnd[kTaskRuns] bounds cur
            auto row = [&]() { return rr + (e >> rsh); };
            put(hbase, cnt, act, lane, seek, row);
        };
        uint32_t i0 = span_beg;
        constexpr int U = kSearchUnroll;
        constexpr uint32_t kStep = 32u * U;
        if (i0 + kStep <= span_end) {  // full steps: no predicates; the entries of step t+1 are fetched while step t gathers
            uint32_t e[U], nx[U];
            Count cn[U];
            const uint32_t* src = region + i0 + lane;
#pragma unroll
            for (int u = 0; u < U; ++u) e[u] = __ldcs(src + 32 * u);
            for (;;) {
#pragma unroll
                for (int u = 0; u < U; ++u) cn[u] = load(e[u]);
                const bool more = i0 + 2u * kStep <= span_end;  // warp-uniform
                if (more) {
                    const uint32_t* nsrc = region + i0 + kStep + lane;
#pragma unroll
                    for (int u = 0; u < U; ++u) nx[u] = __ldcs(nsrc + 32 * u);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) emit(e[u], cn[u], i0 + lane + 32u * u, true);
                i0 += kStep;
                if (!more) break;
#pragma unroll
                for (int u = 0; u < U; ++u) e[u] = nx[u];
            }
        }
        for (; i0 + 128u <= span_end; i0 += 128u) {  // full 128-entry steps that are left
            const uint32_t* src = region + i0 + lane;
            const uint32_t e0 = __ldcs(src), e1 = __ldcs(src + 32), e2 = __ldcs(src + 64), e3 = __ldcs(src + 96);
            const Count c0 = load(e0), c1 = load(e1), c2 = load(e2), c3 = load(e3);
            emit(e0, c0, i0 + lane, true);
            emit(e1, c1, i0 + lane + 32u, true);
            emit(e2, c2, i0 + lane + 64u, true);
            emit(e3, c3, i0 + lane + 96u, true);
        }
        if (i0 < span_end) {  // tail of the span
            uint32_t e[4];
            Count cnt[4];
            bool act[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t i = i0 + 32u * u + lane;
                act[u] = i < span_end;
                e[u] = act[u] ? __ldcs(region + i) : 0u;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) cnt[u] = act[u] ? load(e[u]) : Count{};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (i0 + 32u * u >= span_end) break;  // warp-uniform
                emit(e[u], cnt[u], i0 + 32u * u + lane, act[u]);
            }
        }
    }
}

// load functor of the walk for the full-layout table: the count of the entry's key
__device__ __forceinline__ auto table_load(const uint32_t* __restrict__ table, uint32_t bucket_base, uint32_t hi_mask2) {
    return [=](uint32_t e) { return table[entry_key(e, bucket_base, hi_mask2)]; };
}

// hist[read][bin(table[key])] += 1 for one (bin size, bin count): rows of B bins
__global__ void __launch_bounds__(256)
k_search_keys(const uint32_t* __restrict__ ents, const PartMeta* __restrict__ meta, int bucket0, int n_chunks, ChunkList L,
              StepTables T, uint32_t bucket_base0, uint32_t hi_mask2, int shift, const uint32_t* __restrict__ table, uint32_t S32,
              uint64_t magic, uint32_t B, uint32_t* __restrict__ hist) {
    const int bucket = bucket0 + (int)blockIdx.y;
    const uint32_t bucket_base = bucket_base0 + ((uint32_t)blockIdx.y << shift);
    __shared__ uint32_t s_bnd[8][kTaskRuns + 1];  // per warp: start of each run of the span, [kTaskRuns] = end of the span
    __shared__ uint32_t s_r0[8][kTaskRuns];       // per warp: read index of each run's step relative to the span's first
    if (meta->overflow) return;
    search_keys_body(ents, meta, bucket, n_chunks, L, T, shift, hist, B, s_bnd, s_r0, table_load(table, bucket_base, hi_mask2),
                              [&](uint32_t* hbase, uint32_t cnt, bool act, uint32_t lane, auto seek, auto row) {
                                  uint32_t cell = 0xFFFFFFFFu;
                                  if (act) {
                                      seek();
                                      const uint32_t bin = coverage_bin(cnt, S32, magic, B);
                                      cell = row() * B + bin;
                                  }
                                  const uint32_t peers = __match_any_sync(0xFFFFFFFFu, cell);
                                  if (act && (uint32_t)__ffs(peers) - 1u == lane) atomicAdd(hbase + cell, (uint32_t)__popc(peers));
                              });
}

// Several (bin size, bin count) settings in one pass: the count gathered for a window is binned once per setting, into
// rows of W = sum of B_m words that hold setting 0's bins, then setting 1's, ...  The gather (the cost of the search)
// happens once; each further setting adds one bin computation, one __match_any_sync and the REDs of its cells.
struct CovSettings {
    uint64_t magic[LRB_MAX_COV_SETTINGS];
    uint32_t S32[LRB_MAX_COV_SETTINGS], B[LRB_MAX_COV_SETTINGS], off[LRB_MAX_COV_SETTINGS];
    uint32_t n, W;
};

__global__ void __launch_bounds__(256)
k_search_settings(const uint32_t* __restrict__ ents, const PartMeta* __restrict__ meta, int bucket0, int n_chunks, ChunkList L,
                  StepTables T, uint32_t bucket_base0, uint32_t hi_mask2, int shift, const uint32_t* __restrict__ table,
                  const __grid_constant__ CovSettings C, uint32_t* __restrict__ hist) {
    const int bucket = bucket0 + (int)blockIdx.y;
    const uint32_t bucket_base = bucket_base0 + ((uint32_t)blockIdx.y << shift);
    __shared__ uint32_t s_bnd[8][kTaskRuns + 1];
    __shared__ uint32_t s_r0[8][kTaskRuns];
    if (meta->overflow) return;
    search_keys_body(ents, meta, bucket, n_chunks, L, T, shift, hist, C.W, s_bnd, s_r0, table_load(table, bucket_base, hi_mask2),
                           [&](uint32_t* hbase, uint32_t cnt, bool act, uint32_t lane, auto seek, auto row) {
                               uint32_t base = 0;
                               if (act) {
                                   seek();
                                   base = row() * C.W;
                               }
                               for (uint32_t m = 0; m < C.n; ++m) {
                                   uint32_t cell = 0xFFFFFFFFu;
                                   if (act) cell = base + C.off[m] + coverage_bin(cnt, C.S32[m], C.magic[m], C.B[m]);
                                   const uint32_t peers = __match_any_sync(0xFFFFFFFFu, cell);
                                   if (act && (uint32_t)__ffs(peers) - 1u == lane) atomicAdd(hbase + cell, (uint32_t)__popc(peers));
                               }
                           });
}

// Several sample tables, one walk over the lists per table.  A sample table is held compact (lrb_dev_table_compact): only
// its bit-15-clear keys, entry i = T[((i >> 15) << 16) | (i & 0x7FFF)].  A list entry keeps its key inside the bucket with
// bit 15 dropped in its low shift - 1 bits, so the entry's compact index is (bucket_base >> 1) | (e & (2^(shift-1) - 1))
// and a bucket's slice of a compact table is one contiguous 2^(shift-1)-entry range.  k_search_samples gathers each
// entry's count from one table and bins it with that table's setting into that table's column block.  Walking two tables
// at once saves one read of the lists per pair but measured 1.28-1.30x slower on config #2 (DESIGN.md section 4).
// The fields sit at the offsets of the former two-table layout (the pad words): packed back to back, nvcc schedules
// k_search_samples differently and it measured 0.5 % slower (22.36 against 22.23 ms over the 64 buckets of config #2,
// NVIDIA B200 at a 1000 W limit).
struct SampleGroup {
    const uint32_t* table;     // compact table
    const uint32_t* pad0;
    uint64_t magic, pad1;
    uint32_t S32, pad2, B, pad3, off, pad4;
    uint32_t W;                // row pitch: the bins of every table of the call
};

__global__ void __launch_bounds__(256)
k_search_samples(const uint32_t* __restrict__ ents, const PartMeta* __restrict__ meta, int bucket0, int n_chunks, ChunkList L,
                 StepTables T, uint32_t cbase0, int shift, const __grid_constant__ SampleGroup S, uint32_t* __restrict__ hist) {
    const int bucket = bucket0 + (int)blockIdx.y;
    const uint32_t cbase = cbase0 + ((uint32_t)blockIdx.y << (shift - 1));
    const uint32_t emask = (1u << (shift - 1)) - 1u;
    __shared__ uint32_t s_bnd[8][kTaskRuns + 1];
    __shared__ uint32_t s_r0[8][kTaskRuns];
    if (meta->overflow) return;
    const uint32_t* slice = S.table + cbase;  // the bucket's slice of the table
    search_keys_body(ents, meta, bucket, n_chunks, L, T, shift, hist, S.W, s_bnd, s_r0,
                     [&](uint32_t e) { return __ldg(slice + (e & emask)); },
                     [&](uint32_t* hbase, uint32_t cnt, bool act, uint32_t lane, auto seek, auto row) {
                         uint32_t base = 0;
                         if (act) {
                             seek();
                             base = row() * S.W;
                         }
                         uint32_t cell = 0xFFFFFFFFu;
                         if (act) cell = base + S.off + coverage_bin(cnt, S.S32, S.magic, S.B);
                         const uint32_t peers = __match_any_sync(0xFFFFFFFFu, cell);
                         if (act && (uint32_t)__ffs(peers) - 1u == lane) atomicAdd(hbase + cell, (uint32_t)__popc(peers));
                     });
}

// Bins given by count edges t_0 < ... < t_{n-1} (t_0 >= 2, checked on the host): a count c goes to bin #{i : t_i <= c},
// rows of B = n + 1 bins.  The edges reach the kernel by value (16 380 bytes at most, within the parameter limit) and
// are copied once per CTA into shared memory, padded to P - 1 words (P = the least power of two >= B) with 0xFFFFFFFF.
// The bin is then found by log2(P) warp-uniform halving steps, each one LDS; a padding word compares <= c only when
// c = 0xFFFFFFFF, where every edge does too, so min(pos, n) is exact.  For B <= 32 the edges of one step sit in distinct
// banks.
struct CovEdges {
    uint32_t n, P;                  // edges, the padded search size
    uint32_t t[LRB_MAX_BINS - 1];
};

__global__ void __launch_bounds__(256)
k_search_edges(const uint32_t* __restrict__ ents, const PartMeta* __restrict__ meta, int bucket0, int n_chunks, ChunkList L,
               StepTables T, uint32_t bucket_base0, uint32_t hi_mask2, int shift, const uint32_t* __restrict__ table,
               const __grid_constant__ CovEdges E, uint32_t* __restrict__ hist) {
    const int bucket = bucket0 + (int)blockIdx.y;
    const uint32_t bucket_base = bucket_base0 + ((uint32_t)blockIdx.y << shift);
    __shared__ uint32_t s_bnd[8][kTaskRuns + 1];
    __shared__ uint32_t s_r0[8][kTaskRuns];
    extern __shared__ uint32_t s_edge[];          // P - 1 words (dynamic)
    if (meta->overflow) return;
    for (uint32_t i = threadIdx.x; i + 1u < E.P; i += blockDim.x) s_edge[i] = i < E.n ? E.t[i] : 0xFFFFFFFFu;
    __syncthreads();
    const uint32_t B = E.n + 1u;
    search_keys_body(ents, meta, bucket, n_chunks, L, T, shift, hist, B, s_bnd, s_r0, table_load(table, bucket_base, hi_mask2),
                     [&](uint32_t* hbase, uint32_t cnt, bool act, uint32_t lane, auto seek, auto row) {
                         uint32_t cell = 0xFFFFFFFFu;
                         if (act) {
                             seek();
                             uint32_t pos = 0;
                             for (uint32_t step = E.P >> 1; step; step >>= 1)
                                 pos += s_edge[pos + step - 1u] <= cnt ? step : 0u;
                             cell = row() * B + min(pos, E.n);
                         }
                         const uint32_t peers = __match_any_sync(0xFFFFFFFFu, cell);
                         if (act && (uint32_t)__ffs(peers) - 1u == lane) atomicAdd(hbase + cell, (uint32_t)__popc(peers));
                     });
}

// A mixed row (lrb_dev_partition_search_layout): the blocks of one table, each binned by (bin size, bin count) as in
// k_search_settings or by count edges as in k_search_edges, into its own columns of rows of W words.  One walk per distinct
// table: the gather happens once and every block of that table bins it (several binnings of one gather measured 1.09-1.65x
// faster than separate searches, k_search_settings), while two tables in one walk measured 1.28-1.30x slower (k_search_samples
// with two tables, DESIGN.md section 4).  The edges of the walk's edge blocks sit back to back in t[]; each edge block's are
// copied into its own P - 1 words of dynamic shared memory (P = the least power of two >= its bins, padding 0xFFFFFFFF),
// searched as in k_search_edges.  COMPACT: the table is compact (as in k_search_samples), else full-layout.  Five CTAs
// per SM, as k_search_edges runs: left to itself ptxas gives the compact form 61 registers (4 CTAs) and spills the
// full-layout form at 48; at (256, 5) both take 48 without spills.
struct CovWalk {
    const uint32_t* table;
    uint32_t n, W;                                  // blocks of this walk, row pitch
    uint64_t magic[LRB_MAX_COV_SETTINGS];
    uint32_t by_edges[LRB_MAX_COV_SETTINGS];        // kind: 0 (bin size, bin count), 1 edges
    uint32_t S32[LRB_MAX_COV_SETTINGS], B[LRB_MAX_COV_SETTINGS], off[LRB_MAX_COV_SETTINGS];   // B: the block's bins
    uint32_t eoff[LRB_MAX_COV_SETTINGS];            // edge blocks: first edge in t[], first word in shared memory
    uint32_t soff[LRB_MAX_COV_SETTINGS], P[LRB_MAX_COV_SETTINGS];
    uint32_t t[LRB_MAX_BINS - 1];                   // a row has at most LRB_MAX_BINS - 1 edges in all
};

template <bool COMPACT>
__global__ void __launch_bounds__(256, 5)
k_search_layout(const uint32_t* __restrict__ ents, const PartMeta* __restrict__ meta, int bucket0, int n_chunks, ChunkList L,
                StepTables T, uint32_t base0, uint32_t hi_mask2, int shift, const __grid_constant__ CovWalk C, uint32_t* __restrict__ hist) {
    const int bucket = bucket0 + (int)blockIdx.y;
    __shared__ uint32_t s_bnd[8][kTaskRuns + 1];
    __shared__ uint32_t s_r0[8][kTaskRuns];
    extern __shared__ uint32_t s_edge[];          // sum of P - 1 words over the edge blocks (dynamic)
    if (meta->overflow) return;
    for (uint32_t m = 0; m < C.n; ++m)
        if (C.by_edges[m])
            for (uint32_t i = threadIdx.x; i + 1u < C.P[m]; i += blockDim.x)
                s_edge[C.soff[m] + i] = i + 1u < C.B[m] ? C.t[C.eoff[m] + i] : 0xFFFFFFFFu;
    __syncthreads();
    auto put = [&](uint32_t* hbase, uint32_t cnt, bool act, uint32_t lane, auto seek, auto row) {
        uint32_t base = 0;
        if (act) {
            seek();
            base = row() * C.W;
        }
        for (uint32_t m = 0; m < C.n; ++m) {
            uint32_t cell = 0xFFFFFFFFu;
            if (act) {
                uint32_t bin;
                if (C.by_edges[m]) {   // warp-uniform
                    const uint32_t* se = s_edge + C.soff[m];
                    uint32_t pos = 0;
                    for (uint32_t step = C.P[m] >> 1; step; step >>= 1) pos += se[pos + step - 1u] <= cnt ? step : 0u;
                    bin = min(pos, C.B[m] - 1u);
                } else {
                    bin = coverage_bin(cnt, C.S32[m], C.magic[m], C.B[m]);
                }
                cell = base + C.off[m] + bin;
            }
            const uint32_t peers = __match_any_sync(0xFFFFFFFFu, cell);
            if (act && (uint32_t)__ffs(peers) - 1u == lane) atomicAdd(hbase + cell, (uint32_t)__popc(peers));
        }
    };
    if (COMPACT) {
        const uint32_t* slice = C.table + (base0 >> 1) + ((uint32_t)blockIdx.y << (shift - 1));   // the bucket's slice
        const uint32_t emask = (1u << (shift - 1)) - 1u;
        search_keys_body(ents, meta, bucket, n_chunks, L, T, shift, hist, C.W, s_bnd, s_r0,
                         [&](uint32_t e) { return __ldg(slice + (e & emask)); }, put);
    } else {
        const uint32_t bucket_base = base0 + ((uint32_t)blockIdx.y << shift);
        search_keys_body(ents, meta, bucket, n_chunks, L, T, shift, hist, C.W, s_bnd, s_r0, table_load(C.table, bucket_base, hi_mask2), put);
    }
}

// sums[r] = number of windows of read r that were bucketed so far = sum of the B bins that start its histogram row (every
// setting of a row counts each window once, so the first one does)
__global__ void __launch_bounds__(256) k_row_sums(const uint32_t* __restrict__ hist, uint32_t* __restrict__ sums, uint64_t n_reads, uint32_t B,
                                                  uint32_t pitch) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    const uint32_t* row = hist + r * pitch;
    uint32_t s = 0;
    for (uint32_t i = 0; i < B; ++i) s += row[i];
    sums[r] = s;
}

// search tasks of every chunk of the partition (L.task0 = prefix of tasks per chunk)
ChunkList chunk_list(const lrb_partition* part) {
    ChunkList L;
    L.task0[0] = 0;
    for (int c = 0; c < kMaxChunks; ++c) {
        L.step0[c] = c < part->n_chunks ? part->chunk_step0[c] : 0u;
        L.nsteps[c] = c < part->n_chunks ? part->chunk_nsteps[c] : 0u;
        L.task0[c + 1] = L.task0[c] + (L.nsteps[c] + kTaskRuns - 1) / kTaskRuns;
    }
    return L;
}

int sms() {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n > 0 ? n : 148;
}

unsigned search_grid(const ChunkList& L, int n_chunks) {  // CTAs per bucket of the search: 8 warps (tasks) per CTA
    return (unsigned)std::min<uint64_t>((uint64_t)sms() * 8, (L.task0[n_chunks] + 7) / 8 + 1);
}

}  // namespace

extern "C" uint64_t lrb_partition_step_capacity(uint64_t n_blocks, int max_chunks) {
    if (max_chunks < 1) max_chunks = 1;
    // every chunk owns ceil(blocks/256) steps + one terminal slot; adds larger than 2^26 blocks are split
    return n_blocks / kPartThreads + 2ull * (uint64_t)max_chunks + 2ull * (n_blocks / kMaxChunkBlocks + 1) + 2;
}

extern "C" uint64_t lrb_partition_steps_words(uint64_t step_capacity) {
    return 2ull * kMaxGroups * kMaxBuckets + step_capacity * (1 + kMaxBuckets / 2 + kMaxBuckets);
}

extern "C" int lrb_dev_fill_blk_read(const lrb_reads_view* dev, uint32_t* blk_read, void* stream) {
    if (!dev || !blk_read) return lrb_set_error(LRB_EINVAL, "lrb_dev_fill_blk_read: null argument");
    if (!dev->n_reads) return LRB_OK;
    const uint64_t threads = dev->n_reads * 32;
    LRB_LAUNCH("k_fill_blk_read", (cudaStream_t)stream, k_fill_blk_read<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*dev, blk_read));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

// ---- host side: begin, add chunk(s) of the stream, then count and/or search bucket by bucket -------------------
extern "C" int lrb_dev_partition_begin(lrb_partition* part, int with_rids, uint32_t key_lo, uint32_t key_hi,
                                       int log2_bucket_keys, void* stream) {
    if (!part || !part->keys || !part->small || !part->steps) return lrb_set_error(LRB_EINVAL, "lrb_dev_partition_begin: null argument");
    if (key_hi > kTableEntries) key_hi = kTableEntries;
    const int shift = log2_bucket_keys;
    if (shift < 20 || shift > 25) return lrb_set_error(LRB_EINVAL, "log2_bucket_keys must be in [20, 25]");
    const uint32_t bsz = 1u << shift;
    if (key_lo >= key_hi || (key_lo & (bsz - 1)) || (key_hi & (bsz - 1)))
        return lrb_set_error(LRB_EINVAL, "key range must be non-empty and aligned to the bucket size 2^%d", shift);
    const int nb = (int)((key_hi - key_lo) >> shift);
    if (nb < 1 || nb > kMaxBuckets) return lrb_set_error(LRB_EINVAL, "key range spans %d buckets (max %d): raise log2_bucket_keys", nb, kMaxBuckets);
    part->n_buckets = nb;
    part->shift = shift;
    part->key_lo = key_lo;
    part->key_hi = key_hi;
    part->has_rids = with_rids ? 1 : 0;
    part->n_chunks = 0;
    part->steps_used = 0;
    part->n_reads = 0;
    LRB_CUDA(cudaMemsetAsync(part->small, 0, sizeof(PartMeta), (cudaStream_t)stream));
    // second-level lists (shared-memory count): built chunk by chunk in add() when the workspace has room for them
    part->l2_enabled = 0;
    part->l2_ncta = part->l2_C3 = 0;
    part->l2_seg0 = part->l2_span = part->l2_spill0 = part->l2_cells0 = 0;
    part->l2_spill_cap = 0;
    const int sub_bits = shift - 16;
    if (part->sub && sub_bits >= 0) {
        const uint64_t nsub = 1ull << sub_bits;
        // CTAs of k2_partition: kL2CtasPerSm per SM, fewer when the lists cannot have that many tiles anyway (small inputs keep big segments)
        const uint64_t n_cta = std::max<uint64_t>(1, std::min<uint64_t>(std::min<uint64_t>((uint64_t)sms() * kL2CtasPerSm, 1024), part->capacity / ((uint64_t)kStepSlots * nb)));
        // workspace (u16 units): fill counters | cell table | segments ... spare tile | spill area
        const uint64_t ncell = (uint64_t)nb * nsub;
        const uint64_t fill_u16 = (n_cta * ncell * 2 + 7) & ~7ull;               // fill counters (u32)
        const uint64_t cells_u16 = ((3 * ncell + kMaxBuckets) * 2 + 7) & ~7ull;   // uint2 info[ncell], u32 hist[ncell], u32 run_len[nb]
        const uint64_t seg0 = fill_u16 + cells_u16;
        const uint64_t segs = ncell * n_cta;
        // spill area (u32 keys) at the end of the workspace: 1/8 of the list capacity, i.e. 1/8 of ALL windows may sit in
        // rows or segments that overflowed before any bucket has to fall back to k_count_keys
        const uint64_t spill_cap = std::min<uint64_t>(std::max<uint64_t>(part->capacity / 8, 1u << 16), 0xFFFFFFF0ull);
        const uint64_t spill_u16 = 2 * spill_cap + 8;
        const uint64_t usable = part->sub_capacity > spill_u16 ? (part->sub_capacity - spill_u16) & ~7ull : 0;
        const uint64_t seg_units = usable > seg0 + kStepSlots ? (usable - seg0 - kStepSlots) & ~7ull : 0;   // a spare tile stays behind the last segment
        uint64_t C3 = (seg_units / segs) & ~7ull;                                // uniform capacity (small inputs, too small a sample)
        if (nsub * n_cta * C3 + kStepSlots >= (1ull << 32)) C3 = ((((1ull << 32) - 8 - kStepSlots) / (nsub * n_cta))) & ~7ull;
        // worth building only if the segments could hold every window with some slack (else most rows would spill);
        // cell offsets are 32-bit counts of octets: 64 GB of segments at most
        if (C3 >= 8 && segs * C3 >= part->capacity + part->capacity / 4 && seg_units / 8 < (1ull << 32)) {
            part->l2_enabled = 1;
            part->l2_ncta = (uint32_t)n_cta;
            part->l2_C3 = (uint32_t)C3;
            part->l2_cells0 = fill_u16;
            part->l2_seg0 = seg0;
            part->l2_span = seg_units;
            part->l2_spill0 = usable;
            part->l2_spill_cap = (uint32_t)spill_cap;
            LRB_CUDA(cudaMemsetAsync(part->sub, 0, seg0 * sizeof(uint16_t), (cudaStream_t)stream));   // fill counters and cell histogram
        }
    }
    return LRB_OK;
}

static int add_chunk(const lrb_reads_view* dev, const uint32_t* blk_read, uint64_t blk_lo, uint64_t blk_hi, lrb_partition* part,
                     cudaStream_t st) {
    if (part->n_chunks >= kMaxChunks) return lrb_set_error(LRB_EINVAL, "too many chunks in one partition (max %d)", kMaxChunks);
    const uint64_t nblk = blk_hi - blk_lo;
    const uint32_t n_steps = (uint32_t)((nblk + kPartThreads - 1) / kPartThreads);
    if (part->steps_used + n_steps + 1 > part->step_capacity)
        return lrb_set_error(LRB_ENOMEM, "partition step tables too small: %llu steps needed, %llu available (lrb_partition_step_capacity)",
                             (ull)(part->steps_used + n_steps + 1), (ull)part->step_capacity);
    const int c = part->n_chunks++;
    const uint32_t step0 = (uint32_t)part->steps_used;
    part->chunk_step0[c] = step0;
    part->chunk_nsteps[c] = n_steps;
    part->steps_used += n_steps + 1;
    PartMeta* meta = reinterpret_cast<PartMeta*>(part->small);
    const StepTables T = step_tables(part->steps, part->step_capacity);
    const int nb = part->n_buckets, shift = part->shift;
    // groups of consecutive steps, one CTA each in both passes; enough of them to fill the machine several times
    const uint32_t want_groups = (uint32_t)std::min<uint64_t>((uint64_t)sms() * 32, kMaxGroups);
    const uint32_t G = std::max<uint32_t>(1, (n_steps + want_groups - 1) / want_groups);
    const uint32_t n_groups = (n_steps + G - 1) / G;
    const bool full = part->key_lo == 0 && part->key_hi >= kTableEntries;
    const uint32_t* br = part->has_rids ? blk_read : nullptr;
    if (full)
        LRB_LAUNCH("k_step_hist", st, k_step_hist<true><<<n_groups, kPartThreads, 0, st>>>(dev->codes, dev->valid, br, blk_lo, blk_hi, part->key_lo, part->key_hi, shift, n_steps, G, step0, T));
    else
        LRB_LAUNCH("k_step_hist", st, k_step_hist<false><<<n_groups, kPartThreads, 0, st>>>(dev->codes, dev->valid, br, blk_lo, blk_hi, part->key_lo, part->key_hi, shift, n_steps, G, step0, T));
    LRB_LAUNCH("k_group_scan", st, k_group_scan<<<nb, 256, 0, st>>>(T, n_groups, meta, c, nb, (ull)part->capacity));
#define LRB_LAUNCH_PART(RID, FULLK)                                                                                              \
    LRB_LAUNCH("k_partition", st, k_partition<RID, FULLK><<<n_groups, kPartThreads, 0, st>>>(dev->codes, dev->valid, br, blk_lo, blk_hi, part->key_lo, part->key_hi, \
                                                               shift, nb, n_steps, G, step0, T, meta, c, part->keys))
    if (part->has_rids) { if (full) LRB_LAUNCH_PART(true, true); else LRB_LAUNCH_PART(true, false); }
    else { if (full) LRB_LAUNCH_PART(false, true); else LRB_LAUNCH_PART(false, false); }
#undef LRB_LAUNCH_PART
    if (part->l2_enabled) {
        L2Layout Y;
        Y.nsub = 1u << (shift - 16); Y.n_cta = part->l2_ncta; Y.C3 = part->l2_C3; Y.nb = (uint32_t)nb;
        Y.seg0 = part->l2_seg0; Y.seg_units = part->l2_span; Y.cells0 = part->l2_cells0; Y.windows_est = part->capacity;
        Y.spill0 = part->l2_spill0; Y.spill_cap = part->l2_spill_cap; Y.key_lo = part->key_lo; Y.shift = shift;
        if (c == 0) {   // segment capacities from the key distribution of a sample of the first chunk (see L2Layout)
            const uint64_t stride = std::max<uint64_t>(1, nblk >> 18);   // <= 2^18 blocks = 8 M windows: ~500 per cell, 0.1 ms
            const uint64_t n_samp = (nblk + stride - 1) / stride;
            if (full)
                LRB_LAUNCH("k_sample_cells", st, k_sample_cells<true><<<(unsigned)((n_samp + 255) / 256), 256, 0, st>>>(dev->codes, dev->valid, blk_lo, blk_hi, stride, part->key_lo, part->key_hi, part->sub, Y));
            else
                LRB_LAUNCH("k_sample_cells", st, k_sample_cells<false><<<(unsigned)((n_samp + 255) / 256), 256, 0, st>>>(dev->codes, dev->valid, blk_lo, blk_hi, stride, part->key_lo, part->key_hi, part->sub, Y));
            LRB_LAUNCH("k_plan_cells", st, k_plan_cells<<<1, 1024, 0, st>>>(part->sub, Y));
        }
        constexpr int kSmemL2 = kL2Stage * (int)sizeof(uint16_t);
#define LRB_LAUNCH_K2(LG)                                                                                               \
    case LG:                                                                                                            \
        LRB_CUDA(cudaFuncSetAttribute(k2_partition<LG>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemL2));         \
        LRB_LAUNCH("k2_partition", st, k2_partition<LG><<<Y.n_cta, kL2Threads, kSmemL2, st>>>(part->keys, meta, c, part->sub, Y)); \
        break
        switch (shift - 16) {  // log2 of the sub-slices per bucket (shift is 20..25)
            LRB_LAUNCH_K2(4); LRB_LAUNCH_K2(5); LRB_LAUNCH_K2(6); LRB_LAUNCH_K2(7); LRB_LAUNCH_K2(8); LRB_LAUNCH_K2(9);
            default: return lrb_set_error(LRB_EINVAL, "second-level lists need log2_bucket_keys in [20, 25]");
        }
#undef LRB_LAUNCH_K2
    }
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_partition_add(const lrb_reads_view* dev, const uint32_t* blk_read, uint64_t blk_lo, uint64_t blk_hi,
                                     lrb_partition* part, void* stream) {
    if (!dev || !part || !part->keys || !part->small || !part->steps) return lrb_set_error(LRB_EINVAL, "lrb_dev_partition_add: null argument");
    if (part->has_rids && !blk_read) return lrb_set_error(LRB_EINVAL, "lrb_dev_partition_add: read ids need blk_read");
    if (blk_hi > dev->n_blocks) blk_hi = dev->n_blocks;
    if (blk_lo >= blk_hi) return LRB_OK;
    part->n_reads = std::max<uint64_t>(part->n_reads, dev->n_reads);
    for (uint64_t lo = blk_lo; lo < blk_hi; lo += kMaxChunkBlocks) {
        const int rc = add_chunk(dev, blk_read, lo, std::min(blk_hi, lo + kMaxChunkBlocks), part, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return LRB_OK;
}

// One-shot convenience: begin + a single chunk.
extern "C" int lrb_dev_partition_build(const lrb_reads_view* dev, const uint32_t* blk_read, int with_rids, uint64_t blk_lo,
                                       uint64_t blk_hi, uint32_t key_lo, uint32_t key_hi, int log2_bucket_keys,
                                       lrb_partition* part, void* stream) {
    int rc = lrb_dev_partition_begin(part, with_rids, key_lo, key_hi, log2_bucket_keys, stream);
    if (rc) return rc;
    return lrb_dev_partition_add(dev, blk_read, blk_lo, blk_hi, part, stream);
}

// Synchronises the stream and reports whether the lists are complete; *needed = entries required in total.
extern "C" int lrb_dev_partition_check(const lrb_partition* part, uint64_t* needed, void* stream) {
    if (!part || !part->small) return lrb_set_error(LRB_EINVAL, "lrb_dev_partition_check: null argument");
    ull h[2] = {0, 0};
    const PartMeta* meta = reinterpret_cast<const PartMeta*>(part->small);
    LRB_CUDA(cudaMemcpyAsync(h, &meta->needed, sizeof h, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    LRB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (needed) *needed = h[0];
    if (h[1])
        return lrb_set_error(LRB_ENOMEM, "partition workspace too small: %llu entries needed, %llu available", h[0], (ull)part->capacity);
    return LRB_OK;
}

// mode bit 0: count (table[key] += 1), bit 1: search (hist/sums through table[key]); both = per bucket count then search
extern "C" int lrb_dev_partition_apply(const lrb_partition* part, int mode, uint32_t* table, long bin_size, int bins,
                                       uint32_t* hist, uint32_t* sums, void* stream) {
    return lrb_dev_partition_apply_range(part, mode, 0, LRB_PART_MAX_BUCKETS, table, bin_size, bins, hist, sums, stream);
}

// The same for the buckets [bucket_lo, bucket_hi) only (clamped to the partition's buckets): lets a multi-GPU driver
// exchange the table slice of bucket b+1 while bucket b is searched.  sums are rewritten when the last bucket is included.
extern "C" int lrb_dev_partition_apply_range(const lrb_partition* part, int mode, int bucket_lo, int bucket_hi, uint32_t* table,
                                             long bin_size, int bins, uint32_t* hist, uint32_t* sums, void* stream) {
    if (!part || !table) return lrb_set_error(LRB_EINVAL, "lrb_dev_partition_apply: null argument");
    if (bucket_lo < 0) bucket_lo = 0;
    if (bucket_hi > part->n_buckets) bucket_hi = part->n_buckets;
    const bool do_count = mode & 1, do_search = mode & 2;
    // second-level (shared-memory) counting needs the sub-slice lists built by add(); without them the L2-atomic kernel does the job
    const bool smem_count = do_count && (mode & 4) && part->l2_enabled;
    const bool overwrite = do_count && (mode & 8);   // the caller did not zero the slices of the applied buckets
    L2Layout Y = {};
    if (smem_count) {
        Y.nsub = 1u << (part->shift - 16); Y.n_cta = part->l2_ncta; Y.C3 = part->l2_C3; Y.nb = (uint32_t)part->n_buckets;
        Y.seg0 = part->l2_seg0; Y.seg_units = part->l2_span; Y.cells0 = part->l2_cells0; Y.windows_est = part->capacity;
        Y.spill0 = part->l2_spill0; Y.spill_cap = part->l2_spill_cap; Y.key_lo = part->key_lo; Y.shift = part->shift;
    }
    if (do_search) {
        if (!hist || !sums) return lrb_set_error(LRB_EINVAL, "lrb_dev_partition_apply: search needs hist and sums");
        if (!part->has_rids) return lrb_set_error(LRB_EINVAL, "lrb_dev_partition_apply: partition was built without read ids");
        if (bin_size <= 0) return lrb_set_error(LRB_EINVAL, "bin_size must be >= 1 (the reference divides by it)");
        if (bins <= 0 || bins > LRB_MAX_BINS) return lrb_set_error(LRB_EINVAL, "bins must be in [1, %d]", LRB_MAX_BINS);
    }
    if (part->n_chunks == 0) return LRB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t S32 = bin_size > 0xFFFFFFFFl ? 0xFFFFFFFFu : (uint32_t)(bin_size > 0 ? bin_size : 1);
    const uint64_t magic = coverage_magic(S32);
    const PartMeta* meta = reinterpret_cast<const PartMeta*>(part->small);
    const StepTables T = step_tables(part->steps, part->step_capacity);
    const ChunkList L = chunk_list(part);
    const int shift = part->shift;
    const uint32_t hi_mask2 = ((1u << shift) - 1u) & ~0xFFFFu;
    const unsigned grid = (unsigned)sms() * 8;
    const unsigned sgrid = search_grid(L, part->n_chunks);
    constexpr int kSmemTable = (1 << kSubBits) * (int)sizeof(uint32_t);
    if (smem_count) {
        LRB_CUDA(cudaFuncSetAttribute(k_count_smem<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTable));
        LRB_CUDA(cudaFuncSetAttribute(k_count_smem<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTable));
    }
    if (overwrite && !smem_count && bucket_hi > bucket_lo)   // the L2-atomic kernel adds: zero the slices of these buckets here
        LRB_CUDA(cudaMemsetAsync(table + part->key_lo + ((size_t)bucket_lo << part->shift), 0, sizeof(uint32_t) * ((size_t)(bucket_hi - bucket_lo) << part->shift), st));
    const bool count_batched = do_count && smem_count && !do_search && bucket_hi > bucket_lo;
    if (count_batched) {  // count only: every bucket in one launch each of the two kernels (the second only counts flagged buckets)
        const uint32_t base0 = part->key_lo + ((uint32_t)bucket_lo << shift);
        const dim3 g1(Y.nsub, (unsigned)(bucket_hi - bucket_lo)), g2(grid, (unsigned)(bucket_hi - bucket_lo));
        if (overwrite) LRB_LAUNCH("k_count_smem", st, k_count_smem<true><<<g1, 1024, kSmemTable, st>>>(part->sub, meta, bucket_lo, Y, base0, shift, table));
        else LRB_LAUNCH("k_count_smem", st, k_count_smem<false><<<g1, 1024, kSmemTable, st>>>(part->sub, meta, bucket_lo, Y, base0, shift, table));
        LRB_LAUNCH("k_count_keys", st, k_count_keys<<<g2, 256, 0, st>>>(part->keys, meta, bucket_lo, part->n_chunks, base0, shift, hi_mask2, table, 1));
        LRB_LAUNCH("k_count_spill", st, k_count_spill<<<grid, 256, 0, st>>>(part->sub, meta, Y, bucket_lo, bucket_hi, table));
    }
    const bool search_batched = do_search && !do_count && bucket_hi > bucket_lo;
    if (search_batched) {
        const uint32_t base0 = part->key_lo + ((uint32_t)bucket_lo << shift);
        const dim3 gs(sgrid, (unsigned)(bucket_hi - bucket_lo));
        LRB_LAUNCH("k_search_keys", st, k_search_keys<<<gs, 256, 0, st>>>(part->keys, meta, bucket_lo, part->n_chunks, L, T, base0, hi_mask2, shift,
                                                                         table, S32, magic, (uint32_t)bins, hist));
    }
    for (int b = bucket_lo; b < bucket_hi && !count_batched && !search_batched; ++b) {
        const uint32_t bucket_base = part->key_lo + ((uint32_t)b << shift);
        if (smem_count && overwrite) LRB_LAUNCH("k_count_smem", st, k_count_smem<true><<<Y.nsub, 1024, kSmemTable, st>>>(part->sub, meta, b, Y, bucket_base, shift, table));
        else if (smem_count) LRB_LAUNCH("k_count_smem", st, k_count_smem<false><<<Y.nsub, 1024, kSmemTable, st>>>(part->sub, meta, b, Y, bucket_base, shift, table));
        if (do_count) LRB_LAUNCH("k_count_keys", st, k_count_keys<<<grid, 256, 0, st>>>(part->keys, meta, b, part->n_chunks, bucket_base, shift, hi_mask2, table, smem_count ? 1 : 0));
        if (smem_count) LRB_LAUNCH("k_count_spill", st, k_count_spill<<<grid, 256, 0, st>>>(part->sub, meta, Y, b, b + 1, table));
        if (do_search)
            LRB_LAUNCH("k_search_keys", st, k_search_keys<<<sgrid, 256, 0, st>>>(part->keys, meta, b, part->n_chunks, L, T, bucket_base, hi_mask2, shift,
                                                                                table, S32, magic, (uint32_t)bins, hist));
    }
    if (do_search && part->n_reads && bucket_hi == part->n_buckets)
        LRB_LAUNCH("k_row_sums", st, k_row_sums<<<(unsigned)((part->n_reads + 255) / 256), 256, 0, st>>>(hist, sums, part->n_reads, (uint32_t)bins, (uint32_t)bins));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

// The search of one coverage layout (common.h).  A layout of one of the three shapes runs the kernel tuned for it: a single
// (bin_size, bins) block on the full table is mode 2 of lrb_dev_partition_apply_range (k_search_keys); several such blocks
// are one launch of k_search_settings; (bin_size, bins) blocks on compact tables one launch of k_search_samples each; one
// edge block on the full table one launch of k_search_edges.  Any other layout is one launch of k_search_layout per
// distinct table, in order of first appearance.  Then k_row_sums.
int lrb_partition_search(const char* who, const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* table,
                         const uint32_t* const* compact, const CovLayout& cov, uint32_t* hist, uint32_t* sums, void* stream) {
    if (cov.single())
        return lrb_dev_partition_apply_range(part, 2, bucket_lo, bucket_hi, const_cast<uint32_t*>(table), cov.b[0].bin_size, cov.b[0].bins, hist,
                                             sums, stream);
    if (!part->has_rids) return lrb_set_error(LRB_EINVAL, "%s: partition was built without read ids", who);
    if (cov.reads_slots() && (part->key_lo & ((1u << part->shift) - 1u)))
        return lrb_set_error(LRB_EINVAL, "%s: the partition's key range must start at a bucket boundary (key_lo %u)", who, part->key_lo);
    if (bucket_lo < 0) bucket_lo = 0;
    if (bucket_hi > part->n_buckets) bucket_hi = part->n_buckets;
    if (part->n_chunks == 0) return LRB_OK;
    bool any_edges = false;
    for (int m = 0; m < cov.n; ++m) any_edges = any_edges || cov.b[m].by_edges;
    const bool settings = !any_edges && !cov.reads_slots(), samples = !any_edges && !cov.reads_full();
    const bool edges = cov.n == 1 && cov.b[0].by_edges && cov.b[0].table < 0;
    cudaStream_t st = (cudaStream_t)stream;
    const PartMeta* meta = reinterpret_cast<const PartMeta*>(part->small);
    const ChunkList L = chunk_list(part);
    const StepTables T = step_tables(part->steps, part->step_capacity);
    const int shift = part->shift;
    const uint32_t hi_mask2 = ((1u << shift) - 1u) & ~0xFFFFu;
    const uint32_t base0 = part->key_lo + ((uint32_t)bucket_lo << shift);
    auto s32 = [](long bin_size) { return bin_size > 0xFFFFFFFFl ? 0xFFFFFFFFu : (uint32_t)bin_size; };
    if (bucket_hi > bucket_lo) {
        const dim3 gs(search_grid(L, part->n_chunks), (unsigned)(bucket_hi - bucket_lo));
        if (edges) {
            const CovBlock& b = cov.b[0];
            CovEdges E;
            E.n = (uint32_t)b.n_edges;
            E.P = 1;
            while (E.P < E.n + 1u) E.P <<= 1;
            std::copy(b.edges, b.edges + b.n_edges, E.t);
            std::fill(E.t + b.n_edges, E.t + (LRB_MAX_BINS - 1), 0xFFFFFFFFu);
            const size_t smem = sizeof(uint32_t) * (E.P - 1u);   // at most 16 380 bytes: no opt-in needed
            LRB_LAUNCH("k_search_edges", st, k_search_edges<<<gs, 256, smem, st>>>(part->keys, meta, bucket_lo, part->n_chunks, L, T, base0,
                                                                                   hi_mask2, shift, table, E, hist));
        } else if (samples) {
            for (int t = 0, off = 0; t < cov.n; off += cov.b[t].bins, ++t) {
                SampleGroup S = {};
                S.W = cov.W;
                S.table = compact[cov.b[t].table];
                S.S32 = s32(cov.b[t].bin_size);
                S.magic = coverage_magic(S.S32);
                S.B = (uint32_t)cov.b[t].bins;
                S.off = (uint32_t)off;
                LRB_LAUNCH("k_search_samples", st, k_search_samples<<<gs, 256, 0, st>>>(part->keys, meta, bucket_lo, part->n_chunks, L, T,
                                                                                       base0 >> 1, shift, S, hist));
            }
        } else if (settings) {
            CovSettings C = {};
            C.n = (uint32_t)cov.n;
            C.W = cov.W;
            for (int m = 0, off = 0; m < cov.n; off += cov.b[m].bins, ++m) {
                C.S32[m] = s32(cov.b[m].bin_size);
                C.magic[m] = coverage_magic(C.S32[m]);
                C.B[m] = (uint32_t)cov.b[m].bins;
                C.off[m] = (uint32_t)off;
            }
            LRB_LAUNCH("k_search_settings", st, k_search_settings<<<gs, 256, 0, st>>>(part->keys, meta, bucket_lo, part->n_chunks, L, T, base0,
                                                                                      hi_mask2, shift, table, C, hist));
        } else {
            uint32_t col[LRB_MAX_COV_SETTINGS];   // first column of each block
            for (int m = 0, off = 0; m < cov.n; off += (int)cov.b[m].width(), ++m) col[m] = (uint32_t)off;
            bool done[LRB_MAX_COV_SETTINGS] = {};
            for (int first = 0; first < cov.n; ++first) {
                if (done[first]) continue;
                const int tab = cov.b[first].table;
                CovWalk C;
                C.table = tab < 0 ? table : compact[tab];
                C.n = 0;
                C.W = cov.W;
                uint32_t n_t = 0, smem_words = 0;
                for (int m = first; m < cov.n; ++m) {
                    const CovBlock& b = cov.b[m];
                    if (b.table != tab) continue;
                    done[m] = true;
                    const uint32_t j = C.n++;
                    C.by_edges[j] = b.by_edges;
                    C.B[j] = b.width();
                    C.off[j] = col[m];
                    C.S32[j] = b.by_edges ? 1u : s32(b.bin_size);
                    C.magic[j] = coverage_magic(C.S32[j]);
                    C.eoff[j] = n_t;
                    C.soff[j] = smem_words;
                    C.P[j] = 1;
                    if (b.by_edges) {
                        while (C.P[j] < C.B[j]) C.P[j] <<= 1;
                        std::copy(b.edges, b.edges + b.n_edges, C.t + n_t);
                        n_t += (uint32_t)b.n_edges;
                        smem_words += C.P[j] - 1u;
                    }
                }
                std::fill(C.t + n_t, C.t + (LRB_MAX_BINS - 1), 0xFFFFFFFFu);
                // each edge block pads to less than twice its bins: at most 2 x 4096 words in all, no opt-in needed
                const size_t smem = sizeof(uint32_t) * smem_words;
                if (tab < 0)
                    LRB_LAUNCH("k_search_layout", st, k_search_layout<false><<<gs, 256, smem, st>>>(part->keys, meta, bucket_lo, part->n_chunks, L,
                                                                                                   T, base0, hi_mask2, shift, C, hist));
                else
                    LRB_LAUNCH("k_search_layout", st, k_search_layout<true><<<gs, 256, smem, st>>>(part->keys, meta, bucket_lo, part->n_chunks, L,
                                                                                                  T, base0, hi_mask2, shift, C, hist));
            }
        }
    }
    if (part->n_reads && bucket_hi == part->n_buckets)
        LRB_LAUNCH("k_row_sums", st, k_row_sums<<<(unsigned)((part->n_reads + 255) / 256), 256, 0, st>>>(hist, sums, part->n_reads, cov.b[0].width(), cov.W));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

// Several coverage settings in one search (k_search_settings): hist rows of W = sum of bins[m] words, setting m's bins at
// column sum_{j<m} bins[j]; sums are rewritten by the call that includes the last bucket.  n = 1 is mode 2 of
// lrb_dev_partition_apply_range.
extern "C" int lrb_dev_partition_search_settings(const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* table, int n,
                                                 const long* bin_sizes, const int* bins, uint32_t* hist, uint32_t* sums, void* stream) {
    static const char* who = "lrb_dev_partition_search_settings";
    if (!part || !table || !hist || !sums) return lrb_set_error(LRB_EINVAL, "%s: null argument", who);
    CovLayout L = lrb_cov_settings(n, bin_sizes, bins);
    const int rc = lrb_check_cov_layout(who, &L);
    return rc ? rc : lrb_partition_search(who, part, bucket_lo, bucket_hi, table, nullptr, L, hist, sums, stream);
}

// Several compact sample tables in one search (k_search_samples): hist rows of W = sum of bins[t] words, table t's bins at
// column sum_{j<t} bins[j]; one walk over the lists per table; sums are rewritten by the call that includes the last bucket.
extern "C" int lrb_dev_partition_search_samples(const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* const* compact_tables,
                                                int n, const long* bin_sizes, const int* bins, uint32_t* hist, uint32_t* sums, void* stream) {
    static const char* who = "lrb_dev_partition_search_samples";
    if (!part || !compact_tables || !hist || !sums) return lrb_set_error(LRB_EINVAL, "%s: null argument", who);
    int slots[LRB_MAX_SAMPLE_TABLES] = {};   // block t reads compact_tables[slots[t]], the first entry with its pointer
    for (int t = 0; t < n && t < LRB_MAX_SAMPLE_TABLES; ++t) {
        if (!compact_tables[t]) return lrb_set_error(LRB_EINVAL, "%s: null table %d", who, t);
        while (compact_tables[slots[t]] != compact_tables[t]) ++slots[t];
    }
    CovLayout L = lrb_cov_settings(n, bin_sizes, bins, slots);
    const int rc = lrb_check_cov_layout(who, &L);
    return rc ? rc : lrb_partition_search(who, part, bucket_lo, bucket_hi, nullptr, compact_tables, L, hist, sums, stream);
}

// Coverage bins given by count edges (k_search_edges): hist rows of n_edges + 1 words; edges is a HOST array, checked by
// lrb_check_cov_layout; sums are rewritten by the call that includes the last bucket.
extern "C" int lrb_dev_partition_search_edges(const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* table,
                                              const uint32_t* edges, int n_edges, uint32_t* hist, uint32_t* sums, void* stream) {
    static const char* who = "lrb_dev_partition_search_edges";
    if (!part || !table || !hist || !sums) return lrb_set_error(LRB_EINVAL, "%s: null argument", who);
    CovLayout L = lrb_cov_edges(edges, n_edges);
    const int rc = lrb_check_cov_layout(who, &L);
    return rc ? rc : lrb_partition_search(who, part, bucket_lo, bucket_hi, table, nullptr, L, hist, sums, stream);
}

// A mixed coverage row (k_search_layout, or the kernel of the shape the layout has): blocks is a HOST array, checked by
// lrb_check_cov_layout; block m reads `table` (table -1) or compact_tables[t]; sums are rewritten by the call that includes
// the last bucket.
extern "C" int lrb_dev_partition_search_layout(const lrb_partition* part, int bucket_lo, int bucket_hi, const uint32_t* table,
                                               const uint32_t* const* compact_tables, const lrb_cov_block* blocks, int n, uint32_t* hist,
                                               uint32_t* sums, void* stream) {
    static const char* who = "lrb_dev_partition_search_layout";
    if (!part || !hist || !sums) return lrb_set_error(LRB_EINVAL, "%s: null argument", who);
    CovLayout L = lrb_cov_layout(blocks, n);
    const int rc = lrb_check_cov_layout(who, &L);
    if (rc) return rc;
    for (int m = 0; m < L.n; ++m) {
        const int t = L.b[m].table;
        if (t < 0 && !table) return lrb_set_error(LRB_EINVAL, "%s: null table (block %d reads the full-layout table)", who, m);
        if (t >= 0 && (!compact_tables || !compact_tables[t])) return lrb_set_error(LRB_EINVAL, "%s: null compact table %d (block %d)", who, t, m);
    }
    return lrb_partition_search(who, part, bucket_lo, bucket_hi, table, compact_tables, L, hist, sums, stream);
}
