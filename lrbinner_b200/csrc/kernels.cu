// kernels.cu — sm_100a kernels of the profile stage and their C-ABI launchers (lrb_dev_*).
//
// Work decomposition (DESIGN.md "Kernels"):
//   * composition / search : one WARP per tile (<= 256 blocks of 32 slots of ONE read); lanes take blocks
//     lane, lane+32, ... so every warp load is a fully coalesced 256 B (codes) / 128 B (validity) line;
//     per-warp shared-memory histogram (smem atomics, measured ~1.6 T ops/s on B200), flushed to the
//     read's output row with one RED per non-zero bin.
//   * count  : one THREAD per block, grid-stride; read-oblivious because padding slots are invalid;
//     one RED.ADD.U32 per valid window on the bit-15-clear key of {val, rc(val)}.
//   * mirror : 64x64 tiled "transpose" T[x] = T[rc(x)] for bit-15-set x (coalesced both ways).
//   * spectrum: grid-stride 16-byte reads of the bit-15-clear half; small counts into per-lane shared counters.
// No tensor cores anywhere: nothing here is a dense contraction (BASELINE.json north_star).
#include <cuda_runtime.h>
#include <algorithm>
#include <atomic>
#include <mutex>
#include <stdint.h>
#include <stdio.h>

#include "../../include/lrbinner_b200.h"
#include "common.h"
#include "lane_core.cuh"
#include "fixed6.h"

using namespace lrb;

namespace {

constexpr int kWarpsPerCta = 8;
constexpr int kCtaThreads = kWarpsPerCta * 32;

// canonical-index LUTs of count-kmers (compute_kmer_inds), filled once per device by ensure_luts()
__device__ uint16_t g_lut3[64];
__device__ uint16_t g_lut4[256];
__device__ uint16_t g_lut5[1024];

template <int K> struct CompTraits;
template <> struct CompTraits<3> { static constexpr int P = 32; };
template <> struct CompTraits<4> { static constexpr int P = 136; };
template <> struct CompTraits<5> { static constexpr int P = 512; };

__device__ __forceinline__ uint32_t ld_stream_u32(const uint32_t* p) { return __ldg(p); }
__device__ __forceinline__ uint2 ld_stream_u2(const uint2* p) { return __ldg(p); }

// ------------------------------------------------------------------------------------------------
// composition: count_kmers (count-kmers.cpp:66-95)
// ------------------------------------------------------------------------------------------------
// fire-and-forget shared-memory increment (plain RED; see partition.cu)
__device__ __forceinline__ void smem_inc(uint32_t* p) {
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
}

// Per-warp histogram of the RAW k-mers (4^K bins) — one shared-memory RED per base, no LUT lookup in the inner loop;
// the canonical fold (index of min(x, rc x), count-kmers.cpp:38-64) happens once per tile at flush time.
template <int K>
__global__ void __launch_bounds__(kCtaThreads)
k_composition(lrb_reads_view R, uint32_t* __restrict__ out, uint64_t tile_lo, uint64_t tile_hi) {
    constexpr int P = CompTraits<K>::P;
    constexpr int NK = 1 << (2 * K);
    __shared__ uint16_t s_lut[NK];
    __shared__ uint32_t s_raw[kWarpsPerCta][NK];

    const uint16_t* glut = (K == 3) ? g_lut3 : (K == 4) ? g_lut4 : g_lut5;
    for (int i = threadIdx.x; i < NK; i += kCtaThreads) s_lut[i] = glut[i];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* raw = s_raw[warp];
    for (int i = lane; i < NK; i += 32) raw[i] = 0;
    __syncthreads();

    const uint64_t tile = tile_lo + (uint64_t)blockIdx.x * kWarpsPerCta + warp;
    if (tile >= tile_hi) return;
    const uint32_t r = R.tile_read[tile];
    const uint32_t b0 = R.tile_blk[tile];
    const uint32_t rb0 = R.read_blk[r], rb1 = R.read_blk[r + 1];
    const uint32_t len = R.read_len[r];
    const uint32_t nblk = min((uint32_t)kTileBlocks, rb1 - b0);
    const uint2* codes2 = reinterpret_cast<const uint2*>(R.codes);

    for (uint32_t i = lane; i < nblk; i += 32) {
        const uint32_t gb = b0 + i;
        const uint2 w = ld_stream_u2(codes2 + gb);
        const uint32_t p0 = (gb - rb0) * 32u;            // read position of slot 0 of this block
        const uint32_t pw = (p0 != 0) ? ld_stream_u32(R.codes + 2 * (size_t)gb - 1) : 0u;
        const uint32_t m = comp_block_mask(p0, len, K);
        if (K == 3) comp_block<K>(pw, w.x, w.y, m, [&](uint32_t kmer) { atomicAdd(&raw[kmer], 1u); });  // 64 bins: lanes collide, aggregated form
        else comp_block<K>(pw, w.x, w.y, m, [&](uint32_t kmer) { smem_inc(&raw[kmer]); });
    }
    __syncwarp();
    uint32_t* row = out + (size_t)r * P;
    for (int i = lane; i < NK; i += 32) {   // fold x and rc(x) into the canonical bin; x < rc(x) owns the pair
        const uint32_t rc = rc_small((uint32_t)i, K);
        if ((uint32_t)i > rc) continue;
        const uint32_t c = raw[i] + (((uint32_t)i != rc) ? raw[rc] : 0u);
        if (c) atomicAdd(row + s_lut[i], c);
    }
}

// ------------------------------------------------------------------------------------------------
// 15-mer count: line_to_kmer_counts (kmer_utils.h:114-156), canonical half + later mirror
// ------------------------------------------------------------------------------------------------
template <bool FILTER>
__global__ void __launch_bounds__(256)
k_count15(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ valid, uint32_t* __restrict__ table,
          uint64_t blk_lo, uint64_t blk_hi, uint32_t key_lo, uint32_t key_hi) {
    const uint2* codes2 = reinterpret_cast<const uint2*>(codes);
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t gb = blk_lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; gb < blk_hi; gb += stride) {
        const uint32_t v = ld_stream_u32(valid + gb);
        const uint32_t pv = gb ? ld_stream_u32(valid + gb - 1) : 0u;
        const uint32_t m = window15_mask(pv, v);
        if (m == 0) continue;
        const uint2 w = ld_stream_u2(codes2 + gb);
        const uint32_t pw = gb ? ld_stream_u32(codes + 2 * gb - 1) : 0u;
        canon15_block(pw, w.x, w.y, m, [&](uint32_t key) {
            if (!FILTER || (key >= key_lo && key < key_hi)) atomicAdd(table + key, 1u);
        });
    }
}

// mirror: T[x] = T[rc(x)] for all x with bit 15 set — a 64x64 tiled "transpose" whose index algebra
// (mirror_dst_index / mirror_src_index) lives in lane_core.cuh.  Reads touch only bit-15-clear entries,
// writes only bit-15-set ones, so the pass is race-free in place; both sides move 256 B rows.  Global accesses are
// 16 bytes wide: a source row of the tile is 64 contiguous entries = 16 uint4, and so is a destination row.
__global__ void __launch_bounds__(256) k_mirror(uint32_t* __restrict__ table) {
    __shared__ uint32_t tile[64][65];
    const uint32_t t = blockIdx.x;
    const uint32_t c4 = (threadIdx.x & 15u) * 4u, r = threadIdx.x >> 4;  // 16 uint4 columns x 16 rows per pass
#pragma unroll
    for (uint32_t sb = r; sb < 64; sb += 16) {
        const uint4 v = __ldcs(reinterpret_cast<const uint4*>(table + mirror_src_index(t, sb, c4)));
        tile[sb][c4] = v.x; tile[sb][c4 + 1] = v.y; tile[sb][c4 + 2] = v.z; tile[sb][c4 + 3] = v.w;
    }
    __syncthreads();
    const uint32_t s0 = rc_small(c4, 3), s1 = rc_small(c4 + 1, 3), s2 = rc_small(c4 + 2, 3), s3 = rc_small(c4 + 3, 3);
#pragma unroll
    for (uint32_t a = r; a < 64; a += 16) {
        const uint32_t col = rc_small(a, 3);
        const uint4 o = make_uint4(tile[s0][col], tile[s1][col], tile[s2][col], tile[s3][col]);
        __stcs(reinterpret_cast<uint4*>(table + mirror_dst_index(t, a, c4)), o);
    }
}

// ------------------------------------------------------------------------------------------------
// abundance spectrum of the canonical half (no reference counterpart): spectrum[c] += #keys with T == c (c < M),
// [M] += #keys with T >= M, [M+1] += their sum, [M+2] = max.  Canonical index ci in [0, 2^29) = (row:14 | col:15) maps to
// the table word (row << 16) | col; the kernel walks 16-byte units of 4 canonical entries, which never straddle a row.
// The values are heavily concentrated (zeros of a sparse table, the error floor at small counts), so one shared-memory
// atomic per entry into one histogram would serialise on a few addresses.  Counts below kSpecLaneBins go to counters
// private to the lane instead — s_lane[warp][c][lane], so lane l only ever touches bank l and a warp's update is one
// conflict-free RED whatever the values — and are summed over the lanes once per CTA.  Larger counts are spread out
// (genomic peaks) and take the CTA's shared histogram; counts past that take global u64 atomics.  A thread whose 4
// values are equal adds them as one update of 4.
// ------------------------------------------------------------------------------------------------
constexpr int kSpecThreads = 256;
constexpr int kSpecWarps = kSpecThreads / 32;
constexpr int kSpecUnroll = 4;              // 16-byte loads in flight per thread
constexpr uint32_t kSpecLaneBins = 32;      // counts below this: per-lane counters
constexpr uint32_t kSpecSmemBins = 8192;    // counts below this: the CTA's shared histogram; above: global u64 atomics
constexpr size_t kSpecSmem = sizeof(uint32_t) * (kSpecSmemBins + (size_t)kSpecWarps * kSpecLaneBins * 32);  // 64 KiB

__device__ __forceinline__ uint64_t canon_word(uint64_t ci) { return ((ci >> 15) << 16) | (ci & 0x7FFFu); }

__device__ __forceinline__ void smem_add(uint32_t* p, uint32_t n) {  // fire-and-forget shared-memory add (RED)
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "r"(n) : "memory");
}

struct SpecAcc {
    uint32_t n_over = 0, vmax = 0;
    uint64_t sum_over = 0;
};

// table value v counted w times
__device__ __forceinline__ void spec_add(uint32_t* s_hist, uint32_t* my_lane, unsigned long long* spec, uint32_t M, uint32_t v,
                                         uint32_t w, SpecAcc& a) {
    if (v < M) {
        if (v < kSpecLaneBins) smem_add(my_lane + v * 32u, w);
        else if (v < kSpecSmemBins) smem_add(s_hist + v, w);
        else atomicAdd(spec + v, (unsigned long long)w);
    } else {
        a.n_over += w;
        a.sum_over += (uint64_t)v * w;
    }
    a.vmax = max(a.vmax, v);
}

// FULL: canonical index ci is the table word canon_word(ci); else the table is compact (lrb_dev_table_compact) and ci is
// its entry ci
template <bool FULL>
__device__ __forceinline__ uint64_t spec_word(uint64_t ci) { return FULL ? canon_word(ci) : ci; }

template <bool FULL>
__global__ void __launch_bounds__(kSpecThreads)
k_table_spectrum(const uint32_t* __restrict__ table, uint64_t u_beg, uint64_t u_end, uint64_t e0_lo, uint64_t e0_hi,
                 uint64_t e1_lo, uint64_t e1_hi, uint32_t M, unsigned long long* __restrict__ spec) {
    extern __shared__ uint32_t s_spec[];
    uint32_t* s_hist = s_spec;                                   // [kSpecSmemBins]
    uint32_t* s_lane = s_spec + kSpecSmemBins;                   // [kSpecWarps][kSpecLaneBins][32]
    for (uint32_t i = threadIdx.x; i < kSpecSmemBins + kSpecWarps * kSpecLaneBins * 32; i += kSpecThreads) s_spec[i] = 0;
    __syncthreads();

    SpecAcc a;
    const uint32_t lane = threadIdx.x & 31u, warp_in_cta = threadIdx.x >> 5;
    uint32_t* my_lane = s_lane + warp_in_cta * (kSpecLaneBins * 32) + lane;
    const uint64_t n_units = u_end - u_beg;
    const uint64_t stride = (uint64_t)gridDim.x * kSpecThreads * kSpecUnroll;
    for (uint64_t base = ((uint64_t)blockIdx.x * kSpecWarps + warp_in_cta) * (32 * kSpecUnroll); base < n_units; base += stride) {
        uint4 q[kSpecUnroll];
#pragma unroll
        for (int k = 0; k < kSpecUnroll; ++k) {   // a warp reads 4 x 512 contiguous bytes
            const uint64_t u = base + (uint64_t)k * 32 + lane;
            if (u < n_units) q[k] = __ldcs(reinterpret_cast<const uint4*>(table + spec_word<FULL>((u_beg + u) * 4)));
        }
#pragma unroll
        for (int k = 0; k < kSpecUnroll; ++k) {
            if (base + (uint64_t)k * 32 + lane >= n_units) continue;
            if (q[k].x == q[k].y && q[k].x == q[k].z && q[k].x == q[k].w) {
                spec_add(s_hist, my_lane, spec, M, q[k].x, 4u, a);
            } else {
                spec_add(s_hist, my_lane, spec, M, q[k].x, 1u, a);
                spec_add(s_hist, my_lane, spec, M, q[k].y, 1u, a);
                spec_add(s_hist, my_lane, spec, M, q[k].z, 1u, a);
                spec_add(s_hist, my_lane, spec, M, q[k].w, 1u, a);
            }
        }
    }
    // the < 8 entries before the first / after the last whole unit (key ranges not aligned to 4)
    if (blockIdx.x == 0 && threadIdx.x < 16) {
        const uint64_t ci = threadIdx.x < 8 ? e0_lo + threadIdx.x : e1_lo + (threadIdx.x - 8);
        if (ci < (threadIdx.x < 8 ? e0_hi : e1_hi)) spec_add(s_hist, my_lane, spec, M, __ldg(table + spec_word<FULL>(ci)), 1u, a);
    }

    a.n_over = __reduce_add_sync(0xFFFFFFFFu, a.n_over);
    a.vmax = __reduce_max_sync(0xFFFFFFFFu, a.vmax);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a.sum_over += __shfl_xor_sync(0xFFFFFFFFu, a.sum_over, o);
    if (lane == 0) {
        if (a.n_over) {
            atomicAdd(spec + M, (unsigned long long)a.n_over);
            atomicAdd(spec + M + 1, (unsigned long long)a.sum_over);
        }
        atomicMax(spec + M + 2, (unsigned long long)a.vmax);
    }
    __syncwarp();
    // lane c sums count c over the warp's 32 lane counters (rotated start: the 32 lanes read 32 different banks)
    if (lane < kSpecLaneBins) {
        const uint32_t* row = s_lane + warp_in_cta * (kSpecLaneBins * 32) + lane * 32u;
        uint32_t n = 0;
        for (uint32_t j = 0; j < 32; ++j) n += row[(lane + j) & 31u];
        if (n) smem_add(s_hist + lane, n);
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < min(M, kSpecSmemBins); i += kSpecThreads)
        if (s_hist[i]) atomicAdd(spec + i, (unsigned long long)s_hist[i]);
}

// validity bitmap from the read lengths (one warp per read), then the sparse exceptions on top
__global__ void __launch_bounds__(256) k_default_valid(lrb_reads_view R, uint32_t* __restrict__ valid) {
    const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= R.n_reads) return;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t b0 = R.read_blk[r], b1 = R.read_blk[r + 1], len = R.read_len[r];
    for (uint32_t b = b0 + lane; b < b1; b += 32) valid[b] = default_valid_word(len, (uint64_t)(b - b0) * 32);
    if (r == R.n_reads - 1 && lane == 0) valid[R.n_blocks] = 0u;  // the word after the stream
}

__global__ void __launch_bounds__(256)
k_patch_valid(const uint32_t* __restrict__ exc_blk, const uint32_t* __restrict__ exc_valid, uint64_t n_exc, uint32_t* __restrict__ valid) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_exc) valid[exc_blk[i]] = exc_valid[i];
}

// ------------------------------------------------------------------------------------------------
// search: line_to_vec (kmer_utils.h:24-87)
// ------------------------------------------------------------------------------------------------
template <bool FILTER>
__global__ void __launch_bounds__(kCtaThreads)
k_search15(lrb_reads_view R, const uint32_t* __restrict__ table, uint32_t S32, uint64_t magic, uint32_t B,
           uint32_t* __restrict__ hist_out, uint32_t* __restrict__ sums_out, uint64_t tile_lo, uint64_t tile_hi,
           uint32_t key_lo, uint32_t key_hi) {
    extern __shared__ uint32_t s_dyn[];  // [kWarpsPerCta][B]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* hist = s_dyn + (size_t)warp * B;
    for (uint32_t i = lane; i < B; i += 32) hist[i] = 0;
    __syncwarp();

    const uint64_t tile = tile_lo + (uint64_t)blockIdx.x * kWarpsPerCta + warp;
    if (tile >= tile_hi) return;
    const uint32_t r = R.tile_read[tile];
    const uint32_t b0 = R.tile_blk[tile];
    const uint32_t rb1 = R.read_blk[r + 1];
    const uint32_t nblk = min((uint32_t)kTileBlocks, rb1 - b0);
    const uint2* codes2 = reinterpret_cast<const uint2*>(R.codes);
    uint32_t nwin = 0;

    for (uint32_t i = lane; i < nblk; i += 32) {
        const uint32_t gb = b0 + i;
        const uint32_t v = ld_stream_u32(R.valid + gb);
        const uint32_t pv = gb ? ld_stream_u32(R.valid + gb - 1) : 0u;
        uint32_t m = window15_mask(pv, v);
        if (m == 0) continue;
        const uint2 w = ld_stream_u2(codes2 + gb);
        const uint32_t pw = gb ? ld_stream_u32(R.codes + 2 * (size_t)gb - 1) : 0u;
        uint32_t cnt[32];
        if (FILTER) {
            const uint32_t r0 = rc16(w.y), r1 = rc16(w.x), r2 = rc16(pw);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                cnt[j] = 0;
                if ((m >> j) & 1u) {
                    const uint32_t val = kmer_ending_at<15>(pw, w.x, w.y, j);
                    const uint32_t key = canonical15(val, rc15_ending_at(r0, r1, r2, j));
                    if (key >= key_lo && key < key_hi) cnt[j] = __ldg(table + key);
                    else m &= ~(1u << j);
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                cnt[j] = 0;
                if ((m >> j) & 1u) cnt[j] = __ldg(table + kmer_ending_at<15>(pw, w.x, w.y, j));
            }
        }
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if ((m >> j) & 1u) atomicAdd(&hist[coverage_bin(cnt[j], S32, magic, B)], 1u);
        nwin += (uint32_t)popc32(m);
    }
    __syncwarp();
    uint32_t* row = hist_out + (size_t)r * B;
    for (uint32_t i = lane; i < B; i += 32) {
        const uint32_t c = hist[i];
        if (c) atomicAdd(row + i, c);
    }
    nwin = __reduce_add_sync(0xFFFFFFFFu, nwin);
    if (lane == 0 && nwin) atomicAdd(sums_out + r, nwin);
}

// ------------------------------------------------------------------------------------------------
// ASCII -> packed on the device (same rule as the host packer in ingest.cpp)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_pack_ascii(lrb_reads_view R, const char* __restrict__ bases, const uint64_t* __restrict__ offsets,
             uint32_t* __restrict__ codes, uint32_t* __restrict__ valid) {
    // one warp per read, lanes take blocks
    const uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= R.n_reads) return;
    const uint32_t rb0 = R.read_blk[r], rb1 = R.read_blk[r + 1], len = R.read_len[r];
    const char* s = bases + offsets[r];
    for (uint32_t b = rb0 + lane; b < rb1; b += 32) {
        const uint32_t p0 = (b - rb0) * 32u;
        uint32_t w0 = 0, w1 = 0, v = 0;
        for (int j = 0; j < 32; ++j) {
            const uint32_t p = p0 + j;
            if (p < len) {
                const unsigned char c = (unsigned char)s[p];
                const uint32_t code = (c >> 1) & 3u;
                if (j < 16) w0 |= code << (30 - 2 * j); else w1 |= code << (62 - 2 * j);
                if (c == 'A' || c == 'C' || c == 'G' || c == 'T') v |= 1u << j;
            }
        }
        codes[2 * (size_t)b] = w0;
        codes[2 * (size_t)b + 1] = w1;
        valid[b] = v;
    }
}

// ------------------------------------------------------------------------------------------------
// text epilogue: fixed-width "%f" rows (count-kmers.cpp:110-118, search-15mers.cpp:35-48)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void put_fixed6_dev(char* dst, uint32_t q, char sep) {  // "d.dddddd" + sep
    dst[0] = (char)('0' + q / 1000000u);
    dst[1] = '.';
    uint32_t f = q % 1000000u;
#pragma unroll
    for (int i = 7; i >= 2; --i) { dst[i] = (char)('0' + f % 10u); f /= 10u; }
    dst[8] = sep;
}

// one thread per value; COMP: value followed by ' ' and a '\n' closes the row; coverage: ' ' between, '\n' last
template <bool COMP>
__global__ void __launch_bounds__(256)
k_format_rows(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ denom_src, uint64_t n_rows, uint32_t width,
              int k, char* __restrict__ text) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_rows * width) return;
    const uint64_t r = idx / width;
    const uint32_t j = (uint32_t)(idx - r * width);
    uint32_t den = denom_src[r];
    if (COMP) den = den >= (uint32_t)k ? den - (uint32_t)k + 1u : 0u;  // total = max(0, len-k+1)
    const uint32_t q = fixed6(counts[idx], den, !COMP);
    const size_t row_bytes = COMP ? (size_t)width * 9 + 1 : (size_t)width * 9;
    char* dst = text + r * row_bytes + (size_t)j * 9;
    put_fixed6_dev(dst, q, (!COMP && j == width - 1) ? '\n' : ' ');
    if (COMP && j == width - 1) dst[9] = '\n';
}

// profile values as the downstream stages see them: float(the "%f" text) == fixed6 / 10^6 (both exactly rounded)
template <bool COMP>
__global__ void __launch_bounds__(256)
k_profile_values(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ denom_src, uint64_t n_rows, uint32_t width, int k,
                 double* __restrict__ out) {
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_rows * width) return;
    const uint64_t r = idx / width;
    uint32_t den = denom_src[r];
    if (COMP) den = den >= (uint32_t)k ? den - (uint32_t)k + 1u : 0u;  // total = max(0, len-k+1)
    out[idx] = (double)fixed6(counts[idx], den, !COMP) / 1e6;
}

// the LUTs are per device, not per thread (the multi-GPU host pipeline drives every device from a thread of its own)
std::atomic<bool> g_luts_ready[64];
std::mutex g_luts_mutex;

int ensure_luts() {
    int dev = 0;
    LRB_CUDA(cudaGetDevice(&dev));
    if (dev < 64 && g_luts_ready[dev].load(std::memory_order_acquire)) return LRB_OK;
    std::lock_guard<std::mutex> lock(g_luts_mutex);
    if (dev < 64 && g_luts_ready[dev].load(std::memory_order_acquire)) return LRB_OK;
    uint16_t l3[64], l4[256], l5[1024];
    lrb_kmer_lut(3, l3);
    lrb_kmer_lut(4, l4);
    lrb_kmer_lut(5, l5);
    LRB_CUDA(cudaMemcpyToSymbol(g_lut3, l3, sizeof l3));
    LRB_CUDA(cudaMemcpyToSymbol(g_lut4, l4, sizeof l4));
    LRB_CUDA(cudaMemcpyToSymbol(g_lut5, l5, sizeof l5));
    if (dev < 64) g_luts_ready[dev].store(true, std::memory_order_release);
    return LRB_OK;
}

int sm_count() {
    static thread_local int sms[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev >= 64) return 148;
    if (!sms[dev]) {
        if (cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms[dev] = 148;
    }
    return sms[dev];
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI launchers
// ------------------------------------------------------------------------------------------------
extern "C" int lrb_dev_composition(const lrb_reads_view* dev, int k, uint32_t* counts, uint64_t tile_lo,
                                   uint64_t tile_hi, void* stream) {
    if (!dev || !counts || k < 3 || k > 5) return lrb_set_error(LRB_EINVAL, "lrb_dev_composition: k must be 3, 4 or 5");
    if (tile_hi > dev->n_tiles) tile_hi = dev->n_tiles;
    if (tile_lo >= tile_hi) return LRB_OK;
    int rc = ensure_luts();
    if (rc) return rc;
    const uint64_t ntile = tile_hi - tile_lo;
    const unsigned grid = (unsigned)((ntile + kWarpsPerCta - 1) / kWarpsPerCta);
    cudaStream_t st = (cudaStream_t)stream;
    if (k == 3) LRB_LAUNCH("k_composition", st, k_composition<3><<<grid, kCtaThreads, 0, st>>>(*dev, counts, tile_lo, tile_hi));
    else if (k == 4) LRB_LAUNCH("k_composition", st, k_composition<4><<<grid, kCtaThreads, 0, st>>>(*dev, counts, tile_lo, tile_hi));
    else LRB_LAUNCH("k_composition", st, k_composition<5><<<grid, kCtaThreads, 0, st>>>(*dev, counts, tile_lo, tile_hi));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_count(const lrb_reads_view* dev, uint32_t* table, uint64_t blk_lo, uint64_t blk_hi,
                             uint32_t key_lo, uint32_t key_hi, void* stream) {
    if (!dev || !table) return lrb_set_error(LRB_EINVAL, "lrb_dev_count: null argument");
    if (blk_hi > dev->n_blocks) blk_hi = dev->n_blocks;
    if (blk_lo >= blk_hi || key_lo >= key_hi) return LRB_OK;
    const uint64_t nblk = blk_hi - blk_lo;
    const int threads = 256;
    uint64_t want = (nblk + threads - 1) / threads;
    const uint64_t cap = (uint64_t)sm_count() * 16;  // persistent grid: 16 CTAs of 256 threads per SM
    const unsigned grid = (unsigned)(want < cap ? want : cap);
    cudaStream_t st = (cudaStream_t)stream;
    const bool filter = !(key_lo == 0 && key_hi >= kTableEntries);
    if (filter) LRB_LAUNCH("k_count15", st, k_count15<true><<<grid, threads, 0, st>>>(dev->codes, dev->valid, table, blk_lo, blk_hi, key_lo, key_hi));
    else LRB_LAUNCH("k_count15", st, k_count15<false><<<grid, threads, 0, st>>>(dev->codes, dev->valid, table, blk_lo, blk_hi, key_lo, key_hi));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_mirror(uint32_t* table, void* stream) {
    if (!table) return lrb_set_error(LRB_EINVAL, "lrb_dev_mirror: null table");
    LRB_LAUNCH("k_mirror", (cudaStream_t)stream, k_mirror<<<1u << 17, 256, 0, (cudaStream_t)stream>>>(table));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

// canonical half of every 2^16-entry row (its first 2^15 entries) side by side: one pitched copy on the copy engines
extern "C" int lrb_dev_table_compact(const uint32_t* table, uint32_t* compact, void* stream) {
    if (!table || !compact) return lrb_set_error(LRB_EINVAL, "lrb_dev_table_compact: null argument");
    LRB_CUDA(cudaMemcpy2DAsync(compact, 4u << 15, table, 4u << 16, 4u << 15, (size_t)(LRB_TABLE_ENTRIES >> 16), cudaMemcpyDeviceToDevice,
                               (cudaStream_t)stream));
    return LRB_OK;
}

// canonical (bit-15-clear) keys below `key` (key <= 2^30): 2^15 per complete 2^16-entry row, then the clear half of its row
static uint64_t canon_rank(uint64_t key) { return ((key >> 16) << 15) + std::min<uint64_t>(key & 0xFFFFu, 0x8000u); }

// the spectrum of canonical indices [ci_lo, ci_hi): whole 4-entry units [u_beg, u_end); the entries outside them are the
// edges e0 (head) and e1 (tail), < 8 in all
template <bool FULL>
static int launch_spectrum(const char* name, const uint32_t* table, uint64_t ci_lo, uint64_t ci_hi, uint32_t max_count, uint64_t* spectrum,
                           cudaStream_t st) {
    uint64_t u_beg = (ci_lo + 3) / 4, u_end = ci_hi / 4;
    uint64_t e0_lo = ci_lo, e0_hi = u_beg * 4, e1_lo = u_end * 4, e1_hi = ci_hi;
    if (u_beg >= u_end) { u_end = u_beg; e0_hi = ci_hi; e1_lo = e1_hi = 0; }
    const uint64_t per_cta = (uint64_t)kSpecThreads * kSpecUnroll;
    const uint64_t want = std::max<uint64_t>(1, (u_end - u_beg + per_cta - 1) / per_cta);
    const unsigned grid = (unsigned)std::min<uint64_t>(want, (uint64_t)sm_count() * 3);  // 3 x 64 KiB per SM
    LRB_CUDA(cudaFuncSetAttribute(k_table_spectrum<FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSpecSmem));
    LRB_LAUNCH(name, st, k_table_spectrum<FULL><<<grid, kSpecThreads, kSpecSmem, st>>>(table, u_beg, u_end, e0_lo, e0_hi, e1_lo, e1_hi,
                                                                                      max_count, reinterpret_cast<unsigned long long*>(spectrum)));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_table_spectrum(const uint32_t* table, uint32_t key_lo, uint32_t key_hi, uint32_t max_count,
                                      uint64_t* spectrum, void* stream) {
    if (!table || !spectrum) return lrb_set_error(LRB_EINVAL, "lrb_dev_table_spectrum: null argument");
    if ((uintptr_t)table & 15u) return lrb_set_error(LRB_EINVAL, "lrb_dev_table_spectrum: the table must be 16-byte aligned");
    if (max_count < 2 || max_count > LRB_SPECTRUM_MAX_COUNT)
        return lrb_set_error(LRB_EINVAL, "lrb_dev_table_spectrum: max_count must be in [2, %u] (got %u)", LRB_SPECTRUM_MAX_COUNT, max_count);
    const uint64_t hi = std::min<uint64_t>(key_hi, kTableEntries);
    if (key_lo >= hi) return LRB_OK;
    const uint64_t ci_lo = canon_rank(key_lo), ci_hi = canon_rank(hi);
    if (ci_lo >= ci_hi) return LRB_OK;
    return launch_spectrum<true>("k_table_spectrum", table, ci_lo, ci_hi, max_count, spectrum, (cudaStream_t)stream);
}

extern "C" int lrb_dev_compact_spectrum(const uint32_t* compact, uint32_t max_count, uint64_t* spectrum, void* stream) {
    if (!compact || !spectrum) return lrb_set_error(LRB_EINVAL, "lrb_dev_compact_spectrum: null argument");
    if ((uintptr_t)compact & 15u) return lrb_set_error(LRB_EINVAL, "lrb_dev_compact_spectrum: the table must be 16-byte aligned");
    if (max_count < 2 || max_count > LRB_SPECTRUM_MAX_COUNT)
        return lrb_set_error(LRB_EINVAL, "lrb_dev_compact_spectrum: max_count must be in [2, %u] (got %u)", LRB_SPECTRUM_MAX_COUNT, max_count);
    return launch_spectrum<false>("k_table_spectrum_compact", compact, 0, LRB_COMPACT_ENTRIES, max_count, spectrum, (cudaStream_t)stream);
}

// ---- multi-GPU table exchange helpers (lrbinner_b200/dist.py: PeerExchange) -----------------------------------------
// dst rows (pitched) += sum of n_planes staged copies of the same rows (contiguous planes): 16-byte accesses, one pass.
__global__ void __launch_bounds__(256)
k_add_planes(uint4* __restrict__ dst, uint64_t dst_pitch4, const uint4* __restrict__ src, uint64_t plane4, int n_planes, uint32_t width4,
             uint64_t total4) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r = i / width4, c = i - r * width4;
        uint4 acc = dst[r * dst_pitch4 + c];
        for (int p = 0; p < n_planes; ++p) {
            const uint4 v = __ldcs(src + (uint64_t)p * plane4 + i);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        dst[r * dst_pitch4 + c] = acc;
    }
}

extern "C" int lrb_dev_add_planes(uint32_t* dst, uint64_t dst_pitch_words, const uint32_t* src, uint64_t plane_words, int n_planes,
                                  uint32_t width_words, uint32_t rows, void* stream) {
    if (!dst || !src) return lrb_set_error(LRB_EINVAL, "lrb_dev_add_planes: null argument");
    if ((width_words & 3u) || (dst_pitch_words & 3u) || (plane_words & 3u) || ((uintptr_t)dst & 15u) || ((uintptr_t)src & 15u))
        return lrb_set_error(LRB_EINVAL, "lrb_dev_add_planes: rows, pitches and pointers must be 16-byte aligned");
    if (!rows || !width_words || n_planes <= 0) return LRB_OK;
    const uint64_t total4 = (uint64_t)rows * (width_words / 4);
    const unsigned grid = (unsigned)std::min<uint64_t>((total4 + 255) / 256, (uint64_t)sm_count() * 16);
    LRB_LAUNCH("k_add_planes", (cudaStream_t)stream, k_add_planes<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<uint4*>(dst), dst_pitch_words / 4, reinterpret_cast<const uint4*>(src),
                                                         plane_words / 4, n_planes, width_words / 4, total4));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

// pitched device-to-device copy on the copy engines (src may be a peer's memory mapped into this process)
extern "C" int lrb_dev_copy2d(void* dst, uint64_t dpitch, const void* src, uint64_t spitch, uint64_t width_bytes, uint64_t height,
                              void* stream) {
    if (!dst || !src) return lrb_set_error(LRB_EINVAL, "lrb_dev_copy2d: null argument");
    if (!width_bytes || !height) return LRB_OK;
    LRB_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width_bytes, height, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return LRB_OK;
}

extern "C" int lrb_dev_fill_valid(const lrb_reads_view* dev, const uint32_t* exc_blk, const uint32_t* exc_valid, uint64_t n_exc,
                                  void* stream) {
    if (!dev || !dev->valid || (n_exc && (!exc_blk || !exc_valid))) return lrb_set_error(LRB_EINVAL, "lrb_dev_fill_valid: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t* valid = const_cast<uint32_t*>(dev->valid);
    if (dev->n_reads) {
        const uint64_t threads = dev->n_reads * 32;
        LRB_LAUNCH("k_default_valid", st, k_default_valid<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(*dev, valid));
    } else {
        LRB_CUDA(cudaMemsetAsync(valid, 0, sizeof(uint32_t) * (dev->n_blocks + 1), st));
    }
    if (n_exc) LRB_LAUNCH("k_patch_valid", st, k_patch_valid<<<(unsigned)((n_exc + 255) / 256), 256, 0, st>>>(exc_blk, exc_valid, n_exc, valid));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_search(const lrb_reads_view* dev, const uint32_t* table, long bin_size, int bins,
                              uint32_t* hist, uint32_t* sums, uint64_t tile_lo, uint64_t tile_hi, uint32_t key_lo,
                              uint32_t key_hi, void* stream) {
    if (!dev || !table || !hist || !sums) return lrb_set_error(LRB_EINVAL, "lrb_dev_search: null argument");
    if (bin_size <= 0) return lrb_set_error(LRB_EINVAL, "lrb_dev_search: bin_size must be >= 1 (the reference divides by it)");
    if (bins <= 0 || bins > LRB_MAX_BINS) return lrb_set_error(LRB_EINVAL, "lrb_dev_search: bins must be in [1, 4096]");
    if (tile_hi > dev->n_tiles) tile_hi = dev->n_tiles;
    if (tile_lo >= tile_hi || key_lo >= key_hi) return LRB_OK;
    const uint32_t S32 = bin_size > 0xFFFFFFFFl ? 0xFFFFFFFFu : (uint32_t)bin_size;
    const uint64_t magic = coverage_magic(S32);
    const uint64_t ntile = tile_hi - tile_lo;
    const unsigned grid = (unsigned)((ntile + kWarpsPerCta - 1) / kWarpsPerCta);
    const size_t smem = (size_t)kWarpsPerCta * (size_t)bins * sizeof(uint32_t);
    cudaStream_t st = (cudaStream_t)stream;
    const bool filter = !(key_lo == 0 && key_hi >= kTableEntries);
    if (smem > 48 * 1024) {
        LRB_CUDA(cudaFuncSetAttribute(k_search15<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        LRB_CUDA(cudaFuncSetAttribute(k_search15<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (filter)
        LRB_LAUNCH("k_search15", st, k_search15<true><<<grid, kCtaThreads, smem, st>>>(*dev, table, S32, magic, (uint32_t)bins, hist, sums, tile_lo, tile_hi, key_lo, key_hi));
    else
        LRB_LAUNCH("k_search15", st, k_search15<false><<<grid, kCtaThreads, smem, st>>>(*dev, table, S32, magic, (uint32_t)bins, hist, sums, tile_lo, tile_hi, key_lo, key_hi));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_pack_ascii(const lrb_reads_view* dev, const char* bases, const uint64_t* offsets, void* stream) {
    if (!dev || !bases || !offsets) return lrb_set_error(LRB_EINVAL, "lrb_dev_pack_ascii: null argument");
    if (dev->n_reads == 0) return LRB_OK;
    const uint64_t threads = dev->n_reads * 32;
    const unsigned grid = (unsigned)((threads + 255) / 256);
    LRB_LAUNCH("k_pack_ascii", (cudaStream_t)stream, k_pack_ascii<<<grid, 256, 0, (cudaStream_t)stream>>>(*dev, bases, offsets, const_cast<uint32_t*>(dev->codes),
                                                        const_cast<uint32_t*>(dev->valid)));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_format_composition(const uint32_t* counts, const uint32_t* read_len, uint64_t n_reads, int k,
                                          char* text, void* stream) {
    const int P = (k == 3) ? 32 : (k == 4) ? 136 : (k == 5) ? 512 : 0;
    if (!P || !text || (n_reads && (!counts || !read_len))) return lrb_set_error(LRB_EINVAL, "lrb_dev_format_composition: bad argument");
    if (!n_reads) return LRB_OK;
    const uint64_t total = n_reads * (uint64_t)P;
    LRB_LAUNCH("k_format_rows", (cudaStream_t)stream, k_format_rows<true><<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(counts, read_len, n_reads, (uint32_t)P, k, text));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_profile_values(const uint32_t* counts, const uint32_t* denom, uint64_t n_reads, int width, int k, double* out,
                                      void* stream) {
    if (width <= 0 || !out || (n_reads && (!counts || !denom))) return lrb_set_error(LRB_EINVAL, "lrb_dev_profile_values: bad argument");
    if (k != 0 && ((k == 3 ? 32 : k == 4 ? 136 : k == 5 ? 512 : 0) != width))
        return lrb_set_error(LRB_EINVAL, "lrb_dev_profile_values: width %d does not belong to k = %d", width, k);
    if (!n_reads) return LRB_OK;
    const uint64_t total = n_reads * (uint64_t)width;
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (k) LRB_LAUNCH("k_profile_values", (cudaStream_t)stream, k_profile_values<true><<<grid, 256, 0, (cudaStream_t)stream>>>(counts, denom, n_reads, (uint32_t)width, k, out));
    else LRB_LAUNCH("k_profile_values", (cudaStream_t)stream, k_profile_values<false><<<grid, 256, 0, (cudaStream_t)stream>>>(counts, denom, n_reads, (uint32_t)width, 0, out));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}

extern "C" int lrb_dev_format_coverage(const uint32_t* hist, const uint32_t* sums, uint64_t n_reads, int bins, char* text,
                                       void* stream) {
    if (bins <= 0 || !text || (n_reads && (!hist || !sums))) return lrb_set_error(LRB_EINVAL, "lrb_dev_format_coverage: bad argument");
    if (!n_reads) return LRB_OK;
    const uint64_t total = n_reads * (uint64_t)bins;
    LRB_LAUNCH("k_format_rows", (cudaStream_t)stream, k_format_rows<false><<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(hist, sums, n_reads, (uint32_t)bins, 0, text));
    LRB_CUDA(cudaGetLastError());
    return LRB_OK;
}
