// radix.cu -- stable radix partition passes over (key, payload) pairs, and a generic
// exclusive scan.  Two users:
//
//   * index build  (replaces quicksort/partition, /root/reference/src/index.c:25-46): four
//     8-bit LSD passes on the sign-flipped key give (values ascending, positions) with ties
//     in ascending row order -- the canonical stable order; identical to the reference's
//     unstable quicksort whenever keys are unique (SURVEY.md A3);
//   * hash join    (hash_join.cu): one or two passes on the top bits of a multiplicative
//     hash split both inputs into partitions small enough for a shared-memory table while
//     keeping the original row order inside every partition (stability is what makes the
//     join's output order reproducible); across GPUs, one pass groups keys by owner
//     (route_owner, any owner count);
//   * index build over several GPUs: one pass groups a shard's keys by the index slice that will
//     hold them (digit = number of splitters below the key), and rank_hist_kernel finds those
//     splitters exactly (a multi-target radix select).
//
// One pass = histogram (per-CTA, per-bucket counts) -> row scan of the [bucket][cta] matrix
// -> bucket bases -> stable scatter.  Inside the scatter a step covers 256 consecutive rows:
// lanes that share a bucket are ranked with match_any in lane order, warps are ordered
// through a small per-warp count table, so equal digits keep their input order.
#include "adb_common.cuh"

namespace adb {

constexpr int RX_THREADS = 256;
constexpr int RX_WARPS = RX_THREADS / kWarp;
constexpr int RX_BUCKETS = 256;


// f(key) of RadixPass::hash; the digit is (f >> shift) & mask.  For the signed order (HASH 0)
// the sign flip is folded into one constant xor-ed onto the extracted digit.
template <int HASH>
struct RxDigit {
    uint32_t shift, mask, flip;
    __host__ __device__ explicit RxDigit(const RadixPass &p)
        : shift((uint32_t)p.shift), mask((1u << p.bits) - 1u),
          flip(HASH == 0 ? ((0x80000000u >> p.shift) & ((1u << p.bits) - 1u)) : 0u) {}
    __device__ __forceinline__ uint32_t operator()(uint32_t key) const {
        if (HASH == 1) return ((key * 0x9E3779B1u) >> shift) & mask;
        return ((key >> shift) & mask) ^ flip;
    }
};
// digit = the key's owner among p.parts (any count, not only powers of two)
template <>
struct RxDigit<2> {
    uint32_t parts;
    __host__ __device__ explicit RxDigit(const RadixPass &p) : parts(p.parts) {}
    __device__ __forceinline__ uint32_t operator()(uint32_t key) const { return route_owner(key, parts); }
};
// digit = key / div, at most mask: floor(2^32 / div) as the multiplier is never more than one
// below the quotient
template <>
struct RxDigit<3> {
    uint32_t div, magic, mask;
    __host__ __device__ explicit RxDigit(const RadixPass &p)
        : div(p.div ? p.div : 1u), magic((uint32_t)(0x100000000ull / (p.div ? p.div : 1u) > 0xFFFFFFFFull
                                                        ? 0xFFFFFFFFull : 0x100000000ull / (p.div ? p.div : 1u))),
          mask((1u << p.bits) - 1u) {}
    __device__ __forceinline__ uint32_t operator()(uint32_t key) const {
        uint32_t q = __umulhi(key, magic);
        if ((unsigned long long)(q + 1) * div <= key) ++q;
        return min(q, mask);
    }
};

// digit = the index slice of the key: how many of the 15 sorted splitters lie below it (signed),
// a branchless binary search over L1-cached device memory
template <>
struct RxDigit<4> {
    const int32_t *split;
    __host__ __device__ explicit RxDigit(const RadixPass &p)
        : split(reinterpret_cast<const int32_t *>(((uint64_t)p.split_hi << 32) | (uint32_t)p.shift)) {}
    __device__ __forceinline__ uint32_t operator()(uint32_t key) const {
        static_assert(kRangeSplitters == 15, "the search below covers 8 + 4 + 2 + 1 splitters");
        uint32_t d = 0;
#pragma unroll
        for (uint32_t step = 8; step; step >>= 1)
            if (__ldg(split + d + step - 1) < (int32_t)key) d += step;
        return d;
    }
};

template <int HASH>
__global__ void __launch_bounds__(RX_THREADS)
rx_hist_kernel(const uint32_t *__restrict__ keys, uint32_t n, uint32_t rows_per_cta, RadixPass p,
               uint32_t seg_tiles, uint32_t *__restrict__ hist /* [segment][bucket][seg_tiles] */) {
    __shared__ uint32_t s_h[RX_BUCKETS];
    const RxDigit<HASH> digit(p);
    s_h[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t begin = blockIdx.x * rows_per_cta;
    const uint32_t end = min(n, begin + rows_per_cta);
    if (end - begin == rows_per_cta && (reinterpret_cast<uintptr_t>(keys) & 15) == 0 && (rows_per_cta & 3) == 0) {
        const int4 *k4 = reinterpret_cast<const int4 *>(keys + begin);
        for (uint32_t i = threadIdx.x; i < rows_per_cta / 4; i += RX_THREADS) {
            const int4 k = ld_stream(k4 + i);
            atomicAdd(&s_h[digit((uint32_t)k.x)], 1u);
            atomicAdd(&s_h[digit((uint32_t)k.y)], 1u);
            atomicAdd(&s_h[digit((uint32_t)k.z)], 1u);
            atomicAdd(&s_h[digit((uint32_t)k.w)], 1u);
        }
    } else {
        for (uint32_t i = begin + threadIdx.x; i < end; i += RX_THREADS)
            atomicAdd(&s_h[digit(keys[i])], 1u);
    }
    __syncthreads();
    const uint32_t seg = blockIdx.x / seg_tiles, t = blockIdx.x - seg * seg_tiles;
    hist[((size_t)seg * RX_BUCKETS + threadIdx.x) * seg_tiles + t] = s_h[threadIdx.x];
}

// Exclusive scan of every row of the [segment][bucket][seg_tiles] histogram in place; row totals
// out.  The last segment may hold fewer than seg_tiles tiles.
__global__ void __launch_bounds__(1024)
rx_row_scan_kernel(uint32_t *__restrict__ mat, uint32_t seg_tiles, uint32_t tiles, uint32_t *__restrict__ totals) {
    __shared__ uint32_t s_warp[32];
    uint32_t *row = mat + (size_t)blockIdx.x * seg_tiles;
    const uint32_t seg = blockIdx.x / RX_BUCKETS;
    const uint32_t cols = min(seg_tiles, tiles - seg * seg_tiles);
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t carry = 0;
    // four consecutive columns per thread and step: a 500 M-row pass has 122 K columns, and a
    // step costs three block barriers whatever it covers
    for (uint32_t base = 0; base < cols; base += 4096) {
        const uint32_t i = base + threadIdx.x * 4;
        uint32_t x[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) x[k] = i + k < cols ? row[i + k] : 0u;
        const uint32_t sum = x[0] + x[1] + x[2] + x[3];
        const uint32_t incl = warp_incl_scan(sum, lane);
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) s_warp[lane] = warp_incl_scan(s_warp[lane], lane);
        __syncthreads();
        uint32_t run = carry + (warp ? s_warp[warp - 1] : 0u) + incl - sum;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (i + k < cols) row[i + k] = run;
            run += x[k];
        }
        carry += s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = carry;
}

// The same for short rows (a segmented pass has 256 x segments rows of a few dozen tiles each:
// r02y, 65 K CTAs of 1024 threads for two columns took 278 us): one warp per row.
__global__ void __launch_bounds__(RX_THREADS)
rx_row_scan_warp_kernel(uint32_t *__restrict__ mat, uint32_t seg_tiles, uint32_t tiles, uint32_t rows,
                        uint32_t *__restrict__ totals) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t r = blockIdx.x * RX_WARPS + (threadIdx.x >> 5);
    if (r >= rows) return;
    uint32_t *row = mat + (size_t)r * seg_tiles;
    const uint32_t seg = r / RX_BUCKETS;
    const uint32_t cols = min(seg_tiles, tiles - seg * seg_tiles);
    uint32_t carry = 0;
    for (uint32_t base = 0; base < cols; base += kWarp) {
        const uint32_t i = base + lane;
        const uint32_t x = i < cols ? row[i] : 0u;
        const uint32_t incl = warp_incl_scan(x, lane);
        if (i < cols) row[i] = carry + incl - x;
        carry += __shfl_sync(kFull, incl, 31);
    }
    if (lane == 0) totals[r] = carry;
}

// base[seg][b] = first row of the segment + sum of totals[seg][0..b)  (one CTA of 256 threads
// per segment)
__global__ void rx_bucket_base_kernel(const uint32_t *__restrict__ totals_all, uint32_t *__restrict__ base_all,
                                      uint32_t seg_rows) {
    __shared__ uint32_t s_warp[RX_WARPS];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t *totals = totals_all + blockIdx.x * RX_BUCKETS;
    uint32_t *base = base_all + blockIdx.x * RX_BUCKETS;
    const uint32_t x = totals[threadIdx.x];
    const uint32_t incl = warp_incl_scan(x, lane);
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t wexcl = 0;
    for (uint32_t w = 0; w < warp; ++w) wexcl += s_warp[w];
    base[threadIdx.x] = blockIdx.x * seg_rows + wexcl + incl - x;
}

// Stable scatter, one 4096-row tile per CTA.  Warp w owns the contiguous rows
// tile + w*512 .. +512 (row = ... + i*32 + lane), so ranking its keys round by round gives
// every key its rank among the warp's equal digits in row order.  Per-digit prefixes over the
// eight warps and over the 256 digits turn that into a slot in the tile-sorted order; {key,
// payload} pairs are parked there in shared memory and written out slot by slot, so each
// digit's run leaves as one contiguous (coalesced) piece instead of thirty-two 4-byte scatters
// per warp.
//
// r02t (ncu, 200 M pairs, profiles/r02t_radix_summary.md): the first version of this kernel
// spent 159 warp instructions per 32 keys at 43 % issue utilisation and 37 % occupancy -- a
// run-time loop over the digit's bits around each ballot (9 instructions per bit), the digit
// recomputed with a run-time hash selector, the payload loaded after the ranking (38 % of the
// stall samples).  This version: hash, digit width and tile fullness are template parameters
// (4 instructions per bit, unrolled), the peer masks of all sixteen rounds are computed before
// the dependent counter chain, the payload tile travels global -> shared with cp.async while the
// ranking runs, pairs move through shared memory as 8-byte words, counters are 16-bit:
// 56 KB of shared memory and <= 64 registers = 4 CTAs per SM.
//
// (r01k tried finding the peers through a per-warp shared-memory table -- atomicOr of the
// lane bit, sync, read back, leader clears -- instead of one ballot per digit bit: 20.4 ms
// against 19.6 ms for the 500 M-key sort, so the ballots stayed.  MATCH.ANY: r01f, XU pipe bound.)
// REMOTE: bucket d is a destination rank and is written into that rank's receive buffer over
// NVLink (peer_base[d] + key_off / pay_off) instead of one local output array; `base` then
// holds the offset of this rank's piece inside every destination buffer.  The run-contiguous
// write-out is what makes the remote stores full 128-byte transactions.
constexpr int RX_TILE = (int)kRadixTile;                 // rows per tile = CTA threads x keys per thread
constexpr int RX_ST = RX_TILE / 16 < 256 ? 256 : RX_TILE / 16 > 512 ? 512 : RX_TILE / 16;   // scatter CTA threads (16 keys each at 4096 rows)
constexpr int RX_KPT = RX_TILE / RX_ST, RX_SWARPS = RX_ST / kWarp;
// CTA shape: 256 threads x 16 keys: 64 registers, 56 KB -> 4 CTAs = 32 warps per SM.  512 x 8 was
// measured and dropped: 40 registers, 60 KB -> 3 CTAs = 48 warps per SM, but 13.8 vs 12.0 ms per
// 500 M pairs (r02zc).  Other tile sizes (-DADB_RADIX_TILE, r02zn): 2048 rows x 8 keys per thread
// 17.3 ms (runs of 8 rows, twice the histogram), 8192 rows x 512 threads 12.7 ms.
struct RxShared {
    uint2 kv[RX_TILE];                                   // tile-sorted {key, payload}
    uint32_t pay_in[RX_TILE];                            // the tile's payloads in row order (cp.async)
    uint16_t wcnt[RX_SWARPS][RX_BUCKETS];                // per-warp digit counts -> first slot of (warp, digit)
    uint32_t gofs[RX_BUCKETS];                           // global address = gofs[d] + tile slot
    uint32_t ws[RX_BUCKETS / kWarp];
    uint32_t *peer[kMaxPeers];
};

__device__ __forceinline__ void cp_async_4(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <int HASH, int BITS, bool REMOTE, bool FULL>
__device__ __forceinline__ void rx_scatter_tile(RxShared &sh, const uint32_t *__restrict__ keys,
                                                const uint32_t *__restrict__ pay, uint32_t tile, uint32_t end,
                                                const RadixPass &p, uint32_t my_off, uint32_t *__restrict__ keys_out,
                                                uint32_t *__restrict__ pay_out, unsigned long long key_off,
                                                unsigned long long pay_off) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const RxDigit<HASH> digit(p);
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t wofs = warp * (kWarp * RX_KPT) + lane;  // row in tile of this lane's round-0 key
    const uint32_t wrow = tile + wofs;
    // the payload tile goes straight to shared memory while the keys are ranked
    if (pay) {
        if (FULL && (reinterpret_cast<uintptr_t>(pay) & 15) == 0) {
#pragma unroll
            for (int i = 0; i < RX_KPT / 4; ++i) {
                const uint32_t q = (i * RX_ST + threadIdx.x) * 4;
                cp_async_16(&sh.pay_in[q], pay + tile + q);
            }
        } else {
#pragma unroll
            for (int i = 0; i < RX_KPT; ++i)
                if (FULL || wrow + i * kWarp < end) cp_async_4(&sh.pay_in[wofs + i * kWarp], pay + wrow + i * kWarp);
        }
    }
    uint32_t key[RX_KPT];
#pragma unroll
    for (int i = 0; i < RX_KPT; ++i)
        key[i] = (FULL || wrow + i * kWarp < end)
                     ? (uint32_t)ld_stream(reinterpret_cast<const int32_t *>(keys) + wrow + i * kWarp) : 0u;
    {   // zero the per-warp counters: 4 KB = one 16-byte store per thread
        reinterpret_cast<uint4 *>(&sh.wcnt[0][0])[threadIdx.x] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    // 1a. lanes holding the same digit, one ballot per digit bit (MATCH.ANY runs on the XU pipe
    //     and saturated it, ncu r01f).  dr = digit | rank among the round's equal digits << 8 |
    //     size of that group << 16; 0xFFFFFFFF = past the end.
    uint32_t dr[RX_KPT];
#pragma unroll
    for (int i = 0; i < RX_KPT; ++i) {
        const bool live = FULL || wrow + i * kWarp < end;
        const uint32_t d = digit(key[i]);
        uint32_t peers = FULL ? kFull : __ballot_sync(kFull, live);
        if (BITS > 0) {
#pragma unroll
            for (int b = 0; b < BITS; ++b) peers = warp_match_bit(peers, d, 1u << b);
        } else {
            for (int b = 0; b < p.bits; ++b) {
                const bool bit = (d & (1u << b)) != 0u;
                const uint32_t vote = __ballot_sync(kFull, bit);
                peers &= bit ? vote : ~vote;
            }
        }
        dr[i] = live ? (d | ((uint32_t)__popc(peers & lt) << 8) | ((uint32_t)__popc(peers) << 16)) : 0xFFFFFFFFu;
    }
    // 1b. the dependent part: the warp's running count of every digit
    uint16_t *cnt = sh.wcnt[warp];
#pragma unroll
    for (int i = 0; i < RX_KPT; ++i) {
        const bool live = FULL || dr[i] != 0xFFFFFFFFu;
        const uint32_t d = dr[i] & 0xFFu, r = (dr[i] >> 8) & 0xFFu;
        uint32_t before = 0;
        if (live) before = cnt[d];
        __syncwarp();
        if (live && r == 0) cnt[d] = (uint16_t)(before + (dr[i] >> 16));
        __syncwarp();
        if (live) dr[i] = d | ((before + r) << 8);
    }
    __syncthreads();
    // 2. digit `threadIdx.x` (the first 256 threads): exclusive prefix over the warps, then over
    //    the digits
    {
        const bool digit_thread = RX_ST == RX_BUCKETS || threadIdx.x < RX_BUCKETS;
        uint32_t c[RX_SWARPS], tot = 0;
        if (digit_thread) {
#pragma unroll
            for (int w = 0; w < RX_SWARPS; ++w) { c[w] = sh.wcnt[w][threadIdx.x]; tot += c[w]; }
        }
        const uint32_t incl = warp_incl_scan(tot, lane);
        if (digit_thread && lane == 31) sh.ws[warp] = incl;
        __syncthreads();
        if (digit_thread) {
            uint32_t wexcl = 0;
#pragma unroll
            for (int w = 0; w < RX_BUCKETS / kWarp; ++w) wexcl += (uint32_t)w < warp ? sh.ws[w] : 0u;
            const uint32_t tbase = wexcl + incl - tot;      // first tile slot of this digit
            sh.gofs[threadIdx.x] = my_off - tbase;          // modular: slot >= tbase for this digit
            uint32_t run = tbase;
#pragma unroll
            for (int w = 0; w < RX_SWARPS; ++w) { sh.wcnt[w][threadIdx.x] = (uint16_t)run; run += c[w]; }
        }
    }
    if (pay) cp_async_wait_all();
    __syncthreads();
    // 3. park the pairs in tile-sorted order
#pragma unroll
    for (int i = 0; i < RX_KPT; ++i) {
        if (FULL || dr[i] != 0xFFFFFFFFu) {
            const uint32_t d = dr[i] & 0xFFu, r = dr[i] >> 8;
            const uint32_t slot = sh.wcnt[warp][d] + r;
            sh.kv[slot] = make_uint2(key[i], pay ? sh.pay_in[wofs + i * kWarp] : wrow + i * kWarp);
        }
    }
    __syncthreads();
    // 4. write out, run by run
    const uint32_t count = FULL ? (uint32_t)RX_TILE : end - tile;
#pragma unroll 4
    for (uint32_t slot = threadIdx.x; slot < count; slot += RX_ST) {
        const uint2 kv = sh.kv[slot];
        const uint32_t d = digit(kv.x);
        const uint32_t dst = sh.gofs[d] + slot;
        if (REMOTE) {
            uint32_t *pb = sh.peer[d];
            pb[key_off + dst] = kv.x;
            pb[pay_off + dst] = kv.y;
        } else {
            keys_out[dst] = kv.x;
            pay_out[dst] = kv.y;
        }
    }
}

template <int HASH, int BITS, bool REMOTE>
__global__ void __launch_bounds__(RX_ST, (RX_KPT >= 16 ? 1024 : 1536) / RX_ST)
rx_scatter_kernel(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ pay, uint32_t n,
                  RadixPass p, uint32_t seg_tiles, const uint32_t *__restrict__ hist,
                  const uint32_t *__restrict__ base,
                  uint32_t *__restrict__ keys_out, uint32_t *__restrict__ pay_out,
                  uint32_t *const *__restrict__ peer_base, unsigned long long key_off,
                  unsigned long long pay_off, const uint32_t *__restrict__ abort_flag) {
    extern __shared__ __align__(16) unsigned char rx_smem[];
    RxShared &sh = *reinterpret_cast<RxShared *>(rx_smem);
    if (REMOTE) {
        if (*abort_flag) return;                            // a receive region would overflow
        if (threadIdx.x < (1u << p.bits)) sh.peer[threadIdx.x] = peer_base[threadIdx.x];
    }
    // next free global slot of digit `threadIdx.x` for this tile
    const uint32_t seg = blockIdx.x / seg_tiles, t = blockIdx.x - seg * seg_tiles;
    uint32_t my_off = 0;
    if (RX_ST == RX_BUCKETS || threadIdx.x < RX_BUCKETS)
        my_off = base[seg * RX_BUCKETS + threadIdx.x] +
                 hist[((size_t)seg * RX_BUCKETS + threadIdx.x) * seg_tiles + t];
    const uint32_t tile = blockIdx.x * RX_TILE;
    if (tile + RX_TILE <= n)
        rx_scatter_tile<HASH, BITS, REMOTE, true>(sh, keys, pay, tile, n, p, my_off, keys_out, pay_out, key_off, pay_off);
    else
        rx_scatter_tile<HASH, BITS, REMOTE, false>(sh, keys, pay, tile, n, p, my_off, keys_out, pay_out, key_off, pay_off);
}

// One CTA per 4096-row tile, launched in row order: the CTAs resident at any moment work on
// neighbouring tiles, so each of the 256 output streams is appended to by many CTAs at
// neighbouring addresses (DRAM-page and L2 friendly) instead of every CTA opening its own 256
// far-apart streams.  The price is a [256][tiles] histogram (1 KB per 32 KB of input).
RadixGeom radix_geom(uint32_t n, int sm_count) {
    (void)sm_count;
    RadixGeom g{};
    g.rows_per_cta = RX_TILE;
    g.ctas = (n + RX_TILE - 1) / RX_TILE;
    if (g.ctas == 0) g.ctas = 1;
    return g;
}

// function attributes are per device: once per device the engine launches on
static void rx_set_attributes() {
    static bool done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (done[dev & 63]) return;
    auto allow = [](auto *kernel) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RxShared));
    };
    allow(&rx_scatter_kernel<0, 8, false>);
    allow(&rx_scatter_kernel<1, 8, false>);
    allow(&rx_scatter_kernel<0, 0, false>);
    allow(&rx_scatter_kernel<1, 0, false>);
    allow(&rx_scatter_kernel<2, 0, false>);
    allow(&rx_scatter_kernel<2, 0, true>);
    allow(&rx_scatter_kernel<3, 0, false>);
    allow(&rx_scatter_kernel<4, 0, false>);
    done[dev & 63] = true;
}

static void rx_launch_scatter(uint32_t ctas, const uint32_t *keys_in, const uint32_t *pay_in, uint32_t n, RadixPass p,
                              uint32_t seg_tiles, const uint32_t *hist, const uint32_t *base, uint32_t *keys_out,
                              uint32_t *pay_out, cudaStream_t s) {
    const size_t sm = sizeof(RxShared);
#define RX_LAUNCH(H, B)                                                                                      \
    rx_scatter_kernel<H, B, false><<<ctas, RX_ST, sm, s>>>(keys_in, pay_in, n, p, seg_tiles, hist, base, keys_out, \
                                                           pay_out, nullptr, 0, 0, nullptr)
    if (p.hash == 0 && p.bits == 8) RX_LAUNCH(0, 8);
    else if (p.hash == 1 && p.bits == 8) RX_LAUNCH(1, 8);
    else if (p.hash == 0) RX_LAUNCH(0, 0);
    else if (p.hash == 1) RX_LAUNCH(1, 0);
    else if (p.hash == 3) RX_LAUNCH(3, 0);
    else if (p.hash == 4) RX_LAUNCH(4, 0);
    else RX_LAUNCH(2, 0);
#undef RX_LAUNCH
}

static void launch_hist(const uint32_t *keys_in, uint32_t n, const RadixGeom &g, RadixPass p, uint32_t seg_tiles,
                        uint32_t *hist, cudaStream_t s) {
    if (p.hash == 1) rx_hist_kernel<1><<<g.ctas, RX_THREADS, 0, s>>>(keys_in, n, g.rows_per_cta, p, seg_tiles, hist);
    else if (p.hash == 2) rx_hist_kernel<2><<<g.ctas, RX_THREADS, 0, s>>>(keys_in, n, g.rows_per_cta, p, seg_tiles, hist);
    else if (p.hash == 3) rx_hist_kernel<3><<<g.ctas, RX_THREADS, 0, s>>>(keys_in, n, g.rows_per_cta, p, seg_tiles, hist);
    else if (p.hash == 4) rx_hist_kernel<4><<<g.ctas, RX_THREADS, 0, s>>>(keys_in, n, g.rows_per_cta, p, seg_tiles, hist);
    else rx_hist_kernel<0><<<g.ctas, RX_THREADS, 0, s>>>(keys_in, n, g.rows_per_cta, p, seg_tiles, hist);
}

// A pass over consecutive SEGMENTS of seg_tiles tiles each: every segment is partitioned on its
// own (its rows stay inside its row range), base[seg][d] = first output row of bucket d of
// segment seg.  seg_tiles >= tiles (or 0) is the plain pass.
uint32_t radix_segments(uint32_t n, uint32_t seg_tiles) {
    const uint32_t tiles = (n + RX_TILE - 1) / RX_TILE;
    if (seg_tiles == 0 || seg_tiles >= tiles) return 1;
    return (tiles + seg_tiles - 1) / seg_tiles;
}
uint32_t radix_seg_tiles(uint32_t n, uint32_t seg_tiles) {
    const uint32_t tiles = (n + RX_TILE - 1) / RX_TILE;
    return radix_segments(n, seg_tiles) == 1 ? (tiles ? tiles : 1) : seg_tiles;
}
size_t radix_hist_elems(uint32_t n, uint32_t seg_tiles) {
    const uint32_t tiles = (n + RX_TILE - 1) / RX_TILE;
    const uint32_t segs = radix_segments(n, seg_tiles);
    const uint32_t st = segs == 1 ? (tiles ? tiles : 1) : seg_tiles;
    return (size_t)segs * RX_BUCKETS * st;
}

// scratch: hist = radix_hist_elems(n, seg_tiles) uint32, totals = base = 256 * radix_segments()
int launch_radix_pass_segmented(const uint32_t *keys_in, const uint32_t *pay_in, uint32_t *keys_out,
                                uint32_t *pay_out, uint32_t n, RadixPass p, uint32_t seg_tiles, uint32_t *hist,
                                uint32_t *totals, uint32_t *base, int sm_count, cudaStream_t s) {
    if (n == 0) return 0;
    rx_set_attributes();
    const RadixGeom g = radix_geom(n, sm_count);
    const uint32_t segs = radix_segments(n, seg_tiles);
    if (segs == 1) seg_tiles = g.ctas;
    launch_hist(keys_in, n, g, p, seg_tiles, hist, s);
    if (seg_tiles <= 512)
        rx_row_scan_warp_kernel<<<(segs * RX_BUCKETS + RX_WARPS - 1) / RX_WARPS, RX_THREADS, 0, s>>>(
            hist, seg_tiles, g.ctas, segs * RX_BUCKETS, totals);
    else
        rx_row_scan_kernel<<<segs * RX_BUCKETS, 1024, 0, s>>>(hist, seg_tiles, g.ctas, totals);
    rx_bucket_base_kernel<<<segs, RX_BUCKETS, 0, s>>>(totals, base, seg_tiles * RX_TILE);
    rx_launch_scatter(g.ctas, keys_in, pay_in, n, p, seg_tiles, hist, base, keys_out, pay_out, s);
    return 4;
}

int launch_radix_pass(const uint32_t *keys_in, const uint32_t *pay_in, uint32_t *keys_out,
                      uint32_t *pay_out, uint32_t n, RadixPass p, uint32_t *hist, uint32_t *totals,
                      uint32_t *base, int sm_count, cudaStream_t s) {
    return launch_radix_pass_segmented(keys_in, pay_in, keys_out, pay_out, n, p, 0, hist, totals, base, sm_count, s);
}

int launch_radix_hist(const uint32_t *keys_in, uint32_t n, RadixPass p, uint32_t *hist, uint32_t *totals,
                      int sm_count, cudaStream_t s) {
    if (n == 0) {
        cudaMemsetAsync(totals, 0, sizeof(uint32_t) * RX_BUCKETS, s);
        return 0;
    }
    const RadixGeom g = radix_geom(n, sm_count);
    launch_hist(keys_in, n, g, p, g.ctas, hist, s);
    rx_row_scan_kernel<<<RX_BUCKETS, 1024, 0, s>>>(hist, g.ctas, g.ctas, totals);
    return 2;
}

int launch_radix_scatter_remote(const uint32_t *keys_in, const uint32_t *pay_in, uint32_t n, RadixPass p,
                                const uint32_t *hist, const uint32_t *base, uint32_t *const *peer_base,
                                unsigned long long key_off, unsigned long long pay_off,
                                const uint32_t *abort_flag, int sm_count, cudaStream_t s) {
    if (n == 0) return 0;
    if (p.hash != 2) return -1;                              // the routing hash is the only remote user
    rx_set_attributes();
    const RadixGeom g = radix_geom(n, sm_count);
    rx_scatter_kernel<2, 0, true><<<g.ctas, RX_ST, sizeof(RxShared), s>>>(
        keys_in, pay_in, n, p, g.ctas, hist, base, nullptr, nullptr, peer_base, key_off, pay_off, abort_flag);
    return 1;
}

// ---- multi-target radix select -----------------------------------------------------------------
// Round r of four: every key whose sign-flipped top 8r bits equal one of the (distinct) prefixes
// counts its next 8 bits in that prefix's histogram.  The host sums the contexts' histograms and
// narrows every target's prefix and remaining rank, so four streaming passes give exact order
// statistics.  The prefixes sit in shared memory (an indexed kernel-parameter array would be
// copied to local memory by every thread, DESIGN §3).
constexpr int RS_THREADS = 256;
__global__ void __launch_bounds__(RS_THREADS)
rank_hist_kernel(const int32_t *__restrict__ keys, uint32_t n, const uint32_t *__restrict__ prefixes, uint32_t n_pre,
                 uint32_t round, uint32_t *__restrict__ hist) {
    __shared__ uint32_t s_h[kMaxPeers * 256];
    __shared__ uint32_t s_pre[kMaxPeers];
    for (uint32_t i = threadIdx.x; i < n_pre * 256; i += RS_THREADS) s_h[i] = 0;
    if (threadIdx.x < n_pre) s_pre[threadIdx.x] = prefixes[threadIdx.x];
    __syncthreads();
    const uint32_t dshift = 24 - 8 * round;
    auto count = [&](int32_t key) {
        const uint32_t f = (uint32_t)key ^ 0x80000000u;
        const uint32_t top = round ? f >> (32 - 8 * round) : 0u;
        for (uint32_t i = 0; i < n_pre; ++i)
            if (s_pre[i] == top) {
                atomicAdd(&s_h[i * 256 + ((f >> dshift) & 255u)], 1u);
                break;
            }
    };
    // the unaligned head and the tail one key at a time, the rest 16 bytes at a time
    const uint32_t stride = gridDim.x * RS_THREADS;
    const uint32_t lead = min((uint32_t)((16 - (reinterpret_cast<uintptr_t>(keys) & 15)) & 15) / 4, n);
    const uint32_t n4 = (n - lead) / 4, tail = lead + 4 * n4;
    const int4 *k4 = reinterpret_cast<const int4 *>(keys + lead);
    for (uint32_t i = blockIdx.x * RS_THREADS + threadIdx.x; i < n4; i += stride) {
        const int4 k = ld_stream(k4 + i);
        count(k.x);
        count(k.y);
        count(k.z);
        count(k.w);
    }
    for (uint32_t i = blockIdx.x * RS_THREADS + threadIdx.x; i < lead + (n - tail); i += stride)
        count(keys[i < lead ? i : tail + (i - lead)]);
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n_pre * 256; i += RS_THREADS)
        if (s_h[i]) atomicAdd(&hist[i], s_h[i]);
}

int launch_rank_hist(const int32_t *keys, uint32_t n, const uint32_t *prefixes, uint32_t n_prefixes, uint32_t round,
                     uint32_t *hist, int sm_count, cudaStream_t s) {
    if (n == 0) return 0;
    uint32_t ctas = (n + RS_THREADS * 16 - 1) / (RS_THREADS * 16);
    if (ctas > (uint32_t)sm_count * 4) ctas = (uint32_t)sm_count * 4;
    rank_hist_kernel<<<ctas, RS_THREADS, 0, s>>>(keys, n, prefixes, n_prefixes, round, hist);
    return 1;
}

// ---- generic exclusive scan: out[i] = sum(in[0..i)), *total = sum(in[0..n)) -------------------
constexpr int SC_THREADS = 1024;

__global__ void __launch_bounds__(SC_THREADS)
sc_chunk_sum_kernel(const uint32_t *__restrict__ in, uint32_t in_stride, uint32_t n,
                    uint32_t rows_per_cta, unsigned long long *__restrict__ sums) {
    __shared__ unsigned long long s_w[32];
    const uint32_t begin = blockIdx.x * rows_per_cta, end = min(n, begin + rows_per_cta);
    unsigned long long acc = 0;
    for (uint32_t i = begin + threadIdx.x; i < end; i += SC_THREADS) acc += in[(size_t)i * in_stride];
    acc = (unsigned long long)warp_sum_i64((int64_t)acc);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < 32; ++w) t += s_w[w];
        sums[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(SC_THREADS)
sc_chunk_scan_kernel(const uint32_t *__restrict__ in, uint32_t in_stride, uint32_t n,
                     uint32_t rows_per_cta, const unsigned long long *__restrict__ sums,
                     uint32_t *__restrict__ out, int64_t *__restrict__ total) {
    __shared__ unsigned long long s_w[32];
    __shared__ uint32_t s_warp[32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long acc = 0;
    for (uint32_t c = threadIdx.x; c < blockIdx.x; c += SC_THREADS) acc += sums[c];
    acc = (unsigned long long)warp_sum_i64((int64_t)acc);
    if (lane == 0) s_w[warp] = acc;
    __syncthreads();
    unsigned long long base64 = 0;
    for (int w = 0; w < 32; ++w) base64 += s_w[w];
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *total = (int64_t)(base64 + sums[blockIdx.x]);
    uint32_t carry = (uint32_t)base64;                      // offsets fit 32 bits (total < 2^31 checked by caller)
    const uint32_t begin = blockIdx.x * rows_per_cta, end = min(n, begin + rows_per_cta);
    for (uint32_t b = begin; b < end; b += SC_THREADS) {
        const uint32_t i = b + threadIdx.x;
        const uint32_t x = i < end ? in[(size_t)i * in_stride] : 0u;
        const uint32_t incl = warp_incl_scan(x, lane);
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) s_warp[lane] = warp_incl_scan(s_warp[lane], lane);
        __syncthreads();
        const uint32_t wexcl = warp ? s_warp[warp - 1] : 0u;
        if (i < end) out[i] = carry + wexcl + incl - x;
        carry += s_warp[31];
        __syncthreads();
    }
}

// sums scratch: >= scan_ctas(n) entries of 8 bytes
uint32_t scan_ctas(uint32_t n, int sm_count) {
    uint32_t ctas = (n + 8191) / 8192;
    const uint32_t cap = (uint32_t)sm_count * 2u;
    if (ctas > cap) ctas = cap;
    return ctas ? ctas : 1;
}

int launch_exclusive_scan(const uint32_t *in, uint32_t in_stride, uint32_t *out, uint32_t n,
                          unsigned long long *sums, int64_t *total, int sm_count, cudaStream_t s) {
    if (n == 0) {
        cudaMemsetAsync(total, 0, sizeof(int64_t), s);
        return 0;
    }
    const uint32_t ctas = scan_ctas(n, sm_count);
    uint32_t rows = (n + ctas - 1) / ctas;
    rows = (rows + SC_THREADS - 1) / SC_THREADS * SC_THREADS;
    const uint32_t grid = (n + rows - 1) / rows;
    sc_chunk_sum_kernel<<<grid, SC_THREADS, 0, s>>>(in, in_stride, n, rows, sums);
    sc_chunk_scan_kernel<<<grid, SC_THREADS, 0, s>>>(in, in_stride, n, rows, sums, out, total);
    return 2;
}

// Load this file's kernels now (CUDA loads them lazily, on first launch): a first launch that
// has to load code while another context's kernel spin-waits for this one can stall behind it.
void preload_radix() {
    { auto *fp = &rx_hist_kernel<0>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_hist_kernel<1>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_hist_kernel<2>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_hist_kernel<3>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_hist_kernel<4>; preload_one(reinterpret_cast<const void *>(fp)); }
    preload_one(reinterpret_cast<const void *>(&rx_row_scan_kernel));
    preload_one(reinterpret_cast<const void *>(&rx_row_scan_warp_kernel));
    preload_one(reinterpret_cast<const void *>(&rx_bucket_base_kernel));
    { auto *fp = &rx_scatter_kernel<0, 8, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_scatter_kernel<1, 8, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_scatter_kernel<0, 0, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_scatter_kernel<1, 0, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_scatter_kernel<2, 0, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_scatter_kernel<2, 0, true>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_scatter_kernel<3, 0, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &rx_scatter_kernel<4, 0, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    preload_one(reinterpret_cast<const void *>(&rank_hist_kernel));
    preload_one(reinterpret_cast<const void *>(&sc_chunk_scan_kernel));
    preload_one(reinterpret_cast<const void *>(&sc_chunk_sum_kernel));
    rx_set_attributes();
}

}  // namespace adb
