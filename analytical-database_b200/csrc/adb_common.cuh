// adb_common.cuh -- device helpers shared by the operator kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "adb_engine.h"

namespace adb {

constexpr int kWarp = 32;
constexpr uint32_t kFull = 0xffffffffu;

// ---- streaming global accesses -------------------------------------------------------
// Column scans touch every byte exactly once: keep them out of L1 so the position
// lists / gather targets that *are* reused keep the cache.
__device__ __forceinline__ int4 ld_stream(const int4 *p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ int32_t ld_stream(const int32_t *p) {
    int32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
// Random accesses (gathers over position lists, hash-table probes): a miss of a plain load
// brings a whole 128-byte line in from DRAM on this part whatever the cache operator or
// cudaLimitMaxL2FetchGranularity says (profiles/r01c_gather_probe.md); the .L2::64B prefetch-size
// qualifier (SASS LDG.E.LTC64B) halves that to 64 bytes per miss (r01z: 5 M sparse hits
// 660 -> 340 MB of DRAM reads, 103 -> 82 us).
__device__ __forceinline__ int32_t ld_gather(const int32_t *p) {
    int32_t r;
    asm volatile("ld.global.nc.L2::64B.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 ld_gather(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L2::64B.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream(int4 *p, const int4 &v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x),
                 "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}

// ---- 64-bit status words for the decoupled look-back ------------------------------------
// One word carries {epoch, flag, value}; a single relaxed 64-bit access moves all three
// atomically, so no fence is needed between "value" and "flag".
__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// ---- programmatic dependent launch ----------------------------------------------------------
// The chain is a string of short kernels on one stream (0.31 ms + 0.13 ms per shard); a
// kernel launched with launch_pdl() may be scheduled while its predecessor drains and must
// call pdl_wait() before it reads or overwrites anything the predecessor touches.  Work that
// depends on nothing earlier (the first column tile of the predicate pass) goes before the
// wait.  pdl_launch_dependents() lets the successor's CTAs take the slots this grid frees.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem,
                              cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- warp primitives ------------------------------------------------------------------
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t x, uint32_t lane) {
#pragma unroll
    for (int d = 1; d < kWarp; d <<= 1) {
        uint32_t y = __shfl_up_sync(kFull, x, d);
        if (lane >= (uint32_t)d) x += y;
    }
    return x;
}
__device__ __forceinline__ uint32_t warp_sum(uint32_t x) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(kFull, x, d);
    return x;
}
__device__ __forceinline__ int64_t warp_sum_i64(int64_t x) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x += __shfl_xor_sync(kFull, x, d);
    return x;
}
__device__ __forceinline__ int32_t warp_min_i32(int32_t x) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x = min(x, __shfl_xor_sync(kFull, x, d));
    return x;
}
__device__ __forceinline__ int32_t warp_max_i32(int32_t x) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) x = max(x, __shfl_xor_sync(kFull, x, d));
    return x;
}

// peers &= lanes whose digit agrees with mine in the bit `bitmask`.  Spelled out in PTX: from
// the C form nvcc derives two predicates per bit (bit != 0 for the select, bit != 1 for the
// vote) through a shift, an and and a compare -- six instructions where four do.
__device__ __forceinline__ uint32_t warp_match_bit(uint32_t peers, uint32_t d, uint32_t bitmask) {
    asm("{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b32 t, v;\n\t"
        "and.b32 t, %1, %2;\n\t"
        "setp.ne.u32 p, t, 0;\n\t"
        "vote.sync.ballot.b32 v, p, 0xffffffff;\n\t"
        "selp.b32 t, 0, 0xffffffff, p;\n\t"
        "lop3.b32 %0, %0, v, t, 0x60;\n\t"
        "}"
        : "+r"(peers) : "r"(d), "r"(bitmask));
    return peers;
}

// lanes (of `active`) that hold the same 8-bit value as this one
__device__ __forceinline__ uint32_t warp_match8(uint32_t active, uint32_t v) {
    uint32_t peers = active;
#pragma unroll
    for (int b = 0; b < 8; ++b) peers = warp_match_bit(peers, v, 1u << b);
    return peers;
}

// ---- range predicate -------------------------------------------------------------------
// The reference tests `v >= low && v < high` with either bound optional
// (src/query.c:97-127).  Host code folds that into an inclusive pair [lo, hi_incl]:
// absent low -> INT32_MIN, absent high -> INT32_MAX, high == INT32_MIN or lo > hi_incl ->
// the canonical empty range (1, 0).  Exact for every int32 input.
struct Range {
    int32_t lo, hi_incl;
};
__device__ __forceinline__ bool in_range(int32_t v, const Range &r) {
    return v >= r.lo && v <= r.hi_incl;
}

// ---- aggregate exchange over NVLink peer memory (peer_agg.cu, and the epilogue of the fused
// chain kernel) ------------------------------------------------------------------------------
// One 32-byte record per (bank, source rank) in every rank's mailbox; box[r] is rank r's
// mailbox as mapped into this process (cudaIpcOpenMemHandle; box[rank] is the local
// allocation itself).
constexpr int kMaxPeers = ADB_MAX_PEERS;
struct PeerRecord {
    int64_t sum, count;
    int32_t min, max;
    uint32_t epoch, pad;
};
struct PeerBoxes {
    PeerRecord *box[kMaxPeers];
};
// The whole mailbox: the aggregate records first (box[r] points here), then the control words
// of the join's pair exchange (peer_exchange.cu): every rank's per-destination pair counts
// and two rows of epoch flags.
struct PeerCtl {
    PeerRecord agg[2][kMaxPeers];
    uint32_t jcnt[2][kMaxPeers][kMaxPeers];          // [bank][source rank][destination rank]
    uint32_t jcnt_epoch[2][kMaxPeers];               // [bank][source]: its count row has landed
    uint32_t jdone_epoch[2][kMaxPeers];              // [bank][source]: its pairs have landed
};
constexpr size_t kPeerBoxBytes = sizeof(PeerCtl);
constexpr unsigned long long kPeerTimeoutNs = 2000000000ull;      // 2 s

// What a kernel needs to finish an aggregate across ranks: world == 0 disables it.
struct PeerExchange {
    const PeerBoxes *boxes;       // in DEVICE memory: an array inside a kernel parameter would be
                                  // copied to every thread's local memory as soon as it is indexed
    int32_t rank, world;
    uint32_t epoch;
    const adb_agg *parts;         // this rank's shard partials, all folded in before the exchange
    int32_t k;
    adb_agg *final_out;           // table-wide aggregate, identical on every rank
};

__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// ---- aggregate accumulator + the block -> grid fold shared by aggregate_kernel and the
// fused chain kernel --------------------------------------------------------------------------
struct AggAcc {
    int64_t sum;
    int32_t mn, mx;
    __device__ __forceinline__ void add(int32_t v) {
        sum += v;
        mn = min(mn, v);
        mx = max(mx, v);
    }
    __device__ __forceinline__ void add4(const int4 &v) {
        // pairwise int64 adds keep the carry chain short
        sum += ((int64_t)v.x + (int64_t)v.y) + ((int64_t)v.z + (int64_t)v.w);
        mn = min(min(mn, v.x), min(v.y, min(v.z, v.w)));
        mx = max(max(mx, v.x), max(v.y, max(v.z, v.w)));
    }
};

// One full warp, converged.  Folds this rank's k shard partials, stores the result into every
// rank's mailbox (payload, then the epoch with st.release.sys), acquire-spins on its own
// mailbox until every rank's record of this epoch has arrived, folds them in rank order and
// writes the table-wide aggregate (count = -1 if a peer did not arrive within 2 s).  Two
// banks suffice: a peer can only start epoch e+2 after it received this rank's e+1 record,
// which is sent after this rank has finished reading bank e.
__device__ __forceinline__ void peer_exchange_warp(const PeerExchange &px, int lane) {
    AggAcc g{0, INT32_MAX, INT32_MIN};
    int64_t cnt = 0;
    for (int i = lane; i < px.k; i += kWarp) {
        const volatile adb_agg *p = px.parts + i;           // just written by this grid: no .nc path
        g.sum += p->sum;
        cnt += p->count;
        g.mn = min(g.mn, p->min);
        g.mx = max(g.mx, p->max);
    }
    g.sum = warp_sum_i64(g.sum);
    cnt = warp_sum_i64(cnt);
    g.mn = warp_min_i32(g.mn);
    g.mx = warp_max_i32(g.mx);
    const uint32_t bank = px.epoch & 1u;
    if (lane < px.world) {
        PeerRecord *dst = px.boxes->box[lane] + bank * kMaxPeers + px.rank;
        volatile PeerRecord *v = dst;
        v->sum = g.sum;
        v->count = cnt;
        v->min = g.mn;
        v->max = g.mx;
        st_release_sys(&dst->epoch, px.epoch);
    }
    AggAcc f{0, INT32_MAX, INT32_MIN};
    int64_t fc = 0;
    bool ok = true;
    if (lane < px.world) {
        PeerRecord *src = px.boxes->box[px.rank] + bank * kMaxPeers + lane;
        const unsigned long long t0 = global_ns();
        while (ld_acquire_sys(&src->epoch) != px.epoch) {
            if (global_ns() - t0 > kPeerTimeoutNs) { ok = false; break; }
            __nanosleep(32);
        }
        const volatile PeerRecord *v = src;
        f.sum = v->sum;
        fc = v->count;
        f.mn = v->min;
        f.mx = v->max;
    }
    ok = __all_sync(kFull, ok);
    f.sum = warp_sum_i64(f.sum);
    fc = warp_sum_i64(fc);
    f.mn = warp_min_i32(f.mn);
    f.mx = warp_max_i32(f.mx);
    if (lane == 0) *px.final_out = ok ? adb_agg{f.sum, fc, f.mn, f.mx} : adb_agg{0, -1, INT32_MAX, INT32_MIN};
}

// Every thread of every CTA calls this once with its private accumulator and its share of
// the tuple count.  Warp shuffles -> one partial per CTA in `scratch` -> the last CTA to
// arrive (ticket) folds all partials in a fixed order and writes *out.  The ticket re-arms
// itself, so back-to-back launches on one stream need no reset.  Returns true in (every thread
// of) that last CTA, which may go on to exchange the aggregate with the peers.
template <int THREADS>
__device__ __forceinline__ bool agg_grid_fold(AggAcc acc, int64_t cnt, adb_agg *__restrict__ out,
                                              adb_agg *scratch, unsigned int *ticket) {
    constexpr int W = THREADS / kWarp;
    __shared__ int64_t s_sum[W], s_cnt[W];
    __shared__ int32_t s_mn[W], s_mx[W];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    acc.sum = warp_sum_i64(acc.sum);
    cnt = warp_sum_i64(cnt);
    acc.mn = warp_min_i32(acc.mn);
    acc.mx = warp_max_i32(acc.mx);
    if (lane == 0) { s_sum[warp] = acc.sum; s_cnt[warp] = cnt; s_mn[warp] = acc.mn; s_mx[warp] = acc.mx; }
    __syncthreads();
    if (warp == 0) {
        AggAcc b{lane < W ? s_sum[lane] : 0, lane < W ? s_mn[lane] : INT32_MAX,
                 lane < W ? s_mx[lane] : INT32_MIN};
        int64_t c = lane < W ? s_cnt[lane] : 0;
        b.sum = warp_sum_i64(b.sum);
        c = warp_sum_i64(c);
        b.mn = warp_min_i32(b.mn);
        b.mx = warp_max_i32(b.mx);
        if (lane == 0) {
            scratch[blockIdx.x] = adb_agg{b.sum, c, b.mn, b.mx};
            __threadfence();
            const unsigned int done = atomicAdd(ticket, 1u);
            s_last = (done == gridDim.x - 1);
        }
    }
    __syncthreads();
    if (!s_last) return false;
    __threadfence();
    AggAcc g{0, INT32_MAX, INT32_MIN};
    int64_t gc = 0;
    for (unsigned int k = threadIdx.x; k < gridDim.x; k += THREADS) {
        const volatile adb_agg *p = scratch + k;        // written by other CTAs: no .nc path
        g.sum += p->sum;
        gc += p->count;
        g.mn = min(g.mn, p->min);
        g.mx = max(g.mx, p->max);
    }
    g.sum = warp_sum_i64(g.sum);
    gc = warp_sum_i64(gc);
    g.mn = warp_min_i32(g.mn);
    g.mx = warp_max_i32(g.mx);
    __syncthreads();
    if (lane == 0) { s_sum[warp] = g.sum; s_cnt[warp] = gc; s_mn[warp] = g.mn; s_mx[warp] = g.mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        AggAcc f{0, INT32_MAX, INT32_MIN};
        int64_t fc = 0;
        for (int w = 0; w < W; ++w) {
            f.sum += s_sum[w];
            fc += s_cnt[w];
            f.mn = min(f.mn, s_mn[w]);
            f.mx = max(f.mx, s_mx[w]);
        }
        *out = adb_agg{f.sum, fc, f.mn, f.mx};
        *ticket = 0;                                    // re-arm for the next launch
    }
    return true;
}

// splitmix64 finaliser: the counter-based generator behind adb_synth_uniform
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t seed, uint64_t idx) {
    uint64_t z = seed + (idx + 1) * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

}  // namespace adb

// ---- engine-internal launch interface (engine.cu <-> kernel files) --------------------
namespace adb {
inline void preload_one(const void *kernel) {
    cudaFuncAttributes attr;
    cudaFuncGetAttributes(&attr, kernel);
    cudaGetLastError();
}
void preload_csv_load();
void preload_format_text();
void preload_gather_agg();
void preload_hash_join();
void preload_index_lookup();
void preload_index_ties();
void preload_peer_agg();
void preload_peer_exchange();
void preload_radix();
void preload_select_scan();
void preload_shared_scan();
}  // namespace adb

// Every launch_* returns the number of kernels it enqueued (0 for an empty input).
namespace adb {

struct SelectArgs {
    const int32_t *val;       // values the predicate reads
    const int32_t *pos_in;    // paired positions (select_pairs) or nullptr
    const int64_t *d_n;       // optional device-side length
    uint32_t n;               // host-side length / upper bound (< 2^31)
    bool stable_val;          // val is a base column: no kernel ever writes it (early first-tile request)
    Range range;
    int32_t base_pos;
    int32_t *out;
    int64_t *d_count;
    uint32_t *mask;               // selection bitmap scratch (select_mask_words() words)
    uint32_t *counts;             // per-warp-chunk hit counts (kMaxSelectChunks)
    int sm_count;
    // fused chain (launch_select_expand_fetch_agg): gather + aggregate while expanding
    const int32_t *fetch_col;     // values gathered at every emitted row
    int32_t *val_out;
    adb_agg *agg_out, *agg_scratch;
    unsigned int *agg_ticket;
    PeerExchange px;              // world != 0: the chain kernel finishes with the cross-rank exchange
    // Small results go to the host through a mapped pinned mailbox (engine.cu read_back).  When
    // pub is set, the kernel that produces the count / the aggregate stores it there itself
    // (payload words, fence, then the sequence number at pub[kMboxWords]) and no separate
    // publish kernel is launched.
    unsigned long long *pub;
    unsigned long long pub_seq;
    unsigned int *mask_ticket;    // set: the predicate kernel of a count phase totals the counts itself
};
constexpr uint32_t kMboxWords = 256;                  // 2 KB: 150 batch counts fit
__device__ __forceinline__ void mbox_publish(volatile unsigned long long *pub, unsigned long long seq,
                                             const unsigned long long *words, int n) {
    for (int i = 0; i < n; ++i) pub[i] = words[i];
    __threadfence_system();
    pub[kMboxWords] = seq;
}
// two-phase form: mask + per-chunk counts (+ total into a.d_count), then expand into a.out
int launch_select_mask(const SelectArgs &a, bool with_total, cudaStream_t s);
int launch_select_expand(const SelectArgs &a, cudaStream_t s);
int launch_select_expand_fetch_agg(const SelectArgs &a, cudaStream_t s);     // a.out == a.val_out == NULL: aggregate only
int launch_scan_gather_agg(const SelectArgs &a, cudaStream_t s);
size_t select_mask_words(uint32_t n, int sm_count);
constexpr uint32_t kMaxSelectChunks = 1u << 16;

int launch_fetch(const int32_t *col, const int32_t *pos, int64_t n_max, const int64_t *d_n,
                  int32_t base_pos, int32_t *out, int sm_count, cudaStream_t s);
// a column row-range sharded over several contexts / devices: shard k holds rows
// [k * shard_rows, (k + 1) * shard_rows); remote shards are peer-mapped
struct ShardTable {
    const int32_t *ptr[kMaxPeers];
};
int launch_fetch_sharded(const ShardTable &t, int n_shards, uint32_t shard_rows, const int32_t *pos,
                         int64_t n_max, const int64_t *d_n, int32_t *out, int sm_count, cudaStream_t s);
int launch_aggregate(const int32_t *v, int64_t n_max, const int64_t *d_n, adb_agg *out,
                      adb_agg *scratch, unsigned int *ticket, int sm_count, cudaStream_t s);
int launch_agg_combine(const adb_agg *parts, int32_t k, adb_agg *out, cudaStream_t s);
int launch_agg_export(const adb_agg *a, int64_t *sum_count, int32_t *max_notmin, cudaStream_t s);
int launch_agg_import(const int64_t *sum_count, const int32_t *max_notmin, adb_agg *a, cudaStream_t s);
int launch_ewise(const int32_t *a, const int32_t *b, int64_t n_max, const int64_t *d_n,
                  int32_t *out, bool subtract, int sm_count, cudaStream_t s);
int launch_synth_uniform(int32_t *out, int64_t n, uint64_t seed, uint64_t first_row, int32_t lo,
                          uint32_t span, int sm_count, cudaStream_t s);
int launch_narrow_u64(const unsigned long long *src, int64_t n, int32_t *dst, int sm_count, cudaStream_t s);
int launch_scatter_value(int32_t *col, int64_t n_rows, const int32_t *pos, int64_t n, int32_t base, int32_t value,
                         int sm_count, cudaStream_t s);
int launch_mark_rows(uint32_t *dead, int64_t n_rows, const int32_t *pos, int64_t n, int32_t base, int sm_count,
                     cudaStream_t s);
int launch_compact_rows(const int32_t *col, const uint32_t *dead, const uint32_t *dead_before, int64_t n_rows,
                        int32_t *out, int sm_count, cudaStream_t s);
int launch_synth_affine(int32_t *out, int64_t n, uint64_t first_row, uint64_t mul, uint64_t add, uint64_t modulus,
                        int sm_count, cudaStream_t s);
int launch_iota(int32_t *out, int64_t n, int32_t first, int sm_count, cudaStream_t s);
int launch_widen_i32(const int32_t *src, int64_t n, unsigned long long *dst, int sm_count, cudaStream_t s);
// counts: 128 uint64 (zeroed by the launcher)
int launch_histogram(const int32_t *v, int64_t n, int32_t vmin, int32_t bin_size, unsigned long long *counts,
                     int sm_count, cudaStream_t s);
constexpr int kAggMaxBlocks = 148 * 8;
int launch_agg_combine_allreduce(const PeerExchange &px, cudaStream_t s);

// Pair exchange of the sharded hash join over NVLink peer memory (peer_exchange.cu + the
// REMOTE flavour of the radix scatter): counts all-gather -> every rank scatters its routed
// pairs straight into the destination ranks' receive buffers -> done flags.
struct PairExchange {
    const PeerBoxes *boxes;       // device table of the peers' mailboxes
    int32_t rank, world;
    uint32_t epoch;
    unsigned long long cap;       // pairs a receive region holds
};
// status[0]: 0 ok, 1 a receive region would overflow, 2 a peer did not arrive
int launch_jx_counts(const PairExchange &x, const uint32_t *my_totals, uint32_t *base_out,
                     int64_t *recv_total_out, uint32_t *status, cudaStream_t s);
int launch_jx_done(const PairExchange &x, uint32_t *status, cudaStream_t s);


// Batched shared scan (shared_scan.cu).  All pointers are device addresses.
struct SharedScanPlan {
    const int32_t *bounds;     // m ascending distinct bounds
    const uint16_t *cov_off;   // m + 2 CSR offsets: interval k covers cov_q[cov_off[k] .. cov_off[k+1])
    const uint8_t *cov_q;      // covering query ids, ascending inside an interval
    uint32_t m;
    uint32_t q_count;
    // host-built lookup tables over d = v - lo, d in [0, span):
    const uint16_t *lut;       // kSsLut + 1 entries: bounds below the edge of bucket d >> lut_shift
                               // (bit 15: no query reaches into the bucket)
    const uint32_t *bits;      // kSsBits bits: bucket d >> bit_shift is touched by some query
    uint32_t lut_shift, bit_shift;
    int32_t lo;                // bounds[0]
    uint32_t span;             // bounds[m-1] - bounds[0]
    // query q covers the contiguous interval ids q_first[q] .. q_last[q] (first >= 1; first >
    // last for an empty query): its hit count is a difference of interval-count prefix sums
    const uint16_t *q_first, *q_last;
    // pair lists: when no value is covered by more than a few queries the classify pass lists
    // one {query, row} entry per (row, covering query) pair -- list_rows = chunk_rows * deepest
    // cover entries per chunk -- and the emit pass never looks an interval up; 0 = the chunk
    // lists hold one {interval, row} entry per hit row (heavily overlapping batches)
    uint32_t pair_depth;
    const uint32_t *cov4;      // per interval id: its covering queries by colour, one byte each, 0xFF = none
};
constexpr uint32_t kSsLut = 1024;
constexpr uint32_t kSsBits = 1u << 16;
struct SharedScanGeom {
    uint32_t chunk_rows, num_chunks, grid;
};
SharedScanGeom shared_scan_geom(uint32_t n, int sm_count);
int launch_shared_classify(const int32_t *val, uint32_t n, const SharedScanPlan &plan,
                           const SharedScanGeom &g, uint32_t *hitlist, uint32_t *chunk_hits,
                           uint32_t *counts, int64_t *totals, cudaStream_t s);
int launch_shared_emit(const uint32_t *hitlist, const uint32_t *chunk_hits,
                       const SharedScanPlan &plan, const SharedScanGeom &g, const uint32_t *offsets,
                       int32_t *const *outs, int64_t capacity, uint32_t base_pos, cudaStream_t s);

// Rows per tile of a radix pass (one CTA); the join's partitioned probe gathers its results back
// tile by tile and reads the tiles' places from the pass' histogram, so it shares the constant.
#ifndef ADB_RADIX_TILE
#define ADB_RADIX_TILE 4096
#endif
constexpr uint32_t kRadixTile = ADB_RADIX_TILE;
// Owner of a key among `parts` owners (the multi-GPU exchange's routing): the routing hash
// h = key * 0x85EBCA6B scaled to [0, parts), floor(h * parts / 2^32).  Every owner takes
// floor(2^32 / parts) or that + 1 of the hash values; for parts = 2^k it is h >> (32 - k), the top
// k bits.  The routing pass and the sharded expansion both call this, so a key is always looked
// up on the owner it was sent to.
__device__ __forceinline__ uint32_t route_owner(uint32_t key, uint32_t parts) {
    return __umulhi(key * 0x85EBCA6Bu, parts);
}

// Stable radix partition passes + generic exclusive scan (radix.cu).
struct RadixPass {
    int shift, bits;           // digit = (f(key) >> shift) & ((1 << bits) - 1), bits <= 8
    int hash;                  // f = key ^ 0x80000000 (0: signed order) or key * 0x9E3779B1 (1: join
                               // hash); 2: digit = route_owner(key, parts) (multi-GPU exchange;
                               // shift unused, bits = ceil(log2 parts) so the histograms hold it);
                               // 3: digit = key / div (the shard a row number lives on; shift unused)
                               // 4: digit = #{splitters < key}, signed (the index slice a key
                               // belongs to): 15 nondecreasing int32 splitters in device memory,
                               // padded with INT32_MAX; their address is carried in shift (low
                               // half) and split_hi, so the struct keeps the size every other
                               // pass' kernels take as a parameter
    union {
        uint32_t div = 1;      // hash 3
        uint32_t parts;        // hash 2: the owner count, 1 .. 256
        uint32_t split_hi;     // hash 4
    };
};
constexpr int kRangeSplitters = 15;          // hash 4: slices 0 .. 15 = up to kMaxPeers destinations
struct RadixGeom {
    uint32_t rows_per_cta, ctas;
};
RadixGeom radix_geom(uint32_t n, int sm_count);
int launch_radix_pass(const uint32_t *keys_in, const uint32_t *pay_in, uint32_t *keys_out,
                      uint32_t *pay_out, uint32_t n, RadixPass p, uint32_t *hist, uint32_t *totals,
                      uint32_t *base, int sm_count, cudaStream_t s);
// The pass over consecutive segments of seg_tiles 4096-row tiles, each partitioned inside its own
// row range; base[seg * 256 + d] = first output row of bucket d of segment seg (the join's
// partitioned probe: segments = probe-row windows, buckets = table partitions).  totals and
// base: 256 * radix_segments() words, hist: radix_hist_elems() words.
uint32_t radix_segments(uint32_t n, uint32_t seg_tiles);
uint32_t radix_seg_tiles(uint32_t n, uint32_t seg_tiles);   // tiles per segment the pass really uses (all of them when unsegmented)
size_t radix_hist_elems(uint32_t n, uint32_t seg_tiles);
int launch_radix_pass_segmented(const uint32_t *keys_in, const uint32_t *pay_in, uint32_t *keys_out,
                                uint32_t *pay_out, uint32_t n, RadixPass p, uint32_t seg_tiles, uint32_t *hist,
                                uint32_t *totals, uint32_t *base, int sm_count, cudaStream_t s);
// The same pass split in two for the peer exchange: histogram + per-tile offsets + totals, then
// a scatter whose bucket d is written into peer_base[d] + key_off / pay_off (uint32 units) at
// the offsets `base` holds (skipped when *abort_flag != 0).
int launch_radix_hist(const uint32_t *keys_in, uint32_t n, RadixPass p, uint32_t *hist, uint32_t *totals,
                      int sm_count, cudaStream_t s);
int launch_radix_scatter_remote(const uint32_t *keys_in, const uint32_t *pay_in, uint32_t n, RadixPass p,
                                const uint32_t *hist, const uint32_t *base, uint32_t *const *peer_base,
                                unsigned long long key_off, unsigned long long pay_off,
                                const uint32_t *abort_flag, int sm_count, cudaStream_t s);
// One round of the multi-target radix select: hist[i * 256 + digit] += keys whose sign-flipped
// value f = key ^ 0x80000000 has top 8 * round bits equal to prefixes[i] and next 8 bits = digit
// (round 0..3; n_prefixes <= kMaxPeers distinct prefixes; hist zeroed by the caller).
int launch_rank_hist(const int32_t *keys, uint32_t n, const uint32_t *prefixes, uint32_t n_prefixes, uint32_t round,
                     uint32_t *hist, int sm_count, cudaStream_t s);
uint32_t scan_ctas(uint32_t n, int sm_count);
// in_stride: distance (in uint32) between consecutive inputs (2 reads the .y of a uint2 array)
int launch_exclusive_scan(const uint32_t *in, uint32_t in_stride, uint32_t *out, uint32_t n,
                          unsigned long long *sums, int64_t *total, int sm_count, cudaStream_t s);

// The reference quicksort's tie order (index_ties.cu).  A big segment [lo, hi] of one level
// owns tiles tbase .. tbase + ceil((hi - lo + 1) / kTiesTile); small ones (<= kTiesSmall rows)
// are sorted by one CTA each.  `big` of TiesCounters = segments << 32 | tiles.
constexpr uint32_t kTiesTile = 4096;
constexpr uint32_t kTiesSmall = 4096;
struct TiesBig {
    uint32_t lo, hi, tbase, pad;
};
struct TiesCounters {
    unsigned long long big;
    uint32_t small, pad;
};
struct TiesLevel {
    const int32_t *keys;           // K: the sorted keys
    const uint32_t *dex;           // dex[k] = #{i < k : K[i + 1] == K[i]}
    const int32_t *cv;             // this level's (values, positions)
    const uint32_t *cp;
    int32_t *nv;                   // the next level's
    uint32_t *np;
    uint32_t *ev;                  // partition events, at the segment's own rows
    uint32_t *pos_out;             // final positions
    const TiesBig *big;
    uint32_t nbig, ntiles;
    const uint2 *small;
    uint32_t nsmall;
    uint4 *tile_cnt;               // per tile: L rows, descents, first push
    uint32_t *tile_pre;            // per tile: L rows of the segment's earlier tiles
    uint4 *info;                   // per big segment: mode, nL, lead, rotations
    TiesBig *big_next;
    uint2 *small_next;
    TiesCounters *ctr_next;        // zeroed before the level
};
int launch_ties_dups(const int32_t *keys, uint32_t n, uint32_t *flags, unsigned long long *count, int sm_count,
                     cudaStream_t s);
int launch_ties_init(const int32_t *col, uint32_t n, int32_t *cv, uint32_t *cp, TiesBig *big, uint2 *small,
                     int sm_count, cudaStream_t s);
int launch_ties_level(const TiesLevel &a, cudaStream_t s);

// Bulk CSV load (csv_load.cu).
uint32_t csv_blocks(size_t bytes);
int launch_csv_count(const unsigned char *text, size_t bytes, uint32_t *block_counts, cudaStream_t s);
int launch_csv_index(const unsigned char *text, size_t bytes, const uint32_t *block_base,
                     unsigned long long *line_end, cudaStream_t s);
int launch_csv_parse(const unsigned char *text, size_t bytes, const unsigned long long *line_end,
                     unsigned long long n_newlines, uint32_t skip_lines, unsigned long long rows,
                     uint32_t n_cols, int32_t *const *cols, unsigned char *n_fields, uint32_t *flags,
                     cudaStream_t s);
// forward fill of short rows: per-tile records of the last row with each field, scanned over
// the tiles (summary: the piece's last value of every column, then whether it exists)
uint32_t csv_tiles(unsigned long long rows);
int launch_csv_tile_scan(unsigned long long rows, uint32_t n_cols, int32_t *const *cols,
                         const unsigned char *n_fields, int32_t *tile_last, int32_t *summary, cudaStream_t s);
int launch_csv_last_row(unsigned long long rows, uint32_t n_cols, int32_t *const *cols, int32_t *summary,
                        cudaStream_t s);
int launch_csv_fill(unsigned long long rows, uint32_t n_cols, int32_t *const *cols, const unsigned char *n_fields,
                    const int32_t *tile_prev, const int32_t *carry, cudaStream_t s);

// Result text for print (format_text.cu).
uint32_t fmt_blocks(int64_t n);
int launch_fmt_len(const int32_t *val, int64_t n, uint32_t *block_len, cudaStream_t s);
int launch_fmt_emit(const int32_t *val, int64_t n, const uint32_t *block_off, unsigned char *text,
                    uint64_t text_bytes, cudaStream_t s);

// Hash join (hash_join.cu).
int launch_hj_bounds(const uint32_t *keys, uint32_t n, uint32_t part_bits, uint32_t num_parts,
                     uint32_t *off, cudaStream_t s);
// sums: scratch of (num_parts + 1023) / 1024 + 1 64-bit words
int launch_hj_geometry(const uint32_t *off1, uint32_t num_parts, unsigned long long *toff,
                       unsigned long long *sums, cudaStream_t s);
// toff: num_parts + 1 slot offsets (capacity of partition p = toff[p+1] - toff[p], 0 or a
// power of two); table: toff[num_parts] 16-byte slots
int launch_hj_table_build(const uint32_t *bkeys, const int32_t *bpos, const uint32_t *off1,
                          const unsigned long long *toff, uint32_t num_parts, uint32_t part_bits,
                          uint4 *table, cudaStream_t s);
// Probe and expansion share one geometry: warp w of the grid owns the probe rows
// [w * rows_per_warp, (w + 1) * rows_per_warp).  The probe leaves per-warp match counts, scanned
// in place (warp_sums[w] = first output slot of warp w, *total = all matches).
struct HjProbeGeom {
    uint32_t blocks, warps, rows_per_warp;
};
HjProbeGeom hj_probe_geom(uint32_t n_probe, int sm_count);
int launch_hj_probe(const uint32_t *pkeys, uint32_t n_probe, const HjProbeGeom &pg, const unsigned long long *toff,
                    uint32_t part_bits, const uint4 *table, uint2 *gc_by_j, unsigned long long *warp_sums,
                    unsigned long long *total, cudaStream_t s);
// Probe side partitioned for L2 locality (hash_join.cu): pkeys_part / row_part / cell_base come
// from launch_radix_pass_segmented(probe keys, NULL, ..., RadixPass{24, 8, 1}, seg_tiles).
HjProbeGeom hj_probe_geom_partitioned(uint32_t n_probe);   // one CTA per 4096 rows (its pg goes to the expansion too)
// cell_base / hist / seg_tiles: the segmented pass' base, scanned histogram and effective tiles per
// window (radix_seg_tiles); chunk_sums: pg.warps / 1024 + 2 64-bit words
int launch_hj_probe_partitioned(const uint32_t *pkeys_part, const uint32_t *row_part, const uint32_t *cell_base,
                                const uint32_t *hist, uint32_t segs, uint32_t seg_tiles, uint32_t n_probe,
                                const HjProbeGeom &pg, const unsigned long long *toff, uint32_t part_bits,
                                const uint4 *table, uint2 *res_part, uint2 *gc_by_j,
                                unsigned long long *warp_sums, unsigned long long *chunk_sums,
                                unsigned long long *total, cudaStream_t s);
// The routed probe of the sharded join: an owner probes the keys it received (results in the
// same order; scratch_sums: hj_probe_geom(n).warps words), the rows' home takes the results back
// to row order (cells = owners; cell_base / hist from the unsegmented routing pass).
int launch_hj_probe_plain(const uint32_t *pkeys, uint32_t n_probe, const unsigned long long *toff,
                          uint32_t part_bits, const uint4 *table, uint2 *results, unsigned long long *scratch_sums,
                          int sm_count, cudaStream_t s);
int launch_hj_unpartition_routed(const uint32_t *row_part, const uint2 *res_part, const uint32_t *cell_base,
                                 const uint32_t *hist, uint32_t n_probe, uint32_t cells, const HjProbeGeom &pg,
                                 uint2 *gc_by_j, unsigned long long *warp_sums, unsigned long long *chunk_sums,
                                 unsigned long long *total, cudaStream_t s);
// 4-byte answers of routed rows back to row order (cells = owners; cell_base / hist from the
// unsegmented routing pass, RadixPass::hash 3)
int launch_rows_unpartition32(const uint32_t *row_part, const uint32_t *val_part, const uint32_t *cell_base,
                              const uint32_t *hist, uint32_t n, uint32_t cells, uint32_t *out, cudaStream_t s);
int launch_hj_expand(const uint2 *gc_by_j, const unsigned long long *warp_base, const HjProbeGeom &pg,
                     uint32_t n_probe, const int32_t *build_pos_sorted, const int32_t *probe_pos,
                     int32_t *out_build, int32_t *out_probe, cudaStream_t s);

// The join sharded over several contexts (SURVEY.md 8e): the build side is hash-partitioned
// over the owners (adb_peer_exchange_pairs' route_owner), every owner builds the tables of its
// share, and every context's probe rows -- in their original order -- are answered by the owner
// of each key (the routed probe above).  Output pairs then come out probe-major per context, and
// the contexts' outputs concatenated in shard order are the reference's list.  The expansion
// reads a multi-row group's build positions from its owner over NVLink peer memory.
struct JoinOwners {
    const int32_t *bpos[kMaxPeers];                  // build positions sorted by hash (multi-row groups)
    uint32_t count;                                  // owner of a key = route_owner(key, count)
};
int launch_hj_expand_sharded(const uint2 *gc_by_j, const unsigned long long *warp_base, const HjProbeGeom &pg,
                             uint32_t n_probe, const uint32_t *pkeys, const JoinOwners &owners,
                             const int32_t *probe_pos, int32_t *out_build, int32_t *out_probe, cudaStream_t s);

// Implicit fan-out-32 B+-tree over a sorted value array (index_lookup.cu).
constexpr int kBTreeMaxDepth = 8;
struct BTreeView {
    const int32_t *levels[kBTreeMaxDepth];   // levels[0] sits just above the leaves
    int64_t lens[kBTreeMaxDepth];
    int depth;
};
int launch_btree_level(const int32_t *below, int64_t below_len, int32_t *level, int64_t level_len,
                       int sm_count, cudaStream_t s);
// plain_range: `values` is one slice of a range-partitioned index -- the slice answers
// positions[lb(low) .. lb(high)) and the caller applies the reference's low == high quirk to
// the whole index (it depends on the total count and on the smallest key of all slices)
int launch_index_bounds(const int32_t *values, int64_t n, const BTreeView *tree, const int32_t *lo,
                        const int32_t *hi, bool plain_range, int64_t *bounds, int64_t *d_count,
                        cudaStream_t s);
int launch_index_emit(const int32_t *positions, int64_t n, const int64_t *bounds, int32_t *out,
                      int sm_count, cudaStream_t s);

}  // namespace adb
