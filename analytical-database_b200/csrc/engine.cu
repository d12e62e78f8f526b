// engine.cu -- the C-ABI of libadb_b200.so (include/adb_engine.h): context, memory, and
// the host half of every operator (argument checks, bound folding, launches).
//
// There is deliberately no CPU path in this file: if no CUDA device can be opened,
// adb_init() fails and every operator reports ADB_ERR_NOT_INITIALISED.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <thread>
#include <tuple>
#include <cstdarg>
#include <vector>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>

#include "adb_common.cuh"

namespace {

thread_local std::string g_err;

// A device allocation the engine owns: grown by grow(), freed by release(); reads as a T *.
template <class T> struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;                     // bytes
    operator T *() const { return p; }
};

// Home side of a routed exchange (adb_engine.h), in the arena: this context's items grouped by
// owner, their row numbers, and where the owners' answers are collected
struct RouteState {
    uint32_t *items = nullptr, *rows = nullptr;
    void *answers = nullptr;
    uint32_t n = 0;
};

// Arena buffers the layout functions fill: radix_run's keys and payload, twice; a join build's
// partition bounds, table offsets, geometry scan chunk sums and sort; a probe's (probe_layout).
struct RadixBufs { uint32_t *k[2], *v[2]; };
struct JoinBuildBufs { uint32_t *off1; unsigned long long *toff, *chunk_sums; RadixBufs radix; };
struct ProbeBufs {
    adb::HjProbeGeom pg{};
    unsigned long long *tot = nullptr, *warp_base = nullptr, *chunk_sums = nullptr;
    uint2 *gc_by_j = nullptr, *res = nullptr;
    uint32_t *pk = nullptr, *rows = nullptr, *hist = nullptr, *totals = nullptr, *base = nullptr;
};

struct Engine {
    bool up = false;
    int32_t ctx_index = 0;
    int device = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t marks[ADB_MAX_MARKS] = {};
    // select scratch: selection bitmap (grown on demand) + per-chunk counts
    DevBuf<uint32_t> sel_mask, sel_counts;
    // aggregate fold state: one partial per CTA, and two self-re-arming tickets -- [0] for every
    // grid-wide aggregate fold (one arrival per CTA), [1] for the count phase's fused total
    // (mask_kernel<true>, one arrival per warp-chunk).  The fused count must not share a counter
    // with the fold: each finds its last arrival by comparing the ticket it drew with its own
    // number of arrivals, which only holds while no other kernel draws from the same counter.
    DevBuf<adb_agg> agg_scratch;
    DevBuf<unsigned int> agg_ticket;
    DevBuf<int64_t> idx_bounds;         // {first, count} of the last index select
    int64_t idx_pending_n = -1;         // >= 0 between adb_select_index_count and _emit
    adb::SelectArgs sel_pending{};      // valid between adb_select_*_count and adb_select_emit
    bool sel_ready = false;
    uint64_t sel_generation = 0;        // bumped by every drop_pending (adb_select_generation)
    // small results travel to the host through a mapped pinned mailbox (read_back)
    unsigned long long *mbox = nullptr;  // kMboxWords payload words, then the flag word
    unsigned long long *mbox_dev = nullptr;
    unsigned long long mbox_seq = 0;
    DevBuf<int64_t> scratch_count;      // device int64 for callers that pass no d_count
    // batched shared scan state (count phase -> emit phase)
    DevBuf<unsigned char> ss_plan_mem;  // bounds | cov_off | cov_q
    DevBuf<uint32_t> ss_hits;           // per-chunk hit lists, chunk_rows entries each
    DevBuf<uint32_t> ss_chunk_hits, ss_counts;
    DevBuf<int64_t> ss_totals;
    DevBuf<int32_t *> ss_outs;
    adb::SharedScanPlan ss_plan{};
    adb::SharedScanGeom ss_geom{};
    bool ss_ready = false;
    int32_t ss_base_pos = 0;            // added to every emitted row (shard base)
    // radix / join scratch
    DevBuf<uint32_t> rx_hist, rx_totals, rx_base;
    DevBuf<unsigned long long> sc_sums;
    struct JoinState {
        bool ready = false;
        uint32_t n_probe = 0, n_build = 0;
        int64_t matches = 0;
        ProbeBufs probe;                    // what the expansion reads: gc_by_j, warp_base, pg
        RouteState route;                   // routed probe (adb_join_route_probe), 8-byte answers
        bool routed = false;
        int32_t *build_pos_sorted = nullptr;
        const int32_t *probe_pos = nullptr;
        bool swapped = false;
        // sharded form (adb_join_build ... adb_join_finish_routed): this context's tables, probed
        // here for the keys every context routes to it; the probe keys and the owner table for the
        // expansion
        bool built = false, sharded = false;
        uint32_t part_bits = 1;
        JoinBuildBufs build;                // in the arena, like probe and build_pos_sorted
        const uint32_t *probe_keys = nullptr;
        adb::JoinOwners owners{};
    } join;
    // grow-only scratch arena for the sort / join temporaries: cudaMallocAsync of many
    // differently sized multi-hundred-MB blocks made the pool re-map memory on every join
    DevBuf<unsigned char> arena;
    size_t arena_used = 0;
    // delete plan (adb_delete_rows_plan -> _apply): flags and prefix in the arena
    uint32_t *del_dead = nullptr, *del_before = nullptr;
    int64_t del_rows = -1;
    // join tables: one open-addressing table per build partition, 16-byte slots (grow-only)
    DevBuf<uint4> hj_table;
    // routed fetch (adb_route_rows), 4-byte answers: apart from the join's, which it may run beside
    RouteState fetch_route;
    // routed exchange, owner side: the items other contexts sent here and the answers (grow-only)
    DevBuf<uint32_t> rt_recv_keys;
    DevBuf<uint2> rt_recv_res;
    // bulk CSV load state (adb_csv_index -> adb_csv_parse[_piece] -> adb_csv_fill); scratch is grow-only
    struct CsvState {
        const unsigned char *text = nullptr;
        size_t bytes = 0;
        unsigned long long newlines = 0, rows = 0;
        uint32_t skip = 0, n_cols = 0;
        bool ready = false;
        bool fill_ready = false;            // a piece was parsed and has short rows: adb_csv_fill may run
        DevBuf<uint32_t> block_counts, block_base;
        DevBuf<unsigned long long> line_end;
        DevBuf<unsigned char> n_fields;
        DevBuf<int32_t *> col_table;        // 256 device pointers
        DevBuf<uint32_t> flags;
        DevBuf<int64_t> total;
        DevBuf<int32_t> tile_last;          // per tile and column: last row with the field (scanned)
        DevBuf<int32_t> piece;              // [0, 256) last values, [256, 512) have-flags, [512, 768) carry
    } csv;
    // print formatting state (adb_format_i32_count -> _emit)
    struct FmtState {
        const int32_t *val = nullptr;
        int64_t n = 0, bytes = 0;
        bool ready = false;
        DevBuf<uint32_t> block_len, block_off;
        DevBuf<int64_t> total;
    } fmt;
    // pinned staging lanes for large pageable copies (staged_copy)
    struct StageLane { void *buf[2] = {nullptr, nullptr}; cudaEvent_t ev[2] = {nullptr, nullptr}; cudaStream_t st = nullptr; };
    StageLane stage[8];
    int stage_lanes = 0;
    cudaEvent_t stage_ready = nullptr;
    // aggregate exchange over peer memory (adb_peer_*): own mailbox + the peers' mappings
    DevBuf<adb::PeerRecord> peer_box;
    adb::PeerBoxes peer_boxes{};
    DevBuf<adb::PeerBoxes> peer_boxes_dev;  // the same table in device memory (kernels index it)
    int32_t peer_world = 0, peer_rank = -1;
    bool peer_connected = false;
    uint32_t peer_epoch = 0;
    // pair exchange of the sharded join (adb_peer_join_*): my receive buffer (2 sides x
    // {values, positions} x jx_cap ints), the peers' mapped buffers, a device table of them
    DevBuf<int32_t> jx_recv;
    unsigned long long jx_cap = 0;
    uint32_t *jx_peer_host[ADB_MAX_PEERS] = {};
    DevBuf<uint32_t *> jx_peer_dev;
    bool jx_connected = false;
    uint32_t jx_epoch = 0;
    DevBuf<uint32_t> jx_status;         // device: 0 ok, 1 overflow, 2 timeout
    DevBuf<int64_t> jx_total;           // device: pairs this rank receives
    int64_t launches = 0;
    int32_t chain_mark_base = -1;       // adb_chain_marks(): slots for the next chain call
    bool peer_local = false;            // mailboxes mapped by peer access inside one process (no IPC handles)
    // Front cache of adb_alloc / adb_free.  Result buffers of one query shape come and go in
    // the same few sizes; cudaMallocAsync / cudaFreeAsync cost 5-10 us each (r02h: 14 + 2 x 18 us
    // per select -> fetch -> sum chain on 8 GPUs), a hit here is host bookkeeping.  Blocks keep
    // the stream-ordered semantics of the pool: they are only ever reused on this context's
    // stream.  live: block -> its size class.
    struct CachedBlock { void *p; size_t bytes; };
    static constexpr int kCacheSlots = 64;
    CachedBlock cache[kCacheSlots];
    int cache_n = 0;
    size_t cache_bytes = 0, cache_cap = (size_t)16 << 30;
    std::unordered_map<void *, size_t> *live = nullptr;
    // small host -> device blobs (batch plans, pointer tables) are staged through engine-owned
    // pinned slots: a cudaMemcpyAsync from the caller's memory would read it after the call
    // returned if that memory happened to be pinned (ADVICE r1)
    static constexpr int kBlobSlots = 4;
    static constexpr size_t kBlobBytes = 64 << 10;
    unsigned char *blob[kBlobSlots] = {};
    cudaEvent_t blob_ev[kBlobSlots] = {};
    int blob_next = 0;
};

// Every device buffer a context owns outside its peer connection (peer_close frees those):
// shutting the context down, or an adb_init that failed half way, releases exactly these.
auto context_bufs(Engine &E) {
    return std::tie(E.sel_mask, E.sel_counts, E.agg_scratch, E.agg_ticket, E.idx_bounds, E.scratch_count,
                    E.ss_plan_mem, E.ss_hits, E.ss_chunk_hits, E.ss_counts, E.ss_totals, E.ss_outs, E.rx_hist,
                    E.rx_totals, E.rx_base, E.sc_sums, E.arena, E.hj_table, E.rt_recv_keys, E.rt_recv_res,
                    E.csv.block_counts, E.csv.block_base, E.csv.line_end, E.csv.n_fields, E.csv.col_table,
                    E.csv.flags, E.csv.total, E.csv.tile_last, E.csv.piece, E.fmt.block_len, E.fmt.block_off, E.fmt.total);
}

// One context per GPU of the box (several may share a device: a 1-GPU box then runs the
// multi-shard host path unchanged).  Every entry point works on the calling THREAD's current
// context (adb_ctx_select); a context is only ever driven by one thread at a time.
Engine g_ctx[ADB_MAX_CONTEXTS];
thread_local int g_cur = 0;
#define g (g_ctx[g_cur])


adb_status fail(adb_status code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                       \
    do {                                                                               \
        cudaError_t e_ = (call);                                                       \
        if (e_ != cudaSuccess)                                                         \
            return fail(ADB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                           \
    } while (0)

#define NEED_UP()                                                                      \
    do {                                                                               \
        if (!g.up) return fail(ADB_ERR_NOT_INITIALISED, "adb_init() has not succeeded"); \
    } while (0)

adb_status after_launch(const char *what, int launches) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ADB_ERR_CUDA, "%s launch failed: %s", what, cudaGetErrorString(e));
    g.launches += launches;
    return ADB_OK;
}

// ---- small device -> host results -----------------------------------------------------------
// Every operator of the drop-in API ends by handing a count or an aggregate to the host
// (Result.num_tuples is a plain struct field, src/include/cs165_api.h:179-183).
// cudaMemcpyAsync into pageable memory + cudaStreamSynchronize costs ~20 us of host latency per
// call; here a one-warp kernel at the end of the stream stores the words into mapped pinned
// host memory, then a sequence number, and the host spins on that word.  The stream is polled
// now and then so that a faulted kernel surfaces as an error instead of a hang.
using adb::kMboxWords;
__global__ void publish_kernel(const unsigned long long *__restrict__ src, uint32_t words,
                               volatile unsigned long long *dst, unsigned long long seq) {
    for (uint32_t i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) dst[kMboxWords] = seq;
}

static adb_status mbox_wait(unsigned long long seq, void *h_dst, size_t bytes);
static adb_status read_back(void *h_dst, const void *d_src, size_t bytes) {
    if (bytes == 0) return ADB_OK;
    if (!g.mbox || bytes > kMboxWords * 8 || (bytes & 7u) || (reinterpret_cast<uintptr_t>(d_src) & 7u)) {
        CU(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, g.stream));
        CU(cudaStreamSynchronize(g.stream));
        return ADB_OK;
    }
    const unsigned long long seq = ++g.mbox_seq;
    publish_kernel<<<1, 64, 0, g.stream>>>(static_cast<const unsigned long long *>(d_src), (uint32_t)(bytes / 8),
                                           g.mbox_dev, seq);
    if (adb_status s = after_launch("publish", 1)) return s;
    return mbox_wait(seq, h_dst, bytes);
}

// Spin until the kernel that carries sequence number `seq` has stored its words into the mailbox.
static adb_status mbox_wait(unsigned long long seq, void *h_dst, size_t bytes) {
    const volatile unsigned long long *flag = g.mbox + kMboxWords;
    for (uint32_t spins = 1;; ++spins) {
        if (__atomic_load_n(const_cast<const unsigned long long *>(flag), __ATOMIC_ACQUIRE) == seq) break;
        if ((spins & 0xFFFu) == 0) {
            const cudaError_t e = cudaStreamQuery(g.stream);
            if (e == cudaSuccess) {
                if (__atomic_load_n(const_cast<const unsigned long long *>(flag), __ATOMIC_ACQUIRE) == seq) break;
                return fail(ADB_ERR_CUDA, "result mailbox: the stream drained without publishing");
            }
            if (e != cudaErrorNotReady) return fail(ADB_ERR_CUDA, "result mailbox: %s", cudaGetErrorString(e));
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    memcpy(h_dst, g.mbox, bytes);
    return ADB_OK;
}

// An aggregate a kernel published itself: {sum, count, min | max << 32} (mbox_publish).
static adb_status mbox_wait_agg(unsigned long long seq, adb_agg *h) {
    unsigned long long w[3];
    if (adb_status s = mbox_wait(seq, w, sizeof w)) return s;
    *h = adb_agg{(int64_t)w[0], (int64_t)w[1], (int32_t)(uint32_t)w[2], (int32_t)(uint32_t)(w[2] >> 32)};
    return ADB_OK;
}

// Asynchronous upload of a small blob whose source may go out of scope as soon as the caller
// returns: through a ring of pinned slots (a slot is reused only after its copy has run).
adb_status upload_blob(void *d_dst, const void *h_src, size_t bytes) {
    if (bytes == 0) return ADB_OK;
    if (bytes > Engine::kBlobBytes) {               // large: synchronous
        CU(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, g.stream));
        CU(cudaStreamSynchronize(g.stream));
        return ADB_OK;
    }
    const int k = g.blob_next;
    g.blob_next = (k + 1) % Engine::kBlobSlots;
    if (!g.blob[k]) {
        CU(cudaHostAlloc(reinterpret_cast<void **>(&g.blob[k]), Engine::kBlobBytes, cudaHostAllocDefault));
        CU(cudaEventCreateWithFlags(&g.blob_ev[k], cudaEventDisableTiming));
    } else {
        CU(cudaEventSynchronize(g.blob_ev[k]));
    }
    memcpy(g.blob[k], h_src, bytes);
    CU(cudaMemcpyAsync(d_dst, g.blob[k], bytes, cudaMemcpyHostToDevice, g.stream));
    CU(cudaEventRecord(g.blob_ev[k], g.stream));
    return ADB_OK;
}

// src/server.c:144-154 passes NULL for an absent bound; the predicate is low <= v < high.
adb_status fold_range(const int32_t *lo, const int32_t *hi, adb::Range *out) {
    adb::Range r{lo ? *lo : INT32_MIN, INT32_MAX};
    if (hi) {
        if (*hi == INT32_MIN) r = adb::Range{1, 0};     // v < INT32_MIN: nothing
        else r.hi_incl = *hi - 1;
    }
    if (r.lo > r.hi_incl) r = adb::Range{1, 0};
    *out = r;
    return ADB_OK;
}

adb_status check_len(int64_t n, const char *what) {
    if (n < 0 || n >= (int64_t)1 << 31)
        return fail(ADB_ERR_INVALID, "%s: length %lld outside [0, 2^31) (positions are int32, "
                    "src/query.c:94-95)", what, (long long)n);
    return ADB_OK;
}

// ---- engine-owned device memory --------------------------------------------------------------
// give every cached block back to the pool (before shutdown, or when the device runs short)
void cache_flush(Engine &E) {
    for (int i = 0; i < E.cache_n; ++i) cudaFreeAsync(E.cache[i].p, E.stream);
    E.cache_n = 0;
    E.cache_bytes = 0;
    cudaGetLastError();
}

// Out of device memory: clear the error, flush the front cache and wait until its blocks are free.
void cache_drop(Engine &E) {
    cudaGetLastError();
    cache_flush(E);
    cudaStreamSynchronize(E.stream);
}

template <class T> cudaError_t release(DevBuf<T> &b) {
    const cudaError_t e = b.p ? cudaFree(b.p) : cudaSuccess;
    b = DevBuf<T>{};
    return e;
}

// cudaMalloc of `bytes` into the empty buffer `b`.  Out of memory, the front cache goes back to
// the pool and the pool hands its idle blocks back to the device (its release threshold keeps
// them otherwise, adb_init), then the allocation is tried once more.
template <class T> adb_status dev_alloc(DevBuf<T> &b, size_t bytes, const char *what) {
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e == cudaErrorMemoryAllocation) {
        cache_drop(g);
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, g.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
        cudaGetLastError();
        e = cudaMalloc(&b.p, bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        b = DevBuf<T>{};
        return fail(e == cudaErrorMemoryAllocation ? ADB_ERR_NOMEM : ADB_ERR_CUDA, "%s (%zu bytes): %s", what, bytes,
                    cudaGetErrorString(e));
    }
    b.cap = bytes;
    return ADB_OK;
}

// Grow-only scratch: nothing happens while `need` bytes fit; otherwise the old block is freed
// once the stream is done with it and the new one has room for need + need / 8 + 1 MiB.  The
// routed probe picks its form by the arena's capacity, so this slack is part of its behaviour.
template <class T> adb_status grow(DevBuf<T> &b, size_t need, const char *what) {
    if (need <= b.cap) return ADB_OK;
    if (b.p) {
        CU(cudaStreamSynchronize(g.stream));
        CU(release(b));
    }
    return dev_alloc(b, need + need / 8 + (1 << 20), what);
}

// ---- scratch arena ------------------------------------------------------------------------------
// A bump allocation over the arena in 256-byte steps; dry (no base, no capacity) it only sums its
// takes, so an arena user's layout function run dry is what that user reserves.  Past cap: NULL.
struct Carve {
    unsigned char *base = nullptr;
    size_t cap = SIZE_MAX, used = 0;
    template <class T> T *take(size_t count) {
        const size_t at = used;
        used += (count * sizeof(T) + 255) & ~(size_t)255;
        return base && used <= cap ? reinterpret_cast<T *>(base + at) : nullptr;
    }
};

// Make room for `bytes` of temporaries and start a fresh bump allocation.  Whatever lived in
// the arena before (a join waiting for its emit phase) is gone.
adb_status arena_reserve(size_t bytes) {
    g.join = Engine::JoinState{};
    g.del_rows = -1;
    g.arena_used = 0;
    return grow(g.arena, bytes, "sort/join scratch");
}
// Take what `layout` carves from where the arena's bump allocation stands; with `reserve`, the
// arena is first reserved afresh for exactly that (the layout's dry run).  An overrun fails as `what`.
template <class Layout> adb_status arena_take(Layout &&layout, const char *what, bool reserve = false) {
    if (reserve) {
        Carve dry;
        layout(dry);
        if (adb_status s = arena_reserve(dry.used)) return s;
    }
    Carve c{g.arena.p, g.arena.cap, g.arena_used};
    layout(c);
    if (c.used > c.cap) return fail(ADB_ERR_NOMEM, "%s: scratch arena too small", what);
    g.arena_used = c.used;
    return ADB_OK;
}

void jx_close() {
    for (int r = 0; r < g.peer_world; ++r)
        if (r != g.peer_rank && g.jx_peer_host[r] && !g.peer_local) cudaIpcCloseMemHandle(g.jx_peer_host[r]);
    release(g.jx_recv);
    release(g.jx_peer_dev);
    release(g.jx_status);
    release(g.jx_total);
    cudaGetLastError();
    g.jx_cap = 0;
    for (auto &p : g.jx_peer_host) p = nullptr;
    g.jx_connected = false;
    // jx_epoch is NOT reset: the epoch words live in the aggregate mailbox, which outlives the
    // receive regions -- a new connection that started over at epoch 1 would take the previous
    // connection's count rows for its own (only peer_close, which frees the mailbox, resets it)
}

void peer_close() {
    jx_close();
    for (int r = 0; r < g.peer_world; ++r)
        if (r != g.peer_rank && g.peer_boxes.box[r] && !g.peer_local) cudaIpcCloseMemHandle(g.peer_boxes.box[r]);
    release(g.peer_box);
    release(g.peer_boxes_dev);
    cudaGetLastError();
    g.peer_boxes = adb::PeerBoxes{};
    g.peer_world = 0;
    g.peer_rank = -1;
    g.peer_connected = false;
    g.peer_epoch = 0;
    g.jx_epoch = 0;
    g.peer_local = false;
}

// ---- large host <-> device copies of pageable memory ----------------------------------------
// Loaded columns are plain (mmap'd / malloc'd) host arrays (src/db_manager.c:178-186), which
// cudaMemcpy moves through one internal staging buffer at ~11 GB/s (r01g: 4 GB in 354 ms).
// Here `lanes` host threads each own two pinned 16 MB buffers and a stream: while a lane's
// DMA engine drains one buffer the thread memcpys the next chunk into the other, and the
// lanes together keep the PCIe link busy (the replacement for load_db's row-at-a-time
// ingest, SURVEY.md 8f rank 1).  Synchronous: returns when every byte has landed.
constexpr size_t kStageChunk = 16u << 20;
constexpr size_t kStageMinBytes = 64u << 20;
constexpr int kStageMaxLanes = 8;

bool host_is_pageable(const void *p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

adb_status ensure_stager() {
    if (g.stage_lanes) return ADB_OK;
    int lanes = (int)std::thread::hardware_concurrency() / 2;
    if (const char *e = getenv("ADB_STAGE_LANES")) lanes = atoi(e);
    lanes = lanes < 1 ? 1 : lanes > kStageMaxLanes ? kStageMaxLanes : lanes;
    for (int l = 0; l < lanes; ++l) {
        for (int b = 0; b < 2; ++b) {
            CU(cudaHostAlloc(&g.stage[l].buf[b], kStageChunk, cudaHostAllocDefault));
            CU(cudaEventCreateWithFlags(&g.stage[l].ev[b], cudaEventDisableTiming));
        }
        CU(cudaStreamCreateWithFlags(&g.stage[l].st, cudaStreamNonBlocking));
    }
    CU(cudaEventCreateWithFlags(&g.stage_ready, cudaEventDisableTiming));
    g.stage_lanes = lanes;
    return ADB_OK;
}

// up: host `h` -> device `d`; else device `d` -> host `h`
adb_status staged_copy(void *d, void *h, size_t bytes, bool up) {
    if (adb_status s = ensure_stager()) return s;
    // the device buffer may come from the stream-ordered pool / be written by queued kernels
    CU(cudaEventRecord(g.stage_ready, g.stream));
    const size_t nchunks = (bytes + kStageChunk - 1) / kStageChunk;
    const int lanes = g.stage_lanes;
    std::atomic<int> err{(int)cudaSuccess};
    Engine &E = g;                                  // the helper threads have their own current context
    auto work = [&](int l) {
        auto &L = E.stage[l];
        cudaSetDevice(E.device);
        auto ck = [&](cudaError_t e) { if (e != cudaSuccess) { int ok = (int)cudaSuccess; err.compare_exchange_strong(ok, (int)e); } };
        ck(cudaStreamWaitEvent(L.st, E.stage_ready, 0));
        char *dp = static_cast<char *>(d), *hp = static_cast<char *>(h);
        if (up) {
            int b = 0;
            for (size_t c = l; c < nchunks; c += lanes, b ^= 1) {
                const size_t off = c * kStageChunk, len = std::min(kStageChunk, bytes - off);
                ck(cudaEventSynchronize(L.ev[b]));                    // buffer b's previous DMA is done
                memcpy(L.buf[b], hp + off, len);
                ck(cudaMemcpyAsync(dp + off, L.buf[b], len, cudaMemcpyHostToDevice, L.st));
                ck(cudaEventRecord(L.ev[b], L.st));
            }
        } else {
            // chunk k+1's DMA runs while chunk k is copied out of its pinned buffer
            size_t prev_off = 0, prev_len = 0;
            int b = 0, prev_b = -1;
            for (size_t c = l; c < nchunks; c += lanes, b ^= 1) {
                const size_t off = c * kStageChunk, len = std::min(kStageChunk, bytes - off);
                ck(cudaMemcpyAsync(L.buf[b], dp + off, len, cudaMemcpyDeviceToHost, L.st));
                ck(cudaEventRecord(L.ev[b], L.st));
                if (prev_b >= 0) {
                    ck(cudaEventSynchronize(L.ev[prev_b]));
                    memcpy(hp + prev_off, L.buf[prev_b], prev_len);
                }
                prev_b = b; prev_off = off; prev_len = len;
            }
            if (prev_b >= 0) {
                ck(cudaEventSynchronize(L.ev[prev_b]));
                memcpy(hp + prev_off, L.buf[prev_b], prev_len);
            }
        }
        ck(cudaStreamSynchronize(L.st));
    };
    std::vector<std::thread> th;
    for (int l = 1; l < lanes; ++l) th.emplace_back(work, l);
    work(0);
    for (auto &t : th) t.join();
    if (err.load() != (int)cudaSuccess)
        return fail(ADB_ERR_CUDA, "staged %s of %zu bytes: %s", up ? "upload" : "download", bytes,
                    cudaGetErrorString((cudaError_t)err.load()));
    return ADB_OK;
}

}  // namespace

extern "C" {

const char *adb_last_error(void) { return g_err.c_str(); }
const char *adb_version(void) { return "adb_b200 0.1 (sm_100a)"; }
int adb_sm_count(void) { return g.sm_count; }
int64_t adb_launch_count(void) { return g.launches; }
int64_t adb_launch_count_all(void) {
    int64_t t = 0;
    for (const Engine &e : g_ctx) t += e.up ? e.launches : 0;
    return t;
}

int32_t adb_device_count(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); return 0; }
    return count;
}
int32_t adb_ctx_current(void) { return g_cur; }
adb_status adb_ctx_select(int32_t ctx) {
    if (ctx < 0 || ctx >= ADB_MAX_CONTEXTS) return fail(ADB_ERR_INVALID, "adb_ctx_select: context %d outside [0, %d)", ctx, ADB_MAX_CONTEXTS);
    g_cur = ctx;
    if (g.up) CU(cudaSetDevice(g.device));
    return ADB_OK;
}
adb_status adb_ctx_init(int32_t ctx, int device_ordinal) {
    if (adb_status s = adb_ctx_select(ctx)) return s;
    return adb_init(device_ordinal);
}

static adb_status init_current(int device_ordinal);
static void teardown_current();
adb_status adb_init(int device_ordinal) {
    if (g.up) return ADB_OK;
    const adb_status s = init_current(device_ordinal);
    if (s != ADB_OK) teardown_current();        // nothing stays allocated: a later adb_init starts afresh
    return s;
}

static adb_status init_current(int device_ordinal) {
    // (takes effect when this is the first CUDA call of the process; otherwise the preload_*
    // calls below do the same for the engine's own kernels)
    setenv("CUDA_MODULE_LOADING", "EAGER", 0);
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(ADB_ERR_CUDA, "no CUDA device: %s (this engine has no CPU fallback)",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device_ordinal < 0 || device_ordinal >= count)
        return fail(ADB_ERR_INVALID, "device %d not in [0, %d)", device_ordinal, count);
    CU(cudaSetDevice(device_ordinal));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device_ordinal));
    g.device = device_ordinal;
    g.sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
    g.own_stream = true;
    CU(cudaEventCreate(&g.ev0));
    CU(cudaEventCreate(&g.ev1));
    // keep freed blocks cached in the stream-ordered pool: result buffers are recycled
    cudaMemPool_t pool;
    CU(cudaDeviceGetDefaultMemPool(&pool, device_ordinal));
    uint64_t keep = UINT64_MAX;
    CU(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    if (adb_status s = dev_alloc(g.sel_counts, sizeof(uint32_t) * adb::kMaxSelectChunks, "select chunk counts")) return s;
    if (adb_status s = dev_alloc(g.idx_bounds, 2 * sizeof(int64_t), "index select bounds")) return s;
    if (adb_status s = dev_alloc(g.scratch_count, sizeof(int64_t), "select count")) return s;
    // Gathers over sparse position lists touch one 32-byte sector per hit; ask L2 not to
    // widen those misses (r01b: 570 MB of DRAM reads for 180 MB of requested sectors).
    // A hint only -- streaming kernels request whole lines anyway.  ADB_L2_FETCH overrides.
    {
        size_t gran = 32;
        if (const char *e = getenv("ADB_L2_FETCH")) gran = (size_t)atoi(e);
        if (gran) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, gran);
        cudaGetLastError();
    }
    if (!getenv("ADB_NO_MAILBOX")) {
        void *mb = nullptr;
        if (cudaHostAlloc(&mb, (kMboxWords + 8) * sizeof(unsigned long long), cudaHostAllocMapped) == cudaSuccess) {
            memset(mb, 0, (kMboxWords + 8) * sizeof(unsigned long long));
            void *dv = nullptr;
            if (cudaHostGetDevicePointer(&dv, mb, 0) == cudaSuccess) {
                g.mbox = static_cast<unsigned long long *>(mb);
                g.mbox_dev = static_cast<unsigned long long *>(dv);
            } else {
                cudaGetLastError();
                cudaFreeHost(mb);
            }
        } else {
            cudaGetLastError();                 // readbacks fall back to cudaMemcpyAsync
        }
    }
    if (adb_status s = dev_alloc(g.agg_scratch, sizeof(adb_agg) * adb::kAggMaxBlocks, "aggregate partials")) return s;
    if (adb_status s = dev_alloc(g.agg_ticket, sizeof(unsigned int) * 2, "aggregate tickets")) return s;
    CU(cudaMemset(g.agg_ticket.p, 0, sizeof(unsigned int) * 2));
    // every kernel of the engine is loaded here, per device: see preload_* (adb_common.cuh)
    adb::preload_csv_load(); adb::preload_format_text(); adb::preload_gather_agg(); adb::preload_hash_join();
    adb::preload_index_lookup(); adb::preload_index_ties(); adb::preload_peer_agg(); adb::preload_peer_exchange(); adb::preload_radix();
    adb::preload_select_scan(); adb::preload_shared_scan();
    { cudaFuncAttributes attr; cudaFuncGetAttributes(&attr, publish_kernel); cudaGetLastError(); }
    g.launches = 0;
    g.ctx_index = g_cur;
    g.live = new std::unordered_map<void *, size_t>();
    g.cache_n = 0;
    g.cache_bytes = 0;
    if (const char *e = getenv("ADB_ALLOC_CACHE_MB")) g.cache_cap = (size_t)atol(e) << 20;
    g.up = true;
    return ADB_OK;
}

// Shuts down every context of the process (the hook is called once, from shutdown_server()).
adb_status adb_shutdown(void) {
    const int keep = g_cur;
    // first quiesce every stream: a context's kernels may still touch a peer's mailbox
    for (int c = 0; c < ADB_MAX_CONTEXTS; ++c)
        if (g_ctx[c].up) { cudaSetDevice(g_ctx[c].device); cudaStreamSynchronize(g_ctx[c].stream); }
    for (int c = 0; c < ADB_MAX_CONTEXTS; ++c) {
        g_cur = c;
        if (g.up) teardown_current();
    }
    g_cur = keep;
    return ADB_OK;
}

// Frees everything the current context holds; also a context that adb_init left half built.
static void teardown_current() {
    if (g.device >= 0) cudaSetDevice(g.device);
    cache_flush(g);
    delete g.live;
    g.live = nullptr;
    cudaStreamSynchronize(g.stream);
    std::apply([](auto &...b) { (release(b), ...); }, context_bufs(g));
    for (int k = 0; k < Engine::kBlobSlots; ++k) {
        if (g.blob[k]) cudaFreeHost(g.blob[k]);
        if (g.blob_ev[k]) cudaEventDestroy(g.blob_ev[k]);
    }
    if (g.mbox) cudaFreeHost(g.mbox);
    peer_close();
    for (int l = 0; l < g.stage_lanes; ++l) {
        for (int b = 0; b < 2; ++b) { cudaFreeHost(g.stage[l].buf[b]); cudaEventDestroy(g.stage[l].ev[b]); }
        cudaStreamDestroy(g.stage[l].st);
    }
    if (g.stage_ready) cudaEventDestroy(g.stage_ready);
    if (g.ev0) cudaEventDestroy(g.ev0);
    if (g.ev1) cudaEventDestroy(g.ev1);
    for (cudaEvent_t &m : g.marks)
        if (m) cudaEventDestroy(m);
    if (g.own_stream) cudaStreamDestroy(g.stream);
    cudaGetLastError();
    g = Engine{};
}

void *adb_stream(void) { return g.stream; }

adb_status adb_set_stream(void *cuda_stream) {
    NEED_UP();
    CU(cudaStreamSynchronize(g.stream));
    if (g.own_stream) cudaStreamDestroy(g.stream);
    g.stream = static_cast<cudaStream_t>(cuda_stream);
    g.own_stream = false;
    return ADB_OK;
}

// size classes: 256-byte steps up to 64 KB, then eight steps per power of two (<= 12.5 % slack)
static size_t alloc_class(size_t bytes) {
    if (bytes < 16) bytes = 16;
    if (bytes <= (64u << 10)) return (bytes + 255) & ~(size_t)255;
    size_t p2 = (size_t)1 << 16;
    while (p2 < bytes) p2 <<= 1;                       // smallest power of two >= bytes
    const size_t step = p2 >> 4;                       // 1/8 of the power of two below
    return (bytes + step - 1) / step * step;
}
static void *cache_take(Engine &E, size_t cls) {
    for (int i = 0; i < E.cache_n; ++i)
        if (E.cache[i].bytes == cls) {
            void *p = E.cache[i].p;
            E.cache[i] = E.cache[--E.cache_n];
            E.cache_bytes -= cls;
            return p;
        }
    return nullptr;
}
adb_status adb_alloc(void **d_ptr, size_t bytes) {
    NEED_UP();
    if (!d_ptr) return fail(ADB_ERR_INVALID, "adb_alloc: NULL out pointer");
    const size_t cls = alloc_class(bytes);
    if (void *p = cache_take(g, cls)) {
        (*g.live)[p] = cls;
        *d_ptr = p;
        return ADB_OK;
    }
    cudaError_t e = cudaMallocAsync(d_ptr, cls, g.stream);
    if (e == cudaErrorMemoryAllocation && g.cache_n) {          // short of memory: drop the cache, once more
        cache_drop(g);
        e = cudaMallocAsync(d_ptr, cls, g.stream);
    }
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(ADB_ERR_NOMEM, "adb_alloc: out of device memory for %zu bytes", bytes);
    }
    CU(e);
    (*g.live)[*d_ptr] = cls;
    return ADB_OK;
}
adb_status adb_free(void *d_ptr) {
    NEED_UP();
    if (!d_ptr) return ADB_OK;
    auto it = g.live->find(d_ptr);
    if (it == g.live->end()) {                      // not one of ours (or freed twice): let the runtime judge
        CU(cudaFreeAsync(d_ptr, g.stream));
        return ADB_OK;
    }
    const size_t cls = it->second;
    g.live->erase(it);
    if (g.cache_n < Engine::kCacheSlots && g.cache_bytes + cls <= g.cache_cap) {
        g.cache[g.cache_n++] = Engine::CachedBlock{d_ptr, cls};
        g.cache_bytes += cls;
        return ADB_OK;
    }
    CU(cudaFreeAsync(d_ptr, g.stream));
    return ADB_OK;
}
// The same on context `ctx` from ANOTHER thread's point of view: served only when it needs no
// CUDA call (a cache hit / room in the cache), so the caller neither switches devices nor wakes
// the context's own thread.  ADB_ERR_INVALID-free protocol: returns 1 when served, 0 when the
// caller must go through adb_alloc / adb_free on that context.  The context must be idle.
int32_t adb_alloc_cached_on(int32_t ctx, void **d_ptr, size_t bytes) {
    if (ctx < 0 || ctx >= ADB_MAX_CONTEXTS || !g_ctx[ctx].up || !d_ptr) return 0;
    Engine &E = g_ctx[ctx];
    const size_t cls = alloc_class(bytes);
    void *p = cache_take(E, cls);
    if (!p) return 0;
    (*E.live)[p] = cls;
    *d_ptr = p;
    return 1;
}
int32_t adb_free_cached_on(int32_t ctx, void *d_ptr) {
    if (ctx < 0 || ctx >= ADB_MAX_CONTEXTS || !g_ctx[ctx].up) return 0;
    if (!d_ptr) return 1;
    Engine &E = g_ctx[ctx];
    auto it = E.live->find(d_ptr);
    if (it == E.live->end()) return 0;
    const size_t cls = it->second;
    if (E.cache_n >= Engine::kCacheSlots || E.cache_bytes + cls > E.cache_cap) return 0;
    E.live->erase(it);
    E.cache[E.cache_n++] = Engine::CachedBlock{d_ptr, cls};
    E.cache_bytes += cls;
    return 1;
}
adb_status adb_upload_async(void *d_dst, const void *h_src, size_t bytes) {
    NEED_UP();
    if (bytes) CU(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, g.stream));
    return ADB_OK;
}
adb_status adb_download_async(void *h_dst, const void *d_src, size_t bytes) {
    NEED_UP();
    if (bytes) CU(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, g.stream));
    return ADB_OK;
}
adb_status adb_upload(void *d_dst, const void *h_src, size_t bytes) {
    NEED_UP();
    if (bytes >= kStageMinBytes && host_is_pageable(h_src)) return staged_copy(d_dst, const_cast<void *>(h_src), bytes, true);
    adb_status s = adb_upload_async(d_dst, h_src, bytes);
    return s ? s : adb_sync();
}
adb_status adb_download(void *h_dst, const void *d_src, size_t bytes) {
    NEED_UP();
    if (bytes >= kStageMinBytes && host_is_pageable(h_dst)) return staged_copy(const_cast<void *>(d_src), h_dst, bytes, false);
    adb_status s = adb_download_async(h_dst, d_src, bytes);
    return s ? s : adb_sync();
}
// Page-lock a host range the caller keeps uploading from (a loaded column is an mmap that
// insert_row appends to, src/db_manager.c:164-199: every insert invalidates the HBM copy): from
// registered memory adb_upload is one DMA at the link's rate instead of the staged copy through
// pinned lanes.  Portable: every context's device sees it pinned.  Registration itself is slow
// (it touches and locks every page), so it only pays for memory that is uploaded repeatedly.
adb_status adb_host_register(void *h_ptr, size_t bytes) {
    NEED_UP();
    if (!h_ptr || !bytes) return fail(ADB_ERR_INVALID, "adb_host_register: empty range");
    cudaError_t e = cudaHostRegister(h_ptr, bytes, cudaHostRegisterPortable);
    if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return ADB_OK; }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ADB_ERR_CUDA, "adb_host_register(%zu bytes): %s", bytes, cudaGetErrorString(e));
    }
    return ADB_OK;
}
adb_status adb_host_unregister(void *h_ptr) {
    NEED_UP();
    if (!h_ptr) return ADB_OK;
    cudaError_t e = cudaHostUnregister(h_ptr);
    if (e != cudaSuccess) cudaGetLastError();       // (not registered: nothing to undo)
    return ADB_OK;
}

adb_status adb_memset(void *d_dst, int byte, size_t bytes) {
    NEED_UP();
    if (bytes) CU(cudaMemsetAsync(d_dst, byte, bytes, g.stream));
    return ADB_OK;
}
adb_status adb_sync(void) {
    NEED_UP();
    CU(cudaStreamSynchronize(g.stream));
    return ADB_OK;
}
adb_status adb_host_alloc(void **h_ptr, size_t bytes) {
    NEED_UP();
    CU(cudaMallocHost(h_ptr, bytes ? bytes : 16));
    return ADB_OK;
}
adb_status adb_host_free(void *h_ptr) {
    NEED_UP();
    if (h_ptr) CU(cudaFreeHost(h_ptr));
    return ADB_OK;
}
adb_status adb_timer_start(void) {
    NEED_UP();
    CU(cudaEventRecord(g.ev0, g.stream));
    return ADB_OK;
}
adb_status adb_timer_stop(float *ms) {
    NEED_UP();
    CU(cudaEventRecord(g.ev1, g.stream));
    CU(cudaEventSynchronize(g.ev1));
    if (ms) CU(cudaEventElapsedTime(ms, g.ev0, g.ev1));
    return ADB_OK;
}

adb_status adb_mark(int32_t slot) {
    NEED_UP();
    if (slot < 0 || slot >= ADB_MAX_MARKS) return fail(ADB_ERR_INVALID, "adb_mark: slot %d out of range", slot);
    if (!g.marks[slot]) CU(cudaEventCreate(&g.marks[slot]));
    CU(cudaEventRecord(g.marks[slot], g.stream));
    return ADB_OK;
}
adb_status adb_mark_elapsed(int32_t from_slot, int32_t to_slot, float *ms) {
    NEED_UP();
    if (from_slot < 0 || from_slot >= ADB_MAX_MARKS || to_slot < 0 || to_slot >= ADB_MAX_MARKS ||
        !g.marks[from_slot] || !g.marks[to_slot] || !ms)
        return fail(ADB_ERR_INVALID, "adb_mark_elapsed: unrecorded or invalid slot");
    CU(cudaEventSynchronize(g.marks[to_slot]));
    CU(cudaEventElapsedTime(ms, g.marks[from_slot], g.marks[to_slot]));
    return ADB_OK;
}

adb_status adb_chain_marks(int32_t base_slot) {
    NEED_UP();
    if (base_slot >= 0 && base_slot + 2 >= ADB_MAX_MARKS)
        return fail(ADB_ERR_INVALID, "adb_chain_marks: slot %d out of range", base_slot);
    g.chain_mark_base = base_slot;
    return ADB_OK;
}

// ---- operators ---------------------------------------------------------------------------
static adb_status finish_count(int64_t *d_count, int64_t *h_count) {
    if (!h_count) return ADB_OK;
    return read_back(h_count, d_count, sizeof(int64_t));
}

// The pending select (adb_select_count*) is dropped, and adb_select_generation() bumped, when a
// select is about to overwrite its bitmap and when an emit consumes it.  So whether a refused call
// drops it depends on what was refused: a select that refuses an output pointer (adb_select_scan,
// adb_chain_select_*) leaves it as it was, one that refuses its length or input column has
// dropped it; the deferred emit (adb_select_emit_fetch_agg*) leaves it on any refusal;
// adb_select_emit has taken it before it checks its output.
static void drop_pending() { g.sel_ready = false; ++g.sel_generation; }

// The setup every select runs, in this order: NEED_UP, the entry point's own output-pointer rule
// (null_out), drop_pending, then the length, the input column, the bounds, the bitmap and the
// SelectArgs.
// stable_val: d_val is a base column -- no operator ever writes it, so the predicate pass may
// request its first tile while the previous kernel on the stream is still draining (any other
// input may be that kernel's output and must wait for it: ADVICE r1, select_scan.cu).
static adb_status select_prepare(const char *what, bool null_out, const int32_t *d_val, int64_t n_max,
                                 const int64_t *d_n, const int32_t *lo, const int32_t *hi,
                                 int64_t *d_count, adb::SelectArgs *a, bool stable_val = false) {
    NEED_UP();
    if (null_out) return fail(ADB_ERR_INVALID, "%s: NULL device pointer", what);
    drop_pending();
    if (adb_status s = check_len(n_max, what)) return s;
    if (n_max > 0 && !d_val) return fail(ADB_ERR_INVALID, "%s: NULL device pointer", what);
    *a = adb::SelectArgs{};
    a->val = d_val; a->d_n = d_n; a->n = (uint32_t)n_max;
    a->stable_val = stable_val;
    fold_range(lo, hi, &a->range);
    a->d_count = d_count ? d_count : g.scratch_count;
    // the bitmap only ever grows; a select over the largest shard (2^31 rows) needs 256 MB
    if (adb_status s = grow(g.sel_mask, sizeof(uint32_t) * adb::select_mask_words(a->n, g.sm_count), "select bitmap"))
        return s;
    a->mask = g.sel_mask; a->counts = g.sel_counts; a->sm_count = g.sm_count;
    a->agg_scratch = g.agg_scratch; a->agg_ticket = g.agg_ticket;
    return ADB_OK;
}

adb_status adb_select_scan(const int32_t *d_col, int64_t n, const int32_t *lo, const int32_t *hi,
                           int32_t base_pos, int32_t *d_pos_out, int64_t *d_count,
                           int64_t *h_count) {
    adb::SelectArgs a;
    if (adb_status s = select_prepare("adb_select_scan", !d_count || (n > 0 && !d_pos_out), d_col, n, nullptr,
                                      lo, hi, d_count, &a, true))
        return s;
    a.base_pos = base_pos; a.out = d_pos_out;
    const int k_ = adb::launch_select_mask(a, false, g.stream);
    if (adb_status s = after_launch("select_scan", k_ + adb::launch_select_expand(a, g.stream))) return s;
    return finish_count(d_count, h_count);
}

// Two-phase form: the count phase streams the column once and leaves the selection bitmap in
// the engine's scratch; the emit phase turns it into positions in a buffer of exactly the
// right size.  Any other select in between invalidates the pending bitmap.
adb_status adb_select_count(const int32_t *d_val, int64_t n_max, const int64_t *d_n,
                            const int32_t *lo, const int32_t *hi, int64_t *d_count,
                            int64_t *h_count) {
    adb::SelectArgs a;
    if (adb_status s = select_prepare("adb_select_count", false, d_val, n_max, d_n, lo, hi, d_count, &a)) return s;
    if (adb_status s = after_launch("select_count", adb::launch_select_mask(a, true, g.stream))) return s;
    g.sel_pending = a;
    g.sel_ready = true;
    return finish_count(a.d_count, h_count);
}

// Count phase over rows [base_pos, base_pos + n) of a BASE column (shard): as adb_select_count,
// plus the two things only a base column allows -- the early first-tile request (see
// select_prepare) and a pending select that adb_select_emit_fetch_agg* can resolve, emitting
// base_pos + row.
adb_status adb_select_count_base(const int32_t *d_col, int64_t n, const int32_t *lo, const int32_t *hi,
                                 int32_t base_pos, int64_t *d_count, int64_t *h_count) {
    adb::SelectArgs a;
    if (adb_status s = select_prepare("adb_select_count_base", false, d_col, n, nullptr, lo, hi, d_count, &a, true))
        return s;
    // the host wants the count: the kernel that totals it also hands it over (no publish launch)
    const bool fused_pub = h_count && g.mbox && a.n > 0;
    if (fused_pub) { a.pub = g.mbox_dev; a.pub_seq = ++g.mbox_seq; }
    a.mask_ticket = g.agg_ticket + 1;
    if (adb_status s = after_launch("select_count", adb::launch_select_mask(a, true, g.stream))) return s;
    const unsigned long long seq = a.pub_seq;
    a.pub = nullptr; a.pub_seq = 0; a.mask_ticket = nullptr;
    a.base_pos = base_pos;
    g.sel_pending = a;
    g.sel_ready = true;
    if (fused_pub) return mbox_wait(seq, h_count, sizeof(int64_t));
    return finish_count(a.d_count, h_count);
}

adb_status adb_select_emit(const int32_t *d_pos_in, int32_t base_pos, int32_t *d_pos_out) {
    NEED_UP();
    if (!g.sel_ready) return fail(ADB_ERR_INVALID, "adb_select_emit: no pending adb_select_count");
    drop_pending();                                 // the pending count is consumed
    adb::SelectArgs a = g.sel_pending;
    if (a.n == 0) return ADB_OK;
    if (!d_pos_out) return fail(ADB_ERR_INVALID, "adb_select_emit: NULL output");
    a.pos_in = d_pos_in; a.base_pos = base_pos; a.out = d_pos_out;
    a.d_count = g.scratch_count;                    // expand rewrites the same total
    return after_launch("select_emit", adb::launch_select_expand(a, g.stream));
}

uint64_t adb_select_generation(void) { return g.sel_generation; }

// The second kernel of the materialised chain and of the deferred emit: positions, gather and
// aggregate (with px, the exchange too) in one launch.  Where that kernel cannot run -- an empty
// column, or a grid larger than the fold scratch -- the three-operator form runs instead and reads
// the hit count from d_count; the aggregate-only form (a.out == a.val_out == NULL) has no such
// fallback for a non-empty select.  h_agg (optional) receives the aggregate, straight from the
// kernel when it can publish it itself.
static adb_status fused_finish(const char *what, adb::SelectArgs &a, const int64_t *d_count,
                               const adb::PeerExchange *px, adb_agg *h_agg) {
    if (px) a.px = *px;
    const bool nostore = !a.out && !a.val_out;
    const bool fused_pub = nostore && h_agg && g.mbox && a.n > 0;
    if (fused_pub) { a.pub = g.mbox_dev; a.pub_seq = ++g.mbox_seq; }
    const int f_ = adb::launch_select_expand_fetch_agg(a, g.stream);
    if (f_ > 0) {
        if (adb_status s = after_launch(what, f_)) return s;
    } else if (nostore && a.n > 0) {
        return fail(ADB_ERR_INVALID, "%s: a select over %u rows cannot be aggregated unmaterialised", what, a.n);
    } else {
        if (adb_status s = after_launch(what, adb::launch_select_expand(a, g.stream))) return s;
        if (adb_status s = adb_fetch(a.fetch_col, a.out, a.n, d_count, a.base_pos, a.val_out)) return s;
        if (adb_status s = adb_aggregate(a.val_out, a.n, d_count, a.agg_out, nullptr)) return s;
        if (px)
            if (adb_status s = after_launch("chain exchange", adb::launch_agg_combine_allreduce(*px, g.stream))) return s;
    }
    if (!h_agg) return ADB_OK;
    if (adb_status s = fused_pub ? mbox_wait_agg(a.pub_seq, h_agg)
                                 : read_back(h_agg, px ? px->final_out : a.agg_out, sizeof(adb_agg)))
        return s;
    if (px && h_agg->count < 0)
        return fail(ADB_ERR_CUDA, "%s: a peer did not arrive within 2 s (epoch %u)", what, px->epoch);
    return ADB_OK;
}

// Deferred emit of a select whose consumers turned out to be fetch + aggregate: the fused
// second kernel of the chain, after the host has read the count (SURVEY.md 8f rank 3).
static adb_status emit_fetch_agg_impl(const char *what, const int32_t *d_fetch_col, int32_t *d_pos_out,
                                      int32_t *d_val_out, adb_agg *d_agg, adb_agg *h_agg,
                                      const adb::PeerExchange *px) {
    NEED_UP();
    if (!g.sel_ready) return fail(ADB_ERR_INVALID, "%s: no pending adb_select_count", what);
    adb::SelectArgs a = g.sel_pending;
    if (a.d_n) return fail(ADB_ERR_INVALID, "%s: the pending select is not over a base column", what);
    // both outputs NULL: aggregate only -- nothing is materialised and the pending select stays
    // pending (the bitmap is only read), so a later emit can still write the handles
    const bool nostore = !d_pos_out && !d_val_out;
    if (!d_agg || (a.n > 0 && (!d_fetch_col || (!nostore && (!d_pos_out || !d_val_out)))))
        return fail(ADB_ERR_INVALID, "%s: NULL device pointer", what);
    if (!nostore) drop_pending();                   // the pending count is consumed
    const int64_t *d_count = a.d_count;             // written by the count phase
    a.d_count = g.scratch_count;                    // the expansion rewrites the same total
    a.out = d_pos_out; a.fetch_col = d_fetch_col; a.val_out = d_val_out; a.agg_out = d_agg;
    return fused_finish(what, a, d_count, px, h_agg);     // base_pos: what the count phase recorded
}

adb_status adb_select_emit_fetch_agg(const int32_t *d_fetch_col, int32_t *d_pos_out, int32_t *d_val_out,
                                     adb_agg *d_agg, adb_agg *h_agg) {
    return emit_fetch_agg_impl("adb_select_emit_fetch_agg", d_fetch_col, d_pos_out, d_val_out, d_agg, h_agg, nullptr);
}

// The descriptor of this context's next aggregate exchange (epoch peer_epoch + 1).  Every
// context must take part in every exchange, so a context that advances its epoch and then fails
// has left the group out of step.  The three callers advance it at different points:
//   adb_agg_combine_allreduce            once its arguments are accepted;
//   adb_select_emit_fetch_agg_exchange   once a pending select is found, before the remaining checks;
//   adb_chain_select_fetch_agg_exchange  only when the chain was enqueued.
// Making them agree would change what a group does after one rank fails.
static adb_status peer_exchange(const char *what, const adb_agg *d_parts, int32_t k, adb_agg *d_out,
                                adb::PeerExchange *px) {
    NEED_UP();
    if (!g.peer_connected) return fail(ADB_ERR_INVALID, "%s: adb_peer_connect first", what);
    *px = adb::PeerExchange{g.peer_boxes_dev, g.peer_rank, g.peer_world, g.peer_epoch + 1, d_parts, k, d_out};
    return ADB_OK;
}

// The deferred emit with the cross-context exchange riding in the same kernel: this context's
// partial goes to d_part, the table-wide aggregate to d_out (and h_out) on every context.
// Collective over the contexts / ranks of adb_peer_connect*.
adb_status adb_select_emit_fetch_agg_exchange(const int32_t *d_fetch_col, int32_t *d_pos_out,
                                              int32_t *d_val_out, adb_agg *d_part, adb_agg *d_out,
                                              adb_agg *h_out) {
    const char *what = "adb_select_emit_fetch_agg_exchange";
    adb::PeerExchange px;
    if (adb_status s = peer_exchange(what, d_part, 1, d_out, &px)) return s;
    if (!d_part || !d_out) return fail(ADB_ERR_INVALID, "%s: NULL device pointer", what);
    if (!g.sel_ready) return fail(ADB_ERR_INVALID, "%s: no pending adb_select_count_base", what);
    ++g.peer_epoch;
    return emit_fetch_agg_impl(what, d_fetch_col, d_pos_out, d_val_out, d_part, h_out, &px);
}

adb_status adb_fetch(const int32_t *d_col, const int32_t *d_pos, int64_t n_max,
                     const int64_t *d_n, int32_t base_pos, int32_t *d_val_out) {
    NEED_UP();
    if (adb_status s = check_len(n_max, "adb_fetch")) return s;
    if (n_max == 0) return ADB_OK;
    if (!d_col || !d_pos || !d_val_out) return fail(ADB_ERR_INVALID, "adb_fetch: NULL device pointer");
    const int k_ = adb::launch_fetch(d_col, d_pos, n_max, d_n, base_pos, d_val_out, g.sm_count, g.stream);
    return after_launch("fetch", k_);
}

// fetch over a column that is row-range sharded across contexts: position p lives in shard
// p / shard_rows at row p % shard_rows; remote shards are read over NVLink peer memory
// (adb_peer_connect_local has enabled the access).
adb_status adb_fetch_sharded(const int32_t *const *d_shards, int32_t n_shards, int64_t shard_rows,
                             const int32_t *d_pos, int64_t n_max, const int64_t *d_n, int32_t *d_val_out) {
    NEED_UP();
    if (adb_status s = check_len(n_max, "adb_fetch_sharded")) return s;
    if (n_shards < 1 || n_shards > ADB_MAX_PEERS || shard_rows < 1 || shard_rows >= ((int64_t)1 << 31) || !d_shards)
        return fail(ADB_ERR_INVALID, "adb_fetch_sharded: %d shards of %lld rows", n_shards, (long long)shard_rows);
    if (n_max == 0) return ADB_OK;
    if (!d_pos || !d_val_out) return fail(ADB_ERR_INVALID, "adb_fetch_sharded: NULL device pointer");
    adb::ShardTable t{};
    for (int i = 0; i < n_shards; ++i) t.ptr[i] = d_shards[i];
    const int k_ = adb::launch_fetch_sharded(t, n_shards, (uint32_t)shard_rows, d_pos, n_max, d_n, d_val_out,
                                             g.sm_count, g.stream);
    return after_launch("fetch_sharded", k_);
}

adb_status adb_aggregate(const int32_t *d_val, int64_t n_max, const int64_t *d_n,
                         adb_agg *d_out, adb_agg *h_out) {
    NEED_UP();
    if (adb_status s = check_len(n_max, "adb_aggregate")) return s;
    if (!d_out || (n_max > 0 && !d_val)) return fail(ADB_ERR_INVALID, "adb_aggregate: NULL device pointer");
    const int k_ = adb::launch_aggregate(d_val, n_max, d_n, d_out, g.agg_scratch, g.agg_ticket, g.sm_count, g.stream);
    if (adb_status s = after_launch("aggregate", k_)) return s;
    if (h_out) {
        if (adb_status s = read_back(h_out, d_out, sizeof(adb_agg))) return s;
    }
    return ADB_OK;
}

adb_status adb_agg_combine(const adb_agg *d_parts, int32_t k, adb_agg *d_out, adb_agg *h_out) {
    NEED_UP();
    if (k < 0 || !d_out || (k > 0 && !d_parts)) return fail(ADB_ERR_INVALID, "adb_agg_combine: bad arguments");
    const int k_ = adb::launch_agg_combine(d_parts, k, d_out, g.stream);
    if (adb_status s = after_launch("agg_combine", k_)) return s;
    if (h_out) {
        if (adb_status s = read_back(h_out, d_out, sizeof(adb_agg))) return s;
    }
    return ADB_OK;
}

// ---- aggregate exchange over NVLink peer memory ------------------------------------------
// The peer setup shared by the IPC path (adb_peer_create / _connect, adb_peer_join_create /
// _connect) and the one-process path (adb_peer_connect_local, adb_peer_join_connect_local).
// The mailbox and the receive region may be exported through IPC, so they are plain cudaMalloc
// blocks of exactly their size.

// Closes the current connection and gives this context a fresh mailbox, zeroed (epoch 0 =
// nothing arrived yet) and idle before anyone maps it.
static adb_status peer_mailbox_create() {
    CU(cudaStreamSynchronize(g.stream));
    peer_close();
    if (adb_status s = dev_alloc(g.peer_box, adb::kPeerBoxBytes, "peer mailbox")) return s;
    CU(cudaMemset(g.peer_box.p, 0, adb::kPeerBoxBytes));
    CU(cudaDeviceSynchronize());
    return ADB_OK;
}

// g.peer_boxes (every rank's mailbox, as this context sees it) -> the device table kernels index.
static adb_status peer_boxes_upload() {
    if (adb_status s = grow(g.peer_boxes_dev, sizeof(adb::PeerBoxes), "peer mailbox table")) return s;
    CU(cudaMemcpy(g.peer_boxes_dev.p, &g.peer_boxes, sizeof(adb::PeerBoxes), cudaMemcpyHostToDevice));
    g.peer_connected = true;
    g.peer_epoch = 0;
    return ADB_OK;
}

// Closes the current receive region and makes this context's: 2 sides x {values, positions} x
// `cap` ints, with the table of the peers' regions, the exchange status and the received total.
static adb_status jx_region_create(unsigned long long cap) {
    CU(cudaStreamSynchronize(g.stream));
    jx_close();
    if (adb_status s = dev_alloc(g.jx_recv, cap * 4 * sizeof(int32_t), "join receive buffer")) return s;
    if (adb_status s = grow(g.jx_peer_dev, sizeof(uint32_t *) * ADB_MAX_PEERS, "join receive-buffer table")) return s;
    if (adb_status s = grow(g.jx_status, 4 * sizeof(uint32_t), "join exchange status")) return s;
    if (adb_status s = grow(g.jx_total, 2 * sizeof(int64_t), "join exchange total")) return s;
    g.jx_cap = cap;
    return ADB_OK;
}

// g.jx_peer_host (every rank's receive region, as this context sees it) -> the device table.
static adb_status jx_table_upload() {
    CU(cudaMemcpy(g.jx_peer_dev.p, g.jx_peer_host, sizeof(uint32_t *) * ADB_MAX_PEERS, cudaMemcpyHostToDevice));
    g.jx_connected = true;
    return ADB_OK;
}

adb_status adb_peer_create(int32_t world, int32_t rank, unsigned char *handle_out) {
    NEED_UP();
    static_assert(sizeof(cudaIpcMemHandle_t) == ADB_PEER_HANDLE_BYTES, "handle size");
    if (world < 1 || world > ADB_MAX_PEERS || rank < 0 || rank >= world || !handle_out)
        return fail(ADB_ERR_INVALID, "adb_peer_create: world %d (max %d), rank %d", world, ADB_MAX_PEERS, rank);
    if (adb_status s = peer_mailbox_create()) return s;
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, g.peer_box.p));
    memcpy(handle_out, &h, sizeof h);
    g.peer_world = world;
    g.peer_rank = rank;
    g.peer_boxes.box[rank] = g.peer_box;
    return ADB_OK;
}

adb_status adb_peer_connect(const unsigned char *handles) {
    NEED_UP();
    if (!g.peer_box.p || !handles) return fail(ADB_ERR_INVALID, "adb_peer_connect: adb_peer_create first");
    for (int r = 0; r < g.peer_world; ++r) {
        if (r == g.peer_rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * ADB_PEER_HANDLE_BYTES, sizeof h);
        void *p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(ADB_ERR_CUDA, "adb_peer_connect: cannot map rank %d's mailbox: %s (peer access over "
                        "NVLink is required)", r, cudaGetErrorString(e));
        }
        g.peer_boxes.box[r] = static_cast<adb::PeerRecord *>(p);
    }
    return peer_boxes_upload();
}

adb_status adb_agg_combine_allreduce(const adb_agg *d_parts, int32_t k, adb_agg *d_out, adb_agg *h_out) {
    adb::PeerExchange px;
    if (adb_status s = peer_exchange("adb_agg_combine_allreduce", d_parts, k, d_out, &px)) return s;
    if (k < 0 || !d_out || (k > 0 && !d_parts))
        return fail(ADB_ERR_INVALID, "adb_agg_combine_allreduce: bad arguments");
    ++g.peer_epoch;
    if (adb_status s = after_launch("agg_combine_allreduce", adb::launch_agg_combine_allreduce(px, g.stream))) return s;
    if (!h_out) return ADB_OK;
    if (adb_status s = read_back(h_out, d_out, sizeof(adb_agg))) return s;
    if (h_out->count < 0)
        return fail(ADB_ERR_CUDA, "adb_agg_combine_allreduce: a peer did not arrive within 2 s (epoch %u)", px.epoch);
    return ADB_OK;
}

// ---- pair exchange of the sharded join over peer memory ---------------------------------------
static adb_status ensure_radix_scratch(uint32_t n);          // defined with the radix helpers below
adb_status adb_peer_join_create(int64_t cap_pairs, unsigned char *handle_out) {
    NEED_UP();
    if (!g.peer_connected) return fail(ADB_ERR_INVALID, "adb_peer_join_create: adb_peer_connect first");
    if (cap_pairs < 1 || cap_pairs >= ((int64_t)1 << 31) || !handle_out)
        return fail(ADB_ERR_INVALID, "adb_peer_join_create: capacity %lld outside [1, 2^31)", (long long)cap_pairs);
    const unsigned long long cap = ((unsigned long long)cap_pairs + 63) & ~63ull;     // regions stay 256-byte aligned
    if (adb_status s = jx_region_create(cap)) return s;
    CU(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, g.jx_recv.p));
    memcpy(handle_out, &h, sizeof h);
    g.jx_peer_host[g.peer_rank] = reinterpret_cast<uint32_t *>(g.jx_recv.p);
    return ADB_OK;
}

adb_status adb_peer_join_connect(const unsigned char *handles) {
    NEED_UP();
    if (!g.jx_recv.p || !handles) return fail(ADB_ERR_INVALID, "adb_peer_join_connect: adb_peer_join_create first");
    for (int r = 0; r < g.peer_world; ++r) {
        if (r == g.peer_rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * ADB_PEER_HANDLE_BYTES, sizeof h);
        void *p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(ADB_ERR_CUDA, "adb_peer_join_connect: cannot map rank %d's receive buffer: %s", r, cudaGetErrorString(e));
        }
        g.jx_peer_host[r] = static_cast<uint32_t *>(p);
    }
    return jx_table_upload();
}

// The multi-GPU exchange's pass: digit = route_owner(key, parts), for any parts in [1, 256].  Its
// histograms, bases and scatter cover 2^ceil(log2 parts) buckets as any pass' do; those from parts
// up stay empty.
static adb::RadixPass routing_pass(int parts) {
    adb::RadixPass p{0, 0, 2};
    while ((1 << p.bits) < parts) ++p.bits;
    p.parts = (uint32_t)parts;
    return p;
}

adb_status adb_peer_exchange_pairs(int32_t side, const int32_t *d_val, const int32_t *d_pos, int64_t n,
                                   int64_t *h_recv_count, const int32_t **d_recv_val,
                                   const int32_t **d_recv_pos) {
    NEED_UP();
    if (!g.jx_connected) return fail(ADB_ERR_INVALID, "adb_peer_exchange_pairs: adb_peer_join_connect first");
    if (adb_status s = check_len(n, "adb_peer_exchange_pairs")) return s;
    if (side < 0 || side > 1 || !h_recv_count || !d_recv_val || !d_recv_pos || (n > 0 && (!d_val || !d_pos)))
        return fail(ADB_ERR_INVALID, "adb_peer_exchange_pairs: bad arguments");
    const int world = g.peer_world;
    if (adb_status s = ensure_radix_scratch((uint32_t)(n ? n : 1))) return s;
    const adb::RadixPass pass = routing_pass(world);          // the owners of adb_route_pairs
    const adb::PairExchange x{g.peer_boxes_dev, g.peer_rank, world, ++g.jx_epoch, g.jx_cap};
    const unsigned long long key_off = (unsigned long long)(2 * side) * g.jx_cap;
    const unsigned long long pay_off = (unsigned long long)(2 * side + 1) * g.jx_cap;
    int k_ = 0;
    if (world == 1 && (unsigned long long)n > g.jx_cap)
        return fail(ADB_ERR_NOMEM, "adb_peer_exchange_pairs: %lld pairs do not fit the %llu-pair receive region; "
                    "reserve more with adb_peer_join_create", (long long)n, g.jx_cap);
    if (world == 1) {
        // no routing digit: every pair stays here (still through the flags: one code path)
        CU(cudaMemsetAsync(g.rx_totals, 0, sizeof(uint32_t) * 256, g.stream));
        const uint32_t n32 = (uint32_t)n;
        if (adb_status s = upload_blob(g.rx_totals, &n32, sizeof n32)) return s;
    } else {
        k_ += adb::launch_radix_hist(reinterpret_cast<const uint32_t *>(d_val), (uint32_t)n, pass, g.rx_hist,
                                     g.rx_totals, g.sm_count, g.stream);
    }
    k_ += adb::launch_jx_counts(x, g.rx_totals, g.rx_base, g.jx_total, g.jx_status, g.stream);
    // Nothing of this context may wait in a hardware queue behind its spinning jx_counts_kernel.
    // The contexts' streams share the device's few hardware work queues, and when a peer's stream
    // lands in the same queue, a launch that depends on the spinning kernel (the scatter) blocks
    // that queue's head: the peer's own jx_counts_kernel behind it cannot start, and both give up
    // after 2 s.  Which streams share a queue depends on how many were created before, so this
    // struck some first joins on freshly started contexts only.  The scatter is enqueued once
    // every count row has arrived.
    CU(cudaStreamSynchronize(g.stream));
    if (world == 1) {
        if (n) {
            CU(cudaMemcpyAsync(g.jx_recv + key_off, d_val, (size_t)n * 4, cudaMemcpyDeviceToDevice, g.stream));
            CU(cudaMemcpyAsync(g.jx_recv + pay_off, d_pos, (size_t)n * 4, cudaMemcpyDeviceToDevice, g.stream));
        }
    } else {
        k_ += adb::launch_radix_scatter_remote(reinterpret_cast<const uint32_t *>(d_val),
                                               reinterpret_cast<const uint32_t *>(d_pos), (uint32_t)n, pass,
                                               g.rx_hist, g.rx_base, g.jx_peer_dev, key_off, pay_off,
                                               g.jx_status, g.sm_count, g.stream);
    }
    k_ += adb::launch_jx_done(x, g.jx_status, g.stream);
    if (adb_status s = after_launch("peer_exchange_pairs", k_)) return s;
    int64_t total = 0;
    uint32_t status = 0;
    CU(cudaMemcpyAsync(&total, g.jx_total, sizeof total, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaMemcpyAsync(&status, g.jx_status, sizeof status, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    if (status == 1)
        return fail(ADB_ERR_NOMEM, "adb_peer_exchange_pairs: a rank would receive more than the %llu pairs its region "
                    "holds (this rank: %lld); reserve more with adb_peer_join_create", g.jx_cap, (long long)total);
    if (status == 2) return fail(ADB_ERR_CUDA, "adb_peer_exchange_pairs: a peer did not arrive within 2 s (epoch %u)", x.epoch);
    *h_recv_count = total;
    *d_recv_val = g.jx_recv + key_off;
    *d_recv_pos = g.jx_recv + pay_off;
    return ADB_OK;
}

// ---- the same exchange group inside ONE process: contexts 0 .. world-1 are the ranks --------
// Peer access (cudaDeviceEnablePeerAccess + access to the stream-ordered pools) instead of IPC
// handles; contexts that share a device simply see each other's allocations.
static adb_status enable_peer_access(int world) {
    for (int i = 0; i < world; ++i) {
        const int di = g_ctx[i].device;
        CU(cudaSetDevice(di));
        for (int j = 0; j < world; ++j) {
            const int dj = g_ctx[j].device;
            if (di == dj) continue;
            int can = 0;
            CU(cudaDeviceCanAccessPeer(&can, di, dj));
            if (!can) return fail(ADB_ERR_CUDA, "device %d cannot access device %d's memory (NVLink / PCIe peer access is required)", di, dj);
            cudaError_t e = cudaDeviceEnablePeerAccess(dj, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else CU(e);
            // buffers of device dj's stream-ordered pool (columns, results) readable / writable from di
            cudaMemPool_t pool;
            CU(cudaDeviceGetDefaultMemPool(&pool, dj));
            cudaMemAccessDesc desc{};
            desc.location.type = cudaMemLocationTypeDevice;
            desc.location.id = di;
            desc.flags = cudaMemAccessFlagsProtReadWrite;
            CU(cudaMemPoolSetAccess(pool, &desc, 1));
        }
    }
    return ADB_OK;
}

adb_status adb_peer_connect_local(int32_t world) {
    if (world < 1 || world > ADB_MAX_PEERS || world > ADB_MAX_CONTEXTS)
        return fail(ADB_ERR_INVALID, "adb_peer_connect_local: world %d (max %d)", world, ADB_MAX_PEERS);
    for (int r = 0; r < world; ++r)
        if (!g_ctx[r].up) return fail(ADB_ERR_NOT_INITIALISED, "adb_peer_connect_local: context %d is not initialised", r);
    const int keep = g_cur;
    adb_status rc = enable_peer_access(world);
    for (int r = 0; r < world && rc == ADB_OK; ++r) {
        g_cur = r;
        auto one = [&]() -> adb_status {
            CU(cudaSetDevice(g.device));
            return peer_mailbox_create();
        };
        rc = one();
    }
    for (int r = 0; r < world && rc == ADB_OK; ++r) {
        g_cur = r;
        auto one = [&]() -> adb_status {
            CU(cudaSetDevice(g.device));
            for (int q = 0; q < world; ++q) g.peer_boxes.box[q] = g_ctx[q].peer_box;
            g.peer_world = world;
            g.peer_rank = r;
            g.peer_local = true;
            return peer_boxes_upload();
        };
        rc = one();
    }
    g_cur = keep;
    if (g.up) cudaSetDevice(g.device);
    return rc;
}

adb_status adb_peer_join_connect_local(int64_t cap_pairs) {
    const int world = g.peer_world;
    if (!g.peer_connected || !g.peer_local) return fail(ADB_ERR_INVALID, "adb_peer_join_connect_local: adb_peer_connect_local first");
    if (cap_pairs < 1 || cap_pairs >= ((int64_t)1 << 31))
        return fail(ADB_ERR_INVALID, "adb_peer_join_connect_local: capacity %lld outside [1, 2^31)", (long long)cap_pairs);
    const unsigned long long cap = ((unsigned long long)cap_pairs + 63) & ~63ull;
    const int keep = g_cur;
    adb_status rc = ADB_OK;
    for (int r = 0; r < world && rc == ADB_OK; ++r) {
        g_cur = r;
        auto one = [&]() -> adb_status {
            CU(cudaSetDevice(g.device));
            return jx_region_create(cap);
        };
        rc = one();
    }
    for (int r = 0; r < world && rc == ADB_OK; ++r) {
        g_cur = r;
        auto one = [&]() -> adb_status {
            CU(cudaSetDevice(g.device));
            for (int q = 0; q < world; ++q) g.jx_peer_host[q] = reinterpret_cast<uint32_t *>(g_ctx[q].jx_recv.p);
            return jx_table_upload();
        };
        rc = one();
    }
    g_cur = keep;
    if (g.up) cudaSetDevice(g.device);
    return rc;
}

// The current context's stream waits for everything enqueued so far on context `other`'s stream
// (`what` names the caller in errors).
static adb_status ctx_wait(int32_t other, const char *what) {
    NEED_UP();
    if (other < 0 || other >= ADB_MAX_CONTEXTS || !g_ctx[other].up)
        return fail(ADB_ERR_INVALID, "%s: context %d is not initialised", what, other);
    Engine &o = g_ctx[other];
    if (&o == &g) return ADB_OK;
    cudaEvent_t ev;
    CU(cudaSetDevice(o.device));
    CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CU(cudaEventRecord(ev, o.stream));
    CU(cudaSetDevice(g.device));
    CU(cudaStreamWaitEvent(g.stream, ev, 0));
    CU(cudaEventDestroy(ev));                      // released once the wait has consumed it
    return ADB_OK;
}

adb_status adb_ctx_wait(int32_t other_ctx) { return ctx_wait(other_ctx, "adb_ctx_wait"); }

// Copy between contexts (peer DMA when the devices differ), ordered on the CURRENT context's
// stream after everything already enqueued on the source context's stream: the wait, then the
// _ready copy.
adb_status adb_copy_from_ctx(void *d_dst, int32_t src_ctx, const void *d_src, size_t bytes) {
    if (bytes)
        if (adb_status s = ctx_wait(src_ctx, "adb_copy_from_ctx")) return s;
    return adb_copy_from_ctx_ready(d_dst, src_ctx, d_src, bytes);
}

// The same copy when the caller KNOWS the source bytes are complete (the source context has
// synchronised its stream and a host barrier lies in between): no event, no device switch --
// eight pulls per GPU and phase of the routed join probe would otherwise pay ~15 us each.
adb_status adb_copy_from_ctx_ready(void *d_dst, int32_t src_ctx, const void *d_src, size_t bytes) {
    NEED_UP();
    if (src_ctx < 0 || src_ctx >= ADB_MAX_CONTEXTS || !g_ctx[src_ctx].up)
        return fail(ADB_ERR_INVALID, "adb_copy_from_ctx_ready: context %d is not initialised", src_ctx);
    if (bytes == 0) return ADB_OK;
    if (!d_dst || !d_src) return fail(ADB_ERR_INVALID, "adb_copy_from_ctx_ready: NULL pointer");
    const Engine &src = g_ctx[src_ctx];
    if (src.device == g.device) CU(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, g.stream));
    else CU(cudaMemcpyPeerAsync(d_dst, g.device, d_src, src.device, bytes, g.stream));
    return ADB_OK;
}

adb_status adb_peer_destroy(void) {
    NEED_UP();
    CU(cudaStreamSynchronize(g.stream));
    peer_close();
    return ADB_OK;
}

adb_status adb_agg_export(const adb_agg *d_agg, int64_t *d_sum_count, int32_t *d_max_notmin) {
    NEED_UP();
    if (!d_agg || !d_sum_count || !d_max_notmin) return fail(ADB_ERR_INVALID, "adb_agg_export: NULL pointer");
    return after_launch("agg_export", adb::launch_agg_export(d_agg, d_sum_count, d_max_notmin, g.stream));
}
adb_status adb_agg_import(const int64_t *d_sum_count, const int32_t *d_max_notmin, adb_agg *d_agg) {
    NEED_UP();
    if (!d_agg || !d_sum_count || !d_max_notmin) return fail(ADB_ERR_INVALID, "adb_agg_import: NULL pointer");
    return after_launch("agg_import", adb::launch_agg_import(d_sum_count, d_max_notmin, d_agg, g.stream));
}

static adb_status ewise(const int32_t *a, const int32_t *b, int64_t n_max, const int64_t *d_n,
                        int32_t *out, bool subtract) {
    NEED_UP();
    if (adb_status s = check_len(n_max, subtract ? "adb_sub" : "adb_add")) return s;
    if (n_max == 0) return ADB_OK;
    if (!a || !b || !out) return fail(ADB_ERR_INVALID, "adb_add/adb_sub: NULL device pointer");
    const int k_ = adb::launch_ewise(a, b, n_max, d_n, out, subtract, g.sm_count, g.stream);
    return after_launch("ewise", k_);
}
adb_status adb_add(const int32_t *d_a, const int32_t *d_b, int64_t n_max, const int64_t *d_n,
                   int32_t *d_out) { return ewise(d_a, d_b, n_max, d_n, d_out, false); }
adb_status adb_sub(const int32_t *d_a, const int32_t *d_b, int64_t n_max, const int64_t *d_n,
                   int32_t *d_out) { return ewise(d_a, d_b, n_max, d_n, d_out, true); }

static adb_status chain_impl(const int32_t *d_sel_col, const int32_t *d_fetch_col,
                             int64_t n, const int32_t *lo, const int32_t *hi,
                             int32_t *d_pos_out, int32_t *d_val_out,
                             int64_t *d_count, adb_agg *d_agg, const adb::PeerExchange *px) {
    const char *what = "adb_chain_select_fetch_agg";
    adb::SelectArgs a;
    if (adb_status s = select_prepare(what, !d_count || !d_agg || (n > 0 && (!d_pos_out || !d_val_out || !d_fetch_col)),
                                      d_sel_col, n, nullptr, lo, hi, d_count, &a, true))
        return s;
    a.out = d_pos_out; a.fetch_col = d_fetch_col; a.val_out = d_val_out; a.agg_out = d_agg;
    // two launches: predicate pass -> bitmap, then expansion with the gather and the
    // aggregates fused in (positions and values are still materialised)
    const int32_t mb = g.chain_mark_base;
    g.chain_mark_base = -1;
    if (mb >= 0) adb_mark(mb);
    if (adb_status s = after_launch(what, adb::launch_select_mask(a, false, g.stream))) return s;
    if (mb >= 0) adb_mark(mb + 1);
    const adb_status s = fused_finish(what, a, d_count, px, nullptr);
    if (mb >= 0) adb_mark(mb + 2);
    return s;
}

adb_status adb_chain_select_fetch_agg(const int32_t *d_sel_col, const int32_t *d_fetch_col,
                                      int64_t n, const int32_t *lo, const int32_t *hi,
                                      int32_t *d_pos_out, int32_t *d_val_out,
                                      int64_t *d_count, adb_agg *d_agg) {
    return chain_impl(d_sel_col, d_fetch_col, n, lo, hi, d_pos_out, d_val_out, d_count, d_agg, nullptr);
}

// The chain with NEITHER handle materialised (SURVEY.md 8f rank 3): one kernel scans the select
// column and gathers + folds the fetch column at every hit -- 4N + 4H bytes, no bitmap, no lists.
adb_status adb_chain_select_agg(const int32_t *d_sel_col, const int32_t *d_fetch_col, int64_t n,
                                const int32_t *lo, const int32_t *hi, int64_t *d_count, adb_agg *d_agg,
                                adb_agg *h_agg) {
    adb::SelectArgs a;
    if (adb_status s = select_prepare("adb_chain_select_agg", !d_count || !d_agg || (n > 0 && !d_fetch_col),
                                      d_sel_col, n, nullptr, lo, hi, d_count, &a, true))
        return s;
    a.fetch_col = d_fetch_col; a.agg_out = d_agg;
    const int f_ = adb::launch_scan_gather_agg(a, g.stream);
    if (f_ > 0) {
        if (adb_status s = after_launch("chain (unmaterialised)", f_)) return s;
    } else {
        // empty column: the aggregate of nothing
        CU(cudaMemsetAsync(d_count, 0, sizeof(int64_t), g.stream));
        if (adb_status s = adb_aggregate(d_sel_col, 0, nullptr, d_agg, nullptr)) return s;
    }
    if (h_agg) return read_back(h_agg, d_agg, sizeof(adb_agg));
    return ADB_OK;
}

adb_status adb_chain_select_fetch_agg_exchange(const int32_t *d_sel_col, const int32_t *d_fetch_col,
                                               int64_t n, const int32_t *lo, const int32_t *hi,
                                               int32_t *d_pos_out, int32_t *d_val_out, int64_t *d_count,
                                               adb_agg *d_parts, int32_t k, adb_agg *d_out) {
    adb::PeerExchange px;
    if (adb_status s = peer_exchange("adb_chain_select_fetch_agg_exchange", d_parts, k, d_out, &px)) return s;
    if (k < 1 || !d_parts || !d_out) return fail(ADB_ERR_INVALID, "adb_chain_select_fetch_agg_exchange: bad arguments");
    const adb_status s = chain_impl(d_sel_col, d_fetch_col, n, lo, hi, d_pos_out, d_val_out, d_count,
                                    d_parts + (k - 1), &px);
    if (s == ADB_OK) ++g.peer_epoch;          // the exchange was enqueued: every rank advances together
    return s;
}

// ---- batched shared scan -------------------------------------------------------------------
constexpr size_t kSsBoundsBytes = 4 * 2 * ADB_MAX_BATCH;                 // 1200
// cov_off: 2 * (2 * ADB_MAX_BATCH + 2) = 604 bytes, padded to 640
constexpr size_t kSsLutOff = kSsBoundsBytes + 640;
constexpr size_t kSsLutBytes = ((2 * (adb::kSsLut + 1) + 15) / 16) * 16;
constexpr size_t kSsBitsOff = kSsLutOff + kSsLutBytes;
constexpr size_t kSsQOff = kSsBitsOff + adb::kSsBits / 8;            // q_first | q_last, uint16 each
constexpr size_t kSsCov4Off = kSsQOff + 2 * 2 * ((ADB_MAX_BATCH + 7) / 8) * 8;   // 4 query ids per interval id
// cov_q comes last: a plan is uploaded up to the end of its cover lists (a few hundred bytes for
// the usual batch, 45 KB for 150 nested queries)
constexpr size_t kSsCovOff = kSsCov4Off + 4 * (2 * ADB_MAX_BATCH + 8);
constexpr size_t kSsCovBytes = 2 * ADB_MAX_BATCH * ADB_MAX_BATCH;        // 45000
constexpr size_t kSsPlanBytes = kSsCovOff + ((kSsCovBytes + 15) / 16) * 16;
constexpr size_t kSsMaxChunks = 8192;

// The host half of the batched scan: everything the kernels look up, in one packed buffer
// (bounds | cov_off | cov_q | lut | bits | q_first/q_last | cov4).  Pure host code: also
// reachable without a device through adb_shared_select_plan (tests).
struct SsHostPlan {
    std::vector<unsigned char> bytes;
    uint32_t m = 0, lut_shift = 0, bit_shift = 0, span = 0, deepest = 1;
    int32_t lo = 0;
};
static void ss_build_plan(const int32_t *lows, const int32_t *highs, int32_t q_count, SsHostPlan *hp) {
    // ---- elementary intervals: interval k = [bounds[k-1], bounds[k]), ids 0 and m lie outside
    int32_t bounds[2 * ADB_MAX_BATCH];
    uint32_t m = 0;
    for (int32_t q = 0; q < q_count; ++q)
        if (lows[q] < highs[q]) { bounds[m++] = lows[q]; bounds[m++] = highs[q]; }
    std::sort(bounds, bounds + m);
    m = (uint32_t)(std::unique(bounds, bounds + m) - bounds);
    // query q = [low, high) covers the interval ids (index of low) + 1 .. (index of high)
    uint16_t qf[ADB_MAX_BATCH], ql[ADB_MAX_BATCH];
    uint16_t off[2 * ADB_MAX_BATCH + 2] = {0};               // CSR offsets of the cover lists
    for (int32_t q = 0; q < q_count; ++q) {
        qf[q] = 1;
        ql[q] = 0;
        if (lows[q] < highs[q]) {
            qf[q] = (uint16_t)(std::lower_bound(bounds, bounds + m, lows[q]) - bounds + 1);
            ql[q] = (uint16_t)(std::lower_bound(bounds, bounds + m, highs[q]) - bounds);
            for (uint32_t k = qf[q]; k <= ql[q]; ++k) ++off[k + 1];    // counts first
        }
    }
    uint32_t deepest = 1;                                    // most queries covering one value
    for (uint32_t k = 1; k <= m + 1; ++k) {
        deepest = std::max<uint32_t>(deepest, off[k]);
        off[k] = (uint16_t)(off[k] + off[k - 1]);
    }
    const uint32_t cov_total = m ? off[m + 1] : 0;           // <= 299 * 150 < 2^16
    std::vector<unsigned char> &plan = hp->bytes;
    plan.assign(kSsCovOff + ((cov_total + 15) / 16) * 16, 0);
    if (m) memcpy(plan.data(), bounds, m * sizeof(int32_t));
    memcpy(plan.data() + kSsBoundsBytes, off, (m + 2) * sizeof(uint16_t));
    uint8_t *cov = plan.data() + kSsCovOff;                  // query ids ascending inside an interval
    {
        uint16_t cur[2 * ADB_MAX_BATCH + 2];
        memcpy(cur, off, sizeof cur);
        for (int32_t q = 0; q < q_count; ++q)
            for (uint32_t k = qf[q]; k <= ql[q]; ++k) cov[cur[k]++] = (uint8_t)q;
    }
    memcpy(plan.data() + kSsQOff, qf, sizeof(uint16_t) * (size_t)q_count);
    memcpy(plan.data() + kSsQOff + 2 * (((ADB_MAX_BATCH + 7) / 8) * 8), ql, sizeof(uint16_t) * (size_t)q_count);
    // ---- value -> interval tables over d = v - bounds[0] in [0, span)
    uint32_t lut_shift = 0, bit_shift = 0, span = 0;
    uint16_t *lut = reinterpret_cast<uint16_t *>(plan.data() + kSsLutOff);
    uint32_t *bits = reinterpret_cast<uint32_t *>(plan.data() + kSsBitsOff);
    if (m) {
        const uint32_t ulo = (uint32_t)bounds[0];
        span = (uint32_t)bounds[m - 1] - ulo;
        while ((span >> lut_shift) >= adb::kSsLut) ++lut_shift;
        while ((span >> bit_shift) >= adb::kSsBits) ++bit_shift;
        // lut[k] = number of bounds strictly below the lower edge of bucket k
        uint32_t a = 0;
        for (uint32_t k = 0; k <= adb::kSsLut; ++k) {
            const uint64_t edge = (uint64_t)k << lut_shift;
            while (a < m && (uint64_t)((uint32_t)bounds[a] - ulo) < edge) ++a;
            lut[k] = (uint16_t)a;
        }
        // interval ids reachable from bucket k: lut[k] .. lut[k+1]; none covered -> bit 15
        uint16_t prev = lut[0];
        for (uint32_t k = 0; k < adb::kSsLut; ++k) {
            const uint16_t next = lut[k + 1];
            bool covered = false;
            for (uint32_t i = prev; i <= next && !covered; ++i) covered = off[i + 1] != off[i];
            lut[k] = covered ? prev : (uint16_t)(prev | 0x8000u);
            prev = next;
        }
        // fine bitmap: every bucket a covered interval reaches into; runs of covered intervals
        // are filled a word at a time
        for (uint32_t k = 1; k < m;) {
            if (off[k + 1] == off[k]) { ++k; continue; }
            uint32_t e = k;
            while (e + 1 < m && off[e + 2] != off[e + 1]) ++e;             // covered run k .. e
            const uint32_t t0 = ((uint32_t)bounds[k - 1] - ulo) >> bit_shift;
            const uint32_t t1 = ((uint32_t)bounds[e] - 1u - ulo) >> bit_shift;
            const uint32_t w0 = t0 >> 5, w1 = t1 >> 5;
            const uint32_t head = 0xFFFFFFFFu << (t0 & 31), tail = 0xFFFFFFFFu >> (31 - (t1 & 31));
            if (w0 == w1) {
                bits[w0] |= head & tail;
            } else {
                bits[w0] |= head;
                for (uint32_t w = w0 + 1; w < w1; ++w) bits[w] = 0xFFFFFFFFu;
                bits[w1] |= tail;
            }
            k = e + 1;
        }
    }
    // ---- pair lists (<= 4 queries deep): the queries are coloured so that overlapping ones get
    // different colours -- they are intervals, so going through them by lower bound and taking
    // the lowest colour no still-open query holds needs exactly `deepest` colours -- and every
    // interval id lists its covering queries BY COLOUR (0xFF = none).  The classify pass then
    // emits a batch's pairs colour by colour: a query lives in one colour, so its pairs stay in
    // row order, which is all the emit pass needs.
    uint32_t *cov4 = reinterpret_cast<uint32_t *>(plan.data() + kSsCov4Off);
    for (uint32_t k = 0; k <= m + 1; ++k) cov4[k] = 0xFFFFFFFFu;
    if (deepest <= 4) {
        int32_t order[ADB_MAX_BATCH];
        int32_t live = 0;
        for (int32_t q = 0; q < q_count; ++q) if (lows[q] < highs[q]) order[live++] = q;
        std::sort(order, order + live, [&](int32_t x, int32_t y) {
            return lows[x] != lows[y] ? lows[x] < lows[y] : x < y; });
        int32_t open_high[4];
        bool open_used[4] = {false, false, false, false};
        uint8_t colour[ADB_MAX_BATCH] = {0};
        for (int32_t i = 0; i < live; ++i) {
            const int32_t q = order[i];
            int c = -1;
            for (int k = 0; k < 4; ++k) {
                if (open_used[k] && open_high[k] <= lows[q]) open_used[k] = false;     // closed before q opens
                if (c < 0 && !open_used[k]) c = k;
            }
            if (c < 0) { deepest = 5; break; }               // cannot happen for depth <= 4; stay safe
            open_used[c] = true;
            open_high[c] = highs[q];
            colour[q] = (uint8_t)c;
        }
        if (deepest <= 4)
            for (uint32_t k = 1; k < m; ++k)
                for (uint32_t c = off[k]; c < off[k + 1]; ++c) {
                    const uint32_t q = cov[c], sh = 8u * colour[q];
                    cov4[k] = (cov4[k] & ~(0xFFu << sh)) | (q << sh);
                }
    }
    hp->m = m; hp->lut_shift = lut_shift; hp->bit_shift = bit_shift; hp->span = span;
    hp->deepest = deepest; hp->lo = m ? bounds[0] : 0;
}

static adb_status shared_select_count_impl(const int32_t *d_col, int64_t n, const int32_t *lows,
                                           const int32_t *highs, int32_t q_count, int64_t *h_counts);
adb_status adb_shared_select_count(const int32_t *d_col, int64_t n, const int32_t *lows,
                                   const int32_t *highs, int32_t q_count, int64_t *h_counts) {
    NEED_UP();
    g.ss_base_pos = 0;
    return shared_select_count_impl(d_col, n, lows, highs, q_count, h_counts);
}
// over rows [base_pos, base_pos + n) of a column (shard): the emit phase writes base_pos + row
adb_status adb_shared_select_count_base(const int32_t *d_col, int64_t n, int32_t base_pos, const int32_t *lows,
                                        const int32_t *highs, int32_t q_count, int64_t *h_counts) {
    NEED_UP();
    g.ss_base_pos = base_pos;
    return shared_select_count_impl(d_col, n, lows, highs, q_count, h_counts);
}
static adb_status shared_select_count_impl(const int32_t *d_col, int64_t n, const int32_t *lows,
                                           const int32_t *highs, int32_t q_count, int64_t *h_counts) {
    NEED_UP();
    g.ss_ready = false;
    if (adb_status s = check_len(n, "adb_shared_select_count")) return s;
    if (q_count < 1 || q_count > ADB_MAX_BATCH)
        return fail(ADB_ERR_INVALID, "adb_shared_select_count: q_count %d outside [1, %d] (server.c:366-371 chunks "
                    "batches to 150)", q_count, ADB_MAX_BATCH);
    if (!lows || !highs || (n > 0 && !d_col)) return fail(ADB_ERR_INVALID, "adb_shared_select_count: NULL pointer");
    if (adb_status s = grow(g.ss_plan_mem, kSsPlanBytes, "shared scan plan")) return s;
    if (adb_status s = grow(g.ss_counts, sizeof(uint32_t) * ADB_MAX_BATCH * kSsMaxChunks, "shared scan counts")) return s;
    if (adb_status s = grow(g.ss_totals, sizeof(int64_t) * ADB_MAX_BATCH, "shared scan totals")) return s;
    if (adb_status s = grow(g.ss_outs, sizeof(int32_t *) * ADB_MAX_BATCH, "shared scan outputs")) return s;
    if (adb_status s = grow(g.ss_chunk_hits, sizeof(uint32_t) * kSsMaxChunks, "shared scan chunk hits")) return s;
    SsHostPlan hp;
    ss_build_plan(lows, highs, q_count, &hp);
    // one packed upload, staged through a pinned slot (the host vector goes out of scope below)
    if (adb_status s = upload_blob(g.ss_plan_mem, hp.bytes.data(), hp.bytes.size())) return s;
    const uint32_t m = hp.m, lut_shift = hp.lut_shift, bit_shift = hp.bit_shift, span = hp.span, deepest = hp.deepest;
    g.ss_plan = adb::SharedScanPlan{reinterpret_cast<const int32_t *>(g.ss_plan_mem.p),
                                    reinterpret_cast<const uint16_t *>(g.ss_plan_mem + kSsBoundsBytes),
                                    g.ss_plan_mem + kSsCovOff, m, (uint32_t)q_count,
                                    reinterpret_cast<const uint16_t *>(g.ss_plan_mem + kSsLutOff),
                                    reinterpret_cast<const uint32_t *>(g.ss_plan_mem + kSsBitsOff),
                                    lut_shift, bit_shift, hp.lo, span,
                                    reinterpret_cast<const uint16_t *>(g.ss_plan_mem + kSsQOff),
                                    reinterpret_cast<const uint16_t *>(g.ss_plan_mem + kSsQOff) + ((ADB_MAX_BATCH + 7) / 8) * 8,
                                    0u, reinterpret_cast<const uint32_t *>(g.ss_plan_mem + kSsCov4Off)};
    if (n == 0) {
        for (int32_t q = 0; q < q_count; ++q) if (h_counts) h_counts[q] = 0;
        g.ss_geom = adb::SharedScanGeom{0, 0, 0};
        g.ss_ready = true;
        return ADB_OK;
    }
    g.ss_geom = adb::shared_scan_geom((uint32_t)n, g.sm_count);
    if (g.ss_geom.num_chunks > kSsMaxChunks) return fail(ADB_ERR_INVALID, "shared scan: chunk table overflow");
    // pair lists while they stay small: <= 4 queries deep and <= 4 GB of scratch
    size_t rows = (size_t)g.ss_geom.num_chunks * g.ss_geom.chunk_rows;
    if (deepest <= 4 && rows * deepest * sizeof(uint32_t) <= ((size_t)4 << 30) && !getenv("ADB_SS_INTERVAL_LISTS")) {
        g.ss_plan.pair_depth = deepest;
        rows *= deepest;
    }
    if (adb_status s = grow(g.ss_hits, rows * sizeof(uint32_t), "shared scan hit lists")) return s;
    const int k_ = adb::launch_shared_classify(d_col, (uint32_t)n, g.ss_plan, g.ss_geom, g.ss_hits,
                                               g.ss_chunk_hits, g.ss_counts, g.ss_totals, g.stream);
    if (adb_status s = after_launch("shared_classify", k_)) return s;
    if (h_counts) {
        if (adb_status s = read_back(h_counts, g.ss_totals, sizeof(int64_t) * q_count)) return s;
    }
    g.ss_ready = true;
    return ADB_OK;
}

adb_status adb_shared_select_emit(int32_t *const *d_out_ptrs, int64_t capacity) {
    NEED_UP();
    if (!g.ss_ready) return fail(ADB_ERR_INVALID, "adb_shared_select_emit: no preceding adb_shared_select_count");
    if (!d_out_ptrs) return fail(ADB_ERR_INVALID, "adb_shared_select_emit: NULL pointer");
    g.ss_ready = false;
    if (g.ss_geom.num_chunks == 0) return ADB_OK;
    if (adb_status s = upload_blob(g.ss_outs, d_out_ptrs, sizeof(int32_t *) * g.ss_plan.q_count)) return s;
    const int k_ = adb::launch_shared_emit(g.ss_hits, g.ss_chunk_hits, g.ss_plan, g.ss_geom, g.ss_counts,
                                           g.ss_outs, capacity, (uint32_t)g.ss_base_pos, g.stream);
    return after_launch("shared_emit", k_);
}

// Host-only: the plan adb_shared_select_count would upload for this batch (no device needed).
adb_status adb_shared_select_plan(const int32_t *lows, const int32_t *highs, int32_t q_count,
                                  unsigned char *plan_out, size_t capacity, uint32_t *meta_out) {
    if (q_count < 1 || q_count > ADB_MAX_BATCH || !lows || !highs || !meta_out)
        return fail(ADB_ERR_INVALID, "adb_shared_select_plan: bad arguments");
    SsHostPlan hp;
    ss_build_plan(lows, highs, q_count, &hp);
    const uint32_t meta[16] = {(uint32_t)hp.bytes.size(), hp.m, hp.lut_shift, hp.bit_shift, hp.span,
                               (uint32_t)hp.lo, hp.deepest, (uint32_t)kSsBoundsBytes,
                               (uint32_t)kSsCovOff, (uint32_t)kSsLutOff, (uint32_t)kSsBitsOff,
                               (uint32_t)kSsQOff, (uint32_t)kSsCov4Off, adb::kSsLut, adb::kSsBits,
                               (uint32_t)(((ADB_MAX_BATCH + 7) / 8) * 8)};
    memcpy(meta_out, meta, sizeof meta);
    if (plan_out) {
        if (capacity < hp.bytes.size()) return fail(ADB_ERR_INVALID, "adb_shared_select_plan: buffer too small");
        memcpy(plan_out, hp.bytes.data(), hp.bytes.size());
    }
    return ADB_OK;
}

// ---- radix sort / partition helpers ---------------------------------------------------------
static adb_status ensure_radix_scratch(uint32_t n) {
    // <= 256 segments (segmented pass)
    if (adb_status s = grow(g.rx_totals, sizeof(uint32_t) * 256 * 256, "radix totals")) return s;
    if (adb_status s = grow(g.rx_base, sizeof(uint32_t) * 256 * 256, "radix bases")) return s;
    if (adb_status s = grow(g.sc_sums, sizeof(unsigned long long) * (size_t)(g.sm_count * 2 + 8), "scan chunk sums"))
        return s;
    // [segment][bucket][tiles per segment]: <= 256 segments, the last one padded
    return grow(g.rx_hist, sizeof(uint32_t) * 256 * ((size_t)adb::radix_geom(n, g.sm_count).ctas + 256),
                "radix histogram");
}

static RadixBufs radix_layout(Carve &c, uint32_t n) {
    const size_t m = n ? n : 1;
    return {{c.take<uint32_t>(m), c.take<uint32_t>(m)}, {c.take<uint32_t>(m), c.take<uint32_t>(m)}};
}

// Runs `npass` stable passes over (keys, payload) through the buffers `b`; payload starts as pay0,
// or the row index.  The last pass writes to (final_k, final_v) when given.
static adb_status radix_run(const uint32_t *keys_in, uint32_t n, const adb::RadixPass *passes, int npass,
                            const RadixBufs &b, uint32_t *final_k, uint32_t *final_v, uint32_t **keys_out,
                            uint32_t **pay_out, int *launches, const uint32_t *pay0 = nullptr) {
    *keys_out = nullptr;
    *pay_out = nullptr;
    if (adb_status s = ensure_radix_scratch(n)) return s;
    const uint32_t *src_k = keys_in, *src_v = pay0;       // pay0 == NULL: payload = row index
    int cur = 0;
    for (int p = 0; p < npass; ++p) {
        uint32_t *dk = b.k[cur], *dv = b.v[cur];
        if (p == npass - 1 && final_k && final_v) { dk = final_k; dv = final_v; }
        *launches += adb::launch_radix_pass(src_k, src_v, dk, dv, n, passes[p], g.rx_hist,
                                            g.rx_totals, g.rx_base, g.sm_count, g.stream);
        src_k = dk;
        src_v = dv;
        cur ^= 1;
    }
    *keys_out = const_cast<uint32_t *>(src_k);
    *pay_out = const_cast<uint32_t *>(src_v);
    return ADB_OK;
}

adb_status adb_index_sort(const int32_t *d_col, int64_t n, int32_t *d_values_out,
                          int32_t *d_positions_out) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_index_sort")) return s;
    if (n == 0) return ADB_OK;
    if (!d_col || !d_values_out || !d_positions_out) return fail(ADB_ERR_INVALID, "adb_index_sort: NULL pointer");
    const adb::RadixPass passes[4] = {{0, 8, 0}, {8, 8, 0}, {16, 8, 0}, {24, 8, 0}};
    RadixBufs b;
    if (adb_status s = arena_take([&](Carve &c) { b = radix_layout(c, (uint32_t)n); }, "adb_index_sort", true)) return s;
    uint32_t *k = nullptr, *v = nullptr;
    int launches = 0;
    if (adb_status s = radix_run(reinterpret_cast<const uint32_t *>(d_col), (uint32_t)n, passes, 4, b,
                                 reinterpret_cast<uint32_t *>(d_values_out),
                                 reinterpret_cast<uint32_t *>(d_positions_out), &k, &v, &launches)) return s;
    return after_launch("index_sort", launches);
}

// Scratch of adb_index_sort_ref_ties: the radix sort's buffers (afterwards the two (values,
// positions) pairs the levels alternate between), event slots, the dup prefix, per-tile and
// per-segment tables.  A big segment has more than kTiesSmall rows, so a level holds at most
// n / (kTiesSmall + 1) + 1 of them and hands out at most twice that many small ones.
struct TiesBufs {
    RadixBufs rx;
    uint32_t *ev, *dex;
    uint4 *tile_cnt, *info;
    uint32_t *tile_pre;
    adb::TiesBig *big[2];
    uint2 *small[2];
    adb::TiesCounters *ctr;
    unsigned long long *dups;
    int64_t *dex_total;
};
static TiesBufs ties_layout(Carve &c, uint32_t n) {
    const size_t m = n ? n : 1;
    const size_t max_big = n / (adb::kTiesSmall + 1) + 1;
    const size_t max_tiles = n / adb::kTiesTile + 1 + max_big;
    TiesBufs b;
    b.rx = radix_layout(c, n);
    b.ev = c.take<uint32_t>(m);
    b.dex = c.take<uint32_t>(m);
    b.tile_cnt = c.take<uint4>(max_tiles);
    b.tile_pre = c.take<uint32_t>(max_tiles);
    b.info = c.take<uint4>(max_big);
    for (int k = 0; k < 2; ++k) {
        b.big[k] = c.take<adb::TiesBig>(max_big);
        b.small[k] = c.take<uint2>(2 * max_big + 1);
    }
    b.ctr = c.take<adb::TiesCounters>(1);
    b.dups = c.take<unsigned long long>(1);
    b.dex_total = c.take<int64_t>(1);
    return b;
}

adb_status adb_index_sort_ref_ties(const int32_t *d_col, int64_t n, int32_t *d_values_out,
                                   int32_t *d_positions_out) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_index_sort_ref_ties")) return s;
    if (n == 0) return ADB_OK;
    if (!d_col || !d_values_out || !d_positions_out)
        return fail(ADB_ERR_INVALID, "adb_index_sort_ref_ties: NULL pointer");
    const uint32_t un = (uint32_t)n;
    TiesBufs b;
    if (adb_status s = arena_take([&](Carve &c) { b = ties_layout(c, un); }, "adb_index_sort_ref_ties", true)) return s;
    // the values are the radix sort's; so are the positions when no key repeats
    const adb::RadixPass passes[4] = {{0, 8, 0}, {8, 8, 0}, {16, 8, 0}, {24, 8, 0}};
    uint32_t *k = nullptr, *v = nullptr;
    int launches = 0;
    uint32_t *pos_out = reinterpret_cast<uint32_t *>(d_positions_out);
    if (adb_status s = radix_run(reinterpret_cast<const uint32_t *>(d_col), un, passes, 4, b.rx,
                                 reinterpret_cast<uint32_t *>(d_values_out), pos_out, &k, &v, &launches)) return s;
    launches += adb::launch_ties_dups(d_values_out, un, nullptr, b.dups, g.sm_count, g.stream);
    if (adb_status s = after_launch("index_sort_ref_ties", launches)) return s;
    unsigned long long dups = 0;
    if (adb_status s = read_back(&dups, b.dups, sizeof dups)) return s;
    if (dups == 0) return ADB_OK;

    launches = adb::launch_ties_dups(d_values_out, un, b.ev, b.dups, g.sm_count, g.stream);
    launches += adb::launch_exclusive_scan(b.ev, 1, b.dex, un, g.sc_sums, b.dex_total, g.sm_count, g.stream);
    int32_t *vals[2] = {reinterpret_cast<int32_t *>(b.rx.k[0]), reinterpret_cast<int32_t *>(b.rx.k[1])};
    uint32_t *poss[2] = {b.rx.v[0], b.rx.v[1]};
    launches += adb::launch_ties_init(d_col, un, vals[0], poss[0], b.big[0], b.small[0], g.sm_count, g.stream);
    adb::TiesLevel a{};
    a.keys = d_values_out;
    a.dex = b.dex;
    a.ev = b.ev;
    a.pos_out = pos_out;
    a.tile_cnt = b.tile_cnt;
    a.tile_pre = b.tile_pre;
    a.info = b.info;
    a.ctr_next = b.ctr;
    const bool first_big = un > adb::kTiesSmall;
    uint32_t nbig = first_big, ntiles = first_big ? (un + adb::kTiesTile - 1) / adb::kTiesTile : 0;
    uint32_t nsmall = !first_big;
    int levels = 0;
    for (int cur = 0; nbig || nsmall; cur ^= 1, ++levels) {
        a.cv = vals[cur];
        a.cp = poss[cur];
        a.nv = vals[cur ^ 1];
        a.np = poss[cur ^ 1];
        a.big = b.big[cur];
        a.small = b.small[cur];
        a.big_next = b.big[cur ^ 1];
        a.small_next = b.small[cur ^ 1];
        a.nbig = nbig;
        a.ntiles = ntiles;
        a.nsmall = nsmall;
        CU(cudaMemsetAsync(b.ctr, 0, sizeof *b.ctr, g.stream));
        launches += adb::launch_ties_level(a, g.stream);
        if (adb_status s = after_launch("index_sort_ref_ties level", launches)) return s;
        launches = 0;
        adb::TiesCounters c;
        if (adb_status s = read_back(&c, b.ctr, sizeof c)) return s;
        nbig = (uint32_t)(c.big >> 32);
        ntiles = (uint32_t)c.big;
        nsmall = c.small;
    }
    // ADB_TRACE=1: how deep the quicksort's recursion went (one readback per level)
    if (getenv("ADB_TRACE")) fprintf(stderr, "index_sort_ref_ties: %d levels\n", levels);
    return ADB_OK;
}

// ---- index build over several contexts: exact splitters, range routing, pairs sort -------------
adb_status adb_rank_hist(const int32_t *d_col, int64_t n, const uint32_t *h_prefixes, int32_t n_prefixes,
                         int32_t round, uint32_t *h_hist) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_rank_hist")) return s;
    if (round < 0 || round > 3 || n_prefixes < 1 || n_prefixes > ADB_MAX_PEERS || !h_prefixes || !h_hist)
        return fail(ADB_ERR_INVALID, "adb_rank_hist: round %d must be in [0, 3], prefixes %d in [1, %d]", round,
                    n_prefixes, ADB_MAX_PEERS);
    for (int32_t i = 0; i < n_prefixes; ++i)
        if (((uint64_t)h_prefixes[i] >> (8 * round)) || (i && h_prefixes[i] <= h_prefixes[i - 1]))
            return fail(ADB_ERR_INVALID, "adb_rank_hist: prefixes must be ascending and below 2^%d", 8 * round);
    if (n > 0 && !d_col) return fail(ADB_ERR_INVALID, "adb_rank_hist: NULL pointer");
    uint32_t *pre = nullptr, *hist = nullptr;
    if (adb_status s = arena_take([&](Carve &c) {
            pre = c.take<uint32_t>(ADB_MAX_PEERS);
            hist = c.take<uint32_t>((size_t)ADB_MAX_PEERS * 256);
        }, "adb_rank_hist", true)) return s;
    const size_t hist_bytes = sizeof(uint32_t) * 256 * (size_t)n_prefixes;
    if (adb_status s = upload_blob(pre, h_prefixes, sizeof(uint32_t) * (size_t)n_prefixes)) return s;
    CU(cudaMemsetAsync(hist, 0, hist_bytes, g.stream));
    const int k_ = adb::launch_rank_hist(d_col, (uint32_t)n, pre, (uint32_t)n_prefixes, (uint32_t)round, hist,
                                         g.sm_count, g.stream);
    if (adb_status s = after_launch("rank_hist", k_)) return s;
    return read_back(h_hist, hist, hist_bytes);
}

adb_status adb_route_range(const int32_t *d_keys, int64_t n, int64_t row_base, const int32_t *h_splitters,
                           int32_t parts, int32_t *d_keys_out, int32_t *d_rows_out, int64_t *h_counts) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_route_range")) return s;
    if (parts < 1 || parts > ADB_MAX_PEERS || !h_counts || (parts > 1 && !h_splitters))
        return fail(ADB_ERR_INVALID, "adb_route_range: parts must be in [1, %d]", ADB_MAX_PEERS);
    if (row_base < 0 || row_base + n > ((int64_t)1 << 31))
        return fail(ADB_ERR_INVALID, "adb_route_range: rows %lld + %lld past 2^31", (long long)row_base, (long long)n);
    for (int32_t i = 1; i + 1 < parts; ++i)
        if (h_splitters[i] < h_splitters[i - 1])
            return fail(ADB_ERR_INVALID, "adb_route_range: splitters must not decrease");
    if (n > 0 && (!d_keys || !d_keys_out || !d_rows_out))
        return fail(ADB_ERR_INVALID, "adb_route_range: NULL device pointer");
    for (int32_t r = 0; r < parts; ++r) h_counts[r] = 0;
    if (n == 0) return ADB_OK;
    int32_t split[adb::kRangeSplitters + 1];
    for (int i = 0; i <= adb::kRangeSplitters; ++i) split[i] = i + 1 < parts ? h_splitters[i] : INT32_MAX;
    int32_t *d_split = nullptr;
    uint32_t *rows = nullptr;
    if (adb_status s = arena_take([&](Carve &c) {
            d_split = c.take<int32_t>(adb::kRangeSplitters + 1);
            rows = c.take<uint32_t>((size_t)n);
        }, "adb_route_range", true)) return s;
    if (adb_status s = ensure_radix_scratch((uint32_t)n)) return s;
    if (adb_status s = upload_blob(d_split, split, sizeof split)) return s;
    const uint64_t at = reinterpret_cast<uintptr_t>(d_split);
    adb::RadixPass pass{(int)(uint32_t)at, 0, 4};
    pass.split_hi = (uint32_t)(at >> 32);
    while ((1 << pass.bits) < parts) ++pass.bits;
    int k_ = adb::launch_iota(reinterpret_cast<int32_t *>(rows), n, (int32_t)row_base, g.sm_count, g.stream);
    k_ += adb::launch_radix_pass(reinterpret_cast<const uint32_t *>(d_keys), rows,
                                 reinterpret_cast<uint32_t *>(d_keys_out), reinterpret_cast<uint32_t *>(d_rows_out),
                                 (uint32_t)n, pass, g.rx_hist, g.rx_totals, g.rx_base, g.sm_count, g.stream);
    if (adb_status s = after_launch("route_range", k_)) return s;
    uint32_t totals[ADB_MAX_PEERS];
    CU(cudaMemcpyAsync(totals, g.rx_totals, sizeof(uint32_t) * parts, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    for (int32_t r = 0; r < parts; ++r) h_counts[r] = totals[r];
    return ADB_OK;
}

adb_status adb_index_sort_pairs(const int32_t *d_keys, const int32_t *d_payload, int64_t n, int32_t *d_values_out,
                                int32_t *d_payload_out) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_index_sort_pairs")) return s;
    if (n == 0) return ADB_OK;
    if (!d_keys || !d_payload || !d_values_out || !d_payload_out)
        return fail(ADB_ERR_INVALID, "adb_index_sort_pairs: NULL pointer");
    const adb::RadixPass passes[4] = {{0, 8, 0}, {8, 8, 0}, {16, 8, 0}, {24, 8, 0}};
    RadixBufs b;
    if (adb_status s = arena_take([&](Carve &c) { b = radix_layout(c, (uint32_t)n); }, "adb_index_sort_pairs", true))
        return s;
    uint32_t *k = nullptr, *v = nullptr;
    int launches = 0;
    if (adb_status s = radix_run(reinterpret_cast<const uint32_t *>(d_keys), (uint32_t)n, passes, 4, b,
                                 reinterpret_cast<uint32_t *>(d_values_out),
                                 reinterpret_cast<uint32_t *>(d_payload_out), &k, &v, &launches,
                                 reinterpret_cast<const uint32_t *>(d_payload))) return s;
    return after_launch("index_sort_pairs", launches);
}

// Multi-GPU join exchange, send side: stable partition of a (value, position) pair list by
// destination rank = route_owner of the value (its routing hash is independent of the join's own
// partition hash, so the receiving rank's local partitions stay balanced).
adb_status adb_route_pairs(const int32_t *d_val, const int32_t *d_pos, int64_t n, int32_t parts,
                           int32_t *d_val_out, int32_t *d_pos_out, int64_t *h_counts) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_route_pairs")) return s;
    if (parts < 1 || parts > 256 || !h_counts)
        return fail(ADB_ERR_INVALID, "adb_route_pairs: parts must be in [1, 256]");
    if (n > 0 && (!d_val || !d_pos || !d_val_out || !d_pos_out))
        return fail(ADB_ERR_INVALID, "adb_route_pairs: NULL device pointer");
    for (int32_t r = 0; r < parts; ++r) h_counts[r] = 0;
    if (n == 0) return ADB_OK;
    if (parts == 1) {
        CU(cudaMemcpyAsync(d_val_out, d_val, n * 4, cudaMemcpyDeviceToDevice, g.stream));
        CU(cudaMemcpyAsync(d_pos_out, d_pos, n * 4, cudaMemcpyDeviceToDevice, g.stream));
        h_counts[0] = n;
        return ADB_OK;
    }
    if (adb_status s = ensure_radix_scratch((uint32_t)n)) return s;
    const int k_ = adb::launch_radix_pass(reinterpret_cast<const uint32_t *>(d_val),
                                          reinterpret_cast<const uint32_t *>(d_pos),
                                          reinterpret_cast<uint32_t *>(d_val_out),
                                          reinterpret_cast<uint32_t *>(d_pos_out), (uint32_t)n,
                                          routing_pass(parts), g.rx_hist, g.rx_totals,
                                          g.rx_base, g.sm_count, g.stream);
    if (adb_status s = after_launch("route_pairs", k_)) return s;
    uint32_t totals[256];
    CU(cudaMemcpyAsync(totals, g.rx_totals, sizeof(uint32_t) * parts, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    for (int32_t r = 0; r < parts; ++r) h_counts[r] = totals[r];
    return ADB_OK;
}

// ---- bulk CSV load ---------------------------------------------------------------------------------
adb_status adb_csv_index(const char *d_text, size_t bytes, int32_t skip_lines, int64_t *h_rows) {
    NEED_UP();
    auto &c = g.csv;
    c.ready = false;
    c.fill_ready = false;
    if (skip_lines < 0 || !h_rows || (bytes && !d_text)) return fail(ADB_ERR_INVALID, "adb_csv_index: bad arguments");
    if (adb_status s = grow(c.col_table, 256 * sizeof(int32_t *), "csv column table")) return s;
    if (adb_status s = grow(c.flags, 4 * sizeof(uint32_t), "csv flags")) return s;
    if (adb_status s = grow(c.total, 2 * sizeof(int64_t), "csv line count")) return s;
    c.text = reinterpret_cast<const unsigned char *>(d_text);
    c.bytes = bytes;
    c.skip = (uint32_t)skip_lines;
    c.newlines = 0;
    c.rows = 0;
    if (bytes == 0) { *h_rows = 0; c.ready = true; return ADB_OK; }
    if (reinterpret_cast<uintptr_t>(d_text) & 15u) return fail(ADB_ERR_INVALID, "adb_csv_index: text must be 16-byte aligned (adb_alloc is)");
    const uint32_t blocks = adb::csv_blocks(bytes);
    if (adb_status s = grow(c.block_counts, sizeof(uint32_t) * blocks, "csv block counts")) return s;
    if (adb_status s = grow(c.block_base, sizeof(uint32_t) * blocks, "csv block bases")) return s;
    if (adb_status s = ensure_radix_scratch(1)) return s;            // the scan's chunk sums live there
    int k_ = adb::launch_csv_count(c.text, bytes, c.block_counts, g.stream);
    k_ += adb::launch_exclusive_scan(c.block_counts, 1, c.block_base, blocks, g.sc_sums, c.total, g.sm_count, g.stream);
    int64_t newlines = 0;
    unsigned char last = 0;
    CU(cudaMemcpyAsync(&newlines, c.total, sizeof newlines, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaMemcpyAsync(&last, c.text + bytes - 1, 1, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    if (newlines >= (int64_t)1 << 32) return fail(ADB_ERR_INVALID, "adb_csv_index: %lld lines in one call; split the text at a line boundary", (long long)newlines);
    if (adb_status s = grow(c.line_end, sizeof(unsigned long long) * ((size_t)newlines + 1), "csv line ends")) return s;
    k_ += adb::launch_csv_index(c.text, bytes, c.block_base, c.line_end, g.stream);
    if (adb_status s = after_launch("csv_index", k_)) return s;
    const unsigned long long lines = (unsigned long long)newlines + (last != '\n' ? 1 : 0);
    c.newlines = (unsigned long long)newlines;
    c.rows = lines > c.skip ? lines - c.skip : 0;
    if (adb_status s = check_len((int64_t)c.rows, "adb_csv_index")) return s;
    *h_rows = (int64_t)c.rows;
    c.ready = true;
    return ADB_OK;
}

// Parse the indexed rows into d_cols; *h_short = some row had fewer than n_cols fields.  With
// `summary`, also the piece's last value of every column (c.piece); when a row was short, the
// tile records the fill needs are left in c.tile_last.
static adb_status csv_parse_rows(const char *what, int32_t n_cols, int32_t *const *d_cols, bool summary,
                                 bool *h_short) {
    auto &c = g.csv;
    *h_short = false;
    if (!c.ready) return fail(ADB_ERR_INVALID, "%s: no preceding adb_csv_index", what);
    c.ready = false;
    c.fill_ready = false;
    if (n_cols < 1 || n_cols > 254 || !d_cols) return fail(ADB_ERR_INVALID, "%s: n_cols %d outside [1, 254]", what, n_cols);
    if (c.rows == 0 && !summary) return ADB_OK;
    for (int32_t i = 0; i < n_cols; ++i)
        if (!d_cols[i] && c.rows) return fail(ADB_ERR_INVALID, "%s: column %d is NULL", what, i);
    if (adb_status s = grow(c.n_fields, (size_t)c.rows + 1, "csv field counts")) return s;
    if (adb_status s = grow(c.piece, 3 * 256 * sizeof(int32_t), "csv piece summary")) return s;
    if (adb_status s = upload_blob(c.col_table, d_cols, sizeof(int32_t *) * n_cols)) return s;
    CU(cudaMemsetAsync(c.flags, 0, 4 * sizeof(uint32_t), g.stream));
    int k_ = adb::launch_csv_parse(c.text, c.bytes, c.line_end, c.newlines, c.skip, c.rows, (uint32_t)n_cols,
                                   c.col_table, c.n_fields, c.flags, g.stream);
    uint32_t flags[2] = {0, 0};
    CU(cudaMemcpyAsync(flags, c.flags, sizeof flags, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    if (adb_status s = after_launch("csv_parse", k_)) return s;
    if (flags[1])
        return fail(ADB_ERR_INVALID, "%s: a line is longer than 1023 bytes (fgets would split it, "
                    "src/db_manager.c:23,306)", what);
    c.n_cols = (uint32_t)n_cols;
    *h_short = flags[0] != 0;
    if (*h_short) {
        const uint32_t tiles = adb::csv_tiles(c.rows);
        if (adb_status s = grow(c.tile_last, sizeof(int32_t) * (size_t)tiles * n_cols, "csv fill tiles")) return s;
        k_ = adb::launch_csv_tile_scan(c.rows, (uint32_t)n_cols, c.col_table, c.n_fields, c.tile_last, c.piece,
                                       g.stream);
        if (adb_status s = after_launch("csv_tile_scan", k_)) return s;
        c.fill_ready = true;
    } else if (summary) {
        k_ = adb::launch_csv_last_row(c.rows, (uint32_t)n_cols, c.col_table, c.piece, g.stream);
        if (adb_status s = after_launch("csv_last_row", k_)) return s;
    }
    return ADB_OK;
}

static adb_status csv_fill(const int32_t *h_carry) {
    auto &c = g.csv;
    if (!c.fill_ready) return ADB_OK;                                 // no short row: nothing to fill
    c.fill_ready = false;
    if (h_carry) {
        if (adb_status s = upload_blob(c.piece + 512, h_carry, sizeof(int32_t) * c.n_cols)) return s;
    } else {
        CU(cudaMemsetAsync(c.piece + 512, 0, sizeof(int32_t) * c.n_cols, g.stream));
    }
    const int k_ = adb::launch_csv_fill(c.rows, c.n_cols, c.col_table, c.n_fields, c.tile_last, c.piece + 512, g.stream);
    return after_launch("csv_fill", k_);
}

adb_status adb_csv_parse(int32_t n_cols, int32_t *const *d_cols) {
    NEED_UP();
    bool short_rows = false;
    if (adb_status s = csv_parse_rows("adb_csv_parse", n_cols, d_cols, false, &short_rows)) return s;
    return csv_fill(nullptr);                                          // a missing field of the first rows is 0
}

adb_status adb_csv_parse_piece(int32_t n_cols, int32_t *const *d_cols, int32_t *h_last, int32_t *h_has,
                               int32_t *h_short) {
    NEED_UP();
    if (!h_last || !h_has || !h_short) return fail(ADB_ERR_INVALID, "adb_csv_parse_piece: NULL output");
    bool short_rows = false;
    if (adb_status s = csv_parse_rows("adb_csv_parse_piece", n_cols, d_cols, true, &short_rows)) return s;
    auto &c = g.csv;
    int32_t sum[512];
    CU(cudaMemcpyAsync(sum, c.piece, sizeof sum, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    for (int32_t i = 0; i < n_cols; ++i) {
        h_last[i] = sum[i];
        h_has[i] = sum[256 + i];
    }
    *h_short = short_rows;
    return ADB_OK;
}

adb_status adb_csv_fill(const int32_t *h_carry) {
    NEED_UP();
    return csv_fill(h_carry);
}

// ---- result text ------------------------------------------------------------------------------------
adb_status adb_format_i32_count(const int32_t *d_val, int64_t n, int64_t *h_bytes) {
    NEED_UP();
    auto &f = g.fmt;
    f.ready = false;
    if (adb_status s = check_len(n, "adb_format_i32_count")) return s;
    if (!h_bytes || (n > 0 && !d_val)) return fail(ADB_ERR_INVALID, "adb_format_i32_count: NULL pointer");
    f.val = d_val;
    f.n = n;
    f.bytes = 0;
    if (n == 0) { *h_bytes = 0; f.ready = true; return ADB_OK; }
    if (adb_status s = grow(f.total, 2 * sizeof(int64_t), "print byte count")) return s;
    const uint32_t blocks = adb::fmt_blocks(n);
    if (adb_status s = grow(f.block_len, sizeof(uint32_t) * blocks, "print block lengths")) return s;
    if (adb_status s = grow(f.block_off, sizeof(uint32_t) * blocks, "print block offsets")) return s;
    if (adb_status s = ensure_radix_scratch(1)) return s;
    int k_ = adb::launch_fmt_len(d_val, n, f.block_len, g.stream);
    k_ += adb::launch_exclusive_scan(f.block_len, 1, f.block_off, blocks, g.sc_sums, f.total, g.sm_count, g.stream);
    int64_t total = 0;
    CU(cudaMemcpyAsync(&total, f.total, sizeof total, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    if (adb_status s = after_launch("format_count", k_)) return s;
    if (total - 1 >= (int64_t)1 << 32)
        return fail(ADB_ERR_INVALID, "adb_format_i32_count: %lld bytes of text; format at most 4 GiB per call", (long long)total - 1);
    f.bytes = total - 1;                            // no separator after the last value
    *h_bytes = f.bytes;
    f.ready = true;
    return ADB_OK;
}

adb_status adb_format_i32_emit(char *d_text) {
    NEED_UP();
    auto &f = g.fmt;
    if (!f.ready) return fail(ADB_ERR_INVALID, "adb_format_i32_emit: no preceding adb_format_i32_count");
    f.ready = false;
    if (f.n == 0) return ADB_OK;
    if (!d_text || (reinterpret_cast<uintptr_t>(d_text) & 15u))
        return fail(ADB_ERR_INVALID, "adb_format_i32_emit: the text buffer must be 16-byte aligned device memory");
    const int k_ = adb::launch_fmt_emit(f.val, f.n, f.block_off, reinterpret_cast<unsigned char *>(d_text),
                                        (uint64_t)f.bytes, g.stream);
    return after_launch("format_emit", k_);
}

// ---- hash join ------------------------------------------------------------------------------------
static void join_release() { g.join = Engine::JoinState{}; }      // its buffers are arena memory

// ADB_TRACE=1: synchronise after every stage of a join and print its wall-clock time.
struct StageTrace {
    bool on;
    std::chrono::steady_clock::time_point t;
    StageTrace() : on(getenv("ADB_TRACE") != nullptr), t(std::chrono::steady_clock::now()) {}
    void lap(const char *what) {
        if (!on) return;
        cudaStreamSynchronize(g.stream);
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[adb trace] %-28s %9.3f ms\n", what,
                std::chrono::duration<double, std::milli>(now - t).count());
        t = now;
    }
};

// build = the side whose rows are grouped (the reference's column_one for hash_join);
// probe = the side walked in row order.  Output pair k is (build position, probe position).
//
// join_build: steps 1-3 (sort on the hash, partition boundaries, one table per partition);
// leaves {build_pos_sorted, part_bits} in g.join and the tables in g.hj_table.
// Probe rows partitioned for L2 locality (hash_join.cu, P1-P3) when the tables will not fit L2
// by a wide margin (`by_size`: each caller's own size rule).  ADB_JOIN_PROBE=direct /
// partitioned overrides (tests run both forms on the same inputs).
static bool join_probe_partitioned(bool by_size) {
    const char *e = getenv("ADB_JOIN_PROBE");
    if (e && !strcmp(e, "direct")) return false;
    if (e && !strcmp(e, "partitioned")) return true;
    return by_size;
}

static uint32_t join_part_bits(uint32_t nb) {
    uint32_t part_bits = 1;                    // >= 1: the table's key tag needs one spare bit
    // (up to 2^20 partitions: a 500 M-row build side still gets ~500-row partitions that fit the
    // shared-memory table, instead of 2^16 oversized ones built slot by slot in global memory)
    while (part_bits < 20 && (nb >> part_bits) > 1024) ++part_bits;
    return part_bits;
}

static JoinBuildBufs join_build_layout(Carve &c, uint32_t nb) {
    const uint32_t num_parts = 1u << join_part_bits(nb);
    return {c.take<uint32_t>(num_parts + 1), c.take<unsigned long long>(num_parts + 1),
            c.take<unsigned long long>(num_parts / 1024 + 2), radix_layout(c, nb)};
}

// The partitioned probe's (P1-P3) windows: <= 256 of whole 4096-row tiles.
static uint32_t probe_window_tiles(uint32_t n) { return ((n + adb::kRadixTile - 1) / adb::kRadixTile + 255) / 256; }

// A probe of n keys by the one-GPU join, by adb_join_finish_routed (partitioned geometry; the rows
// come back probed) or by the owner of received keys (answers straight into g.rt_recv_res).
// warp_base: per-warp match counts, scanned into every warp's first output slot.
enum ProbeUser { kJoinProbe, kFinishProbe, kOwnerProbe };
static ProbeBufs probe_layout(Carve &c, uint32_t n, bool partitioned, ProbeUser who) {
    ProbeBufs b;
    b.pg = partitioned ? adb::hj_probe_geom_partitioned(n) : adb::hj_probe_geom(n, g.sm_count);
    b.tot = c.take<unsigned long long>(2);
    if (who != kOwnerProbe) b.gc_by_j = c.take<uint2>(n);
    b.warp_base = c.take<unsigned long long>(b.pg.warps);
    if (!partitioned) return b;
    b.chunk_sums = c.take<unsigned long long>(b.pg.warps / 1024 + 2);
    if (who == kFinishProbe) return b;
    b.pk = c.take<uint32_t>(n);
    b.rows = c.take<uint32_t>(n);
    b.res = c.take<uint2>(n);
    if (who == kJoinProbe) return b;
    // the owner's own: g.rx_hist / g.rx_base still hold the routing pass adb_join_finish_routed reads
    const uint32_t segs = adb::radix_segments(n, probe_window_tiles(n));
    b.hist = c.take<uint32_t>(adb::radix_hist_elems(n, probe_window_tiles(n)));
    b.totals = c.take<uint32_t>((size_t)segs * 256);
    b.base = c.take<uint32_t>((size_t)segs * 256);
    return b;
}

static RouteState route_layout(Carve &c, uint32_t n, size_t answer_bytes) {
    return {c.take<uint32_t>(n), c.take<uint32_t>(n), c.take<unsigned char>((size_t)n * answer_bytes), n};
}

// What adb_join_build reserves for nb build rows and np probe rows of this context: the build, the
// routed rows, the owner's probe of about as many received keys and the finish.  The owner picks
// its probe form from what is left, so adb_peer_exchange_reserve reserves exactly this.
static size_t join_arena_bytes(uint32_t nb, uint32_t np) {
    Carve c;
    join_build_layout(c, nb);
    route_layout(c, np, sizeof(uint2));
    probe_layout(c, np, true, kOwnerProbe);
    probe_layout(c, INT32_MAX, false, kOwnerProbe);   // the direct probe's sums stop growing at 8 CTAs per SM
    probe_layout(c, np, true, kFinishProbe);
    return c.used;
}

// P1-P3 of the partitioned probe (hash_join.cu): a segmented pass on the top 8 hash bits over the
// windows, then the probe slice by slice, the results gathered back into key order in gc_by_j.
static int probe_partitioned(const uint32_t *keys, uint32_t n, const ProbeBufs &b, uint32_t *hist, uint32_t *totals,
                             uint32_t *base, uint2 *gc_by_j, StageTrace *tr) {
    const uint32_t want_tiles = probe_window_tiles(n);
    int k_ = adb::launch_radix_pass_segmented(keys, nullptr, b.pk, b.rows, n, adb::RadixPass{24, 8, 1}, want_tiles,
                                              hist, totals, base, g.sm_count, g.stream);
    if (tr) tr->lap("probe rows by window and table slice");
    return k_ + adb::launch_hj_probe_partitioned(b.pk, b.rows, base, hist, adb::radix_segments(n, want_tiles),
                                                 adb::radix_seg_tiles(n, want_tiles), n, b.pg, g.join.build.toff,
                                                 g.join.part_bits, g.hj_table, b.res, gc_by_j, b.warp_base,
                                                 b.chunk_sums, b.tot, g.stream);
}

static adb_status join_build(const int32_t *bv, const int32_t *bp, uint32_t nb, int *launches, StageTrace &tr) {
    const uint32_t part_bits = join_part_bits(nb);
    const uint32_t num_parts = 1u << part_bits;
    auto &j = g.join;
    j.part_bits = part_bits;
    j.n_build = nb;
    const JoinBuildBufs &b = j.build;
    if (nb == 0) {                             // an owner without build rows: every partition is empty
        CU(cudaMemsetAsync(b.toff, 0, (size_t)(num_parts + 1) * 8, g.stream));
        j.build_pos_sorted = nullptr;
        return ADB_OK;
    }
    // 1. build side: full stable sort on the bijective hash; the payload carried through the
    //    passes is the build position itself, so nothing is gathered afterwards
    const adb::RadixPass sort4[4] = {{0, 8, 1}, {8, 8, 1}, {16, 8, 1}, {24, 8, 1}};
    uint32_t *bk = nullptr, *bi = nullptr;
    if (adb_status s = radix_run(reinterpret_cast<const uint32_t *>(bv), nb, sort4, 4, b.radix, nullptr, nullptr, &bk,
                                 &bi, launches, reinterpret_cast<const uint32_t *>(bp))) return s;
    j.build_pos_sorted = reinterpret_cast<int32_t *>(bi);
    tr.lap("build sort");
    // 2. partition boundaries -> table geometry: partition p gets a power-of-two slot range
    //    holding its rows at <= 80 % load (<= 4096 slots: built in shared memory)
    *launches += adb::launch_hj_bounds(bk, nb, part_bits, num_parts, b.off1, g.stream);
    *launches += adb::launch_hj_geometry(b.off1, num_parts, b.toff, b.chunk_sums, g.stream);
    unsigned long long slots = 0;
    if (adb_status s = read_back(&slots, b.toff + num_parts, sizeof slots)) return s;
    if (adb_status s = grow(g.hj_table, slots * 16, "join tables")) return s;
    tr.lap("partition boundaries");
    // 3. one table per partition
    *launches += adb::launch_hj_table_build(bk, j.build_pos_sorted, b.off1, b.toff, num_parts, part_bits,
                                            g.hj_table, g.stream);
    tr.lap("per-partition tables");
    return ADB_OK;
}

static adb_status join_count(const int32_t *bv, const int32_t *bp, int64_t nb64, const int32_t *pv,
                             const int32_t *pp, int64_t np64, bool swapped, int64_t *h_matches) {
    NEED_UP();
    join_release();
    if (adb_status s = check_len(nb64, "adb_join")) return s;
    if (adb_status s = check_len(np64, "adb_join")) return s;
    if ((nb64 > 0 && (!bv || !bp)) || (np64 > 0 && (!pv || !pp)))
        return fail(ADB_ERR_INVALID, "adb_join: NULL device pointer");
    const uint32_t nb = (uint32_t)nb64, np = (uint32_t)np64;
    if (nb == 0 || np == 0) {
        auto &j0 = g.join;
        j0.swapped = swapped; j0.n_probe = np; j0.probe_pos = pp; j0.matches = 0; j0.ready = true;
        if (h_matches) *h_matches = 0;
        return ADB_OK;
    }
    int launches = 0;
    StageTrace tr;
    // ~21 bytes of table per build row against 126 MB of L2
    const bool partitioned = join_probe_partitioned(nb >= (6u << 20) && np >= (4u << 20));
    if (partitioned)
        if (adb_status s = ensure_radix_scratch(np > nb ? np : nb)) return s;
    if (adb_status s = arena_take([&](Carve &c) {
            g.join.build = join_build_layout(c, nb);
            g.join.probe = probe_layout(c, np, partitioned, kJoinProbe);
        }, "adb_join", true)) return s;
    if (adb_status s = join_build(bv, bp, nb, &launches, tr)) return s;
    auto &j = g.join;
    j.swapped = swapped;
    j.n_probe = np;
    j.probe_pos = pp;
    // 4. probe in row order; every warp leaves the matches of its piece, their scan = the
    //    first output slot of every piece (the expansion computes the slots inside a piece)
    const ProbeBufs &pb = j.probe;
    const uint32_t *pkeys = reinterpret_cast<const uint32_t *>(pv);
    launches += partitioned ? probe_partitioned(pkeys, np, pb, g.rx_hist, g.rx_totals, g.rx_base, pb.gc_by_j, &tr)
                            : adb::launch_hj_probe(pkeys, np, pb.pg, j.build.toff, j.part_bits, g.hj_table, pb.gc_by_j,
                                                   pb.warp_base, pb.tot, g.stream);
    if (adb_status s = read_back(&j.matches, pb.tot, sizeof(int64_t))) return s;
    tr.lap(partitioned ? "probe slice by slice + back to row order" : "probe + piece offsets");
    if (adb_status s = after_launch("join_count", launches)) return s;
    if (j.matches >= (int64_t)1 << 31) {
        const long long m = j.matches;
        join_release();
        return fail(ADB_ERR_INVALID, "join produces %lld pairs; the reference indexes its output with an int "
                    "(query.c:657) so the result must stay below 2^31", m);
    }
    j.ready = true;
    if (h_matches) *h_matches = j.matches;
    return ADB_OK;
}

// ---- the join sharded over the contexts of one process (SURVEY.md 8e) ----------------------------
// Every context calls adb_join_build on its share of the build side (what adb_peer_exchange_pairs
// delivered), the host waits for all of them, then every context's probe rows go through the
// routed probe below and adb_join_emit.  The probe rows keep their original order, so the
// contexts' outputs concatenated in shard order are the reference's probe-major list.
adb_status adb_join_build(const int32_t *d_v, const int32_t *d_p, int64_t n, int64_t probe_rows_hint) {
    NEED_UP();
    join_release();
    if (adb_status s = check_len(n, "adb_join_build")) return s;
    if (adb_status s = check_len(probe_rows_hint, "adb_join_build")) return s;
    if (n > 0 && (!d_v || !d_p)) return fail(ADB_ERR_INVALID, "adb_join_build: NULL device pointer");
    int launches = 0;
    StageTrace tr;
    if (adb_status s = ensure_radix_scratch((uint32_t)(n ? n : 1))) return s;
    if (adb_status s = arena_reserve(join_arena_bytes((uint32_t)n, (uint32_t)probe_rows_hint))) return s;
    if (adb_status s = arena_take([&](Carve &c) { g.join.build = join_build_layout(c, (uint32_t)n); }, "adb_join_build"))
        return s;
    if (adb_status s = join_build(d_v, d_p, (uint32_t)n, &launches, tr)) return s;
    if (adb_status s = after_launch("join_build", launches)) return s;
    CU(cudaStreamSynchronize(g.stream));               // the other contexts' probes read these tables
    g.join.built = true;
    g.join.n_probe = (uint32_t)probe_rows_hint;
    return ADB_OK;
}

// ---- routed exchange (adb_engine.h): the sharded join's probe and the routed fetch ---------------
// Step 1 on the home side: one stable pass (`pass` picks the owner's digit) groups this context's n
// items by owner into the arena, with their row numbers and room for answer_bytes of answer each;
// h_counts[o] = items bound for owner o.  The arena is reserved here for this exchange alone when
// `reserve` (a join waiting for its emit phase is dropped), else the one adb_join_build reserved
// is used.  The pass' scanned histogram stays in g.rx_hist / g.rx_base for step 3.
static adb_status route_partition(const char *what, int32_t world, const int32_t *d_in, int64_t n64,
                                  adb::RadixPass pass, size_t answer_bytes, bool reserve, RouteState &rt,
                                  int64_t *h_counts, const int32_t **d_routed, void **d_answers) {
    if (adb_status s = check_len(n64, what)) return s;
    if (!h_counts || !d_routed || !d_answers || (n64 > 0 && !d_in)) return fail(ADB_ERR_INVALID, "%s: NULL pointer", what);
    for (int r = 0; r < world; ++r) h_counts[r] = 0;
    *d_routed = nullptr;
    *d_answers = nullptr;
    const uint32_t n = (uint32_t)n64;
    rt.n = n;
    if (n == 0) return ADB_OK;
    if (adb_status s = ensure_radix_scratch(n)) return s;
    if (adb_status s = arena_take([&](Carve &c) { rt = route_layout(c, n, answer_bytes); }, what, reserve)) return s;
    const int k_ = adb::launch_radix_pass_segmented(reinterpret_cast<const uint32_t *>(d_in), nullptr, rt.items,
                                                    rt.rows, n, pass, 0, g.rx_hist, g.rx_totals, g.rx_base,
                                                    g.sm_count, g.stream);
    if (adb_status s = after_launch(what, k_)) return s;
    uint32_t totals[ADB_MAX_PEERS];
    CU(cudaMemcpyAsync(totals, g.rx_totals, sizeof(uint32_t) * world, cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    for (int r = 0; r < world; ++r) h_counts[r] = totals[r];
    *d_routed = reinterpret_cast<const int32_t *>(rt.items);
    *d_answers = rt.answers;
    return ADB_OK;
}

// The sharded join's probe routes the keys to their route_owner; the owner probes
// them against its own tables and the rows' home puts the 8-byte answers back in row order (the
// same gather as the one-GPU partitioned probe; cells = owners).  Probing in place and reading
// each remote key's slot over NVLink instead costs one 32-byte response per 16 useful bytes, 8.8 G
// reads/s per GPU: 1.2 ms for the 11 M remote rows of an 8-GPU 100 M-row probe, and the whole
// 100 M x 100 M join on 8 GPUs took 2.71 ms that way against 2.08 ms routed
// (profiles/r02_join_sharded.md).
adb_status adb_join_route_probe(int32_t world, const int32_t *d_pv, int64_t np64, int64_t *h_counts,
                                const int32_t **d_routed_keys, void **d_answers) {
    NEED_UP();
    auto &j = g.join;
    if (!j.built) return fail(ADB_ERR_INVALID, "adb_join_route_probe: no preceding adb_join_build on this context");
    if (world < 2 || world > ADB_MAX_PEERS)
        return fail(ADB_ERR_INVALID, "adb_join_route_probe: world %d must be in [2, %d]", world, ADB_MAX_PEERS);
    if (np64 > (int64_t)j.n_probe) return fail(ADB_ERR_INVALID, "adb_join_route_probe: more probe rows than adb_join_build reserved for");
    if (adb_status s = route_partition("adb_join_route_probe", world, d_pv, np64, routing_pass(world),
                                       sizeof(uint2), false, j.route, h_counts, d_routed_keys, d_answers))
        return s;
    j.routed = true;
    return ADB_OK;
}

adb_status adb_join_recv_buffers(int64_t n_recv, int32_t **d_keys, void **d_answers) {
    NEED_UP();
    if (adb_status s = check_len(n_recv, "adb_join_recv_buffers")) return s;
    if (!d_keys || !d_answers) return fail(ADB_ERR_INVALID, "adb_join_recv_buffers: NULL pointer");
    if (adb_status s = grow(g.rt_recv_keys, (size_t)n_recv * 4, "routed probe: received keys")) return s;
    if (adb_status s = grow(g.rt_recv_res, (size_t)n_recv * 8, "routed probe: answers")) return s;
    *d_keys = reinterpret_cast<int32_t *>(g.rt_recv_keys.p);
    *d_answers = g.rt_recv_res.p;
    return ADB_OK;
}

adb_status adb_join_probe_received(int64_t n_recv) {
    NEED_UP();
    auto &j = g.join;
    if (!j.built) return fail(ADB_ERR_INVALID, "adb_join_probe_received: no tables on this context");
    if (adb_status s = check_len(n_recv, "adb_join_probe_received")) return s;
    if ((size_t)n_recv * 4 > g.rt_recv_keys.cap || (size_t)n_recv * 8 > g.rt_recv_res.cap)
        return fail(ADB_ERR_INVALID, "adb_join_probe_received: more keys than adb_join_recv_buffers made room for");
    if (n_recv == 0) return ADB_OK;
    const uint32_t n = (uint32_t)n_recv;
    StageTrace tr;
    // A table well beyond L2 (two or four GPUs: >= 24 M build rows here) is probed slice by slice like
    // the one-GPU join's.  No room for that next to what adb_join_finish_routed still takes for this
    // context's own probe rows (a skewed key set sent most of the probe side here): the direct probe.
    Carve need;
    probe_layout(need, n, true, kOwnerProbe);
    probe_layout(need, j.route.n, true, kFinishProbe);
    const bool partitioned = join_probe_partitioned(n >= (4u << 20) && j.n_build >= (24u << 20)) &&
                             g.arena_used + need.used <= g.arena.cap;
    ProbeBufs b;
    if (adb_status s = arena_take([&](Carve &c) { b = probe_layout(c, n, partitioned, kOwnerProbe); },
                                  "adb_join_probe_received")) return s;
    const int k_ = partitioned
        ? probe_partitioned(g.rt_recv_keys, n, b, b.hist, b.totals, b.base, g.rt_recv_res, nullptr)
        : adb::launch_hj_probe_plain(g.rt_recv_keys, n, j.build.toff, j.part_bits, g.hj_table, g.rt_recv_res,
                                     b.warp_base, g.sm_count, g.stream);
    if (adb_status s = after_launch("join_probe_received", k_)) return s;
    CU(cudaStreamSynchronize(g.stream));               // the rows' homes pull the answers next
    tr.lap("received keys in + probe");
    return ADB_OK;
}

adb_status adb_join_finish_routed(int32_t world, const int32_t *d_pv, const int32_t *d_pp, int64_t np64,
                                  int32_t swapped, int64_t *h_matches) {
    NEED_UP();
    auto &j = g.join;
    if (!j.built || !j.routed) return fail(ADB_ERR_INVALID, "adb_join_finish_routed: no preceding adb_join_route_probe");
    if (world < 2 || world > ADB_MAX_PEERS)
        return fail(ADB_ERR_INVALID, "adb_join_finish_routed: world %d must be in [2, %d]", world, ADB_MAX_PEERS);
    if ((uint32_t)np64 != j.route.n) return fail(ADB_ERR_INVALID, "adb_join_finish_routed: row count differs from adb_join_route_probe");
    if (np64 > 0 && (!d_pv || !d_pp)) return fail(ADB_ERR_INVALID, "adb_join_finish_routed: NULL device pointer");
    const uint32_t np = (uint32_t)np64;
    adb::JoinOwners o{};
    for (int r = 0; r < world; ++r) {
        const Engine &E = g_ctx[r];
        if (!E.up || !E.join.built) return fail(ADB_ERR_INVALID, "adb_join_finish_routed: context %d has built no tables", r);
        o.bpos[r] = E.join.build_pos_sorted;
    }
    o.count = (uint32_t)world;
    j.owners = o;
    j.sharded = true;
    j.swapped = swapped != 0;
    j.n_probe = np;
    j.probe_pos = d_pp;
    j.probe_keys = reinterpret_cast<const uint32_t *>(d_pv);
    j.matches = 0;
    j.routed = false;
    if (np == 0) {
        j.ready = true;
        if (h_matches) *h_matches = 0;
        return ADB_OK;
    }
    if (adb_status s = arena_take([&](Carve &c) { j.probe = probe_layout(c, np, true, kFinishProbe); },
                                  "adb_join_finish_routed")) return s;
    const ProbeBufs &b = j.probe;
    StageTrace tr;
    int launches = adb::launch_hj_unpartition_routed(j.route.rows, static_cast<const uint2 *>(j.route.answers),
                                                     g.rx_base, g.rx_hist, np, (uint32_t)world, b.pg, b.gc_by_j,
                                                     b.warp_base, b.chunk_sums, b.tot, g.stream);
    if (adb_status s = read_back(&j.matches, b.tot, sizeof(int64_t))) return s;
    tr.lap("answers back to row order + piece offsets");
    if (adb_status s = after_launch("join_finish_routed", launches)) return s;
    if (j.matches >= (int64_t)1 << 31)
        return fail(ADB_ERR_INVALID, "join produces %lld pairs on one context; the result must stay below 2^31",
                    (long long)j.matches);
    j.ready = true;
    if (h_matches) *h_matches = j.matches;
    return ADB_OK;
}

// ---- routed fetch over a position list that is not aligned with the column's shards ---------------
// adb_fetch_sharded reads every remote row over NVLink, 4 useful bytes per 32-byte response
// (~12 G rows/s per GPU: an index-ordered 10 % select + fetch over 500 M rows took 3.6 ms on two
// GPUs against 1.2 ms on one).  Routed instead: the positions go to the GPUs that hold the rows
// (the digit is the shard, position / shard_rows), those gather locally (adb_fetch with the
// shard's base) and the list's home puts the 4-byte values back in list order.  It reserves the
// sort / join arena afresh: a join waiting for its emit phase is dropped.
adb_status adb_route_rows(int32_t world, int64_t shard_rows, const int32_t *d_pos, int64_t n64, int64_t *h_counts,
                          const int32_t **d_routed_pos, void **d_answers) {
    NEED_UP();
    if (world < 2 || world > ADB_MAX_PEERS) return fail(ADB_ERR_INVALID, "adb_route_rows: world %d must be in [2, %d]", world, ADB_MAX_PEERS);
    if (shard_rows < 1 || shard_rows > 0x7FFFFFFF) return fail(ADB_ERR_INVALID, "adb_route_rows: bad shard size");
    int bits = 1;
    while ((1 << bits) < world) ++bits;
    adb::RadixPass pass{0, bits, 3};
    pass.div = (uint32_t)shard_rows;
    return route_partition("adb_route_rows", world, d_pos, n64, pass, sizeof(uint32_t), true, g.fetch_route, h_counts,
                           d_routed_pos, d_answers);
}

adb_status adb_route_finish32(int32_t world, int32_t *d_out, int64_t n64) {
    NEED_UP();
    RouteState &rt = g.fetch_route;
    if (world < 2 || world > ADB_MAX_PEERS) return fail(ADB_ERR_INVALID, "adb_route_finish32: world %d must be in [2, %d]", world, ADB_MAX_PEERS);
    if ((uint32_t)n64 != rt.n) return fail(ADB_ERR_INVALID, "adb_route_finish32: row count differs from adb_route_rows");
    if (n64 == 0) return ADB_OK;
    if (!d_out) return fail(ADB_ERR_INVALID, "adb_route_finish32: NULL output");
    const int k_ = adb::launch_rows_unpartition32(rt.rows, static_cast<const uint32_t *>(rt.answers), g.rx_base,
                                                  g.rx_hist, rt.n, (uint32_t)world, reinterpret_cast<uint32_t *>(d_out),
                                                  g.stream);
    rt.n = 0;
    return after_launch("route_finish32", k_);
}

// Everything adb_peer_exchange_pairs / adb_join_build allocate, sized up front.  Device memory
// management can wait for the device to go idle; a context that did that while a peer context
// ON THE SAME DEVICE sits in the exchange's spin-wait for it would stall both (contexts sharing
// a device is the 1-GPU test configuration).  Call on every context, wait for all, then start
// the collective.
adb_status adb_peer_exchange_reserve(int64_t send_pairs, int64_t build_pairs, int64_t probe_rows) {
    NEED_UP();
    if (adb_status s = check_len(send_pairs, "adb_peer_exchange_reserve")) return s;
    if (adb_status s = check_len(build_pairs, "adb_peer_exchange_reserve")) return s;
    if (adb_status s = check_len(probe_rows, "adb_peer_exchange_reserve")) return s;
    uint32_t big = (uint32_t)(send_pairs > build_pairs ? send_pairs : build_pairs);
    if ((uint32_t)probe_rows > big) big = (uint32_t)probe_rows;            // the routed probe's partition pass
    if (adb_status s = ensure_radix_scratch(big ? big : 1)) return s;
    const uint32_t nb = (uint32_t)build_pairs, np = (uint32_t)probe_rows;
    if (adb_status s = arena_reserve(join_arena_bytes(nb, np))) return s;
    const uint32_t num_parts = 1u << join_part_bits(nb);
    // tables: <= 2.5 slots per build row (power-of-two capacity at <= 80 % load) + 16 per partition
    const unsigned long long slots = (unsigned long long)nb * 5 / 2 + 16ull * num_parts + 4096;
    return grow(g.hj_table, slots * 16, "join tables");
}

adb_status adb_hash_join_count(const int32_t *d_v1, const int32_t *d_p1, int64_t n1,
                               const int32_t *d_v2, const int32_t *d_p2, int64_t n2,
                               int64_t *h_matches) {
    return join_count(d_v1, d_p1, n1, d_v2, d_p2, n2, false, h_matches);
}
adb_status adb_nested_loop_join_count(const int32_t *d_v1, const int32_t *d_p1, int64_t n1,
                                      const int32_t *d_v2, const int32_t *d_p2, int64_t n2,
                                      int64_t *h_matches) {
    // outer-major over side one (query.c:597-611) == probe-major with side one probing
    return join_count(d_v2, d_p2, n2, d_v1, d_p1, n1, true, h_matches);
}
adb_status adb_join_emit(int32_t *d_out1, int32_t *d_out2) {
    NEED_UP();
    auto &j = g.join;
    if (!j.ready) return fail(ADB_ERR_INVALID, "adb_join_emit: no preceding *_join_count");
    adb_status rc = ADB_OK;
    if (j.matches > 0) {
        if (!d_out1 || !d_out2) return fail(ADB_ERR_INVALID, "adb_join_emit: NULL output");
        int32_t *ob = j.swapped ? d_out2 : d_out1, *op = j.swapped ? d_out1 : d_out2;
        const int k_ = j.sharded
            ? adb::launch_hj_expand_sharded(j.probe.gc_by_j, j.probe.warp_base, j.probe.pg, j.n_probe, j.probe_keys, j.owners,
                                            j.probe_pos, ob, op, g.stream)
            : adb::launch_hj_expand(j.probe.gc_by_j, j.probe.warp_base, j.probe.pg, j.n_probe, j.build_pos_sorted,
                                    j.probe_pos, ob, op, g.stream);
        rc = after_launch("join_expand", k_);
    }
    if (j.sharded) {
        StageTrace tr;
        tr.lap("expand (sharded)");
        // the other contexts' expansions may still be reading this context's tables and sorted
        // build positions: they stay until the next join on this context (the host waits for
        // every context's emit before it starts one)
        j.ready = false;
        if (rc == ADB_OK) CU(cudaStreamSynchronize(g.stream));
        return rc;
    }
    join_release();
    return rc;
}

// ---- sorted index / B+-tree --------------------------------------------------------------
struct adb_index {
    const int32_t *values;
    const int32_t *positions;
    int64_t n;
    DevBuf<int32_t> tree_mem;
    adb::BTreeView tree;
    bool slice = false;
};

adb_status adb_index_create(const int32_t *d_values, const int32_t *d_positions, int64_t n,
                            int32_t with_btree, adb_index **out) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_index_create")) return s;
    if (!out || (n > 0 && (!d_values || !d_positions)))
        return fail(ADB_ERR_INVALID, "adb_index_create: NULL pointer");
    adb_index *ix = new adb_index{d_values, d_positions, n, DevBuf<int32_t>{}, adb::BTreeView{}, false};
    if (with_btree && n > 32) {
        int64_t lens[adb::kBTreeMaxDepth], total = 0;
        int depth = 0;
        for (int64_t len = (n + 31) / 32;; len = (len + 31) / 32) {
            lens[depth++] = len;
            total += len;
            if (len <= 32 || depth == adb::kBTreeMaxDepth) break;
        }
        if (adb_status s = dev_alloc(ix->tree_mem, total * sizeof(int32_t), "adb_index_create: B+-tree")) {
            delete ix;
            return s;
        }
        int32_t *p = ix->tree_mem;
        const int32_t *below = d_values;
        int64_t below_len = n;
        int launches = 0;
        for (int l = 0; l < depth; ++l) {
            ix->tree.levels[l] = p;
            ix->tree.lens[l] = lens[l];
            launches += adb::launch_btree_level(below, below_len, p, lens[l], g.sm_count, g.stream);
            below = p;
            below_len = lens[l];
            p += lens[l];
        }
        ix->tree.depth = depth;
        if (adb_status s = after_launch("btree_level", launches)) { release(ix->tree_mem); delete ix; return s; }
    }
    *out = ix;
    return ADB_OK;
}

// `ix` is one slice of an index that is range-partitioned (by index order) over several
// contexts: it answers positions[lb(low) .. lb(high)) of its slice, and the caller applies the
// reference's low == high quirk (query.c:181-188) to the whole index -- it depends on the total
// count and on the smallest key of all slices.
adb_status adb_index_set_slice(adb_index *ix, int32_t is_slice) {
    if (!ix) return fail(ADB_ERR_INVALID, "adb_index_set_slice: NULL index");
    ix->slice = is_slice != 0;
    return ADB_OK;
}

adb_status adb_index_destroy(adb_index *ix) {
    NEED_UP();
    if (!ix) return ADB_OK;
    CU(cudaStreamSynchronize(g.stream));
    release(ix->tree_mem);
    delete ix;
    return ADB_OK;
}

adb_status adb_select_index_count(const adb_index *ix, int32_t use_btree, const int32_t *lo,
                                  const int32_t *hi, int64_t *d_count, int64_t *h_count) {
    NEED_UP();
    g.idx_pending_n = -1;
    if (!ix) return fail(ADB_ERR_INVALID, "adb_select_index_count: NULL index");
    int64_t *dc = d_count ? d_count : g.scratch_count;
    const int k_ = adb::launch_index_bounds(ix->values, ix->n,
                                            use_btree && ix->tree.depth > 0 ? &ix->tree : nullptr,
                                            lo, hi, ix->slice, g.idx_bounds, dc, g.stream);
    if (adb_status s = after_launch("index_bounds", k_)) return s;
    g.idx_pending_n = ix->n;
    return finish_count(dc, h_count);
}

adb_status adb_select_index_emit(const adb_index *ix, int32_t *d_pos_out) {
    NEED_UP();
    if (!ix || g.idx_pending_n != ix->n)
        return fail(ADB_ERR_INVALID, "adb_select_index_emit: no pending adb_select_index_count on this index");
    g.idx_pending_n = -1;
    if (ix->n == 0) return ADB_OK;
    if (!d_pos_out) return fail(ADB_ERR_INVALID, "adb_select_index_emit: NULL output");
    return after_launch("index_emit", adb::launch_index_emit(ix->positions, ix->n, g.idx_bounds,
                                                             d_pos_out, g.sm_count, g.stream));
}

// ColumnIndex.positions are size_t on the host (src/include/cs165_api.h:65-68) and truncated to
// int when emitted (src/query.c:187): upload the 8-byte array as it is and narrow it here.
adb_status adb_narrow_u64_to_i32(const void *d_src_u64, int64_t n, int32_t *d_dst) {
    NEED_UP();
    if (n < 0 || (n > 0 && (!d_src_u64 || !d_dst))) return fail(ADB_ERR_INVALID, "adb_narrow_u64_to_i32: bad arguments");
    if (n == 0) return ADB_OK;
    const int k_ = adb::launch_narrow_u64(static_cast<const unsigned long long *>(d_src_u64), n, d_dst, g.sm_count, g.stream);
    return after_launch("narrow_u64", k_);
}

// ---- updates and deletes (SURVEY.md 8f rank 4; milestone5.py:123-262) --------------------------------
adb_status adb_update_rows(int32_t *d_col, int64_t n_rows, const int32_t *d_pos, int64_t n_pos, int32_t base_pos,
                           int32_t value) {
    NEED_UP();
    if (adb_status s = check_len(n_pos, "adb_update_rows")) return s;
    if (adb_status s = check_len(n_rows, "adb_update_rows")) return s;
    if (n_pos > 0 && n_rows > 0 && (!d_col || !d_pos)) return fail(ADB_ERR_INVALID, "adb_update_rows: NULL device pointer");
    return after_launch("update_rows", adb::launch_scatter_value(d_col, n_rows, d_pos, n_pos, base_pos, value,
                                                                  g.sm_count, g.stream));
}

// Plan: which of n_rows rows die (positions d_pos[0 .. n_pos), duplicates allowed) and where the
// survivors move.  *h_rows_left = rows left.  The plan lives in the engine's scratch arena until
// the next sort / join / plan; adb_delete_rows_apply compacts one column with it.
adb_status adb_delete_rows_plan(int64_t n_rows, const int32_t *d_pos, int64_t n_pos, int32_t base_pos,
                                int64_t *h_rows_left) {
    NEED_UP();
    g.del_rows = -1;
    if (adb_status s = check_len(n_rows, "adb_delete_rows_plan")) return s;
    if (adb_status s = check_len(n_pos, "adb_delete_rows_plan")) return s;
    if (!h_rows_left || (n_pos > 0 && !d_pos)) return fail(ADB_ERR_INVALID, "adb_delete_rows_plan: NULL pointer");
    if (n_rows == 0) { *h_rows_left = 0; g.del_rows = 0; return ADB_OK; }
    if (adb_status s = ensure_radix_scratch(1)) return s;
    int64_t *tot = nullptr;
    if (adb_status s = arena_take([&](Carve &c) {
            g.del_dead = c.take<uint32_t>(n_rows);
            g.del_before = c.take<uint32_t>(n_rows);
            tot = c.take<int64_t>(2);
        }, "adb_delete_rows_plan", true)) return s;
    CU(cudaMemsetAsync(g.del_dead, 0, (size_t)n_rows * 4, g.stream));
    int k_ = adb::launch_mark_rows(g.del_dead, n_rows, d_pos, n_pos, base_pos, g.sm_count, g.stream);
    k_ += adb::launch_exclusive_scan(g.del_dead, 1, g.del_before, (uint32_t)n_rows, g.sc_sums, tot, g.sm_count, g.stream);
    if (adb_status s = after_launch("delete_rows_plan", k_)) return s;
    int64_t dead = 0;
    if (adb_status s = read_back(&dead, tot, sizeof dead)) return s;
    g.del_rows = n_rows;
    *h_rows_left = n_rows - dead;
    return ADB_OK;
}
adb_status adb_delete_rows_apply(const int32_t *d_col, int32_t *d_col_out) {
    NEED_UP();
    if (g.del_rows < 0) return fail(ADB_ERR_INVALID, "adb_delete_rows_apply: no preceding adb_delete_rows_plan");
    if (g.del_rows == 0) return ADB_OK;
    if (!d_col || !d_col_out || d_col == d_col_out)
        return fail(ADB_ERR_INVALID, "adb_delete_rows_apply: needs distinct input and output columns");
    return after_launch("delete_rows_apply", adb::launch_compact_rows(d_col, g.del_dead, g.del_before, g.del_rows,
                                                                      d_col_out, g.sm_count, g.stream));
}

adb_status adb_synth_affine(int32_t *d_out, int64_t n, uint64_t first_row, uint64_t mul, uint64_t add,
                            uint64_t modulus) {
    NEED_UP();
    if (n < 0 || (n > 0 && !d_out) || modulus == 0 || modulus > ((uint64_t)1 << 31) || mul >= modulus || add >= modulus)
        return fail(ADB_ERR_INVALID, "adb_synth_affine: bad arguments");
    return after_launch("synth_affine", adb::launch_synth_affine(d_out, n, first_row, mul, add, modulus, g.sm_count, g.stream));
}

adb_status adb_iota_i32(int32_t *d_out, int64_t n, int32_t first) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_iota_i32")) return s;
    if (n > 0 && !d_out) return fail(ADB_ERR_INVALID, "adb_iota_i32: NULL output");
    return after_launch("iota", adb::launch_iota(d_out, n, first, g.sm_count, g.stream));
}

// d_dst[i] = (size_t) d_src[i]; d_src == NULL: d_dst[i] = i (identity positions of a clustered index)
adb_status adb_widen_i32_to_u64(const int32_t *d_src, int64_t n, void *d_dst_u64) {
    NEED_UP();
    if (n < 0 || (n > 0 && !d_dst_u64)) return fail(ADB_ERR_INVALID, "adb_widen_i32_to_u64: bad arguments");
    if (n == 0) return ADB_OK;
    const int k_ = adb::launch_widen_i32(d_src, n, static_cast<unsigned long long *>(d_dst_u64), g.sm_count, g.stream);
    return after_launch("widen_i32", k_);
}

// build_histogram, src/index.c:63-84: h_counts[b] = rows with (v - vmin) / bin_size == b, b < 100.
adb_status adb_histogram_i32(const int32_t *d_val, int64_t n, int32_t vmin, int32_t bin_size, uint64_t *h_counts) {
    NEED_UP();
    if (adb_status s = check_len(n, "adb_histogram_i32")) return s;
    if (bin_size <= 0 || !h_counts || (n > 0 && !d_val)) return fail(ADB_ERR_INVALID, "adb_histogram_i32: bad arguments");
    void *d = nullptr;
    if (adb_status s = adb_alloc(&d, 128 * sizeof(unsigned long long))) return s;
    const int k_ = adb::launch_histogram(d_val, n, vmin, bin_size, static_cast<unsigned long long *>(d), g.sm_count, g.stream);
    adb_status rc = after_launch("histogram", k_);
    unsigned long long host[128];
    if (rc == ADB_OK) rc = adb_download(host, d, sizeof host);
    adb_free(d);
    if (rc == ADB_OK) for (int b = 0; b < 100; ++b) h_counts[b] = host[b];
    return rc;
}

adb_status adb_synth_uniform(int32_t *d_out, int64_t n, uint64_t seed, uint64_t first_row,
                             int32_t lo, uint32_t span) {
    NEED_UP();
    if (n < 0 || (n > 0 && !d_out)) return fail(ADB_ERR_INVALID, "adb_synth_uniform: bad arguments");
    if (n == 0) return ADB_OK;
    const int k_ = adb::launch_synth_uniform(d_out, n, seed, first_row, lo, span, g.sm_count, g.stream);
    return after_launch("synth_uniform", k_);
}

}  // extern "C"
