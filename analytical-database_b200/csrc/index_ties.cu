// index_ties.cu -- the reference's quicksort (src/index.c:25-46, Lomuto: pivot = last element,
// strict <) reproduced on the GPU, equal keys in exactly the order its swaps leave them.
//
// The recursion runs level by level: the two sides of a partition are disjoint, so every live
// segment of one level is handled at once.  K = the radix-sorted keys (adb_index_sort's values,
// which are also this sort's values); a segment [lo, hi] always holds the keys K[lo..hi].
//
//   * pairwise-distinct segment (no K[k] == K[k-1] for k in (lo, hi], one difference of `dex`,
//     the exclusive prefix count of such k): every row goes to lower_bound(K[lo..hi], key);
//   * non-decreasing segment: each run of equal keys is rotated right by one (the recursion
//     would take the last element first, then the rest in order, one level per row);
//   * segment of <= kTiesSmall rows: one CTA finishes its whole sub-sort in shared memory;
//   * any other segment is partitioned in closed form.  Of the m = hi - lo scanned rows, the
//     L rows (< pivot) keep their order at lo.., the pivot lands at lo + nL, and the rows
//     >= pivot behave as a FIFO queue: from the first push on (`lead` = L rows before it)
//     every scanned row is an event k = (j - lo) - lead, a push holding its own row, an L row
//     a rotation holding S[Lb - lead] (Lb = L rows before it); if anything was pushed, a closing
//     rotation k = m - lead holds S[nL - lead].  With R rotations, S[R + s] lands at
//     lo + nL + 1 + s.  A rotation points at a strictly smaller event index, so each output
//     slot resolves its row by chasing those pointers (tests/test_index_ties_model.py states
//     the same in Python against the quicksort).
//
// Every row's final position is written to the output once: a pivot, a one-row side, or a row
// of a finished segment.  Live sides go to the other (values, positions) buffer for the next
// level; the host reads back one 16-byte counter per level (big segments | their tiles, small
// segments).
#include "adb_common.cuh"

namespace adb {

constexpr int QT_THREADS = 512;
constexpr int QT_WARPS = QT_THREADS / kWarp;
constexpr uint32_t QT_TILE = kTiesTile;
constexpr int QT_RPT = (int)(QT_TILE / QT_THREADS);            // rows per thread
constexpr uint32_t QT_ROT = 0x80000000u;                         // event = rotation, low bits: index
constexpr uint32_t QT_NONE = 0xFFFFFFFFu;
constexpr int QT_SMALL_THREADS = 512;
constexpr int QT_STACK = 32;                                      // >= log2(kTiesSmall) + 1
static_assert(QT_TILE % QT_THREADS == 0, "tile = threads x rows per thread");

enum : uint32_t { QT_PARTITION = 0, QT_DISTINCT = 1, QT_NONDEC = 2 };

// first index in a[0 .. len) whose value is >= x
__device__ __forceinline__ uint32_t qt_lower_bound(const int32_t *a, uint32_t len, int32_t x) {
    uint32_t lo = 0, hi = len;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// block-wide exclusive scan of one count per thread; returns the exclusive prefix, *total the sum
template <int THREADS>
__device__ __forceinline__ uint32_t qt_block_scan(uint32_t x, uint32_t *s_warp, uint32_t *total) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t incl = warp_incl_scan(x, lane);
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < THREADS / kWarp; ++w) {
        const uint32_t t = s_warp[w];
        before += (uint32_t)w < warp ? t : 0u;
        all += t;
    }
    *total = all;
    __syncthreads();                                   // s_warp is reused by the next scan
    return before + incl - x;
}

// ---- set-up ---------------------------------------------------------------------------------
// count (and with flags, mark) the k with K[k + 1] == K[k]; flags[n - 1] = 0
template <bool FLAGS>
__global__ void __launch_bounds__(256)
qt_dups_kernel(const int32_t *__restrict__ keys, uint32_t n, uint32_t *__restrict__ flags,
               unsigned long long *__restrict__ count) {
    uint32_t c = 0;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const uint32_t d = k + 1 < n && keys[k + 1] == keys[k];
        if (FLAGS) flags[k] = d;
        c += d;
    }
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, (unsigned long long)c);
}

// (values, positions) = (column, identity); the whole column is the first segment
__global__ void __launch_bounds__(256)
qt_init_kernel(const int32_t *__restrict__ col, uint32_t n, int32_t *__restrict__ cv, uint32_t *__restrict__ cp,
               TiesBig *__restrict__ big, uint2 *__restrict__ small) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        cv[i] = col[i];
        cp[i] = i;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (n > kTiesSmall) big[0] = TiesBig{0, n - 1, 0, 0};
        else small[0] = make_uint2(0, n - 1);
    }
}

// ---- one level of big segments ----------------------------------------------------------------
// the segment a tile belongs to: tiles were handed out in segment order (tbase ascending)
__device__ __forceinline__ uint32_t qt_tile_segment(const TiesBig *__restrict__ big, uint32_t nbig, uint32_t tile) {
    uint32_t lo = 0, hi = nbig;                        // last s with big[s].tbase <= tile
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (big[mid].tbase <= tile) lo = mid; else hi = mid;
    }
    return lo;
}

// per tile: L rows, descents (v[i] > v[i + 1]) and the segment-relative row of the first push
__global__ void __launch_bounds__(QT_THREADS)
qt_count_kernel(TiesLevel a) {
    __shared__ uint32_t s_l[QT_WARPS], s_d[QT_WARPS], s_f[QT_WARPS];
    const TiesBig sg = a.big[qt_tile_segment(a.big, a.nbig, blockIdx.x)];
    const uint32_t r0 = sg.lo + (blockIdx.x - sg.tbase) * QT_TILE;
    const uint32_t r1 = min(r0 + QT_TILE, sg.hi);      // scanned rows stop before the pivot
    const int32_t x = a.cv[sg.hi];
    uint32_t nl = 0, nd = 0, first = QT_NONE;
    for (uint32_t j = r0 + threadIdx.x; j < r1; j += QT_THREADS) {
        const int32_t v = a.cv[j];
        if (v < x) ++nl;
        else first = min(first, j - sg.lo);
        nd += v > a.cv[j + 1];
    }
    nl = warp_sum(nl);
    nd = warp_sum(nd);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) first = min(first, __shfl_xor_sync(kFull, first, d));
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_l[warp] = nl; s_d[warp] = nd; s_f[warp] = first; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < QT_WARPS; ++w) { nl += s_l[w]; nd += s_d[w]; first = min(first, s_f[w]); }
        a.tile_cnt[blockIdx.x] = make_uint4(nl, nd, first, 0);
    }
}

// one warp per segment: prefix of the tiles' L counts, the segment's mode, its live sides
// handed out as next-level segments
__global__ void __launch_bounds__(256)
qt_segment_kernel(TiesLevel a) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t s = blockIdx.x * (256 / kWarp) + (threadIdx.x >> 5);
    if (s >= a.nbig) return;
    const TiesBig sg = a.big[s];
    const uint32_t m = sg.hi - sg.lo;
    const uint32_t tiles = (m + QT_TILE) / QT_TILE;    // ceil((m + 1) / tile)
    uint32_t carry = 0, nd = 0, first = QT_NONE;
    for (uint32_t t0 = 0; t0 < tiles; t0 += kWarp) {
        const uint32_t t = t0 + lane;
        const uint4 c = t < tiles ? a.tile_cnt[sg.tbase + t] : make_uint4(0, 0, QT_NONE, 0);
        const uint32_t incl = warp_incl_scan(c.x, lane);
        if (t < tiles) a.tile_pre[sg.tbase + t] = carry + incl - c.x;
        carry += __shfl_sync(kFull, incl, 31);
        nd += c.y;
        first = min(first, c.z);
    }
    nd = warp_sum(nd);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) first = min(first, __shfl_xor_sync(kFull, first, d));
    if (lane != 0) return;
    const uint32_t nl = carry, q = m - nl;
    uint32_t mode = QT_PARTITION;
    if (a.dex[sg.hi] == a.dex[sg.lo]) mode = QT_DISTINCT;
    else if (nd == 0) mode = QT_NONDEC;
    const uint32_t lead = q ? first : m;
    a.info[s] = make_uint4(mode, nl, lead, q ? nl - lead + 1 : 0);
    if (mode != QT_PARTITION) return;
    const uint2 side[2] = {make_uint2(sg.lo, sg.lo + nl - 1), make_uint2(sg.lo + nl + 1, sg.hi)};
    const uint32_t len[2] = {nl, q};
    for (int k = 0; k < 2; ++k) {
        if (len[k] < 2) continue;
        if (len[k] <= kTiesSmall) {
            a.small_next[atomicAdd(&a.ctr_next->small, 1u)] = side[k];
        } else {
            const uint32_t t = (len[k] + QT_TILE - 1) / QT_TILE;
            // one atomic for slot and tiles: slots in tile order, which qt_tile_segment needs
            const unsigned long long old = atomicAdd(&a.ctr_next->big, (1ull << 32) | t);
            a.big_next[old >> 32] = TiesBig{side[k].x, side[k].y, (uint32_t)old, 0};
        }
    }
}

// partition, first half: L rows to their places, the pivot, every event into ev[lo + k]
__global__ void __launch_bounds__(QT_THREADS)
qt_events_kernel(TiesLevel a) {
    __shared__ uint32_t s_warp[QT_WARPS];
    const uint32_t s = qt_tile_segment(a.big, a.nbig, blockIdx.x);
    const uint4 inf = a.info[s];
    if (inf.x != QT_PARTITION) return;
    const TiesBig sg = a.big[s];
    const uint32_t nl = inf.y, lead = inf.z, m = sg.hi - sg.lo, q = m - nl;
    const uint32_t r0 = sg.lo + (blockIdx.x - sg.tbase) * QT_TILE;
    const uint32_t r1 = min(r0 + QT_TILE, sg.hi);
    const int32_t x = a.cv[sg.hi];
    const uint32_t j0 = r0 + threadIdx.x * QT_RPT;     // this thread's rows, in row order
    int32_t v[QT_RPT];
    uint32_t mine = 0;
#pragma unroll
    for (int i = 0; i < QT_RPT; ++i) {
        v[i] = j0 + i < r1 ? a.cv[j0 + i] : INT32_MAX;
        mine += j0 + i < r1 && v[i] < x;
    }
    uint32_t tot;
    uint32_t lb = a.tile_pre[blockIdx.x] + qt_block_scan<QT_THREADS>(mine, s_warp, &tot);
#pragma unroll
    for (int i = 0; i < QT_RPT; ++i) {
        const uint32_t j = j0 + i;
        if (j >= r1) break;
        const uint32_t rel = j - sg.lo, p = a.cp[j];
        if (v[i] < x) {
            const uint32_t dst = sg.lo + lb;
            if (nl == 1) a.pos_out[dst] = p;
            else { a.nv[dst] = v[i]; a.np[dst] = p; }
            if (rel > lead) a.ev[sg.lo + rel - lead] = QT_ROT | (lb - lead);
            ++lb;
        } else {
            a.ev[sg.lo + rel - lead] = j;
        }
    }
    if (r1 == sg.hi && threadIdx.x == 0) {             // the tile that holds the pivot
        a.pos_out[sg.lo + nl] = a.cp[sg.hi];
        if (q) a.ev[sg.lo + m - lead] = QT_ROT | (nl - lead);
    }
}

// partition, second half: the rows >= pivot from the queue; the two closed-form finishes
__global__ void __launch_bounds__(QT_THREADS)
qt_gather_kernel(TiesLevel a) {
    const uint32_t s = qt_tile_segment(a.big, a.nbig, blockIdx.x);
    const uint4 inf = a.info[s];
    const TiesBig sg = a.big[s];
    const uint32_t r0 = sg.lo + (blockIdx.x - sg.tbase) * QT_TILE;
    const uint32_t r1 = min(r0 + QT_TILE, sg.hi + 1);
    if (inf.x == QT_PARTITION) {
        const uint32_t nl = inf.y, rot = inf.w, q = sg.hi - sg.lo - nl;
        const uint32_t g0 = sg.lo + nl + 1;
        for (uint32_t d = max(r0, g0) + threadIdx.x; d < r1; d += QT_THREADS) {
            uint32_t e = a.ev[sg.lo + rot + (d - g0)];
            while (e & QT_ROT) e = a.ev[sg.lo + (e & ~QT_ROT)];
            if (q == 1) a.pos_out[d] = a.cp[e];
            else { a.nv[d] = a.cv[e]; a.np[d] = a.cp[e]; }
        }
    } else if (inf.x == QT_DISTINCT) {
        const int32_t *k = a.keys + sg.lo;
        const uint32_t len = sg.hi - sg.lo + 1;
        for (uint32_t i = r0 + threadIdx.x; i < r1; i += QT_THREADS)
            a.pos_out[sg.lo + qt_lower_bound(k, len, a.cv[i])] = a.cp[i];
    } else {                                           // non-decreasing: cv[lo..hi] == K[lo..hi]
        for (uint32_t i = r0 + threadIdx.x; i < r1; i += QT_THREADS) {
            const int32_t v = a.cv[i];
            const bool last = i == sg.hi || a.cv[i + 1] != v;
            const uint32_t dst = last ? sg.lo + qt_lower_bound(a.cv + sg.lo, i - sg.lo, v) : i + 1;
            a.pos_out[dst] = a.cp[i];
        }
    }
}

// ---- small segments: one CTA sorts the whole segment in shared memory ------------------------
struct QtSmall {
    int32_t v[kTiesSmall], tv[kTiesSmall];
    uint32_t p[kTiesSmall], tp[kTiesSmall], ev[kTiesSmall];
    uint2 stack[QT_STACK];
    uint32_t warp[QT_SMALL_THREADS / kWarp];
    uint32_t first;
    int32_t a, b, top;
};

__global__ void __launch_bounds__(QT_SMALL_THREADS)
qt_small_kernel(TiesLevel a) {
    extern __shared__ __align__(16) unsigned char qt_smem[];
    QtSmall &sh = *reinterpret_cast<QtSmall *>(qt_smem);
    const uint2 seg = a.small[blockIdx.x];
    const uint32_t base = seg.x;                        // rows below are relative to it
    for (uint32_t i = threadIdx.x; i <= seg.y - base; i += QT_SMALL_THREADS) {
        sh.v[i] = a.cv[base + i];
        sh.p[i] = a.cp[base + i];
    }
    if (threadIdx.x == 0) { sh.a = 0; sh.b = (int32_t)(seg.y - base); sh.top = 0; }
    __syncthreads();
    for (;;) {
        const int32_t lo = sh.a, hi = sh.b;
        if (lo > hi) break;                             // stack empty
        const uint32_t len = (uint32_t)(hi - lo + 1), m = len - 1;
        uint32_t next = 0;                              // 0: pop; else the sides to go on with
        uint32_t nl = 0;
        if (a.dex[base + hi] == a.dex[base + lo]) {
            const int32_t *k = a.keys + base + lo;
            for (uint32_t i = threadIdx.x; i < len; i += QT_SMALL_THREADS)
                a.pos_out[base + lo + qt_lower_bound(k, len, sh.v[lo + i])] = sh.p[lo + i];
        } else {
            bool desc = false;
            for (uint32_t i = threadIdx.x; i < m; i += QT_SMALL_THREADS) desc |= sh.v[lo + i] > sh.v[lo + i + 1];
            if (!__syncthreads_or(desc)) {
                for (uint32_t i = threadIdx.x; i < len; i += QT_SMALL_THREADS) {
                    const int32_t v = sh.v[lo + i];
                    const bool last = i == m || sh.v[lo + i + 1] != v;
                    const uint32_t dst = last ? qt_lower_bound(sh.v + lo, i, v) : i + 1;
                    a.pos_out[base + lo + dst] = sh.p[lo + i];
                }
            } else {
                // partition [lo, hi]: each thread scans a contiguous run of rows
                const int32_t x = sh.v[hi];
                const uint32_t per = (m + QT_SMALL_THREADS - 1) / QT_SMALL_THREADS;
                const uint32_t j0 = min(m, threadIdx.x * per), j1 = min(m, j0 + per);
                if (threadIdx.x == 0) sh.first = QT_NONE;
                uint32_t mine = 0;
                for (uint32_t r = j0; r < j1; ++r) mine += sh.v[lo + r] < x;
                uint32_t lb = qt_block_scan<QT_SMALL_THREADS>(mine, sh.warp, &nl);   // (syncs)
                if (j1 - j0 > mine) {
                    uint32_t r = j0;
                    while (sh.v[lo + r] < x) ++r;
                    atomicMin(&sh.first, r);
                }
                __syncthreads();
                const uint32_t q = m - nl, lead = q ? sh.first : m;
                for (uint32_t r = j0; r < j1; ++r) {
                    const int32_t v = sh.v[lo + r];
                    if (v < x) {
                        sh.tv[lo + lb] = v;
                        sh.tp[lo + lb] = sh.p[lo + r];
                        if (r > lead) sh.ev[lo + r - lead] = QT_ROT | (lb - lead);
                        ++lb;
                    } else {
                        sh.ev[lo + r - lead] = lo + r;
                    }
                }
                if (threadIdx.x == 0) {
                    sh.tv[lo + nl] = x;
                    sh.tp[lo + nl] = sh.p[hi];
                    if (q) sh.ev[lo + m - lead] = QT_ROT | (nl - lead);
                }
                __syncthreads();
                const uint32_t rot = q ? nl - lead + 1 : 0;
                for (uint32_t s = threadIdx.x; s < q; s += QT_SMALL_THREADS) {
                    uint32_t e = sh.ev[lo + rot + s];
                    while (e & QT_ROT) e = sh.ev[lo + (e & ~QT_ROT)];
                    sh.tv[lo + nl + 1 + s] = sh.v[e];
                    sh.tp[lo + nl + 1 + s] = sh.p[e];
                }
                __syncthreads();
                for (uint32_t i = threadIdx.x; i < len; i += QT_SMALL_THREADS) {
                    sh.v[lo + i] = sh.tv[lo + i];
                    sh.p[lo + i] = sh.tp[lo + i];
                }
                if (threadIdx.x == 0) {
                    a.pos_out[base + lo + nl] = sh.tp[lo + nl];
                    if (nl == 1) a.pos_out[base + lo] = sh.tp[lo];
                    if (q == 1) a.pos_out[base + hi] = sh.tp[hi];
                }
                next = (nl >= 2 ? 1u : 0u) | (q >= 2 ? 2u : 0u);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            // the smaller side next, the larger one deferred: the stack stays <= log2(len) deep
            const int32_t l0 = lo, l1 = lo + (int32_t)nl - 1, g0 = lo + (int32_t)nl + 1, g1 = hi;
            if (next == 3) {
                const bool left_small = l1 - l0 <= g1 - g0;
                sh.stack[sh.top++] = left_small ? make_uint2(g0, g1) : make_uint2(l0, l1);
                sh.a = left_small ? l0 : g0;
                sh.b = left_small ? l1 : g1;
            } else if (next == 1) {
                sh.a = l0; sh.b = l1;
            } else if (next == 2) {
                sh.a = g0; sh.b = g1;
            } else if (sh.top > 0) {
                const uint2 t = sh.stack[--sh.top];
                sh.a = (int32_t)t.x; sh.b = (int32_t)t.y;
            } else {
                sh.a = 1; sh.b = 0;
            }
        }
        __syncthreads();
    }
}

// ---- launches -------------------------------------------------------------------------------
static void qt_set_attributes() {
    static bool done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (done[dev & 63]) return;
    cudaFuncSetAttribute(qt_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(QtSmall));
    done[dev & 63] = true;
}

int launch_ties_dups(const int32_t *keys, uint32_t n, uint32_t *flags, unsigned long long *count, int sm_count,
                     cudaStream_t s) {
    const uint32_t grid = min((n + 255) / 256, (uint32_t)sm_count * 8);
    cudaMemsetAsync(count, 0, sizeof *count, s);
    if (flags) qt_dups_kernel<true><<<grid, 256, 0, s>>>(keys, n, flags, count);
    else qt_dups_kernel<false><<<grid, 256, 0, s>>>(keys, n, nullptr, count);
    return 1;
}

int launch_ties_init(const int32_t *col, uint32_t n, int32_t *cv, uint32_t *cp, TiesBig *big, uint2 *small,
                     int sm_count, cudaStream_t s) {
    qt_init_kernel<<<min((n + 255) / 256, (uint32_t)sm_count * 8), 256, 0, s>>>(col, n, cv, cp, big, small);
    return 1;
}

int launch_ties_level(const TiesLevel &a, cudaStream_t s) {
    int k = 0;
    if (a.nsmall) {
        qt_set_attributes();
        qt_small_kernel<<<a.nsmall, QT_SMALL_THREADS, sizeof(QtSmall), s>>>(a);
        ++k;
    }
    if (a.nbig) {
        qt_count_kernel<<<a.ntiles, QT_THREADS, 0, s>>>(a);
        qt_segment_kernel<<<(a.nbig + 7) / 8, 256, 0, s>>>(a);
        qt_events_kernel<<<a.ntiles, QT_THREADS, 0, s>>>(a);
        qt_gather_kernel<<<a.ntiles, QT_THREADS, 0, s>>>(a);
        k += 4;
    }
    return k;
}

void preload_index_ties() {
    { auto *fp = &qt_dups_kernel<true>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &qt_dups_kernel<false>; preload_one(reinterpret_cast<const void *>(fp)); }
    preload_one(reinterpret_cast<const void *>(&qt_init_kernel));
    preload_one(reinterpret_cast<const void *>(&qt_count_kernel));
    preload_one(reinterpret_cast<const void *>(&qt_segment_kernel));
    preload_one(reinterpret_cast<const void *>(&qt_events_kernel));
    preload_one(reinterpret_cast<const void *>(&qt_gather_kernel));
    preload_one(reinterpret_cast<const void *>(&qt_small_kernel));
    qt_set_attributes();
}

}  // namespace adb
