// select_scan.cu -- range select as a dependency-free, order-preserving bitmap compaction.
//
// Replaces select_column_scan (/root/reference/src/query.c:92-137) and select_result
// (query.c:38-86).  The reference appends `position[index++] = i` in one sequential
// loop, so the output must be the ascending list of qualifying rows.
//
// r01a tried the textbook single-pass design (decoupled look-back over 16 KB tiles).  ncu
// showed DRAM traffic == algorithmic bytes but only 24 % of peak: with ~1200 resident
// tiles the look-back chain, not HBM, was the critical path (profiles/r01a_*).  This
// version has no inter-CTA dependency at all:
//
//   mask_kernel    streams the column once (16-byte loads, one contiguous row range per
//                  warp, next tile prefetched into registers), writes a 1-bit-per-row
//                  selection bitmap (N/8 bytes) and one hit count per warp-chunk;
//   expand_kernel  each CTA sums the counts of the chunks before it (<= 9472 ints, from
//                  L2), then every warp turns its slice of the bitmap into positions at
//                  its exact output offset -- sparse words store straight from registers,
//                  dense words are compacted in shared memory and written as full rows.
//
// DRAM traffic: 4N (column) + N/8 + N/8 (bitmap out and back, mostly L2-resident) + 4H
// (positions) against the algorithmic 4N + 4H of SURVEY.md section 8d.
#include "adb_common.cuh"

namespace adb {

constexpr int SEL_THREADS = 256;
constexpr int SEL_WARPS = SEL_THREADS / kWarp;           // 8
constexpr int SEL_VEC = 4;                               // int4 loads per thread per tile
constexpr int SEL_WTILE = kWarp * SEL_VEC * 4;           // 512 rows per warp-tile (16 mask words)
constexpr int EXP_WORDS = 4;                             // mask words per lane per step

// ------------------------------------------------------------------------------------------
// mask_kernel: warp `c` (global) owns rows [c*chunk_rows, (c+1)*chunk_rows).
// Bit (4*j + k) of a thread's nibble set is row  tile + 128*j + 4*lane + k, so 8 adjacent
// lanes own one 32-row mask word; the nibbles are OR-combined with three xor-shuffles.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_tile(int4 (&v)[SEL_VEC], const int32_t *__restrict__ val,
                                          uint32_t row0, uint32_t lane) {
#pragma unroll
    for (int j = 0; j < SEL_VEC; ++j)
        v[j] = ld_stream(reinterpret_cast<const int4 *>(val + row0 + j * 128 + lane * 4));
}

__device__ __forceinline__ uint32_t tile_nibbles(const int4 (&v)[SEL_VEC], const Range &rg) {
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < SEL_VEC; ++j) {
        m |= (in_range(v[j].x, rg) ? 1u : 0u) << (4 * j);
        m |= (in_range(v[j].y, rg) ? 2u : 0u) << (4 * j);
        m |= (in_range(v[j].z, rg) ? 4u : 0u) << (4 * j);
        m |= (in_range(v[j].w, rg) ? 8u : 0u) << (4 * j);
    }
    return m;
}

__device__ __forceinline__ uint32_t tile_nibbles_guarded(const int32_t *__restrict__ val,
                                                         uint32_t row0, uint32_t lane, uint32_t n,
                                                         const Range &rg) {
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < SEL_VEC; ++j)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t idx = row0 + j * 128 + lane * 4 + k;
            if (idx < n && in_range(ld_stream(val + idx), rg)) m |= 1u << (4 * j + k);
        }
    return m;
}

// nibbles -> the 16 natural-order mask words of the warp-tile, stored as one 64-byte row
__device__ __forceinline__ void store_mask_words(uint32_t nib, uint32_t lane,
                                                 uint32_t *__restrict__ words) {
    const uint32_t sh = 4 * (lane & 7);
    uint32_t w[SEL_VEC];
#pragma unroll
    for (int j = 0; j < SEL_VEC; ++j) {
        uint32_t x = ((nib >> (4 * j)) & 0xFu) << sh;
        x |= __shfl_xor_sync(kFull, x, 1);
        x |= __shfl_xor_sync(kFull, x, 2);
        x |= __shfl_xor_sync(kFull, x, 4);
        w[j] = x;                                       // rows tile + 128*j + 32*(lane>>3) ...
    }
    const uint32_t j = lane & 7;                        // lanes with (lane & 7) < 4 write
    if (j < SEL_VEC) {
        const uint32_t x = j == 0 ? w[0] : j == 1 ? w[1] : j == 2 ? w[2] : w[3];
        words[j * 4 + (lane >> 3)] = x;
    }
}

// TOTAL: the count phase of the two-phase select.  The last warp to finish (a ticket) also sums
// the per-chunk counts into *d_count and, when the host is waiting for the count, hands it over
// through the mailbox: no count kernel, no publish kernel behind the predicate pass.  A separate
// instantiation, so the chain's kernel is compiled exactly as before.
struct MaskTotal {
    int64_t *d_count;
    unsigned int *ticket;             // zeroed; re-armed by the last warp
    unsigned long long *pub;          // mapped host mailbox or nullptr
    unsigned long long pub_seq;
};
template <bool TOTAL>
__global__ void __launch_bounds__(SEL_THREADS)
mask_kernel(const int32_t *__restrict__ val, const int64_t *__restrict__ d_n, uint32_t n_host,
            Range rg, uint32_t chunk_rows, uint32_t num_chunks, uint32_t *__restrict__ mask,
            uint32_t *__restrict__ counts, bool stable_val, MaskTotal tot) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t chunk = blockIdx.x * SEL_WARPS + (threadIdx.x >> 5);
    pdl_launch_dependents();
    if (chunk >= num_chunks) return;
    // Anything but a base column may be the output of the kernel this one was launched behind
    // (select_result over a just-fetched vector): wait for it before the first load.
    if (!stable_val) pdl_wait();
    uint32_t n = n_host;
    if (d_n) {
        pdl_wait();                                          // the length comes from an earlier kernel
        const long long dn = *d_n;
        n = dn < (long long)n_host ? (uint32_t)(dn < 0 ? 0 : dn) : n_host;
    }
    const uint32_t row_begin = chunk * chunk_rows;
    const uint32_t tiles = chunk_rows / SEL_WTILE;
    uint32_t *__restrict__ words = mask + row_begin / 32;
    const bool aligned = (reinterpret_cast<uintptr_t>(val) & 15u) == 0;
    uint32_t hits = 0;

    // number of leading tiles that are completely inside [0, n) -> vector path
    uint32_t full = 0;
    if (aligned && n > row_begin) {
        const uint32_t avail = (n - row_begin) / SEL_WTILE;
        full = avail < tiles ? avail : tiles;
    }
    if (full) {
        int4 cur[SEL_VEC];
        load_tile(cur, val, row_begin, lane);
        // a base column is never written by an operator: its first tile is requested while the
        // previous kernel (which still reads the bitmap) drains
        pdl_wait();
        for (uint32_t t = 0; t < full; ++t) {
            int4 nxt[SEL_VEC];
            if (t + 1 < full) load_tile(nxt, val, row_begin + (t + 1) * SEL_WTILE, lane);
            const uint32_t nib = tile_nibbles(cur, rg);
            hits += __popc(nib);
            store_mask_words(nib, lane, words + t * (SEL_WTILE / 32));
            if (t + 1 < full) {
#pragma unroll
                for (int j = 0; j < SEL_VEC; ++j) cur[j] = nxt[j];
            }
        }
    }
    pdl_wait();
    for (uint32_t t = full; t < tiles; ++t) {            // ragged tail / unaligned view / past n
        const uint32_t row0 = row_begin + t * SEL_WTILE;
        const uint32_t nib = row0 < n ? tile_nibbles_guarded(val, row0, lane, n, rg) : 0u;
        hits += __popc(nib);
        store_mask_words(nib, lane, words + t * (SEL_WTILE / 32));
    }
    hits = warp_sum(hits);
    if (lane == 0) counts[chunk] = hits;
    if constexpr (TOTAL) {
        // one ticket per warp-chunk; whoever draws the last one totals the counts (9472 words from
        // L2) while every other warp has long retired
        uint32_t done = 0;
        if (lane == 0) {
            __threadfence();
            done = atomicAdd(tot.ticket, 1u);
        }
        done = __shfl_sync(kFull, done, 0);
        if (done != num_chunks - 1) return;
        __threadfence();
        unsigned long long acc = 0;
        for (uint32_t i = lane; i < num_chunks; i += kWarp) acc += *reinterpret_cast<volatile uint32_t *>(counts + i);
        acc = (unsigned long long)warp_sum_i64((int64_t)acc);
        if (lane == 0) {
            *tot.d_count = (int64_t)acc;
            *tot.ticket = 0;
            if (tot.pub) mbox_publish(tot.pub, tot.pub_seq, &acc, 1);
        }
    }
}

// ------------------------------------------------------------------------------------------
// expand_kernel: bitmap -> ascending positions.
// ------------------------------------------------------------------------------------------
// FETCH fuses the rest of the north-star chain into the expansion: every emitted row is
// also gathered from `fetch_col` into `val_out` and folded into {sum, min, max, count}
// (fetch_column + sum/min/max, query.c:223-243,325-437), so the position list and the value
// vector are still materialised but neither is read back from HBM by a later kernel.
struct ChainArgs {
    const int32_t *fetch_col;
    int32_t *val_out;
    adb_agg *agg_out, *agg_scratch;
    unsigned int *agg_ticket;
};
// EXCH: the chain kernel of a rank's last shard also carries the cross-rank exchange.  A
// separate parameter type and instantiation, so the single-GPU kernel is compiled exactly as
// before (r01o: growing ChainArgs itself cost the fused kernel 0.131 -> 0.180 ms).
struct ChainArgsX {
    ChainArgs c;
    PeerExchange px;
};
// Out of line on purpose: inlined, the exchange (system-scope loads, a spin loop) changed the
// register allocation and scheduling of the whole kernel (48 -> 40 registers, 0.131 -> 0.186 ms).
__device__ __noinline__ void chain_exchange(PeerExchange px, int lane) { peer_exchange_warp(px, lane); }

template <bool EXCH> struct ChainOf { using type = ChainArgs; };
template <> struct ChainOf<true> { using type = ChainArgsX; };
__device__ __forceinline__ const ChainArgs &chain_of(const ChainArgs &a) { return a; }
__device__ __forceinline__ const ChainArgs &chain_of(const ChainArgsX &a) { return a.c; }

template <bool PAIRS, bool FETCH, bool EXCH = false>
__global__ void __launch_bounds__(SEL_THREADS)
expand_kernel(const uint32_t *__restrict__ mask, const uint32_t *__restrict__ counts,
              uint32_t chunk_rows, uint32_t num_chunks, const int32_t *__restrict__ pos_in,
              int32_t base_pos, int32_t *__restrict__ out, int64_t *__restrict__ d_count,
              const typename ChainOf<EXCH>::type chx) {
    const ChainArgs &ch = chain_of(chx);
    pdl_launch_dependents();
    pdl_wait();                                              // bitmap + counts come from mask_kernel
    __shared__ uint32_t s_red[SEL_WARPS];
    __shared__ int32_t s_stage[SEL_WARPS][kWarp * 32 * EXP_WORDS / 4];   // 1024 positions per warp
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t first_chunk = blockIdx.x * SEL_WARPS;
    const int32_t *__restrict__ fcol = ch.fetch_col;
    int32_t *__restrict__ vout = ch.val_out;
    AggAcc acc{0, INT32_MAX, INT32_MIN};

    // exclusive prefix of this CTA: sum of every chunk count before it
    uint32_t accum = 0;
    for (uint32_t i = threadIdx.x; i < first_chunk; i += SEL_THREADS) accum += counts[i];
    accum = warp_sum(accum);
    if (lane == 0) s_red[warp] = accum;
    __syncthreads();
    uint32_t base = 0;
#pragma unroll
    for (int w = 0; w < SEL_WARPS; ++w) base += s_red[w];
    uint32_t my_count = 0;
    for (uint32_t w = 0; w < SEL_WARPS; ++w) {
        const uint32_t c = first_chunk + w < num_chunks ? counts[first_chunk + w] : 0u;
        if (w < warp) base += c;
        if (w == warp) my_count = c;
    }
    const uint32_t chunk = first_chunk + warp;
    if (chunk == num_chunks - 1 && lane == 0) *d_count = (int64_t)base + my_count;
    const bool active = chunk < num_chunks && my_count != 0;
    if (!FETCH && !active) return;

    if (active) {
        const uint32_t row_begin = chunk * chunk_rows;
        const uint32_t nwords = chunk_rows / 32;
        const uint32_t *__restrict__ words = mask + row_begin / 32;
        int32_t *stage = s_stage[warp];
        uint32_t out_off = base;
        // each step: lane owns EXP_WORDS consecutive words (128 rows); warp covers 4096 rows.
        // The next step's words are requested before this step's hits are written out.
        uint4 m_next = make_uint4(0, 0, 0, 0);
        if (lane * EXP_WORDS < nwords) m_next = *reinterpret_cast<const uint4 *>(words + lane * EXP_WORDS);
        for (uint32_t w0 = 0; w0 < nwords && out_off < base + my_count; w0 += kWarp * EXP_WORDS) {
            const uint32_t wi = w0 + lane * EXP_WORDS;
            const uint4 m = m_next;
            const uint32_t wn = wi + kWarp * EXP_WORDS;
            m_next = make_uint4(0, 0, 0, 0);
            if (wn < nwords) m_next = *reinterpret_cast<const uint4 *>(words + wn);   // nwords % 16 == 0
            const uint32_t c = __popc(m.x) + __popc(m.y) + __popc(m.z) + __popc(m.w);
            const uint32_t incl = warp_incl_scan(c, lane);
            const uint32_t step_total = __shfl_sync(kFull, incl, 31);
            if (step_total == 0) continue;
            uint32_t r = incl - c;                               // rank of this lane's first hit
            const uint32_t row0 = row_begin + wi * 32;
            const uint32_t mm[EXP_WORDS] = {m.x, m.y, m.z, m.w};
            if (!FETCH && step_total <= 2 * kWarp) {
                // sparse: straight from registers (stores only, nothing waits on them)
#pragma unroll
                for (int q = 0; q < EXP_WORDS; ++q) {
                    uint32_t bits = mm[q];
                    while (bits) {
                        const uint32_t b = __ffs(bits) - 1;
                        bits &= bits - 1;
                        const uint32_t row = row0 + q * 32 + b;
                        out[out_off + r] = PAIRS ? ld_gather(pos_in + row) : (int32_t)row + base_pos;
                        if (FETCH) {
                            const int32_t v = ld_gather(fcol + row);
                            vout[out_off + r] = v;
                            acc.add(v);
                        }
                        ++r;
                    }
                }
            } else {
                // dense: compact into shared memory (<= 1024 at a time), write full rows
                uint32_t done = 0;                               // positions already flushed
                while (done < step_total) {
                    const uint32_t lim = done + 1024;
                    uint32_t rr = r;
#pragma unroll
                    for (int q = 0; q < EXP_WORDS; ++q) {
                        uint32_t bits = mm[q];
                        while (bits) {
                            const uint32_t b = __ffs(bits) - 1;
                            bits &= bits - 1;
                            if (rr >= done && rr < lim) {
                                const uint32_t row = row0 + q * 32 + b;
                                stage[rr - done] = (PAIRS && !FETCH) ? ld_gather(pos_in + row) : (int32_t)row;
                            }
                            ++rr;
                        }
                    }
                    __syncwarp();
                    const uint32_t cnt = step_total - done < 1024 ? step_total - done : 1024;
                    if (FETCH) {
                        // The gathers are the long pole (one 128-byte line each).  Rows were
                        // dealt out by rank, so every lane issues up to GB independent loads
                        // before the first value is consumed: one round trip per 32*GB hits
                        // instead of one per hit of the busiest lane.
                        constexpr int GB = 4;
                        for (uint32_t i0 = 0; i0 < cnt; i0 += GB * kWarp) {
                            int32_t row[GB], v[GB], p[GB];
#pragma unroll
                            for (int k = 0; k < GB; ++k) {
                                const uint32_t i = i0 + k * kWarp + lane;
                                row[k] = i < cnt ? stage[i] : -1;
                            }
#pragma unroll
                            for (int k = 0; k < GB; ++k) {
                                v[k] = row[k] >= 0 ? ld_gather(fcol + row[k]) : 0;
                                p[k] = PAIRS ? (row[k] >= 0 ? ld_gather(pos_in + row[k]) : 0) : row[k] + base_pos;
                            }
#pragma unroll
                            for (int k = 0; k < GB; ++k)
                                if (row[k] >= 0) {
                                    const uint32_t o = out_off + done + i0 + k * kWarp + lane;
                                    out[o] = p[k];
                                    vout[o] = v[k];
                                    acc.add(v[k]);
                                }
                        }
                    } else {
                        for (uint32_t i = lane; i < cnt; i += kWarp) {
                            const int32_t row = stage[i];
                            out[out_off + done + i] = PAIRS ? row : row + base_pos;
                        }
                    }
                    __syncwarp();
                    done += cnt;
                }
            }
            out_off += step_total;
        }
    }
    if (FETCH) {
        const bool last = agg_grid_fold<SEL_THREADS>(acc, lane == 0 && chunk < num_chunks ? (int64_t)my_count : 0,
                                                     ch.agg_out, ch.agg_scratch, ch.agg_ticket);
        // multi-GPU: the CTA that completed this shard's aggregate folds the rank's partials and
        // exchanges them with every peer over NVLink (agg_out is one of px.parts: publish it first)
        if constexpr (EXCH) {
            if (last) {
                __threadfence();
                __syncthreads();
                if (warp == 0) chain_exchange(chx.px, (int)lane);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// bitmap_gather_agg_kernel: the aggregate-only resolution of a pending select (SURVEY.md 8f rank
// 3).  No ranking, no staging, no stores: order does not matter to sum / min / max, so every
// lane walks its own bitmap words and gathers + folds the fetch column at each set bit.  A
// lane's gathers are serialised by their round trip, the 9472 warps' are not.  The bitmap is
// only read: the select stays pending for whoever wants its handles written later.
// ------------------------------------------------------------------------------------------
template <bool EXCH>
__global__ void __launch_bounds__(SEL_THREADS)
bitmap_gather_agg_kernel(const uint32_t *__restrict__ mask, const uint32_t *__restrict__ counts,
                         uint32_t chunk_rows, uint32_t num_chunks, const typename ChainOf<EXCH>::type chx,
                         unsigned long long *pub, unsigned long long pub_seq) {
    const ChainArgs &ch = chain_of(chx);
    pdl_launch_dependents();
    pdl_wait();
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t chunk = blockIdx.x * SEL_WARPS + warp;
    const int32_t *__restrict__ fcol = ch.fetch_col;
    AggAcc acc{0, INT32_MAX, INT32_MIN};
    uint32_t my_count = 0;
    if (chunk < num_chunks) my_count = counts[chunk];
    if (my_count) {
        const uint32_t row_begin = chunk * chunk_rows;
        const uint32_t nwords = chunk_rows / 32;                // a multiple of 16
        const uint32_t *__restrict__ words = mask + row_begin / 32;
        // BG words per lane and step.  A lane's gathers would be serialised by their round trip
        // if it walked one word after the other; instead every round takes the next hit of EACH
        // of the lane's words, so up to BG independent gathers are in flight per lane.
        constexpr int BG = 8;
        for (uint32_t w0 = 0; w0 < nwords; w0 += BG * kWarp) {
            uint32_t m[BG];
#pragma unroll
            for (int k = 0; k < BG; ++k) {
                const uint32_t w = w0 + k * kWarp + lane;
                m[k] = w < nwords ? words[w] : 0u;
            }
            const uint32_t row0 = row_begin + (w0 + lane) * 32;
            uint32_t any = 0;
#pragma unroll
            for (int k = 0; k < BG; ++k) any |= m[k];
            while (any) {
                int32_t v[BG];
                uint32_t has = 0;
#pragma unroll
                for (int k = 0; k < BG; ++k) {
                    v[k] = 0;
                    if (m[k]) {
                        const uint32_t b = __ffs(m[k]) - 1;
                        m[k] &= m[k] - 1;
                        v[k] = ld_gather(fcol + row0 + k * (kWarp * 32) + b);
                        has |= 1u << k;
                    }
                }
                any = 0;
#pragma unroll
                for (int k = 0; k < BG; ++k) {
                    if (has & (1u << k)) acc.add(v[k]);
                    any |= m[k];
                }
            }
        }
    }
    const bool last = agg_grid_fold<SEL_THREADS>(acc, lane == 0 ? (int64_t)my_count : 0, ch.agg_out, ch.agg_scratch,
                                                 ch.agg_ticket);
    if (!last) return;
    if constexpr (EXCH) {
        __threadfence();
        __syncthreads();
        if (warp == 0) chain_exchange(chx.px, (int)lane);
        __syncwarp();
    }
    // the host is waiting for the aggregate: hand it over from here (no publish kernel)
    if (pub && threadIdx.x == 0) {
        const volatile adb_agg *r = ch.agg_out;
        if constexpr (EXCH) r = chx.px.final_out;
        unsigned long long w[3];
        w[0] = (unsigned long long)r->sum;
        w[1] = (unsigned long long)r->count;
        w[2] = (unsigned long long)(uint32_t)r->min | ((unsigned long long)(uint32_t)r->max << 32);
        mbox_publish(pub, pub_seq, w, 3);
    }
}

// ------------------------------------------------------------------------------------------
// scan_gather_agg_kernel: the whole chain in ONE pass when neither handle is materialised
// (SURVEY.md 8f rank 3: 4N + 4H bytes).  The predicate pass as in mask_kernel, but a hit row is
// gathered from the fetch column and folded on the spot: no bitmap, no position list, no value
// vector.  The next tile's loads are in flight while this tile's (rare) gathers wait.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SEL_THREADS)
scan_gather_agg_kernel(const int32_t *__restrict__ val, const int32_t *__restrict__ fcol, uint32_t n, Range rg,
                       uint32_t chunk_rows, uint32_t num_chunks, adb_agg *__restrict__ agg_out, adb_agg *agg_scratch,
                       unsigned int *agg_ticket, int64_t *__restrict__ d_count) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t chunk = blockIdx.x * SEL_WARPS + (threadIdx.x >> 5);
    pdl_launch_dependents();
    AggAcc acc{0, INT32_MAX, INT32_MIN};
    uint32_t hits = 0;
    if (chunk < num_chunks) {
        const uint32_t row_begin = chunk * chunk_rows;
        const uint32_t tiles = chunk_rows / SEL_WTILE;
        const bool aligned = (reinterpret_cast<uintptr_t>(val) & 15u) == 0;
        uint32_t full = 0;
        if (aligned && n > row_begin) {
            const uint32_t avail = (n - row_begin) / SEL_WTILE;
            full = avail < tiles ? avail : tiles;
        }
        auto fold = [&](uint32_t nib, uint32_t row0) {
            hits += __popc(nib);
            while (nib) {                                   // bit 4j+k = row row0 + 128j + 4 lane + k
                const uint32_t b = __ffs(nib) - 1;
                nib &= nib - 1;
                acc.add(ld_gather(fcol + row0 + (b >> 2) * 128 + lane * 4 + (b & 3)));
            }
        };
        if (full) {
            int4 cur[SEL_VEC];
            load_tile(cur, val, row_begin, lane);           // both columns are base columns
            pdl_wait();
            for (uint32_t t = 0; t < full; ++t) {
                int4 nxt[SEL_VEC];
                if (t + 1 < full) load_tile(nxt, val, row_begin + (t + 1) * SEL_WTILE, lane);
                fold(tile_nibbles(cur, rg), row_begin + t * SEL_WTILE);
                if (t + 1 < full) {
#pragma unroll
                    for (int j = 0; j < SEL_VEC; ++j) cur[j] = nxt[j];
                }
            }
        }
        pdl_wait();
        for (uint32_t t = full; t < tiles; ++t) {
            const uint32_t row0 = row_begin + t * SEL_WTILE;
            if (row0 < n) fold(tile_nibbles_guarded(val, row0, lane, n, rg), row0);
        }
    } else {
        pdl_wait();
    }
    const bool last = agg_grid_fold<SEL_THREADS>(acc, (int64_t)hits, agg_out, agg_scratch, agg_ticket);
    if (last && threadIdx.x == 0) {
        __threadfence();
        *d_count = reinterpret_cast<volatile adb_agg *>(agg_out)->count;
    }
}

// ------------------------------------------------------------------------------------------
// launch geometry shared by both kernels
// ------------------------------------------------------------------------------------------
struct SelectGeom {
    uint32_t chunk_rows, num_chunks, grid;
};
static SelectGeom select_geom(uint32_t n, int sm_count) {
    SelectGeom g{};
    const uint32_t wtiles = (n + SEL_WTILE - 1) / SEL_WTILE;
    const uint32_t max_chunks = (uint32_t)sm_count * 8u * SEL_WARPS;             // 8 CTAs per SM resident
    uint32_t tiles_per_chunk = (wtiles + max_chunks - 1) / max_chunks;
    if (tiles_per_chunk == 0) tiles_per_chunk = 1;
    g.chunk_rows = tiles_per_chunk * SEL_WTILE;
    g.num_chunks = (wtiles + tiles_per_chunk - 1) / tiles_per_chunk;
    g.grid = (g.num_chunks + SEL_WARPS - 1) / SEL_WARPS;
    return g;
}

size_t select_mask_words(uint32_t n, int sm_count) {
    const SelectGeom g = select_geom(n, sm_count);
    return (size_t)g.num_chunks * (g.chunk_rows / 32);
}

// One CTA folds the per-chunk hit counts into the select's total (count phase of the
// two-phase form: the caller sizes the position list before expand_kernel runs).
__global__ void __launch_bounds__(1024)
count_total_kernel(const uint32_t *__restrict__ counts, uint32_t num_chunks,
                   int64_t *__restrict__ d_count, unsigned long long *pub, unsigned long long pub_seq) {
    __shared__ unsigned long long s_w[32];
    unsigned long long acc = 0;
    for (uint32_t i = threadIdx.x; i < num_chunks; i += 1024) acc += counts[i];
    acc = (unsigned long long)warp_sum_i64((int64_t)acc);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < 32; ++w) t += s_w[w];
        *d_count = (int64_t)t;
        if (pub) mbox_publish(pub, pub_seq, &t, 1);         // the host is waiting for this count
    }
}

int launch_select_mask(const SelectArgs &a, bool with_total, cudaStream_t s) {
    if (a.n == 0) {
        cudaMemsetAsync(a.d_count, 0, sizeof(int64_t), s);
        return 0;
    }
    const SelectGeom g = select_geom(a.n, a.sm_count);
    if (with_total && a.mask_ticket) {
        launch_pdl(mask_kernel<true>, g.grid, SEL_THREADS, 0, s, a.val, a.d_n, a.n, a.range, g.chunk_rows,
                   g.num_chunks, a.mask, a.counts, a.stable_val,
                   MaskTotal{a.d_count, a.mask_ticket, a.pub, a.pub_seq});
        return 1;
    }
    launch_pdl(mask_kernel<false>, g.grid, SEL_THREADS, 0, s, a.val, a.d_n, a.n, a.range, g.chunk_rows,
               g.num_chunks, a.mask, a.counts, a.stable_val, MaskTotal{});
    if (!with_total) return 1;
    count_total_kernel<<<1, 1024, 0, s>>>(a.counts, g.num_chunks, a.d_count, a.pub, a.pub_seq);
    return 2;
}

int launch_select_expand(const SelectArgs &a, cudaStream_t s) {
    if (a.n == 0) return 0;
    const SelectGeom g = select_geom(a.n, a.sm_count);
    if (a.pos_in)
        expand_kernel<true, false><<<g.grid, SEL_THREADS, 0, s>>>(
            a.mask, a.counts, g.chunk_rows, g.num_chunks, a.pos_in, a.base_pos, a.out, a.d_count, ChainArgs{});
    else
        expand_kernel<false, false><<<g.grid, SEL_THREADS, 0, s>>>(
            a.mask, a.counts, g.chunk_rows, g.num_chunks, nullptr, a.base_pos, a.out, a.d_count, ChainArgs{});
    return 1;
}

// select_column_scan's expansion with fetch_column and the aggregates fused in.  Row r of the
// scanned column pairs with row r of fetch_col (same table, same shard).
int launch_select_expand_fetch_agg(const SelectArgs &a, cudaStream_t s) {
    const SelectGeom g = select_geom(a.n ? a.n : 1, a.sm_count);
    if (a.n == 0 || (int)g.grid > kAggMaxBlocks) return -1;          // caller falls back to 3 launches
    const ChainArgs c{a.fetch_col, a.val_out, a.agg_out, a.agg_scratch, a.agg_ticket};
    if (!a.out && !a.val_out) {                     // aggregate only: nothing is materialised
        if (a.px.world)
            launch_pdl(bitmap_gather_agg_kernel<true>, g.grid, SEL_THREADS, 0, s, a.mask, a.counts, g.chunk_rows,
                       g.num_chunks, ChainArgsX{c, a.px}, a.pub, a.pub_seq);
        else
            launch_pdl(bitmap_gather_agg_kernel<false>, g.grid, SEL_THREADS, 0, s, a.mask, a.counts, g.chunk_rows,
                       g.num_chunks, c, a.pub, a.pub_seq);
        return 1;
    }
    if (a.px.world)
        launch_pdl(expand_kernel<false, true, true>, g.grid, SEL_THREADS, 0, s, a.mask, a.counts, g.chunk_rows,
                   g.num_chunks, (const int32_t *)nullptr, a.base_pos, a.out, a.d_count, ChainArgsX{c, a.px});
    else
        launch_pdl(expand_kernel<false, true, false>, g.grid, SEL_THREADS, 0, s, a.mask, a.counts, g.chunk_rows,
                   g.num_chunks, (const int32_t *)nullptr, a.base_pos, a.out, a.d_count, c);
    return 1;
}

// the chain with neither handle materialised: one kernel, 4N + 4H bytes
int launch_scan_gather_agg(const SelectArgs &a, cudaStream_t s) {
    const SelectGeom g = select_geom(a.n ? a.n : 1, a.sm_count);
    if (a.n == 0 || (int)g.grid > kAggMaxBlocks) return -1;
    launch_pdl(scan_gather_agg_kernel, g.grid, SEL_THREADS, 0, s, a.val, a.fetch_col, a.n, a.range, g.chunk_rows,
               g.num_chunks, a.agg_out, a.agg_scratch, a.agg_ticket, a.d_count);
    return 1;
}

// Load this file's kernels now (CUDA loads them lazily, on first launch): a first launch that
// has to load code while another context's kernel spin-waits for this one can stall behind it.
void preload_select_scan() {
    { auto *fp = &bitmap_gather_agg_kernel<true>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &bitmap_gather_agg_kernel<false>; preload_one(reinterpret_cast<const void *>(fp)); }
    preload_one(reinterpret_cast<const void *>(&count_total_kernel));
    { auto *fp = &expand_kernel<true, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &expand_kernel<false, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &expand_kernel<false, true, false>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &expand_kernel<false, true, true>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &mask_kernel<true>; preload_one(reinterpret_cast<const void *>(fp)); }
    { auto *fp = &mask_kernel<false>; preload_one(reinterpret_cast<const void *>(fp)); }
    preload_one(reinterpret_cast<const void *>(&scan_gather_agg_kernel));
}

}  // namespace adb
