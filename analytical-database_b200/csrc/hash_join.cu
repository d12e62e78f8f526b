// hash_join.cu -- equi-join of two (value, position) pair lists with a reproducible order.
//
// Replaces hash_join + multimap (/root/reference/src/query.c:652-696, src/multimap.c) and,
// with the sides swapped, nested_loop_join (query.c:585-650).  The reference inserts the
// build side (column_one, the larger input, parse.c:798-813) row by row into an open
// addressing multimap and then walks the probe side in row order, appending for every
// probe row all stored positions of its key in insertion order.  The output is therefore
// probe-major, build-insertion order inside a key -- and must be reproduced exactly.
//
// GPU formulation (shared-memory-partitioned hash build, probe in row order):
//   1. build side: stable LSD radix sort on h = key * 0x9E3779B1 (radix.cu), payload = the
//      build position.  The odd multiplier is a bijection on 32 bits, so equal h <=> equal
//      key: one sort both groups equal keys (insertion order kept inside a group: the sort
//      is stable) and orders the groups by partition id = top bits of h;
//   2. partition boundaries by binary search; one CTA per partition builds an open
//      addressing table {key tag -> group start / single build position, group size} in
//      shared memory and streams it to the partition's slot range in global memory;
//   3. probe rows, in their original order, look their key up in their partition's table:
//      {group start or build position, match count} per probe row, stored coalesced;
//   4. exclusive scan of the match counts in probe-row order = output offsets (radix.cu);
//   5. expand: probe row j copies its group's positions to out1[off[j] ..] and its own
//      position to out2[off[j] ..]; long groups (skewed keys) are spread over a warp.
// Partitions too large for the shared-memory table (heavy skew) build directly in their
// global slots.
#include "adb_common.cuh"

namespace adb {

constexpr int HJ_THREADS = 256;
constexpr uint32_t kHashMul = 0x9E3779B1u;

__device__ __forceinline__ uint32_t hj_pid(uint32_t key, uint32_t part_bits) {
    return part_bits ? (key * kHashMul) >> (32 - part_bits) : 0u;
}

// ---- partition boundaries -----------------------------------------------------------------
// The build side arrives sorted on the whole hash, so partition p starts at the first row
// whose id is >= p: one binary search per partition instead of one global atomic per row.
__global__ void hj_bounds_kernel(const uint32_t *__restrict__ keys, uint32_t n, uint32_t part_bits,
                                 uint32_t num_parts, uint32_t *__restrict__ off) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p > num_parts) return;
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (hj_pid(keys[mid], part_bits) < p) lo = mid + 1; else hi = mid;
    }
    off[p] = lo;                                  // off[num_parts] == n
}

// ---- table geometry ------------------------------------------------------------------------------
// Partition p gets a power-of-two slot range holding its rows at <= 80 % load (0 slots when it
// is empty); toff = exclusive scan of the capacities, toff[num_parts] = total.  Three small
// launches (r02u: one CTA walking 2^17-2^20 partitions 1024 at a time took 0.3 ms): every CTA
// scans the capacities of 1024 partitions and leaves their sum, one CTA scans the sums, every
// CTA adds its base.
constexpr uint32_t HJ_GEOM_CHUNK = 1024;

__device__ __forceinline__ unsigned long long hj_block_incl_scan_u64(unsigned long long x, unsigned long long *s_w,
                                                                      unsigned long long *block_total) {
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long incl = x;
#pragma unroll
    for (int d = 1; d < kWarp; d <<= 1) {
        const unsigned long long y = __shfl_up_sync(kFull, incl, d);
        if (lane >= (uint32_t)d) incl += y;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    unsigned long long wexcl = 0, tot = 0;
    for (uint32_t w = 0; w < blockDim.x / kWarp; ++w) {
        if (w < warp) wexcl += s_w[w];
        tot += s_w[w];
    }
    __syncthreads();
    *block_total = tot;
    return wexcl + incl;
}

__global__ void __launch_bounds__(HJ_GEOM_CHUNK)
hj_geometry_local_kernel(const uint32_t *__restrict__ off1, uint32_t num_parts,
                         unsigned long long *__restrict__ toff, unsigned long long *__restrict__ chunk_sums) {
    __shared__ unsigned long long s_w[32];
    const uint32_t p = blockIdx.x * HJ_GEOM_CHUNK + threadIdx.x;
    unsigned long long cap = 0;
    if (p < num_parts) {
        const unsigned long long sz = off1[p + 1] - off1[p];
        if (sz) {
            cap = 16;
            while (cap < sz + sz / 4 + 1) cap <<= 1;
        }
    }
    unsigned long long tot;
    const unsigned long long incl = hj_block_incl_scan_u64(cap, s_w, &tot);
    if (p < num_parts) toff[p] = incl - cap;              // exclusive inside the chunk
    if (threadIdx.x == 0) chunk_sums[blockIdx.x] = tot;
}

// in-place exclusive scan of 64-bit sums by one CTA (a few thousand, or the partitioned probe's
// 8 per 4096 rows: four per thread and step); the total goes to *total
__global__ void __launch_bounds__(1024)
hj_sums_scan_kernel(unsigned long long *__restrict__ sums, uint32_t n, unsigned long long *__restrict__ total) {
    __shared__ unsigned long long s_w[32];
    unsigned long long carry = 0;
    for (uint32_t base = 0; base < n; base += 4096) {
        const uint32_t i = base + threadIdx.x * 4;
        unsigned long long x[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) x[k] = i + k < n ? sums[i + k] : 0ull;
        unsigned long long tot;
        const unsigned long long incl = hj_block_incl_scan_u64(x[0] + x[1] + x[2] + x[3], s_w, &tot);
        unsigned long long run = carry + incl - (x[0] + x[1] + x[2] + x[3]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (i + k < n) sums[i + k] = run;
            run += x[k];
        }
        carry += tot;
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(HJ_GEOM_CHUNK)
hj_geometry_add_kernel(unsigned long long *__restrict__ toff, uint32_t num_parts,
                       const unsigned long long *__restrict__ chunk_base) {
    const uint32_t p = blockIdx.x * HJ_GEOM_CHUNK + threadIdx.x;
    if (p < num_parts) toff[p] += chunk_base[blockIdx.x];
}

// exclusive scan of n 64-bit sums in place, 1024 per CTA (the partitioned probe leaves 8 per 4096
// rows: one CTA walking 195 K of them took 207 us, r02z)
__global__ void __launch_bounds__(HJ_GEOM_CHUNK)
hj_sums_local_kernel(unsigned long long *__restrict__ sums, uint32_t n, unsigned long long *__restrict__ chunk_sums) {
    __shared__ unsigned long long s_w[32];
    const uint32_t i = blockIdx.x * HJ_GEOM_CHUNK + threadIdx.x;
    const unsigned long long x = i < n ? sums[i] : 0ull;
    unsigned long long tot;
    const unsigned long long incl = hj_block_incl_scan_u64(x, s_w, &tot);
    if (i < n) sums[i] = incl - x;
    if (threadIdx.x == 0) chunk_sums[blockIdx.x] = tot;
}

// ---- per-partition tables ---------------------------------------------------------------------
// All keys of a partition share the top `part_bits` bits of h = key * kHashMul, and the
// multiplier is a bijection, so the remaining low bits of h identify the key: a slot stores
// that 32-bit tag (+1, 0 = free), the group's size, and -- for a single-row group, the common
// case -- the build position itself, else the group's start in the sorted build arrays.
//
// r01k history.  (1) One CTA per partition built a shared-memory table and probed it with the
// partition's probe rows (probe side radix-partitioned too), scattering {start, count} to slot
// j: ncu showed 7.9 GB of DRAM traffic at 1.8 TB/s for 100 M probes -- every 8-byte store is a
// 32-byte read-modify-write at a random address (3.1 GB of fill reads, 3.2 GB of writes), and
// shrinking the table from 64 KB to 32 KB per CTA (35 % -> 80 % occupancy) changed nothing:
// the random-access rate of HBM was the limit.  (2) Now the tables are written to global
// memory (16-byte slots, one coalesced burst per partition) and the probe side is walked in
// its ORIGINAL order: one random 16-byte read per probe row, every store coalesced, no probe
// partitioning passes, no scatter.
struct HjSlot {                       // 16 bytes, read with one ld.global.v4
    uint32_t tag;                     // hj_tag(key), 0 = free
    uint32_t x, y;                    // what a probe of this key gets, see hj_matches()
    uint32_t pad;
};
static_assert(sizeof(HjSlot) == 16, "slot layout");

// A probe row's result {x, y}:  y == 0: no match;  y == 1: one build row, x = its position;
// y with bit 31 set: two build rows, x and y & 0x7FFFFFFF their positions in insertion order
// (positions are row numbers < 2^31);  else: y >= 2 rows, x = start of the group in the sorted
// build positions.  r02w: on uniform keys 26 % of the probe rows meet a group of two or more and
// each of those cost the expansion a random read of the sorted build positions (1.7 GB of DRAM
// lines per 100 M probes); pairs -- two thirds of them -- now travel inside the slot.
__device__ __forceinline__ uint32_t hj_matches(uint32_t y) { return (y >> 31) ? 2u : y; }
__device__ __forceinline__ uint2 hj_slot_value(uint32_t group_start, uint32_t size, const int32_t *__restrict__ bpos) {
    if (size == 1) return make_uint2((uint32_t)bpos[group_start], 1u);
    if (size == 2) {
        const uint32_t p0 = (uint32_t)bpos[group_start], p1 = (uint32_t)bpos[group_start + 1];
        if (!(p1 >> 31)) return make_uint2(p0, 0x80000000u | p1);
    }
    return make_uint2(group_start, size);
}

__device__ __forceinline__ uint32_t hj_tag(uint32_t key, uint32_t part_bits) {
    return (((key * kHashMul) << part_bits) >> part_bits) + 1u;       // part_bits >= 1: never wraps to 0
}
// well-mixed 32 bits of the tag; the caller masks with capacity - 1 (a power of two)
__device__ __forceinline__ uint32_t hj_mix(uint32_t tag) {
    return (uint32_t)(((unsigned long long)tag * 0x9E3779B97F4A7C15ull) >> 29);
}

// One CTA per partition.  Partitions whose slot range is at most HJ_BUILD_SLOTS (<= 1638 build rows)
// build in shared memory in ONE phase -- every build row claims / finds its key's slot and
// adds 1 to the size, the group leader (first row of the run of equal keys) adds its offset
// in the same atomic -- and stream the finished table out.  Larger partitions (heavy skew)
// run the same steps directly on their global slots.
// CTA shape (r02za: 256 threads around a 4096-slot table = 32 KB kept 7 CTAs per SM resident
// and the kernel, a string of dependent round trips per partition, ran at 2.9 TB/s): partitions
// average <= 1024 rows, i.e. <= 2048 slots, so the CTA is 128 threads around 2048 slots
// (16 KB, 14 CTAs per SM); the few larger partitions take the global-memory path.
constexpr int HJ_BUILD_THREADS = 128;
constexpr uint32_t HJ_BUILD_SLOTS = 2048;                // shared-memory table slots
__global__ void __launch_bounds__(HJ_BUILD_THREADS)
hj_table_build_kernel(const uint32_t *__restrict__ bkeys /* sorted by hash */,
                      const int32_t *__restrict__ bpos /* build positions in the same order */,
                      const uint32_t *__restrict__ off1, const unsigned long long *__restrict__ toff,
                      uint32_t part_bits, uint4 *__restrict__ table) {
    __shared__ uint32_t s_tag[HJ_BUILD_SLOTS];
    __shared__ uint32_t s_gc[HJ_BUILD_SLOTS];           // {group start within the partition : 16, size : 16}
    const uint32_t p = blockIdx.x;
    const uint32_t b0 = off1[p], b1 = off1[p + 1];
    if (b1 == b0) return;                               // capacity 0: nothing to write
    const unsigned long long t0 = toff[p], cap64 = toff[p + 1] - t0;
    if (cap64 <= HJ_BUILD_SLOTS) {
        const uint32_t cap = (uint32_t)cap64, mask = cap - 1;
        for (uint32_t s = threadIdx.x; s < cap; s += HJ_BUILD_THREADS) { s_tag[s] = 0u; s_gc[s] = 0u; }
        __syncthreads();
        for (uint32_t i = b0 + threadIdx.x; i < b1; i += HJ_BUILD_THREADS) {
            const uint32_t k = bkeys[i];
            const bool leader = i == b0 || bkeys[i - 1] != k;
            const uint32_t tag = hj_tag(k, part_bits);
            uint32_t s = hj_mix(tag) & mask;
            while (true) {
                const uint32_t cur = atomicCAS(&s_tag[s], 0u, tag);
                if (cur == 0u || cur == tag) break;
                s = (s + 1) & mask;
            }
            atomicAdd(&s_gc[s], 1u + (leader ? (i - b0) << 16 : 0u));
        }
        __syncthreads();
        uint4 *__restrict__ out = table + t0;
        for (uint32_t s = threadIdx.x; s < cap; s += HJ_BUILD_THREADS) {
            const uint32_t w = s_gc[s], c = w & 0xFFFFu, gs = b0 + (w >> 16);
            const uint2 v = c ? hj_slot_value(gs, c, bpos) : make_uint2(0u, 0u);
            out[s] = make_uint4(s_tag[s], v.x, v.y, 0u);
        }
        return;
    }
    uint32_t *T = reinterpret_cast<uint32_t *>(table + t0);          // 4 words per slot
    const unsigned long long mask = cap64 - 1;
    for (unsigned long long s = threadIdx.x; s < cap64; s += HJ_BUILD_THREADS)
        reinterpret_cast<uint4 *>(T)[s] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    for (uint32_t i = b0 + threadIdx.x; i < b1; i += HJ_BUILD_THREADS) {
        const uint32_t k = bkeys[i];
        const bool leader = i == b0 || bkeys[i - 1] != k;
        const uint32_t tag = hj_tag(k, part_bits);
        unsigned long long s = hj_mix(tag) & mask;
        while (true) {
            const uint32_t cur = atomicCAS(&T[4 * s], 0u, tag);
            if (cur == 0u || cur == tag) break;
            s = (s + 1) & mask;
        }
        atomicAdd(&T[4 * s + 2], 1u);
        if (leader) T[4 * s + 1] = i;                    // only the leader writes this word
    }
    __syncthreads();
    for (unsigned long long s = threadIdx.x; s < cap64; s += HJ_BUILD_THREADS) {
        const uint32_t c = T[4 * s + 2];
        if (c == 1u || c == 2u) {
            const uint2 v = hj_slot_value(T[4 * s + 1], c, bpos);
            T[4 * s + 1] = v.x;
            T[4 * s + 2] = v.y;
        }
    }
}

// Probe side in its original row order: one random 16-byte slot read per row (linear probing
// almost always ends inside the same 64-byte half line, which is what a miss fetches: ld_gather), results stored coalesced.
// Every warp walks ONE contiguous piece of the probe side and leaves the number of matches it
// found: the scan of those ~9 K sums is all the expansion needs to compute its output offsets
// itself (r02u: the separate offsets pass over the 100 M counts cost 0.52 ms, and reading them
// back in the expansion another 400 MB).
__device__ __forceinline__ void hj_warp_range(uint32_t rows_per_warp, uint32_t n_probe, uint32_t *j0, uint32_t *j1) {
    const unsigned long long w = blockIdx.x * (HJ_THREADS / kWarp) + (threadIdx.x >> 5);
    const unsigned long long b = w * rows_per_warp, e = b + rows_per_warp;
    *j0 = (uint32_t)(b < n_probe ? b : n_probe);
    *j1 = (uint32_t)(e < n_probe ? e : n_probe);
}
__device__ __forceinline__ void hj_warp_sum_out(unsigned long long acc, unsigned long long *__restrict__ warp_sums) {
    acc = (unsigned long long)warp_sum_i64((int64_t)acc);
    if ((threadIdx.x & 31) == 0) warp_sums[blockIdx.x * (HJ_THREADS / kWarp) + (threadIdx.x >> 5)] = acc;
}

__global__ void __launch_bounds__(HJ_THREADS)
hj_probe_kernel(const uint32_t *__restrict__ pkeys, uint32_t n_probe, uint32_t rows_per_warp,
                const unsigned long long *__restrict__ toff, uint32_t part_bits,
                const uint4 *__restrict__ table, uint2 *__restrict__ gc_by_j,
                unsigned long long *__restrict__ warp_sums) {
    uint32_t j0, j1;
    hj_warp_range(rows_per_warp, n_probe, &j0, &j1);
    unsigned long long acc = 0;
    for (uint32_t j = j0 + (threadIdx.x & 31); j < j1; j += kWarp) {
        const uint32_t k = (uint32_t)ld_stream(reinterpret_cast<const int32_t *>(pkeys) + j);
        const uint32_t p = hj_pid(k, part_bits);
        const unsigned long long t0 = toff[p], cap = toff[p + 1] - t0;
        uint2 r = make_uint2(0u, 0u);
        if (cap) {
            const uint32_t tag = hj_tag(k, part_bits);
            const unsigned long long mask = cap - 1;
            unsigned long long s = hj_mix(tag) & mask;
            while (true) {
                const uint4 sl = ld_gather(table + t0 + s);
                if (sl.x == tag) { r = make_uint2(sl.y, sl.z); break; }
                if (sl.x == 0u) break;
                s = (s + 1) & mask;
            }
        }
        gc_by_j[j] = r;
        acc += hj_matches(r.y);
    }
    hj_warp_sum_out(acc, warp_sums);
}

// ---- the probe side partitioned for L2 locality ---------------------------------------------------
// tools/random_read_probe.cu (r02v): 100 M random 16-byte reads of a 2 GB table run at 36 G/s
// whatever the miss size -- the DRAM's random-access rate -- and at 145-165 G/s when consecutive
// reads stay inside a 32 MB slice of it.  For a table well beyond L2 the probe therefore goes:
//   P1  the probe rows, cut into <= 256 WINDOWS of consecutive rows, are partitioned window by
//       window on the top 8 bits of the join hash (one segmented radix pass, payload = the row
//       number): cell (w, p) = the rows of window w whose slots lie in 1/256 of the table;
//   P2  the cells are probed partition-major -- p = 0: all windows, p = 1: all windows ... -- so
//       the slice of the table in use stays in L2; results are stored where the row sits;
//   P3  one linear pass takes {row number, result} back to probe order: consecutive entries
//       belong to one window, i.e. to a 3 MB piece of the result array, so these scattered
//       8-byte stores meet in L2 and leave it as full sectors (r01k's scatter straight from the
//       partitions was a 32-byte read-modify-write in DRAM per row: 1.8 TB/s of traffic).
// A row is a chain of dependent loads (key -> slot range of its table partition -> slot); a
// thread keeps two rows in flight and loads the keys of the next two before it resolves the
// current ones.  (r02zd: four rows per thread without the look-ahead made the kernel slower,
// 0.92 -> 1.17 ms -- cells are ~1500 rows, the last trip of a CTA then runs half empty; r02ze:
// asking L2 for the next table slice with prefetch.global.L2, one line per thread in address
// order, changed nothing: 0.92 ms, +0.3 GB of DRAM reads.)
__device__ __forceinline__ uint2 hj_lookup(uint32_t k, const unsigned long long *__restrict__ toff,
                                           uint32_t part_bits, const uint4 *__restrict__ table) {
    const uint32_t pid = hj_pid(k, part_bits);
    const unsigned long long t0 = toff[pid], cap = toff[pid + 1] - t0;
    if (!cap) return make_uint2(0u, 0u);
    const uint32_t tag = hj_tag(k, part_bits);
    const unsigned long long mask = cap - 1;
    unsigned long long s = hj_mix(tag) & mask;
    while (true) {
        const uint4 sl = ld_gather(table + t0 + s);
        if (sl.x == tag) return make_uint2(sl.y, sl.z);
        if (sl.x == 0u) return make_uint2(0u, 0u);
        s = (s + 1) & mask;
    }
}

__global__ void __launch_bounds__(HJ_THREADS)
hj_probe_cells_kernel(const uint32_t *__restrict__ pkeys_part, const uint32_t *__restrict__ cell_base,
                      uint32_t segs, uint32_t seg_rows, uint32_t n_probe,
                      const unsigned long long *__restrict__ toff, uint32_t part_bits,
                      const uint4 *__restrict__ table, uint2 *__restrict__ res_part) {
    const uint32_t p = blockIdx.x / segs, w = blockIdx.x - p * segs;
    const uint32_t b = cell_base[w * 256 + p];
    const unsigned long long seg_end = (unsigned long long)(w + 1) * seg_rows;
    const uint32_t e = p < 255 ? cell_base[w * 256 + p + 1] : (uint32_t)(seg_end < n_probe ? seg_end : n_probe);
    const int32_t *__restrict__ pk = reinterpret_cast<const int32_t *>(pkeys_part);
    uint32_t i = b + threadIdx.x;
    uint32_t k0 = i < e ? (uint32_t)ld_stream(pk + i) : 0u;
    uint32_t k1 = i + HJ_THREADS < e ? (uint32_t)ld_stream(pk + i + HJ_THREADS) : 0u;
    while (i < e) {
        const uint32_t i2 = i + 2 * HJ_THREADS;
        const uint32_t n0 = i2 < e ? (uint32_t)ld_stream(pk + i2) : 0u;
        const uint32_t n1 = i2 + HJ_THREADS < e ? (uint32_t)ld_stream(pk + i2 + HJ_THREADS) : 0u;
        const bool two = i + HJ_THREADS < e;
        // both rows' first loads are issued before either is waited for
        const uint32_t pid0 = hj_pid(k0, part_bits), pid1 = hj_pid(k1, part_bits);
        const unsigned long long a0 = toff[pid0], c0 = toff[pid0 + 1] - a0;
        const unsigned long long a1 = two ? toff[pid1] : 0ull, c1 = two ? toff[pid1 + 1] - a1 : 0ull;
        const uint32_t tag0 = hj_tag(k0, part_bits), tag1 = hj_tag(k1, part_bits);
        unsigned long long s0 = c0 ? hj_mix(tag0) & (c0 - 1) : 0ull, s1 = c1 ? hj_mix(tag1) & (c1 - 1) : 0ull;
        uint4 sl0 = make_uint4(0u, 0u, 0u, 0u), sl1 = sl0;
        if (c0) sl0 = ld_gather(table + a0 + s0);
        if (c1) sl1 = ld_gather(table + a1 + s1);
        uint2 r0 = make_uint2(0u, 0u), r1 = r0;
        while (c0) {                                        // linear probing past the first slot is rare
            if (sl0.x == tag0) { r0 = make_uint2(sl0.y, sl0.z); break; }
            if (sl0.x == 0u) break;
            s0 = (s0 + 1) & (c0 - 1);
            sl0 = ld_gather(table + a0 + s0);
        }
        while (c1) {
            if (sl1.x == tag1) { r1 = make_uint2(sl1.y, sl1.z); break; }
            if (sl1.x == 0u) break;
            s1 = (s1 + 1) & (c1 - 1);
            sl1 = ld_gather(table + a1 + s1);
        }
        res_part[i] = r0;
        if (two) res_part[i + HJ_THREADS] = r1;
        i = i2;
        k0 = n0;
        k1 = n1;
    }
}

// P3.  r02y: scattering {row number -> result} entry by entry, even though consecutive entries
// stay inside one 3 MB window of the result array, still cost a DRAM read-modify-write per
// 8-byte store (3.9 GB read + 3.0 GB written for 100 M rows, 3.6 ms): partially written sectors
// do not wait in L2 for their other rows.  So the rows are gathered instead: a CTA owns 4096
// consecutive probe rows, takes their entries out of each of the window's 256 cells (~16 per
// cell, row numbers ascending), parks the results in shared memory by row and writes them out
// as whole lines.  Its eight warps are the expansion's pieces (512 rows each): their match
// counts go to warp_sums.
constexpr uint32_t HJ_SUB = kRadixTile;               // = the radix pass' tile
constexpr uint32_t HJ_SUB_WARP = HJ_SUB / (HJ_THREADS / kWarp);

// Where do the entries of the CTA's 4096 rows sit inside cell (w, p)?  A sub-window is one
// 4096-row tile of the segmented radix pass, and that pass' histogram, scanned along the tiles
// of a window, holds exactly this: hist[w][p][t] = entries of the window's tiles before t in
// bucket p.  (r02z searched the cells' ascending row numbers instead: two binary searches per
// cell in front of every gather made the kernel 1.58 ms; r02za moved them into a kernel of
// their own, 0.18 ms; reading the histogram costs nothing.)
__global__ void __launch_bounds__(HJ_THREADS)
hj_unpartition_kernel(const uint32_t *__restrict__ row_part, const uint2 *__restrict__ res_part,
                      const uint32_t *__restrict__ cell_base, const uint32_t *__restrict__ hist,
                      uint32_t seg_tiles, uint32_t tiles, uint32_t n_probe,
                      uint2 *__restrict__ gc_by_j, unsigned long long *__restrict__ warp_sums) {
    __shared__ uint2 s_res[HJ_SUB];
    __shared__ uint32_t s_lo[256], s_n[256];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t j_lo = blockIdx.x * HJ_SUB;
    const uint32_t j_hi = min(n_probe, j_lo + HJ_SUB);
    const uint32_t w = blockIdx.x / seg_tiles, t = blockIdx.x - w * seg_tiles;
    {
        const uint32_t p = threadIdx.x;
        const uint32_t b = cell_base[w * 256 + p];
        const uint32_t *h = hist + ((size_t)w * 256 + p) * seg_tiles;
        const uint32_t tiles_here = min(seg_tiles, tiles - w * seg_tiles);
        const unsigned long long seg_end = (unsigned long long)(w + 1) * seg_tiles * HJ_SUB;
        const uint32_t e = p < 255 ? cell_base[w * 256 + p + 1] : (uint32_t)(seg_end < n_probe ? seg_end : n_probe);
        const uint32_t lo = b + h[t];
        const uint32_t hi = t + 1 < tiles_here ? b + h[t + 1] : e;
        s_lo[p] = lo;
        s_n[p] = hi - lo;
    }
    __syncthreads();
    // warp `warp` gathers cells warp*32 .. +32, eight cells' loads in flight at a time
    constexpr int U = 8;
    for (uint32_t c0 = warp * 32; c0 < warp * 32 + 32; c0 += U) {
        uint32_t row[U];
        int2 val[U];
        bool more = false;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t cnt = s_n[c0 + u];
            row[u] = 0xFFFFFFFFu;
            if (lane < cnt) {
                row[u] = row_part[s_lo[c0 + u] + lane];
                val[u] = *reinterpret_cast<const int2 *>(res_part + s_lo[c0 + u] + lane);
            }
            more |= cnt > kWarp;
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (row[u] != 0xFFFFFFFFu) s_res[row[u] - j_lo] = make_uint2((uint32_t)val[u].x, (uint32_t)val[u].y);
        if (more) {                                          // a cell with more than 32 rows in here (skew)
            for (int u = 0; u < U; ++u) {
                const uint32_t lo = s_lo[c0 + u], cnt = s_n[c0 + u];
                for (uint32_t q = kWarp + lane; q < cnt; q += kWarp) {
                    const int2 t = *reinterpret_cast<const int2 *>(res_part + lo + q);
                    s_res[row_part[lo + q] - j_lo] = make_uint2((uint32_t)t.x, (uint32_t)t.y);
                }
            }
        }
    }
    __syncthreads();
    const uint32_t rows = j_hi - j_lo;
    for (uint32_t r = threadIdx.x; r < rows; r += HJ_THREADS) gc_by_j[j_lo + r] = s_res[r];
    uint32_t acc = 0;
    for (uint32_t r = warp * HJ_SUB_WARP + lane; r < min(rows, (warp + 1) * HJ_SUB_WARP); r += kWarp)
        acc += hj_matches(s_res[r].y);
    acc = warp_sum(acc);
    if (lane == 0) warp_sums[blockIdx.x * (HJ_THREADS / kWarp) + warp] = acc;
}

// The same gather when a tile's rows sit in a FEW fat cells (the routed probe of the sharded
// join: cells = the owner GPUs, ~4096 / G entries each): the tile's entries, cell after cell,
// are dealt out to the threads sixteen apiece, all loads issued before the first store.
constexpr int HJ_FAT_CELLS = ADB_MAX_PEERS;
__global__ void __launch_bounds__(HJ_THREADS)
hj_unpartition_routed_kernel(const uint32_t *__restrict__ row_part, const uint2 *__restrict__ res_part,
                             const uint32_t *__restrict__ cell_base, const uint32_t *__restrict__ hist,
                             uint32_t tiles, uint32_t n_probe, uint32_t cells,
                             uint2 *__restrict__ gc_by_j, unsigned long long *__restrict__ warp_sums) {
    __shared__ uint2 s_res[HJ_SUB];
    __shared__ uint32_t s_lo[HJ_FAT_CELLS], s_pre[HJ_FAT_CELLS + 1];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t t = blockIdx.x;
    const uint32_t j_lo = t * HJ_SUB, j_hi = min(n_probe, j_lo + HJ_SUB);
    const uint32_t rows = j_hi - j_lo;
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (uint32_t c = 0; c < cells; ++c) {
            const uint32_t b = cell_base[c];
            const uint32_t *h = hist + (size_t)c * tiles;      // one segment: [bucket][tiles]
            const uint32_t lo = b + h[t];
            const uint32_t hi = t + 1 < tiles ? b + h[t + 1] : cell_base[c + 1];   // bucket c + 1 <= 255 exists
            s_lo[c] = lo;
            s_pre[c] = run;
            run += hi - lo;
        }
        s_pre[cells] = run;                                     // == rows
    }
    __syncthreads();
    constexpr int PER = HJ_SUB / HJ_THREADS;                    // 16
    uint32_t row[PER];
    int2 val[PER];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const uint32_t e = threadIdx.x + i * HJ_THREADS;
        row[i] = 0xFFFFFFFFu;
        if (e < rows) {
            uint32_t c = 0;
            while (c + 1 < cells && s_pre[c + 1] <= e) ++c;
            const uint32_t src = s_lo[c] + (e - s_pre[c]);
            row[i] = row_part[src];
            val[i] = *reinterpret_cast<const int2 *>(res_part + src);
        }
    }
#pragma unroll
    for (int i = 0; i < PER; ++i)
        if (row[i] != 0xFFFFFFFFu) s_res[row[i] - j_lo] = make_uint2((uint32_t)val[i].x, (uint32_t)val[i].y);
    __syncthreads();
    for (uint32_t r = threadIdx.x; r < rows; r += HJ_THREADS) gc_by_j[j_lo + r] = s_res[r];
    uint32_t acc = 0;
    for (uint32_t r = warp * HJ_SUB_WARP + lane; r < min(rows, (warp + 1) * HJ_SUB_WARP); r += kWarp)
        acc += hj_matches(s_res[r].y);
    acc = warp_sum(acc);
    if (lane == 0) warp_sums[blockIdx.x * (HJ_THREADS / kWarp) + warp] = acc;
}

// The same gather for 4-byte answers without any counting: the routed fetch over a position list
// that is not aligned with the column's shards (engine.cu: adb_route_rows ... adb_route_finish32).
__global__ void __launch_bounds__(HJ_THREADS)
rows_unpartition32_kernel(const uint32_t *__restrict__ row_part, const uint32_t *__restrict__ val_part,
                          const uint32_t *__restrict__ cell_base, const uint32_t *__restrict__ hist,
                          uint32_t tiles, uint32_t n, uint32_t cells, uint32_t *__restrict__ out) {
    __shared__ uint32_t s_val[HJ_SUB];
    __shared__ uint32_t s_lo[HJ_FAT_CELLS], s_pre[HJ_FAT_CELLS + 1];
    const uint32_t t = blockIdx.x;
    const uint32_t j_lo = t * HJ_SUB, j_hi = min(n, j_lo + HJ_SUB);
    const uint32_t rows = j_hi - j_lo;
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (uint32_t c = 0; c < cells; ++c) {
            const uint32_t b = cell_base[c];
            const uint32_t *h = hist + (size_t)c * tiles;
            const uint32_t lo = b + h[t];
            const uint32_t hi = t + 1 < tiles ? b + h[t + 1] : cell_base[c + 1];
            s_lo[c] = lo;
            s_pre[c] = run;
            run += hi - lo;
        }
        s_pre[cells] = run;
    }
    __syncthreads();
    constexpr int PER = HJ_SUB / HJ_THREADS;
    uint32_t row[PER], val[PER];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const uint32_t e = threadIdx.x + i * HJ_THREADS;
        row[i] = 0xFFFFFFFFu;
        if (e < rows && e < s_pre[cells]) {                  // (fewer entries than rows: positions outside every shard)
            uint32_t c = 0;
            while (c + 1 < cells && s_pre[c + 1] <= e) ++c;
            const uint32_t src = s_lo[c] + (e - s_pre[c]);
            row[i] = row_part[src];
            val[i] = val_part[src];
        }
    }
#pragma unroll
    for (int i = 0; i < PER; ++i)
        if (row[i] != 0xFFFFFFFFu) s_val[row[i] - j_lo] = val[i];
    __syncthreads();
    for (uint32_t r = threadIdx.x; r < rows; r += HJ_THREADS) out[j_lo + r] = s_val[r];
}

// ---- expand ---------------------------------------------------------------------------------------
// A warp expands the piece of the probe side it probed: its first output slot comes from the
// scan of the warps' match counts, the slots inside the piece from a running warp scan.  Four
// 32-row steps are loaded at once (r02u: one step at a time kept 16 KB per SM in flight and
// ran at 2.2 TB/s).
constexpr int HJ_EXP_STEPS = 4;

struct HjLocalBuild {
    const int32_t *__restrict__ bpos;
    __device__ __forceinline__ const int32_t *list(uint32_t) const { return bpos; }
};

template <class BuildLists, class OwnerOf>
__device__ __forceinline__ void hj_expand_body(const uint2 *__restrict__ gc_by_j,
                                               const unsigned long long *__restrict__ warp_base,
                                               uint32_t rows_per_warp, uint32_t n_probe,
                                               const BuildLists &lists, const OwnerOf &owner_of,
                                               const int32_t *__restrict__ probe_pos,
                                               int32_t *__restrict__ out_build, int32_t *__restrict__ out_probe) {
    const uint32_t lane = threadIdx.x & 31;
    uint32_t j0, j1;
    hj_warp_range(rows_per_warp, n_probe, &j0, &j1);
    if (j0 >= j1) return;
    uint32_t running = (uint32_t)warp_base[blockIdx.x * (HJ_THREADS / kWarp) + (threadIdx.x >> 5)];
    for (uint32_t jb = j0; jb < j1; jb += kWarp * HJ_EXP_STEPS) {
        uint2 gcv[HJ_EXP_STEPS];
        int32_t ppv[HJ_EXP_STEPS];
#pragma unroll
        for (int u = 0; u < HJ_EXP_STEPS; ++u) {
            const uint32_t j = jb + u * kWarp + lane;
            gcv[u] = make_uint2(0u, 0u);
            ppv[u] = 0;
            if (j < j1) {
                const int2 t = *reinterpret_cast<const int2 *>(gc_by_j + j);
                gcv[u] = make_uint2((uint32_t)t.x, (uint32_t)t.y);
                ppv[u] = ld_stream(probe_pos + j);
            }
        }
#pragma unroll
        for (int u = 0; u < HJ_EXP_STEPS; ++u) {
            if (jb + u * kWarp >= j1) break;                 // warp-uniform
            const bool pair = gcv[u].y >> 31;
            const uint32_t cnt = hj_matches(gcv[u].y), gs = gcv[u].x;
            const int32_t pp = ppv[u];
            const uint32_t incl = warp_incl_scan(cnt, lane);
            const uint32_t off = running + incl - cnt;
            running += __shfl_sync(kFull, incl, 31);
            if (cnt == 1) {                                  // gs already is the build position
                out_build[off] = (int32_t)gs;
                out_probe[off] = pp;
            } else if (pair) {                               // both build positions came with the slot
                out_build[off] = (int32_t)gs;
                out_build[off + 1] = (int32_t)(gcv[u].y & 0x7FFFFFFFu);
                out_probe[off] = pp;
                out_probe[off + 1] = pp;
            } else if (cnt && cnt <= 8) {
                // all of the group's (random) reads are issued before the first is waited for: nearly
                // every warp step has a lane in here (8 % of the rows on uniform keys)
                const int32_t *__restrict__ bp = lists.list(owner_of(jb + u * kWarp + lane));
                int32_t v[8];
#pragma unroll
                for (uint32_t r = 0; r < 8; ++r)
                    if (r < cnt) v[r] = ld_gather(bp + gs + r);
#pragma unroll
                for (uint32_t r = 0; r < 8; ++r)
                    if (r < cnt) {
                        out_build[off + r] = v[r];
                        out_probe[off + r] = pp;
                    }
            }
            uint32_t longs = __ballot_sync(kFull, cnt > 8);
            while (longs) {
                const int src = __ffs(longs) - 1;
                longs &= longs - 1;
                const uint32_t c = __shfl_sync(kFull, cnt, src), g = __shfl_sync(kFull, gs, src);
                const uint32_t o = __shfl_sync(kFull, off, src);
                const int32_t q = __shfl_sync(kFull, pp, src);
                const int32_t *__restrict__ bp = lists.list(owner_of(jb + u * kWarp + src));
                for (uint32_t r = lane; r < c; r += kWarp) {
                    out_build[o + r] = bp[g + r];
                    out_probe[o + r] = q;
                }
            }
        }
    }
}

struct HjNoOwner {
    __device__ __forceinline__ uint32_t operator()(uint32_t) const { return 0u; }
};

__global__ void __launch_bounds__(HJ_THREADS)
hj_expand_kernel(const uint2 *__restrict__ gc_by_j, const unsigned long long *__restrict__ warp_base,
                 uint32_t rows_per_warp, uint32_t n_probe,
                 const int32_t *__restrict__ build_pos_sorted, const int32_t *__restrict__ probe_pos,
                 int32_t *__restrict__ out_build, int32_t *__restrict__ out_probe) {
    hj_expand_body(gc_by_j, warp_base, rows_per_warp, n_probe, HjLocalBuild{build_pos_sorted}, HjNoOwner{},
                   probe_pos, out_build, out_probe);
}

// ---- the expansion when the tables live on several contexts -------------------------------------
// The owner table travels as a kernel parameter and is copied to shared memory once per CTA.
struct HjOwnersShared {
    const int32_t *bpos[kMaxPeers];
};
__device__ __forceinline__ void hj_load_owners(const JoinOwners &o, HjOwnersShared &s) {
    if (threadIdx.x == 0)
#pragma unroll
        for (int k = 0; k < kMaxPeers; ++k) s.bpos[k] = o.bpos[k];
    __syncthreads();
}
struct HjOwnerLists {
    const HjOwnersShared *so;
    __device__ __forceinline__ const int32_t *list(uint32_t w) const { return so->bpos[w]; }
};
struct HjOwnerOfRow {                                   // whose sorted build list holds row j's group
    const uint32_t *__restrict__ pkeys;
    uint32_t owners;
    __device__ __forceinline__ uint32_t operator()(uint32_t j) const { return route_owner(pkeys[j], owners); }
};

__global__ void __launch_bounds__(HJ_THREADS)
hj_expand_sharded_kernel(const uint2 *__restrict__ gc_by_j, const unsigned long long *__restrict__ warp_base,
                         uint32_t rows_per_warp, uint32_t n_probe, const uint32_t *__restrict__ pkeys,
                         const JoinOwners owners, const int32_t *__restrict__ probe_pos,
                         int32_t *__restrict__ out_build, int32_t *__restrict__ out_probe) {
    __shared__ HjOwnersShared so;
    hj_load_owners(owners, so);
    hj_expand_body(gc_by_j, warp_base, rows_per_warp, n_probe, HjOwnerLists{&so},
                   HjOwnerOfRow{pkeys, owners.count}, probe_pos, out_build, out_probe);
}

// ---- launchers --------------------------------------------------------------------------------------
int launch_hj_bounds(const uint32_t *keys, uint32_t n, uint32_t part_bits, uint32_t num_parts,
                     uint32_t *off, cudaStream_t s) {
    hj_bounds_kernel<<<(num_parts + 1 + 255) / 256, 256, 0, s>>>(keys, n, part_bits, num_parts, off);
    return 1;
}

// sums: scratch of (num_parts + 1023) / 1024 + 1 64-bit words
int launch_hj_geometry(const uint32_t *off1, uint32_t num_parts, unsigned long long *toff,
                       unsigned long long *sums, cudaStream_t s) {
    const uint32_t chunks = (num_parts + HJ_GEOM_CHUNK - 1) / HJ_GEOM_CHUNK;
    hj_geometry_local_kernel<<<chunks, HJ_GEOM_CHUNK, 0, s>>>(off1, num_parts, toff, sums);
    hj_sums_scan_kernel<<<1, 1024, 0, s>>>(sums, chunks, toff + num_parts);
    hj_geometry_add_kernel<<<chunks, HJ_GEOM_CHUNK, 0, s>>>(toff, num_parts, sums);
    return 3;
}

int launch_hj_table_build(const uint32_t *bkeys, const int32_t *bpos, const uint32_t *off1,
                          const unsigned long long *toff, uint32_t num_parts, uint32_t part_bits,
                          uint4 *table, cudaStream_t s) {
    hj_table_build_kernel<<<num_parts, HJ_BUILD_THREADS, 0, s>>>(bkeys, bpos, off1, toff, part_bits, table);
    return 1;
}

int launch_rows_unpartition32(const uint32_t *row_part, const uint32_t *val_part, const uint32_t *cell_base,
                              const uint32_t *hist, uint32_t n, uint32_t cells, uint32_t *out, cudaStream_t s) {
    if (n == 0) return 0;
    const uint32_t tiles = (n + HJ_SUB - 1) / HJ_SUB;
    rows_unpartition32_kernel<<<tiles, HJ_THREADS, 0, s>>>(row_part, val_part, cell_base, hist, tiles, n, cells, out);
    return 1;
}

HjProbeGeom hj_probe_geom(uint32_t n_probe, int sm_count) {
    HjProbeGeom pg{};
    pg.blocks = (n_probe + HJ_THREADS - 1) / HJ_THREADS;
    if (pg.blocks > (uint32_t)sm_count * 8) pg.blocks = sm_count * 8;
    if (pg.blocks == 0) pg.blocks = 1;
    pg.warps = pg.blocks * (HJ_THREADS / kWarp);
    pg.rows_per_warp = ((n_probe + pg.warps - 1) / pg.warps + kWarp - 1) / kWarp * kWarp;
    if (pg.rows_per_warp == 0) pg.rows_per_warp = kWarp;
    return pg;
}

// warp_sums: pg.warps 64-bit words; after the call warp_sums[w] = matches of the warps before w,
// *total = all matches
int launch_hj_probe(const uint32_t *pkeys, uint32_t n_probe, const HjProbeGeom &pg, const unsigned long long *toff,
                    uint32_t part_bits, const uint4 *table, uint2 *gc_by_j, unsigned long long *warp_sums,
                    unsigned long long *total, cudaStream_t s) {
    if (n_probe == 0) return 0;
    hj_probe_kernel<<<pg.blocks, HJ_THREADS, 0, s>>>(pkeys, n_probe, pg.rows_per_warp, toff, part_bits, table,
                                                     gc_by_j, warp_sums);
    hj_sums_scan_kernel<<<1, 1024, 0, s>>>(warp_sums, pg.warps, total);
    return 2;
}

// The partitioned form of launch_hj_probe (P2 + P3 above; P1 is launch_radix_pass_segmented with
// RadixPass{24, 8, 1}, payload = row number): pkeys_part / row_part = its outputs, cell_base = its
// `base`, res_part = n_probe scratch entries.
// in-place exclusive scan of the pieces' match counts; chunk_sums: warps / 1024 + 2 words
static int hj_piece_scan(unsigned long long *warp_sums, uint32_t warps, unsigned long long *chunk_sums,
                         unsigned long long *total, cudaStream_t s) {
    const uint32_t chunks = (warps + HJ_GEOM_CHUNK - 1) / HJ_GEOM_CHUNK;
    hj_sums_local_kernel<<<chunks, HJ_GEOM_CHUNK, 0, s>>>(warp_sums, warps, chunk_sums);
    hj_sums_scan_kernel<<<1, 1024, 0, s>>>(chunk_sums, chunks, total);
    hj_geometry_add_kernel<<<chunks, HJ_GEOM_CHUNK, 0, s>>>(warp_sums, warps, chunk_sums);
    return 3;
}

// cell_base / hist / seg_tiles: the segmented pass' base, scanned histogram and (effective)
// tiles per window; chunk_sums: pg.warps / 1024 + 2 64-bit words
int launch_hj_probe_partitioned(const uint32_t *pkeys_part, const uint32_t *row_part, const uint32_t *cell_base,
                                const uint32_t *hist, uint32_t segs, uint32_t seg_tiles, uint32_t n_probe,
                                const HjProbeGeom &pg, const unsigned long long *toff, uint32_t part_bits,
                                const uint4 *table, uint2 *res_part, uint2 *gc_by_j,
                                unsigned long long *warp_sums, unsigned long long *chunk_sums,
                                unsigned long long *total, cudaStream_t s) {
    if (n_probe == 0) return 0;
    hj_probe_cells_kernel<<<segs * 256, HJ_THREADS, 0, s>>>(pkeys_part, cell_base, segs, seg_tiles * HJ_SUB, n_probe,
                                                            toff, part_bits, table, res_part);
    hj_unpartition_kernel<<<pg.blocks, HJ_THREADS, 0, s>>>(row_part, res_part, cell_base, hist, seg_tiles,
                                                           (n_probe + HJ_SUB - 1) / HJ_SUB, n_probe, gc_by_j,
                                                           warp_sums);
    return 2 + hj_piece_scan(warp_sums, pg.warps, chunk_sums, total, s);
}

// The routed probe of the sharded join (engine.cu: adb_join_route_probe ... adb_join_finish_routed).
// launch_hj_probe_plain: the keys an owner received, against its own tables, results in place.
int launch_hj_probe_plain(const uint32_t *pkeys, uint32_t n_probe, const unsigned long long *toff,
                          uint32_t part_bits, const uint4 *table, uint2 *results, unsigned long long *scratch_sums,
                          int sm_count, cudaStream_t s) {
    if (n_probe == 0) return 0;
    const HjProbeGeom pg = hj_probe_geom(n_probe, sm_count);
    hj_probe_kernel<<<pg.blocks, HJ_THREADS, 0, s>>>(pkeys, n_probe, pg.rows_per_warp, toff, part_bits, table,
                                                     results, scratch_sums);
    return 1;
}
// back to row order on the rows' home: cells = the owners (one window, unsegmented pass)
int launch_hj_unpartition_routed(const uint32_t *row_part, const uint2 *res_part, const uint32_t *cell_base,
                                 const uint32_t *hist, uint32_t n_probe, uint32_t cells, const HjProbeGeom &pg,
                                 uint2 *gc_by_j, unsigned long long *warp_sums, unsigned long long *chunk_sums,
                                 unsigned long long *total, cudaStream_t s) {
    if (n_probe == 0) return 0;
    hj_unpartition_routed_kernel<<<pg.blocks, HJ_THREADS, 0, s>>>(row_part, res_part, cell_base, hist,
                                                                  (n_probe + HJ_SUB - 1) / HJ_SUB, n_probe, cells,
                                                                  gc_by_j, warp_sums);
    return 1 + hj_piece_scan(warp_sums, pg.warps, chunk_sums, total, s);
}

// the partitioned probe's geometry: one CTA per 4096 probe rows, 512 rows per warp
HjProbeGeom hj_probe_geom_partitioned(uint32_t n_probe) {
    HjProbeGeom pg{};
    pg.blocks = (n_probe + HJ_SUB - 1) / HJ_SUB;
    if (pg.blocks == 0) pg.blocks = 1;
    pg.warps = pg.blocks * (HJ_THREADS / kWarp);
    pg.rows_per_warp = HJ_SUB_WARP;
    return pg;
}

int launch_hj_expand(const uint2 *gc_by_j, const unsigned long long *warp_base, const HjProbeGeom &pg,
                     uint32_t n_probe, const int32_t *build_pos_sorted, const int32_t *probe_pos,
                     int32_t *out_build, int32_t *out_probe, cudaStream_t s) {
    if (n_probe == 0) return 0;
    hj_expand_kernel<<<pg.blocks, HJ_THREADS, 0, s>>>(gc_by_j, warp_base, pg.rows_per_warp, n_probe,
                                                      build_pos_sorted, probe_pos, out_build, out_probe);
    return 1;
}

int launch_hj_expand_sharded(const uint2 *gc_by_j, const unsigned long long *warp_base, const HjProbeGeom &pg,
                             uint32_t n_probe, const uint32_t *pkeys, const JoinOwners &owners,
                             const int32_t *probe_pos, int32_t *out_build, int32_t *out_probe, cudaStream_t s) {
    if (n_probe == 0) return 0;
    hj_expand_sharded_kernel<<<pg.blocks, HJ_THREADS, 0, s>>>(gc_by_j, warp_base, pg.rows_per_warp, n_probe, pkeys,
                                                              owners, probe_pos, out_build, out_probe);
    return 1;
}

// Load this file's kernels now (CUDA loads them lazily, on first launch): a first launch that
// has to load code while another context's kernel spin-waits for this one can stall behind it.
void preload_hash_join() {
    preload_one(reinterpret_cast<const void *>(&hj_expand_sharded_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_expand_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_geometry_local_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_geometry_add_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_sums_scan_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_probe_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_probe_cells_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_unpartition_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_unpartition_routed_kernel));
    preload_one(reinterpret_cast<const void *>(&rows_unpartition32_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_sums_local_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_table_build_kernel));
    preload_one(reinterpret_cast<const void *>(&hj_bounds_kernel));
}

}  // namespace adb
