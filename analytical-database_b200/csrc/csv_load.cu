// csv_load.cu -- bulk load: CSV text -> int32 columns, on the device.
//
// Replaces the ingest loop of load_db (/root/reference/src/db_manager.c:304-318): after the
// header line, every fgets() line is split at ',' with strsep, the first col_count tokens go
// through atoi(), and insert_row() appends one value to every column (db_manager.c:164-199,
// one row at a time, doubling and re-mmap-ing the columns as they grow).  SURVEY.md 8f ranks
// this first among the callers of the operator path: once the operators run in well under a
// millisecond, 93 MB/s of atoi-per-cell is what a user waits for.
//
// Device formulation (the text is already in HBM; adb_upload stages it over PCIe):
//   csv_count_kernel   newlines per 4 KB block (16-byte loads, byte-compare + popc);
//   exclusive scan     of the block counts (radix.cu) -> first line number of every block;
//   csv_index_kernel   line_end[k] = offset just past the k-th '\n';
//   csv_parse_kernel   one thread per row: fields split at ',', each parsed with atoi's exact
//                      semantics -- leading isspace() skipped, optional sign, digits until
//                      the first non-digit, strtol's saturation at LONG_MAX / LONG_MIN
//                      followed by the truncating cast to int -- and stored column-wise
//                      (coalesced: consecutive threads write consecutive rows of a column).
//   rows with fewer than n_cols fields: the reference's `int row[]` lives outside the loop, so
//   a missing field keeps the value of the nearest earlier row that had it (db_manager.c:304-311;
//   a short FIRST row reads uninitialised stack in the reference and is defined as 0 here).
//   That is a forward fill, a scan with the associative "last present value" operator.  Rare
//   path, only launched when a short row was seen:
//   csv_tile_last_kernel  per tile of 256 rows and column c, the last row that has field c;
//   csv_tile_scan_kernel  exclusive max-scan of those records over the tiles, one CTA per column
//                         -> the last row BEFORE every tile that has field c, and the piece's
//                         last value of every column (what the next piece of a file inherits);
//   csv_fill_kernel       one CTA per tile: one ballot per warp and column finds the nearest
//                         earlier row inside the tile, the scan the one before it, and a row
//                         with no such row takes the caller's carry-in.
//   Work: the scan is tiles x n_cols, the fill one ballot per warp for each column that some row
//   of the tile lacks -- linear in rows plus missing cells.
// A line longer than MAX_LINE_SIZE - 1 = 1023 bytes would be split in two by fgets
// (db_manager.c:23,306); the parse flags it and the host reports ADB_ERR_INVALID.
#include "adb_common.cuh"

namespace adb {

constexpr int CSV_THREADS = 256;
constexpr uint32_t CSV_BLOCK_BYTES = CSV_THREADS * 16;      // 4 KB of text per CTA step
constexpr uint32_t kCsvMaxLine = 1023;                       // MAX_LINE_SIZE - 1

__device__ __forceinline__ uint32_t newline_mask4(uint32_t w) {
    return __vcmpeq4(w, 0x0A0A0A0Au);                        // 0xFF in every byte equal to '\n'
}

// newlines in the 16 bytes at byte offset `off` (clipped to `bytes`): one bit per byte
__device__ __forceinline__ uint32_t newline_bits16(const unsigned char *__restrict__ text, size_t off,
                                                   size_t bytes) {
    uint32_t bits = 0;
    if (off + 16 <= bytes) {
        const uint4 v = *reinterpret_cast<const uint4 *>(text + off);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t m = newline_mask4(w[i]);
            bits |= ((m & 1u) | ((m >> 7) & 2u) | ((m >> 14) & 4u) | ((m >> 21) & 8u)) << (4 * i);
        }
    } else {
        for (int i = 0; i < 16; ++i)
            if (off + i < bytes && text[off + i] == '\n') bits |= 1u << i;
    }
    return bits;
}

__global__ void __launch_bounds__(CSV_THREADS)
csv_count_kernel(const unsigned char *__restrict__ text, size_t bytes, uint32_t *__restrict__ block_counts) {
    __shared__ uint32_t s_w[CSV_THREADS / kWarp];
    const size_t off = ((size_t)blockIdx.x * CSV_THREADS + threadIdx.x) * 16;
    uint32_t c = off < bytes ? __popc(newline_bits16(text, off, bytes)) : 0u;
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < CSV_THREADS / kWarp; ++w) t += s_w[w];
        block_counts[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(CSV_THREADS)
csv_index_kernel(const unsigned char *__restrict__ text, size_t bytes, const uint32_t *__restrict__ block_base,
                 unsigned long long *__restrict__ line_end) {
    __shared__ uint32_t s_w[CSV_THREADS / kWarp];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t off = ((size_t)blockIdx.x * CSV_THREADS + threadIdx.x) * 16;
    uint32_t bits = off < bytes ? newline_bits16(text, off, bytes) : 0u;
    const uint32_t c = __popc(bits);
    const uint32_t incl = warp_incl_scan(c, lane);
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    uint32_t wexcl = 0;
    for (uint32_t w = 0; w < warp; ++w) wexcl += s_w[w];
    size_t k = (size_t)block_base[blockIdx.x] + wexcl + incl - c;
    while (bits) {
        const uint32_t b = __ffs(bits) - 1;
        bits &= bits - 1;
        line_end[k++] = (unsigned long long)(off + b + 1);
    }
}

__device__ __forceinline__ bool csv_isspace(unsigned char c) {
    return c == ' ' || (c >= '\t' && c <= '\r');             // ' ', \t \n \v \f \r: isspace() in the C locale
}

// flags[0]: some row had fewer than n_cols fields; flags[1]: some line exceeds kCsvMaxLine
__global__ void __launch_bounds__(CSV_THREADS)
csv_parse_kernel(const unsigned char *__restrict__ text, size_t bytes,
                 const unsigned long long *__restrict__ line_end, unsigned long long n_newlines,
                 uint32_t skip_lines, unsigned long long rows, uint32_t n_cols,
                 int32_t *const *__restrict__ cols, unsigned char *__restrict__ n_fields,
                 uint32_t *__restrict__ flags) {
    const unsigned long long r = (unsigned long long)blockIdx.x * CSV_THREADS + threadIdx.x;
    if (r >= rows) return;
    const unsigned long long k = r + skip_lines;
    size_t i = k ? (size_t)line_end[k - 1] : 0;
    const size_t end = k < n_newlines ? (size_t)line_end[k] : bytes;
    if (end - i > kCsvMaxLine) atomicOr(&flags[1], 1u);
    uint32_t col = 0;
    bool line_done = false;
    while (col < n_cols && !line_done) {
        // one token: [i, next ',' or end of line or NUL)
        while (i < end && csv_isspace(__ldg(text + i))) ++i;
        bool neg = false;
        if (i < end) {
            const unsigned char c = __ldg(text + i);
            if (c == '-') { neg = true; ++i; }
            else if (c == '+') ++i;
        }
        unsigned long long acc = 0;
        bool over = false;
        const unsigned long long lim = neg ? 0x8000000000000000ull : 0x7FFFFFFFFFFFFFFFull;
        while (i < end) {
            const unsigned char c = __ldg(text + i);
            if (c < '0' || c > '9') break;
            const unsigned long long d = c - '0';
            if (over || acc > (lim - d) / 10) over = true;          // strtol: saturate, keep consuming
            else acc = acc * 10 + d;
            ++i;
        }
        const unsigned long long v64 = over ? lim : acc;
        const long long sv = neg ? (long long)(0ull - v64) : (long long)v64;
        cols[col][r] = (int32_t)sv;                                  // (int) strtol(...)
        ++col;
        // skip the rest of the token; a NUL ends the C string the reference tokenises
        while (true) {
            if (i >= end) { line_done = true; break; }
            const unsigned char c = __ldg(text + i);
            ++i;
            if (c == ',') break;
            if (c == 0) { line_done = true; break; }
        }
    }
    n_fields[r] = (unsigned char)(col > 255 ? 255 : col);
    if (col < n_cols) atomicOr(&flags[0], 1u);
}

__device__ __forceinline__ int32_t warp_incl_max(int32_t x, uint32_t lane) {
#pragma unroll
    for (int d = 1; d < kWarp; d <<= 1) {
        const int32_t y = __shfl_up_sync(kFull, x, d);
        if (lane >= (uint32_t)d) x = max(x, y);
    }
    return x;
}

// tile_last[c * tiles + t] = the last row of tile t (rows [256 t, 256 t + 256)) that has field c,
// -1 if none.  A row has field c when its field count exceeds c, so this is the suffix maximum
// over k > c of "last row whose field count is k": a 256-entry table in shared memory.
__global__ void __launch_bounds__(CSV_THREADS)
csv_tile_last_kernel(unsigned long long rows, uint32_t n_cols, const unsigned char *__restrict__ n_fields,
                     uint32_t tiles, int32_t *__restrict__ tile_last) {
    __shared__ int32_t s_last[256];
    __shared__ int32_t s_w[CSV_THREADS / kWarp];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    s_last[threadIdx.x] = -1;
    __syncthreads();
    const unsigned long long r = (unsigned long long)blockIdx.x * CSV_THREADS + threadIdx.x;
    if (r < rows) atomicMax(&s_last[n_fields[r]], (int32_t)r);
    __syncthreads();
    // thread i holds entry 255 - i; its inclusive prefix max is the max over k >= 255 - i
    int32_t v = warp_incl_max(s_last[255 - threadIdx.x], lane);
    if (lane == 31) s_w[warp] = v;
    __syncthreads();
    for (uint32_t w = 0; w < warp; ++w) v = max(v, s_w[w]);
    const uint32_t c = 254u - threadIdx.x;                           // max over k >= c + 1
    if (threadIdx.x < 255 && c < n_cols) tile_last[(size_t)c * tiles + blockIdx.x] = v;
}

// One CTA per column c: tile_last[c][t] <- max(tile_last[c][0 .. t)), -1 for tile 0 (the last row
// before tile t that has field c).  summary[c] = the value of the piece's last row that has
// field c (0 if none), summary[256 + c] = whether one exists.
__global__ void __launch_bounds__(CSV_THREADS)
csv_tile_scan_kernel(uint32_t tiles, int32_t *__restrict__ tile_last, int32_t *const *__restrict__ cols,
                     int32_t *__restrict__ summary) {
    __shared__ int32_t s_w[CSV_THREADS / kWarp];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, c = blockIdx.x;
    int32_t *rec = tile_last + (size_t)c * tiles;
    int32_t run = -1;
    for (uint32_t base = 0; base < tiles; base += CSV_THREADS) {
        const uint32_t t = base + threadIdx.x;
        const int32_t incl = warp_incl_max(t < tiles ? rec[t] : -1, lane);
        int32_t excl = __shfl_up_sync(kFull, incl, 1);
        if (lane == 0) excl = -1;
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        int32_t before = run, total = run;
        for (uint32_t w = 0; w < CSV_THREADS / kWarp; ++w) {
            if (w < warp) before = max(before, s_w[w]);
            total = max(total, s_w[w]);
        }
        if (t < tiles) rec[t] = max(before, excl);
        run = total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        summary[c] = run >= 0 ? cols[c][run] : 0;
        summary[256 + c] = run >= 0;
    }
}

// No short row: every column's last value is in the last row.
__global__ void csv_last_row_kernel(unsigned long long rows, uint32_t n_cols, int32_t *const *__restrict__ cols,
                                    int32_t *__restrict__ summary) {
    const uint32_t c = threadIdx.x;
    if (c >= n_cols) return;
    summary[c] = rows ? cols[c][rows - 1] : 0;
    summary[256 + c] = rows != 0;
}

// One CTA per tile.  A missing field c of row r takes the value of the nearest earlier row that
// has it: inside r's warp (ballot), in an earlier warp of the tile (s_w), before the tile
// (tile_prev, from csv_tile_scan_kernel) or, if the piece has none, carry[c].  Rows that have
// field c are never written, so the reads race with nothing.
__global__ void __launch_bounds__(CSV_THREADS)
csv_fill_kernel(unsigned long long rows, uint32_t n_cols, int32_t *const *__restrict__ cols,
                const unsigned char *__restrict__ n_fields, uint32_t tiles, const int32_t *__restrict__ tile_prev,
                const int32_t *__restrict__ carry) {
    __shared__ int32_t s_w[2][CSV_THREADS / kWarp];
    __shared__ int32_t s_min;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long r = (unsigned long long)blockIdx.x * CSV_THREADS + threadIdx.x;
    const uint32_t have = r < rows ? n_fields[r] : 255u;
    if (threadIdx.x == 0) s_min = 255;
    __syncthreads();
    const int32_t wmin = warp_min_i32((int32_t)have);
    if (lane == 0) atomicMin(&s_min, wmin);
    __syncthreads();
    for (uint32_t c = (uint32_t)s_min; c < n_cols; ++c) {
        const uint32_t b = __ballot_sync(kFull, have > c);
        int32_t *const slot = s_w[c & 1];                            // double-buffered: one barrier per column
        if (lane == 0) slot[warp] = b ? (int32_t)(r + 31 - __clz(b)) : -1;
        __syncthreads();
        if (have <= c) {
            const uint32_t below = b & ((1u << lane) - 1);
            int32_t src;
            if (below) {
                src = (int32_t)(r - lane + 31 - __clz(below));
            } else {
                src = tile_prev[(size_t)c * tiles + blockIdx.x];
                for (uint32_t w = 0; w < warp; ++w) src = max(src, slot[w]);
            }
            cols[c][r] = src >= 0 ? cols[c][src] : carry[c];
        }
    }
}

uint32_t csv_blocks(size_t bytes) { return (uint32_t)((bytes + CSV_BLOCK_BYTES - 1) / CSV_BLOCK_BYTES); }

int launch_csv_count(const unsigned char *text, size_t bytes, uint32_t *block_counts, cudaStream_t s) {
    csv_count_kernel<<<csv_blocks(bytes), CSV_THREADS, 0, s>>>(text, bytes, block_counts);
    return 1;
}
int launch_csv_index(const unsigned char *text, size_t bytes, const uint32_t *block_base,
                     unsigned long long *line_end, cudaStream_t s) {
    csv_index_kernel<<<csv_blocks(bytes), CSV_THREADS, 0, s>>>(text, bytes, block_base, line_end);
    return 1;
}
int launch_csv_parse(const unsigned char *text, size_t bytes, const unsigned long long *line_end,
                     unsigned long long n_newlines, uint32_t skip_lines, unsigned long long rows,
                     uint32_t n_cols, int32_t *const *cols, unsigned char *n_fields, uint32_t *flags,
                     cudaStream_t s) {
    if (rows == 0) return 0;
    const unsigned int grid = (unsigned int)((rows + CSV_THREADS - 1) / CSV_THREADS);
    csv_parse_kernel<<<grid, CSV_THREADS, 0, s>>>(text, bytes, line_end, n_newlines, skip_lines, rows,
                                                  n_cols, cols, n_fields, flags);
    return 1;
}
uint32_t csv_tiles(unsigned long long rows) { return (uint32_t)((rows + CSV_THREADS - 1) / CSV_THREADS); }
int launch_csv_tile_scan(unsigned long long rows, uint32_t n_cols, int32_t *const *cols,
                         const unsigned char *n_fields, int32_t *tile_last, int32_t *summary, cudaStream_t s) {
    const uint32_t tiles = csv_tiles(rows);
    csv_tile_last_kernel<<<tiles, CSV_THREADS, 0, s>>>(rows, n_cols, n_fields, tiles, tile_last);
    csv_tile_scan_kernel<<<n_cols, CSV_THREADS, 0, s>>>(tiles, tile_last, cols, summary);
    return 2;
}
int launch_csv_last_row(unsigned long long rows, uint32_t n_cols, int32_t *const *cols, int32_t *summary,
                        cudaStream_t s) {
    csv_last_row_kernel<<<1, 256, 0, s>>>(rows, n_cols, cols, summary);
    return 1;
}
int launch_csv_fill(unsigned long long rows, uint32_t n_cols, int32_t *const *cols, const unsigned char *n_fields,
                    const int32_t *tile_prev, const int32_t *carry, cudaStream_t s) {
    if (rows == 0) return 0;
    const uint32_t tiles = csv_tiles(rows);
    csv_fill_kernel<<<tiles, CSV_THREADS, 0, s>>>(rows, n_cols, cols, n_fields, tiles, tile_prev, carry);
    return 1;
}

// Load this file's kernels now (CUDA loads them lazily, on first launch): a first launch that
// has to load code while another context's kernel spin-waits for this one can stall behind it.
void preload_csv_load() {
    preload_one(reinterpret_cast<const void *>(&csv_count_kernel));
    preload_one(reinterpret_cast<const void *>(&csv_fill_kernel));
    preload_one(reinterpret_cast<const void *>(&csv_index_kernel));
    preload_one(reinterpret_cast<const void *>(&csv_last_row_kernel));
    preload_one(reinterpret_cast<const void *>(&csv_parse_kernel));
    preload_one(reinterpret_cast<const void *>(&csv_tile_last_kernel));
    preload_one(reinterpret_cast<const void *>(&csv_tile_scan_kernel));
}

}  // namespace adb
