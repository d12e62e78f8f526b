/*
 * adb_engine.h -- C-ABI of the B200 operator engine (libadb_b200.so).
 *
 * This is the drop-in boundary for the reference column store's operator path: the
 * functions a C host (the reference's server.c dispatcher through the query.h shim in
 * analytical-database_b200/host/query_shim.c, or any FFI) binds instead of the loops in
 * /root/reference/src/query.c, multimap.c and the lookup half of index.c.  Plain
 * pointers and sizes only.  Each entry point cites the reference interface it
 * replaces (path:line under /root/reference).
 *
 * Conventions
 *  - Every function returns ADB_OK (0) or a negative adb_status; adb_last_error()
 *    returns the message of the calling thread's last failure.  There is no CPU
 *    fallback: without a CUDA device adb_init() fails and every operator returns
 *    ADB_ERR_NOT_INITIALISED.
 *  - Pointers named d_* are device (HBM) addresses obtained from adb_alloc(); all
 *    others are host addresses.  Columns, position lists and value vectors are int32
 *    (reference: `int`, src/include/cs165_api.h:77-92,179-183); row counts and hit
 *    counts are int64 but must stay below 2^31 per column shard because positions
 *    are int32 (src/query.c:94-95).
 *  - An absent range bound is a NULL `lo` / `hi` pointer, exactly as the dispatcher
 *    passes it (src/server.c:144-154).  The predicate is lo <= v < hi
 *    (src/query.c:101).
 *  - Operators are enqueued on the engine stream (adb_stream()); they are asynchronous
 *    unless a host out-parameter (h_count, h_value ...) is non-NULL, in which case the
 *    call synchronises and fills it.  Every operator that produces a variable-length
 *    result also writes its length to a device int64 (d_count) so the next operator
 *    can consume it without a host round trip.
 */
#ifndef ADB_ENGINE_H
#define ADB_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADB_API __attribute__((visibility("default")))

typedef int32_t adb_status;
enum {
    ADB_OK = 0,
    ADB_ERR_NOT_INITIALISED = -1,
    ADB_ERR_CUDA = -2,          /* a CUDA runtime call failed; see adb_last_error() */
    ADB_ERR_INVALID = -3,       /* bad argument (NULL pointer, n >= 2^31, misalignment) */
    ADB_ERR_NOMEM = -4,
    ADB_ERR_NCCL = -5
};

/* ---- lifecycle (no reference equivalent; SURVEY.md section 8b "new hooks") ---------- */
ADB_API adb_status adb_init(int device_ordinal);      /* call from main(), src/server.c:616 */
ADB_API adb_status adb_shutdown(void);                /* call from shutdown_server(), src/server.c:40 */
/* Several engine contexts in one process -- one per GPU of the box (north_star: "columns are
 * row-range partitioned across the 8 B200s of one box"; the reference server is ONE process,
 * src/server.c:616-656, so its operator API can only reach several GPUs from inside it).
 * Every entry point of this header works on the calling THREAD's current context (context 0
 * until adb_ctx_select is called); adb_init() initialises the current context.  Contexts may
 * share a device, so the multi-shard host path also runs on a 1-GPU box.  A context must only
 * be driven by one thread at a time.  adb_shutdown() shuts down every context. */
#define ADB_MAX_CONTEXTS 16
ADB_API int32_t adb_device_count(void);
ADB_API adb_status adb_ctx_init(int32_t ctx, int device_ordinal);   /* select + adb_init */
ADB_API adb_status adb_ctx_select(int32_t ctx);
ADB_API int32_t adb_ctx_current(void);
/* the current context's stream waits for everything enqueued so far on other_ctx's stream */
ADB_API adb_status adb_ctx_wait(int32_t other_ctx);
/* copy into the current context from a buffer of src_ctx (peer DMA across devices), ordered
 * after src_ctx's stream */
ADB_API adb_status adb_copy_from_ctx(void *d_dst, int32_t src_ctx, const void *d_src, size_t bytes);
/* the same when the source context has already synchronised its stream (no cross-stream wait) */
ADB_API adb_status adb_copy_from_ctx_ready(void *d_dst, int32_t src_ctx, const void *d_src, size_t bytes);
ADB_API const char *adb_last_error(void);
ADB_API const char *adb_version(void);
ADB_API int adb_sm_count(void);

/* ---- device memory and stream plumbing ----------------------------------------------- */
ADB_API adb_status adb_alloc(void **d_ptr, size_t bytes);            /* stream-ordered pool */
ADB_API adb_status adb_free(void *d_ptr);
/* adb_alloc / adb_free keep a small front cache of freed blocks per context (size classes with
 * <= 12.5 % slack; ADB_ALLOC_CACHE_MB caps it, default 16384): a hit is host bookkeeping where
 * cudaMallocAsync / cudaFreeAsync cost microseconds.  Blocks keep the pool's stream-ordered
 * semantics (reused on this context's stream only).  The *_cached_on forms serve context `ctx`
 * from another thread when -- and only when -- no CUDA call is needed (return 1), so a host that
 * drives several contexts releases and re-acquires result buffers without switching devices;
 * on 0 the caller goes through adb_alloc / adb_free on that context.  The context must be idle. */
ADB_API int32_t adb_alloc_cached_on(int32_t ctx, void **d_ptr, size_t bytes);
ADB_API int32_t adb_free_cached_on(int32_t ctx, void *d_ptr);
ADB_API adb_status adb_upload(void *d_dst, const void *h_src, size_t bytes);     /* H2D, synchronous */
ADB_API adb_status adb_download(void *h_dst, const void *d_src, size_t bytes);   /* D2H, synchronous */
ADB_API adb_status adb_upload_async(void *d_dst, const void *h_src, size_t bytes);
ADB_API adb_status adb_download_async(void *h_dst, const void *d_src, size_t bytes);
ADB_API adb_status adb_memset(void *d_dst, int byte, size_t bytes);
ADB_API adb_status adb_sync(void);
ADB_API void *adb_stream(void);                       /* the cudaStream_t operators run on */
ADB_API adb_status adb_set_stream(void *cuda_stream); /* adopt a caller's stream (NULL = legacy default) */
ADB_API adb_status adb_host_alloc(void **h_ptr, size_t bytes);       /* pinned host memory */
ADB_API adb_status adb_host_free(void *h_ptr);
/* page-lock / unlock a host range that is uploaded from repeatedly (then adb_upload is one DMA at
 * the link's rate instead of a staged copy); failures of the unlock are ignored */
ADB_API adb_status adb_host_register(void *h_ptr, size_t bytes);
ADB_API adb_status adb_host_unregister(void *h_ptr);
/* CUDA-event stopwatch on the engine stream: start, run operators, stop -> milliseconds. */
ADB_API adb_status adb_timer_start(void);
ADB_API adb_status adb_timer_stop(float *ms);
/* Per-kernel timing: record CUDA event `slot` on the engine stream between operators,
 * then read the milliseconds between two recorded slots (synchronises on to_slot). */
#define ADB_MAX_MARKS 8192
ADB_API adb_status adb_mark(int32_t slot);
ADB_API adb_status adb_mark_elapsed(int32_t from_slot, int32_t to_slot, float *ms);
/* Per-kernel timing inside the fused chain: the next adb_chain_select_fetch_agg records
 * slots base, base+1, base+2 before the predicate pass, between its two kernels and after
 * the fused expansion.  One-shot; a negative base cancels. */
ADB_API adb_status adb_chain_marks(int32_t base_slot);
/* number of engine kernels launched since adb_init (bench.py's gpu_launches) */
ADB_API int64_t adb_launch_count(void);
ADB_API int64_t adb_launch_count_all(void);           /* summed over every context */

/* ---- range select over a base column -- replaces select_column_scan, src/query.c:92-137
 * d_pos_out must hold n int32 (the reference mallocs row_count ints, query.c:94).
 * Emits base_pos + row for every row with lo <= d_col[row] < hi, ascending.
 * d_count (device int64, required) receives the hit count; h_count optional. */
ADB_API adb_status adb_select_scan(const int32_t *d_col, int64_t n, const int32_t *lo, const int32_t *hi,
                           int32_t base_pos, int32_t *d_pos_out, int64_t *d_count,
                           int64_t *h_count);

/* ---- two-phase select: size the position list exactly (the reference mallocs row_count
 * ints per select, query.c:94; 2 GB per handle on a 500 M-row shard is not an option in
 * HBM).  adb_select_count runs the predicate pass over d_val (a base column or the value
 * half of a pair list) and returns the hit count; adb_select_emit then writes the positions:
 * base_pos + row when d_pos_in is NULL (select_column_scan), d_pos_in[row] otherwise
 * (select_result, src/query.c:38-86).  n_max bounds the input length; when d_n is non-NULL
 * the actual length is read from that device int64 (<= n_max).  d_count may be NULL.  Any
 * other select between the two calls invalidates the pending count. */
ADB_API adb_status adb_select_count(const int32_t *d_val, int64_t n_max, const int64_t *d_n,
                            const int32_t *lo, const int32_t *hi, int64_t *d_count,
                            int64_t *h_count);
ADB_API adb_status adb_select_emit(const int32_t *d_pos_in, int32_t base_pos, int32_t *d_pos_out);
/* Count phase over rows [base_pos, base_pos + n) of a BASE column (shard).  A base column is
 * never written by an operator, so the predicate pass may request its first tile while the
 * previous kernel on the stream is still draining (adb_select_count cannot: its input may be
 * that kernel's output), and the pending select can be resolved by adb_select_emit_fetch_agg*,
 * which then emit base_pos + row. */
ADB_API adb_status adb_select_count_base(const int32_t *d_col, int64_t n, const int32_t *lo, const int32_t *hi,
                                 int32_t base_pos, int64_t *d_count, int64_t *h_count);

/* ---- fetch (gather) -- replaces fetch_column, src/query.c:223-243
 * d_val_out[i] = d_col[d_pos[i] - base_pos], i < n (n from d_n when non-NULL). */
ADB_API adb_status adb_fetch(const int32_t *d_col, const int32_t *d_pos, int64_t n_max,
                     const int64_t *d_n, int32_t base_pos, int32_t *d_val_out);
/* fetch over a column that is row-range sharded across contexts (SURVEY.md 8e): d_shards is a
 * HOST array of n_shards device pointers, shard k holding rows [k * shard_rows, (k+1) *
 * shard_rows); d_pos holds global positions in any order.  Remote shards are read over NVLink
 * peer memory (adb_peer_connect_local enables the access). */
ADB_API adb_status adb_fetch_sharded(const int32_t *const *d_shards, int32_t n_shards, int64_t shard_rows,
                             const int32_t *d_pos, int64_t n_max, const int64_t *d_n, int32_t *d_val_out);

/* ---- aggregates -- replace sum / average / min / max, src/query.c:306-437
 * One pass produces all three partials; sum is int64 (query.c:326-327).  Empty input:
 * sum 0, min INT32_MAX, max INT32_MIN (the reference reads payload[0], query.c:395,420:
 * oracle-undefined).  average = (double)sum / (double)count on the host
 * (query.c:314).  d_out is a device adb_agg; h_out optional (synchronises). */
typedef struct adb_agg {
    int64_t sum;
    int64_t count;
    int32_t min;
    int32_t max;
} adb_agg;
ADB_API adb_status adb_aggregate(const int32_t *d_val, int64_t n_max, const int64_t *d_n,
                         adb_agg *d_out, adb_agg *h_out);
/* Emit phase of a pending adb_select_count over a base column with fetch_column and the
 * aggregates fused in (SURVEY.md 8f rank 3: a select whose only consumers so far are a fetch
 * and an aggregate is resolved when the aggregate is asked for): one kernel writes the
 * positions, d_val_out[i] = d_fetch_col[d_pos_out[i]] and the {sum, count, min, max} of those
 * values -- the second kernel of adb_chain_select_fetch_agg, with the host having read the hit
 * count in between to size both lists.  d_agg is a device adb_agg; h_agg optional
 * (synchronises). */
ADB_API adb_status adb_select_emit_fetch_agg(const int32_t *d_fetch_col, int32_t *d_pos_out,
                                             int32_t *d_val_out, adb_agg *d_agg,
                                             adb_agg *h_agg);
/* Serial number of the select whose bitmap sits in the engine's scratch: it changes whenever
 * any select (of any form) starts and whenever a pending count is consumed by an emit.  A
 * caller that defers adb_select_emit compares it with the value it read right after its
 * adb_select_count to learn whether the count is still pending. */
ADB_API uint64_t adb_select_generation(void);
/* Combine `k` device partials (one per shard) into d_out[0] on the device. */
ADB_API adb_status adb_agg_combine(const adb_agg *d_parts, int32_t k, adb_agg *d_out, adb_agg *h_out);

/* Multi-GPU: split a device partial into allreduce operands -- {sum, count} (int64 x 2,
 * ncclSum) and {max, ~min} (int32 x 2, ncclMax) -- and fold the reduced operands back. */
ADB_API adb_status adb_agg_export(const adb_agg *d_agg, int64_t *d_sum_count, int32_t *d_max_notmin);
ADB_API adb_status adb_agg_import(const int64_t *d_sum_count, const int32_t *d_max_notmin, adb_agg *d_agg);

/* ---- bulk load: CSV text -> int32 columns -- replaces the ingest loop of load_db,
 * src/db_manager.c:304-318 (fgets line by line, strsep at ',', atoi per token, insert_row
 * per row); SURVEY.md 8f rank 1.  The text (the file's bytes) is already in device memory
 * (adb_alloc + adb_upload, which stages large pageable buffers through pinned lanes).
 *   adb_csv_index   builds the line index; *h_rows = lines after `skip_lines` header lines
 *                   (load_db consumes one, db_manager.c:263), counted as fgets counts them:
 *                   every '\n'-terminated line, plus a non-empty unterminated last line.
 *   adb_csv_parse   fills n_cols caller-allocated device columns of >= *h_rows ints.  Field
 *                   values are bit-identical to atoi's (glibc: (int) strtol): leading
 *                   whitespace, sign, digits to the first non-digit, saturation at
 *                   LONG_MAX/LONG_MIN then truncation.  Fields beyond n_cols are ignored; a
 *                   missing field repeats the value of the nearest earlier row that had the
 *                   field, as the reference's reused row[] does (0 if no earlier row had it,
 *                   where the reference reads uninitialised stack).  A line longer than 1023
 *                   bytes (fgets would split it, db_manager.c:23) is ADB_ERR_INVALID.
 *                   n_cols <= 254.  It is adb_csv_parse_piece + adb_csv_fill with a zero carry.
 * d_cols is a HOST array of n_cols device pointers.
 *
 * A file cut into pieces at line boundaries (one per GPU): the first rows of a piece may inherit
 * a value from an earlier piece, so the parse and the fill are split:
 *   adb_csv_parse_piece  after adb_csv_index: adb_csv_parse without the fill.  For every column
 *                        c < n_cols, h_has[c] = some row of the piece has field c, h_last[c] = its
 *                        value in the last such row (0 if none); *h_short = some row had fewer
 *                        than n_cols fields.  Synchronises.
 *   adb_csv_fill         fills the missing fields of that piece: the nearest earlier row of the
 *                        piece that has the field, else h_carry[c] (n_cols ints; NULL = zeros).
 *                        Enqueued on the stream, not waited for; nothing to do without a short
 *                        row.  Linear in rows plus missing cells.
 * The carry into piece g is piece g-1's h_last[c] where h_has[c], else the carry into g-1. */
ADB_API adb_status adb_csv_index(const char *d_text, size_t bytes, int32_t skip_lines, int64_t *h_rows);
ADB_API adb_status adb_csv_parse(int32_t n_cols, int32_t *const *d_cols);
ADB_API adb_status adb_csv_parse_piece(int32_t n_cols, int32_t *const *d_cols, int32_t *h_last, int32_t *h_has,
                                       int32_t *h_short);
ADB_API adb_status adb_csv_fill(const int32_t *h_carry);

/* ---- result text: the INT branch of print, src/query.c:262-269 ("%d" per tuple, "\n"
 * between tuples, nothing after the last); SURVEY.md 8f rank 2.  Two-phase like the
 * selects: adb_format_i32_count sizes the text (*h_bytes, without a terminating NUL),
 * adb_format_i32_emit writes it to a 16-byte-aligned device buffer of that size; the caller
 * downloads text instead of integers and never runs sprintf.  The text must stay below
 * 4 GiB per call (the reference's reply path stops at a few MB, server.c:522). */
ADB_API adb_status adb_format_i32_count(const int32_t *d_val, int64_t n, int64_t *h_bytes);
ADB_API adb_status adb_format_i32_emit(char *d_text);

/* ---- multi-GPU aggregate exchange over NVLink peer memory (no reference equivalent: the
 * reference is single-process; SURVEY.md 8e "sum / min / max / avg: one exchange step").
 * One process per GPU.  Every rank calls adb_peer_create, the 64-byte handles are exchanged
 * by the host plumbing (any all-gather), every rank calls adb_peer_connect with all `world`
 * handles in rank order.  adb_agg_combine_allreduce then folds this rank's `k` shard
 * partials and exchanges the result with every peer inside ONE kernel (stores into the
 * peers' mailboxes, acquire-spin on its own): d_out holds the table-wide aggregate on every
 * rank.  Collective: all ranks must call it, in the same order.  A peer that does not
 * arrive within 2 s yields count = -1 (and ADB_ERR_CUDA from the next adb_sync-ing call
 * that reads it through h_out). */
#define ADB_MAX_PEERS 16
#define ADB_PEER_HANDLE_BYTES 64
ADB_API adb_status adb_peer_create(int32_t world, int32_t rank, unsigned char *handle_out);
ADB_API adb_status adb_peer_connect(const unsigned char *handles);
ADB_API adb_status adb_agg_combine_allreduce(const adb_agg *d_parts, int32_t k, adb_agg *d_out,
                                             adb_agg *h_out);
/* The north-star chain of this rank's LAST shard of a step with the exchange fused in: the
 * shard's partial goes to d_parts[k-1] (earlier shards of the step filled d_parts[0..k-1)
 * through adb_chain_select_fetch_agg), and the CTA that completes it folds all k partials and
 * exchanges them with every peer in the same kernel: no launch and no collective call is left
 * between the last gather and the table-wide result in d_out.  Collective. */
ADB_API adb_status adb_chain_select_fetch_agg_exchange(const int32_t *d_sel_col, const int32_t *d_fetch_col,
                                                       int64_t n, const int32_t *lo, const int32_t *hi,
                                                       int32_t *d_pos_out, int32_t *d_val_out,
                                                       int64_t *d_count, adb_agg *d_parts, int32_t k,
                                                       adb_agg *d_out);
/* Pair exchange of the sharded hash join (SURVEY.md 8e: "hash-partition both (key, pos)
 * lists by key to G GPUs ... all-to-all-v") over NVLink peer memory.  After adb_peer_connect:
 * every rank reserves a receive buffer (adb_peer_join_create: cap_pairs pairs per side), the
 * 64-byte handles are all-gathered by the host plumbing, every rank calls
 * adb_peer_join_connect.  adb_peer_exchange_pairs(side, ...) then routes this rank's
 * (value, position) pairs by the routing hash of adb_route_pairs and writes every
 * destination's run straight into that rank's receive region: the pieces land ordered by
 * source rank and in source order inside a piece -- the layout of an all-to-all-v.  On
 * return (*h_recv_count pairs at *d_recv_val / *d_recv_pos, valid until the next exchange
 * of the same side) every source's pairs have landed.  side is 0 or 1, so both inputs of a
 * join can be resident at once.  Collective; any world size.
 * ADB_ERR_NOMEM when some rank would receive more than cap_pairs (no rank writes anything). */
ADB_API adb_status adb_peer_join_create(int64_t cap_pairs, unsigned char *handle_out);
ADB_API adb_status adb_peer_join_connect(const unsigned char *handles);
ADB_API adb_status adb_peer_exchange_pairs(int32_t side, const int32_t *d_val, const int32_t *d_pos, int64_t n,
                                           int64_t *h_recv_count, const int32_t **d_recv_val,
                                           const int32_t **d_recv_pos);
ADB_API adb_status adb_peer_destroy(void);
/* The same exchange group inside ONE process: contexts 0 .. world-1 become ranks 0 .. world-1.
 * Mailboxes and receive regions are reached through peer access (cudaDeviceEnablePeerAccess,
 * plus access to the peers' stream-ordered pools so that columns and results can be read
 * across devices) instead of IPC handles.  Call from one thread while no other thread drives
 * a context. */
ADB_API adb_status adb_peer_connect_local(int32_t world);
ADB_API adb_status adb_peer_join_connect_local(int64_t cap_pairs);
/* adb_select_emit_fetch_agg with the exchange riding in the same kernel (the deferred form of
 * adb_chain_select_fetch_agg_exchange): this context's partial goes to d_part, the table-wide
 * aggregate to d_out (h_out optional) on every context.  Collective. */
ADB_API adb_status adb_select_emit_fetch_agg_exchange(const int32_t *d_fetch_col, int32_t *d_pos_out,
                                              int32_t *d_val_out, adb_agg *d_part, adb_agg *d_out,
                                              adb_agg *h_out);

/* ---- element-wise add / sub -- replace add / sub, src/query.c:356-390 (int32, wraps) */
ADB_API adb_status adb_add(const int32_t *d_a, const int32_t *d_b, int64_t n_max, const int64_t *d_n,
                   int32_t *d_out);
ADB_API adb_status adb_sub(const int32_t *d_a, const int32_t *d_b, int64_t n_max, const int64_t *d_n,
                   int32_t *d_out);

/* ---- fused north-star chain: select -> fetch -> sum/min/max on one shard ---------------
 * Equivalent to adb_select_scan + adb_fetch + adb_aggregate with the position list and
 * the fetched values still materialised in d_pos_out / d_val_out (the handles stay
 * observable, src/server.c:184,205), enqueued back to back with no host round trip. */
ADB_API adb_status adb_chain_select_fetch_agg(const int32_t *d_sel_col, const int32_t *d_fetch_col,
                                      int64_t n, const int32_t *lo, const int32_t *hi,
                                      int32_t *d_pos_out, int32_t *d_val_out,
                                      int64_t *d_count, adb_agg *d_agg);
/* The chain with NEITHER handle materialised (SURVEY.md 8f rank 3: "select -> fetch -> sum
 * without materialising s / f ... cuts the chain from 4N + 20H to 4N + 4H bytes"): one kernel
 * scans d_sel_col and gathers + folds d_fetch_col at every hit.  d_count and d_agg are device
 * outputs, h_agg optional (synchronises).  Likewise adb_select_emit_fetch_agg[_exchange] with
 * d_pos_out == d_val_out == NULL aggregates the pending select's hits without writing them and
 * leaves the select pending. */
ADB_API adb_status adb_chain_select_agg(const int32_t *d_sel_col, const int32_t *d_fetch_col, int64_t n,
                                const int32_t *lo, const int32_t *hi, int64_t *d_count, adb_agg *d_agg,
                                adb_agg *h_agg);

/* ---- batched shared scan -- replaces shared_select + select_task, src/query.c:450-583
 * One pass over d_col evaluates q_count (<= ADB_MAX_BATCH, the dispatcher's chunk,
 * src/server.c:366-371) predicates lows[q] <= v < highs[q]; has_low/has_high are ignored
 * exactly as query.c:474 does.  Two phases so the caller can size each position list
 * exactly (the reference mallocs row_count ints per query, query.c:556):
 *   adb_shared_select_count  scans, classifies, returns every query's hit count;
 *   adb_shared_select_emit   writes query q's ascending positions to d_out_ptrs[q]
 *                            (a HOST array of q_count device pointers), at most `capacity`
 *                            positions each. */
#define ADB_MAX_BATCH 150
ADB_API adb_status adb_shared_select_count(const int32_t *d_col, int64_t n, const int32_t *lows,
                                           const int32_t *highs, int32_t q_count, int64_t *h_counts);
ADB_API adb_status adb_shared_select_emit(int32_t *const *d_out_ptrs, int64_t capacity);
/* count phase over rows [base_pos, base_pos + n) of a column (shard): the emit phase then
 * writes base_pos + row (global positions of a row-range sharded column) */
ADB_API adb_status adb_shared_select_count_base(const int32_t *d_col, int64_t n, int32_t base_pos,
                                                const int32_t *lows, const int32_t *highs, int32_t q_count,
                                                int64_t *h_counts);

/* Host-only (no device, no adb_init): the lookup tables adb_shared_select_count would upload
 * for this batch, for inspection and tests.  plan_out may be NULL to size the buffer.
 * meta_out[16] = {bytes, m (distinct bounds), lut_shift, bit_shift, span, lo (bounds[0]),
 * deepest cover, then the byte offsets of cov_off, cov_q, lut, bits, q_first/q_last, cov4,
 * then the lut and bitmap sizes and the q_first -> q_last stride}.  Layout: bounds[m] int32
 * ascending; interval id k = number of bounds <= v (0 and m lie outside every query);
 * cov_off[m+2] uint16 + cov_q[] uint8: the queries covering interval k, ascending; lut /
 * bits: value -> interval tables over d = v - lo (shared_scan.cu); q_first/q_last uint16:
 * the interval ids query q covers; cov4[m+1] uint32: for batches at most four queries deep,
 * interval k's covering queries one byte per colour (0xFF = none), overlapping queries in
 * different colours. */
ADB_API adb_status adb_shared_select_plan(const int32_t *lows, const int32_t *highs, int32_t q_count,
                                          unsigned char *plan_out, size_t capacity, uint32_t *meta_out);

/* ---- sorted index and B+-tree range select -- replace select_column_sorted_index +
 * binary_search, src/query.c:143-198 (and the stub src/btree.c, whose only defined
 * behaviour is "same as sorted", query.c:205-217).
 * An adb_index wraps a device-resident sorted copy of a column (d_values ascending) and
 * its row permutation (d_positions, int32: the reference truncates its size_t positions
 * to int when it emits them, query.c:187).  The arrays stay owned by the caller -- upload
 * the reference's own ColumnIndex for bit-exact tie order, or build one with
 * adb_index_sort().  with_btree additionally bulk-loads a fan-out-32 implicit B+-tree.
 * adb_select_index_emit writes d_positions[first .. first+count) in index order with exactly the
 * reference's result in its defined domain (including the low == high quirk) and scan
 * semantics where the reference crashes (low/high below the minimum, NULL bounds). */
typedef struct adb_index adb_index;
ADB_API adb_status adb_index_create(const int32_t *d_values, const int32_t *d_positions, int64_t n,
                                    int32_t with_btree, adb_index **out);
ADB_API adb_status adb_index_destroy(adb_index *ix);
/* `ix` is one slice of an index range-partitioned (by index order) over several contexts: it
 * answers positions[lb(low) .. lb(high)) of its slice; the caller applies the low == high quirk
 * of query.c:181-188 to the whole index. */
ADB_API adb_status adb_index_set_slice(adb_index *ix, int32_t is_slice);

/* two phases, as adb_select_count / adb_select_emit */
ADB_API adb_status adb_select_index_count(const adb_index *ix, int32_t use_btree, const int32_t *lo,
                                          const int32_t *hi, int64_t *d_count, int64_t *h_count);
ADB_API adb_status adb_select_index_emit(const adb_index *ix, int32_t *d_pos_out);

/* ---- index build -- replaces quicksort / partition / init_column_index, src/index.c:25-101
 * (values ascending, positions) of d_col by a stable LSD radix sort: ties come out in
 * ascending row order.  The reference's unstable Lomuto quicksort leaves another tie
 * order (SURVEY.md A3); the two agree whenever keys are unique.  A clustered index then
 * permutes the sibling columns with adb_fetch(sibling, positions) (index.c:105-135). */
ADB_API adb_status adb_index_sort(const int32_t *d_col, int64_t n, int32_t *d_values_out,
                                  int32_t *d_positions_out);
/* The same (values, positions) with equal keys in exactly the order the reference's quicksort
 * leaves them (init_column_index + quicksort, src/index.c:25-46,89-101), positions narrowed to
 * int32.  Same arguments and refusals as adb_index_sort; the values always equal its values,
 * the positions differ only inside runs of equal keys.  When no key repeats it costs the radix
 * sort plus one pass over the sorted keys; otherwise the quicksort's levels run on the GPU, all
 * segments of a level at once. */
ADB_API adb_status adb_index_sort_ref_ties(const int32_t *d_col, int64_t n, int32_t *d_values_out,
                                           int32_t *d_positions_out);
/* The index build over several contexts (range-partitioned slices, see adb_index_set_slice):
 *   adb_rank_hist        one round of a multi-target radix select over this context's keys.  With
 *                        f = key ^ 0x80000000 (signed order), h_hist[i * 256 + d] = keys whose top
 *                        8 * round bits of f equal h_prefixes[i] and whose next 8 bits are d.  round
 *                        in [0, 3]; 1 .. ADB_MAX_PEERS prefixes, ascending, each below 2^(8 * round)
 *                        (round 0: the one prefix 0).  Summed over the contexts, four rounds narrow
 *                        any number of ranks to their exact keys.
 *   adb_route_range      stable partition of this context's keys by the slice that holds them:
 *                        slice(k) = #{i < parts - 1 : h_splitters[i] < k} (signed), the splitters
 *                        nondecreasing, parts in [1, ADB_MAX_PEERS].  Rows bound for slice s land
 *                        contiguously, in row order, at offset sum(h_counts[0..s)) of d_keys_out,
 *                        their row numbers row_base + local row at the same offsets of d_rows_out
 *                        (row_base + n <= 2^31).  Synchronises.
 *   adb_index_sort_pairs adb_index_sort of d_keys carrying the given payload instead of the input
 *                        index: the same four stable 8-bit LSD passes, equal keys keep their input
 *                        order.  The outputs must not overlap the inputs. */
ADB_API adb_status adb_rank_hist(const int32_t *d_col, int64_t n, const uint32_t *h_prefixes, int32_t n_prefixes,
                                 int32_t round, uint32_t *h_hist);
ADB_API adb_status adb_route_range(const int32_t *d_keys, int64_t n, int64_t row_base, const int32_t *h_splitters,
                                   int32_t parts, int32_t *d_keys_out, int32_t *d_rows_out, int64_t *h_counts);
ADB_API adb_status adb_index_sort_pairs(const int32_t *d_keys, const int32_t *d_payload, int64_t n,
                                        int32_t *d_values_out, int32_t *d_payload_out);
/* ColumnIndex.positions are size_t on the host (src/include/cs165_api.h:65-68) and truncated
 * to int when emitted (src/query.c:187): d_dst[i] = (int32_t) d_src_u64[i]. */
ADB_API adb_status adb_narrow_u64_to_i32(const void *d_src_u64, int64_t n, int32_t *d_dst);
/* the other direction, for handing a device-built index back to the host catalog:
 * d_dst_u64[i] = (size_t) d_src[i]; d_src == NULL writes the identity (the positions of a
 * clustered index stay 0..n-1, src/index.c:89-101,119-135) */
ADB_API adb_status adb_widen_i32_to_u64(const int32_t *d_src, int64_t n, void *d_dst_u64);
/* d_out[i] = first + i (identity positions: init_column_index, src/index.c:89-101) */
ADB_API adb_status adb_iota_i32(int32_t *d_out, int64_t n, int32_t first);
/* build_histogram, src/index.c:63-84: h_counts[b] (b < 100) = rows with (v - vmin) / bin_size == b;
 * bins past 99 (the reference writes out of bounds there) are dropped */
ADB_API adb_status adb_histogram_i32(const int32_t *d_val, int64_t n, int32_t vmin, int32_t bin_size,
                                     uint64_t *h_counts);

/* ---- updates and deletes (SURVEY.md 8f rank 4) -- relational_update / relational_delete of
 * milestone 5 (project_tests/data_generation_scripts/milestone5.py:123-262: `UPDATE tbl SET col =
 * v WHERE ...` as u=select(...); relational_update(col, u, v), `DELETE FROM tbl WHERE ...` as
 * d=select(...); relational_delete(tbl, d)).  The reference's parser has no branch for either
 * (src/parse.c:876-960), so these have no reference function to replace; the semantics are the
 * generator's pandas model: an update overwrites col[pos] for every listed position, a delete
 * removes the listed rows from every column of the table, survivors keep their order.
 *   adb_update_rows        d_col[d_pos[i] - base_pos] = value for the positions that fall into
 *                          [base_pos, base_pos + n_rows) (a shard ignores the other shards' rows)
 *   adb_delete_rows_plan   marks the rows of d_pos (duplicates allowed) among n_rows rows and
 *                          computes where the survivors move; *h_rows_left = rows left
 *   adb_delete_rows_apply  compacts one column with the plan (d_col_out != d_col, >= rows left) */
ADB_API adb_status adb_update_rows(int32_t *d_col, int64_t n_rows, const int32_t *d_pos, int64_t n_pos,
                                   int32_t base_pos, int32_t value);
ADB_API adb_status adb_delete_rows_plan(int64_t n_rows, const int32_t *d_pos, int64_t n_pos, int32_t base_pos,
                                        int64_t *h_rows_left);
ADB_API adb_status adb_delete_rows_apply(const int32_t *d_col, int32_t *d_col_out);

/* ---- joins -- replace hash_join + multimap (src/query.c:652-696, src/multimap.c) and
 * nested_loop_join (src/query.c:585-650).  Inputs are two (value, position) pair lists;
 * outputs two aligned position lists.  Order is the reference's: hash join probe-major
 * over side two with side one's insertion order inside a key; nested-loop outer-major
 * over side one.  Two phases so the result can be sized exactly:
 *   *_join_count   does all the work up to the output offsets, returns the pair count;
 *   adb_join_emit  writes the pairs (d_out1 = side-one positions, d_out2 = side-two).
 * Negative keys and an empty build side, on which the reference crashes (SURVEY.md A5),
 * follow the equi-join definition.  The pair count must stay below 2^31 (query.c:657). */
ADB_API adb_status adb_hash_join_count(const int32_t *d_v1, const int32_t *d_p1, int64_t n1,
                                       const int32_t *d_v2, const int32_t *d_p2, int64_t n2,
                                       int64_t *h_matches);
ADB_API adb_status adb_nested_loop_join_count(const int32_t *d_v1, const int32_t *d_p1, int64_t n1,
                                              const int32_t *d_v2, const int32_t *d_p2, int64_t n2,
                                              int64_t *h_matches);
ADB_API adb_status adb_join_emit(int32_t *d_out1, int32_t *d_out2);
/* ---- routed exchange (several contexts of one process) --------------------------------------
 * Items travel in bulk to the context that owns them, the owner answers them, and the answers
 * travel back in bulk to their home, which puts them in the items' original order.  The sharded
 * join's probe and the routed fetch below take it; every step on every context, a host barrier
 * after each:
 *   1. partition (adb_join_route_probe / adb_route_rows): a stable partition of this context's
 *      items by owner.  h_counts[o] = items bound for context o; they sit at offset
 *      sum(h_counts[0..o)) of *d_routed_keys / *d_routed_pos, in row order.  *d_answers = where
 *      context o's answers belong, at the same offsets.  Synchronises;
 *   2. owner: adb_join_recv_buffers(n_recv) + one adb_copy_from_ctx[_ready] per source context
 *      (pieces in source-context order), then the owner's own work writes one answer per received
 *      item, in the order received, into *d_answers of adb_join_recv_buffers.  Synchronises;
 *   3. home: one adb_copy_from_ctx[_ready] per owner into step 1's *d_answers, then the finish
 *      call (adb_join_finish_routed / adb_route_finish32) puts the answers back in row order.
 * Steps 1 and 2 end synchronised, so with a host barrier after each the _ready copies are safe. */
/* The join sharded over the contexts of ONE process (SURVEY.md 8e "hash join: hash-partition both
 * (key, pos) lists by key to G GPUs"), keeping the reference's output order.  world = number of
 * contexts, 2 .. ADB_MAX_PEERS; swapped as in adb_nested_loop_join_count.  Every step on every
 * context, a host barrier after each:
 *   1. every context routes its slice of the BUILD side to the keys' owners
 *      (adb_peer_exchange_pairs, side 0: pieces land in source-rank order = insertion order);
 *   2. every context calls adb_join_build on what it received (sort on the hash + one table per
 *      partition, as steps 1-3 of adb_hash_join_count); probe_rows_hint = the probe rows this
 *      context will bring (scratch is reserved for them).  Synchronises;
 *   3. each context's slice of the PROBE side, in its original order, is answered by the keys'
 *      owners through the routed exchange above, 8 bytes per answer (reading every remote slot
 *      over NVLink instead costs one 32-byte response per 16-byte slot, ~9 G reads/s per GPU):
 *      3a. partition: adb_join_route_probe, the owner taken from the keys' routing hash;
 *      3b. owner: adb_join_probe_received(n_recv) probes what it received;
 *      3c. home: adb_join_finish_routed sets *h_matches = this context's pair count.
 *   4. adb_join_emit writes this context's pairs (multi-row groups read the owner's sorted build
 *      positions over peer memory).  Synchronises.
 * Each context's pairs are probe-major over its own probe rows, so the contexts' outputs
 * concatenated in context order are the reference's probe-major list. */
/* Sizes every scratch buffer steps 1-3 will need on this context (exchange of send_pairs pairs,
 * build over up to build_pairs received pairs, probe_rows probe rows) BEFORE the collective
 * starts: device memory management may wait for the device to go idle, which must not happen
 * while a context sharing the device spin-waits for this one.  Every context, then a barrier. */
ADB_API adb_status adb_peer_exchange_reserve(int64_t send_pairs, int64_t build_pairs, int64_t probe_rows);
ADB_API adb_status adb_join_build(const int32_t *d_v, const int32_t *d_p, int64_t n, int64_t probe_rows_hint);
ADB_API adb_status adb_join_route_probe(int32_t world, const int32_t *d_pv, int64_t np, int64_t *h_counts,
                                        const int32_t **d_routed_keys, void **d_answers);
ADB_API adb_status adb_join_recv_buffers(int64_t n_recv, int32_t **d_keys, void **d_answers);
ADB_API adb_status adb_join_probe_received(int64_t n_recv);
ADB_API adb_status adb_join_finish_routed(int32_t world, const int32_t *d_pv, const int32_t *d_pp, int64_t np,
                                          int32_t swapped, int64_t *h_matches);

/* ---- routed fetch (several contexts, a position list that is not aligned with the shards) ----
 * Instead of adb_fetch_sharded's one NVLink read per remote row, the routed exchange above with
 * 4-byte answers: (1) partition: adb_route_rows, the owner being the shard that holds the row
 * (shard = position / shard_rows, at most world - 1); (2) owner: adb_fetch(column shard, received
 * positions, n, NULL, shard base, answers) + adb_sync; (3) home: adb_route_finish32 writes
 * d_out[i] = value of position i.  Uses the sort / join scratch arena (a join waiting for its emit
 * phase is dropped). */
ADB_API adb_status adb_route_rows(int32_t world, int64_t shard_rows, const int32_t *d_pos, int64_t n,
                                  int64_t *h_counts, const int32_t **d_routed_pos, void **d_answers);
ADB_API adb_status adb_route_finish32(int32_t world, int32_t *d_out, int64_t n);

/* ---- multi-GPU join exchange, send side (no reference equivalent: SURVEY.md 8e) ----------
 * Stable partition of a (value, position) pair list by destination rank = the routing hash
 * h = value * 0x85EBCA6B (mod 2^32) scaled to the ranks, floor(h * parts / 2^32); parts (the
 * world size) is in [1, 256].  Every rank owns floor(2^32 / parts) or that + 1 hash values; for
 * a power of two parts = 2^k the rank is the top k bits of h.  Pairs bound for rank r land
 * contiguously, in their original order, at offset sum(h_counts[0..r)) of the outputs --
 * exactly the send buffer and split sizes of an all-to-all-v.  Equal keys always meet on the
 * same rank. */
ADB_API adb_status adb_route_pairs(const int32_t *d_val, const int32_t *d_pos, int64_t n, int32_t parts,
                                   int32_t *d_val_out, int32_t *d_pos_out, int64_t *h_counts);

/* ---- synthetic data (bench / tests): counter-based generator, identical on host ------
 * d_out[i] = lo + mix64(seed, first_row + i) % span, the same sequence
 * analytical-database_b200/synth.py produces with numpy. */
ADB_API adb_status adb_synth_uniform(int32_t *d_out, int64_t n, uint64_t seed, uint64_t first_row,
                             int32_t lo, uint32_t span);
/* d_out[i] = ((first_row + i) * mul + add) mod modulus (mul, add < modulus <= 2^31): with
 * gcd(mul, modulus) = 1 a permutation of 0 .. modulus-1 -- the unique-key indexed column of
 * BASELINE config 3 (the reference's own M3 experiment uses a random permutation,
 * project_tests/experiment_scripts/data_generation.py:216-218). */
ADB_API adb_status adb_synth_affine(int32_t *d_out, int64_t n, uint64_t first_row, uint64_t mul, uint64_t add,
                            uint64_t modulus);

#ifdef __cplusplus
}
#endif
#endif /* ADB_ENGINE_H */
