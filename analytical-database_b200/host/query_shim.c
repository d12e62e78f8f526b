/*
 * query_shim.c -- the reference's operator API (src/include/query.h:20-44) on the B200
 * engine.  This file is the C host side of the drop-in: it replaces
 * /root/reference/src/query.c and src/multimap.c in the server's link line
 * (src/Makefile:62) and forwards every operator to the C-ABI of libadb_b200.so
 * (include/adb_engine.h).  It computes nothing itself and has no CPU fallback: if the
 * engine cannot start, every operator sets ret_status->code = ERROR and returns NULL,
 * which the dispatcher turns into a "Failed ..." reply (src/server.c:171-174).
 *
 * One process, G GPUs (adb_host_init_multi(G) or ADB_GPUS=G; G = 1 by default)
 *   The reference server is one process serving one client (src/server.c:616-656), so the
 *   multi-GPU path lives here, behind the unchanged operator API: one engine context per GPU
 *   (adb_ctx_*), one host thread per context (the calling thread drives context 0), peer
 *   access between all devices.
 *   base columns    row-range sharded: shard g holds rows [g*S, (g+1)*S) of the column in the
 *                   HBM of GPU g (S = rows per shard, the same for every column of a table, so
 *                   the columns of a table are co-partitioned).
 *   results         a position list / value vector is the concatenation, in shard order, of
 *                   G device buffers; positions are GLOBAL row numbers, so the concatenation
 *                   is exactly the reference's list.  A list produced by a scan select is
 *                   "row-aligned" (shard g's entries name rows of shard g): fetch, the fused
 *                   chain and select_result then run shard-local with no data movement.
 *                   Any other list (index order, join output, host arrays) is fetched with
 *                   peer loads over NVLink (adb_fetch_sharded).
 *   aggregates      per-shard partial + one exchange step over peer memory, fused into the
 *                   kernel that produces the partial (adb_select_emit_fetch_agg_exchange /
 *                   adb_agg_combine_allreduce); the host reads context 0's copy.
 *   indexes         range-partitioned BY INDEX ORDER: slice g holds entries [b_g, b_{g+1}) of
 *                   the sorted (values, positions) arrays, equal keys never straddle a
 *                   boundary.  Every slice answers the range lookup; the concatenation in
 *                   slice order is the reference's value-ordered list, bit for bit.
 *
 * Where things live
 *   base columns    Column.data stays the host mmap the catalog owns; the first operator
 *                   that touches a column uploads it to HBM (int32 array) and the copy is
 *                   reused until the column's data pointer or row_count changes
 *                   (insert_row may re-mmap, src/db_manager.c:178-186).  A column with a
 *                   ColumnIndex also gets its (values, positions) uploaded -- exactly the
 *                   arrays src/index.c built, so tie order is the reference's -- plus the
 *                   implicit B+-tree for `btree` indexes.
 *   results         position lists and value vectors stay in HBM.  Result.payload is a
 *                   plain malloc block of max(16, 4*num_tuples) bytes, so the unchanged
 *                   plumbing may free() it (src/client_context.c:35,82) and may read
 *                   num_tuples ints from it (the dispatcher's no-op log loop,
 *                   src/server.c:177-181); a registry maps that address to the device
 *                   buffers.  The block's bytes are NOT the tuples unless ADB_SHIM_MIRROR=1
 *                   (then every result is also copied back to the host).  Scalars
 *                   (sum / avg / min / max) are ordinary host values, as in the reference.
 *   reclaiming HBM  adb_host_result_release() (two-line patch), the free() interposer
 *                   (host/free_interpose.c, no patch), or -- last resort -- the registry
 *                   notices malloc handing out a payload address again.
 *
 * Behaviour the reference leaves undefined (it reads out of bounds or crashes; SURVEY.md
 * appendix A) is defined here and listed in DESIGN.md: NULL bounds on an indexed column,
 * bounds below the index minimum, min/max/print of an empty result, add/sub of lists of
 * different length (ERROR), negative join keys and an empty join side.
 */
#ifndef _GNU_SOURCE
#define _GNU_SOURCE
#endif
#include <limits.h>
#include <malloc.h>
#include <pthread.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "adb_engine.h"
#include "adb_load_api.h"
#include "adb_query_api.h"

#define MAXG ADB_MAX_PEERS
#define REGISTER_MIN_BYTES ((size_t)64 << 20)

/* ---- state ----------------------------------------------------------------------------- */
typedef struct DevColumn {
    const Column *key;
    const int *host_data;
    size_t rows;
    size_t shard_rows;          /* S: shard g = rows [g*S, min(rows, (g+1)*S)) */
    int32_t *d_data[MAXG];
    int adopted;                /* d_data belongs to the caller (adb_host_column_adopt*) */
    const int *uploaded_from;   /* host array of the last upload, and how often it was uploaded: */
    size_t uploaded_bytes;      /* a large array uploaded a second time is page-locked (insert_row */
    int uploads, registered;    /* invalidates the HBM copy again and again, db_manager.c:164-199)  */
    /* index: slice g = entries [ix_begin[g], ix_begin[g+1]) of the sorted arrays */
    const int *host_ix_values;
    size_t ix_rows;
    size_t ix_begin[MAXG + 1];
    int32_t *d_ix_values[MAXG], *d_ix_positions[MAXG];
    adb_index *ix[MAXG];
    int ix_min;                 /* smallest key of the whole index */
} DevColumn;

/* several results carved out of one allocation per context (shared_select) */
typedef struct Slab {
    int32_t *base[MAXG];
    long refs;
} Slab;

/* One list as G device buffers: d[g] holds n[g] entries on context g, the list is their
 * concatenation in context order.  An operator's output, an operator's input and a registered
 * result are all one of these; list_release() frees what the list owns. */
typedef struct ShardList {
    int32_t *d[MAXG];
    size_t n[MAXG];
    size_t total;               /* sum of n[]: stage() and new_dev_result() set it */
    size_t aligned;             /* S > 0: shard g's entries are positions inside rows [g*S, (g+1)*S) */
    Slab *slab;                 /* the buffers are views into this slab, which owns them */
    int borrowed;               /* the buffers are a registered result's: this view owns nothing */
} ShardList;

typedef struct DevResult {
    void *payload;              /* key: the host block handed out as Result.payload */
    ShardList list;
} DevResult;

#define SLOT_EMPTY ((void *)0)
#define SLOT_TOMB ((void *)1)

static struct {
    int up, failed, mirror, lazy;
    int G;                      /* contexts = shards */
    int register_uploads;       /* page-lock host columns that are uploaded repeatedly (ADB_SHIM_NO_REGISTER=1: never) */
    size_t shard_min_rows;
    size_t rebalance_min;       /* index-ordered lists at least this long are re-cut evenly (ADB_REBALANCE_MIN) */
    int ref_ties;               /* index builds keep the reference quicksort's tie order (ADB_INDEX_TIES=reference) */
    DevColumn *cols;
    int ncols, capcols;
    DevResult *slots;           /* open addressing on payload address */
    size_t nslots, nused;       /* nused counts live + tombstones */
    volatile long nlive;
    adb_agg *d_part[MAXG], *d_out[MAXG];
    pthread_mutex_t mu;
    int mu_ready;
} S;

static size_t jx_cap_now;                           /* pairs a GPU's join receive region holds */
static __thread char t_err[384];

const char *adb_host_last_error(void) { return t_err; }
long adb_host_live_device_results(void) { return S.nlive; }
int adb_host_gpus(void) { return S.up ? S.G : 0; }

static void set_err(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof t_err, fmt, ap);
    va_end(ap);
}

static void lock(void) {
    if (!S.mu_ready) {
        pthread_mutexattr_t a;
        pthread_mutexattr_init(&a);
        pthread_mutexattr_settype(&a, PTHREAD_MUTEX_RECURSIVE);
        pthread_mutex_init(&S.mu, &a);
        pthread_mutexattr_destroy(&a);
        S.mu_ready = 1;
    }
    pthread_mutex_lock(&S.mu);
}
static void unlock(void) { pthread_mutex_unlock(&S.mu); }

/* Every operator must set ret_status->code on every path: the dispatcher's Status locals
 * are uninitialised (src/server.c:141,192). */
static void *op_fail(Status *st, const char *what) {
    if (t_err[0] == '\0') set_err("%s failed", what);
    if (st) {
        st->code = ERROR;
        st->error_message = t_err;
    }
    return NULL;
}
static void op_ok(Status *st) {
    if (st) {
        st->code = OK;
        st->error_message = NULL;
    }
}

/* ---- optional host-side profile (ADB_SHIM_PROFILE=1): wall time per phase, printed by
 * adb_host_shutdown / adb_host_profile_dump ------------------------------------------------- */
#include <time.h>
enum { PF_SELECT, PF_SELECT_JOB, PF_FETCH, PF_FETCH_JOB, PF_AGG, PF_AGG_JOB, PF_NEWRESULT, PF_RELEASE,
       PF_FREE_JOB, PF_LOAD_UPLOAD, PF_LOAD_PARSE, PF_LOAD_FILL, PF_LOAD_RECUT, PF_LOAD_AGG, PF_LOAD_DOWNLOAD,
       PF_IX_SPLIT, PF_IX_ROUTE, PF_IX_RESERVE, PF_IX_PULL, PF_IX_SORT, PF_IX_CATALOG, PF_IX_GLOBAL, PF_IX_SIBLINGS,
       PF_IX_SLICES, PF_COUNT };
static const char *const pf_names[PF_COUNT] = {"select_column", "  its shard job", "fetch_column", "  its shard job",
                                               "aggregate", "  its shard job", "new_dev_result", "payload release",
                                               "  free job", "load: upload", "load: index+parse", "load: fill",
                                               "load: re-cut", "load: aggregate", "load: download",
                                               "index: splitters", "index: route", "index: reserve", "index: pulls",
                                               "index: sort", "index: catalog", "index: sort on GPU 0",
                                               "index: siblings", "index: slices"};
static struct { int on; double t[PF_COUNT]; long n[PF_COUNT]; } PF;
static inline double pf_now(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec * 1e6 + (double)ts.tv_nsec * 1e-3;
}
#define PF_BEGIN(id) const double pf_t0_##id = PF.on ? pf_now() : 0.0
#define PF_END(id)                                   \
    do {                                             \
        if (PF.on) {                                 \
            PF.t[id] += pf_now() - pf_t0_##id;       \
            ++PF.n[id];                              \
        }                                            \
    } while (0)
void adb_host_profile_dump(void) {
    if (!PF.on) return;
    fprintf(stderr, "[adb shim profile] phase                 calls   total us    us/call\n");
    for (int i = 0; i < PF_COUNT; ++i)
        if (PF.n[i])
            fprintf(stderr, "[adb shim profile] %-20s %7ld %10.0f %10.2f\n", pf_names[i], PF.n[i], PF.t[i],
                    PF.t[i] / (double)PF.n[i]);
    memset(PF.t, 0, sizeof PF.t);
    memset(PF.n, 0, sizeof PF.n);
}

/* ---- one host thread per context ---------------------------------------------------------
 * An operator is a function run once per shard: the calling thread runs shard 0 (it stays on
 * context 0), worker g runs shard g on context g.  Workers spin for the next job for a while
 * (operators of one query arrive microseconds apart), then sleep on a condition variable. */
typedef void (*shard_fn)(int g, void *arg);
typedef struct ShardErr {
    char msg[MAXG][256];
    int failed[MAXG];
} ShardErr;

static struct {
    pthread_t th[MAXG];
    int started;
    volatile unsigned long seq;
    shard_fn fn;
    void *arg;
    struct { volatile unsigned long v; char pad[56]; } done[MAXG];
    pthread_mutex_t mu;
    pthread_cond_t cv;
    volatile int sleepers, quit;
    long spin_limit;
} W;

static inline void cpu_relax(void) {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
}

static void *worker_main(void *p) {
    const int g = (int)(intptr_t)p;
    adb_ctx_select(g);
    unsigned long seen = 0;
    for (;;) {
        long spins = 0;
        unsigned long s;
        while ((s = __atomic_load_n(&W.seq, __ATOMIC_ACQUIRE)) == seen && !W.quit) {
            if (++spins > W.spin_limit) {
                pthread_mutex_lock(&W.mu);
                __atomic_add_fetch(&W.sleepers, 1, __ATOMIC_SEQ_CST);
                while (__atomic_load_n(&W.seq, __ATOMIC_SEQ_CST) == seen && !W.quit)
                    pthread_cond_wait(&W.cv, &W.mu);
                __atomic_sub_fetch(&W.sleepers, 1, __ATOMIC_SEQ_CST);
                pthread_mutex_unlock(&W.mu);
                spins = 0;
            } else {
                cpu_relax();
            }
        }
        if (W.quit) break;
        seen = s;
        W.fn(g, W.arg);
        __atomic_store_n(&W.done[g].v, s, __ATOMIC_RELEASE);
    }
    return NULL;
}

static void run_shards(shard_fn fn, void *arg) {
    if (S.G == 1) {
        fn(0, arg);
        return;
    }
    W.fn = fn;
    W.arg = arg;
    const unsigned long s = __atomic_add_fetch(&W.seq, 1, __ATOMIC_SEQ_CST);
    if (__atomic_load_n(&W.sleepers, __ATOMIC_SEQ_CST) > 0) {
        pthread_mutex_lock(&W.mu);
        pthread_cond_broadcast(&W.cv);
        pthread_mutex_unlock(&W.mu);
    }
    fn(0, arg);
    for (int g = 1; g < S.G; ++g)
        while (__atomic_load_n(&W.done[g].v, __ATOMIC_ACQUIRE) != s) cpu_relax();
}

static int workers_start(void) {
    if (S.G == 1 || W.started) return 0;
    pthread_mutex_init(&W.mu, NULL);
    pthread_cond_init(&W.cv, NULL);
    W.quit = 0;
    W.seq = 0;
    const char *sp = getenv("ADB_SHIM_SPIN");
    W.spin_limit = sp ? atol(sp) : 200000;          /* ~ a millisecond or two of pause loops */
    for (int g = 1; g < S.G; ++g) {
        W.done[g].v = 0;
        if (pthread_create(&W.th[g], NULL, worker_main, (void *)(intptr_t)g)) {
            set_err("cannot start the host thread of GPU %d", g);
            return -1;
        }
    }
    W.started = 1;
    return 0;
}
static void workers_stop(void) {
    if (!W.started) return;
    pthread_mutex_lock(&W.mu);
    W.quit = 1;
    pthread_cond_broadcast(&W.cv);
    pthread_mutex_unlock(&W.mu);
    for (int g = 1; g < S.G; ++g) pthread_join(W.th[g], NULL);
    W.started = 0;
}

/* per-shard failure -> the caller's t_err (first failing shard) */
static void shard_fail(ShardErr *e, int g, const char *what) {
    e->failed[g] = 1;
    snprintf(e->msg[g], sizeof e->msg[g], "%s (GPU %d): %s", what, g, adb_last_error());
}
static int shard_errs(const ShardErr *e) {
    for (int g = 0; g < S.G; ++g)
        if (e->failed[g]) {
            set_err("%s", e->msg[g]);
            return -1;
        }
    return 0;
}
#define SCK(call)                                   \
    do {                                            \
        if ((call) != ADB_OK) {                     \
            shard_fail(&a->err, g, #call);          \
            return;                                 \
        }                                           \
    } while (0)

/* ---- routed exchange (adb_engine.h), phases 1-3 of a job with a host barrier after each.  Phases 1
 * and 2 end synchronised, so the pulls are _ready copies. */
typedef struct Route {
    int64_t sent[MAXG][MAXG];                       /* sent[g][o] = items of GPU g owned by GPU o */
    const int32_t *items[MAXG];                     /* GPU g's items grouped by owner */
    void *answers_home[MAXG];                       /* where GPU g collects the owners' answers */
    void *answers_owner[MAXG];                      /* GPU o's answers, in the order it received the items */
} Route;

static int run_routed(shard_fn fn, void *arg, int *phase, const ShardErr *err) {
    for (*phase = 1; *phase <= 3; ++*phase) {
        run_shards(fn, arg);
        if (shard_errs(err)) return -1;
    }
    return 0;
}

/* Owner g: room for what every GPU sent it, its pieces pulled in in source order.  The pulls start
 * at g's own piece and go round, so that at any moment every GPU reads from a different source
 * (r02zj: all eight starting at GPU 0 queued up behind one another on its port). */
static adb_status route_pull(int g, Route *r, int32_t **items, int64_t *n_recv) {
    *n_recv = 0;
    for (int s = 0; s < S.G; ++s) *n_recv += r->sent[s][g];
    adb_status st = adb_join_recv_buffers(*n_recv, items, &r->answers_owner[g]);
    for (int k = 0; k < S.G && st == ADB_OK; ++k) {
        const int s = (g + k) % S.G;
        int64_t at = 0, from = 0;
        for (int t = 0; t < s; ++t) at += r->sent[t][g];
        for (int o = 0; o < g; ++o) from += r->sent[s][o];
        if (r->sent[s][g])
            st = adb_copy_from_ctx_ready(*items + at, s, r->items[s] + from, 4 * (size_t)r->sent[s][g]);
    }
    return st;
}

/* Home g: its answers (elem_bytes each) from every owner, in the same rotated order. */
static adb_status route_return(int g, const Route *r, size_t elem_bytes) {
    adb_status st = ADB_OK;
    for (int k = 0; k < S.G && st == ADB_OK; ++k) {
        const int o = (g + k) % S.G;
        int64_t at = 0, from = 0;                   /* g's piece inside owner o's received list */
        for (int t = 0; t < o; ++t) at += r->sent[g][t];
        for (int s = 0; s < g; ++s) from += r->sent[s][o];
        if (r->sent[g][o])
            st = adb_copy_from_ctx_ready((char *)r->answers_home[g] + elem_bytes * (size_t)at, o,
                                         (const char *)r->answers_owner[o] + elem_bytes * (size_t)from,
                                         elem_bytes * (size_t)r->sent[g][o]);
    }
    return st;
}

/* Main-thread engine calls on another context (cheap bookkeeping: allocations, frees). */
static void on_ctx(int g) {
    if (S.G > 1) adb_ctx_select(g);
}
static void free_on(int g, void *d) {
    if (!d) return;
    on_ctx(g);
    adb_free(d);
    on_ctx(0);
}

/* release one buffer per context: each context's thread frees its own */
typedef struct FreeJob {
    int32_t *d[MAXG];
} FreeJob;
static void free_shard(int g, void *arg) {
    FreeJob *a = arg;
    if (a->d[g]) adb_free(a->d[g]);
}
static void free_shards(int32_t *const d[]) {
    FreeJob job;
    int any = 0;
    for (int g = 0; g < MAXG; ++g) {
        job.d[g] = g < S.G ? d[g] : NULL;
        /* the engine's front cache takes the block back without a CUDA call (and without waking
         * GPU g's thread) whenever it has room */
        if (job.d[g] && adb_free_cached_on(g, job.d[g])) job.d[g] = NULL;
        any |= job.d[g] != NULL;
    }
    if (any) {
        PF_BEGIN(PF_FREE_JOB);
        run_shards(free_shard, &job);
        PF_END(PF_FREE_JOB);
    }
}

/* rows of shard g of a list of `rows` rows cut every S rows */
static size_t shard_len(size_t rows, size_t S_, int g) {
    const size_t b = (size_t)g * S_;
    if (b >= rows) return 0;
    return rows - b < S_ ? rows - b : S_;
}

/* ---- lazy handles (SURVEY.md 8f rank 3) ----------------------------------------------------
 * select_column over an un-indexed column returns as soon as the hit count is known: the
 * predicate pass has left its bitmap in the engine's scratch (one per context), the position
 * buffers are allocated, their contents are NOT written.  fetch_column of that handle
 * launches nothing either.  An aggregate of that fetch -- the s=select / f=fetch / a=sum(f)
 * pattern of src/server.c:137-290 -- gathers and folds the hit rows straight from the bitmap
 * without writing the positions or the values (and with G > 1 exchanges the partials over
 * NVLink in the same kernel): the chain costs 4N + 4H bytes instead of 4N + 20H.  A handle is
 * written only when somebody reads it: print, a second fetch, add / sub, a join,
 * select_result, a second aggregate, a foreign reader (adb_host_result_to_host), or the
 * invalidation of a column it depends on.  The record of the newest select (P) still has its
 * bitmap and is written from it; when the next select takes the bitmap over, the record is
 * demoted to a recipe (R: column, bounds, fetch column, buffers) and writing it re-runs the
 * predicate pass.  A handle that is released unread is never written at all.  To the unchanged
 * plumbing the handles are indistinguishable from eager ones.  ADB_SHIM_EAGER=1 (or the mirror
 * mode) turns all of this off. */
typedef struct Lazy {
    int active;
    const void *sel_payload;        /* registry key of the select handle; NULL once it was released */
    const void *fetch_payload;      /* fetch_column of that select, values not written yet */
    int32_t *sel_d[MAXG];           /* position buffers, h[g] entries */
    int32_t *fetch_d[MAXG];
    int owns_sel;                   /* the select handle is gone: its buffers belong to this record */
    size_t h[MAXG];
    const int32_t *d_col[MAXG];     /* what was scanned, to redo the predicate pass */
    size_t rows[MAXG];
    size_t shard_rows;
    const int32_t *d_fetch_col[MAXG];
    int has_lo, has_hi, lo, hi;
    uint64_t generation[MAXG];      /* adb_select_generation() right after the count (P only) */
    int aggregated;                 /* an aggregate has been answered without writing the handles */
} Lazy;
static Lazy P;                      /* the newest select: its bitmaps sit in the engines' scratch */
static Lazy *R;                     /* older unwritten selects: recipes */
static int nR, capR;

typedef struct LazyJob {
    ShardErr err;
    Lazy *z;
    int have_bitmap;
} LazyJob;

static int32_t shard_base(int g, size_t shard_rows) { return (int32_t)((size_t)g * shard_rows); }

/* runs on context g: redo the predicate pass unless this record's bitmap is still in scratch */
static int lazy_recount_shard(Lazy *z, int have_bitmap, int g, ShardErr *e) {
    if (have_bitmap && adb_select_generation() == z->generation[g]) return 0;
    int64_t h = -1;
    if (adb_select_count_base(z->d_col[g], (int64_t)z->rows[g], z->has_lo ? &z->lo : NULL,
                              z->has_hi ? &z->hi : NULL, shard_base(g, z->shard_rows), NULL, &h) != ADB_OK) {
        shard_fail(e, g, "lazy select");
        return -1;
    }
    if ((size_t)h != z->h[g]) {
        e->failed[g] = 1;
        snprintf(e->msg[g], sizeof e->msg[g],
                 "lazy select: the column changed under an unwritten select (%zu hits, now %lld)",
                 z->h[g], (long long)h);
        return -1;
    }
    z->generation[g] = adb_select_generation();
    return 0;
}

static void lazy_write_shard(int g, void *arg) {
    LazyJob *a = arg;
    Lazy *z = a->z;
    if (lazy_recount_shard(z, a->have_bitmap, g, &a->err)) return;
    if (z->fetch_payload)
        SCK(adb_select_emit_fetch_agg(z->d_fetch_col[g], z->sel_d[g], z->fetch_d[g], S.d_part[g], NULL));
    else
        SCK(adb_select_emit(NULL, shard_base(g, z->shard_rows), z->sel_d[g]));
}

static void lazy_done(Lazy *z) {
    if (z->owns_sel) free_shards(z->sel_d);
    z->owns_sel = 0;
    z->active = 0;
    if (z != &P) {                               /* a recipe: close the gap */
        const int k = (int)(z - R);
        R[k] = R[nR - 1];
        --nR;
    }
}

/* Write the handles of one record; afterwards they are ordinary device results. */
static int lazy_write(Lazy *z) {
    if (!z->active) return 0;
    int rc = 0;
    if (z->sel_payload || z->fetch_payload) {
        LazyJob job;
        memset(&job, 0, sizeof job);
        job.z = z;
        job.have_bitmap = z == &P;
        run_shards(lazy_write_shard, &job);
        rc = shard_errs(&job.err);
    }
    lazy_done(z);
    return rc;
}

static Lazy *lazy_find(const void *payload) {
    if (!payload) return NULL;
    if (P.active && (payload == P.sel_payload || payload == P.fetch_payload)) return &P;
    for (int k = 0; k < nR; ++k)
        if (payload == R[k].sel_payload || payload == R[k].fetch_payload) return &R[k];
    return NULL;
}

/* `payload` is about to be read: write its handle if it is still unwritten */
static int resolve_payload(const void *payload) {
    if (!P.active && nR == 0) return 0;
    Lazy *z = lazy_find(payload);
    return z ? lazy_write(z) : 0;
}

/* a new select is about to take the bitmaps over: P becomes a recipe (no GPU work) */
static int demote_pending(void) {
    if (!P.active) return 0;
    if (!P.sel_payload && !P.fetch_payload) {
        lazy_done(&P);
        return 0;
    }
    if (nR == capR) {
        const int cap = capR ? 2 * capR : 8;
        Lazy *n = realloc(R, (size_t)cap * sizeof *n);
        if (!n) return lazy_write(&P);          /* out of host memory: write it now instead */
        R = n;
        capR = cap;
    }
    R[nR++] = P;
    P.active = 0;
    P.owns_sel = 0;
    return 0;
}

/* The plumbing is about to free (or has freed) this payload.  Returns 1 when the handle's
 * device buffers must NOT be released: an unwritten fetch still needs the select's position
 * buffers as scratch should it ever be written -- they now belong to the record. */
static int pending_payload_gone(const void *payload) {
    if (!P.active && nR == 0) return 0;
    Lazy *z = lazy_find(payload);
    if (!z) return 0;
    if (payload == z->fetch_payload) {           /* nobody can read those values any more */
        z->fetch_payload = NULL;
        if (!z->sel_payload) lazy_done(z);
        return 0;
    }
    if (z->fetch_payload) {                      /* the select goes, its unwritten fetch stays */
        z->sel_payload = NULL;
        z->owns_sel = 1;
        return 1;
    }
    lazy_done(z);
    return 0;
}

/* a column's device copy is about to go: write every handle that would have to re-read it */
static void lazy_column_gone(int32_t *const d_data[]) {
    for (int pass = 0; pass < 2; ++pass)
        for (int k = pass ? nR - 1 : 0; k >= 0; --k) {
            Lazy *z = pass ? &R[k] : &P;
            if (!z->active) continue;
            int uses = 0;
            for (int g = 0; g < S.G; ++g)
                if (d_data[g] && (d_data[g] == z->d_col[g] || d_data[g] == z->d_fetch_col[g])) uses = 1;
            if (uses) lazy_write(z);
        }
}

/* ---- engine lifecycle ------------------------------------------------------------------ */
static int host_init(int first_device, int gpus) {
    if (S.up) return 0;
    if (gpus < 1 || gpus > MAXG) {
        set_err("adb_host_init_multi: %d GPUs outside [1, %d]", gpus, MAXG);
        return -1;
    }
    const int ndev = adb_device_count();
    for (int g = 0; g < gpus; ++g) {
        /* fewer devices than contexts: contexts share devices (a 1-GPU box runs the same path) */
        const int dev = ndev > 0 ? (first_device + g) % ndev : first_device + g;
        if (adb_ctx_init(g, dev) != ADB_OK) {
            set_err("adb_init(device %d): %s", dev, adb_last_error());
            S.failed = 1;
            adb_ctx_select(0);
            return -1;
        }
    }
    adb_ctx_select(0);
    if (gpus > 1 && adb_peer_connect_local(gpus) != ADB_OK) {
        set_err("adb_peer_connect_local(%d): %s", gpus, adb_last_error());
        S.failed = 1;
        return -1;
    }
    S.G = gpus;
    for (int g = 0; g < gpus; ++g) {
        void *p = NULL, *q = NULL;
        on_ctx(g);
        if (adb_alloc(&p, sizeof(adb_agg)) != ADB_OK || adb_alloc(&q, sizeof(adb_agg)) != ADB_OK) {
            set_err("adb_alloc: %s", adb_last_error());
            on_ctx(0);
            return -1;
        }
        S.d_part[g] = p;
        S.d_out[g] = q;
    }
    on_ctx(0);
    const char *m = getenv("ADB_SHIM_MIRROR");
    S.mirror = m && m[0] && m[0] != '0';
    /* Result payloads are plain malloc blocks of 4 * num_tuples bytes that nobody writes
     * (the plumbing only frees them): above glibc's mmap threshold every handle costs an
     * mmap + munmap pair (~10 us for a 20 MB list).  Serve them from the heap instead (up to 32 MB) and
     * keep the freed space.  ADB_SHIM_NO_MALLOPT=1 leaves the process's malloc policy alone. */
    const char *nm = getenv("ADB_SHIM_NO_MALLOPT");
    if (!(nm && nm[0] && nm[0] != '0')) {
        /* no mmap'd blocks at all: a 20 M-tuple handle's 80 MB payload would otherwise cost an
         * mmap + munmap pair per operator (the threshold cannot be raised past 32 MB) */
        mallopt(M_MMAP_MAX, 0);
        mallopt(M_TRIM_THRESHOLD, -1);               /* never give heap back */
        mallopt(M_TOP_PAD, 256 << 20);
    }
    const char *pf = getenv("ADB_SHIM_PROFILE");
    PF.on = pf && pf[0] && pf[0] != '0';
    const char *eager = getenv("ADB_SHIM_EAGER");
    S.lazy = !S.mirror && !(eager && eager[0] && eager[0] != '0');
    const char *mn = getenv("ADB_SHARD_MIN_ROWS");
    S.shard_min_rows = mn ? (size_t)atol(mn) : 32;
    if (S.shard_min_rows < 1) S.shard_min_rows = 1;
    const char *nr = getenv("ADB_SHIM_NO_REGISTER");
    S.register_uploads = !(nr && nr[0] && nr[0] != '0');
    const char *rb = getenv("ADB_REBALANCE_MIN");
    S.rebalance_min = rb ? (size_t)atol(rb) : ((size_t)1 << 20);   /* shorter lists: the re-cut costs more than it saves */
    const char *ties = getenv("ADB_INDEX_TIES");
    S.ref_ties = ties && strcmp(ties, "reference") == 0;          /* default: stable */
    if (workers_start()) return -1;
    S.up = 1;
    S.failed = 0;
    return 0;
}

int adb_host_init(int device) { return host_init(device, 1); }
int adb_host_init_multi(int gpus) {
    const char *d = getenv("ADB_DEVICE");
    return host_init(d ? atoi(d) : 0, gpus);
}

static int ensure_up(void) {
    if (S.up) return 0;
    const char *d = getenv("ADB_DEVICE");
    const char *n = getenv("ADB_GPUS");
    return host_init(d ? atoi(d) : 0, n && atoi(n) > 0 ? atoi(n) : 1);
}

static void dev_index_drop(DevColumn *c) {
    for (int g = 0; g < S.G; ++g) {
        if (!c->ix[g] && !c->d_ix_values[g] && !c->d_ix_positions[g]) continue;
        on_ctx(g);
        if (c->ix[g]) adb_index_destroy(c->ix[g]);
        if (c->d_ix_values[g]) adb_free(c->d_ix_values[g]);
        if (c->d_ix_positions[g]) adb_free(c->d_ix_positions[g]);
        c->ix[g] = NULL;
        c->d_ix_values[g] = c->d_ix_positions[g] = NULL;
    }
    on_ctx(0);
    c->host_ix_values = NULL;
    c->ix_rows = 0;
}

/* kernels of any context may still be reading a buffer that is about to go back to its pool
 * (peer gathers read other contexts' column shards) */
static void sync_all(void) {
    if (S.G == 1) return;
    for (int g = 0; g < S.G; ++g) {
        on_ctx(g);
        adb_sync();
    }
    on_ctx(0);
}

static void dev_column_drop(DevColumn *c) {
    if (c->d_data[0] || c->ix[0]) sync_all();
    if (P.active || nR) lazy_column_gone(c->d_data);
    dev_index_drop(c);
    if (!c->adopted)
        for (int g = 0; g < S.G; ++g) free_on(g, c->d_data[g]);
    const Column *key = c->key;
    const int *from = c->uploaded_from;             /* the upload history survives an invalidation */
    const size_t fbytes = c->uploaded_bytes;
    const int uploads = c->uploads, registered = c->registered;
    memset(c, 0, sizeof *c);
    c->key = key;
    c->uploaded_from = from;
    c->uploaded_bytes = fbytes;
    c->uploads = uploads;
    c->registered = registered;
}

static void column_unregister(DevColumn *c) {
    if (c->registered) adb_host_unregister((void *)c->uploaded_from);
    c->registered = 0;
    c->uploads = 0;
    c->uploaded_from = NULL;
    c->uploaded_bytes = 0;
}

/* give back `refs` references to a slab; the last one frees it */
static void slab_drop(Slab *slab, long refs) {
    slab->refs -= refs;
    if (slab->refs == 0) {
        for (int g = 0; g < S.G; ++g) free_on(g, slab->base[g]);
        free(slab);
    }
}

/* release what the list owns (stream-ordered: safe right after the last launch that reads it) */
static void list_release(ShardList *l) {
    if (!l->borrowed) {
        if (l->slab) slab_drop(l->slab, 1);
        else free_shards(l->d);
    }
    memset(l, 0, sizeof *l);
}

static void load_release(void);
void adb_host_shutdown(void) {
    if (!S.up) return;
    adb_host_profile_dump();
    load_release();
    lock();
    if (P.active) lazy_done(&P);
    while (nR) lazy_done(&R[nR - 1]);
    free(R);
    R = NULL;
    capR = 0;
    for (size_t i = 0; i < S.nslots; ++i)
        if (S.slots[i].payload != SLOT_EMPTY && S.slots[i].payload != SLOT_TOMB)
            list_release(&S.slots[i].list);
    DevResult *old = S.slots;
    S.slots = NULL;
    S.nslots = S.nused = 0;
    S.nlive = 0;
    for (int i = 0; i < S.ncols; ++i) {
        dev_column_drop(&S.cols[i]);
        column_unregister(&S.cols[i]);
    }
    DevColumn *oldc = S.cols;
    S.cols = NULL;
    S.ncols = S.capcols = 0;
    for (int g = 0; g < S.G; ++g) {
        free_on(g, S.d_part[g]);
        free_on(g, S.d_out[g]);
        S.d_part[g] = S.d_out[g] = NULL;
    }
    workers_stop();
    jx_cap_now = 0;
    S.up = 0;
    unlock();
    free(old);
    free(oldc);
    adb_shutdown();
    S.G = 0;
}

/* ---- base columns ----------------------------------------------------------------------- */
static DevColumn *dev_column_slot(Column *column) {
    if (!column) {
        set_err("NULL column");
        return NULL;
    }
    if (column->row_count >= ((size_t)1 << 31)) {
        set_err("column of %zu rows: positions are int (src/query.c:94-95), shard it below 2^31",
                column->row_count);
        return NULL;
    }
    DevColumn *c = NULL;
    for (int i = 0; i < S.ncols; ++i)
        if (S.cols[i].key == column) c = &S.cols[i];
    if (!c) {
        if (S.ncols == S.capcols) {
            int cap = S.capcols ? 2 * S.capcols : 16;
            DevColumn *n = realloc(S.cols, (size_t)cap * sizeof *n);
            if (!n) {
                set_err("out of host memory");
                return NULL;
            }
            S.cols = n;
            S.capcols = cap;
        }
        c = &S.cols[S.ncols++];
        memset(c, 0, sizeof *c);
        c->key = column;
    }
    return c;
}

/* rows per shard: an even split, rounded up to 32 rows so that every shard but the last is a
 * whole number of bitmap words; never below ADB_SHARD_MIN_ROWS */
static size_t shard_rows_for(size_t rows) {
    size_t s = (rows + (size_t)S.G - 1) / (size_t)S.G;
    if (s < S.shard_min_rows) s = S.shard_min_rows;
    s = (s + 31) & ~(size_t)31;
    return s ? s : 32;
}

typedef struct UploadJob {
    ShardErr err;
    DevColumn *c;
    const int *host;
} UploadJob;
static void upload_shard(int g, void *arg) {
    UploadJob *a = arg;
    DevColumn *c = a->c;
    const size_t n = shard_len(c->rows, c->shard_rows, g);
    void *p = NULL;
    SCK(adb_alloc(&p, 4 * n));
    c->d_data[g] = p;
    if (n) SCK(adb_upload(p, a->host + (size_t)g * c->shard_rows, 4 * n));
}

static DevColumn *dev_column(Column *column) {
    DevColumn *c = dev_column_slot(column);
    if (!c) return NULL;
    if (c->d_data[0] && c->host_data == column->data && c->rows == column->row_count) return c;
    dev_column_drop(c);
    c->rows = column->row_count;
    c->shard_rows = shard_rows_for(c->rows);
    /* the same large array again (the column was invalidated, not re-mapped): page-lock it once,
     * this and every later upload is then a single DMA per GPU at the link's rate */
    if (c->uploaded_from != column->data || c->uploaded_bytes != 4 * column->row_count) {
        column_unregister(c);
        c->uploaded_from = column->data;
        c->uploaded_bytes = 4 * column->row_count;
    }
    if (++c->uploads == 2 && !c->registered && c->uploaded_bytes >= REGISTER_MIN_BYTES && S.register_uploads)
        c->registered = adb_host_register((void *)column->data, c->uploaded_bytes) == ADB_OK;
    UploadJob job;
    memset(&job, 0, sizeof job);
    job.c = c;
    job.host = column->data;
    run_shards(upload_shard, &job);
    if (shard_errs(&job.err)) {
        for (int g = 0; g < S.G; ++g) free_on(g, c->d_data[g]);
        memset(c->d_data, 0, sizeof c->d_data);
        return NULL;
    }
    c->host_data = column->data;
    return c;
}

int adb_host_column_upload(Column *column) {
    if (ensure_up()) return -1;
    return dev_column(column) ? 0 : -1;
}

/* The column's rows are already in HBM (a GPU-side loader put them there: SURVEY.md 8f
 * rank 1).  The shim uses the buffers as they are until the column's data pointer or
 * row_count changes; they stay the caller's.  adb_host_column_adopt: one buffer on context 0
 * (G = 1).  adb_host_column_adopt_shards: d_shards[g] holds rows [g*shard_rows, (g+1)*shard_rows)
 * on context g; shard_rows must be a multiple of 32. */
int adb_host_column_adopt_shards(Column *column, const void *const *d_shards, size_t shard_rows) {
    if (ensure_up()) return -1;
    DevColumn *c = dev_column_slot(column);
    if (!c || !d_shards || shard_rows == 0 || (shard_rows & 31) ||
        shard_rows * (size_t)S.G < column->row_count) {
        set_err("adb_host_column_adopt_shards: %d shards of %zu rows cannot hold %zu rows (shard_rows must be "
                "a multiple of 32)", S.G, shard_rows, column ? column->row_count : 0);
        return -1;
    }
    dev_column_drop(c);
    for (int g = 0; g < S.G; ++g) c->d_data[g] = (int32_t *)d_shards[g];
    c->adopted = 1;
    c->host_data = column->data;
    c->rows = column->row_count;
    c->shard_rows = shard_rows;
    return 0;
}
int adb_host_column_adopt(Column *column, const void *d_data) {
    if (ensure_up()) return -1;
    if (S.G != 1 || !column) {
        set_err("adb_host_column_adopt: one buffer per GPU is needed with %d GPUs (adb_host_column_adopt_shards)", S.G);
        return -1;
    }
    const void *one[1] = {d_data};
    if (!d_data) return -1;
    size_t sr = (column->row_count + 31) & ~(size_t)31;
    return adb_host_column_adopt_shards(column, one, sr ? sr : 32);
}

void adb_host_column_invalidate(Column *column) {
    for (int i = 0; i < S.ncols; ++i)
        if (S.cols[i].key == column) dev_column_drop(&S.cols[i]);
}

/* Upload the ColumnIndex the reference built (src/index.c:89-101,119-146), cut into G slices
 * by index order.  Its positions are size_t on the host and are truncated to int when emitted
 * (src/query.c:187), so the device copy is int32 (narrowed on the device). */
typedef struct IndexJob {
    ShardErr err;
    DevColumn *c;
    Column *column;
} IndexJob;
static void index_shard(int g, void *arg) {
    IndexJob *a = arg;
    DevColumn *c = a->c;
    const size_t b = c->ix_begin[g], n = c->ix_begin[g + 1] - b;
    void *dv = NULL, *dp = NULL, *d64 = NULL;
    SCK(adb_alloc(&dv, 4 * n));
    c->d_ix_values[g] = dv;
    SCK(adb_alloc(&dp, 4 * n));
    c->d_ix_positions[g] = dp;
    if (n) {
        SCK(adb_upload(dv, a->column->index->values + b, 4 * n));
        SCK(adb_alloc(&d64, 8 * n));
        if (adb_upload(d64, a->column->index->positions + b, 8 * n) != ADB_OK ||
            adb_narrow_u64_to_i32(d64, (int64_t)n, dp) != ADB_OK) {
            shard_fail(&a->err, g, "index upload");
            adb_free(d64);
            return;
        }
        adb_free(d64);
    }
    SCK(adb_index_create(dv, dp, (int64_t)n, /*with_btree=*/!a->column->sorted, &c->ix[g]));
    if (S.G > 1) SCK(adb_index_set_slice(c->ix[g], 1));
}

static int slice_bounds(DevColumn *c, const int *v, size_t n);
static int dev_index(DevColumn *c, Column *column) {
    if (!column->index || !column->index->values || !column->index->positions) {
        set_err("column '%s' is flagged clustered/has_index but carries no ColumnIndex", column->name);
        return -1;
    }
    if (c->ix[0] && c->host_ix_values == column->index->values && c->ix_rows == column->row_count) return 0;
    dev_index_drop(c);
    const size_t n = column->row_count;
    const int *v = column->index->values;
    slice_bounds(c, v, n);
    IndexJob job;
    memset(&job, 0, sizeof job);
    job.c = c;
    job.column = column;
    run_shards(index_shard, &job);
    if (shard_errs(&job.err)) {
        dev_index_drop(c);
        return -1;
    }
    c->host_ix_values = column->index->values;
    c->ix_rows = n;
    return 0;
}

/* ---- index build on the engine (src/index.c:25-178) --------------------------------------------
 * build_unclustered_index: (values ascending, positions) of the column; build_clustered_index:
 * the same sort on a COPY, every other column of the table permuted into that order, the
 * indexed column's own data and its index->positions (identity) left untouched (SURVEY.md A2).
 * Here the sort is the engine's stable LSD radix sort (adb_index_sort): ties come out in
 * ascending row order where the reference's unstable quicksort leaves another order
 * (SURVEY.md A3) -- identical whenever the keys are unique.  With ADB_INDEX_TIES=reference the
 * sort is adb_index_sort_ref_ties instead: the quicksort's own tie order, so the index, the
 * clustered siblings' layout and every rebuild after an update or delete equal the reference's.
 * Equal keys never straddle two slices, so either order survives the cut by index order.  The host arrays the catalog owns
 * (ColumnIndex.values / .positions, the siblings' data) are filled from the device, because the
 * unchanged plumbing persists them at shutdown (src/db_manager.c:396-397); the device-side
 * index slices are installed directly, so the first select re-uploads nothing.
 *
 * cols[0 .. n_cols) are the table's columns in declaration order, `which` the indexed one
 * (its sorted / clustered flags say what to build).  With one GPU, or with ADB_INDEX_TIES=reference
 * (the quicksort's tie order depends on the whole array), the sort runs on context 0 and the slices
 * are copied out to the contexts that hold them.  With G > 1 and the stable order every context
 * sorts its own slice (sharded_build_sort below): the keys are routed to the slice that will hold
 * them first.  The sibling permutation is one peer gather per GPU either way. */
static int slice_bounds(DevColumn *c, const int *v, size_t n) {
    const size_t per = (n + (size_t)S.G - 1) / (size_t)S.G;
    c->ix_begin[0] = 0;
    for (int g = 1; g <= S.G; ++g) {
        size_t b = (size_t)g * per;
        if (b >= n || g == S.G) {
            b = n;
        } else {
            if (b < c->ix_begin[g - 1]) b = c->ix_begin[g - 1];
            if (b > 0 && b < n && v[b] == v[b - 1]) {       /* upper bound of the run of v[b-1] */
                size_t lo = b, hi = n;
                const int key = v[b - 1];
                while (lo < hi) {
                    const size_t mid = lo + (hi - lo) / 2;
                    if (v[mid] <= key) lo = mid + 1; else hi = mid;
                }
                b = lo;
            }
        }
        c->ix_begin[g] = b;
    }
    c->ix_min = n ? v[0] : 0;
    return 0;
}

typedef struct PermuteJob {
    ShardErr err;
    DevColumn *sib;
    int32_t *const *order;      /* entries [begin[d], begin[d+1]) of the sorted positions, on context d */
    const size_t *begin;
    int *host_out;
    int32_t *fresh[MAXG];
} PermuteJob;
static void permute_shard(int g, void *arg) {
    PermuteJob *a = arg;
    DevColumn *c = a->sib;
    const size_t n = shard_len(c->rows, c->shard_rows, g);
    void *ord = NULL, *out = NULL;
    SCK(adb_alloc(&out, 4 * n));
    a->fresh[g] = out;
    if (!n) return;
    SCK(adb_alloc(&ord, 4 * n));
    /* rows [lo, hi) of index order, from every slice that covers them */
    const size_t lo = (size_t)g * c->shard_rows, hi = lo + n;
    adb_status st = ADB_OK;
    for (int d = 0; d < S.G && st == ADB_OK; ++d) {
        const size_t a0 = lo > a->begin[d] ? lo : a->begin[d], a1 = hi < a->begin[d + 1] ? hi : a->begin[d + 1];
        if (a0 < a1)
            st = adb_copy_from_ctx((int32_t *)ord + (a0 - lo), d, a->order[d] + (a0 - a->begin[d]), 4 * (a1 - a0));
    }
    if (st != ADB_OK ||
        (S.G == 1 ? adb_fetch(c->d_data[0], ord, (int64_t)n, NULL, 0, out)
                  : adb_fetch_sharded((const int32_t *const *)c->d_data, S.G, (int64_t)c->shard_rows, ord,
                                      (int64_t)n, NULL, out)) != ADB_OK ||
        adb_download(a->host_out + (size_t)g * c->shard_rows, out, 4 * n) != ADB_OK)
        shard_fail(&a->err, g, "clustered index: sibling permutation");
    adb_free(ord);
}

typedef struct SliceJob {
    ShardErr err;
    DevColumn *c;
    const int32_t *vals0, *poss0;       /* on context 0; poss0 NULL = identity */
    int with_btree;
} SliceJob;
static void slice_shard(int g, void *arg) {
    SliceJob *a = arg;
    DevColumn *c = a->c;
    const size_t b = c->ix_begin[g], n = c->ix_begin[g + 1] - b;
    void *dv = NULL, *dp = NULL;
    SCK(adb_alloc(&dv, 4 * n));
    c->d_ix_values[g] = dv;
    SCK(adb_alloc(&dp, 4 * n));
    c->d_ix_positions[g] = dp;
    SCK(adb_copy_from_ctx(dv, 0, a->vals0 + b, 4 * n));
    if (a->poss0) SCK(adb_copy_from_ctx(dp, 0, a->poss0 + b, 4 * n));
    else SCK(adb_iota_i32(dp, (int64_t)n, (int32_t)b));
    SCK(adb_index_create(dv, dp, (int64_t)n, a->with_btree, &c->ix[g]));
    if (S.G > 1) SCK(adb_index_set_slice(c->ix[g], 1));
    SCK(adb_sync());                    /* the sort buffers on context 0 are released next */
}

/* ---- index build on every context (G > 1, stable tie order) ------------------------------------
 * slice_bounds ends slice g after #{keys <= t_g}, t_g = the key of rank g*per - 1 in sorted order
 * (+inf when g*per >= n): a plain cut at g*per and a cut moved to the end of a run of equal keys
 * both land there, and t_g never decreases, so its clamp never fires.  A key k therefore belongs
 * to slice #{g : t_g < k}.  With the exact t_g (a radix select summed over the contexts) every
 * context routes its own rows to the slice that will hold them and each slice is sorted where it
 * lives: the same slices, entry for entry.  Each slice receives its pieces in source order, i.e.
 * in ascending row order, so the stable sort leaves equal keys in row order, as adb_index_sort of
 * the whole column does. */
typedef struct ShardedBuild {
    ShardErr err;
    int phase;
    DevColumn *c;
    ColumnIndex *ix;
    int clustered, with_btree;
    size_t begin[MAXG + 1];             /* slice d = entries [begin[d], begin[d+1]) */
    /* phase SB_SELECT: one radix-select round over every context's keys */
    uint32_t prefixes[MAXG];
    int n_prefixes, round;
    uint32_t hist[MAXG][MAXG * 256];    /* [context][prefix * 256 + digit] */
    /* phase SB_ROUTE: context g's keys and row numbers grouped by slice; sent[g][d] of them for d */
    int32_t split[MAXG];                /* t_1 .. t_{G-1} */
    int32_t *rk[MAXG], *rr[MAXG];
    int64_t sent[MAXG][MAXG];
    /* slice d: what it received (keys, then row numbers; afterwards the catalog staging), then its
     * sorted values and positions, which become the device index slice */
    int32_t *recv[MAXG], *vals[MAXG], *poss[MAXG];
    adb_index *handle[MAXG];
} ShardedBuild;
enum { SB_SELECT, SB_ROUTE, SB_RESERVE, SB_PULL, SB_SORT, SB_CATALOG, SB_FINISH };

static void sharded_build_shard(int g, void *arg) {
    ShardedBuild *a = arg;
    const size_t b = a->begin[g], m = a->begin[g + 1] - b;
    switch (a->phase) {
    case SB_SELECT: {
        const DevColumn *c = a->c;
        SCK(adb_rank_hist(c->d_data[g], (int64_t)shard_len(c->rows, c->shard_rows, g), a->prefixes, a->n_prefixes,
                          a->round, a->hist[g]));
        break;
    }
    case SB_ROUTE: {
        const DevColumn *c = a->c;
        const size_t len = shard_len(c->rows, c->shard_rows, g);
        void *k = NULL, *r = NULL;
        SCK(adb_alloc(&k, 4 * len));
        a->rk[g] = k;
        SCK(adb_alloc(&r, 4 * len));
        a->rr[g] = r;
        SCK(adb_route_range(c->d_data[g], (int64_t)len, (int64_t)g * (int64_t)c->shard_rows, a->split, S.G, a->rk[g],
                            a->rr[g], a->sent[g]));
        break;
    }
    case SB_RESERVE: {                  /* everything this slice needs, before any pull starts */
        void *p = NULL;
        SCK(adb_alloc(&p, 8 * m));
        a->recv[g] = p;
        SCK(adb_alloc(&p, 4 * m));
        a->vals[g] = p;
        SCK(adb_alloc(&p, 4 * m));
        a->poss[g] = p;
        break;
    }
    case SB_PULL:                       /* source order; starting at its own piece, as route_pull */
        for (int k = 0; k < S.G; ++k) {
            const int src = (g + k) % S.G;
            size_t at = 0, from = 0;
            for (int t = 0; t < src; ++t) at += (size_t)a->sent[t][g];
            for (int o = 0; o < g; ++o) from += (size_t)a->sent[src][o];
            const size_t cnt = (size_t)a->sent[src][g];
            if (!cnt) continue;
            SCK(adb_copy_from_ctx_ready(a->recv[g] + at, src, a->rk[src] + from, 4 * cnt));
            SCK(adb_copy_from_ctx_ready(a->recv[g] + m + at, src, a->rr[src] + from, 4 * cnt));
        }
        SCK(adb_sync());
        break;
    case SB_SORT:                       /* every pull has finished: the routed pieces can go */
        adb_free(a->rk[g]);
        adb_free(a->rr[g]);
        a->rk[g] = a->rr[g] = NULL;
        SCK(adb_index_sort_pairs(a->recv[g], a->recv[g] + m, (int64_t)m, a->vals[g], a->poss[g]));
        SCK(adb_sync());
        break;
    case SB_CATALOG:                    /* over every context's own host link at once */
        if (m) SCK(adb_download(a->ix->values + b, a->vals[g], 4 * m));
        if (m && !a->clustered) {
            SCK(adb_widen_i32_to_u64(a->poss[g], (int64_t)m, a->recv[g]));
            SCK(adb_download(a->ix->positions + b, a->recv[g], 8 * m));
        }
        SCK(adb_sync());
        break;
    case SB_FINISH:                     /* a clustered index's positions are the identity */
        if (a->clustered) {
            SCK(adb_iota_i32(a->poss[g], (int64_t)m, (int32_t)b));
            if (m) {
                SCK(adb_widen_i32_to_u64(a->poss[g], (int64_t)m, a->recv[g]));
                SCK(adb_download(a->ix->positions + b, a->recv[g], 8 * m));
            }
        }
        SCK(adb_index_create(a->vals[g], a->poss[g], (int64_t)m, a->with_btree, &a->handle[g]));
        SCK(adb_index_set_slice(a->handle[g], 1));
        adb_free(a->recv[g]);
        a->recv[g] = NULL;
        break;
    }
}

static int sharded_build_run(ShardedBuild *a, int phase) {
    static const int pf[] = {PF_IX_SPLIT, PF_IX_ROUTE, PF_IX_RESERVE, PF_IX_PULL, PF_IX_SORT, PF_IX_CATALOG, PF_IX_SLICES};
    const double t0 = PF.on ? pf_now() : 0.0;
    a->phase = phase;
    run_shards(sharded_build_shard, a);
    if (PF.on) {
        PF.t[pf[phase]] += pf_now() - t0;
        ++PF.n[pf[phase]];
    }
    return shard_errs(&a->err);
}

/* what a failed build leaves behind */
static void sharded_build_free(ShardedBuild *a) {
    for (int g = 0; g < S.G; ++g) {
        on_ctx(g);
        if (a->handle[g]) adb_index_destroy(a->handle[g]);
        int32_t *bufs[5] = {a->rk[g], a->rr[g], a->recv[g], a->vals[g], a->poss[g]};
        for (int i = 0; i < 5; ++i)
            if (bufs[i]) adb_free(bufs[i]);
    }
    on_ctx(0);
}

/* t_1 .. t_{G-1} (INT32_MAX past the end) and the smallest key by a radix select of their ranks
 * over all contexts: four rounds of 8 bits of the sign-flipped key, histograms summed here. */
static int sharded_build_splitters(ShardedBuild *a, size_t n, int *min_key) {
    const size_t per = (n + (size_t)S.G - 1) / (size_t)S.G;
    size_t rank[MAXG];                  /* target 0: rank 0 (the minimum); target i: t_slice[i] */
    int slice[MAXG], nt = 0;
    if (n) {
        rank[nt] = 0;
        slice[nt++] = 0;
    }
    for (int g = 1; g < S.G; ++g) {
        a->split[g - 1] = INT32_MAX;
        if ((size_t)g * per < n) {
            rank[nt] = (size_t)g * per - 1;
            slice[nt++] = g;
        }
    }
    uint32_t prefix[MAXG] = {0};        /* the targets' high bits found so far, in increasing order */
    for (int round = 0; round < 4 && nt; ++round) {
        int which[MAXG];                /* target -> its prefix's row of the histogram */
        a->n_prefixes = 0;
        for (int t = 0; t < nt; ++t) {
            if (!a->n_prefixes || a->prefixes[a->n_prefixes - 1] != prefix[t]) a->prefixes[a->n_prefixes++] = prefix[t];
            which[t] = a->n_prefixes - 1;
        }
        a->round = round;
        if (sharded_build_run(a, SB_SELECT)) return -1;
        for (int t = 0; t < nt; ++t) {
            size_t left = rank[t];
            int d = 0;
            for (;; ++d) {
                size_t cnt = 0;
                for (int g = 0; g < S.G; ++g) cnt += a->hist[g][which[t] * 256 + d];
                if (left < cnt || d == 255) break;
                left -= cnt;
            }
            rank[t] = left;
            prefix[t] = prefix[t] << 8 | (uint32_t)d;
        }
    }
    for (int t = 0; t < nt; ++t) {
        const int32_t key = (int32_t)(prefix[t] ^ 0x80000000u);
        if (slice[t]) a->split[slice[t] - 1] = key;
        else *min_key = key;
    }
    return 0;
}

/* Sorts the column into its slices on the contexts that hold them and fills the catalog's arrays;
 * a clustered index's positions are filled by SB_FINISH, after the siblings have been permuted. */
static int sharded_build_sort(ShardedBuild *a, size_t n, int *min_key) {
    *min_key = 0;
    if (sharded_build_splitters(a, n, min_key) || sharded_build_run(a, SB_ROUTE)) return -1;
    a->begin[0] = 0;
    for (int d = 0; d < S.G; ++d) {
        a->begin[d + 1] = a->begin[d];
        for (int src = 0; src < S.G; ++src) a->begin[d + 1] += (size_t)a->sent[src][d];
    }
    if (a->begin[S.G] != n) {
        set_err("index build: the slices hold %zu of %zu rows", a->begin[S.G], n);
        return -1;
    }
    return sharded_build_run(a, SB_RESERVE) || sharded_build_run(a, SB_PULL) || sharded_build_run(a, SB_SORT) ||
                   sharded_build_run(a, SB_CATALOG) ? -1 : 0;
}

int adb_host_index_build(Column **cols, int n_cols, int which) {
    t_err[0] = '\0';
    if (ensure_up()) return -1;
    if (!cols || which < 0 || which >= n_cols || !cols[which]) {
        set_err("adb_host_index_build: bad arguments");
        return -1;
    }
    Column *column = cols[which];
    const size_t n = column->row_count;
    DevColumn *c = dev_column(column);
    if (!c) return -1;
    int rc = -1;
    int32_t *all = NULL, *vals = NULL, *poss = NULL;
    void *wide = NULL;
    ColumnIndex *ix = NULL;
    ShardedBuild *sb = NULL;
    int own_all = 0, min_key = 0;
    /* where the sorted positions are: slice d of them on context d */
    int32_t *order[MAXG] = {0};
    size_t order_begin[MAXG + 1];
    /* the catalog's host copy (plain malloc: release_index frees it, db_manager.c:614-626) */
    ix = malloc(sizeof *ix);
    if (ix) {
        ix->values = malloc(n ? n * sizeof(int) : 1);
        ix->positions = malloc(n ? n * sizeof(size_t) : 1);
    }
    if (!ix || !ix->values || !ix->positions) {
        set_err("out of host memory for the index of %zu rows", n);
        goto fail;
    }
    if (S.G > 1 && !S.ref_ties) {
        sb = calloc(1, sizeof *sb);
        if (!sb) {
            set_err("out of host memory for the index build");
            goto fail;
        }
        sb->c = c;
        sb->ix = ix;
        sb->clustered = column->clustered;
        sb->with_btree = !column->sorted;
        if (sharded_build_sort(sb, n, &min_key)) goto fail;
        for (int d = 0; d < S.G; ++d) order[d] = sb->poss[d];
        memcpy(order_begin, sb->begin, sizeof order_begin);
    } else {
        PF_BEGIN(PF_IX_GLOBAL);
        /* the whole column on context 0 */
        if (S.G == 1) {
            all = c->d_data[0];
        } else {
            void *p = NULL;
            if (adb_alloc(&p, 4 * n) != ADB_OK) goto dev_fail;
            all = p;
            own_all = 1;
            for (int g = 0; g < S.G; ++g) {
                const size_t len = shard_len(c->rows, c->shard_rows, g);
                if (len && adb_copy_from_ctx(all + (size_t)g * c->shard_rows, g, c->d_data[g], 4 * len) != ADB_OK)
                    goto dev_fail;
            }
        }
        {
            void *p = NULL, *q = NULL;
            if (adb_alloc(&p, 4 * n) != ADB_OK || adb_alloc(&q, 4 * n) != ADB_OK) {
                if (p) adb_free(p);
                goto dev_fail;
            }
            vals = p;
            poss = q;
        }
        if ((S.ref_ties ? adb_index_sort_ref_ties : adb_index_sort)(all, (int64_t)n, vals, poss) != ADB_OK) goto dev_fail;
        if (n) {
            if (adb_alloc(&wide, 8 * n) != ADB_OK) goto dev_fail;
            if (adb_download(ix->values, vals, 4 * n) != ADB_OK ||
                adb_widen_i32_to_u64(column->clustered ? NULL : poss, (int64_t)n, wide) != ADB_OK ||
                adb_download(ix->positions, wide, 8 * n) != ADB_OK)
                goto dev_fail;
            adb_free(wide);
            wide = NULL;
        }
        PF_END(PF_IX_GLOBAL);
        order[0] = poss;
        order_begin[0] = 0;
        for (int g = 1; g <= S.G; ++g) order_begin[g] = n;
    }
    PF_BEGIN(PF_IX_SIBLINGS);
    if (column->clustered) {
        /* every OTHER column (by name, index.c:128-133) moves into index order */
        for (int j = 0; j < n_cols; ++j) {
            Column *sib = cols[j];
            if (!sib || strcmp(sib->name, column->name) == 0) continue;
            if (sib->row_count != n) {
                set_err("clustered index: column '%s' has %zu rows, '%s' has %zu", sib->name, sib->row_count,
                        column->name, n);
                goto fail;
            }
            DevColumn *dc = dev_column(sib);
            c = dev_column_slot(column);            /* the registry may have moved */
            if (!dc || !c) goto fail;
            if (dc->adopted) {
                set_err("clustered index: column '%s' lives in caller-owned device memory", sib->name);
                goto fail;
            }
            PermuteJob job;
            memset(&job, 0, sizeof job);
            job.sib = dc;
            job.order = order;
            job.begin = order_begin;
            job.host_out = sib->data;               /* in place: the mmap is the catalog's truth */
            run_shards(permute_shard, &job);
            if (shard_errs(&job.err)) {
                for (int g = 0; g < S.G; ++g) free_on(g, job.fresh[g]);
                goto fail;
            }
            sync_all();                             /* every gather has read the old shards */
            if (P.active || nR) lazy_column_gone(dc->d_data);
            for (int g = 0; g < S.G; ++g) {
                free_on(g, dc->d_data[g]);
                dc->d_data[g] = job.fresh[g];
            }
        }
    }
    PF_END(PF_IX_SIBLINGS);
    /* device-side index slices, cut by index order */
    if (sb) {
        if (sharded_build_run(sb, SB_FINISH)) goto fail;
        dev_index_drop(c);
        memcpy(c->ix_begin, sb->begin, sizeof c->ix_begin);
        c->ix_min = min_key;
        for (int d = 0; d < S.G; ++d) {
            c->d_ix_values[d] = sb->vals[d];
            c->d_ix_positions[d] = sb->poss[d];
            c->ix[d] = sb->handle[d];
            sb->vals[d] = sb->poss[d] = NULL;
            sb->handle[d] = NULL;
        }
    } else {
        PF_BEGIN(PF_IX_SLICES);
        dev_index_drop(c);
        slice_bounds(c, ix->values, n);
        SliceJob job;
        memset(&job, 0, sizeof job);
        job.c = c;
        job.vals0 = vals;
        job.poss0 = column->clustered ? NULL : poss;
        job.with_btree = !column->sorted;
        run_shards(slice_shard, &job);
        PF_END(PF_IX_SLICES);
        if (shard_errs(&job.err)) {
            dev_index_drop(c);
            goto fail;
        }
    }
    column->index = ix;
    ix = NULL;
    c->host_ix_values = column->index->values;
    c->ix_rows = n;
    rc = 0;
    goto done;
dev_fail:
    set_err("index build: %s", adb_last_error());
fail:
    if (ix) {
        free(ix->values);
        free(ix->positions);
        free(ix);
    }
done:
    if (sb) {
        sharded_build_free(sb);
        free(sb);
    }
    if (wide) adb_free(wide);
    if (vals) adb_free(vals);
    if (poss) adb_free(poss);
    if (own_all && all) adb_free(all);
    return rc;
}

/* build_histogram (src/index.c:63-84) on the device: counts[b] for the 100 bins of width
 * (max - min) / 99 starting at column->min.  Returns -1 when the bin width is 0 (the reference
 * divides by it). */
int adb_host_column_histogram(Column *column, int bin_size, unsigned long counts[100]) {
    t_err[0] = '\0';
    if (ensure_up() || !column || !counts) return -1;
    if (bin_size <= 0) {
        set_err("histogram: bin width %d (the reference divides by it, index.c:77)", bin_size);
        return -1;
    }
    DevColumn *c = dev_column(column);
    if (!c) return -1;
    memset(counts, 0, 100 * sizeof counts[0]);
    for (int g = 0; g < S.G; ++g) {
        uint64_t part[100];
        const size_t len = shard_len(c->rows, c->shard_rows, g);
        on_ctx(g);
        if (adb_histogram_i32(c->d_data[g], (int64_t)len, column->min, bin_size, part) != ADB_OK) {
            set_err("histogram: %s", adb_last_error());
            on_ctx(0);
            return -1;
        }
        for (int b = 0; b < 100; ++b) counts[b] += part[b];
    }
    on_ctx(0);
    return 0;
}

/* ---- device-resident results ------------------------------------------------------------- */
/* Every payload block the shim hands out starts with a tag derived from its own address.  A
 * registry hit is only trusted when the tag is still there: if the plumbing freed the payload
 * behind the shim's back and malloc gave the address to somebody else (a foreign host Result),
 * that somebody has written its own bytes over the tag (ADVICE r1).  Not in mirror mode, where
 * the block holds the tuples themselves. */
#define PAYLOAD_MAGIC 0xADB200C5EEDULL
static uint64_t payload_tag(const void *payload) { return PAYLOAD_MAGIC ^ ((uint64_t)(uintptr_t)payload * 0x9E3779B97F4A7C15ULL); }
static void payload_stamp(void *payload) {
    if (!S.mirror) {
        ((uint64_t *)payload)[0] = payload_tag(payload);
        ((uint64_t *)payload)[1] = ~payload_tag(payload);
    }
}
static int payload_is_ours(const void *payload) {
    return S.mirror || (((const uint64_t *)payload)[0] == payload_tag(payload) &&
                        ((const uint64_t *)payload)[1] == ~payload_tag(payload));
}

static size_t slot_of(const void *p, size_t nslots) {
    uint64_t x = (uint64_t)(uintptr_t)p;
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 29;
    return (size_t)x & (nslots - 1);
}

static DevResult *registry_find(const void *payload) {
    if (!S.nslots || !payload) return NULL;
    for (size_t i = slot_of(payload, S.nslots);; i = (i + 1) & (S.nslots - 1)) {
        if (S.slots[i].payload == SLOT_EMPTY) return NULL;
        if (S.slots[i].payload == payload) return &S.slots[i];
    }
}

static int registry_grow(void) {
    const size_t n = S.nslots ? 2 * S.nslots : 256;
    DevResult *ns = calloc(n, sizeof *ns), *old = S.slots;
    if (!ns) return -1;
    size_t used = 0;
    for (size_t i = 0; i < S.nslots; ++i) {
        void *p = old[i].payload;
        if (p == SLOT_EMPTY || p == SLOT_TOMB) continue;
        size_t j = slot_of(p, n);
        while (ns[j].payload != SLOT_EMPTY) j = (j + 1) & (n - 1);
        ns[j] = old[i];
        ++used;
    }
    S.slots = ns;
    S.nslots = n;
    S.nused = used;
    free(old);
    return 0;
}

/* Detach the device buffers registered under `payload` (if any); returns 1 and fills *out. */
static int registry_take(const void *payload, ShardList *out) {
    int found = 0;
    lock();
    DevResult *r = registry_find(payload);
    if (r) {
        *out = r->list;
        memset(r, 0, sizeof *r);
        r->payload = SLOT_TOMB;
        --S.nlive;
        found = 1;
    }
    unlock();
    return found;
}

void adb_host_payload_freed(void *payload) {
    if (S.nlive <= 0 || !payload) return;
    /* With the free() interposer every free() of the process lands here, from any thread (the
     * CUDA runtime's included): only an address the registry knows goes any further -- the lazy
     * records below are the calling plumbing's (single-threaded) state. */
    lock();
    const int known = registry_find(payload) != NULL;
    unlock();
    if (!known) return;
    PF_BEGIN(PF_RELEASE);
    const int keep = pending_payload_gone(payload);
    ShardList dead;
    if (registry_take(payload, &dead) && !keep) list_release(&dead);
    PF_END(PF_RELEASE);
}

void adb_host_result_release(Result *result) {
    if (result) adb_host_payload_freed(result->payload);
}

/* What update_result / free_client_context do with a handle's old value (src/client_context.c:
 * 31-45,76-90) plus the release hook, for a batch of Results: release the device buffers, free
 * the payload, free the Result.  For hosts (and harnesses) that drop many handles at once. */
void adb_host_results_drop(Result **results, int n) {
    for (int i = 0; i < n; ++i) {
        Result *r = results ? results[i] : NULL;
        if (!r) continue;
        adb_host_payload_freed(r->payload);
        free(r->payload);
        free(r);
    }
}

static int download_shards(void *dst, const ShardList *l) {
    size_t off = 0;
    int rc = 0;
    for (int g = 0; g < S.G; ++g) {
        if (!l->n[g]) continue;
        on_ctx(g);
        if (adb_download((char *)dst + 4 * off, l->d[g], 4 * l->n[g]) != ADB_OK) {
            set_err("adb_download: %s", adb_last_error());
            rc = -1;
            break;
        }
        off += l->n[g];
    }
    on_ctx(0);
    return rc;
}

/* Register a list as a Result the plumbing can own; the result takes its buffers over and *l
 * still describes them afterwards (with total set).  On failure an owned list is released; a
 * slab view is not -- shared_select gives the slab's references back itself. */
static Result *new_dev_result_impl(ShardList *l);
static Result *new_dev_result(ShardList *l) {
    PF_BEGIN(PF_NEWRESULT);
    Result *r = new_dev_result_impl(l);
    PF_END(PF_NEWRESULT);
    return r;
}
static Result *new_dev_result_impl(ShardList *l) {
    l->total = 0;
    for (int g = 0; g < S.G; ++g) l->total += l->n[g];
    const size_t tuples = l->total;
    Result *r = malloc(sizeof *r);
    size_t bytes = 4 * tuples < 16 ? 16 : 4 * tuples;
    void *payload = malloc(bytes);
    if (!r || !payload) {
        set_err("out of host memory for a %zu-tuple result", tuples);
        goto fail;
    }
    if (S.mirror && tuples && download_shards(payload, l)) goto fail;
    /* malloc returned an address we still hold buffers for: that payload was freed by the
     * plumbing without telling us -- reclaim its HBM now.  No engine call is made with the
     * registry lock held (with the free() interposer other threads' frees wait on it). */
    const int keep_dead = pending_payload_gone(payload);    /* an unwritten fetch may keep the dead select's buffers */
    ShardList dead;
    int have_dead = 0;
    lock();
    DevResult *e = registry_find(payload);
    if (e) {
        dead = e->list;
        have_dead = 1;
    } else {
        if (4 * (S.nused + 1) > 3 * S.nslots && registry_grow()) {
            unlock();
            set_err("out of host memory");
            goto fail;
        }
        size_t j = slot_of(payload, S.nslots);
        while (S.slots[j].payload != SLOT_EMPTY && S.slots[j].payload != SLOT_TOMB)
            j = (j + 1) & (S.nslots - 1);
        if (S.slots[j].payload == SLOT_EMPTY) ++S.nused;
        e = &S.slots[j];
        ++S.nlive;
    }
    e->payload = payload;
    e->list = *l;
    unlock();
    if (have_dead && !keep_dead) list_release(&dead);
    payload_stamp(payload);
    r->num_tuples = tuples;
    r->data_type = INT;
    r->payload = payload;
    return r;
fail:
    free(r);
    free(payload);
    if (!l->slab) list_release(l);
    return NULL;
}

static void drop_result(Result *r) {
    if (!r) return;
    adb_host_result_release(r);
    free(r->payload);
    free(r);
}

/* Hand an operator's list out as its Result and set the Status. */
static Result *hand_out(ShardList *l, Status *st, const char *what) {
    Result *r = new_dev_result(l);
    if (!r) return op_fail(st, what);
    op_ok(st);
    return r;
}

/* The same for the two lists of a join (results[0], results[1]); on failure both are released. */
static Result **hand_out_pair(ShardList *l1, ShardList *l2, Status *st, const char *what) {
    Result **results = malloc(2 * sizeof *results);
    if (!results) {
        set_err("out of host memory");
        list_release(l1);
        list_release(l2);
        return op_fail(st, what);
    }
    results[0] = new_dev_result(l1);
    if (!results[0]) {
        list_release(l2);
        goto fail;
    }
    results[1] = new_dev_result(l2);
    if (!results[1]) {
        drop_result(results[0]);
        goto fail;
    }
    op_ok(st);
    return results;
fail:
    free(results);
    return op_fail(st, what);
}

/* The device buffers registered under r's payload, as a borrowed view cut to r->num_tuples.
 * Returns 1 and fills *v; 0 when the payload is no device result (a scalar or a host array
 * built by a test or by foreign code); -1 (t_err set) when the result cannot be read. */
static int result_view(const Result *r, ShardList *v) {
    if (resolve_payload(r->payload)) return -1; /* about to be read: write it if it is unwritten */
    lock();
    DevResult *e = registry_find(r->payload);
    if (e) *v = e->list;
    unlock();
    if (!e) return 0;
    if (!payload_is_ours(r->payload)) {
        /* the address was recycled: the registered device buffers belong to a dead handle */
        adb_host_payload_freed(r->payload);
        return 0;
    }
    if (v->total < r->num_tuples) {
        set_err("result claims %zu tuples but its device buffers hold %zu", r->num_tuples, v->total);
        return -1;
    }
    size_t left = r->num_tuples;                /* a caller shortened the list: drop the tail */
    for (int g = 0; g < S.G; ++g) {
        v->n[g] = v->n[g] < left ? v->n[g] : left;
        left -= v->n[g];
    }
    v->total = r->num_tuples;
    v->borrowed = 1;
    return 1;
}

static int same_split(const size_t a[], const size_t b[]) {
    for (int g = 0; g < S.G; ++g)
        if (a[g] != b[g]) return 0;
    return 1;
}

/* dst (context g, `want[g]` entries each) <- the list whose shards are src/have, re-cut */
static int recut(int32_t *const src[], const size_t have[], const size_t want[], int32_t *dst[]) {
    size_t src_begin[MAXG + 1];
    src_begin[0] = 0;
    for (int s = 0; s < S.G; ++s) src_begin[s + 1] = src_begin[s] + have[s];
    size_t dst_begin = 0;
    int rc = 0;
    for (int g = 0; g < S.G && !rc; ++g) {
        void *p = NULL;
        on_ctx(g);
        if (adb_alloc(&p, 4 * want[g]) != ADB_OK) {
            set_err("adb_alloc(%zu): %s", 4 * want[g], adb_last_error());
            rc = -1;
            break;
        }
        dst[g] = p;
        const size_t b = dst_begin, e = dst_begin + want[g];
        for (int s = 0; s < S.G; ++s) {
            const size_t lo = b > src_begin[s] ? b : src_begin[s];
            const size_t hi = e < src_begin[s + 1] ? e : src_begin[s + 1];
            if (lo >= hi) continue;
            if (adb_copy_from_ctx(dst[g] + (lo - b), s, src[s] + (lo - src_begin[s]), 4 * (hi - lo)) != ADB_OK) {
                set_err("adb_copy_from_ctx: %s", adb_last_error());
                rc = -1;
                break;
            }
        }
        dst_begin = e;
    }
    /* The copies run on each destination context's own stream -- the stream its consumer runs
     * on -- but the SOURCE buffers belong to other contexts' pools and may be released as soon as
     * the operator returns: wait for the copies here (a rare path: operands cut differently). */
    for (int g = 0; g < S.G; ++g) {
        on_ctx(g);
        if (adb_sync() != ADB_OK && !rc) {
            set_err("adb_sync: %s", adb_last_error());
            rc = -1;
        }
    }
    on_ctx(0);
    return rc;
}

/* An operator input: the device buffers behind a Result, released with list_release().  A
 * device result is borrowed; a host array (built by a test or by foreign code) is uploaded into
 * buffers the list owns.  `like` (optional): the split the operand must have -- a device result
 * cut differently is re-cut with peer copies, a host array is uploaded that way. */
static int stage(const Result *r, const size_t *like, ShardList *out) {
    memset(out, 0, sizeof *out);
    if (!r) {
        set_err("NULL result operand");
        return -1;
    }
    if (r->num_tuples >= ((size_t)1 << 31)) {
        set_err("result of %zu tuples exceeds the int position domain (src/query.c:40-43)", r->num_tuples);
        return -1;
    }
    ShardList v;
    const int found = result_view(r, &v);
    if (found < 0) return -1;
    out->total = r->num_tuples;
    if (found) {
        if (!like || same_split(v.n, like)) {
            *out = v;
            return 0;
        }
        memcpy(out->n, like, sizeof(size_t) * (size_t)S.G);
        if (recut(v.d, v.n, like, out->d)) {
            list_release(out);
            return -1;
        }
        return 0;
    }
    if (r->num_tuples && !r->payload) {
        set_err("result operand has no payload");
        return -1;
    }
    /* host array: upload, cut like the partner or evenly */
    const size_t per = (r->num_tuples + (size_t)S.G - 1) / (size_t)S.G;
    size_t off = 0;
    int rc = 0;
    for (int g = 0; g < S.G; ++g) {
        const size_t n = like ? like[g] : shard_len(r->num_tuples, per ? per : 1, g);
        void *p = NULL;
        on_ctx(g);
        if (adb_alloc(&p, 4 * n) != ADB_OK ||
            (n && adb_upload(p, (const char *)r->payload + 4 * off, 4 * n) != ADB_OK)) {
            set_err("operand upload: %s", adb_last_error());
            if (p) adb_free(p);
            rc = -1;
            break;
        }
        out->d[g] = p;
        out->n[g] = n;
        off += n;
    }
    on_ctx(0);
    if (rc) list_release(out);
    return rc;
}

int adb_host_result_to_host(const Result *result, void *dst) {
    if (!result) return -1;
    if (result->num_tuples == 0) return 0;
    ShardList v;
    const int found = result_view(result, &v);
    if (found) return found < 0 ? -1 : download_shards(dst, &v);
    /* scalar or foreign host payload */
    size_t w = result->data_type == INT || result->data_type == FLOAT ? 4 : 8;
    memcpy(dst, result->payload, w * result->num_tuples);
    return 0;
}

/* allocate n[g] ints on every context (each context's thread allocates its own) */
typedef struct AllocJob {
    ShardErr err;
    ShardList *l;
} AllocJob;
static void alloc_shard(int g, void *arg) {
    AllocJob *a = arg;
    void *p = NULL;
    if (a->l->d[g]) return;                         /* served from the cache already */
    SCK(adb_alloc(&p, 4 * a->l->n[g]));
    a->l->d[g] = p;
}
static int alloc_shards(ShardList *l) {
    AllocJob job;
    memset(&job, 0, sizeof job);
    job.l = l;
    int missing = 0;
    for (int g = 0; g < S.G; ++g) {
        void *p = NULL;
        l->d[g] = adb_alloc_cached_on(g, &p, 4 * l->n[g]) ? p : NULL;
        missing |= l->d[g] == NULL;
    }
    if (missing) run_shards(alloc_shard, &job);
    if (shard_errs(&job.err)) {
        list_release(l);
        return -1;
    }
    return 0;
}

/* ---- updates and deletes (SURVEY.md 8f rank 4) ------------------------------------------------
 * relational_update(col, positions, value) and relational_delete(tbl, positions) of milestone 5
 * (project_tests/data_generation_scripts/milestone5.py:123-262).  The reference's parser has no
 * branch for them (src/parse.c:876-960) and query.c no function, so these are hooks a parser
 * branch would call; the semantics are the generator's pandas model.  The host arrays
 * (Column.data, the catalog's truth: they are what shutdown persists) are brought up to date
 * from the device after every change.  Handles created before the change keep their values
 * (unwritten ones are written first).  Indexes: an unclustered index of a changed column (update)
 * or of any column of the table (delete) is rebuilt on the engine; a table with a CLUSTERED index
 * is refused -- the reference's clustered layout (SURVEY.md A2) has no defined update semantics. */
typedef struct UpdateJob {
    ShardErr err;
    DevColumn *c;
    int32_t *pos[MAXG];             /* the positions this context applies */
    size_t n[MAXG];
    int value;
    int *host;
} UpdateJob;
static void update_shard(int g, void *arg) {
    UpdateJob *a = arg;
    DevColumn *c = a->c;
    const size_t rows = shard_len(c->rows, c->shard_rows, g);
    if (!rows) return;
    SCK(adb_update_rows(c->d_data[g], (int64_t)rows, a->pos[g], (int64_t)a->n[g], shard_base(g, c->shard_rows), a->value));
    SCK(adb_download(a->host + (size_t)g * c->shard_rows, c->d_data[g], 4 * rows));
}

static int table_has_clustered(Column **cols, int n_cols) {
    for (int j = 0; j < n_cols; ++j)
        if (cols[j] && cols[j]->clustered) return 1;
    return 0;
}
static int rebuild_index(Column **cols, int n_cols, int j) {
    Column *col = cols[j];
    if (col->index) {                       /* plain mallocs of init_column_index / adb_host_index_build */
        free(col->index->values);
        free(col->index->positions);
        free(col->index);
        col->index = NULL;
    }
    return adb_host_index_build(cols, n_cols, j);
}

int adb_host_relational_update(Column **cols, int n_cols, int which, Result *positions, int value) {
    t_err[0] = '\0';
    if (ensure_up()) return -1;
    if (!cols || which < 0 || which >= n_cols || !cols[which] || !positions) {
        set_err("relational_update: bad arguments");
        return -1;
    }
    if (table_has_clustered(cols, n_cols)) {
        set_err("relational_update: the table has a clustered index (no defined update semantics, SURVEY.md A2)");
        return -1;
    }
    Column *column = cols[which];
    ShardList p;
    memset(&p, 0, sizeof p);
    int32_t *all[MAXG] = {0};
    int rc = -1;
    DevColumn *c = dev_column(column);
    if (!c || c->adopted || !column->data) {
        if (c) set_err("relational_update: column '%s' has no host array to keep up to date", column->name);
        return -1;
    }
    if (stage(positions, NULL, &p)) return -1;
    c = dev_column_slot(column);
    if (P.active || nR) lazy_column_gone(c->d_data);        /* handles that still have to read the old values */
    UpdateJob job;
    memset(&job, 0, sizeof job);
    job.c = c;
    job.value = value;
    job.host = column->data;
    if (S.G == 1 || (p.aligned && p.aligned == c->shard_rows)) {
        for (int g = 0; g < S.G; ++g) {
            job.pos[g] = p.d[g];
            job.n[g] = p.n[g];
        }
    } else {
        /* positions anywhere: every GPU gets the whole list and applies the rows it owns */
        size_t allto[MAXG];
        for (int g = 0; g < S.G; ++g) {
            memset(allto, 0, sizeof allto);
            allto[g] = p.total;
            int32_t *tmp[MAXG] = {0};
            if (recut(p.d, p.n, allto, tmp)) {
                for (int k = 0; k < S.G; ++k) free_on(k, tmp[k]);
                goto done;
            }
            all[g] = tmp[g];
            for (int k = 0; k < S.G; ++k)
                if (k != g) free_on(k, tmp[k]);
            job.pos[g] = all[g];
            job.n[g] = p.total;
        }
    }
    run_shards(update_shard, &job);
    if (shard_errs(&job.err)) goto done;
    if (value < column->min) column->min = value;           /* insert_row keeps these (db_manager.c:193-194) */
    if (value > column->max) column->max = value;
    rc = 0;
    if (column->has_index) rc = rebuild_index(cols, n_cols, which);
done:
    for (int g = 0; g < S.G; ++g) free_on(g, all[g]);
    list_release(&p);
    return rc;
}

int adb_host_relational_delete(Column **cols, int n_cols, Result *positions) {
    t_err[0] = '\0';
    if (ensure_up()) return -1;
    if (!cols || n_cols < 1 || !positions) {
        set_err("relational_delete: bad arguments");
        return -1;
    }
    if (table_has_clustered(cols, n_cols)) {
        set_err("relational_delete: the table has a clustered index (no defined delete semantics, SURVEY.md A2)");
        return -1;
    }
    const size_t rows = cols[0] ? cols[0]->row_count : 0;
    for (int j = 0; j < n_cols; ++j)
        if (!cols[j] || cols[j]->row_count != rows || !cols[j]->data) {
            set_err("relational_delete: the table's columns must be host-backed and equally long");
            return -1;
        }
    ShardList p;
    memset(&p, 0, sizeof p);
    size_t all0[MAXG] = {0};
    all0[0] = positions->num_tuples;
    if (stage(positions, all0, &p)) return -1;              /* the whole list on GPU 0 (a global compaction) */
    int rc = -1;
    int64_t left = -1;
    void *gathered = NULL, *out = NULL;
    if (adb_delete_rows_plan((int64_t)rows, p.d[0], (int64_t)p.total, 0, &left) != ADB_OK) {
        set_err("relational_delete: %s", adb_last_error());
        goto done;
    }
    if (adb_alloc(&out, 4 * (size_t)(left > 0 ? left : 1)) != ADB_OK ||
        (S.G > 1 && adb_alloc(&gathered, 4 * (rows ? rows : 1)) != ADB_OK)) {
        set_err("relational_delete: %s", adb_last_error());
        goto done;
    }
    for (int j = 0; j < n_cols; ++j) {
        DevColumn *c = dev_column(cols[j]);
        if (!c) goto done;
        if (P.active || nR) lazy_column_gone(c->d_data);    /* handles that still have to read the old rows */
        const int32_t *src = c->d_data[0];
        if (S.G > 1) {
            for (int g = 0; g < S.G; ++g) {
                const size_t len = shard_len(c->rows, c->shard_rows, g);
                if (len && adb_copy_from_ctx((int32_t *)gathered + (size_t)g * c->shard_rows, g, c->d_data[g], 4 * len) != ADB_OK) {
                    set_err("relational_delete: %s", adb_last_error());
                    goto done;
                }
            }
            src = gathered;
        }
        if (adb_delete_rows_apply(src, out) != ADB_OK ||
            (left > 0 && adb_download(cols[j]->data, out, 4 * (size_t)left) != ADB_OK)) {
            set_err("relational_delete: %s", adb_last_error());
            goto done;
        }
    }
    for (int j = 0; j < n_cols; ++j) {
        adb_host_column_invalidate(cols[j]);                /* re-sharded at the next touch */
        cols[j]->row_count = (size_t)left;
    }
    rc = 0;
    for (int j = 0; j < n_cols && rc == 0; ++j)
        if (cols[j]->has_index) rc = rebuild_index(cols, n_cols, j);
done:
    if (out) adb_free(out);
    if (gathered) adb_free(gathered);
    list_release(&p);
    return rc;
}

/* ---- bulk load (SURVEY.md 8f rank 1): CSV text -> row-sharded device columns ---------------------
 * What load_db's ingest loop does (src/db_manager.c:304-318), with every GPU parsing a piece of the
 * file that came over its own host link.  Two phases, because the catalog grows its mmap'd columns
 * between them:
 *   count  the text after `skip_lines` lines is cut into G pieces: piece g > 0 starts right after
 *          the first '\n' at or after byte g*len/G (pieces may be empty; no line spans two).  Every
 *          GPU uploads, indexes and parses its piece (adb_csv_parse_piece); the host resolves the
 *          carry chain (a missing field takes the value of the nearest earlier row of the FILE that
 *          had it); pieces with short rows are filled; then the pieces are re-cut into shards of
 *          shard_rows_for(rows) rows and every shard's min / max is taken.
 *   emit   every GPU downloads its shard into Column.data + old_rows + g*S; min / max are folded as
 *          insert_row folds them (db_manager.c:193-194) and row_count is set.  Into an empty table
 *          the shards become the columns' device copies, so the next operator uploads nothing. */
typedef struct Load {
    int pending, n_cols;
    size_t rows, shard_rows;                        /* rows of the text; S of the new shards */
    int32_t **d[MAXG];                              /* d[g][c]: shard g of column c (context g) */
    int mn[256], mx[256];                           /* the new rows' min / max per column */
} Load;
static Load L;

typedef struct LoadJob {
    ShardErr err;
    int step, n_cols;
    const char *text;
    size_t begin[MAXG + 1];                         /* piece g = text[begin[g], begin[g+1]) */
    void *d_text[MAXG];
    int32_t **piece[MAXG];                          /* piece[g][c], rows[g] ints */
    size_t rows[MAXG];
    int32_t last[MAXG][256], has[MAXG][256], carry[MAXG][256];
    int32_t shorts[MAXG];
    adb_agg agg[MAXG][256];
} LoadJob;

static void load_shard(int g, void *arg) {
    LoadJob *a = arg;
    const size_t bytes = a->begin[g + 1] - a->begin[g];
    switch (a->step) {
    case 0: {                                       /* this GPU's piece over its own link */
        void *p = NULL;
        SCK(adb_alloc(&p, bytes ? bytes : 16));
        a->d_text[g] = p;
        if (bytes) SCK(adb_upload(p, a->text + a->begin[g], bytes));
        break;
    }
    case 1: {                                       /* index + parse, without the fill */
        int64_t rows = 0;
        SCK(adb_csv_index(a->d_text[g], bytes, 0, &rows));
        a->rows[g] = (size_t)rows;
        for (int c = 0; c < a->n_cols; ++c) {
            void *p = NULL;
            SCK(adb_alloc(&p, 4 * (rows ? (size_t)rows : 1)));
            a->piece[g][c] = p;
        }
        SCK(adb_csv_parse_piece(a->n_cols, a->piece[g], a->last[g], a->has[g], &a->shorts[g]));
        SCK(adb_free(a->d_text[g]));
        a->d_text[g] = NULL;
        break;
    }
    case 2:                                         /* enqueued only: the re-cut's copies wait for it */
        if (a->shorts[g]) SCK(adb_csv_fill(a->carry[g]));
        break;
    case 3: {                                       /* min / max of the new shards */
        const size_t n = shard_len(L.rows, L.shard_rows, g);
        for (int c = 0; c < a->n_cols && n; ++c)
            SCK(adb_aggregate(L.d[g][c], (int64_t)n, NULL, S.d_part[g], &a->agg[g][c]));
        break;
    }
    }
}

/* the pending load's shard buffers (NULL: none) */
static void load_release(void) {
    for (int g = 0; g < MAXG; ++g) {
        if (!L.d[g]) continue;
        for (int c = 0; c < L.n_cols; ++c) free_on(g, L.d[g][c]);
        free(L.d[g]);
        L.d[g] = NULL;
    }
    L.pending = 0;
}

static void load_job_free(LoadJob *job) {
    for (int g = 0; g < S.G; ++g) {
        free_on(g, job->d_text[g]);
        if (!job->piece[g]) continue;
        for (int c = 0; c < job->n_cols; ++c) free_on(g, job->piece[g][c]);
        free(job->piece[g]);
    }
    free(job);
}

static int load_step(LoadJob *job, int step, int pf) {
    PF_BEGIN(load);
    job->step = step;
    run_shards(load_shard, job);
    if (PF.on) {
        PF.t[pf] += pf_now() - pf_t0_load;
        ++PF.n[pf];
    }
    return shard_errs(&job->err);
}

int adb_host_load_csv_count(const char *text, size_t bytes, int skip_lines, int n_cols, size_t *rows) {
    t_err[0] = '\0';
    if (ensure_up()) return -1;
    load_release();                                 /* a second count drops a pending one */
    if (!rows || (bytes && !text) || skip_lines < 0 || n_cols < 1 || n_cols > 254) {
        set_err("adb_host_load_csv_count: bad arguments (n_cols %d outside [1, 254]?)", n_cols);
        return -1;
    }
    size_t off = 0;                                 /* the header lines load_db consumes (db_manager.c:263) */
    for (int k = 0; k < skip_lines && off < bytes; ++k) {
        const char *nl = memchr(text + off, '\n', bytes - off);
        off = nl ? (size_t)(nl - text) + 1 : bytes;
    }
    LoadJob *job = calloc(1, sizeof *job);
    if (!job) {
        set_err("out of host memory");
        return -1;
    }
    job->text = text;
    job->n_cols = n_cols;
    const size_t len = bytes - off;
    job->begin[0] = off;
    for (int g = 1; g < S.G; ++g) {
        const size_t at = off + (size_t)((unsigned __int128)g * len / (unsigned)S.G);
        const char *nl = at < bytes ? memchr(text + at, '\n', bytes - at) : NULL;
        job->begin[g] = nl ? (size_t)(nl - text) + 1 : bytes;
    }
    job->begin[S.G] = bytes;
    for (int g = 0; g < S.G; ++g)
        if (!(job->piece[g] = calloc((size_t)n_cols, sizeof(int32_t *)))) {
            set_err("out of host memory");
            load_job_free(job);
            return -1;
        }
    if (load_step(job, 0, PF_LOAD_UPLOAD) || load_step(job, 1, PF_LOAD_PARSE)) {
        load_job_free(job);
        return -1;
    }
    size_t total = 0;
    for (int g = 0; g < S.G; ++g) total += job->rows[g];
    if (total >= ((size_t)1 << 31)) {
        set_err("adb_host_load_csv_count: %zu rows: positions are int (src/query.c:94-95)", total);
        load_job_free(job);
        return -1;
    }
    /* the carry chain: what the reference's row[] holds when piece g starts */
    for (int g = 1; g < S.G; ++g)
        for (int c = 0; c < n_cols; ++c)
            job->carry[g][c] = job->has[g - 1][c] ? job->last[g - 1][c] : job->carry[g - 1][c];
    if (load_step(job, 2, PF_LOAD_FILL)) {
        load_job_free(job);
        return -1;
    }
    /* every fill is enqueued: the re-cut's copies (adb_copy_from_ctx) wait for them */
    PF_BEGIN(recut);
    L.n_cols = n_cols;
    L.rows = total;
    L.shard_rows = shard_rows_for(total);
    size_t want[MAXG];
    for (int g = 0; g < S.G; ++g) {
        want[g] = shard_len(total, L.shard_rows, g);
        if (!(L.d[g] = calloc((size_t)n_cols, sizeof(int32_t *)))) {
            set_err("out of host memory");
            goto fail;
        }
    }
    for (int c = 0; c < n_cols; ++c) {
        int32_t *src[MAXG], *dst[MAXG] = {0};
        for (int g = 0; g < S.G; ++g) src[g] = job->piece[g][c];
        const int rc = recut(src, job->rows, want, dst);
        for (int g = 0; g < S.G; ++g) L.d[g][c] = dst[g];
        if (rc) goto fail;
        for (int g = 0; g < S.G; ++g) {            /* recut waited for its copies */
            free_on(g, job->piece[g][c]);
            job->piece[g][c] = NULL;
        }
    }
    if (PF.on) {
        PF.t[PF_LOAD_RECUT] += pf_now() - pf_t0_recut;
        ++PF.n[PF_LOAD_RECUT];
    }
    if (load_step(job, 3, PF_LOAD_AGG)) goto fail;
    for (int c = 0; c < n_cols; ++c) {
        L.mn[c] = INT_MAX;
        L.mx[c] = INT_MIN;
        for (int g = 0; g < S.G; ++g) {
            if (!shard_len(total, L.shard_rows, g)) continue;
            if (job->agg[g][c].min < L.mn[c]) L.mn[c] = job->agg[g][c].min;
            if (job->agg[g][c].max > L.mx[c]) L.mx[c] = job->agg[g][c].max;
        }
    }
    load_job_free(job);
    L.pending = 1;
    *rows = total;
    return 0;
fail:
    load_release();
    load_job_free(job);
    return -1;
}

typedef struct EmitJob {
    ShardErr err;
    Column **cols;
    size_t old_rows;
} EmitJob;
static void load_emit_shard(int g, void *arg) {
    EmitJob *a = arg;
    const size_t n = shard_len(L.rows, L.shard_rows, g);
    for (int c = 0; c < L.n_cols && n; ++c)
        SCK(adb_download(a->cols[c]->data + a->old_rows + (size_t)g * L.shard_rows, L.d[g][c], 4 * n));
}

int adb_host_load_csv_emit(Column **cols, int n_cols) {
    t_err[0] = '\0';
    if (ensure_up()) return -1;
    if (!L.pending) {
        set_err("adb_host_load_csv_emit: no pending adb_host_load_csv_count");
        return -1;
    }
    int rc = -1;
    const size_t old = cols && n_cols > 0 && cols[0] ? cols[0]->row_count : 0;
    if (!cols || n_cols != L.n_cols) {
        set_err("adb_host_load_csv_emit: %d columns, the count parsed %d", n_cols, L.n_cols);
        goto done;
    }
    for (int c = 0; c < n_cols; ++c)
        if (!cols[c] || !cols[c]->data || cols[c]->row_count != old) {
            set_err("adb_host_load_csv_emit: the table's columns must be host-backed and equally long");
            goto done;
        }
    if (old + L.rows >= ((size_t)1 << 31)) {
        set_err("adb_host_load_csv_emit: %zu + %zu rows: positions are int (src/query.c:94-95)", old, L.rows);
        goto done;
    }
    for (int c = 0; c < n_cols; ++c) {              /* handles and indexes of the old rows go first */
        DevColumn *dc = dev_column_slot(cols[c]);
        if (!dc) goto done;
        dev_column_drop(dc);
    }
    PF_BEGIN(download);
    EmitJob job;
    memset(&job, 0, sizeof job);
    job.cols = cols;
    job.old_rows = old;
    run_shards(load_emit_shard, &job);
    if (PF.on) {
        PF.t[PF_LOAD_DOWNLOAD] += pf_now() - pf_t0_download;
        ++PF.n[PF_LOAD_DOWNLOAD];
    }
    if (shard_errs(&job.err)) goto done;
    for (int c = 0; c < n_cols; ++c) {
        Column *col = cols[c];
        if (L.rows && L.mn[c] < col->min) col->min = L.mn[c];
        if (L.rows && L.mx[c] > col->max) col->max = L.mx[c];
        col->row_count = old + L.rows;
        if (old || !L.rows) continue;               /* an append: the next operator uploads the whole column */
        DevColumn *dc = dev_column_slot(col);
        if (dc->uploaded_from != col->data || dc->uploaded_bytes != 4 * L.rows) {
            column_unregister(dc);
            dc->uploaded_from = col->data;
            dc->uploaded_bytes = 4 * L.rows;
        }
        ++dc->uploads;
        for (int g = 0; g < S.G; ++g) {
            dc->d_data[g] = L.d[g][c];
            L.d[g][c] = NULL;                       /* the column owns them now (adopted = 0) */
        }
        dc->host_data = col->data;
        dc->rows = L.rows;
        dc->shard_rows = L.shard_rows;
    }
    rc = 0;
done:
    load_release();
    return rc;
}

/* ---- selects ------------------------------------------------------------------------------ */
/* src/index.c:180-185: the cost model is the constant `true` (the drop-in links
 * host/index_shim.c in place of index.c, so the definition lives here in both builds). */
bool should_use_index(Column *column, int low, int high) {
    (void)column; (void)low; (void)high;
    return true;
}

void log_result(Result *result) { (void)result; }        /* src/query.c:26-28: returns at once */

typedef struct SelectJob {
    ShardErr err;
    DevColumn *c;
    int *low, *high;
    int use_btree, defer;
    ShardList out;
    uint64_t generation[MAXG];
} SelectJob;

/* select_column_sorted_index (src/query.c:165-198) through the uploaded index slices. */
static void select_index_shard(int g, void *arg) {
    SelectJob *a = arg;
    DevColumn *c = a->c;
    int64_t h = 0;
    SCK(adb_select_index_count(c->ix[g], a->use_btree, a->low, a->high, NULL, &h));
    void *p = NULL;
    SCK(adb_alloc(&p, 4 * (size_t)h));
    a->out.d[g] = p;
    a->out.n[g] = (size_t)h;
    SCK(adb_select_index_emit(c->ix[g], p));
}

static Result *select_index_path(Column *column, DevColumn *c, int *low, int *high, Status *st) {
    if (dev_index(c, column)) return op_fail(st, "select_column");
    SelectJob job;
    memset(&job, 0, sizeof job);
    job.c = c;
    job.low = low;
    job.high = high;
    job.use_btree = !column->sorted;                 /* create_index(... sorted=false) = btree */
    run_shards(select_index_shard, &job);
    if (shard_errs(&job.err)) goto fail;
    if (S.G > 1) {
        /* the slices answered positions[lb(low) .. lb(high)); the reference's low == high quirk
         * (query.c:181-188; closed form in index_lookup.cu) belongs to the whole index: in the
         * defined domain, an empty range whose upper bound is a key yields the first tuple
         * carrying that key */
        size_t total = 0;
        for (int g = 0; g < S.G; ++g) total += job.out.n[g];
        if (total == 0 && c->ix_rows > 0 && low && high && *low <= *high && *low >= c->ix_min) {
            SelectJob q2;
            memset(&q2, 0, sizeof q2);
            int lo2 = *high, hi2 = *high == INT_MAX ? 0 : *high + 1;
            q2.c = c;
            q2.low = &lo2;
            q2.high = *high == INT_MAX ? NULL : &hi2;
            q2.use_btree = job.use_btree;
            run_shards(select_index_shard, &q2);
            if (shard_errs(&q2.err)) {
                list_release(&q2.out);
                goto fail;
            }
            int first = -1;
            for (int g = 0; g < S.G; ++g)
                if (q2.out.n[g] && first < 0) first = g;
            if (first >= 0) {                       /* keep the first tuple only */
                list_release(&job.out);
                job.out = q2.out;
                for (int g = 0; g < S.G; ++g) job.out.n[g] = g == first ? 1 : 0;
            } else {
                list_release(&q2.out);
            }
        }
    }
    job.out.aligned = 0;                            /* index order: positions anywhere */
    if (S.G > 1) {
        /* A range of a range-partitioned index lives in one or two slices, so one or two GPUs hold
         * the whole (long) list and would do every later fetch / aggregate over it alone.  The
         * list is the concatenation of the shards' buffers whatever the cut: re-cut it evenly over
         * the GPUs with peer copies (order untouched). */
        size_t total = 0, most = 0;
        for (int g = 0; g < S.G; ++g) {
            total += job.out.n[g];
            if (job.out.n[g] > most) most = job.out.n[g];
        }
        if (total >= S.rebalance_min && most > 2 * (total / (size_t)S.G)) {
            ShardList even;
            memset(&even, 0, sizeof even);
            const size_t per = (total + (size_t)S.G - 1) / (size_t)S.G;
            for (int g = 0; g < S.G; ++g) even.n[g] = shard_len(total, per, g);
            if (recut(job.out.d, job.out.n, even.n, even.d)) {
                list_release(&even);
                goto fail;
            }
            list_release(&job.out);
            job.out = even;
        }
    }
    return hand_out(&job.out, st, "select_column");
fail:
    list_release(&job.out);
    return op_fail(st, "select_column");
}

static void select_scan_shard(int g, void *arg) {
    SelectJob *a = arg;
    DevColumn *c = a->c;
    const size_t n = shard_len(c->rows, c->shard_rows, g);
    int64_t h = 0;
    SCK(adb_select_count_base(c->d_data[g], (int64_t)n, a->low, a->high, shard_base(g, c->shard_rows), NULL, &h));
    a->generation[g] = adb_select_generation();
    void *p = NULL;
    SCK(adb_alloc(&p, 4 * (size_t)h));
    a->out.d[g] = p;
    a->out.n[g] = (size_t)h;
    if (!a->defer) SCK(adb_select_emit(NULL, shard_base(g, c->shard_rows), p));
}

/* src/query.c:203-220: clustered or indexed columns go through the index, others scan. */
static Result *select_column_impl(Column *column, int *low, int *high, Status *ret_status);
Result *select_column(Column *column, int *low, int *high, Status *ret_status) {
    PF_BEGIN(PF_SELECT);
    Result *r = select_column_impl(column, low, high, ret_status);
    PF_END(PF_SELECT);
    return r;
}
static Result *select_column_impl(Column *column, int *low, int *high, Status *ret_status) {
    t_err[0] = '\0';
    if (ensure_up()) return op_fail(ret_status, "select_column");
    DevColumn *c = dev_column(column);
    if (!c) return op_fail(ret_status, "select_column");
    if (column->clustered ||
        (column->has_index && should_use_index(column, low ? *low : 0, high ? *high : 0)))
        return select_index_path(column, c, low, high, ret_status);
    SelectJob job;
    memset(&job, 0, sizeof job);
    if (demote_pending()) goto fail;                /* this select takes the bitmaps over */
    job.c = c;
    job.low = low;
    job.high = high;
    job.defer = S.lazy;
    PF_BEGIN(PF_SELECT_JOB);
    run_shards(select_scan_shard, &job);
    PF_END(PF_SELECT_JOB);
    if (shard_errs(&job.err)) goto fail;
    job.out.aligned = c->shard_rows;
    Result *r = hand_out(&job.out, ret_status, "select_column");
    if (r && job.defer && job.out.total > 0) {      /* positions are written by whoever needs them first */
        memset(&P, 0, sizeof P);
        P.sel_payload = r->payload;
        for (int g = 0; g < S.G; ++g) {
            P.sel_d[g] = job.out.d[g];
            P.h[g] = job.out.n[g];
            P.d_col[g] = c->d_data[g];
            P.rows[g] = shard_len(c->rows, c->shard_rows, g);
            P.generation[g] = job.generation[g];
        }
        P.shard_rows = c->shard_rows;
        P.has_lo = low != NULL;
        P.has_hi = high != NULL;
        P.lo = low ? *low : 0;
        P.hi = high ? *high : 0;
        P.active = 1;
    }
    return r;
fail:
    list_release(&job.out);
    return op_fail(ret_status, "select_column");
}

/* src/query.c:38-86: predicate over a fetched value vector, emits the paired positions. */
typedef struct PairsJob {
    ShardErr err;
    ShardList *v, *p;
    int *low, *high;
    ShardList out;
} PairsJob;
static void select_pairs_shard(int g, void *arg) {
    PairsJob *a = arg;
    int64_t h = 0;
    SCK(adb_select_count(a->v->d[g], (int64_t)a->v->n[g], NULL, a->low, a->high, NULL, &h));
    void *p = NULL;
    SCK(adb_alloc(&p, 4 * (size_t)h));
    a->out.d[g] = p;
    a->out.n[g] = (size_t)h;
    SCK(adb_select_emit(a->p->d[g], 0, p));
}

Result *select_result(Result *column, Result *position, int *low_pointer, int *high_pointer,
                      Status *ret_status) {
    t_err[0] = '\0';
    ShardList v, p;
    memset(&v, 0, sizeof v);
    memset(&p, 0, sizeof p);
    PairsJob job;
    memset(&job, 0, sizeof job);
    if (ensure_up() || stage(column, NULL, &v)) goto fail;
    if (!position || position->num_tuples < column->num_tuples) {
        set_err("select: %zu values but only %zu positions", column->num_tuples,
                position ? position->num_tuples : (size_t)0);
        goto fail;
    }
    {
        /* the positions are cut like the values (a longer list: the extra tail is ignored, as
         * the reference's loop over column->num_tuples does) */
        Result head = *position;
        head.num_tuples = column->num_tuples;
        if (stage(&head, v.n, &p)) goto fail;
    }
    job.v = &v;
    job.p = &p;
    job.low = low_pointer;
    job.high = high_pointer;
    run_shards(select_pairs_shard, &job);
    if (shard_errs(&job.err)) goto fail;
    job.out.aligned = p.aligned;
    list_release(&v);
    list_release(&p);
    return hand_out(&job.out, ret_status, "select_result");
fail:
    list_release(&job.out);
    list_release(&v);
    list_release(&p);
    return op_fail(ret_status, "select_result");
}

/* src/query.c:450-583: query_count range selects in one pass; reads .low/.high only and
 * ignores has_low/has_high and indexes, exactly as query.c:474 does.  Per context ONE slab holds
 * all the batch's position lists (one allocation instead of query_count); every Result is a
 * view into it and the slab goes back to the pool when the last of them is released. */
typedef struct SharedJob {
    ShardErr err;
    DevColumn *c;
    int q_count;
    int32_t *lows, *highs;
    int64_t counts[MAXG][ADB_MAX_BATCH];
    size_t off[MAXG][ADB_MAX_BATCH];
    int32_t *slab[MAXG];
} SharedJob;
static void shared_shard(int g, void *arg) {
    SharedJob *a = arg;
    DevColumn *c = a->c;
    const size_t n = shard_len(c->rows, c->shard_rows, g);
    SCK(adb_shared_select_count_base(c->d_data[g], (int64_t)n, shard_base(g, c->shard_rows), a->lows, a->highs,
                                     a->q_count, a->counts[g]));
    size_t total = 0;
    int64_t cap = 1;
    for (int q = 0; q < a->q_count; ++q) {
        a->off[g][q] = total;
        total += ((size_t)a->counts[g][q] + 3) & ~(size_t)3;         /* every list 16-byte aligned */
        if (a->counts[g][q] > cap) cap = a->counts[g][q];
    }
    void *p = NULL;
    SCK(adb_alloc(&p, 4 * total));
    a->slab[g] = p;
    int32_t *outs[ADB_MAX_BATCH];
    for (int q = 0; q < a->q_count; ++q) outs[q] = a->slab[g] + a->off[g][q];
    SCK(adb_shared_select_emit(outs, cap));
}

Result **shared_select(SelectOperator *operators, int query_count, Column *column,
                       Status *ret_status) {
    t_err[0] = '\0';
    Result **results = NULL;
    SharedJob *job = NULL;
    Slab *slab = NULL;
    int made = 0;
    if (ensure_up()) goto fail;
    if (query_count < 1 || query_count > ADB_MAX_BATCH || !operators) {
        set_err("shared_select: query_count %d outside [1, %d] (the dispatcher chunks batches "
                "to 150, src/server.c:366-371)", query_count, ADB_MAX_BATCH);
        goto fail;
    }
    DevColumn *c = dev_column(column);
    if (!c) goto fail;                              /* (the batched scan has its own scratch: P stays) */
    results = calloc((size_t)query_count, sizeof *results);
    job = calloc(1, sizeof *job);
    slab = calloc(1, sizeof *slab);
    if (job) {
        job->lows = malloc(sizeof(int32_t) * (size_t)query_count);
        job->highs = malloc(sizeof(int32_t) * (size_t)query_count);
    }
    if (!results || !job || !slab || !job->lows || !job->highs) {
        set_err("out of host memory");
        goto fail;
    }
    for (int q = 0; q < query_count; ++q) {
        job->lows[q] = operators[q].low;
        job->highs[q] = operators[q].high;
    }
    job->c = c;
    job->q_count = query_count;
    run_shards(shared_shard, job);
    if (shard_errs(&job->err)) {
        for (int g = 0; g < S.G; ++g) free_on(g, job->slab[g]);
        goto fail;
    }
    for (int g = 0; g < S.G; ++g) slab->base[g] = job->slab[g];
    slab->refs = query_count;
    for (int q = 0; q < query_count; ++q) {
        ShardList view;
        memset(&view, 0, sizeof view);
        for (int g = 0; g < S.G; ++g) {
            view.d[g] = job->slab[g] + job->off[g][q];
            view.n[g] = (size_t)job->counts[g][q];
        }
        view.aligned = c->shard_rows;
        view.slab = slab;
        results[q] = new_dev_result(&view);
        if (!results[q]) {
            slab_drop(slab, query_count - q);       /* the views not handed out yet give their references back */
            slab = NULL;
            goto fail;
        }
        made = q + 1;
    }
    free(job->lows);
    free(job->highs);
    free(job);
    op_ok(ret_status);
    return results;
fail:
    for (int q = 0; q < made; ++q) drop_result(results[q]);
    if (made == 0) free(slab);
    free(results);
    if (job) {
        free(job->lows);
        free(job->highs);
        free(job);
    }
    return op_fail(ret_status, "shared_select");
}

/* ---- fetch --------------------------------------------------------------------------------- */
/* src/query.c:223-243: values[i] = column->data[position[i]]. */
typedef struct FetchJob {
    ShardErr err;
    DevColumn *c;
    ShardList *p;
    ShardList out;
    int phase;
    Route route;                                    /* routed form (phases 1-3): items = positions */
} FetchJob;
/* A position list that is not aligned with the column's shards (index order, a join's output):
 * above this many positions they are routed to the GPUs that hold the rows and the values come
 * back in bulk (adb_route_rows); below, every remote row is one NVLink read (adb_fetch_sharded).
 * ADB_FETCH_ROUTE_MIN overrides (0 = always route, a huge value = never). */
/* Measured (r02zo / r02zp, 500 M-row column, index-ordered lists): two GPUs, 5 M positions 0.39 ->
 * 0.23 ms, 50 M 3.58 -> 1.40 ms; eight GPUs, 5 M 0.20 -> 0.43 ms, 50 M 0.92 -> 0.98 ms -- the routed
 * form pays three host phases (~0.3 ms), the peer loads of eight GPUs spread over seven links each.
 * Default: 1 M positions on two GPUs, 16 x that per doubling of the GPU count. */
static size_t fetch_route_min(void) {
    const char *e = getenv("ADB_FETCH_ROUTE_MIN");
    if (e) {
        const long long v = atoll(e);
        return v < 0 ? 0 : (size_t)v;
    }
    size_t m = (size_t)1 << 20;
    for (int g = 2; g < S.G; g *= 2) m *= 16;
    return m;
}
static void fetch_shard(int g, void *arg) {
    FetchJob *a = arg;
    DevColumn *c = a->c;
    const size_t n = a->p->n[g];
    Route *r = &a->route;
    if (a->phase == 2) {                            /* owner: gather my pieces from my shard */
        int32_t *pos = NULL;
        int64_t n_recv = 0;
        SCK(route_pull(g, r, &pos, &n_recv));
        if (n_recv)
            SCK(adb_fetch(c->d_data[g], pos, n_recv, NULL, shard_base(g, c->shard_rows), r->answers_owner[g]));
        SCK(adb_sync());
        return;
    }
    if (a->phase == 3) {                            /* home: the values back into list order */
        SCK(route_return(g, r, 4));
        SCK(adb_route_finish32(S.G, a->out.d[g], (int64_t)n));
        return;
    }
    void *out = NULL;
    SCK(adb_alloc(&out, 4 * n));
    a->out.d[g] = out;
    a->out.n[g] = n;
    if (a->phase == 1) {                            /* home: my positions grouped by the shard they name */
        SCK(adb_route_rows(S.G, (int64_t)c->shard_rows, a->p->d[g], (int64_t)n, r->sent[g], &r->items[g],
                           &r->answers_home[g]));
        return;
    }
    if (!n) return;
    if (S.G == 1 || (a->p->aligned && a->p->aligned == c->shard_rows))
        SCK(adb_fetch(c->d_data[g], a->p->d[g], (int64_t)n, NULL, shard_base(g, c->shard_rows), out));
    else
        SCK(adb_fetch_sharded((const int32_t *const *)c->d_data, S.G, (int64_t)c->shard_rows, a->p->d[g],
                              (int64_t)n, NULL, out));
}

static Result *fetch_column_impl(Column *column, Result *position_result, Status *ret_status);
Result *fetch_column(Column *column, Result *position_result, Status *ret_status) {
    PF_BEGIN(PF_FETCH);
    Result *r = fetch_column_impl(column, position_result, ret_status);
    PF_END(PF_FETCH);
    return r;
}
static Result *fetch_column_impl(Column *column, Result *position_result, Status *ret_status) {
    t_err[0] = '\0';
    ShardList p;
    memset(&p, 0, sizeof p);
    FetchJob job;
    memset(&job, 0, sizeof job);
    if (ensure_up()) goto fail;
    DevColumn *c = dev_column(column);
    if (!c) goto fail;
    /* fetch of the pending select: nothing is launched yet -- the values are written together
     * with the positions, by the aggregate that usually follows or by the first other reader */
    if (P.active && position_result && position_result->payload == P.sel_payload && !P.fetch_payload &&
        c->shard_rows == P.shard_rows) {
        size_t total = 0;
        int fits = 1;
        for (int g = 0; g < S.G; ++g) {
            total += P.h[g];
            if (shard_len(c->rows, c->shard_rows, g) < P.rows[g]) fits = 0;
        }
        if (fits && position_result->num_tuples == total) {
            ShardList vals;
            memset(&vals, 0, sizeof vals);
            memcpy(vals.n, P.h, sizeof vals.n);
            PF_BEGIN(PF_FETCH_JOB);
            const int arc = alloc_shards(&vals);
            PF_END(PF_FETCH_JOB);
            if (arc) goto fail;
            Result *r = new_dev_result(&vals);
            if (!r) return op_fail(ret_status, "fetch_column");
            if (P.active) {                         /* (new_dev_result may have flushed) */
                P.fetch_payload = r->payload;
                for (int g = 0; g < S.G; ++g) {
                    P.fetch_d[g] = vals.d[g];
                    P.d_fetch_col[g] = c->d_data[g];
                }
                op_ok(ret_status);
                return r;
            }
            drop_result(r);                         /* rare: take the ordinary path below */
        }
    }
    if (stage(position_result, NULL, &p)) goto fail;
    job.c = c;
    job.p = &p;
    if (S.G > 1 && !(p.aligned && p.aligned == c->shard_rows) && p.total >= fetch_route_min() &&
        c->shard_rows > 0) {
        if (run_routed(fetch_shard, &job, &job.phase, &job.err)) goto fail;
    } else {
        run_shards(fetch_shard, &job);
        if (shard_errs(&job.err)) goto fail;
    }
    job.out.aligned = p.aligned;                    /* values pair with their positions shard by shard */
    list_release(&p);
    return hand_out(&job.out, ret_status, "fetch_column");
fail:
    list_release(&job.out);
    list_release(&p);
    return op_fail(ret_status, "fetch_column");
}

/* ---- aggregates ------------------------------------------------------------------------------ */
typedef struct AggJob {
    ShardErr err;
    int32_t *const *d;
    const size_t *n;
    int fused;                   /* resolve the pending select + fetch in the same kernel */
    adb_agg h;
} AggJob;
static void agg_shard(int g, void *arg) {
    AggJob *a = arg;
    adb_agg *h = g == 0 ? &a->h : NULL;
    if (a->fused) {
        /* the newest select's bitmap: gather + fold its hit rows, unwritten (fused == 1) or
         * writing both handles on the way (fused == 2); a context whose bitmap was overwritten
         * meanwhile redoes its predicate pass first */
        if (lazy_recount_shard(&P, 1, g, &a->err)) return;
        int32_t *pos = a->fused == 2 ? P.sel_d[g] : NULL, *val = a->fused == 2 ? P.fetch_d[g] : NULL;
        if (S.G == 1)
            SCK(adb_select_emit_fetch_agg(P.d_fetch_col[g], pos, val, S.d_part[g], h));
        else
            SCK(adb_select_emit_fetch_agg_exchange(P.d_fetch_col[g], pos, val, S.d_part[g], S.d_out[g], h));
        return;
    }
    if (S.G == 1) {
        SCK(adb_aggregate(a->d[g], (int64_t)a->n[g], NULL, S.d_part[g], h));
    } else {
        SCK(adb_aggregate(a->d[g], (int64_t)a->n[g], NULL, S.d_part[g], NULL));
        SCK(adb_agg_combine_allreduce(S.d_part[g], 1, S.d_out[g], h));
    }
}

static int aggregate_shards(int32_t *const d[], const size_t n[], adb_agg *h) {
    AggJob job;
    memset(&job, 0, sizeof job);
    job.d = d;
    job.n = n;
    run_shards(agg_shard, &job);
    if (shard_errs(&job.err)) return -1;
    *h = job.h;
    return 0;
}

static int aggregate_result_impl(const Result *r, adb_agg *h);
static int aggregate_result(const Result *r, adb_agg *h) {
    PF_BEGIN(PF_AGG);
    const int rc = aggregate_result_impl(r, h);
    PF_END(PF_AGG);
    return rc;
}
static int aggregate_result_impl(const Result *r, adb_agg *h) {
    ShardList v;
    memset(&v, 0, sizeof v);
    if (ensure_up()) return -1;
    /* aggregate of the unwritten fetch of the newest select: the hit rows are gathered and
     * folded straight from the bitmap.  The first aggregate writes nothing (4N + 4H bytes for the
     * chain); a second one on the same handle writes both handles on the way -- whoever asks
     * twice will probably ask again. */
    if (P.active && r && P.fetch_payload && r->payload == P.fetch_payload && r->data_type == INT) {
        size_t total = 0;
        for (int g = 0; g < S.G; ++g) total += P.h[g];
        if (r->num_tuples == total) {
            AggJob job;
            memset(&job, 0, sizeof job);
            job.fused = P.aggregated ? 2 : 1;
            PF_BEGIN(PF_AGG_JOB);
            run_shards(agg_shard, &job);
            PF_END(PF_AGG_JOB);
            if (job.fused == 2) lazy_done(&P);
            else P.aggregated = 1;
            if (shard_errs(&job.err)) return -1;
            *h = job.h;
            return 0;
        }
    }
    if (stage(r, NULL, &v)) return -1;
    int rc = aggregate_shards(v.d, v.n, h);
    list_release(&v);
    return rc;
}

static Result *scalar_result(DataType t, const void *value, size_t width, Status *st, const char *what) {
    Result *r = malloc(sizeof *r);
    void *p = malloc(width);
    if (!r || !p) {
        free(r);
        free(p);
        set_err("out of host memory");
        return op_fail(st, what);
    }
    /* malloc handed out an address we still hold a device result for: the plumbing freed that
     * payload without telling us (no release hook, no interposer) -- it is dead, drop it */
    adb_host_payload_freed(p);
    memcpy(p, value, width);
    r->num_tuples = 1;
    r->data_type = t;
    r->payload = p;
    op_ok(st);
    return r;
}

/* src/query.c:306-323: long sum, then (double)sum / (double)num_tuples on the host -- the
 * same two conversions and one division, so the double is bit-identical (empty -> -nan). */
Result *average(Result *column, Status *ret_status) {
    t_err[0] = '\0';
    adb_agg a;
    if (aggregate_result(column, &a)) return op_fail(ret_status, "average");
    long s = (long)a.sum;
    double avg = (double)s / (double)column->num_tuples;
    return scalar_result(DOUBLE, &avg, sizeof avg, ret_status, "average");
}

/* src/query.c:325-354: long sum over a Result or over a whole base column. */
Result *sum(GeneralizedColumn *column, Status *ret_status) {
    t_err[0] = '\0';
    adb_agg a;
    if (!column) {
        set_err("NULL operand");
        return op_fail(ret_status, "sum");
    }
    if (column->column_type == RESULT) {
        if (aggregate_result(column->column_pointer.result, &a)) return op_fail(ret_status, "sum");
    } else {
        if (ensure_up()) return op_fail(ret_status, "sum");
        DevColumn *c = dev_column(column->column_pointer.column);
        if (!c) return op_fail(ret_status, "sum");
        size_t n[MAXG];
        for (int g = 0; g < S.G; ++g) n[g] = shard_len(c->rows, c->shard_rows, g);
        if (aggregate_shards(c->d_data, n, &a)) return op_fail(ret_status, "sum");
    }
    long s = (long)a.sum;
    return scalar_result(LONG, &s, sizeof s, ret_status, "sum");
}

/* src/query.c:392-437.  The reference seeds with payload[0]; on an empty input that is an
 * out-of-bounds read (oracle-undefined) -- here min is INT_MAX and max INT_MIN. */
Result *min(Result *column, Status *ret_status) {
    t_err[0] = '\0';
    adb_agg a;
    if (aggregate_result(column, &a)) return op_fail(ret_status, "min");
    int v = a.min;
    return scalar_result(INT, &v, sizeof v, ret_status, "min");
}
Result *max(Result *column, Status *ret_status) {
    t_err[0] = '\0';
    adb_agg a;
    if (aggregate_result(column, &a)) return op_fail(ret_status, "max");
    int v = a.max;
    return scalar_result(INT, &v, sizeof v, ret_status, "max");
}

/* ---- add / sub -------------------------------------------------------------------------------- */
/* src/query.c:356-390: length is column_one's; the reference does not check column_two's
 * length (it would read out of bounds) -- here a shorter column_two is an ERROR. */
typedef struct EwiseJob {
    ShardErr err;
    ShardList *a, *b;
    int subtract;
    ShardList out;
} EwiseJob;
static void ewise_shard(int g, void *arg) {
    EwiseJob *a = arg;
    const size_t n = a->a->n[g];
    void *out = NULL;
    SCK(adb_alloc(&out, 4 * n));
    a->out.d[g] = out;
    a->out.n[g] = n;
    SCK((a->subtract ? adb_sub : adb_add)(a->a->d[g], a->b->d[g], (int64_t)n, NULL, out));
}
static Result *ewise(Result *one, Result *two, int subtract, Status *st) {
    t_err[0] = '\0';
    const char *what = subtract ? "sub" : "add";
    ShardList a, b;
    memset(&a, 0, sizeof a);
    memset(&b, 0, sizeof b);
    EwiseJob job;
    memset(&job, 0, sizeof job);
    if (ensure_up() || stage(one, NULL, &a)) goto fail;
    if (!two || two->num_tuples < one->num_tuples) {
        set_err("%s: operands of %zu and %zu tuples", what, one->num_tuples, two ? two->num_tuples : (size_t)0);
        goto fail;
    }
    {
        Result head = *two;
        head.num_tuples = one->num_tuples;
        if (stage(&head, a.n, &b)) goto fail;
    }
    job.a = &a;
    job.b = &b;
    job.subtract = subtract;
    run_shards(ewise_shard, &job);
    if (shard_errs(&job.err)) goto fail;
    job.out.aligned = a.aligned;
    list_release(&a);
    list_release(&b);
    return hand_out(&job.out, st, what);
fail:
    list_release(&job.out);
    list_release(&a);
    list_release(&b);
    return op_fail(st, what);
}
Result *add(Result *column_one, Result *column_two, Status *ret_status) {
    return ewise(column_one, column_two, 0, ret_status);
}
Result *sub(Result *column_one, Result *column_two, Status *ret_status) {
    return ewise(column_one, column_two, 1, ret_status);
}

/* ---- joins --------------------------------------------------------------------------------------- */
/* src/query.c:585-696.  results[0] lists side-one positions, results[1] side-two positions;
 * hash join is probe-major over side two, nested-loop outer-major over side one.  The
 * caller frees the two-element array (src/server.c:432).
 * One GPU, or an empty side: the single-context join on context 0. */
/* G > 1: the join itself is sharded.  A key's owner is its routing hash scaled to [0, G), so every
 * GPU count splits the keys near evenly.  The build side is hash-partitioned over the GPUs
 * through peer memory (adb_peer_exchange_pairs), every GPU builds the tables of its keys, and
 * every GPU's slice of the probe side, in its original order, is routed to the keys' owners,
 * probed there, and the answers come home in bulk.  The slices' outputs concatenated in shard
 * order are the reference's probe-major list, so nothing is gathered and nothing re-sorted. */
typedef struct JoinJob {
    ShardErr err;
    ShardList *bv, *bp, *pv, *pp;
    int swapped, phase, overflow;
    size_t cap;                                     /* pairs a GPU can receive */
    size_t pairs[MAXG];                             /* each context's share of the output (phase 3) */
    ShardList o1, o2;
    Route route;                                    /* routed probe (phases 1-3): items = probe keys */
} JoinJob;

static void join_shard(int g, void *arg) {
    JoinJob *a = arg;
    if (a->phase == -1) {
        /* all scratch sized before anybody starts the collective (see adb_peer_exchange_reserve) */
        SCK(adb_peer_exchange_reserve((int64_t)a->bv->n[g], (int64_t)a->cap, (int64_t)a->pv->n[g]));
        return;
    }
    if (a->phase == 0) {
        int64_t rn = 0;
        const int32_t *rv = NULL, *rp = NULL;
        const adb_status s = adb_peer_exchange_pairs(0, a->bv->d[g], a->bp->d[g], (int64_t)a->bv->n[g], &rn, &rv, &rp);
        if (s == ADB_ERR_NOMEM) {                   /* every GPU sees the same verdict: retry with more room */
            a->overflow = 1;
            return;
        }
        if (s != ADB_OK) {
            shard_fail(&a->err, g, "adb_peer_exchange_pairs");
            return;
        }
        SCK(adb_join_build(rv, rp, rn, (int64_t)a->pv->n[g]));
        return;
    }
    Route *r = &a->route;
    if (a->phase == 1) {                            /* routed probe, 3a: my keys grouped by owner */
        SCK(adb_join_route_probe(S.G, a->pv->d[g], (int64_t)a->pv->n[g], r->sent[g], &r->items[g],
                                 &r->answers_home[g]));
        return;
    }
    if (a->phase == 2) {                            /* 3b: I own what the others sent me */
        int32_t *keys = NULL;
        int64_t n_recv = 0;
        SCK(route_pull(g, r, &keys, &n_recv));
        SCK(adb_join_probe_received(n_recv));
        return;
    }
    if (a->phase == 3) {                            /* 3c: the owners' answers come home, back to row order */
        SCK(route_return(g, r, 8));
        int64_t m = 0;
        SCK(adb_join_finish_routed(S.G, a->pv->d[g], a->pp->d[g], (int64_t)a->pv->n[g], a->swapped, &m));
        a->pairs[g] = (size_t)m;
        return;
    }
    /* phase 4: expand into this context's share of the output */
    const size_t m = a->pairs[g];
    void *x = NULL, *y = NULL;
    SCK(adb_alloc(&x, 4 * (size_t)m));
    a->o1.d[g] = x;
    SCK(adb_alloc(&y, 4 * (size_t)m));
    a->o2.d[g] = y;
    a->o1.n[g] = a->o2.n[g] = (size_t)m;
    SCK(adb_join_emit(x, y));
}

static int ensure_join_exchange(size_t cap) {
    if (cap <= jx_cap_now) return 0;
    size_t p2 = (size_t)1 << 17;                    /* grow in powers of two: reconnecting is a device-wide affair */
    while (p2 < cap) p2 <<= 1;
    if (p2 < ((size_t)1 << 31)) cap = p2;
    sync_all();
    if (adb_peer_join_connect_local((int64_t)cap) != ADB_OK) {
        set_err("adb_peer_join_connect_local(%zu): %s", cap, adb_last_error());
        return -1;
    }
    jx_cap_now = cap;
    return 0;
}

static Result **join_sharded(Result *v1, Result *p1, Result *v2, Result *p2, int nested, Status *st) {
    const char *what = nested ? "nested_loop_join" : "hash_join";
    ShardList a, b, c, d;
    memset(&a, 0, sizeof a); memset(&b, 0, sizeof b); memset(&c, 0, sizeof c); memset(&d, 0, sizeof d);
    JoinJob job;
    memset(&job, 0, sizeof job);
    {
        Result h1 = *p1, h2 = *p2;
        h1.num_tuples = v1->num_tuples;
        h2.num_tuples = v2->num_tuples;
        if (stage(v1, NULL, &a) || stage(&h1, a.n, &b) || stage(v2, NULL, &c) || stage(&h2, c.n, &d)) goto fail;
    }
    /* hash join: side one is grouped (build), side two walked in order (probe); nested-loop
     * join is outer-major over side one: side one probes (src/query.c:597-611,669-681) */
    job.bv = nested ? &c : &a;
    job.bp = nested ? &d : &b;
    job.pv = nested ? &a : &c;
    job.pp = nested ? &b : &d;
    job.swapped = nested;
    const size_t nb = job.bv->total;
    for (int attempt = 0; attempt < 2; ++attempt) {
        /* head room of 50 % over an even split; a skewed key set gets the whole side's worth */
        if (ensure_join_exchange(attempt ? nb + 64 : nb / (size_t)S.G + nb / (2 * (size_t)S.G) + 65536)) goto fail;
        job.cap = jx_cap_now < nb ? jx_cap_now : nb;
        job.phase = -1;
        run_shards(join_shard, &job);
        if (shard_errs(&job.err)) goto fail;
        job.phase = 0;
        job.overflow = 0;
        run_shards(join_shard, &job);
        if (shard_errs(&job.err)) goto fail;
        if (!job.overflow) break;
        if (attempt) {
            set_err("%s: the build side does not fit the exchange regions", what);
            goto fail;
        }
    }
    if (run_routed(join_shard, &job, &job.phase, &job.err)) goto fail;
    {
        /* the one-context join's bound (join_count, engine.cu) on the whole result, before any
         * output is allocated: every context's share can stay below 2^31 while their sum does not */
        size_t total = 0;
        for (int g = 0; g < S.G; ++g) total += job.pairs[g];
        if (total >= ((size_t)1 << 31)) {
            set_err("%s: join produces %zu pairs; the reference indexes its output with an int "
                    "(query.c:657) so the result must stay below 2^31", what, total);
            goto fail;
        }
    }
    job.phase = 4;
    run_shards(join_shard, &job);
    if (shard_errs(&job.err)) goto fail;
    list_release(&a); list_release(&b); list_release(&c); list_release(&d);
    return hand_out_pair(&job.o1, &job.o2, st, what);
fail:
    list_release(&job.o1);
    list_release(&job.o2);
    list_release(&a); list_release(&b); list_release(&c); list_release(&d);
    return op_fail(st, what);
}

static Result **join(Result *v1, Result *p1, Result *v2, Result *p2, int nested, Status *st) {
    t_err[0] = '\0';
    const char *what = nested ? "nested_loop_join" : "hash_join";
    if (ensure_up()) return op_fail(st, what);
    if (S.G > 1 && v1 && p1 && v2 && p2 && v1->num_tuples && v2->num_tuples &&
        p1->num_tuples >= v1->num_tuples && p2->num_tuples >= v2->num_tuples)
        return join_sharded(v1, p1, v2, p2, nested, st);
    ShardList a, b, c, d, o1, o2;
    memset(&a, 0, sizeof a); memset(&b, 0, sizeof b); memset(&c, 0, sizeof c); memset(&d, 0, sizeof d);
    memset(&o1, 0, sizeof o1); memset(&o2, 0, sizeof o2);
    int64_t m = 0;
    size_t all1[MAXG] = {0}, all2[MAXG] = {0};
    if (ensure_up() || !v1 || !p1 || !v2 || !p2) goto fail;
    if (p1->num_tuples < v1->num_tuples || p2->num_tuples < v2->num_tuples) {
        set_err("%s: fewer positions than values", what);
        goto fail;
    }
    all1[0] = v1->num_tuples;
    all2[0] = v2->num_tuples;
    {
        Result h1 = *p1, h2 = *p2;
        h1.num_tuples = v1->num_tuples;
        h2.num_tuples = v2->num_tuples;
        if (stage(v1, all1, &a) || stage(&h1, all1, &b) || stage(v2, all2, &c) || stage(&h2, all2, &d)) goto fail;
    }
    if ((nested ? adb_nested_loop_join_count : adb_hash_join_count)(
            a.d[0], b.d[0], (int64_t)v1->num_tuples, c.d[0], d.d[0], (int64_t)v2->num_tuples, &m) != ADB_OK) {
        set_err("%s: %s", what, adb_last_error());
        goto fail;
    }
    {
        void *x = NULL, *y = NULL;
        const int ok = adb_alloc(&x, 4 * (size_t)m) == ADB_OK && adb_alloc(&y, 4 * (size_t)m) == ADB_OK;
        o1.d[0] = x;
        o2.d[0] = y;
        if (!ok) {
            set_err("adb_alloc: %s", adb_last_error());
            goto fail;
        }
        o1.n[0] = o2.n[0] = (size_t)m;
    }
    if (adb_join_emit(o1.d[0], o2.d[0]) != ADB_OK) {
        set_err("adb_join_emit: %s", adb_last_error());
        goto fail;
    }
    list_release(&a); list_release(&b); list_release(&c); list_release(&d);
    for (int g = 1; g < S.G; ++g) {                 /* the other contexts hold empty pieces */
        void *x = NULL, *y = NULL;
        on_ctx(g);
        adb_alloc(&x, 0);
        adb_alloc(&y, 0);
        o1.d[g] = x;
        o2.d[g] = y;
    }
    on_ctx(0);
    return hand_out_pair(&o1, &o2, st, what);
fail:
    list_release(&o1);
    list_release(&o2);
    list_release(&a); list_release(&b); list_release(&c); list_release(&d);
    return op_fail(st, what);
}
Result **nested_loop_join(Result *column_one, Result *position_one, Result *column_two,
                          Result *position_two, Status *ret_status) {
    return join(column_one, position_one, column_two, position_two, 1, ret_status);
}
Result **hash_join(Result *column_one, Result *position_one, Result *column_two,
                   Result *position_two, Status *ret_status) {
    return join(column_one, position_one, column_two, position_two, 0, ret_status);
}

/* ---- print ------------------------------------------------------------------------------------------ */
#define PRINT_ON_DEVICE_MIN 4096       /* shorter results: the download + host loop is cheaper than three launches */
typedef struct Text {
    char *s;
    size_t len, cap;
} Text;
static int text_room(Text *t, size_t extra) {
    if (t->len + extra + 1 <= t->cap) return 0;
    size_t cap = t->cap ? t->cap : 64;
    while (cap < t->len + extra + 1) cap *= 2;
    char *n = realloc(t->s, cap);
    if (!n) return -1;
    t->s = n;
    t->cap = cap;
    return 0;
}
static void text_i64(Text *t, long long v) {          /* "%d" / "%ld" without the printf cost */
    char buf[24];
    int k = 0;
    unsigned long long u = v < 0 ? 0ULL - (unsigned long long)v : (unsigned long long)v;
    do {
        buf[k++] = (char)('0' + u % 10);
        u /= 10;
    } while (u);
    if (v < 0) buf[k++] = '-';
    while (k) t->s[t->len++] = buf[--k];
}

/* device-side "%d\n%d..." of every shard, concatenated */
typedef struct FormatJob {
    ShardErr err;
    int32_t *const *d;
    const size_t *n;
    int64_t bytes[MAXG];
    void *d_text[MAXG];
    char *dst[MAXG];
    int phase;
} FormatJob;
static void format_shard(int g, void *arg) {
    FormatJob *a = arg;
    if (!a->n[g]) return;
    if (a->phase == 0) {
        SCK(adb_format_i32_count(a->d[g], (int64_t)a->n[g], &a->bytes[g]));
        SCK(adb_alloc(&a->d_text[g], (size_t)a->bytes[g]));
        SCK(adb_format_i32_emit(a->d_text[g]));
    } else {
        adb_status s = adb_download(a->dst[g], a->d_text[g], (size_t)a->bytes[g]);
        adb_free(a->d_text[g]);
        a->d_text[g] = NULL;
        if (s != ADB_OK) shard_fail(&a->err, g, "adb_download");
    }
}

/* src/query.c:245-304: results are rendered one after another (column-major), values of a
 * result separated by '\n', results separated by ','; ints "%d", longs "%ld", floats and
 * doubles "%.2f".  Device-resident payloads are copied to the host first.  The reference
 * sizes its buffer at 11 bytes per tuple and overruns it for wide values (SURVEY.md A8);
 * this one grows.  An all-empty print returns "" (the reference returns uninitialised
 * bytes). */
char *print(Result **results, int result_num, Status *ret_status) {
    t_err[0] = '\0';
    Text t = {0};
    void *host = NULL;
    if (text_room(&t, 16)) goto oom;
    t.s[0] = '\0';
    for (int i = 0; i < result_num; ++i) {
        Result *r = results[i];
        if (i > 0) {
            if (text_room(&t, 1)) goto oom;
            t.s[t.len++] = ',';
        }
        const size_t n = r->num_tuples;
        const size_t w = r->data_type == INT || r->data_type == FLOAT ? 4 : 8;
        if (r->data_type == INT && n >= PRINT_ON_DEVICE_MIN) {
            /* a long device-resident INT result is formatted where it lives; the text, not
             * the integers, crosses PCIe and no sprintf runs (SURVEY.md 8f rank 2) */
            ShardList v;
            const int found = result_view(r, &v);
            if (found < 0) goto dev_fail;
            if (found) {
                FormatJob job;
                memset(&job, 0, sizeof job);
                job.d = v.d;
                job.n = v.n;
                run_shards(format_shard, &job);
                size_t bytes = 0;
                int pieces = 0;
                for (int g = 0; g < S.G; ++g)
                    if (v.n[g]) { bytes += (size_t)job.bytes[g]; ++pieces; }
                bytes += pieces ? (size_t)pieces - 1 : 0;            /* '\n' between the shards' texts */
                int bad = shard_errs(&job.err);
                if (!bad && text_room(&t, bytes)) bad = 2;
                if (!bad) {
                    size_t off = t.len;
                    int seen = 0;
                    for (int g = 0; g < S.G; ++g) {
                        if (!v.n[g]) continue;
                        if (seen++) t.s[off++] = '\n';
                        job.dst[g] = t.s + off;
                        off += (size_t)job.bytes[g];
                    }
                    job.phase = 1;
                    run_shards(format_shard, &job);
                    bad = shard_errs(&job.err);
                    if (!bad) t.len += bytes;
                } else {
                    for (int g = 0; g < S.G; ++g) free_on(g, job.d_text[g]);
                }
                if (bad == 2) goto oom;
                if (bad) goto dev_fail;
                continue;
            }
        }
        host = malloc(n ? n * w : 1);
        if (!host) goto oom;
        if (adb_host_result_to_host(r, host)) {
            free(host);
            free(t.s);
            return op_fail(ret_status, "print");
        }
        for (size_t k = 0; k < n; ++k) {
            if (text_room(&t, 400)) goto oom;       /* "%.2f" of a double: at most 312 chars */
            if (r->data_type == INT) text_i64(&t, ((int *)host)[k]);
            else if (r->data_type == LONG) text_i64(&t, ((long *)host)[k]);
            else if (r->data_type == FLOAT) t.len += (size_t)sprintf(t.s + t.len, "%.2f", ((float *)host)[k]);
            else t.len += (size_t)sprintf(t.s + t.len, "%.2f", ((double *)host)[k]);
            if (k != n - 1) t.s[t.len++] = '\n';
        }
        free(host);
        host = NULL;
    }
    t.s[t.len] = '\0';
    op_ok(ret_status);
    return t.s;
dev_fail:
    free(t.s);
    return op_fail(ret_status, "print");
oom:
    free(host);
    free(t.s);
    set_err("out of host memory");
    return op_fail(ret_status, "print");
}
