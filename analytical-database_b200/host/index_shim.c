/*
 * index_shim.c -- build_index(Db*) of the reference (src/index.c:152-178) on the B200 engine.
 * Drop-in build only (it walks the reference's Db / Table structs, so it needs the
 * reference's headers): it replaces src/index.c's build_index in the server's link line.  The
 * loop is the reference's -- tables and columns in declaration order, which is what makes an
 * unclustered index on an EARLIER column keep pre-permutation positions when a later column
 * is clustered (SURVEY.md A2) -- and every build goes to the engine
 * (adb_host_index_build: radix sort on the GPU, sibling permutation as peer gathers,
 * histogram kernel).
 *
 * Tie order: the engine's sort is stable (ties in ascending row order), the reference's
 * quicksort is not (SURVEY.md A3); the two agree whenever the indexed keys are unique.
 * ADB_INDEX_TIES=reference keeps the build on the GPU with the quicksort's own tie order
 * (adb_index_sort_ref_ties, chosen in adb_host_index_build), so the clustered siblings'
 * layout and every select on them equal the reference's too.
 * ADB_INDEX_BUILD=reference hands the build to the reference's own, unmodified index.c
 * (compiled into the drop-in under the name reference_build_index, oracle/Makefile) for hosts
 * that need its exact tie order; the shim then uploads what it built, as in round 1.
 */
#include <stdlib.h>
#include <string.h>

#include "adb_query_api.h"        /* with ADB_WITH_REFERENCE_HEADERS: cs165_api.h, db_manager.h */
#include "utils.h"

void reference_build_index(Db *db);               /* src/index.c's build_index, renamed at compile time */

/* src/index.c:63-84 with the counting loop on the device */
static void engine_histogram(Column *column) {
    Histogram *histogram = malloc(sizeof(Histogram));
    if (!histogram) return;
    histogram->bin_size = (column->max - column->min) / (BIN_NUM - 1);
    memset(histogram->values, 0, sizeof(int) * BIN_NUM);
    memset(histogram->counts, 0, sizeof(size_t) * BIN_NUM);
    column->histogram = histogram;
    size_t bin_start = 0;
    for (int bin = 0; bin < BIN_NUM; bin++) {
        histogram->values[bin] = bin_start;
        bin_start += histogram->bin_size;
    }
    unsigned long counts[100];
    if (histogram->bin_size > 0 && adb_host_column_histogram(column, histogram->bin_size, counts) == 0)
        for (int bin = 0; bin < BIN_NUM && bin < 100; bin++) histogram->counts[bin] = counts[bin];
}

void build_index(Db *db) {
    const char *mode = getenv("ADB_INDEX_BUILD");
    if (mode && strcmp(mode, "reference") == 0) {
        reference_build_index(db);
        return;
    }
    for (size_t i = 0; i < db->tables_size; i++) {
        Table *table = &(db->tables[i]);
        Column **cols = malloc((table->col_count ? table->col_count : 1) * sizeof *cols);
        if (!cols) return;
        for (size_t j = 0; j < table->col_count; j++) cols[j] = &(table->columns[j]);
        for (size_t j = 0; j < table->col_count; j++) {
            Column *column = cols[j];
            if (!column->has_index) continue;
            if (adb_host_index_build(cols, (int)table->col_count, (int)j) != 0) {
                log_err("index build of %s on the engine failed: %s\n", column->name, adb_host_last_error());
                continue;                           /* selects on it will answer "Failed" */
            }
            if (!column->clustered) engine_histogram(column);
        }
        free(cols);
    }
}
