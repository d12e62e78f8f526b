/*
 * adb_load_api.h -- bulk load for the operator-API host (analytical-database_b200/host/query_shim.c):
 * what load_db's ingest loop does (src/db_manager.c:304-318), on every GPU at once.  Its own
 * header because it is not part of the reference's query.h surface: load_db lives in the catalog
 * (db_manager.c), and the binding a maintainer adds there is in INTEGRATION.md ("Bulk load").
 * Column comes from adb_query_api.h (the reference's cs165_api.h with
 * -DADB_WITH_REFERENCE_HEADERS).
 */
#ifndef ADB_LOAD_API_H
#define ADB_LOAD_API_H

#include <stddef.h>

#include "adb_query_api.h"

#ifdef __cplusplus
extern "C" {
#endif
/* Bulk load -- load_db's ingest loop (src/db_manager.c:304-318) on every GPU at once (SURVEY.md 8f
 * rank 1).  Two phases, because the catalog grows its columns in between:
 *   count  parses the data rows of a CSV file (`text`: the bytes after load_db's header line,
 *          skip_lines more lines are skipped first) into n_cols columns, in [1, 254]; *rows = the
 *          lines, as fgets counts them.  The text is cut into one piece per GPU at line boundaries
 *          (piece g > 0 starts right after the first '\n' at or after byte g*len/G of the text
 *          after the skipped lines); every GPU uploads its piece over its own link and parses it,
 *          and the rows are re-cut into the shim's row-range shards.  Values are atoi's; a missing
 *          field repeats the nearest earlier row's (0 if none), as the reference's reused row[]
 *          does.  A line over 1023 bytes (fgets would split it) is refused.  A second count drops
 *          a pending one.
 *   emit   cols[0 .. n_cols): the table's columns in file order, equally long, each Column.data
 *          with room for row_count + rows ints.  Appends the rows to the host arrays, folds
 *          min / max as insert_row does, sets row_count.  Into an empty table the parsed shards
 *          become the columns' device copies (the next operator uploads nothing); an append leaves
 *          the columns to be uploaded again.  On failure the columns are untouched.
 * Both return 0 on success, -1 with adb_host_last_error() set. */
int adb_host_load_csv_count(const char *text, size_t bytes, int skip_lines, int n_cols, size_t *rows);
int adb_host_load_csv_emit(Column **cols, int n_cols);
#ifdef __cplusplus
}
#endif

#endif /* ADB_LOAD_API_H */
