"""The stand-in types of include/adb_query_api.h must be byte-compatible with the
reference's headers (SURVEY.md section 8a "keep byte-compatible"), and libadb_query.so must
export the whole operator API.  CPU-only."""
import ctypes as C
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_INC = "/root/reference/src/include"

PROBE = r'''
#include <stdio.h>
#include <stddef.h>
#include "adb_query_api.h"
#define S(t) printf(#t " %zu\n", sizeof(t))
#define O(t, f) printf(#t "." #f " %zu\n", offsetof(t, f))
int main(void) {
    S(Column); O(Column, data); O(Column, fd); O(Column, row_count); O(Column, sorted);
    O(Column, clustered); O(Column, has_index); O(Column, index); O(Column, btree_node);
    O(Column, histogram); O(Column, max); O(Column, min);
    S(ColumnIndex); O(ColumnIndex, values); O(ColumnIndex, positions);
    S(Result); O(Result, num_tuples); O(Result, data_type); O(Result, payload);
    S(Status); O(Status, code); O(Status, error_message);
    S(GeneralizedColumn); O(GeneralizedColumn, column_type); O(GeneralizedColumn, column_pointer);
    S(SelectOperator); O(SelectOperator, handle); O(SelectOperator, low); O(SelectOperator, high);
    O(SelectOperator, has_low); O(SelectOperator, has_high); O(SelectOperator, column);
    O(SelectOperator, col_result); O(SelectOperator, pos_result); O(SelectOperator, comparator);
    printf("enums %d %d %d %d %d %d %d %d %d %d\n", INT, LONG, FLOAT, DOUBLE, OK, ERROR, RESULT,
           COLUMN, COLUMN_SELECT, RESULT_SELECT);
    printf("consts %d %d %d\n", MAX_SIZE_NAME, HANDLE_MAX_SIZE, LONG_INT_LENGTH);
    return 0;
}
'''


def _run_probe(extra):
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "p.c"), os.path.join(d, "p")
        open(src, "w").write(PROBE)
        subprocess.run(["gcc", "-std=c99", "-w", "-I" + os.path.join(ROOT, "include")] + extra +
                       ["-o", exe, src], check=True)
        return subprocess.run([exe], check=True, stdout=subprocess.PIPE).stdout.decode()


def test_stand_in_types_have_the_expected_layout():
    out = dict(line.rsplit(" ", 1) for line in _run_probe([]).splitlines() if not line.startswith(("enums", "consts")))
    assert out["Column"] == "128" and out["Result"] == "24" and out["SelectOperator"] == "136"
    assert out["Column.data"] == "64" and out["Column.row_count"] == "80" and out["Column.index"] == "96"


def test_stand_in_types_match_the_reference_headers():
    """tests/golden/reference_layout.txt is the probe's output compiled against the reference's
    own headers (recorded from the stand-ins at a commit where the two outputs were equal); where
    the reference headers are present the probe is compiled against them as well."""
    mine = _run_probe([])
    with open(os.path.join(ROOT, "tests", "golden", "reference_layout.txt")) as f:
        assert mine == f.read()
    if os.path.isdir(REF_INC):
        assert mine == _run_probe(["-DADB_WITH_REFERENCE_HEADERS", "-I" + REF_INC])


def test_ctypes_view_matches_the_header():
    import query_api as q
    out = dict(line.rsplit(" ", 1) for line in _run_probe([]).splitlines() if not line.startswith(("enums", "consts")))
    for name in ("Column", "ColumnIndex", "Result", "Status", "GeneralizedColumn", "SelectOperator"):
        assert C.sizeof(getattr(q, name)) == int(out[name]), name
    assert q.Column.row_count.offset == int(out["Column.row_count"])
    assert q.SelectOperator.column.offset == int(out["SelectOperator.column"])


def test_operator_library_exports_the_whole_api():
    import analytical_database_b200 as adb
    import query_api as q
    if not os.path.exists(q.LIB):
        adb.build_native()
    lib = C.CDLL(q.LIB)
    missing = [n for n in list(q.OPERATORS) + list(q.HOOKS) if not hasattr(lib, n)]
    assert not missing, missing
    # every function include/adb_query_api.h declares is covered by the list above
    import re
    src = open(os.path.join(ROOT, "include", "adb_query_api.h")).read()
    declared = set(re.findall(r"^\w[\w \*]*?\b(\w+)\(", src, flags=re.M)) - {"defined"}
    assert declared <= set(q.OPERATORS) | set(q.HOOKS), declared - set(q.OPERATORS) - set(q.HOOKS)


NO_DEVICE_PROBE = r'''
import ctypes as C
import numpy as np
import query_api as q
api = q.Api()
col = api.column(np.arange(10, dtype=np.int32))
st = q.Status(99, None)
lo = C.c_int(1)
assert not api.lib.select_column(C.byref(col), C.byref(lo), None, C.byref(st))
assert st.code == q.ERROR and b"no CPU fallback" in api.lib.adb_host_last_error()
'''


def test_operators_fail_loudly_without_a_device():
    """In a process that sees no CUDA device (none visible on a GPU host either)."""
    import analytical_database_b200 as adb
    import query_api as q
    if not os.path.exists(q.LIB):
        adb.build_native()
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    subprocess.run([sys.executable, "-c", NO_DEVICE_PROBE], cwd=os.path.join(ROOT, "tests"), env=env, check=True)
