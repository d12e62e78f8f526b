"""CPU-side check of include/adb_load_api.h (the bulk-load hooks of the operator-API host):
libadb_query.so exports every function the header declares, and the ctypes binding the GPU
tests use (tests/test_gpu_load_csv.py) covers all of them."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_load_hooks_are_exported_and_bound():
    import analytical_database_b200 as adb
    import query_api as q
    from test_gpu_load_csv import LOAD_HOOKS
    if not os.path.exists(q.LIB):
        adb.build_native()
    src = open(os.path.join(ROOT, "include", "adb_load_api.h")).read()
    declared = set(re.findall(r"^\w[\w \*]*?\b(\w+)\(", src, flags=re.M))
    assert declared == set(LOAD_HOOKS)
    lib = C.CDLL(q.LIB)
    assert all(hasattr(lib, n) for n in declared)
