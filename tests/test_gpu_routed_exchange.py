"""The routed exchange (include/adb_engine.h) at four engine contexts: one routed fetch and one
sharded hash join launch the same kernels, and the join runs the same stages, as when the fetch and
the join's probe each wrote out the exchange on their own.  The answers are checked as well."""
import ctypes as C
import re
from collections import Counter

import numpy as np
import pytest

from query_api import Api

pytestmark = pytest.mark.gpu

CONTEXTS = 4
# adb_launch_count_all() over one operator call, and the join's ADB_TRACE=1 stage lines with how
# often each appears (all four contexts), recorded on the inputs below
FETCH_LAUNCHES = 24
JOIN_LAUNCHES = 152
JOIN_STAGES = {stage: CONTEXTS for stage in (
    "build sort", "partition boundaries", "per-partition tables", "received keys in + probe",
    "answers back to row order + piece offsets", "expand (sharded)")}


@pytest.fixture(scope="module")
def api():
    with pytest.MonkeyPatch.context() as mp:
        # shim switches read at init that change how lists are cut, staged or written
        for var in ("ADB_SHIM_MIRROR", "ADB_SHIM_EAGER", "ADB_SHARD_MIN_ROWS", "ADB_REBALANCE_MIN"):
            mp.delenv(var, raising=False)
        a = Api()
        assert a.lib.adb_host_init_multi(CONTEXTS) == 0, a.lib.adb_host_last_error()
        yield a
        a.lib.adb_host_shutdown()


@pytest.fixture(scope="module")
def launch_count():
    import analytical_database_b200 as adb
    lib = C.CDLL(adb.lib_path())                      # the engine libadb_query.so drives
    lib.adb_launch_count_all.restype = C.c_int64
    return lib.adb_launch_count_all


@pytest.fixture(autouse=True)
def default_forms(monkeypatch):
    for var in ("ADB_JOIN_PROBE", "ADB_TRACE", "ADB_FETCH_ROUTE_MIN"):
        monkeypatch.delenv(var, raising=False)


def test_routed_fetch_launches(api, launch_count, monkeypatch):
    monkeypatch.setenv("ADB_FETCH_ROUTE_MIN", "0")
    rng = np.random.default_rng(7)
    other = rng.integers(-10**6, 10**6, 100_003).astype(np.int32)
    perm = rng.permutation(other.size)[:7777].astype(np.int32)
    col, hp = api.column(other), api.host_result(perm)
    api.drop(api.fetch_column(col, C.pointer(hp)))    # the first call also uploads the column
    before = launch_count()
    f = api.fetch_column(col, C.pointer(hp))
    launches = launch_count() - before
    assert np.array_equal(api.tuples(f), other[perm])
    api.drop(f)
    assert launches == FETCH_LAUNCHES


def test_sharded_join_launches_and_stages(api, port, launch_count, capfd, monkeypatch):
    monkeypatch.setenv("ADB_TRACE", "1")
    rng = np.random.default_rng(11)
    n1, n2 = 70_000, 50_000
    k1, k2 = rng.integers(1, 30_000, n1).astype(np.int32), rng.integers(1, 30_000, n2).astype(np.int32)
    p1, p2 = rng.permutation(n1).astype(np.int32), rng.permutation(n2).astype(np.int32)
    R = [C.pointer(api.host_result(x)) for x in (k1, p1, k2, p2)]
    for r in api.join("hash_join", *R):               # the first call also sizes the exchange
        api.drop(r)
    capfd.readouterr()
    before = launch_count()
    o1, o2 = api.join("hash_join", *R)
    launches = launch_count() - before
    trace = capfd.readouterr().err
    stages = Counter(m.group(1) for m in re.finditer(r"^\[adb trace\] (.*?)\s+-?[\d.]+ ms$", trace, re.M))
    e1, e2 = port.hash_join(k1, p1, k2, p2)
    assert np.array_equal(api.tuples(o1), e1) and np.array_equal(api.tuples(o2), e2)
    api.drop(o1), api.drop(o2)
    assert launches == JOIN_LAUNCHES
    assert dict(stages) == JOIN_STAGES
