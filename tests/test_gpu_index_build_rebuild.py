"""The index build across several contexts in the shim's other situations: the rebuild after an
update and a delete, ADB_INDEX_TIES=reference (which keeps the one-context sort), and BASELINE
config 3 at full size on eight devices.  Each test brings up its own shim."""
import ctypes as C
import os

import numpy as np
import pytest

from query_api import Api, Column

pytestmark = pytest.mark.gpu

INT_MIN, INT_MAX = -(1 << 31), (1 << 31) - 1


@pytest.fixture
def five():
    a = Api()
    assert a.lib.adb_host_init_multi(5) == 0, a.lib.adb_host_last_error()
    yield a
    a.lib.adb_host_shutdown()


def test_rebuild_after_update_and_delete_at_five_contexts(five, rng):
    """relational_update / relational_delete rebuild the index (test_gpu_updates' generator model)."""
    api = five
    n = 60_013
    key = rng.integers(0, 5000, n).astype(np.int32)
    pay = rng.integers(0, 500, n).astype(np.int32)
    cols = api.table([key, pay], {0: (False, False)})
    ptrs = (C.POINTER(Column) * 2)(*[C.pointer(c) for c, _ in cols])
    api.build_index(cols, 0)
    model = [key.copy(), pay.copy()]
    u = api.select_column(cols[1][0], 10, 40)
    assert api.lib.adb_host_relational_update(ptrs, 2, 0, u, -77) == 0, api.lib.adb_host_last_error()
    model[0][(model[1] >= 10) & (model[1] < 40)] = -77
    api.drop(u)
    d = api.select_column(cols[1][0], 300, 380)
    assert api.lib.adb_host_relational_delete(ptrs, 2, d) == 0, api.lib.adb_host_last_error()
    keep = ~((model[1] >= 300) & (model[1] < 380))
    model = [m[keep] for m in model]
    api.drop(d)
    m = model[0].size
    assert cols[0][0].row_count == m
    ix = cols[0][0].index.contents
    order = np.argsort(model[0], kind="stable")
    assert np.array_equal(np.ctypeslib.as_array(ix.values, shape=(m,)), model[0][order])
    assert np.array_equal(np.ctypeslib.as_array(ix.positions, shape=(m,)), order.astype(np.uint64))
    for lo, hi in [(-77, -76), (100, 2000), (INT_MIN, 7)]:
        s = api.select_column(cols[0][0], lo, hi)
        f = api.fetch_column(cols[1][0], s)
        v = model[0][order]
        exp = order[np.searchsorted(v, lo):np.searchsorted(v, hi)].astype(np.int32)
        assert np.array_equal(api.tuples(s), exp) and np.array_equal(api.tuples(f), model[1][exp])
        api.drop(s), api.drop(f)


def test_reference_ties_keep_the_reference_order_at_three_contexts(cpu_ref, rng):
    old = os.environ.get("ADB_INDEX_TIES")
    os.environ["ADB_INDEX_TIES"] = "reference"
    try:
        api = Api()
        assert api.lib.adb_host_init_multi(3) == 0, api.lib.adb_host_last_error()
        try:
            key = rng.integers(0, 300, 50_021).astype(np.int32)
            cols = api.table([np.arange(key.size, dtype=np.int32), key], {1: (False, False)})
            values, positions = api.build_index(cols, 1)
            ev, ep = cpu_ref.index_sort(key)
            assert np.array_equal(values, ev) and np.array_equal(positions, ep)
        finally:
            api.lib.adb_host_shutdown()
    finally:
        if old is None:
            os.environ.pop("ADB_INDEX_TIES", None)
        else:
            os.environ["ADB_INDEX_TIES"] = old


@pytest.fixture(scope="module")
def cpu_ref():
    from oracle import oracle
    return oracle.reference("O2") or oracle.port()


def test_config3_full_size_at_eight_contexts():
    """BASELINE config 3 (500 M permutation keys) at 8 contexts, one per device; the 1- and
    2-context runs are test_gpu_index_build's.  Needs eight devices."""
    import analytical_database_b200 as adb
    import query_api as q
    n, mul, add, G = 500_000_000, 387_420_489, 123_456_789, 8
    inv = pow(mul, -1, n)
    api = Api()
    assert api.lib.adb_host_init_multi(G) == 0, api.lib.adb_host_last_error()
    eng = adb.Engine(0)
    if eng.lib.adb_device_count() < G:
        api.lib.adb_host_shutdown()
        pytest.skip("fewer than eight devices")
    S = ((n + G - 1) // G + 31) // 32 * 32
    ptrs, bufs = (C.c_void_p * G)(), []
    for g in range(G):
        eng._ck(eng.lib.adb_ctx_select(g))
        b = eng.alloc_i32(max(1, min(S, n - g * S)))
        eng._ck(eng.lib.adb_synth_affine(b.i32(), max(1, min(S, n - g * S)), g * S, mul, add, n))
        eng.sync()
        bufs.append(b)
        ptrs[g] = b.ptr
    eng._ck(eng.lib.adb_ctx_select(0))
    key = q.Column()
    key.name, key.row_count, key.has_index = b"key", n, True
    assert api.lib.adb_host_column_adopt_shards(C.byref(key), ptrs, S) == 0
    arr = (C.POINTER(q.Column) * 1)(C.pointer(key))
    assert api.lib.adb_host_index_build(arr, 1, 0) == 0, api.lib.adb_host_last_error()
    hv = np.ctypeslib.as_array(key.index.contents.values, shape=(n,))
    hp = np.ctypeslib.as_array(key.index.contents.positions, shape=(n,))
    for a0 in (0, n // 3, n - (1 << 18)):
        vs = np.arange(a0, a0 + (1 << 18), dtype=np.int64)
        assert np.array_equal(hv[a0:a0 + (1 << 18)], vs.astype(np.int32))
        assert np.array_equal(hp[a0:a0 + (1 << 18)], ((vs - add) % n * inv % n).astype(np.uint64))
    ix = key.index.contents
    for ptr in (ix.values, ix.positions, key.index):
        q._libc.free(C.cast(ptr, C.c_void_p))
    api.lib.adb_host_shutdown()
