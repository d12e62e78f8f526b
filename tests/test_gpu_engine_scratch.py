"""The engine's own device scratch, which grows on demand and is never shrunk.

Every operator that keeps scratch runs small, then large, then small inputs on a context that
starts with none: the first call allocates, the large one replaces the block with a bigger one,
and the last runs in a block larger than it needs.  Every answer is compared with the oracle or
numpy.  The same module drives the IPC peer path (adb_peer_create / _connect,
adb_peer_join_create / _connect) at world size 1, the path the one-process-per-GPU sharded runs
take."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from analytical_database_b200 import Engine
    Engine(0).close()                    # drop whatever an earlier module left: no scratch yet
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(autouse=True)
def default_forms(monkeypatch):
    for var in ("ADB_JOIN_PROBE", "ADB_SS_INTERVAL_LISTS"):
        monkeypatch.delenv(var, raising=False)


def test_select_scan(eng, rng):
    # the bitmap's first block covers ~8 M rows; 20 M need a larger one
    for n in (5000, 20_000_000, 5000):
        data = rng.integers(0, 1 << 20, n).astype(np.int32)
        col = eng.upload(data)
        pos, dc, h = eng.select_scan(col, n, 1000, 300_000, base=7)
        exp = np.flatnonzero((data >= 1000) & (data < 300_000)).astype(np.int32) + 7
        assert h == exp.size and np.array_equal(pos.to_host(h), exp), n
        for b in (col, pos, dc):
            b.free()


@pytest.mark.parametrize("form", ["pair lists", "interval lists"])
def test_shared_select(eng, port, rng, form):
    """Pair lists take batches at most four queries deep; six overlapping queries take interval
    lists."""
    for n in (4000, 3_000_000, 4000):
        data = rng.integers(0, 100_000, n).astype(np.int32)
        if form == "pair lists":
            lows = np.array([1000, 20_000, 30_000], np.int32)
            highs = np.array([40_000, 50_000, 90_000], np.int32)
        else:
            lows = (np.arange(6) * 1000).astype(np.int32)
            highs = (lows + 60_000).astype(np.int32)
        col = eng.upload(data)
        got = eng.shared_select(col, n, lows, highs)
        exp = port.shared_select(data, lows, highs)
        for q, ((buf, cnt), e) in enumerate(zip(got, exp)):
            assert cnt == e.size and np.array_equal(buf.to_host(cnt), e), (n, q)
            buf.free()
        col.free()


def test_index_sort(eng, rng):
    for n in (1000, 3_000_000, 1000):
        data = rng.integers(-2**31, 2**31 - 1, n, dtype=np.int64).astype(np.int32)
        col = eng.upload(data)
        dv, dp = eng.index_sort(col, n)
        order = np.argsort(data, kind="stable").astype(np.int32)
        assert np.array_equal(dp.to_host(n), order) and np.array_equal(dv.to_host(n), data[order]), n
        for b in (col, dv, dp):
            b.free()


def test_hash_join(eng, rng):
    """Many-one joins (unique build keys), so the expected pairs are one lookup per probe row in
    probe order.  The large one is past the partitioned probe's threshold (build >= 6 M rows,
    probe >= 4 M), the small ones take the direct probe."""
    for n1, n2 in ((2000, 1500), (6_500_000, 4_500_000), (2000, 1500)):
        k1 = rng.permutation(n1).astype(np.int32)
        k2 = rng.integers(0, int(1.25 * n1), n2).astype(np.int32)
        p1 = rng.permutation(n1).astype(np.int32)
        p2 = rng.permutation(n2).astype(np.int32)
        d = [eng.upload(x) for x in (k1, p1, k2, p2)]
        o1, o2, m = eng.join(d[0], d[1], n1, d[2], d[3], n2)
        row_of_key = np.full(int(1.25 * n1) + 1, -1, np.int64)
        row_of_key[k1] = np.arange(n1)
        hit = row_of_key[k2]
        e1, e2 = p1[hit[hit >= 0]], p2[hit >= 0]
        assert m == e1.size, (n1, n2)
        assert np.array_equal(o1.to_host(m), e1) and np.array_equal(o2.to_host(m), e2), (n1, n2)
        for b in d + [o1, o2]:
            b.free()


def test_csv_load(eng):
    r = np.random.default_rng(3)
    for rows in (50, 1_200_000, 50):
        vals = r.integers(-2**31, 2**31 - 1, (rows, 2), dtype=np.int64).astype(np.int32)
        text = ("a,b\n" + "\n".join(f"{x},{y}" for x, y in vals.tolist()) + "\n").encode()
        cols, n = eng.csv_load(text, 2)
        assert n == rows
        for i, c in enumerate(cols):
            assert np.array_equal(c.to_host(n), vals[:, i]), (rows, i)
            c.free()


def test_format_i32(eng, port, rng):
    for n in (100, 2_000_000, 100):
        vals = rng.integers(-2**31, 2**31 - 1, n, dtype=np.int64).astype(np.int32)
        d = eng.upload(vals)
        assert eng.format_i32(d, n) == port.print_i32(vals), n
        d.free()


def test_world_one_ipc_peer_path(eng, rng):
    """adb_peer_create(1, 0) + adb_peer_connect: the allreduce over the one rank's own mailbox
    equals adb_agg_combine.  adb_peer_join_create + _connect: adb_peer_exchange_pairs hands back
    the input pairs."""
    from analytical_database_b200.engine import _AggStruct
    lib = eng.lib
    handle = C.create_string_buffer(64)
    eng._ck(lib.adb_peer_create(1, 0, handle))
    try:
        eng._ck(lib.adb_peer_connect(handle.raw))
        agg_t = np.dtype([("sum", "<i8"), ("count", "<i8"), ("min", "<i4"), ("max", "<i4")])
        assert agg_t.itemsize == C.sizeof(_AggStruct)
        out = eng.alloc(2 * agg_t.itemsize)
        for k in (1, 3, 7):
            chunks = [rng.integers(-10**6, 10**6, int(rng.integers(1, 1000))) for _ in range(k)]
            parts = np.array([(c.sum(), c.size, c.min(), c.max()) for c in chunks], agg_t)
            d_parts = eng.upload(parts)
            p_parts = C.cast(d_parts.void(), C.POINTER(_AggStruct))
            plain, fused = _AggStruct(), _AggStruct()
            eng._ck(lib.adb_agg_combine(p_parts, k, eng.agg_ptr(out, 0), C.byref(plain)))
            eng._ck(lib.adb_agg_combine_allreduce(p_parts, k, eng.agg_ptr(out, 1), C.byref(fused)))
            whole = np.concatenate(chunks)
            expected = (int(whole.sum()), whole.size, int(whole.min()), int(whole.max()))
            assert (plain.sum, plain.count, plain.min, plain.max) == expected, k
            assert (fused.sum, fused.count, fused.min, fused.max) == expected, k
            d_parts.free()
        out.free()

        cap = 300_000
        jhandle = C.create_string_buffer(64)
        eng._ck(lib.adb_peer_join_create(cap, jhandle))
        eng._ck(lib.adb_peer_join_connect(jhandle.raw))
        for n in (1000, cap, 1000):
            val = rng.integers(-2**31, 2**31 - 1, n, dtype=np.int64).astype(np.int32)
            pos = rng.permutation(n).astype(np.int32)
            dv, dp = eng.upload(val), eng.upload(pos)
            for side in (0, 1):
                cnt, rv, rp = C.c_int64(-1), C.c_void_p(), C.c_void_p()
                eng._ck(lib.adb_peer_exchange_pairs(side, dv.i32(), dp.i32(), n, C.byref(cnt), C.byref(rv),
                                                    C.byref(rp)))
                assert cnt.value == n, (n, side)
                for ptr, exp in ((rv, val), (rp, pos)):
                    got = np.empty(n, np.int32)
                    eng._ck(lib.adb_download(got.ctypes.data_as(C.c_void_p), ptr, got.nbytes))
                    assert np.array_equal(got, exp), (n, side)
            dv.free()
            dp.free()
    finally:
        eng._ck(lib.adb_peer_destroy())
