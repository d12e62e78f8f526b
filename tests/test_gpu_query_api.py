"""GPU parity of the drop-in operator API (host/query_shim.c -> libadb_query.so): the
reference's own function names (src/include/query.h:20-44) driven the way the dispatcher
drives them (src/server.c:137-435), compared bit for bit with the reference's objects
(oracle/_ref) or the oracle port on the same seeded inputs."""
import ctypes as C

import numpy as np
import pytest

from query_api import Api, ERROR, GeneralizedColumn, RESULT, SelectOperator, Status

pytestmark = pytest.mark.gpu
I32MAX = 2**31 - 1


@pytest.fixture(scope="module", params=[1, 2, 3, 4], ids=["1gpu", "2gpus", "3gpus", "4gpus"])
def api(request):
    """The whole module runs three times: on one GPU, and with every column row-range sharded
    over 2 and 3 engine contexts driven from ONE process (host/query_shim.c, adb_host_init_multi).
    On a 1-GPU box the contexts share the device -- same host code, same kernels, same peer
    exchange, the mailboxes simply live in one HBM."""
    import os
    os.environ["ADB_REBALANCE_MIN"] = "1000"      # index-ordered lists of the test sizes get re-cut too
    a = Api()
    if request.param == 1:
        assert a.lib.adb_host_init(0) == 0, a.lib.adb_host_last_error()
    else:
        assert a.lib.adb_host_init_multi(request.param) == 0, a.lib.adb_host_last_error()
    assert a.lib.adb_host_gpus() == request.param
    yield a
    a.lib.adb_host_shutdown()


@pytest.fixture(scope="module")
def cpu():
    from oracle import oracle
    return oracle.reference("O2") or oracle.port()


def table(rng, n):
    """milestone1.py:112-121: col1,col2 in [-n/2, n/2), col3 in [0,100), col4 near INT_MAX."""
    return (rng.integers(-n // 2, n // 2, n).astype(np.int32),
            rng.integers(-n // 2, n // 2, n).astype(np.int32),
            rng.integers(0, 100, n).astype(np.int32),
            rng.integers(I32MAX - 10000, I32MAX, n, dtype=np.int64).astype(np.int32))


@pytest.mark.parametrize("n", [1, 1000, 4097, 250_003])
def test_select_fetch_aggregate_print(api, cpu, rng, n):
    c1, c2, c3, c4 = table(rng, n)
    col1, col4 = api.column(c1), api.column(c4)
    for lo, hi in [(None, None), (None, 20), (-17, None), (-n // 8, n // 8), (5, 5), (n, None)]:
        s = api.select_column(col1, lo, hi)
        epos = cpu.select_scan(c1, lo, hi)
        assert s.contents.num_tuples == epos.size and s.contents.data_type == 0
        assert np.array_equal(api.tuples(s), epos)
        f = api.fetch_column(col4, s)
        evals = cpu.fetch(c4, epos)
        assert np.array_equal(api.tuples(f), evals)
        a = api.sum_result(f)
        assert a.contents.data_type == 1 and a.contents.num_tuples == 1
        assert int(api.tuples(a)[0]) == cpu.sum(evals)
        assert api.print(a) == "%d" % cpu.sum(evals)                   # "%ld", query.c:284
        if epos.size:
            avg, mn, mx = api.unary("average", f), api.unary("min", f), api.unary("max", f)
            assert api.tuples(avg)[0].tobytes() == np.float64(cpu.avg(evals)).tobytes()
            assert int(api.tuples(mn)[0]) == cpu.min(evals) and int(api.tuples(mx)[0]) == cpu.max(evals)
            assert api.print(avg) == "%.2f" % cpu.avg(evals)           # query.c:293
            assert api.print(mn, mx) == "%d,%d" % (cpu.min(evals), cpu.max(evals))   # query.c:255-260
            # short results are rendered on the host, >= 4096 tuples on the device
            assert api.print(f) == "\n".join(str(int(v)) for v in evals)
            if 4096 <= epos.size <= 100_000:                          # two long results: column-major, ','
                assert api.print(s, f) == "\n".join(map(str, epos.tolist())) + "," + \
                    "\n".join(map(str, evals.tolist()))
            for r in (avg, mn, mx):
                api.drop(r)
        else:
            avg = api.unary("average", f)
            assert np.isnan(api.tuples(avg)[0]) and api.print(avg) == "-nan"   # A7: empty avg
            assert api.print(f) == ""
            api.drop(avg)
        for r in (s, f, a):
            api.drop(r)
    assert api.lib.adb_host_live_device_results() == 0


def test_sum_over_a_whole_column_and_ewise(api, cpu, rng):
    n = 123_457
    c1, c2, c3, c4 = table(rng, n)
    col1, col2, col4 = api.column(c1), api.column(c2), api.column(c4)
    a = api.sum_column(col4)                                           # query.c:336-341
    assert int(api.tuples(a)[0]) == cpu.sum_column(c4)
    s = api.select_column(col1, -1000, 30000)
    f2, f4 = api.fetch_column(col2, s), api.fetch_column(col4, s)
    epos = cpu.select_scan(c1, -1000, 30000)
    e2, e4 = cpu.fetch(c2, epos), cpu.fetch(c4, epos)
    ad, sb = api.binary("add", f2, f4), api.binary("sub", f2, f4)      # wraps in int32 (A7)
    assert np.array_equal(api.tuples(ad), cpu.add(e2, e4))
    assert np.array_equal(api.tuples(sb), cpu.sub(e2, e4))
    # chained select over an intermediate: s2=select(s1,f1,lo,hi), milestone1.py:300
    s2 = api.select_result(f2, s, -500, 500)
    assert np.array_equal(api.tuples(s2), cpu.select_result(e2, epos, -500, 500))
    s3 = api.select_result(f2, s, None, None)
    assert np.array_equal(api.tuples(s3), epos)
    for r in (a, s, f2, f4, ad, sb, s2, s3):
        api.drop(r)
    assert api.lib.adb_host_live_device_results() == 0


def test_host_payload_operands_are_staged(api, cpu, rng):
    """A Result built by foreign code (plain host int array) is a valid operand."""
    n = 5000
    c1, c2, _, _ = table(rng, n)
    col2 = api.column(c2)
    pos = np.sort(rng.choice(n, 700, replace=False)).astype(np.int32)
    hp = api.host_result(pos)
    f = api.fetch_column(col2, C.pointer(hp))
    assert np.array_equal(api.tuples(f), c2[pos])
    hv = api.host_result(c2[pos])
    s = api.select_result(C.pointer(hv), C.pointer(hp), 0, None)
    assert np.array_equal(api.tuples(s), cpu.select_result(c2[pos], pos, 0, None))
    api.drop(f)
    api.drop(s)


@pytest.mark.parametrize("kind", ["sorted_unclustered", "btree_unclustered", "sorted_clustered",
                                  "btree_clustered"])
def test_indexed_select_matches_the_reference_index_path(api, cpu, rng, kind):
    """select_column routes clustered / indexed columns through the ColumnIndex
    (query.c:203-217); the shim uploads the index the reference built (its own quicksort
    tie order, SURVEY.md A3) and must return positions in exactly the reference's order."""
    n = 60_000
    data = rng.integers(0, 3000, n).astype(np.int32)                   # heavy duplicates
    values, positions = cpu.index_sort(data)
    clustered = kind.endswith("_clustered")
    if clustered:                                                      # index.c:119-135: identity
        positions = np.arange(n, dtype=np.uint64)
    col = api.column(data, index=(values, positions), sorted_=kind.startswith("sorted"),
                     clustered=clustered)
    vmin = int(values[0])
    for lo, hi in [(vmin, vmin + 1), (10, 20), (100, 100), (2990, 5000), (vmin, 4000), (1500, 1400),
                   (17, 18), (2999, 3000)]:
        s = api.select_column(col, lo, hi)
        exp, undefined = cpu.select_sorted_index(values, positions, lo, hi)
        assert not undefined
        assert np.array_equal(api.tuples(s), exp), (kind, lo, hi)
        api.drop(s)
    # oracle-undefined inputs (the reference crashes): scan semantics in index order
    for lo, hi in [(-50, 5), (None, 7), (2995, None)]:
        s = api.select_column(col, lo, hi)
        got = api.tuples(s)
        scan = cpu.select_scan(data, lo, hi)
        if clustered:
            v = values[got]                   # positions are identity over the sorted copy
            assert got.size == scan.size and np.all((v >= (lo if lo is not None else -2**31)))
        else:
            assert np.array_equal(np.sort(got), scan), (kind, lo, hi)
        api.drop(s)


def test_shared_select(api, cpu, rng):
    n, q = 200_003, 100
    data = rng.integers(0, n, n).astype(np.int32)
    col = api.column(data)
    lows = rng.integers(0, n, q)
    highs = lows + rng.integers(0, n // 50, q)
    highs[3] = lows[3] - 5                                             # an empty range
    res = api.shared_select(col, lows, highs)
    from oracle import oracle
    exp = oracle.port().shared_select(data, lows, highs)
    for r, e in zip(res, exp):
        assert np.array_equal(api.tuples(r), e)
        api.drop(r)
    # has_low / has_high are ignored exactly as query.c:474 does
    ops = (SelectOperator * 1)()
    ops[0].low, ops[0].high, ops[0].has_low, ops[0].has_high = 10, 500, 0, 0
    st = Status(99, None)
    r = api.lib.shared_select(ops, 1, C.byref(col), C.byref(st))
    assert st.code == 0 and np.array_equal(api.tuples(r[0]), cpu.select_scan(data, 10, 500))


@pytest.mark.parametrize("nested", [False, True])
def test_joins(api, cpu, rng, nested):
    n1, n2 = (3000, 1200) if nested else (90_000, 40_000)
    v1 = rng.integers(1, 20_000, n1).astype(np.int32)
    v2 = rng.integers(1, 20_000, n2).astype(np.int32)
    p1 = rng.permutation(n1).astype(np.int32)
    p2 = rng.permutation(n2).astype(np.int32)
    R = [C.pointer(api.host_result(x)) for x in (v1, p1, v2, p2)]
    name = "nested_loop_join" if nested else "hash_join"
    o1, o2 = api.join(name, *R)
    e1, e2 = getattr(cpu, name)(v1, p1, v2, p2)
    assert o1.contents.num_tuples == e1.size
    assert np.array_equal(api.tuples(o1), e1) and np.array_equal(api.tuples(o2), e2)
    api.drop(o1)
    api.drop(o2)


def test_error_behaviour(api, rng):
    """Failures set code = ERROR and return NULL (the dispatcher replies "Failed",
    src/server.c:171-174); nothing is computed on the host instead."""
    a, b = api.host_result(np.arange(10)), api.host_result(np.arange(4))
    st = Status(99, None)
    assert not api.lib.add(C.pointer(a), C.pointer(b), C.byref(st)) and st.code == ERROR
    col = api.column(np.arange(100, dtype=np.int32))
    ops = (SelectOperator * 151)()
    st = Status(99, None)
    assert not api.lib.shared_select(ops, 151, C.byref(col), C.byref(st)) and st.code == ERROR
    flagged = api.column(np.arange(100, dtype=np.int32))
    flagged.has_index = True                                           # but no ColumnIndex
    st = Status(99, None)
    lo = C.c_int(1)
    assert not api.lib.select_column(C.byref(flagged), C.byref(lo), C.byref(lo), C.byref(st))
    assert st.code == ERROR and b"ColumnIndex" in api.lib.adb_host_last_error()


def test_column_reupload_after_insert(api, cpu):
    """insert_row appends in place or re-mmaps (db_manager.c:164-199): the shim notices a
    changed row_count / data pointer and refreshes the HBM copy."""
    buf = np.arange(1000, dtype=np.int32)
    col = api.column(buf[:600])
    s = api.select_column(col, 0, 10_000)
    assert s.contents.num_tuples == 600
    col.row_count = 1000                                               # 400 rows appended in place
    s2 = api.select_column(col, 0, 10_000)
    assert s2.contents.num_tuples == 1000
    api.drop(s)
    api.drop(s2)


def test_payload_registry_reclaims_on_address_reuse(api):
    """No patch and no interposer: freeing a payload behind the shim's back leaks HBM only
    until malloc hands the address out again."""
    import query_api
    col = api.column(np.arange(50_000, dtype=np.int32))
    base = api.lib.adb_host_live_device_results()
    freed = set()
    for _ in range(20):
        s = api.select_column(col, 100, 200)                           # same size -> same malloc bin
        freed.add(s.contents.payload)
        query_api._libc.free(s.contents.payload)                       # plumbing-style free, no hook
        query_api._libc.free(C.cast(s, C.c_void_p))
    assert api.lib.adb_host_live_device_results() <= base + 3
    # the same with a deferred select + fetch pending behind the freed payloads: the next chain
    # is still answered correctly, whatever addresses malloc recycles
    data = np.arange(50_000, dtype=np.int32)
    for i in range(20):
        lo, hi = 100 + i, 5000 + 3 * i
        s = api.select_column(col, lo, hi)
        f = api.fetch_column(col, s)
        if i % 2:
            a = api.sum_result(f)
            assert int(api.tuples(a)[0]) == int(data[lo:hi].sum())
            api.drop(a)
        for h in (f, s) if i % 3 else (s, f):
            freed.add(h.contents.payload)
            query_api._libc.free(h.contents.payload)
            query_api._libc.free(C.cast(h, C.c_void_p))
    s = api.select_column(col, 7, 9000)
    f = api.fetch_column(col, s)
    a = api.unary("max", f)
    assert int(api.tuples(a)[0]) == 8999 and np.array_equal(api.tuples(s), np.arange(7, 9000))
    for h in (s, f, a):
        api.drop(h)
    # these payloads had 40 different sizes: whether malloc has handed their addresses out again
    # by now depends on its bins and the process's malloc policy (the shim's own mallopt), so
    # only the upper bound is fixed -- nothing beyond the 40 leaked-on-purpose entries is live
    assert api.lib.adb_host_live_device_results() <= base + 3 + 40
    release_leaked(api, freed)


def release_leaked(api, freed):
    """Late release hooks for payloads a test freed behind the shim's back (none of them is a live
    Result's any more): the entries still registered under those addresses go, so that a later
    malloc cannot reclaim one of them inside another test and shift that test's live count."""
    for p in freed:
        api.lib.adb_host_payload_freed(p)


# ---- deferred select (SURVEY.md 8f rank 3): every order in which the plumbing can touch the
# handles of s=select / f=fetch / a=agg(f) gives the eager answer ---------------------------
def _chain_inputs(rng, n):
    c1, _c2, _c3, c4 = table(rng, n)
    return c1, c4, -n // 6, n // 5


@pytest.mark.parametrize("n", [33, 4097, 300_001])
@pytest.mark.parametrize("agg", ["sum", "average", "min", "max"])
def test_deferred_chain_resolves_in_the_aggregate(api, cpu, rng, n, agg):
    c1, c4, lo, hi = _chain_inputs(rng, n)
    col1, col4 = api.column(c1), api.column(c4)
    epos = cpu.select_scan(c1, lo, hi)
    evals = cpu.fetch(c4, epos)
    s = api.select_column(col1, lo, hi)
    assert s.contents.num_tuples == epos.size            # known before anything is written
    f = api.fetch_column(col4, s)
    assert f.contents.num_tuples == epos.size
    a = api.sum_result(f) if agg == "sum" else api.unary(agg, f)
    got = api.tuples(a)[0]
    if agg == "sum":
        assert int(got) == cpu.sum(evals)
    elif agg == "average":
        assert got.tobytes() == np.float64(cpu.avg(evals)).tobytes()
    else:
        assert int(got) == getattr(cpu, agg)(evals)
    # the handles the aggregate resolved on the way are the eager ones
    assert np.array_equal(api.tuples(s), epos)
    assert np.array_equal(api.tuples(f), evals)
    # and stay usable: a second aggregate, a second fetch, a select over the pair
    assert int(api.tuples(api.unary("max", f))[0]) == cpu.max(evals)
    f2 = api.fetch_column(col1, s)
    assert np.array_equal(api.tuples(f2), cpu.fetch(c1, epos))
    s2 = api.select_result(f2, s, 0, None)
    assert np.array_equal(api.tuples(s2), cpu.select_result(cpu.fetch(c1, epos), epos, 0, None))
    for r in (s, f, a, f2, s2):
        api.drop(r)


def test_deferred_handles_under_every_other_first_use(api, cpu, rng):
    n = 70_001
    c1, c4, lo, hi = _chain_inputs(rng, n)
    col1, col4 = api.column(c1), api.column(c4)
    epos = cpu.select_scan(c1, lo, hi)
    evals = cpu.fetch(c4, epos)
    live0 = api.lib.adb_host_live_device_results()

    # the select is read first
    s = api.select_column(col1, lo, hi)
    assert np.array_equal(api.tuples(s), epos)
    api.drop(s)
    # the fetch is read first
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    assert np.array_equal(api.tuples(f), evals)
    assert np.array_equal(api.tuples(s), epos)
    api.drop(s), api.drop(f)
    # the select is released while the fetch is pending (s is re-bound, client_context.c:31-45)
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    api.drop(s)
    a = api.sum_result(f)
    assert int(api.tuples(a)[0]) == cpu.sum(evals)
    assert np.array_equal(api.tuples(f), evals)
    api.drop(f), api.drop(a)
    # the fetch is released while pending, the select lives on
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    api.drop(f)
    assert np.array_equal(api.tuples(s), epos)
    api.drop(s)
    # both released untouched
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    api.drop(f), api.drop(s)
    # another select takes the bitmap over
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    t = api.select_column(col4, None, I32MAX - 5000)
    a = api.unary("min", f)
    assert int(api.tuples(a)[0]) == cpu.min(evals)
    assert np.array_equal(api.tuples(t), cpu.select_scan(c4, None, I32MAX - 5000))
    assert np.array_equal(api.tuples(s), epos)
    for r in (s, f, t, a):
        api.drop(r)
    # two fetches of one pending select, print, add, a batch and a join in between
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    g = api.fetch_column(col1, s)
    d = api.binary("sub", f, g)
    assert np.array_equal(api.tuples(d), (evals.astype(np.int64) - cpu.fetch(c1, epos)).astype(np.int32))
    for r in (s, f, g, d):
        api.drop(r)
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    assert api.print(f) == "\n".join(str(int(v)) for v in evals)
    api.drop(s), api.drop(f)
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    batch = api.shared_select(col1, [lo, 0], [hi, 10])
    assert np.array_equal(api.tuples(batch[0]), epos)
    a = api.sum_result(f)
    assert int(api.tuples(a)[0]) == cpu.sum(evals)
    for r in (s, f, a, *batch):
        api.drop(r)
    # the column is invalidated (insert_row re-mmaps it, db_manager.c:178-186) while pending
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    api.lib.adb_host_column_invalidate(C.byref(col4))
    api.lib.adb_host_column_invalidate(C.byref(col1))
    a = api.sum_result(f)
    assert int(api.tuples(a)[0]) == cpu.sum(evals)
    assert np.array_equal(api.tuples(s), epos)
    for r in (s, f, a):
        api.drop(r)
    assert api.lib.adb_host_live_device_results() == live0


def test_deferred_select_survives_a_foreign_engine_select(api, cpu, rng):
    """Another user of the engine in the same process overwrites the pending bitmap: the
    shim notices (adb_select_generation) and re-runs the predicate pass."""
    import analytical_database_b200 as adb
    n = 50_021
    c1, c4, lo, hi = _chain_inputs(rng, n)
    col1, col4 = api.column(c1), api.column(c4)
    epos = cpu.select_scan(c1, lo, hi)
    evals = cpu.fetch(c4, epos)
    eng = adb.Engine(0)
    other = eng.upload(np.arange(1000, dtype=np.int32))
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    pos, cnt = eng.select_exact(other, 1000, 10, 20)
    assert cnt == 10
    a = api.sum_result(f)
    assert int(api.tuples(a)[0]) == cpu.sum(evals)
    assert np.array_equal(api.tuples(s), epos) and np.array_equal(api.tuples(f), evals)
    for r in (s, f, a):
        api.drop(r)
    # ... or consumes the pending count outright (an emit without a count of its own)
    s = api.select_column(col1, lo, hi)
    f = api.fetch_column(col4, s)
    stolen = eng.alloc_i32(epos.size)
    eng._ck(eng.lib.adb_select_emit(None, 0, stolen.i32()))
    # (the foreign caller sits on context 0: with several GPUs it steals the first shard's rows)
    G = api.lib.adb_host_gpus()
    shard_rows = ((n + G - 1) // G + 31) // 32 * 32
    m = int(np.searchsorted(epos, shard_rows)) if G > 1 else epos.size
    assert np.array_equal(stolen.to_host(epos.size)[:m], epos[:m])
    a = api.unary("max", f)
    assert int(api.tuples(a)[0]) == cpu.max(evals)
    assert np.array_equal(api.tuples(s), epos) and np.array_equal(api.tuples(f), evals)
    for r in (s, f, a):
        api.drop(r)
    # the engine-level deferred form agrees with the fused chain
    d1, d4 = eng.upload(c1), eng.upload(c4)
    p_, v_, h_, agg = eng.select_fetch_agg_deferred(d1, d4, n, lo, hi)
    assert h_ == epos.size and agg.sum == cpu.sum(evals) and agg.count == epos.size
    assert agg.min == cpu.min(evals) and agg.max == cpu.max(evals)
    assert np.array_equal(p_.to_host(h_), epos) and np.array_equal(v_.to_host(h_), evals)


def test_random_walk_over_the_operator_api(api, cpu):
    """A seeded random sequence of 600 operator calls over a pool of handles, every observable
    value compared with a numpy model built from the oracle: whatever order the plumbing uses,
    re-binds and releases handles in (client_context.c:31-45,76-90), deferred or not."""
    rng = np.random.default_rng(2026)
    n = 60_000
    data = [rng.integers(-n // 2, n // 2, n).astype(np.int32) for _ in range(3)]
    cols = [api.column(d) for d in data]
    live0 = api.lib.adb_host_live_device_results()
    pos, val = [], []                      # (handle, model array) pools

    def bounds():
        a, b = sorted(int(x) for x in rng.integers(-n // 2 - 10, n // 2 + 10, 2))
        return [(a, b), (None, b), (a, None), (a, a + int(rng.integers(0, 50)))][int(rng.integers(0, 4))]

    def check(h, model):
        assert h.contents.num_tuples == model.size
        assert np.array_equal(api.tuples(h), model)

    for step in range(600):
        op = int(rng.integers(0, 12))
        if op <= 1 or not pos:                                   # select over a base column
            c = int(rng.integers(0, 3))
            lo, hi = bounds()
            pos.append((api.select_column(cols[c], lo, hi), cpu.select_scan(data[c], lo, hi)))
        elif op <= 3:                                            # fetch through some position list
            c = int(rng.integers(0, 3))
            h, m = pos[int(rng.integers(0, len(pos)))]
            val.append((api.fetch_column(cols[c], h), cpu.fetch(data[c], m), h, m))
        elif op == 4 and val:                                    # aggregate
            h, m, _, _ = val[int(rng.integers(0, len(val)))]
            if m.size:
                name = ["sum", "average", "min", "max"][int(rng.integers(0, 4))]
                r = api.sum_result(h) if name == "sum" else api.unary(name, h)
                got = api.tuples(r)[0]
                if name == "average":
                    assert got.tobytes() == np.float64(cpu.avg(m)).tobytes()
                else:
                    assert int(got) == {"sum": cpu.sum, "min": cpu.min, "max": cpu.max}[name](m)
                api.drop(r)
        elif op == 5 and val:                                    # read a value vector
            h, m, _, _ = val[int(rng.integers(0, len(val)))]
            check(h, m)
        elif op == 6:                                            # read a position list
            h, m = pos[int(rng.integers(0, len(pos)))]
            check(h, m)
        elif op == 7 and val:                                    # select over (values, their positions)
            h, m, ph, pm = val[int(rng.integers(0, len(val)))]
            if any(ph is p for p, _ in pos):                     # the position list is still bound
                lo, hi = bounds()
                pos.append((api.select_result(h, ph, lo, hi), cpu.select_result(m, pm, lo, hi)))
        elif op == 8 and len(val) >= 2:                          # add / sub of equally long vectors
            i, j = rng.integers(0, len(val), 2)
            (h1, m1, _, _), (h2, m2, _, _) = val[int(i)], val[int(j)]
            if m1.size == m2.size:
                sub = bool(rng.integers(0, 2))
                r = api.binary("sub" if sub else "add", h1, h2)
                exp = (m1.astype(np.int64) - m2 if sub else m1.astype(np.int64) + m2).astype(np.int32)
                check(r, exp)
                api.drop(r)
        elif op == 9 and val:                                    # release a value vector
            h, _, _, _ = val.pop(int(rng.integers(0, len(val))))
            api.drop(h)
        elif op == 10 and len(pos) > 1:                          # release a position list
            h, _ = pos.pop(int(rng.integers(0, len(pos))))
            api.drop(h)
        elif op == 11:
            which = int(rng.integers(0, 3))
            if which == 0:                                       # insert_row re-mmaps: db_manager.c:178-186
                api.lib.adb_host_column_invalidate(C.byref(cols[int(rng.integers(0, 3))]))
            elif which == 1 and val:                             # print of a short vector
                h, m, _, _ = val[int(rng.integers(0, len(val)))]
                if 0 < m.size <= 5000:
                    assert api.print(h) == "\n".join(str(int(v)) for v in m)
            else:                                                # a small batch in between
                c = int(rng.integers(0, 3))
                lows, highs = [-100, 5, 2000], [300, 6, 2100]
                res = api.shared_select(cols[c], lows, highs)
                for r, lo, hi in zip(res, lows, highs):
                    check(r, cpu.select_scan(data[c], lo, hi))
                    api.drop(r)
        if len(pos) > 12:
            api.drop(pos.pop(0)[0])
        if len(val) > 12:
            api.drop(val.pop(0)[0])
    for h, m, _, _ in val:
        check(h, m)
        api.drop(h)
    for h, m in pos:
        check(h, m)
        api.drop(h)
    # (<=: entries an earlier test leaked on purpose -- payloads freed behind the shim's back --
    # may have been reclaimed meanwhile, when malloc handed their addresses out again)
    assert api.lib.adb_host_live_device_results() <= live0


def test_joins_of_growing_size_reconnect_the_exchange(api, cpu, rng):
    """Every join larger than the exchange's receive regions re-creates them; the epoch words of
    the exchange protocol live in a mailbox that survives, so epochs must keep counting (r02: a
    restart at epoch 1 took the previous connection's count rows for its own)."""
    for n1, n2 in [(300, 40), (2000, 299), (150_000, 90_000), (400_000, 1000), (700, 650)]:
        v1 = rng.integers(0, max(n2, 50), n1).astype(np.int32)
        v2 = rng.permutation(n2).astype(np.int32)
        p1, p2 = np.arange(n1, dtype=np.int32), np.arange(n2, dtype=np.int32)
        R = [C.pointer(api.host_result(x)) for x in (v1, p1, v2, p2)]
        o1, o2 = api.join("hash_join", *R)
        e1, e2 = cpu.hash_join(v1, p1, v2, p2)
        assert np.array_equal(api.tuples(o1), e1) and np.array_equal(api.tuples(o2), e2), (n1, n2)
        api.drop(o1), api.drop(o2)


def test_recycled_payload_address_is_not_mistaken_for_a_device_result(api, rng):
    """A payload freed behind the shim's back whose address malloc then gives to a foreign host
    Result: the registry still knows the address, the tag the shim stamped into its own blocks is
    gone, so the operand is read as the host array it is (ADVICE r1)."""
    import query_api
    from query_api import Result, INT
    libc = query_api._libc
    libc.malloc.restype, libc.malloc.argtypes = C.c_void_p, [C.c_size_t]
    n = 30_000
    data = rng.integers(0, 1000, n).astype(np.int32)
    col = api.column(data)
    hit = False
    freed = set()
    for _ in range(50):
        s = api.select_column(col, 0, 500)
        m = s.contents.num_tuples
        api.tuples(s)                                     # written, registered
        addr = s.contents.payload
        freed.add(addr)
        libc.free(addr)                                   # plumbing-style free, no hook
        libc.free(C.cast(s, C.c_void_p))
        p = libc.malloc(4 * m)                            # same size: usually the same address
        foreign = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_int)), shape=(m,))
        foreign[:] = np.arange(m, dtype=np.int32)[::-1] % n
        r = Result(m, INT, p)
        f = api.fetch_column(col, C.pointer(r))
        assert np.array_equal(api.tuples(f), data[foreign])
        got = np.empty(m, np.int32)
        assert api.lib.adb_host_result_to_host(C.byref(r), got.ctypes.data_as(C.c_void_p)) == 0
        assert np.array_equal(got, foreign)
        api.drop(f)
        hit = hit or p == addr
        libc.free(p)
    assert hit                                            # the scenario did occur
    release_leaked(api, freed)


def test_ten_thousand_exchanges(api, rng):
    """The aggregate exchange's two-bank epoch protocol (adb_common.cuh: peer_exchange_warp) over
    10 000 back-to-back rounds, alternating the fused and the stand-alone form: every round's
    table-wide aggregate must be exact (a late or early peer record would corrupt a sum)."""
    n = 40_000
    data = rng.integers(-10**6, 10**6, n).astype(np.int32)
    col = api.column(data)
    total = int(data.astype(np.int64).sum())
    s = api.select_column(col, None, 0)
    f = api.fetch_column(col, s)
    neg = int(data[data < 0].astype(np.int64).sum())
    st = Status(99, None)
    g1, g2 = GeneralizedColumn(1), GeneralizedColumn(RESULT)      # COLUMN, RESULT
    g1.column_pointer.column = C.pointer(col)
    g2.column_pointer.result = f
    drop3 = (type(f) * 1)()
    for k in range(5_000):
        a = api.lib.sum(C.byref(g1), C.byref(st))
        b = api.lib.sum(C.byref(g2), C.byref(st))
        assert C.cast(a.contents.payload, C.POINTER(C.c_long))[0] == total, k
        assert C.cast(b.contents.payload, C.POINTER(C.c_long))[0] == neg, k
        for r in (a, b):
            drop3[0] = r
            api.lib.adb_host_results_drop(drop3, 1)
    api.drop(s), api.drop(f)


def test_lazy_handles_are_written_only_when_read(api, cpu, rng):
    """SURVEY.md 8f rank 3: s=select / f=fetch / a=sum(f) answers the aggregate without writing s
    or f (4N + 4H bytes); the handles are written when -- and only when -- somebody reads them,
    also after later selects have taken the bitmap over (recipes re-run the predicate pass)."""
    import analytical_database_b200 as adb
    eng = adb.Engine(0)                                   # same library: launch counters
    n = 200_003
    c1, c4, lo, hi = _chain_inputs(rng, n)
    col1, col4 = api.column(c1), api.column(c4)
    api.lib.adb_host_column_upload(C.byref(col1)), api.lib.adb_host_column_upload(C.byref(col4))
    epos = cpu.select_scan(c1, lo, hi)
    evals = cpu.fetch(c4, epos)
    G = api.lib.adb_host_gpus()
    live0 = api.lib.adb_host_live_device_results()

    def chain(lo_, hi_):
        s_ = api.select_column(col1, lo_, hi_)
        f_ = api.fetch_column(col4, s_)
        a_ = api.sum_result(f_)
        return s_, f_, a_
    # (1) released unread: per GPU the predicate pass (mask, total, publish) and ONE gather+fold
    # kernel (+ publish on GPU 0) -- no expansion writes, no fetch kernel, no aggregate kernel
    l0 = eng.lib.adb_launch_count_all()
    s, f, a = chain(lo, hi)
    assert int(api.tuples(a)[0]) == cpu.sum(evals)
    launches = eng.lib.adb_launch_count_all() - l0
    assert launches <= 4 * G + 1, launches
    for r in (s, f, a):                                   # select first: the fetch stays unwritten
        api.drop(r)
    assert api.lib.adb_host_live_device_results() == live0
    # (2) several chains in a row, all handles alive (the server's handles live until the client
    # disconnects): nothing is written until the end, then everything is read back in any order
    kept = []
    for k in range(5):
        lo_k, hi_k = lo + 37 * k, hi - 11 * k
        s, f, a = chain(lo_k, hi_k)
        ep = cpu.select_scan(c1, lo_k, hi_k)
        assert int(api.tuples(a)[0]) == cpu.sum(cpu.fetch(c4, ep))
        kept.append((s, f, a, ep))
    for k in (3, 0, 4, 1, 2):
        s, f, a, ep = kept[k]
        if k % 2:
            assert np.array_equal(api.tuples(f), cpu.fetch(c4, ep))
            assert np.array_equal(api.tuples(s), ep)
        else:
            assert np.array_equal(api.tuples(s), ep)
            mx = api.unary("max", f)                      # an aggregate of a demoted handle
            assert int(api.tuples(mx)[0]) == cpu.max(cpu.fetch(c4, ep))
            assert np.array_equal(api.tuples(f), cpu.fetch(c4, ep))
            api.drop(mx)
    for s, f, a, _ in kept:
        for r in (f, s, a):
            api.drop(r)
    # (3) second aggregate on the same handle writes on the way; a third reads the written vector
    s, f, a = chain(lo, hi)
    av = api.unary("average", f)
    assert api.tuples(av)[0].tobytes() == np.float64(cpu.avg(evals)).tobytes()
    mn = api.unary("min", f)
    assert int(api.tuples(mn)[0]) == cpu.min(evals)
    assert np.array_equal(api.tuples(s), epos) and np.array_equal(api.tuples(f), evals)
    for r in (s, f, a, av, mn):
        api.drop(r)
    # (4) the select is released, its unwritten fetch lives on through two more selects and a
    # column invalidation, and is then read
    s, f, a = chain(lo, hi)
    api.drop(s)
    t1 = api.select_column(col4, None, I32MAX - 9000)
    t2 = api.select_column(col1, 0, 5)
    api.lib.adb_host_column_invalidate(C.byref(col4))
    assert np.array_equal(api.tuples(f), evals)
    assert np.array_equal(api.tuples(t1), cpu.select_scan(c4, None, I32MAX - 9000))
    for r in (f, a, t1, t2):
        api.drop(r)
    assert api.lib.adb_host_live_device_results() == live0


# ---- one process, several GPUs: the cases only a sharded layout has ---------------------------
@pytest.mark.parametrize("route_min", ["0", "1000000000"])
def test_sharded_lists_that_are_not_row_aligned(api, cpu, rng, monkeypatch, route_min):
    """Position lists in index order, from a join, or built by foreign code name rows of any
    shard: fetch routes the positions to the GPUs that hold the rows and gathers the values back
    into list order (adb_route_rows; ADB_FETCH_ROUTE_MIN=0 forces it at any size) or reads every
    remote row with a peer load (adb_fetch_sharded), and must still be the reference's gather,
    element for element."""
    monkeypatch.setenv("ADB_FETCH_ROUTE_MIN", route_min)
    n = 100_003
    live0 = api.lib.adb_host_live_device_results()
    data = rng.integers(0, 5000, n).astype(np.int32)
    other = rng.integers(-10**6, 10**6, n).astype(np.int32)
    values, positions = cpu.index_sort(data)
    col = api.column(data, index=(values, positions), sorted_=True)
    ocol = api.column(other)
    s = api.select_column(col, 1000, 1200)
    exp, undefined = cpu.select_sorted_index(values, positions, 1000, 1200)
    assert not undefined and np.array_equal(api.tuples(s), exp)
    f = api.fetch_column(ocol, s)
    assert np.array_equal(api.tuples(f), other[exp])
    a = api.sum_result(f)
    assert int(api.tuples(a)[0]) == int(other[exp].astype(np.int64).sum())
    s2 = api.select_result(f, s, 0, None)
    assert np.array_equal(api.tuples(s2), cpu.select_result(other[exp], exp, 0, None))
    # a host-built list in no order at all
    perm = rng.permutation(n)[:7777].astype(np.int32)
    hp = api.host_result(perm)
    f2 = api.fetch_column(ocol, C.pointer(hp))
    assert np.array_equal(api.tuples(f2), other[perm])
    # operands cut differently: f (cut like the index slices) + f3 (cut like the rows)
    rows = api.select_column(ocol, None, None)
    f3 = api.fetch_column(ocol, rows)
    short = api.host_result(np.arange(exp.size, dtype=np.int32))
    d = api.binary("add", f, C.pointer(short))
    assert np.array_equal(api.tuples(d), (other[exp].astype(np.int64) + np.arange(exp.size)).astype(np.int32))
    d2 = api.binary("sub", f, f3)                     # f3 is longer: its head is used (query.c:361)
    assert np.array_equal(api.tuples(d2), (other[exp].astype(np.int64) - other[:exp.size]).astype(np.int32))
    for r in (s, f, a, s2, f2, rows, f3, d, d2):
        api.drop(r)
    assert api.lib.adb_host_live_device_results() == live0


@pytest.mark.parametrize("n", [1, 31, 33, 65, 200])
def test_columns_shorter_than_the_shard_grid(api, cpu, rng, n):
    """Fewer rows than shards x 32: trailing shards are empty and every operator still agrees."""
    live0 = api.lib.adb_host_live_device_results()
    c1 = rng.integers(-50, 50, n).astype(np.int32)
    c2 = rng.integers(-1000, 1000, n).astype(np.int32)
    col1, col2 = api.column(c1), api.column(c2)
    for lo, hi in [(None, None), (-10, 10), (49, None), (7, 7)]:
        s = api.select_column(col1, lo, hi)
        epos = cpu.select_scan(c1, lo, hi)
        f = api.fetch_column(col2, s)
        a = api.sum_result(f)
        assert int(api.tuples(a)[0]) == cpu.sum(cpu.fetch(c2, epos))
        assert np.array_equal(api.tuples(s), epos) and np.array_equal(api.tuples(f), cpu.fetch(c2, epos))
        if epos.size:
            mx = api.unary("max", f)
            assert int(api.tuples(mx)[0]) == cpu.max(cpu.fetch(c2, epos))
            api.drop(mx)
        for r in (s, f, a):
            api.drop(r)
    tot = api.sum_column(col2)
    assert int(api.tuples(tot)[0]) == cpu.sum_column(c2)
    api.drop(tot)
    res = api.shared_select(col1, [-5, 0, 60], [5, 1, 70])
    for r, (lo, hi) in zip(res, [(-5, 5), (0, 1), (60, 70)]):
        assert np.array_equal(api.tuples(r), cpu.select_scan(c1, lo, hi))
        api.drop(r)
    assert api.lib.adb_host_live_device_results() == live0


def test_index_quirk_across_slices(api, cpu, rng):
    """low == high on a key (query.c:181-188) and bounds around slice boundaries of the
    range-partitioned index: runs of equal keys never straddle a slice, and the quirk is decided
    for the whole index, not per slice."""
    n = 9_000
    data = np.repeat(np.arange(0, 90, dtype=np.int32), 100)            # 90 runs of 100 equal keys
    rng.shuffle(data)
    values, positions = cpu.index_sort(data)
    col = api.column(data, index=(values, positions), sorted_=True)
    cases = [(k, k) for k in (0, 29, 30, 44, 45, 59, 60, 89)] + [(29, 31), (44, 46), (0, 90), (30, 30), (88, 200)]
    for lo, hi in cases:
        s = api.select_column(col, lo, hi)
        exp, undefined = cpu.select_sorted_index(values, positions, lo, hi)
        assert not undefined
        assert np.array_equal(api.tuples(s), exp), (lo, hi)
        api.drop(s)


def test_long_print_across_shards(api, rng):
    n = 50_000
    data = rng.integers(-2**31, 2**31 - 1, n, dtype=np.int64).astype(np.int32)
    col = api.column(data)
    s = api.select_column(col, None, None)
    f = api.fetch_column(col, s)
    assert api.print(f) == "\n".join(str(int(v)) for v in data)
    api.drop(s), api.drop(f)


@pytest.mark.parametrize("sharded_probe", ["routed", "routed-partitioned", "peer"])
def test_join_of_sharded_operands(api, cpu, rng, monkeypatch, sharded_probe):
    """With several GPUs the probe keys are routed to their owners and the answers gathered back
    into row order (default; the owner probes what it received directly or, for a table far
    beyond L2, slice by slice: ADB_JOIN_PROBE=partitioned forces that at any size), or every GPU
    probes in place and reads remote slots over peer memory (ADB_JOIN_SHARDED_PROBE=peer): same
    pairs, same order."""
    monkeypatch.setenv("ADB_JOIN_SHARDED_PROBE", sharded_probe.split("-")[0])
    if sharded_probe.endswith("partitioned"):
        monkeypatch.setenv("ADB_JOIN_PROBE", "partitioned")
    n1, n2 = 70_000, 50_000
    live0 = api.lib.adb_host_live_device_results()
    k1 = rng.integers(1, 30_000, n1).astype(np.int32)
    k2 = rng.integers(1, 30_000, n2).astype(np.int32)
    f1 = rng.integers(0, 100, n1).astype(np.int32)
    f2 = rng.integers(0, 100, n2).astype(np.int32)
    ck1, ck2, cf1, cf2 = (api.column(x) for x in (k1, k2, f1, f2))
    p1, p2 = api.select_column(cf1, None, 80), api.select_column(cf2, None, 15)   # milestone4.py:332-339
    v1, v2 = api.fetch_column(ck1, p1), api.fetch_column(ck2, p2)
    o1, o2 = api.join("hash_join", v1, p1, v2, p2)
    e_p1, e_p2 = cpu.select_scan(f1, None, 80), cpu.select_scan(f2, None, 15)
    e1, e2 = cpu.hash_join(k1[e_p1], e_p1, k2[e_p2], e_p2)
    assert np.array_equal(api.tuples(o1), e1) and np.array_equal(api.tuples(o2), e2)
    g1 = api.fetch_column(cf1, o1)                     # join output feeds a fetch (tests 32-37)
    assert np.array_equal(api.tuples(g1), f1[e1])
    a = api.unary("average", g1)
    assert api.tuples(a)[0].tobytes() == np.float64(cpu.avg(f1[e1])).tobytes()
    for r in (p1, p2, v1, v2, o1, o2, g1, a):
        api.drop(r)
    # heavy skew: a few hundred keys, groups of hundreds of rows spread over every GPU (the probing
    # GPU reads the owner's sorted build positions over peer memory), both join kinds
    s1, s2 = rng.integers(1, 300, 40_000).astype(np.int32), rng.integers(1, 400, 900).astype(np.int32)
    q1, q2 = rng.permutation(40_000).astype(np.int32), rng.permutation(900).astype(np.int32)
    R = [C.pointer(api.host_result(x)) for x in (s1, q1, s2, q2)]
    for name in ("hash_join", "nested_loop_join"):
        if name == "nested_loop_join":                       # quadratic in the oracle: smaller
            R = [C.pointer(api.host_result(x)) for x in (s1[:3000], q1[:3000], s2, q2)]
        o1, o2 = api.join(name, *R)
        args = (s1, q1, s2, q2) if name == "hash_join" else (s1[:3000], q1[:3000], s2, q2)
        e1, e2 = getattr(cpu, name)(*args)
        assert np.array_equal(api.tuples(o1), e1) and np.array_equal(api.tuples(o2), e2), name
        api.drop(o1), api.drop(o2)
    assert api.lib.adb_host_live_device_results() == live0
