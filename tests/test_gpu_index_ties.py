"""adb_index_sort_ref_ties and ADB_INDEX_TIES=reference: the index build on the GPU with equal
keys in exactly the order the reference's quicksort leaves them (init_column_index + quicksort,
src/index.c:25-46,89-101; oracle: index_sort of the reference library when built, else the
restatement that is diff-tested against it).

C-ABI level: values and positions element for element, over sizes on both sides of the
one-CTA threshold (4096 rows) and sizes that take several global levels, and key shapes from
all-distinct to all-equal.  The reference is quadratic on long runs of equal keys, so each shape
goes only up to the size its sort finishes in seconds.  Shim level: the catalog's index, the
clustered siblings, the declaration-order quirk and the rebuilds after an update or a delete all
equal the reference's, positions and order included."""
import ctypes as C
import functools
import os

import numpy as np
import pytest

from query_api import Api, Column

pytestmark = pytest.mark.gpu

I32_MIN, I32_MAX = np.iinfo(np.int32).min, np.iinfo(np.int32).max


@pytest.fixture(scope="module", params=[1, 3], ids=["1gpu", "3gpus"])
def api(request):
    old = os.environ.get("ADB_INDEX_TIES")
    os.environ["ADB_INDEX_TIES"] = "reference"
    a = Api()
    try:
        assert a.lib.adb_host_init_multi(request.param) == 0, a.lib.adb_host_last_error()
        yield a
        a.lib.adb_host_shutdown()
    finally:
        if old is None:
            os.environ.pop("ADB_INDEX_TIES", None)
        else:
            os.environ["ADB_INDEX_TIES"] = old


@pytest.fixture(scope="module")
def cpu():
    from oracle import oracle
    return oracle.reference("O2") or oracle.port()


@pytest.fixture
def eng(api):
    import analytical_database_b200 as adb
    return adb.Engine(0)                                  # the shim's context 0, same library


def _shape(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind.startswith("distinct"):
        return rng.integers(0, int(kind[-1]) + 1, n)       # keys 0 .. d
    if kind == "uniform300":
        return rng.integers(-150, 150, n)
    if kind == "zipf":
        return np.minimum(rng.zipf(1.5, n), 100_000)
    if kind == "all_equal":
        return np.full(n, -3)
    if kind == "permutation":
        return rng.permutation(n) - n // 2
    if kind == "nondecreasing_runs":
        return np.sort(rng.integers(0, max(2, n // 50), n))
    if kind == "reverse_dups":
        return np.sort(rng.integers(0, max(2, n // 4), n))[::-1]
    if kind == "extremes":
        v = rng.integers(I32_MIN, I32_MAX, n, endpoint=True)
        pick = rng.random(n)
        v[pick < 0.05] = I32_MIN
        v[pick > 0.95] = I32_MAX
        v[(pick > 0.45) & (pick < 0.5)] = -1
        return v
    if kind == "alternating":
        return np.where(np.arange(n) % 2 == 0, 9, -9)
    raise AssertionError(kind)


# largest size at which the reference's quicksort (quadratic in the length of a run of equal
# keys) stays within seconds, per shape
MAX_N = {"distinct0": 100_003, "distinct1": 100_003, "distinct2": 100_003, "distinct3": 100_003,
         "uniform300": 1_000_003, "zipf": 100_003, "all_equal": 100_003, "permutation": 1_000_003,
         "nondecreasing_runs": 1_000_003, "reverse_dups": 20_000, "extremes": 100_003, "alternating": 100_003}
SIZES = [1, 2, 3, 33, 4097, 20_000, 100_003, 1_000_003]
CASES = [(k, n) for k in MAX_N for n in SIZES if n <= MAX_N[k]]


@functools.lru_cache(maxsize=None)
def _expected(kind, n):
    from oracle import oracle
    cpu = oracle.reference("O2") or oracle.port()
    col = _shape(kind, n, n).astype(np.int32)
    ev, ep = cpu.index_sort(col)
    return col, ev, ep.astype(np.int64)


@pytest.mark.parametrize("kind,n", CASES, ids=[f"{k}-{n}" for k, n in CASES])
def test_ref_ties_equal_the_reference_sort(eng, kind, n):
    col, ev, ep = _expected(kind, n)
    d = eng.upload(col)
    vals, poss = eng.index_sort_ref_ties(d, n)
    gv, gp = vals.to_host(n), poss.to_host(n)
    assert np.array_equal(gv, ev)
    bad = np.flatnonzero(gp != ep)
    assert bad.size == 0, (bad[:10], gp[bad[:10]], ep[bad[:10]])
    sv, sp = eng.index_sort(d, n)                          # values always equal adb_index_sort's
    assert np.array_equal(sv.to_host(n), gv)
    if kind == "permutation" or n == 1:
        assert np.array_equal(sp.to_host(n), gp)
    for b in (d, vals, poss, sv, sp):
        b.free()


def test_ref_ties_refuses_what_index_sort_refuses(eng):
    d = eng.alloc_i32(4)
    for n in (-1, 1 << 31):
        assert eng.lib.adb_index_sort_ref_ties(d.i32(), n, d.i32(), d.i32()) != 0
    assert eng.lib.adb_index_sort_ref_ties(None, 4, d.i32(), d.i32()) != 0
    assert eng.lib.adb_index_sort_ref_ties(None, 0, None, None) == 0
    d.free()


# ---- the host shim with ADB_INDEX_TIES=reference -------------------------------------------------
@pytest.mark.parametrize("n", [1000, 150_001])
def test_unclustered_duplicate_keys_equal_the_reference(api, cpu, rng, n):
    key = rng.integers(0, 300, n).astype(np.int32)
    sib = np.arange(n, dtype=np.int32)
    cols = api.table([sib, key], {1: (True, False)})
    values, positions = api.build_index(cols, 1)
    ev, ep = cpu.index_sort(key)
    assert np.array_equal(values, ev) and np.array_equal(positions, ep)
    for lo, hi in [(17, 42), (int(ev[0]) + 1, 100), (150, int(ev[-1]))]:
        s = api.select_column(cols[1][0], lo, hi)
        exp, undefined = cpu.select_sorted_index(ev, ep, lo, hi)
        assert not undefined and np.array_equal(api.tuples(s), exp), (lo, hi)
        api.drop(s)


@pytest.mark.parametrize("n", [4099, 200_003])
def test_clustered_duplicate_keys_permute_siblings_as_the_reference(api, cpu, rng, n):
    key = rng.integers(-50, 50, n).astype(np.int32)
    a, b = rng.integers(0, 1000, n).astype(np.int32), np.arange(n, dtype=np.int32)
    cols = api.table([a, key, b], {1: (True, True)})
    values, positions = api.build_index(cols, 1)
    ev, ep = cpu.index_sort(key)
    assert np.array_equal(values, ev)
    assert np.array_equal(positions, np.arange(n, dtype=np.uint64))
    ra, rb = cpu.reorder(a, ep), cpu.reorder(b, ep)
    assert np.array_equal(cols[0][1], ra) and np.array_equal(cols[2][1], rb)
    # the device copies moved the same way: a full select on the clustered column fetches them
    s = api.select_column(cols[1][0], -50, 50)
    exp, undefined = cpu.select_sorted_index(ev, np.arange(n, dtype=np.uint64), -50, 50)
    assert not undefined and np.array_equal(api.tuples(s), exp)
    fa, fb = api.fetch_column(cols[0][0], s), api.fetch_column(cols[2][0], s)
    assert np.array_equal(api.tuples(fa), ra[exp]) and np.array_equal(api.tuples(fb), rb[exp])
    for r in (s, fa, fb):
        api.drop(r)


def test_declaration_order_quirk_with_duplicate_keys(api, cpu, rng):
    """tbl4 of milestone 3 (test 25): an unclustered index on an earlier column keeps
    pre-permutation positions when a later column's clustered index, here on duplicate keys,
    permutes the table.  Which rows a select on it then fetches depends on the clustered
    column's tie order."""
    n = 20_011
    c1 = rng.integers(0, 10**6, n).astype(np.int32)
    c2 = rng.integers(0, 2000, n).astype(np.int32)
    c3 = rng.integers(-100, 100, n).astype(np.int32)
    cols = api.table([c1, c2, c3], {1: (False, False), 2: (True, True)})
    v2, p2 = api.build_index(cols, 1)
    v3, p3 = api.build_index(cols, 2)
    e2v, e2p = cpu.index_sort(c2)
    e3v, e3p = cpu.index_sort(c3)
    assert np.array_equal(v2, e2v) and np.array_equal(p2, e2p)
    assert np.array_equal(v3, e3v) and np.array_equal(p3, np.arange(n, dtype=np.uint64))
    assert np.array_equal(cols[0][1], cpu.reorder(c1, e3p)) and np.array_equal(cols[1][1], cpu.reorder(c2, e3p))
    s = api.select_column(cols[1][0], 100, 300)
    exp, undefined = cpu.select_sorted_index(e2v, e2p, 100, 300)
    assert not undefined and np.array_equal(api.tuples(s), exp)
    f = api.fetch_column(cols[0][0], s)
    assert np.array_equal(api.tuples(f), cpu.reorder(c1, e3p)[exp])
    api.drop(s), api.drop(f)


def test_update_and_delete_rebuild_the_index_in_reference_order(api, cpu, rng):
    n = 30_000
    key = rng.integers(0, 400, n).astype(np.int32)
    pay = rng.integers(0, 500, n).astype(np.int32)
    cols = api.table([key, pay], {0: (True, False)})
    ptrs = (C.POINTER(Column) * 2)(*[C.pointer(c) for c, _ in cols])
    api.build_index(cols, 0)
    model = [key.copy(), pay.copy()]
    # UPDATE key = 7 WHERE pay in [100, 140): the indexed key itself changes, its index is rebuilt
    u = api.select_column(cols[1][0], 100, 140)
    assert api.lib.adb_host_relational_update(ptrs, 2, 0, u, 7) == 0, api.lib.adb_host_last_error()
    model[0][(model[1] >= 100) & (model[1] < 140)] = 7
    api.drop(u)
    _check_index(api, cpu, cols, model)
    dele = rng.choice(n, 4000, replace=False).astype(np.int32)
    hd = api.host_result(dele)
    assert api.lib.adb_host_relational_delete(ptrs, 2, C.pointer(hd)) == 0, api.lib.adb_host_last_error()
    keep = np.ones(n, bool)
    keep[dele] = False
    model = [m[keep] for m in model]
    _check_index(api, cpu, cols, model)


def _check_index(api, cpu, cols, model):
    m = model[0].size
    col = cols[0][0]
    assert col.row_count == m
    ev, ep = cpu.index_sort(model[0])
    ix = col.index.contents
    assert np.array_equal(np.ctypeslib.as_array(ix.values, shape=(m,)), ev)
    assert np.array_equal(np.ctypeslib.as_array(ix.positions, shape=(m,)), ep)
    for lo, hi in [(7, 8), (int(ev[m // 4]), int(ev[m // 2]))]:
        s = api.select_column(col, lo, hi)
        exp, undefined = cpu.select_sorted_index(ev, ep, lo, hi)
        assert not undefined and np.array_equal(api.tuples(s), exp), (lo, hi)
        f = api.fetch_column(cols[1][0], s)
        assert np.array_equal(api.tuples(f), model[1][exp])
        api.drop(s), api.drop(f)
