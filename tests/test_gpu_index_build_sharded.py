"""The index build with every context sorting its own slice (G > 1, the stable tie order): the
catalog arrays, the device slices, index selects and fetches, and clustered siblings must be what
the one-context build gives, byte for byte.  Contexts may share one device."""
import ctypes as C

import numpy as np
import pytest

from query_api import Api, Column

pytestmark = pytest.mark.gpu

INT_MIN, INT_MAX = -(1 << 31), (1 << 31) - 1
SIZES = [0, 3, 100_003, 2_000_011]


def keys_of(shape, n, seed):
    rng = np.random.default_rng(seed)
    if shape == "permutation":
        return rng.permutation(n).astype(np.int32)
    if shape == "uniform20":
        return rng.integers(0, 1 << 20, n).astype(np.int32)
    if shape == "uniform1000":
        return rng.integers(0, 1000, n).astype(np.int32)
    if shape == "zipf":
        return np.minimum(rng.zipf(1.5, n), INT_MAX).astype(np.int32)
    if shape == "equal":
        return np.full(n, 42, np.int32)
    if shape == "extremes":
        k = rng.integers(-5000, 5000, n).astype(np.int32)
        k[rng.random(n) < 0.1] = INT_MIN
        k[rng.random(n) < 0.1] = INT_MAX
        return k
    if shape == "sorted":
        return np.sort(rng.integers(-10**6, 10**6, n)).astype(np.int32)
    if shape == "reversed":
        return np.sort(rng.integers(-10**6, 10**6, n))[::-1].astype(np.int32)
    raise ValueError(shape)


SHAPES = ["permutation", "uniform20", "uniform1000", "zipf", "equal", "extremes", "sorted", "reversed"]
CASES = [(s, n) for s in SHAPES for n in SIZES if n < 1_000_000 or s in ("permutation", "zipf", "equal", "reversed")]


def ranges_of(v):
    n = v.size
    if not n:
        return [(0, 10)]
    return [(int(v[n // 5]), int(v[(3 * n) // 5]) + 1), (int(v[0]), int(v[0]) + 1), (INT_MIN, int(v[n // 2])),
            (int(v[-1]), INT_MAX)]


def run_case(api, shape, n, clustered):
    key = keys_of(shape, n, n + len(shape))
    sib = np.arange(n, dtype=np.int32) * 3 - 7
    cols = api.table([sib, key], {1: (False, clustered)})             # btree
    values, positions = api.build_index(cols, 1)
    out = {"values": values.tobytes(), "positions": positions.tobytes(), "sib": cols[0][1].tobytes()}
    for lo, hi in ranges_of(np.sort(key)):
        s = api.select_column(cols[1][0], lo, hi)
        f = api.fetch_column(cols[0][0], s)
        out[(lo, hi)] = (api.tuples(s).tobytes(), api.tuples(f).tobytes())
        api.drop(s), api.drop(f)
    if n:                                                             # the sibling's device shards, row order
        s = api.select_column(cols[0][0], INT_MIN, None)
        f = api.fetch_column(cols[0][0], s)
        out["sib_dev"] = api.tuples(f).tobytes()
        api.drop(s), api.drop(f)
    return key, out


@pytest.fixture(scope="module")
def one_context():
    """Every case built with one context (the reference layout of the slices' concatenation)."""
    api = Api()
    assert api.lib.adb_host_init_multi(1) == 0, api.lib.adb_host_last_error()
    res = {(s, n, cl): run_case(api, s, n, cl)[1] for s, n in CASES for cl in (False, True)}
    api.lib.adb_host_shutdown()
    return res


@pytest.fixture(scope="module", params=[2, 3, 4, 5, 8], ids=lambda g: f"{g}ctx")
def api(request, one_context):
    a = Api()
    assert a.lib.adb_host_init_multi(request.param) == 0, a.lib.adb_host_last_error()
    a.G = request.param
    yield a
    a.lib.adb_host_shutdown()


@pytest.mark.parametrize("clustered", [False, True], ids=["unclustered", "clustered"])
def test_sharded_build_equals_one_context(api, one_context, clustered):
    for shape, n in CASES:
        key, got = run_case(api, shape, n, clustered)
        exp = one_context[(shape, n, clustered)]
        assert got.keys() == exp.keys(), (shape, n)
        for k in exp:
            assert got[k] == exp[k], (api.G, shape, n, k)
        order = np.argsort(key, kind="stable")
        assert got["values"] == key[order].tobytes()
        assert got["positions"] == (np.arange(n) if clustered else order).astype(np.uint64).tobytes()


def test_declaration_order_quirk(api, rng):
    """index.c:158-175: an unclustered index on an earlier column keeps its pre-permutation
    positions when a later column's clustered index permutes the table (test_gpu_index_build)."""
    n = 20_011
    c1 = rng.integers(0, 10**6, n).astype(np.int32)
    c2 = rng.integers(0, 500, n).astype(np.int32)                    # ties
    c3 = (rng.permutation(n) - 500).astype(np.int32)
    cols = api.table([c1, c2, c3], {1: (False, False), 2: (True, True)})
    v2, p2 = api.build_index(cols, 1)
    v3, p3 = api.build_index(cols, 2)
    o2, o3 = np.argsort(c2, kind="stable"), np.argsort(c3, kind="stable")
    assert np.array_equal(v2, c2[o2]) and np.array_equal(p2, o2.astype(np.uint64))
    assert np.array_equal(v3, c3[o3]) and np.array_equal(p3, np.arange(n, dtype=np.uint64))
    assert np.array_equal(cols[0][1], c1[o3]) and np.array_equal(cols[1][1], c2[o3])
    s = api.select_column(cols[1][0], 100, 300)
    lo, hi = np.searchsorted(c2[o2], [100, 300])
    exp = o2[lo:hi].astype(np.int32)                                   # stale positions, value order
    assert np.array_equal(api.tuples(s), exp)
    f = api.fetch_column(cols[0][0], s)
    assert np.array_equal(api.tuples(f), c1[o3][exp])
    api.drop(s), api.drop(f)


def test_sort_runs_on_every_context(api):
    """The slices are sorted where they live: every context that holds rows launches the sort's
    radix passes (4 passes x 4 kernels) during the build, not context 0 alone."""
    from analytical_database_b200.engine import lib_path
    n = 4_000_037
    key = np.random.default_rng(5).permutation(n).astype(np.int32)
    cols = api.table([key], {0: (False, False)})
    eng = C.CDLL(lib_path())
    eng.adb_launch_count.restype = C.c_int64

    def counts():
        out = []
        for g in range(api.G):
            eng.adb_ctx_select(g)
            out.append(eng.adb_launch_count())
        eng.adb_ctx_select(0)
        return np.array(out)

    api.lib.adb_host_column_upload.argtypes = [C.POINTER(Column)]
    assert api.lib.adb_host_column_upload(C.pointer(cols[0][0])) == 0              # the column is on the devices
    before = counts()
    values, positions = api.build_index(cols, 0)
    launched = counts() - before
    assert np.array_equal(values, np.arange(n, dtype=np.int32))
    assert (launched >= 16).all(), launched.tolist()
