"""GPU parity for batch_queries/batch_execute (BASELINE config 2): adb_shared_select_count/_emit against
the oracle's restatement of shared_select (query.c:450-583) and, on the value domain where
the reference's slicing is valid (SURVEY A6), against the unmodified reference objects.
Mirrors milestone2.py: 2 queries disjoint / partial / subsumed (:42-160), 10 queries, and
100 queries batched vs unbatched (:218-255)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from analytical_database_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(autouse=True, params=["pair lists", "interval lists"])
def list_form(request, monkeypatch):
    """Both hit-list forms of the batched scan (shared_scan.cu): batches at most four queries
    deep take pair lists unless ADB_SS_INTERVAL_LISTS is set; deeper ones always take interval
    lists."""
    if request.param == "interval lists":
        monkeypatch.setenv("ADB_SS_INTERVAL_LISTS", "1")
    else:
        monkeypatch.delenv("ADB_SS_INTERVAL_LISTS", raising=False)
    return request.param


def check(eng, port, data, lows, highs, ref=None):
    col = eng.upload(data)
    got = eng.shared_select(col, data.size, lows, highs)
    exp = port.shared_select(data, lows, highs)
    for q, ((buf, cnt), e) in enumerate(zip(got, exp)):
        assert cnt == e.size, (q, cnt, e.size)
        assert np.array_equal(buf.to_host(cnt), e), q
    if ref is not None:
        r = ref.shared_select(data, lows, highs)
        for q, ((buf, cnt), e) in enumerate(zip(got, r)):
            assert cnt == e.size and np.array_equal(buf.to_host(cnt), e), q
    for buf, _ in got:
        buf.free()
    col.free()


def test_two_queries_shapes(eng, port, ref, rng):
    n = 30000
    data = rng.integers(0, n, n).astype(np.int32)
    for lows, highs in [([100, 20000], [5000, 25000]),       # disjoint
                        ([100, 3000], [5000, 9000]),         # partial overlap
                        ([100, 1000], [20000, 2000]),        # subsumed
                        ([500, 500], [900, 900]),            # identical
                        ([7, 7], [7, 8])]:                   # empty + single value
        check(eng, port, data, np.array(lows, np.int32), np.array(highs, np.int32), ref)


@pytest.mark.parametrize("n,q", [(1, 1), (511, 3), (4097, 10), (30000, 100), (100003, 150)])
def test_random_batches(eng, port, ref, rng, n, q):
    data = rng.integers(0, max(n, 2), n).astype(np.int32)
    lows = rng.integers(0, max(n, 2), q).astype(np.int32)
    highs = (lows + rng.integers(0, n // 8 + 2, q)).astype(np.int32)
    if q > 3:
        lows[1], highs[1] = 0, n          # everything
        lows[2], highs[2] = 50, 10        # inverted -> empty
        lows[3], highs[3] = lows[0], highs[0]   # duplicate query
    check(eng, port, data, lows, highs, ref if n >= 30000 else None)


@pytest.mark.parametrize("depth", [1, 2, 3, 4, 5])
def test_cover_depths(eng, port, rng, depth):
    """Batches exactly `depth` queries deep: staggered ranges, each overlapping its depth - 1
    successors (1 = disjoint); 4 is the deepest batch that takes pair lists.  More than one
    1024-entry tile per chunk (dense hits), ties on the bounds, duplicates of a query."""
    n, q = 300_000, 60
    data = rng.integers(0, 6000, n).astype(np.int32)
    lows = (np.arange(q) * 100).astype(np.int32)
    highs = (lows + 100 * depth).astype(np.int32)
    check(eng, port, data, lows, highs)
    if depth >= 2:                                           # the same depth out of identical queries
        lows2 = np.repeat(lows[::depth], depth)[:q].astype(np.int32)
        check(eng, port, data, lows2, (lows2 + 100).astype(np.int32))


def test_negative_and_extreme_values(eng, port, rng):
    """Outside the reference's valid slicing domain (A6): compared with the restatement."""
    n = 50001
    data = rng.integers(-2**31, 2**31 - 1, n, dtype=np.int64).astype(np.int32)
    lows = np.array([-2**31, -5, 2**31 - 100000, 0, -2**30], np.int32)
    highs = np.array([2**31 - 1, 5, 2**31 - 1, 2**30, 2**30], np.int32)
    check(eng, port, data, lows, highs)


def test_heavily_overlapping(eng, port, rng):
    n = 20000
    data = rng.integers(0, 1000, n).astype(np.int32)
    lows = np.arange(0, 150, dtype=np.int32)
    highs = (1000 - np.arange(0, 150)).astype(np.int32)      # nested ranges: every row hits many
    check(eng, port, data, lows, highs)


def test_config2_scale_matches_unbatched(eng, port):
    """BASELINE config 2: 100 range selects over a 100 M-row column.  Every batched list must
    equal the engine's own (separately oracle-checked) single select, and three of them are
    diffed against the oracle on a 4 M-row window regenerated on the host."""
    from analytical_database_b200 import synth
    n, q = 100_000_000, 100
    col = eng.synth_uniform(n, 42, 0, 0, n)
    r = np.random.default_rng(42)
    lows = r.integers(0, n - n // 1000, q).astype(np.int32)
    highs = (lows + n // 1000).astype(np.int32)
    got = eng.shared_select(col, n, lows, highs)
    for i, (buf, cnt) in enumerate(got):
        pos, dc, h = eng.select_scan(col, n, int(lows[i]), int(highs[i]))
        assert h == cnt, i
        assert np.array_equal(pos.to_host(h), buf.to_host(cnt)), i
        pos.free(); dc.free()
    w = 4_000_000
    host = synth.uniform(w, 42, 0, 0, n)
    exp = port.shared_select(host, lows[:3], highs[:3])
    for i in range(3):
        g = got[i][0].to_host(got[i][1])
        assert np.array_equal(g[g < w], exp[i])
