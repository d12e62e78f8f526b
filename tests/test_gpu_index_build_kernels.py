"""The engine pieces of the index build over several contexts: the multi-target radix select
(adb_rank_hist), the range routing pass (adb_route_range) and the stable pairs sort
(adb_index_sort_pairs), each against numpy."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

INT_MIN, INT_MAX = -(1 << 31), (1 << 31) - 1


@pytest.fixture(scope="module")
def eng():
    from analytical_database_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


def key_sets(rng, n):
    yield "unique", (rng.permutation(n) - n // 2).astype(np.int32)
    yield "uniform20", rng.integers(0, 1 << 20, n).astype(np.int32)
    yield "few", rng.integers(0, 1000, n).astype(np.int32)
    yield "zipf", np.minimum(rng.zipf(1.3, n), INT_MAX).astype(np.int32)
    yield "equal", np.full(n, -12345, np.int32)
    yield "extremes", rng.choice(np.array([INT_MIN, INT_MIN + 1, -1, 0, INT_MAX - 1, INT_MAX], np.int32), n)
    yield "full", rng.integers(INT_MIN, INT_MAX, n, endpoint=True).astype(np.int32)


def radix_select(eng, bufs, ranks):
    """Exact keys of `ranks` over the concatenation of the device arrays bufs = [(buf, n)], as the
    host shim narrows them: four rounds, histograms summed over the arrays."""
    prefix = [0] * len(ranks)
    left = list(ranks)
    for rnd in range(4):
        pres = sorted(set(prefix))
        hist = sum(eng.rank_hist(b, n, pres, rnd).astype(np.int64) for b, n in bufs)
        for t in range(len(ranks)):
            row = hist[pres.index(prefix[t])]
            cum = np.cumsum(row)
            d = int(np.searchsorted(cum, left[t], side="right"))
            left[t] -= int(cum[d - 1]) if d else 0
            prefix[t] = prefix[t] << 8 | d
    keys = [p ^ 0x80000000 for p in prefix]
    return [k - (1 << 32) if k > INT_MAX else k for k in keys]


@pytest.mark.parametrize("n", [1, 7, 4099, 1_000_003])
def test_radix_select_equals_numpy_partition(eng, rng, n):
    for name, keys in key_sets(rng, n):
        ranks = sorted({0, n - 1, n // 2, n // 3, (2 * n) // 3, max(0, n - 2)})
        # the keys cut into three arrays, as three contexts would hold them
        cuts = [0, n // 3, (2 * n) // 3, n]
        bufs = [(eng.upload(keys[a:b]), b - a) for a, b in zip(cuts, cuts[1:])]
        got = radix_select(eng, bufs, ranks)
        exp = np.partition(keys, ranks)[ranks]
        assert got == exp.tolist(), (name, n)
        for b, _ in bufs:
            b.free()


def test_rank_hist_one_round_and_refusals(eng, rng):
    keys = rng.integers(INT_MIN, INT_MAX, 100_001, endpoint=True).astype(np.int32)
    d = eng.upload(keys)
    f = keys.view(np.uint32) ^ np.uint32(0x80000000)
    pres = sorted(set((f[:5] >> np.uint32(16)).tolist()))
    h = eng.rank_hist(d, keys.size, pres, 2)
    for i, p in enumerate(pres):
        sel = f[(f >> np.uint32(16)) == p]
        assert np.array_equal(h[i], np.bincount((sel >> np.uint32(8)) & np.uint32(255), minlength=256))
    from analytical_database_b200.engine import EngineError
    for pres, rnd in [([1], 0), ([0], 4), ([5, 5], 1), ([256], 1), (list(range(17)), 2), ([], 1)]:
        with pytest.raises(EngineError):
            eng.rank_hist(d, keys.size, pres, rnd)
    d.free()


@pytest.mark.parametrize("parts", range(1, 17))
def test_route_range_is_a_stable_partition_by_slice(eng, rng, parts):
    n = 300_017
    for name, keys in key_sets(rng, n):
        split = np.sort(rng.choice(keys, parts - 1)) if parts > 1 else np.zeros(0, np.int32)
        if name == "extremes" and parts > 2:
            split[-1] = INT_MAX                                           # a slice past the end
        base = 1_000_000
        d = eng.upload(keys)
        ko, ro, counts = eng.route_range(d, n, base, split, parts)
        dest = np.searchsorted(split.astype(np.int64), keys.astype(np.int64), side="left")
        order = np.argsort(dest, kind="stable")
        assert counts == np.bincount(dest, minlength=parts).tolist(), (name, parts)
        assert np.array_equal(ko.to_host(n), keys[order]), (name, parts)
        assert np.array_equal(ro.to_host(n), (order + base).astype(np.int32)), (name, parts)
        for b in (d, ko, ro):
            b.free()


def test_route_range_refusals(eng):
    from analytical_database_b200.engine import EngineError
    d = eng.upload(np.arange(100, dtype=np.int32))
    for parts in (0, 17, -1):
        with pytest.raises(EngineError, match="parts"):
            eng.route_range(d, 100, 0, np.zeros(max(parts - 1, 0), np.int32), parts)
    with pytest.raises(EngineError, match="decrease"):
        eng.route_range(d, 100, 0, np.array([5, 3], np.int32), 3)
    with pytest.raises(EngineError):
        eng.route_range(d, 100, (1 << 31) - 50, np.array([5], np.int32), 2)
    assert eng.route_range(d, 0, 0, np.array([5], np.int32), 2)[2] == [0, 0]
    d.free()


@pytest.mark.parametrize("n", [1, 33, 4097, 2_000_003])
def test_index_sort_pairs_equals_lexsort(eng, rng, n):
    for name, keys in key_sets(rng, n):
        pay = rng.integers(INT_MIN, INT_MAX, n, endpoint=True).astype(np.int32)
        dk, dp = eng.upload(keys), eng.upload(pay)
        v, p = eng.index_sort_pairs(dk, dp, n)
        order = np.lexsort((np.arange(n), keys))                  # stable: input order within a key
        assert np.array_equal(v.to_host(n), keys[order]), name
        assert np.array_equal(p.to_host(n), pay[order]), name
        for b in (dk, dp, v, p):
            b.free()
