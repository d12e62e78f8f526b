"""The rule the multi-GPU index build routes keys by (host/query_shim.c, sharded_build_sort):
key k belongs to slice d(k) = #{g in 1..G-1 : t_g < k}, t_g = the key of rank g*per - 1 in sorted
order (per = ceil(n / G); +inf when g*per >= n).  It must cut exactly where slice_bounds cuts the
sorted array -- at g*per, moved to the end of a run of equal keys -- or the index slices, and so
every answer of the index path, would change.  Both restated in Python, compared on random sorted
arrays."""
import numpy as np
import pytest

INT_MIN, INT_MAX = -(1 << 31), (1 << 31) - 1


def slice_bounds(v, G):
    """query_shim.c slice_bounds, line for line."""
    n = len(v)
    per = (n + G - 1) // G
    begin = [0]
    for g in range(1, G + 1):
        b = g * per
        if b >= n or g == G:
            b = n
        else:
            b = max(b, begin[g - 1])
            if 0 < b < n and v[b] == v[b - 1]:
                b = int(np.searchsorted(v, v[b - 1], side="right"))
        begin.append(b)
    return begin


def routed_bounds(keys, G):
    """Slice sizes from d(k) over the UNSORTED keys, scanned: what the sharded build installs."""
    n = len(keys)
    per = (n + G - 1) // G
    s = np.sort(keys, kind="stable")
    t = np.array([s[g * per - 1] if g * per < n else INT_MAX for g in range(1, G)], dtype=np.int64)
    d = np.searchsorted(t, np.asarray(keys, dtype=np.int64), side="left")     # #{t_g < k}
    sizes = np.bincount(d, minlength=G) if n else np.zeros(G, np.int64)
    return [0] + np.cumsum(sizes).tolist()


def shapes(rng, n):
    yield "unique", rng.permutation(n).astype(np.int64) - n // 2
    yield "few", rng.integers(0, 3, n)
    yield "zipf", np.minimum(rng.zipf(1.3, n), 10**6)
    yield "equal", np.full(n, 7)
    yield "extremes", rng.choice(np.array([INT_MIN, INT_MIN + 1, -1, 0, INT_MAX - 1, INT_MAX]), n)
    yield "uniform", rng.integers(INT_MIN, INT_MAX, n, endpoint=True)


@pytest.mark.parametrize("G", range(2, 17))
def test_the_routing_rule_cuts_where_slice_bounds_cuts(G):
    rng = np.random.default_rng(G)
    for n in sorted({0, 1, G - 1, G, G + 1, 33, 31 * G + 5, 1000, 4099}):
        for name, keys in shapes(rng, n):
            keys = np.asarray(keys, dtype=np.int64).clip(INT_MIN, INT_MAX)
            assert routed_bounds(keys, G) == slice_bounds(np.sort(keys), G), (G, n, name)


def test_all_equal_keys_land_in_one_slice():
    keys = np.full(1001, -3)
    for G in (2, 5, 8, 16):
        b = routed_bounds(keys, G)
        assert b[1] == 1001 and b[-1] == 1001
