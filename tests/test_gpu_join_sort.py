"""GPU parity for the joins (BASELINE config 4) and the index build.

hash_join / nested_loop_join: pair lists must equal the oracle's element for element --
probe-major over side two with side one's insertion order inside a key for the hash join,
outer-major over side one for the nested loop (SURVEY A5).  Inputs mirror milestone4.py:
many-one and many-many joins, zipfian keys (:31-53), selective prefilters; plus the
oracle-undefined domain (negative keys, empty sides) as equi-join semantics.
index sort: stable order; equals the reference's quicksort whenever keys are unique (A3)."""
import numpy as np
import pytest

import join_reference

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from analytical_database_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(params=["direct", "partitioned"])
def probe_mode(request, monkeypatch):
    """Both forms of the probe on the same inputs: rows in their original order (one random slot
    read each) and rows partitioned by window and table slice (hash_join.cu, P1-P3) -- the engine
    picks by size, ADB_JOIN_PROBE forces."""
    monkeypatch.setenv("ADB_JOIN_PROBE", request.param)
    return request.param


def run_join(eng, k1, p1, k2, p2, nested=False):
    d = [eng.upload(x) for x in (k1, p1, k2, p2)]
    o1, o2, m = eng.join(d[0], d[1], k1.size, d[2], d[3], k2.size, nested_loop=nested)
    a, b = o1.to_host(m), o2.to_host(m)
    for x in d + [o1, o2]:
        x.free()
    return a, b


def inputs(rng, n1, n2, kind):
    if kind == "zipf":
        k1 = (rng.zipf(1.3, n1) % 1000).astype(np.int32)
        k2 = (rng.zipf(1.3, n2) % 1000).astype(np.int32)
    elif kind == "unique":
        k1 = rng.permutation(4 * max(n1, 1))[:n1].astype(np.int32)
        k2 = rng.permutation(4 * max(n1, 1))[:n2].astype(np.int32)
    elif kind == "negative":
        k1 = rng.integers(-max(n1 // 4, 2), max(n1 // 4, 2), n1).astype(np.int32)
        k2 = rng.integers(-max(n1 // 4, 2), max(n1 // 4, 2), n2).astype(np.int32)
    else:
        k1 = rng.integers(0, max(n1 // 4, 2), n1).astype(np.int32)
        k2 = rng.integers(0, max(n1 // 4, 2), n2).astype(np.int32)
    p1 = rng.permutation(10 * max(n1, 1))[:n1].astype(np.int32)
    p2 = rng.permutation(10 * max(n2, 1) + 1)[:n2].astype(np.int32)
    return k1, p1, k2, p2


@pytest.mark.parametrize("kind", ["uniform", "unique", "zipf", "negative"])
@pytest.mark.parametrize("n1,n2", [(1, 1), (4, 1), (100, 7), (2000, 1500), (1500, 0), (0, 9),
                                   (5000, 5000), (40000, 9000)])
def test_hash_join_order(eng, port, rng, probe_mode, kind, n1, n2):
    if kind == "zipf" and n1 * n2 > 3e7:
        n2 = 2000                                  # keep the many-many blow-up bounded
    k1, p1, k2, p2 = inputs(rng, n1, n2, kind)
    a, b = run_join(eng, k1, p1, k2, p2)
    e1, e2 = port.hash_join(k1, p1, k2, p2)
    assert a.size == e1.size, (kind, n1, n2)
    assert np.array_equal(a, e1) and np.array_equal(b, e2), (kind, n1, n2)


@pytest.mark.parametrize("kind", ["uniform", "zipf"])
@pytest.mark.parametrize("n1,n2", [(1, 1), (300, 200), (1500, 1500), (1500, 0)])
def test_nested_loop_join_order(eng, port, rng, probe_mode, kind, n1, n2):
    k1, p1, k2, p2 = inputs(rng, n1, n2, kind)
    a, b = run_join(eng, k1, p1, k2, p2, nested=True)
    e1, e2 = port.nested_loop_join(k1, p1, k2, p2)
    assert np.array_equal(a, e1) and np.array_equal(b, e2), (kind, n1, n2)


def test_hash_join_vs_reference_objects(eng, ref, rng, probe_mode):
    k1, p1, k2, p2 = inputs(rng, 30000, 20000, "uniform")
    a, b = run_join(eng, k1, p1, k2, p2)
    e1, e2 = ref.hash_join(k1, p1, k2, p2)
    assert np.array_equal(a, e1) and np.array_equal(b, e2)


def test_hash_join_skewed_partition(eng, port, rng, probe_mode):
    """One key owns 40 % of the build side: its partition overflows the shared-memory table
    and takes the global-memory path; the probe side hits it a few times."""
    n1, n2 = 60000, 300
    k1 = rng.integers(0, 50000, n1).astype(np.int32)
    k1[rng.random(n1) < 0.4] = 777
    k2 = rng.integers(0, 50000, n2).astype(np.int32)
    k2[:5] = 777
    p1 = np.arange(n1, dtype=np.int32)[::-1].copy()
    p2 = np.arange(n2, dtype=np.int32) + 5
    a, b = run_join(eng, k1, p1, k2, p2)
    e1, e2 = port.hash_join(k1, p1, k2, p2)
    assert np.array_equal(a, e1) and np.array_equal(b, e2)


def test_hash_join_multi_pass_partitioning(eng, port, rng, probe_mode):
    """3 M x 2 M many-one join: 12 partition bits (two probe passes).  Keys stay below the
    reference's table size (1.3 n1): its identity hash `key % size` (multimap.c:60-63) wraps
    larger keys onto an already full region and the CPU probe goes quadratic."""
    n1, n2 = 3_000_000, 2_000_000
    k1 = rng.permutation(n1).astype(np.int32)
    k2 = rng.integers(0, int(1.25 * n1), n2).astype(np.int32)
    p1 = rng.permutation(n1).astype(np.int32)
    p2 = rng.permutation(n2).astype(np.int32)
    a, b = run_join(eng, k1, p1, k2, p2)
    e1, e2 = port.hash_join(k1, p1, k2, p2)
    assert a.size == e1.size
    assert np.array_equal(a, e1) and np.array_equal(b, e2)


@pytest.mark.parametrize("n", [1, 255, 256, 257, 5000, 1_000_003])
def test_index_sort(eng, port, rng, n):
    for data in (rng.integers(-2**31, 2**31 - 1, n, dtype=np.int64).astype(np.int32),
                 rng.integers(-50, 50, n).astype(np.int32),
                 rng.permutation(n).astype(np.int32)):
        col = eng.upload(data)
        dv, dp = eng.index_sort(col, n)
        values, positions = dv.to_host(n), dp.to_host(n)
        order = np.argsort(data, kind="stable").astype(np.int32)
        assert np.array_equal(positions, order)
        assert np.array_equal(values, data[order])
        for x in (col, dv, dp):
            x.free()
    if n <= 5000:                                 # unique keys: identical to the reference quicksort
        data = rng.permutation(n).astype(np.int32)
        col = eng.upload(data)
        dv, dp = eng.index_sort(col, n)
        ev, ep = port.index_sort(data)
        assert np.array_equal(dv.to_host(n), ev) and np.array_equal(dp.to_host(n), ep.astype(np.int32))


def test_full_size_join_properties(eng):
    """BASELINE config 4 at its full size on one GPU: 100 M x 100 M rows, prefilters at 80 % and
    15 %, hash join of the (value, position) pair lists.  The oracle's multimap needs minutes
    there, so the pair lists are compared element for element with the numpy join
    (join_reference.py, pinned to the oracle in test_gpu_join_geometry.py) of the very lists the
    GPU joined.  Also: the pair count equals sum_k count1(k) * count2(k) from a host histogram,
    every pair joins equal keys and every output position passed its side's prefilter."""
    n = 100_000_000
    k1, k2 = eng.synth_uniform(n, 11, 0, 1, n), eng.synth_uniform(n, 12, 0, 1, n)
    f1, f2 = eng.synth_uniform(n, 13, 0, 0, 1000), eng.synth_uniform(n, 14, 0, 0, 1000)
    p1, c1 = eng.select_exact(f1, n, None, 800)
    p2, c2 = eng.select_exact(f2, n, None, 150)
    v1, v2 = eng.fetch(k1, p1, c1), eng.fetch(k2, p2, c2)
    assert c1 > c2                                            # parse.c:798-813: larger side builds
    o1, o2, m = eng.join(v1, p1, c1, v2, p2, c2)
    h1 = np.bincount(v1.to_host(c1), minlength=n + 1)
    hv2 = v2.to_host(c2)
    assert m == int(h1[hv2].sum())                            # sum_k count1(k) * count2(k)
    # equal keys on both sides of every pair
    z = eng.aggregate(eng.ewise(eng.fetch(k1, o1, m), eng.fetch(k2, o2, m), m, True), m)
    assert z.min == 0 and z.max == 0
    # every output position passed its side's prefilter
    a1, a2 = eng.aggregate(eng.fetch(f1, o1, m), m), eng.aggregate(eng.fetch(f2, o2, m), m)
    assert a1.max < 800 and a2.max < 150
    # the pair lists themselves: probe-major, build order inside a probe row
    e1, e2 = join_reference.hash_join(v1.to_host(c1), p1.to_host(c1), hv2, p2.to_host(c2))
    ho1, ho2 = o1.to_host(m), o2.to_host(m)
    bad = np.flatnonzero((ho1 != e1) | (ho2 != e2))
    assert bad.size == 0, ("first wrong pair", int(bad[0]), "of", bad.size)
    assert np.any(ho2[1:] == ho2[:-1])                        # probe rows with several build rows
