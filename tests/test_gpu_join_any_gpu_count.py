"""The sharded joins at any number of engine contexts, not only powers of two.

A key's owner is its routing hash h = key * 0x85EBCA6B (mod 2^32) scaled to the G owners,
floor(h * G / 2^32): the top log2(G) bits of h when G is a power of two, near-even shares of the
hash range otherwise.  CPU: route_owner, the numpy twin of that function, and where it meets
the power-of-two rule the sharded tests route with (sharded_cpu_ops.route_dest).  GPU: the
routing pass of the engine against the twin, and hash_join / nested_loop_join through query.h
at 3, 5, 6 and 7 contexts against the oracle, pair for pair and in order, with every context
running its share of the join."""
import ctypes as C
import re
from collections import Counter

import numpy as np
import pytest


I32MIN, I32MAX = -2**31, 2**31 - 1
ROUTE_MUL = 0x85EBCA6B


def route_hash(keys):
    return (keys.astype(np.int64).astype(np.uint64) * np.uint64(ROUTE_MUL)) & np.uint64(0xFFFFFFFF)


def route_owner(keys, parts):
    """Owner of every key among `parts` owners: floor(h * parts / 2^32)."""
    return ((route_hash(keys) * np.uint64(parts)) >> np.uint64(32)).astype(np.int64)


def top_bits_owner(keys, parts):
    """The owner rule before any owner count was allowed: the top log2(parts) bits of the hash."""
    k = parts.bit_length() - 1
    if k == 0:
        return np.zeros(keys.size, np.int64)
    return (route_hash(keys) >> np.uint64(32 - k)).astype(np.int64)


# ---- CPU: the owner function ----------------------------------------------------------------------
def test_owner_is_the_top_bits_at_powers_of_two():
    keys = np.random.default_rng(3).integers(I32MIN, I32MAX, 10**6, endpoint=True).astype(np.int32)
    keys[:4] = [I32MIN, -1, 0, I32MAX]
    from sharded_cpu_ops import route_dest
    for k in range(9):
        assert np.array_equal(route_owner(keys, 1 << k), top_bits_owner(keys, 1 << k)), 1 << k
        assert np.array_equal(route_owner(keys, 1 << k), route_dest(keys, 1 << k)), 1 << k


@pytest.mark.parametrize("G", range(3, 17))
def test_owners_split_the_hash_range_evenly(G):
    # owner o takes the hash values [ceil(o * 2^32 / G), ceil((o + 1) * 2^32 / G))
    first = [-(-(o << 32) // G) for o in range(G)] + [1 << 32]
    shares = np.diff(first)
    assert shares.sum() == 1 << 32 and shares.max() - shares.min() <= 1
    # the twin puts both sides of every boundary, and both ends of the range, where those say
    hs = [0, (1 << 32) - 1] + [b + d for b in first[1:-1] for d in (-1, 0)]
    want = [0, G - 1] + [o + d for o in range(1, G) for d in (-1, 0)]
    inv = pow(ROUTE_MUL, -1, 1 << 32)                  # the key whose hash is h
    keys = np.array([h * inv % (1 << 32) for h in hs], np.uint64).astype(np.uint32).view(np.int32)
    assert np.array_equal(route_hash(keys), np.array(hs, np.uint64))
    assert route_owner(keys, G).tolist() == want


# ---- GPU, engine: adb_route_pairs at any owner count ----------------------------------------------
@pytest.fixture
def eng():
    from analytical_database_b200 import Engine
    return Engine(0)                                   # context 0 (also the host's, when it is up)


def route_pairs(eng, val, pos, parts):
    n = val.size
    dv, dp = eng.upload(val), eng.upload(pos)
    ov, op = eng.alloc_i32(n), eng.alloc_i32(n)
    counts = (C.c_int64 * parts)()
    eng._ck(eng.lib.adb_route_pairs(dv.i32(), dp.i32(), n, parts, ov.i32(), op.i32(), counts))
    out = list(counts), ov.to_host(n), op.to_host(n)
    for b in (dv, dp, ov, op):
        b.free()
    return out


def route_inputs(n, seed):
    rng = np.random.default_rng(seed)
    val = rng.integers(I32MIN, I32MAX, n, endpoint=True).astype(np.int32)
    val[:6] = [I32MIN, I32MIN, I32MAX, -1, 0, I32MAX]
    val[6:n // 3] = rng.integers(-2000, 2000, n // 3 - 6)           # repeated keys: order inside a run
    return val, rng.permutation(n).astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("parts", [3, 5, 6, 7, 12, 255, 2, 4, 8])
def test_route_pairs_at_any_owner_count(eng, parts):
    n = 300_007
    val, pos = route_inputs(n, parts)
    counts, ov, op = route_pairs(eng, val, pos, parts)
    # powers of two: the top bits of the hash, as before; any other count: the twin
    d = top_bits_owner(val, parts) if parts & (parts - 1) == 0 else route_owner(val, parts)
    assert d.min() >= 0 and d.max() < parts
    assert counts == np.bincount(d, minlength=parts).tolist()
    order = np.argsort(d, kind="stable")               # input order kept inside every destination
    assert np.array_equal(ov, val[order]) and np.array_equal(op, pos[order])


@pytest.mark.gpu
@pytest.mark.parametrize("parts", [0, -1, 257])
def test_route_pairs_refuses_owner_counts_out_of_range(eng, parts):
    d = eng.upload(np.arange(16, dtype=np.int32))
    o = eng.alloc_i32(16)
    counts = (C.c_int64 * 300)()
    assert eng.lib.adb_route_pairs(d.i32(), d.i32(), 16, parts, o.i32(), o.i32(), counts) != 0
    d.free(), o.free()


# ---- GPU, query.h: the joins at 3, 5, 6 and 7 contexts ------------------------------------------
SHIM_VARS = ("ADB_SHIM_MIRROR", "ADB_SHIM_EAGER", "ADB_SHARD_MIN_ROWS", "ADB_REBALANCE_MIN", "ADB_TRACE",
             "ADB_JOIN_PROBE", "ADB_FETCH_ROUTE_MIN")
SHARDED_STAGES = ("build sort", "received keys in + probe", "answers back to row order + piece offsets",
                  "expand (sharded)")


@pytest.fixture(scope="module", params=[3, 5, 6, 7], ids=lambda g: f"{g}ctx")
def api(request):
    """G engine contexts in one process; on a box with fewer devices they share them."""
    from query_api import Api
    with pytest.MonkeyPatch.context() as mp:
        for var in SHIM_VARS:
            mp.delenv(var, raising=False)
        a = Api()
        a.lib.adb_host_shutdown()                      # a fresh host: exchange regions sized from scratch
        assert a.lib.adb_host_init_multi(request.param) == 0, a.lib.adb_host_last_error()
        assert a.lib.adb_host_gpus() == request.param
        yield a
        a.lib.adb_host_shutdown()


@pytest.fixture(autouse=True)
def default_forms(monkeypatch):
    for var in SHIM_VARS:
        monkeypatch.delenv(var, raising=False)


def join_both(api, port, name, k1, p1, k2, p2):
    """One join of host arrays through query.h against the oracle, element for element."""
    R = [C.pointer(api.host_result(x)) for x in (k1, p1, k2, p2)]
    o1, o2 = api.join(name, *R)
    e1, e2 = getattr(port, name)(k1, p1, k2, p2)
    got1, got2 = api.tuples(o1), api.tuples(o2)
    api.drop(o1), api.drop(o2)
    assert got1.size == e1.size, name
    assert np.array_equal(got1, e1) and np.array_equal(got2, e2), name


def positions(rng, n):
    return rng.permutation(10 * n + 3)[:n].astype(np.int32)


def zipf_keys(rng, n, cap):
    """Many-to-many keys (milestone 4's skew): a few keys with thousands of rows, a long tail."""
    return np.minimum(rng.zipf(1.5, n), cap).astype(np.int32)


CASES = ("uniform", "zipf", "extremes", "build smaller than G")


def case_inputs(case, G, nested):
    """(side one keys, side two keys).  The hash join builds side one, the nested-loop join side
    two; the nested-loop oracle is quadratic, so its sides are smaller."""
    rng = np.random.default_rng(sum(map(ord, case)) + 10 * G + nested)
    if case == "uniform":
        n1, n2 = (3000, 1200) if nested else (60_000, 40_000)
        return rng.integers(1, 20_000, n1).astype(np.int32), rng.integers(1, 20_000, n2).astype(np.int32)
    if case == "zipf":
        n1, n2 = (3000, 2000) if nested else (8000, 3000)
        return zipf_keys(rng, n1, 5000), zipf_keys(rng, n2, 5000)
    if case == "extremes":
        pool = np.array([I32MIN, I32MIN + 1, -65536, -7, -1, 0, 1, 65536, I32MAX - 1, I32MAX], np.int32)
        n1, n2 = (2500, 1500) if nested else (50_000, 20_000)

        def side(n):
            k = rng.integers(I32MIN, 0, n).astype(np.int32)        # negative keys, mostly unique
            hot = rng.random(n) < 0.05
            k[hot] = rng.choice(pool, int(hot.sum()))
            return k
        return side(n1), side(n2)
    # fewer build rows than contexts: most owners receive nothing
    small = np.array([5, -3, 5, 11, I32MAX, I32MIN][:G - 1], np.int32)
    big = rng.choice(np.array([5, -3, 11, 12, I32MAX, I32MIN, 0], np.int32), 5000).astype(np.int32)
    return (big, small) if nested else (small, big)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("name", ["hash_join", "nested_loop_join"])
def test_joins_match_the_oracle(api, port, case, name):
    G = api.lib.adb_host_gpus()
    k1, k2 = case_inputs(case, G, name == "nested_loop_join")
    rng = np.random.default_rng(k1.size + k2.size)
    join_both(api, port, name, k1, positions(rng, k1.size), k2, positions(rng, k2.size))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hash_join", "nested_loop_join"])
def test_operands_whose_last_contexts_are_empty(api, port, name):
    """Columns shorter than the shard grid (shards of at least 32 rows): a select + fetch leaves
    the last contexts with empty slices of both join sides."""
    G = api.lib.adb_host_gpus()
    rng = np.random.default_rng(G)
    live0 = api.lib.adb_host_live_device_results()
    n1, n2 = 70, 45                                    # 3 and 2 shards of 32 rows hold them
    k1, k2 = rng.integers(0, 12, n1).astype(np.int32), rng.integers(0, 12, n2).astype(np.int32)
    f1, f2 = rng.integers(0, 100, n1).astype(np.int32), rng.integers(0, 100, n2).astype(np.int32)
    ck1, ck2, cf1, cf2 = (api.column(x) for x in (k1, k2, f1, f2))
    p1, p2 = api.select_column(cf1, None, 90), api.select_column(cf2, None, 70)
    v1, v2 = api.fetch_column(ck1, p1), api.fetch_column(ck2, p2)
    o1, o2 = api.join(name, v1, p1, v2, p2)
    e_p1, e_p2 = port.select_scan(f1, None, 90), port.select_scan(f2, None, 70)
    e1, e2 = getattr(port, name)(k1[e_p1], e_p1, k2[e_p2], e_p2)
    assert e1.size > 0
    assert np.array_equal(api.tuples(o1), e1) and np.array_equal(api.tuples(o2), e2)
    for r in (p1, p2, v1, v2, o1, o2):
        api.drop(r)
    assert api.lib.adb_host_live_device_results() == live0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["hash_join", "nested_loop_join"])
def test_build_side_dominated_by_one_key(api, port, name):
    """95 % of the build side carries one key, so its owner receives far more than the exchange's
    first receive regions hold (an even split with 50 % head room); the join is retried with
    regions of the whole build side and must still give the reference's pairs."""
    G = api.lib.adb_host_gpus()
    api.lib.adb_host_shutdown()                        # the receive regions start at their first size
    assert api.lib.adb_host_init_multi(G) == 0, api.lib.adb_host_last_error()
    rng = np.random.default_rng(40 + G)
    nb, n_probe, hot = 600_000, 200 if name == "nested_loop_join" else 2000, 7
    kb = rng.integers(1, 5000, nb).astype(np.int32)
    kb[rng.random(nb) < 0.95] = hot
    kp = rng.integers(1, 5000, n_probe).astype(np.int32)
    kp[kp == hot] = hot + 1
    kp[[3, n_probe // 2]] = hot
    # the hot owner's share exceeds the first attempt's region (query_shim.c, join_sharded)
    first = nb // G + nb // (2 * G) + 65536
    region = 1 << max(17, (first - 1).bit_length())
    assert np.bincount(route_owner(kb, G), minlength=G).max() > region
    if name == "hash_join":                            # builds side one
        join_both(api, port, name, kb, positions(rng, nb), kp, positions(rng, n_probe))
    else:                                              # builds side two
        join_both(api, port, name, kp, positions(rng, n_probe), kb, positions(rng, nb))


@pytest.mark.gpu
def test_join_output_feeds_fetch_and_sum(api, port):
    """DSL tests 32-37: prefiltered sides joined, the join's positions fetched and summed."""
    G = api.lib.adb_host_gpus()
    rng = np.random.default_rng(70 + G)
    live0 = api.lib.adb_host_live_device_results()
    n1, n2 = 70_000, 50_000
    k1, k2 = rng.integers(1, 30_000, n1).astype(np.int32), rng.integers(1, 30_000, n2).astype(np.int32)
    f1, f2 = rng.integers(0, 100, n1).astype(np.int32), rng.integers(0, 100, n2).astype(np.int32)
    ck1, ck2, cf1, cf2 = (api.column(x) for x in (k1, k2, f1, f2))
    p1, p2 = api.select_column(cf1, None, 80), api.select_column(cf2, None, 15)   # milestone4.py:332-339
    v1, v2 = api.fetch_column(ck1, p1), api.fetch_column(ck2, p2)
    o1, o2 = api.join("hash_join", v1, p1, v2, p2)
    e_p1, e_p2 = port.select_scan(f1, None, 80), port.select_scan(f2, None, 15)
    e1, e2 = port.hash_join(k1[e_p1], e_p1, k2[e_p2], e_p2)
    assert np.array_equal(api.tuples(o1), e1) and np.array_equal(api.tuples(o2), e2)
    g1, g2 = api.fetch_column(cf1, o1), api.fetch_column(cf2, o2)
    s1, s2 = api.sum_result(g1), api.sum_result(g2)
    assert int(api.tuples(s1)[0]) == port.sum(f1[e1]) and int(api.tuples(s2)[0]) == port.sum(f2[e2])
    for r in (p1, p2, v1, v2, o1, o2, g1, g2, s1, s2):
        api.drop(r)
    assert api.lib.adb_host_live_device_results() == live0


@pytest.mark.gpu
def test_every_context_runs_its_share(api, port, capfd, monkeypatch):
    """The join is sharded, not gathered onto one GPU: every context sorts its share of the build
    side, probes the keys it owns, puts its rows' answers back in order and expands them."""
    G = api.lib.adb_host_gpus()
    rng = np.random.default_rng(90 + G)
    n1, n2 = 70_000, 50_000
    k1, k2 = rng.integers(1, 30_000, n1).astype(np.int32), rng.integers(1, 30_000, n2).astype(np.int32)
    p1, p2 = rng.permutation(n1).astype(np.int32), rng.permutation(n2).astype(np.int32)
    capfd.readouterr()
    monkeypatch.setenv("ADB_TRACE", "1")
    join_both(api, port, "hash_join", k1, p1, k2, p2)
    monkeypatch.delenv("ADB_TRACE")
    trace = capfd.readouterr().err
    stages = Counter(m.group(1) for m in re.finditer(r"^\[adb trace\] (.*?)\s+-?[\d.]+ ms$", trace, re.M))
    assert {s: stages[s] for s in SHARDED_STAGES} == {s: G for s in SHARDED_STAGES}
