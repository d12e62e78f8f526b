"""GPU parity tests (run with ``-m gpu`` on the B200 box): every operator of the engine's
C-ABI against the CPU oracle on the same seeded inputs.  Integer work: bit-exact.
avg: the same int64 sum and one fp64 divide, so also bit-exact (tolerance 1e-9 relative
is what north_star allows; the tests assert equality and would report any drift).

Edge cases follow the reference's own suite: absent bounds (milestone1.py:47-110),
negative values and the INT_MAX neighbourhood (milestone1.py:115-119), empty and
all-hit ranges, ragged sizes around the 4096-row tile, unaligned column views.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

I32MAX = 2**31 - 1
I32MIN = -2**31


@pytest.fixture(scope="module")
def eng():
    from analytical_database_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


def columns(rng, n):
    return {
        "uniform": rng.integers(-n // 2 - 1, n // 2 + 1, n, dtype=np.int64).astype(np.int32),
        "small": rng.integers(0, 100, n).astype(np.int32),
        "near_max": rng.integers(I32MAX - 10000, I32MAX, n, dtype=np.int64).astype(np.int32),
        "full": rng.integers(I32MIN, I32MAX, n, dtype=np.int64, endpoint=True).astype(np.int32),
    }


BOUNDS = [(None, None), (None, 10), (-5, None), (-100, 100), (0, 0), (50, 10), (7, 8),
          (I32MIN, I32MAX), (I32MAX - 5000, I32MAX), (I32MIN, I32MIN + 5000), (None, I32MIN),
          (I32MAX, None), (I32MAX, I32MAX)]


@pytest.mark.parametrize("n", [0, 1, 31, 4095, 4096, 4097, 100003, (1 << 20) + 5])
def test_select_scan(eng, port, rng, n):
    for name, data in columns(rng, n).items():
        col = eng.upload(data)
        for lo, hi in BOUNDS:
            pos, dcnt, h = eng.select_scan(col, n, lo, hi)
            exp = port.select_scan(data, lo, hi)
            assert h == exp.size, (name, lo, hi)
            assert np.array_equal(pos.to_host(h), exp), (name, lo, hi)
            assert int(dcnt.to_host(1, np.int64)[0]) == h
            pos.free(); dcnt.free()
        col.free()


def test_select_scan_selectivities_and_base(eng, port, rng):
    """Sparse (register) and dense (staged) write-out paths, mixed inside one column."""
    n = 300007
    data = rng.integers(0, 1000, n).astype(np.int32)
    data[50000:90000] = 5          # a dense run inside sparse surroundings
    col = eng.upload(data)
    for hi in [1, 2, 6, 10, 100, 126, 500, 1000]:
        pos, dcnt, h = eng.select_scan(col, n, 0, hi, base=1000)
        exp = port.select_scan(data, 0, hi) + 1000
        assert h == exp.size and np.array_equal(pos.to_host(h), exp), hi
        pos.free(); dcnt.free()
    col.free()


def test_select_scan_unaligned_view(eng, port, rng):
    """A column view that is only 4-byte aligned takes the scalar-load path."""
    n = 70001
    data = rng.integers(-50, 50, n + 3).astype(np.int32)
    col = eng.upload(data)
    for off in (1, 2, 3):
        pos, dcnt, h = eng.select_scan(col, n, -10, 10, col_offset=off)
        exp = port.select_scan(data[off:off + n], -10, 10)
        assert h == exp.size and np.array_equal(pos.to_host(h), exp), off
        pos.free(); dcnt.free()
    col.free()


@pytest.mark.parametrize("n", [0, 1, 4096, 50001])
def test_select_pairs(eng, port, rng, n):
    val = rng.integers(-100, 100, n).astype(np.int32)
    posin = rng.permutation(max(n, 1) * 3)[:n].astype(np.int32)
    dv, dp = eng.upload(val), eng.upload(posin)
    for lo, hi in BOUNDS[:8]:
        out, dcnt, h = eng.select_pairs(dv, dp, n, lo, hi)
        exp = port.select_result(val, posin, lo, hi)
        assert h == exp.size and np.array_equal(out.to_host(h), exp), (lo, hi)
        out.free(); dcnt.free()
    # device-side length: only the first n//2 pairs are live
    live = n // 2
    dn = eng.upload(np.array([live], np.int64))
    out, dcnt, h = eng.select_pairs(dv, dp, n, -20, 30, d_n=dn)
    exp = port.select_result(val[:live], posin[:live], -20, 30)
    assert h == exp.size and np.array_equal(out.to_host(h), exp)


@pytest.mark.parametrize("n,h", [(1, 1), (1000, 0), (1000, 1000), (100003, 33331), (1 << 20, 777777)])
def test_fetch(eng, port, rng, n, h):
    data = rng.integers(I32MIN, I32MAX, n, dtype=np.int64).astype(np.int32)
    pos = np.sort(rng.integers(0, n, h)).astype(np.int32)
    col, dp = eng.upload(data), eng.upload(pos)
    out = eng.fetch(col, dp, h)
    assert np.array_equal(out.to_host(h), port.fetch(data, pos))
    # unsorted positions + base offset + device-side length
    pos2 = rng.integers(0, n, h).astype(np.int32)
    dp2 = eng.upload(pos2 + 77)
    dn = eng.upload(np.array([h // 2], np.int64))
    out2 = eng.fetch(col, dp2, h, d_n=dn, base=77)
    assert np.array_equal(out2.to_host(h // 2), port.fetch(data, pos2[:h // 2]))


@pytest.mark.parametrize("n", [0, 1, 3, 4, 1023, 100003, (1 << 21) + 3])
def test_aggregate(eng, port, rng, n):
    for name, data in columns(rng, n + 3).items():
        buf = eng.upload(data)
        for off in (0, 1, 3):
            v = data[off:off + n]
            a = eng.aggregate(buf, n, offset=off)
            assert a.sum == port.sum(v) and a.count == n, (name, off)
            if n:
                assert a.min == port.min(v) and a.max == port.max(v), (name, off)
                assert a.avg == port.avg(v)
                assert abs(a.avg - port.avg(v)) <= 1e-9 * abs(port.avg(v))
            else:
                assert a.min == I32MAX and a.max == I32MIN and np.isnan(a.avg)
        buf.free()


@pytest.mark.parametrize("n", [1, 5, 4096, 100003])
def test_add_sub_wrap(eng, port, rng, n):
    a = rng.integers(I32MIN, I32MAX, n, dtype=np.int64).astype(np.int32)
    b = rng.integers(I32MAX - 10000, I32MAX, n, dtype=np.int64).astype(np.int32)
    da, db = eng.upload(a), eng.upload(b)
    assert np.array_equal(eng.ewise(da, db, n, False).to_host(n), port.add(a, b))
    assert np.array_equal(eng.ewise(da, db, n, True).to_host(n), port.sub(a, b))


@pytest.mark.parametrize("n", [0, 1, 513, 4097, 1_000_003])
def test_chain_matches_oracle_and_reference(eng, port, rng, n):
    """s=select(col1,lo,hi); f=fetch(col2,s); a=sum(f)/min/max/avg -- the north-star chain
    (predicate pass + expansion with the gather and the aggregates fused in): the same positions,
    values and aggregates as the oracle and the reference."""
    import ctypes as C
    from oracle import oracle
    ref = oracle.reference("O2")
    sel = rng.integers(-n // 2 - 1, n // 2 + 1, n).astype(np.int32)
    if n > 100000:
        sel[200000:260000] = 7          # a dense run: the shared-memory staged write-out
    fet = rng.integers(I32MAX - 10000, I32MAX, n, dtype=np.int64).astype(np.int32)   # milestone1 col4
    ds, df = eng.upload(sel), eng.upload(fet)
    pos, val, dcnt, dagg = eng.alloc_i32(n), eng.alloc_i32(n), eng.alloc(8), eng.alloc(64)
    for lo, hi in [(None, None), (-100, 5000), (0, None), (None, -490000), (5, 5), (-1000, 1000),
                   (7, 8)]:
        (plo, _a), (phi, _b) = (None, None), (None, None)
        blo = C.c_int32(lo) if lo is not None else None
        bhi = C.c_int32(hi) if hi is not None else None
        eng._ck(eng.lib.adb_chain_select_fetch_agg(
            ds.i32(), df.i32(), n, C.byref(blo) if blo is not None else None,
            C.byref(bhi) if bhi is not None else None, pos.i32(), val.i32(), dcnt.i64(),
            eng.agg_ptr(dagg)))
        h = int(dcnt.to_host(1, np.int64)[0])
        agg = eng.read_agg(dagg)
        exp_pos = port.select_scan(sel, lo, hi)
        exp_val = port.fetch(fet, exp_pos)
        assert h == exp_pos.size and agg.count == h
        assert np.array_equal(pos.to_host(h), exp_pos)
        assert np.array_equal(val.to_host(h), exp_val)
        assert agg.sum == port.sum(exp_val)
        assert (agg.sum, h) == port.chain_select_fetch_sum(sel, fet, lo, hi)
        if ref is not None:
            assert (agg.sum, h) == ref.chain_select_fetch_sum(sel, fet, lo, hi)
        if h:
            assert agg.min == port.min(exp_val) and agg.max == port.max(exp_val)
            assert agg.avg == port.avg(exp_val)


@pytest.mark.parametrize("n", [0, 1, 513, 4097, 1_000_003])
def test_unmaterialised_chain_matches_oracle(eng, port, rng, n):
    """adb_chain_select_agg: select -> fetch -> sum/min/max in ONE kernel with neither handle
    materialised (SURVEY.md 8f rank 3, 4N + 4H bytes), and the aggregate-only form of the deferred
    emit (adb_select_emit_fetch_agg with NULL outputs), against the oracle's chain."""
    import ctypes as C
    from analytical_database_b200.engine import _AggStruct
    sel = rng.integers(-n // 2 - 1, n // 2 + 1, n).astype(np.int32)
    if n > 100000:
        sel[200000:260000] = 7
    fet = rng.integers(I32MAX - 10000, I32MAX, n, dtype=np.int64).astype(np.int32)
    ds, df = eng.upload(sel), eng.upload(fet)
    dcnt, dagg = eng.alloc(8), eng.alloc(64)
    for lo, hi in [(None, None), (-100, 5000), (0, None), (None, -490000), (5, 5), (7, 8)]:
        blo = C.c_int32(lo) if lo is not None else None
        bhi = C.c_int32(hi) if hi is not None else None
        plo = C.byref(blo) if blo is not None else None
        phi = C.byref(bhi) if bhi is not None else None
        hagg = _AggStruct()
        eng._ck(eng.lib.adb_chain_select_agg(ds.i32(), df.i32(), n, plo, phi, dcnt.i64(), eng.agg_ptr(dagg),
                                             C.byref(hagg)))
        exp_pos = port.select_scan(sel, lo, hi)
        exp_val = port.fetch(fet, exp_pos)
        h = int(dcnt.to_host(1, np.int64)[0])
        assert h == exp_pos.size and hagg.count == h and hagg.sum == port.sum(exp_val)
        if h:
            assert hagg.min == port.min(exp_val) and hagg.max == port.max(exp_val)
        # the deferred form: count, aggregate unwritten, aggregate again, then write
        hc = C.c_int64(0)
        eng._ck(eng.lib.adb_select_count_base(ds.i32(), n, plo, phi, 0, None, C.byref(hc)))
        gen = eng.lib.adb_select_generation()
        for _ in range(2):
            h2 = _AggStruct()
            eng._ck(eng.lib.adb_select_emit_fetch_agg(df.i32(), None, None, eng.agg_ptr(dagg), C.byref(h2)))
            assert (h2.sum, h2.count) == (hagg.sum, h) and eng.lib.adb_select_generation() == gen
        pos, val = eng.alloc_i32(max(h, 1)), eng.alloc_i32(max(h, 1))
        h3 = _AggStruct()
        eng._ck(eng.lib.adb_select_emit_fetch_agg(df.i32(), pos.i32(), val.i32(), eng.agg_ptr(dagg), C.byref(h3)))
        assert (h3.sum, h3.count) == (hagg.sum, h)
        assert np.array_equal(pos.to_host(h), exp_pos) and np.array_equal(val.to_host(h), exp_val)
        pos.free(), val.free()


def test_synth_twin(eng):
    from analytical_database_b200 import synth
    for n, seed, first, lo, span in [(1000, 42, 0, 0, 1 << 31), (100003, 7, 12345678901, -500, 1000),
                                     (4097, 42, 1 << 33, I32MAX - 10000, 10000)]:
        d = eng.synth_uniform(n, seed, first, lo, span)
        assert np.array_equal(d.to_host(n), synth.uniform(n, seed, first, lo, span))


def test_full_size_shard_properties(eng, port):
    """One 500 M-row shard of BASELINE config 5 (4 B rows / 8), far beyond what the oracle
    scans in seconds: checked through size-independent properties, plus an exact oracle
    diff on two sampled row windows regenerated on the host from the counter-based
    generator."""
    from analytical_database_b200 import synth
    n, seed = 500_000_000, 42
    span = 1 << 30
    col = eng.synth_uniform(n, seed, 0, 0, span)
    lo, hi = 1000, 1000 + span // 100                       # ~1 % selectivity
    pos, dcnt, h = eng.select_scan(col, n, lo, hi)
    # (1) partition property: counts of a split range add up; null/null selects everything
    mid = lo + (hi - lo) // 3
    p1, c1, h1 = eng.select_scan(col, n, lo, mid)
    p2, c2, h2 = eng.select_scan(col, n, mid, hi)
    assert h1 + h2 == h
    p1.free(); p2.free()
    assert abs(h - n / 100) < 5 * (n / 100) ** 0.5 * 3       # binomial sanity
    # (2) positions strictly ascending: min(pos[1:] - pos[:-1]) >= 1, via the engine's sub/min
    import ctypes as C
    from analytical_database_b200.engine import DevBuf
    shifted = DevBuf.__new__(DevBuf); shifted.eng, shifted.nbytes, shifted.ptr = eng, 0, pos.ptr + 4
    diff = eng.ewise(shifted, pos, h - 1, True)
    d = eng.aggregate(diff, h - 1)
    assert d.min >= 1 and d.sum == int(pos.to_host(1, offset_bytes=4 * (h - 1))[0]) - int(pos.to_host(1)[0])
    # (3) every fetched value satisfies the predicate; fetch is idempotent w.r.t. select
    val = eng.fetch(col, pos, h, d_n=dcnt)
    a = eng.aggregate(val, h, d_n=dcnt)
    assert a.count == h and lo <= a.min and a.max < hi
    # (4) exact diff against the oracle on two windows of the shard
    for first in (0, 377_000_123):
        w = 3_000_000
        host = synth.uniform(w, seed, first, 0, span)
        exp = port.select_scan(host, lo, hi) + first
        allpos = None
        # positions inside the window are a contiguous slice of the ascending list
        before = eng.select_scan(col, first, lo, hi)[2] if first else 0
        got = pos.to_host(exp.size, offset_bytes=4 * before)
        assert np.array_equal(got, exp)
        assert np.array_equal(val.to_host(exp.size, offset_bytes=4 * before), port.fetch(host, exp - first))
