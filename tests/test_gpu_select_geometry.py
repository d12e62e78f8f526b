"""The select family at the launch geometry of real-size columns, against numpy and the pinned
oracle.

select_geom (csrc/select_scan.cu) gives every warp k = ceil(tiles / (sm_count * 64)) tiles of
512 rows, so on a B200 (148 SMs) every column of up to 4 849 664 rows runs with k = 1.  The
kernels only take their multi-tile paths at larger k: the next-tile prefetch of the predicate
pass, the expansion's later 4096-row steps and its 1024-entry flush rounds, the later words and
rounds of the aggregate-only gather.  Here every entry point runs at k in {1, 2, 3, 8, 9, 16,
17}, at both ends of each regime, on inputs whose hit count is set per 4096-row expansion step
(0, 1, the sparse limit 64, 65, 1023-1025, 2048, 2049, every row), with dense runs across a
step boundary, a chunk boundary and into the ragged last chunk.  The streaming operators run past
their grid caps, the operator API runs with 2 and 3 contexts whose shards are at k >= 17 and
k >= 9, and (opt-in, ADB_TEST_MAX_SHARD=1) the chain runs over the largest legal shard."""
import ctypes as C
import os

import numpy as np
import pytest

I32MAX = 2**31 - 1
I32MIN = -2**31
LO, HI = -1000, 1000                    # the select bounds of the stepped inputs: [LO, HI)
BASE = 12_345                           # base_pos of the entry points that take one

SEL_WTILE = 512                         # rows per warp-tile (select_scan.cu: SEL_WTILE)
STEP_ROWS = 4096                        # rows per expansion step: 32 lanes x 4 mask words x 32 rows
STEP_HITS = (0, 1, 64, 65, 1023, 1024, 1025, 2048, 2049, STEP_ROWS)   # STEP_ROWS: every row


def select_geom(n, sm_count):
    """Python mirror of select_geom (csrc/select_scan.cu): (tiles per warp k, chunk_rows,
    num_chunks).  A chunk is one warp's contiguous row range in mask_kernel, expand_kernel,
    bitmap_gather_agg_kernel and scan_gather_agg_kernel alike."""
    wtiles = -(-n // SEL_WTILE)
    max_chunks = sm_count * 8 * 8                        # 8 CTAs of 8 warps per SM
    k = max(1, -(-wtiles // max_chunks))
    return k, k * SEL_WTILE, -(-wtiles // k)


def regime(k, sm_count):
    """(smallest, largest) n that select_geom runs with k tiles per warp.  The smallest is ragged
    (n % 32 == 1): its last chunk has whole tiles past n and the grid's trailing warps are idle."""
    per_k = sm_count * 64 * SEL_WTILE
    return (k - 1) * per_k + 1, k * per_k


def sizes(sm_count):
    out = []
    for k in (1, 2, 3, 8, 9, 16, 17):
        lo, hi = regime(k, sm_count)
        out += [1_000_003 if k == 1 else lo, hi]         # k = 1: a ragged n instead of n = 1
    return out


def stepped_mask(n, sm_count, rng):
    """A hit mask over n rows whose hit count is drawn from STEP_HITS for every expansion step of
    the chunk grid (k = 8: one step of 128 words per chunk; k = 16: two, i.e. one 256-word
    round of bitmap_gather_agg), plus dense runs across a step boundary, a chunk boundary and
    into the ragged last chunk."""
    k, chunk_rows, num_chunks = select_geom(n, sm_count)
    full, tail = divmod(chunk_rows, STEP_ROWS)
    grid = np.empty((num_chunks, chunk_rows), dtype=bool)

    def steps(m, rows):                                   # m steps of `rows` rows, exact counts
        perms = np.stack([rng.permutation(rows) for _ in range(16)]).astype(np.int16)
        want = np.minimum(rng.choice(STEP_HITS, m), rows).astype(np.int16)
        return perms[rng.integers(0, 16, m)] < want[:, None]

    if full:
        grid[:, :full * STEP_ROWS] = steps(num_chunks * full, STEP_ROWS).reshape(num_chunks, -1)
    if tail:
        grid[:, full * STEP_ROWS:] = steps(num_chunks, tail)
    mask = grid.reshape(-1)[:n]
    c = num_chunks // 2
    mask[c * chunk_rows - 1500:c * chunk_rows + 1500] = True            # chunk boundary
    if full >= 2 or (full == 1 and tail):
        s = (num_chunks // 3) * chunk_rows + STEP_ROWS
        mask[s - 1500:s + 1500] = True                                  # step boundary
    mask[n - 3000:] = True                                               # into the last chunk
    return mask


class Case:
    """One stepped select column, a full-range fetch column, a permutation for select_result and
    the answers, on the device and the host."""

    def __init__(self, eng, port, n):
        rng = np.random.default_rng(n)
        self.eng, self.n = eng, n
        self.k = select_geom(n, eng.sm_count)[0]
        mask = stepped_mask(n, eng.sm_count, rng)
        fet = rng.integers(I32MIN, I32MAX, n, dtype=np.int32, endpoint=True)
        pos = np.flatnonzero(mask).astype(np.int32)
        fet[pos[[0, pos.size // 2]]] = I32MIN, I32MAX                   # both extremes are hits
        # hits: [LO, HI) incl. both edges; misses: the fetch column's value, or just outside
        sel = np.where(mask, fet % (HI - LO) + LO, np.where((fet >= LO) & (fet < HI), HI, fet)).astype(np.int32)
        sel[pos[:2]] = LO, HI - 1
        miss = np.flatnonzero(~mask[:4 * STEP_ROWS])
        sel[miss[:3]] = LO - 1, I32MIN, I32MAX
        assert np.array_equal(port.select_scan(sel, LO, HI), pos)
        self.mask, self.fet, self.exp_pos = mask, fet, pos
        self.exp_val = fet[pos]
        self.perm = ((np.arange(n, dtype=np.int64) * 7_368_787 + 12_345) % n).astype(np.int32)
        assert np.gcd(7_368_787, n) == 1                                 # a permutation of 0..n-1
        self.ds, self.df, self.dperm = eng.upload(sel), eng.upload(fet), eng.upload(self.perm)
        h = max(pos.size, 1)
        self.pos, self.val = eng.alloc_i32(h), eng.alloc_i32(h)
        self.dcnt, self.dagg, self.dout = eng.alloc(8), eng.alloc(64), eng.alloc(64)
        self.blo, self.bhi = C.c_int32(LO), C.c_int32(HI)

    def free(self):
        for b in (self.ds, self.df, self.dperm, self.pos, self.val, self.dcnt, self.dagg, self.dout):
            b.free()

    @property
    def bounds(self):
        return C.byref(self.blo), C.byref(self.bhi)

    def count(self):
        return int(self.dcnt.to_host(1, np.int64)[0])

    def check_pos(self, exp, what):
        got = self.pos.to_host(exp.size)
        bad = np.flatnonzero(got != exp)
        assert bad.size == 0, (what, self.n, self.k, "first wrong position at", bad[:1], got[bad[:1]], exp[bad[:1]])

    def check_lists(self, what, base=0):
        self.check_pos(self.exp_pos + base, what)
        assert np.array_equal(self.val.to_host(self.exp_val.size), self.exp_val), (what, self.n, self.k)


def agg_of(a):
    from analytical_database_b200.engine import Agg
    return Agg(a.sum, a.count, a.min, a.max)


def check_agg(port, a, vals, what):
    a = agg_of(a)
    assert (a.count, a.sum) == (vals.size, int(vals.sum(dtype=np.int64))), what
    if vals.size:
        assert (a.min, a.max) == (int(vals.min()), int(vals.max())), what
        assert a.avg == port.avg(vals), what
    else:
        assert (a.min, a.max) == (I32MAX, I32MIN), what


@pytest.fixture(scope="module")
def eng():
    from analytical_database_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


def test_geometry_mirror():
    """The mirror's regimes on a B200: k = 1 up to 4 849 664 rows, k = 8 is one expansion step
    per chunk, k = 16 one aggregate-only gather round, and the largest shard's grid covers
    2^31 + 10 240 rows."""
    assert regime(1, 148) == (1, 4_849_664)
    assert select_geom(4_849_664, 148) == (1, 512, 9472) and select_geom(4_849_665, 148)[0] == 2
    assert select_geom(regime(8, 148)[1], 148)[1] == 32 * 4 * 32
    assert select_geom(regime(16, 148)[1], 148)[1] // 32 == 8 * 32
    k, chunk_rows, num_chunks = select_geom(I32MAX, 148)
    assert (k, num_chunks * chunk_rows) == (443, 2**31 + 10_240)
    for n in sizes(148):
        k = select_geom(n, 148)[0]
        assert regime(k, 148)[0] <= n <= regime(k, 148)[1]


@pytest.fixture(scope="module", params=sizes(148), ids=lambda n: f"n{n}")
def case(request, eng, port):
    n = request.param
    if eng.sm_count != 148:                               # place n in the same regime on this device
        per_k = eng.sm_count * 64 * SEL_WTILE
        k = select_geom(n, 148)[0]
        n = (k - 1) * per_k + 1 if n % 32 else k * per_k
    c = Case(eng, port, n)
    yield c
    c.free()


@pytest.mark.gpu
def test_select_scan(eng, port, case):
    c, lib = case, eng.lib
    lo, hi = c.bounds
    h = C.c_int64(-1)
    eng._ck(lib.adb_select_scan(c.ds.i32(), c.n, lo, hi, BASE, c.pos.i32(), c.dcnt.i64(), C.byref(h)))
    assert h.value == c.exp_pos.size and c.count() == h.value
    c.check_pos(c.exp_pos + BASE, "select_scan")


@pytest.mark.gpu
def test_select_count_emit(eng, port, case):
    """select_result's form: pairs through a permuted position list, then a device-side length
    that cuts into the last chunks."""
    c, lib = case, eng.lib
    lo, hi = c.bounds
    h = C.c_int64(-1)
    eng._ck(lib.adb_select_count(c.ds.i32(), c.n, None, lo, hi, c.dcnt.i64(), C.byref(h)))
    assert h.value == c.exp_pos.size and c.count() == h.value
    eng._ck(lib.adb_select_emit(c.dperm.i32(), 0, c.pos.i32()))
    c.check_pos(c.perm[c.exp_pos], "select_emit(d_pos_in)")
    live = c.n - 5000
    dn = eng.upload(np.array([live], np.int64))
    exp = c.exp_pos[:int(np.searchsorted(c.exp_pos, live))]
    eng._ck(lib.adb_select_count(c.ds.i32(), c.n, dn.i64(), lo, hi, None, C.byref(h)))
    assert h.value == exp.size
    eng._ck(lib.adb_select_emit(None, 7, c.pos.i32()))
    c.check_pos(exp + 7, "select_emit(d_n)")
    dn.free()


@pytest.mark.gpu
def test_select_count_base_emit(eng, port, case):
    """The count phase that totals its own counts (mask_kernel<true>, one ticket per warp)."""
    c, lib = case, eng.lib
    lo, hi = c.bounds
    h = C.c_int64(-1)
    eng._ck(lib.adb_select_count_base(c.ds.i32(), c.n, lo, hi, 0, c.dcnt.i64(), C.byref(h)))
    assert h.value == c.exp_pos.size and c.count() == h.value
    eng._ck(lib.adb_select_emit(None, BASE, c.pos.i32()))
    c.check_pos(c.exp_pos + BASE, "count_base + emit")


@pytest.mark.gpu
def test_chain_select_fetch_agg(eng, port, case):
    c, lib = case, eng.lib
    lo, hi = c.bounds
    eng._ck(lib.adb_chain_select_fetch_agg(c.ds.i32(), c.df.i32(), c.n, lo, hi, c.pos.i32(), c.val.i32(),
                                           c.dcnt.i64(), eng.agg_ptr(c.dagg)))
    assert c.count() == c.exp_pos.size
    check_agg(port, eng.read_agg(c.dagg), c.exp_val, "chain_select_fetch_agg")
    c.check_lists("chain_select_fetch_agg")


@pytest.mark.gpu
def test_chain_select_agg(eng, port, case):
    """The one-pass chain, on the column and on views that are only 4-byte aligned."""
    from analytical_database_b200.engine import _AggStruct
    c, lib = case, eng.lib
    lo, hi = c.bounds
    for off in (0, 1, 3):
        a = _AggStruct()
        eng._ck(lib.adb_chain_select_agg(c.ds.i32(off), c.df.i32(off), c.n - off, lo, hi, c.dcnt.i64(),
                                         eng.agg_ptr(c.dagg), C.byref(a)))
        vals = c.exp_val[c.exp_pos >= off]
        assert c.count() == vals.size, off
        check_agg(port, a, vals, ("chain_select_agg", off))


@pytest.mark.gpu
def test_deferred_emit_fetch_agg(eng, port, case):
    """count_base, the aggregate-only emit twice (the select stays pending: same generation),
    then the storing emit with the base_pos the count phase recorded."""
    from analytical_database_b200.engine import _AggStruct
    c, lib = case, eng.lib
    lo, hi = c.bounds
    h = C.c_int64(-1)
    eng._ck(lib.adb_select_count_base(c.ds.i32(), c.n, lo, hi, BASE, None, C.byref(h)))
    assert h.value == c.exp_pos.size
    gen = lib.adb_select_generation()
    for _ in range(2):
        a = _AggStruct()
        eng._ck(lib.adb_select_emit_fetch_agg(c.df.i32(), None, None, eng.agg_ptr(c.dagg), C.byref(a)))
        check_agg(port, a, c.exp_val, "emit_fetch_agg(NULL, NULL)")
        assert lib.adb_select_generation() == gen
    a = _AggStruct()
    eng._ck(lib.adb_select_emit_fetch_agg(c.df.i32(), c.pos.i32(), c.val.i32(), eng.agg_ptr(c.dagg), C.byref(a)))
    check_agg(port, a, c.exp_val, "emit_fetch_agg")
    c.check_lists("emit_fetch_agg", BASE)


@pytest.mark.gpu
def test_exchange_forms(eng, port, case):
    """The forms that carry the cross-context exchange, on a group of one context."""
    from analytical_database_b200.engine import _AggStruct
    c, lib = case, eng.lib
    lo, hi = c.bounds
    assert lib.adb_peer_connect_local(1) == 0, lib.adb_last_error()
    h = C.c_int64(-1)
    eng._ck(lib.adb_select_count_base(c.ds.i32(), c.n, lo, hi, 0, None, C.byref(h)))
    assert h.value == c.exp_pos.size
    a = _AggStruct()
    eng._ck(lib.adb_select_emit_fetch_agg_exchange(c.df.i32(), None, None, eng.agg_ptr(c.dagg),
                                                   eng.agg_ptr(c.dout), C.byref(a)))
    check_agg(port, a, c.exp_val, "emit_fetch_agg_exchange(NULL, NULL)")
    eng._ck(lib.adb_select_emit_fetch_agg_exchange(c.df.i32(), c.pos.i32(), c.val.i32(), eng.agg_ptr(c.dagg),
                                                   eng.agg_ptr(c.dout), C.byref(a)))
    check_agg(port, a, c.exp_val, "emit_fetch_agg_exchange")
    check_agg(port, eng.read_agg(c.dout), c.exp_val, "emit_fetch_agg_exchange d_out")
    c.check_lists("emit_fetch_agg_exchange")
    eng._ck(lib.adb_chain_select_fetch_agg_exchange(c.ds.i32(), c.df.i32(), c.n, lo, hi, c.pos.i32(), c.val.i32(),
                                                    c.dcnt.i64(), eng.agg_ptr(c.dagg), 1, eng.agg_ptr(c.dout)))
    assert c.count() == c.exp_pos.size
    check_agg(port, eng.read_agg(c.dagg), c.exp_val, "chain_select_fetch_agg_exchange")
    check_agg(port, eng.read_agg(c.dout), c.exp_val, "chain_select_fetch_agg_exchange d_out")
    c.check_lists("chain_select_fetch_agg_exchange")


# ---- the streaming operators past their grid caps (stream_grid in csrc/gather_agg.cu: 8 CTAs of
# 256 threads per SM; fetch's two-wide body runs once h / 4 > 1184 x 256, i.e. from 1 212 420
# positions, aggregate's grid stops growing at 16 x 1184 x 256 = 4 849 664 rows, add / sub's at
# 2 424 832) ----
@pytest.mark.gpu
@pytest.mark.parametrize("h", [1_212_420, 2_500_001, 5_000_003])
def test_fetch_past_the_grid_cap(eng, port, h):
    rng = np.random.default_rng(h)
    n = 6_000_000
    data = rng.integers(I32MIN, I32MAX, n, dtype=np.int32, endpoint=True)
    col = eng.upload(data)
    pos = np.sort(rng.integers(0, n, h)).astype(np.int32)
    dp = eng.upload(pos)
    out = eng.fetch(col, dp, h)
    assert np.array_equal(out.to_host(h), port.fetch(data, pos))
    # unsorted positions + base offset + a device-side length that leaves a ragged tail
    pos2 = rng.integers(0, n, h).astype(np.int32)
    dp2 = eng.upload(pos2 + 77)
    live = h - 3
    dn = eng.upload(np.array([live], np.int64))
    out2 = eng.fetch(col, dp2, h, d_n=dn, base=77)
    assert np.array_equal(out2.to_host(live), port.fetch(data, pos2[:live]))
    for b in (col, dp, out, dp2, dn, out2):
        b.free()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4_849_665, 20_000_003])
def test_aggregate_past_the_grid_cap(eng, port, n):
    rng = np.random.default_rng(n)
    near_max = rng.integers(I32MAX - 10000, I32MAX, n + 3, dtype=np.int32, endpoint=True)
    full = rng.integers(I32MIN, I32MAX, n + 3, dtype=np.int32, endpoint=True)
    full[[5, n - 7]] = I32MIN, I32MAX
    for name, data in (("near_max", near_max), ("full", full)):
        buf = eng.upload(data)
        for off in (0, 1, 3):
            v = data[off:off + n]
            a = eng.aggregate(buf, n, offset=off)
            assert a.count == n and a.sum == port.sum(v), (name, off)
            assert (a.min, a.max) == (port.min(v), port.max(v)), (name, off)
            assert a.avg == port.avg(v), (name, off)
            if name == "near_max":
                assert a.sum > 2**53                     # beyond what a double holds exactly
        buf.free()


@pytest.mark.gpu
def test_add_sub_past_the_grid_cap(eng, port):
    n = 5_000_011
    rng = np.random.default_rng(n)
    a = rng.integers(I32MIN, I32MAX, n, dtype=np.int32, endpoint=True)
    b = rng.integers(I32MIN, I32MAX, n, dtype=np.int32, endpoint=True)
    da, db = eng.upload(a), eng.upload(b)
    for sub in (False, True):
        out = eng.ewise(da, db, n, sub)
        assert np.array_equal(out.to_host(n), port.sub(a, b) if sub else port.add(a, b)), sub
        out.free()
    da.free(), db.free()


# ---- the largest legal shard: n = 2^31 - 1, positions up to 2^31 - 2 (opt-in) ----------------------
@pytest.mark.gpu
@pytest.mark.skipif(not os.environ.get("ADB_TEST_MAX_SHARD"),
                    reason="set ADB_TEST_MAX_SHARD=1: two 2^31 - 1 row columns, ~22 GB of HBM")
def test_largest_shard(eng, port):
    """The chain in its three forms (materialised, one pass, deferred aggregate-only) at about
    30 % and 1 %: they agree with each other and with select + fetch + aggregate, and the lists
    are exact over windows regenerated on the host at the start and the end of the shard."""
    from analytical_database_b200 import synth
    from analytical_database_b200.engine import _AggStruct
    lib = eng.lib
    n, seed, w = I32MAX, 2031, 4_000_000
    sel = eng.synth_uniform(n, seed, 0, 0, 1 << 31)
    fet = eng.synth_uniform(n, seed + 1, 0, I32MIN, (1 << 32) - 1)
    windows = [(first, synth.uniform(w, seed, first, 0, 1 << 31), synth.uniform(w, seed + 1, first, I32MIN, (1 << 32) - 1))
               for first in (0, n - w)]
    dcnt, dagg = eng.alloc(8), eng.alloc(64)
    for lo, hi in ((0, int(0.3 * 2**31)), (1000, 1000 + 2**31 // 100)):
        blo, bhi = C.c_int32(lo), C.c_int32(hi)
        plo, phi = C.byref(blo), C.byref(bhi)
        h = C.c_int64(-1)
        eng._ck(lib.adb_select_count_base(sel.i32(), n, plo, phi, 0, None, C.byref(h)))
        h = h.value
        deferred = _AggStruct()
        eng._ck(lib.adb_select_emit_fetch_agg(fet.i32(), None, None, eng.agg_ptr(dagg), C.byref(deferred)))
        one_pass = _AggStruct()
        eng._ck(lib.adb_chain_select_agg(sel.i32(), fet.i32(), n, plo, phi, dcnt.i64(), eng.agg_ptr(dagg),
                                         C.byref(one_pass)))
        assert int(dcnt.to_host(1, np.int64)[0]) == h
        pos, val = eng.alloc_i32(h), eng.alloc_i32(h)
        eng._ck(lib.adb_chain_select_fetch_agg(sel.i32(), fet.i32(), n, plo, phi, pos.i32(), val.i32(), dcnt.i64(),
                                               eng.agg_ptr(dagg)))
        fused = eng.read_agg(dagg)
        assert int(dcnt.to_host(1, np.int64)[0]) == h

        def check_windows(what):
            for first, s_w, f_w in windows:
                exp = np.flatnonzero((s_w >= lo) & (s_w < hi)).astype(np.int64) + first
                at = 0 if first == 0 else h - exp.size
                assert np.array_equal(pos.to_host(exp.size, offset_bytes=4 * at), exp), (what, lo, first)
                assert np.array_equal(val.to_host(exp.size, offset_bytes=4 * at), f_w[exp - first]), (what, lo, first)
        check_windows("chain_select_fetch_agg")
        assert pos.to_host(1, offset_bytes=4 * (h - 1))[0] > n - 1000          # positions reach the shard's end
        p2, _, h2 = eng.select_scan(sel, n, lo, hi, out=pos, d_count=dcnt)
        val = eng.fetch(fet, pos, h, d_n=dcnt, out=val)
        plain = eng.aggregate(val, h, d_n=dcnt)
        assert h2 == h
        check_windows("select_scan + fetch")
        got = [agg_of(a) for a in (deferred, one_pass)] + [fused, plain]
        assert all(g == plain for g in got), (lo, hi, got)
        assert plain.count == h and abs(h - n * (hi - lo) / 2**31) < 10 * (n * (hi - lo) / 2**31) ** 0.5
        pos.free(), val.free()
    for b in (sel, fet, dcnt, dagg):
        b.free()


# ---- through the operator API (host/query_shim.c): select_column -> fetch_column -> aggregates, then
# the handles are read -- the lazy bitmap_gather_agg<true> answers the first aggregate, the
# materialising expand<false,true,true> the next, on every context's shard ----------------------------
def shard_sizes(n, gpus):
    """The shim's row-range shards (query_shim.c: ceil(n / G) rounded up to 32 rows)."""
    rows = ((n + gpus - 1) // gpus + 31) // 32 * 32
    return [max(0, min(rows, n - g * rows)) for g in range(gpus)]


API_CASES = {2: 17, 3: 9}                # contexts: the least k of every shard


def api_rows(gpus, k_min):
    """The fewest rows whose every shard (of `gpus`) runs with at least k_min tiles per warp on a
    B200, plus a ragged tail."""
    per_k = 148 * 64 * SEL_WTILE
    return gpus * ((k_min - 1) * per_k + 32 * gpus) + 5


def test_api_rows_place_every_shard():
    for gpus, k_min in API_CASES.items():
        assert all(select_geom(s, 148)[0] >= k_min for s in shard_sizes(api_rows(gpus, k_min), gpus))


@pytest.fixture(scope="module", params=sorted(API_CASES), ids=lambda g: f"{g}ctx")
def api(request, eng):
    """Like test_gpu_query_api.py's: every column row-range sharded over the contexts of ONE
    process.  The shim starts from contexts of its own and shuts every context down when it
    ends, so the module's engine is closed first and these tests run last in this module."""
    from query_api import Api
    eng.close()
    a = Api()
    assert a.lib.adb_host_init_multi(request.param) == 0, a.lib.adb_host_last_error()
    yield a
    a.lib.adb_host_shutdown()


@pytest.mark.gpu
@pytest.mark.parametrize("bound", ["dense", "sparse"])
def test_operator_api_chain_on_large_shards(api, port, bound):
    gpus = api.lib.adb_host_gpus()
    n = api_rows(gpus, API_CASES[gpus])
    rng = np.random.default_rng(n)
    c1 = rng.integers(-n // 2, n // 2, n, dtype=np.int32)
    c4 = rng.integers(I32MIN, I32MAX, n, dtype=np.int32, endpoint=True)
    lo, hi = (-n // 4, n // 4) if bound == "dense" else (100, 100 + n // 300)
    epos = np.flatnonzero((c1 >= lo) & (c1 < hi)).astype(np.int32)
    c4[epos[[1, -2]]] = I32MIN, I32MAX
    evals = c4[epos]
    col1, col4 = api.column(c1), api.column(c4)
    s = api.select_column(col1, lo, hi)
    assert s.contents.num_tuples == epos.size
    f = api.fetch_column(col4, s)
    a = api.sum_result(f)                                  # lazy: nothing written yet
    assert int(api.tuples(a)[0]) == int(evals.sum(dtype=np.int64))
    av = api.unary("average", f)                           # writes the handles on the way
    assert api.tuples(av)[0].tobytes() == np.float64(port.avg(evals)).tobytes()
    mn, mx = api.unary("min", f), api.unary("max", f)
    assert (int(api.tuples(mn)[0]), int(api.tuples(mx)[0])) == (I32MIN, I32MAX)
    assert np.array_equal(api.tuples(f), evals)
    assert np.array_equal(api.tuples(s), epos)
    for r in (s, f, a, av, mn, mx):
        api.drop(r)
