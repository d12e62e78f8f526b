"""The hash and nested-loop joins at the launch geometry of real-size inputs, exact against numpy.

join_reference.py restates the oracle's joins in numpy (pinned to the oracle here, on the CPU)
and mirrors where the join's geometry changes.  The one-context cases sit on both sides of every
boundary of it: partition bits (nb = 2049 / 2050, 1 049 599 / 1 049 600), the shared- vs
global-memory table build (partitions of exactly 1638 and 1639 rows), one key of 70 000 rows,
partitions made of 2-, 3-, 8- and 9-row groups only, the direct probe's 32 / 64 rows per warp
(np = 303 104 / 303 105, and a ragged 10 M), the partitioned probe's one / two tiles per window
(np = 1 048 576 / 1 048 577, and 30 M with a ragged last window), a tile whose rows share one
table slice, and per-row match counts of 0, 1, 2, 3, 8, 9, 32, 33 and 4097 inside one expansion
step and across pieces and windows.  Every case runs both ADB_JOIN_PROBE forms and the default,
which must take the form the size rule names.  Then the 2^31-pair bound on one context and on
several, the sharded join at sizes where every owner probes slice by slice, and the sharded join
in a fresh process whose streams all share one hardware work queue.  Opt-in
(ADB_TEST_MAX_JOIN=1): a join just below the bound (~17 GB of output), and a build side past
the 20-bit partition cap."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import join_reference as jr
from join_reference import I32MAX, I32MIN

SM = 148                                # the B200's SMs: the geometry the cases are placed for
MIX = (0, 1, 2, 3, 8, 9, 32, 33, 4097)  # per-probe-row match counts
PROBE_P = (0.3, 0.33, 0.15, 0.1, 0.05, 0.04, 0.015, 0.015)      # of MIX[:-1]; MIX[-1] takes BIG_P
BIG_P = 2e-5
FILL = np.array([1, 2, 3, 8, 9, 32, 33])
FILL_P = (0.55, 0.2, 0.12, 0.05, 0.05, 0.02, 0.01)
STAGE = {False: "probe + piece offsets", True: "probe slice by slice + back to row order"}
FORMS = ("direct", "partitioned", None)                      # None: the engine's own size rule
HOT_ROWS = 70_000                                            # > 65 535: past a 16-bit group size


# ---- inputs ----------------------------------------------------------------------------------------
def distinct_keys(rng, part_lo, part_hi, bits, n):
    """n distinct keys whose join partitions (of `bits`) lie in [part_lo, part_hi)."""
    lo, hi = part_lo << (32 - bits), part_hi << (32 - bits)
    h = np.sort(rng.integers(lo, hi, n + n // 4 + 16, dtype=np.uint64))
    h = h[np.concatenate([[True], h[1:] != h[:-1]])]
    assert h.size >= n
    rng.shuffle(h)
    return jr.keys_of_hashes(h[:n])


def fill_sizes(rng, total, big=0):
    """Group sizes summing to `total`: `big` groups of 4097 rows, the rest drawn from FILL."""
    s = np.concatenate([np.full(big, 4097), rng.choice(FILL, total // 2 + 16, p=FILL_P)])
    c = np.cumsum(s)
    cut = int(np.searchsorted(c, total))
    s = s[:cut + 1].copy()
    s[-1] -= c[cut] - total
    return s


def positions(rng, n):
    """Distinct positions (an affine permutation of 0 .. n-1), a quarter of them with bit 31 set."""
    a = int(rng.integers(n // 3 + 1, 2 * n // 3 + 2)) if n else 1
    while np.gcd(a, max(n, 1)) != 1:
        a += 1
    p = (np.arange(n, dtype=np.int64) * a + int(rng.integers(0, max(n, 1)))) % max(n, 1)
    p[rng.random(n) < 0.25] |= 1 << 31
    return p.astype(np.uint32).view(np.int32)


class Build:
    """A build side made of groups of known size; spec = [(first partition, end, sizes)]."""

    def __init__(self, rng, nb, spec, bits=None):
        self.bits = bits or jr.part_bits(nb)
        keys = [distinct_keys(rng, lo, hi, self.bits, len(sz)) for lo, hi, sz in spec]
        self.gkeys = np.concatenate(keys)
        self.gsizes = np.concatenate([np.asarray(sz, np.int64) for _, _, sz in spec])
        assert self.gsizes.sum() == nb
        self.keys = np.repeat(self.gkeys, self.gsizes)
        rng.shuffle(self.keys)                          # groups interleave in insertion order
        self.pos = positions(rng, nb)
        # the second row of a 2-row group at INT32_MAX (fits the slot's pair form) and at -1
        # (bit 31 set: the slot falls back to the group form)
        self.pair_keys = self.gkeys[self.gsizes == 2][:2]
        for key, p in zip(self.pair_keys, (I32MAX, -1)):
            self.pos[np.flatnonzero(self.keys == key)[1]] = p
        self._sorted, order = jr.stable_sort(self.gkeys)
        self._sizes = self.gsizes[order]
        assert np.all(self._sorted[1:] != self._sorted[:-1])            # one group per key

    def counts(self, probe_keys):
        """Matches of every probe key."""
        i = np.minimum(np.searchsorted(self._sorted, probe_keys), self._sorted.size - 1)
        return np.where(self._sorted[i] == probe_keys, self._sizes[i], 0)

    def misses(self, rng, n, slice_=None):
        h = rng.integers(0, 1 << 32, n, dtype=np.uint64)
        if slice_ is not None:
            h = (h & np.uint64(0xFFFFFF)) | np.uint64(slice_ << 24)
        k = jr.keys_of_hashes(h)
        return k[self.counts(k) == 0]


def general_build(rng, nb):
    return Build(rng, nb, [(0, 1 << jr.part_bits(nb), fill_sizes(rng, nb, big=nb // 500_000 + 2))])


def boundary_rows(n):
    """Rows that end a piece of the direct probe, a piece of the partitioned probe or a window."""
    rows = set()
    rpw = jr.probe_geom(n, SM)[2]
    wrows = jr.window_tiles(n) * jr.RADIX_TILE
    for step, count in ((rpw, -(-n // rpw)), (jr.PIECE_PARTITIONED, -(-n // jr.PIECE_PARTITIONED)),
                        (wrows, jr.windows(n))):
        rows |= {step * i for i in (1, 2, count // 2, count - 1) if 2 <= step * i < n - 2}
    return sorted(rows)


def probe_keys(rng, n, b, one_slice=True):
    """n probe keys whose match counts are drawn from MIX, with every class in one expansion step,
    the heaviest at piece and window edges, the pair groups with the special positions, and (n
    of a tile or more) 300 rows of one tile in one table slice."""
    by = {s: b.gkeys[b.gsizes == s] for s in MIX[1:]}
    by = {s: k for s, k in by.items() if k.size}
    miss = b.misses(rng, max(1024, n // 64))
    classes = [0] + sorted(by)
    p = np.array([dict(zip(MIX, PROBE_P + (BIG_P,)))[s] for s in classes])
    cls = rng.choice(np.array(classes), n, p=p / p.sum())
    k = np.empty(n, np.int32)
    for s in classes:
        at = np.flatnonzero(cls == s)
        k[at] = rng.choice(by[s] if s else miss, at.size)
    def one_of(s):
        return by[s][0] if s in by else by[max(by)][0]
    if n >= jr.STEP_ROWS * 6:
        step = jr.STEP_ROWS * 5 + 7                     # one step, not at its start
        k[step:step + len(MIX)] = [miss[0]] + [one_of(s) for s in MIX[1:]]
    for r in boundary_rows(n):
        k[r - 2:r + 2] = [one_of(2), one_of(4097), one_of(33), one_of(9)]
    if n >= 8:
        k[3:3 + len(b.pair_keys)] = b.pair_keys
    if one_slice and n >= 3 * jr.RADIX_TILE:
        t0 = (n // jr.RADIX_TILE // 2) * jr.RADIX_TILE + 700
        s = int(jr.slice_of(b.gkeys[:1])[0])
        hits = b.gkeys[(jr.slice_of(b.gkeys) == s) & (b.gsizes <= 3)]
        pool = np.concatenate([hits, b.misses(rng, 4096, s)])
        k[t0:t0 + 300] = rng.choice(pool, 300)
        assert np.all(jr.slice_of(k[t0:t0 + 300]) == s)
    return k


def probe_side(rng, n, b, one_slice=True):
    k = probe_keys(rng, n, b, one_slice)
    p = positions(rng, n)
    if n >= 2:
        p[[0, n - 1]] = I32MAX, -1
    return k, p


# ---- CPU: the reference against the oracle, the geometry mirror, the inputs ------------------------
def oracle_inputs(kind, n1, n2, rng):
    if kind == "uniform":
        k1, k2 = rng.integers(0, max(n1 // 4, 2), n1), rng.integers(0, max(n1 // 4, 2), n2)
    elif kind == "unique":
        k1, k2 = rng.permutation(4 * max(n1, n2, 1))[:n1], rng.permutation(4 * max(n1, n2, 1))[:n2]
    elif kind == "zipf":
        k1, k2 = rng.zipf(1.3, n1) % 1000, rng.zipf(1.3, n2) % 1000
    elif kind == "negative":
        k1, k2 = rng.integers(-max(n1 // 4, 2), max(n1 // 4, 2), n1), rng.integers(-max(n1 // 4, 2), max(n1 // 4, 2), n2)
    else:                                               # hot: one key on most rows of both sides
        k1, k2 = rng.integers(0, 50, n1), rng.integers(0, 50, n2)
        k1[rng.random(n1) < 0.6], k2[rng.random(n2) < 0.3] = 7, 7
    return (k1.astype(np.int32), positions(rng, n1), k2.astype(np.int32), positions(rng, n2))


@pytest.mark.parametrize("kind", ["uniform", "unique", "zipf", "negative", "hot"])
@pytest.mark.parametrize("n1,n2", [(0, 0), (0, 9), (9, 0), (1, 1), (2, 3), (300, 200), (3000, 1500)])
def test_reference_equals_the_oracle(port, kind, n1, n2):
    rng = np.random.default_rng(n1 * 7 + n2 + len(kind))
    k1, p1, k2, p2 = oracle_inputs(kind, n1, n2, rng)
    if n1 > 1 and n2 > 1:
        p1[1], p2[0] = I32MAX, I32MAX                  # both ends of the position domain
        p1[0], p2[1] = I32MIN, -1
    for name in ("hash_join", "nested_loop_join"):
        got, want = getattr(jr, name)(k1, p1, k2, p2), getattr(port, name)(k1, p1, k2, p2)
        assert got[0].dtype == np.int32 and got[1].dtype == np.int32, name
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (name, kind, n1, n2)


def test_geometry_mirror():
    """The boundaries of the join's geometry at 148 SMs."""
    assert [jr.part_bits(n) for n in (1, 2049, 2050, 1_049_599, 1_049_600)] == [1, 1, 2, 10, 11]
    assert jr.part_bits(537_395_199) == 19 and jr.part_bits(537_395_200) == 20 == jr.part_bits(I32MAX)
    assert jr.builds_in_shared_memory(1638) and not jr.builds_in_shared_memory(1639)
    assert (jr.table_slots(1638), jr.table_slots(1639), jr.table_slots(1)) == (2048, 4096, 16)
    assert jr.probe_geom(303_104, SM) == (1184, 9472, 32) and jr.probe_geom(303_105, SM)[2] == 64
    assert jr.probe_geom(10_000_019, SM)[2] * 9472 > 10_000_019 > (jr.probe_geom(10_000_019, SM)[2] - 32) * 9472
    assert (jr.window_tiles(1_048_576), jr.windows(1_048_576)) == (1, 256)
    assert (jr.window_tiles(1_048_577), jr.windows(1_048_577)) == (2, 129)
    assert jr.window_tiles(100_000_000) == 96
    assert (jr.window_tiles(30_000_017), jr.windows(30_000_017)) == (29, 253)
    assert -(-30_000_017 // 4096) - 252 * 29 == 17                  # the last window: 17 of 29 tiles
    assert jr.row_scan_is_warp_wide(536_870_912) and not jr.row_scan_is_warp_wide(536_870_913)
    assert jr.partitioned_by_default(6 << 20, 4 << 20)
    assert not jr.partitioned_by_default((6 << 20) - 1, 4 << 20)
    assert not jr.partitioned_by_default(6 << 20, (4 << 20) - 1)
    for gpus, (nb, n) in SHARDED.items():                          # an even split meets the owner's rule
        assert jr.owner_partitioned_by_default(n // gpus, nb // gpus)


def build_side_spec(rng, nb):
    """nb = 2049 / 2050: partition 0 holds 1638 / 1639 rows.  nb ~ 1 M: partitions 0-6 hold 1638
    rows, 1639 rows, the hot key, and 2-, 3-, 8- and 9-row groups only; the rest is mixed."""
    bits = jr.part_bits(nb)
    if nb < 4096:
        first = 1638 if nb == 2049 else 1639
        return [(0, 1, fill_sizes(rng, first)), (1, 1 << bits, fill_sizes(rng, nb - first))]
    spec = [(0, 1, fill_sizes(rng, 1638)), (1, 2, fill_sizes(rng, 1639)),
            (2, 3, np.concatenate([[HOT_ROWS], np.ones(300, np.int64)])),
            (3, 4, np.full(600, 2)), (4, 5, np.full(400, 3)), (5, 6, np.full(150, 8)), (6, 7, np.full(133, 9))]
    used = sum(int(np.sum(s)) for _, _, s in spec)
    return spec + [(7, 1 << bits, fill_sizes(rng, nb - used, big=2))]


BUILD_NB = (2049, 2050, 1_049_599, 1_049_600)


@pytest.mark.parametrize("nb", BUILD_NB)
def test_build_sides_place_their_partitions(nb):
    b = Build(np.random.default_rng(nb), nb, build_side_spec(np.random.default_rng(nb), nb))
    rows = np.bincount(jr.partition_of(b.keys, b.bits), minlength=1 << b.bits)
    if nb < 4096:
        assert rows[0] == (1638 if nb == 2049 else 1639) and rows.sum() == nb
        return
    assert (rows[0], rows[1], rows[2]) == (1638, 1639, HOT_ROWS + 300)
    for p, g in zip(range(3, 7), (2, 3, 8, 9)):
        assert set(b.counts(b.keys[jr.partition_of(b.keys, b.bits) == p]).tolist()) == {g}
    assert np.bincount(b.gsizes)[[2, 8, 9, 32, 33, 4097]].min() > 0


# ---- GPU, one context ----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from analytical_database_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(autouse=True)
def default_env(monkeypatch):
    for var in ("ADB_JOIN_PROBE", "ADB_TRACE"):
        monkeypatch.delenv(var, raising=False)


def check_pairs(got1, got2, want, what):
    bad = np.flatnonzero((got1 != want[0]) | (got2 != want[1]))
    assert bad.size == 0, (what, "first wrong pair", int(bad[0]), (got1[bad[0]], got2[bad[0]]),
                           (want[0][bad[0]], want[1][bad[0]]), "of", bad.size)


def run_forms(eng, monkeypatch, capfd, sides, want, forms=FORMS, nested=False, what=""):
    """The join of `sides` in every form: exact, and with the stage its form names."""
    k1, p1, k2, p2 = sides
    nb, n_probe = (k2.size, k1.size) if nested else (k1.size, k2.size)
    d = [eng.upload(x) for x in sides]
    monkeypatch.setenv("ADB_TRACE", "1")
    for form in forms:
        if form:
            monkeypatch.setenv("ADB_JOIN_PROBE", form)
        else:
            monkeypatch.delenv("ADB_JOIN_PROBE", raising=False)
        capfd.readouterr()
        o1, o2, m = eng.join(d[0], d[1], k1.size, d[2], d[3], k2.size, nested_loop=nested)
        trace = capfd.readouterr().err
        partitioned = form == "partitioned" if form else jr.partitioned_by_default(nb, n_probe)
        assert STAGE[partitioned] in trace and STAGE[not partitioned] not in trace, (what, form, trace)
        assert m == want[0].size, (what, form, m, want[0].size)
        if m:
            check_pairs(o1.to_host(m), o2.to_host(m), want, (what, form))
        o1.free(), o2.free()
    for x in d:
        x.free()


@pytest.mark.gpu
@pytest.mark.parametrize("nb", BUILD_NB)
def test_build_side_geometry(eng, monkeypatch, capfd, nb):
    rng = np.random.default_rng(nb)
    b = Build(rng, nb, build_side_spec(np.random.default_rng(nb), nb))
    k2, p2 = probe_side(rng, 1_000_003, b)
    if nb > 4096:
        k2[[11, 500_000, 999_990]] = b.gkeys[b.gsizes == HOT_ROWS][0]
        for p, g in zip(range(3, 7), (2, 3, 8, 9)):     # every row of the one-size partitions, in order
            pk = np.unique(b.keys[jr.partition_of(b.keys, b.bits) == p])
            k2[20_000 * p:20_000 * p + pk.size] = pk
    sides = (b.keys, b.pos, k2, p2)
    run_forms(eng, monkeypatch, capfd, sides, jr.hash_join(*sides), what=nb)


@pytest.mark.gpu
@pytest.mark.parametrize("n_probe", [303_104, 303_105, 10_000_019])
def test_direct_probe_geometry(eng, monkeypatch, capfd, n_probe):
    rng = np.random.default_rng(n_probe)
    b = general_build(rng, 1_500_000)
    k2, p2 = probe_side(rng, n_probe, b)
    sides = (b.keys, b.pos, k2, p2)
    run_forms(eng, monkeypatch, capfd, sides, jr.hash_join(*sides), what=n_probe)


@pytest.mark.gpu
@pytest.mark.parametrize("n_probe", [1_048_576, 1_048_577, 30_000_017])
def test_partitioned_probe_geometry(eng, monkeypatch, capfd, n_probe):
    rng = np.random.default_rng(n_probe)
    b = general_build(rng, 2_000_000)
    k2, p2 = probe_side(rng, n_probe, b)
    sides = (b.keys, b.pos, k2, p2)
    run_forms(eng, monkeypatch, capfd, sides, jr.hash_join(*sides), what=n_probe)


@pytest.mark.gpu
@pytest.mark.parametrize("nb,n_probe", [(6 << 20, 4 << 20), ((6 << 20) - 1, 4 << 20), (6 << 20, (4 << 20) - 1)])
def test_default_form_thresholds(eng, monkeypatch, capfd, nb, n_probe):
    rng = np.random.default_rng(nb + n_probe)
    b = general_build(rng, nb)
    k2, p2 = probe_side(rng, n_probe, b)
    sides = (b.keys, b.pos, k2, p2)
    run_forms(eng, monkeypatch, capfd, sides, jr.hash_join(*sides), forms=(None,), what=(nb, n_probe))


@pytest.mark.gpu
def test_nested_loop_join_geometry(eng, monkeypatch, capfd):
    """10 M outer rows (side one, probed) against 3 M inner rows (side two, built)."""
    rng = np.random.default_rng(103)
    b = general_build(rng, 3_000_000)
    k1, p1 = probe_side(rng, 10_000_019, b)
    sides = (k1, p1, b.keys, b.pos)
    run_forms(eng, monkeypatch, capfd, sides, jr.nested_loop_join(*sides), nested=True, what="nested")


# ---- the 2^31-pair bound ---------------------------------------------------------------------------
BOUND_ROWS = 46_341                     # 46 341^2 = 2 147 488 281 pairs of one key: >= 2^31


def small_join(rng):
    k1, k2 = rng.integers(0, 20_000, 70_000).astype(np.int32), rng.integers(0, 20_000, 50_000).astype(np.int32)
    return k1, positions(rng, k1.size), k2, positions(rng, k2.size)


@pytest.mark.gpu
def test_pair_bound_one_context(eng):
    from analytical_database_b200.engine import EngineError
    k = eng.upload(np.full(BOUND_ROWS, 7, np.int32))
    p = eng.upload(np.arange(BOUND_ROWS, dtype=np.int32))
    with pytest.raises(EngineError, match="2147488281 pairs"):
        eng.join(k, p, BOUND_ROWS, k, p, BOUND_ROWS)
    k.free(), p.free()
    sides = small_join(np.random.default_rng(1))
    d = [eng.upload(x) for x in sides]
    o1, o2, m = eng.join(d[0], d[1], sides[0].size, d[2], d[3], sides[2].size)
    want = jr.hash_join(*sides)
    assert m == want[0].size
    check_pairs(o1.to_host(m), o2.to_host(m), want, "after the refused join")
    for x in d + [o1, o2]:
        x.free()


@pytest.mark.gpu
@pytest.mark.skipif(not os.environ.get("ADB_TEST_MAX_JOIN"),
                    reason="set ADB_TEST_MAX_JOIN=1: ~17 GB of output")
def test_largest_join(eng):
    """46 340 x 46 341 rows of one key: 2 147 441 940 pairs, just below the bound.  Windows at the
    start, middle and end of the output must be the reference's."""
    n1, n2, w = BOUND_ROWS, BOUND_ROWS - 1, 3_000_000
    rng = np.random.default_rng(2)
    p1, p2 = positions(rng, n1), positions(rng, n2)
    k = eng.upload(np.full(n1, 7, np.int32))
    d1, d2 = eng.upload(p1), eng.upload(p2)
    o1, o2, m = eng.join(k, d1, n1, k, d2, n2)
    assert m == n1 * n2 == 2_147_441_940
    for at in (0, m // 2 - w // 2, m - w):
        i = np.arange(at, at + w, dtype=np.int64)
        assert np.array_equal(o1.to_host(w, offset_bytes=4 * at), p1[i % n1]), at
        assert np.array_equal(o2.to_host(w, offset_bytes=4 * at), p2[i // n1]), at
    for x in (k, d1, d2, o1, o2):
        x.free()


@pytest.mark.gpu
@pytest.mark.skipif(not os.environ.get("ADB_TEST_MAX_JOIN"),
                    reason="set ADB_TEST_MAX_JOIN=1: a 1.76 G-row build side")
def test_build_past_the_partition_cap(eng):
    """1.76 G unique build keys: 20 partition bits, ~1678 rows per partition, so most partitions
    build in global memory.  Build key i has position (i * MUL + ADD) mod 2^31."""
    nb, n_probe, mul, add = 1_760_000_000, 20_000_003, 1_000_003, 12_345
    assert jr.part_bits(nb) == 20 and not jr.builds_in_shared_memory(nb >> 20)
    rng = np.random.default_rng(3)
    bk, bp = eng.alloc_i32(nb), eng.alloc_i32(nb)
    eng._ck(eng.lib.adb_iota_i32(bk.i32(), nb, 0))
    eng._ck(eng.lib.adb_synth_affine(bp.i32(), nb, 0, mul, add, 1 << 31))
    k2 = rng.integers(0, nb + nb // 8, n_probe).astype(np.int32)
    p2 = positions(rng, n_probe)
    d2, dp2 = eng.upload(k2), eng.upload(p2)
    o1, o2, m = eng.join(bk, bp, nb, d2, dp2, n_probe)
    hit = k2 < nb
    want = (((k2[hit].astype(np.int64) * mul + add) % (1 << 31)).astype(np.int32), p2[hit])
    assert m == want[0].size
    check_pairs(o1.to_host(m), o2.to_host(m), want, "past the partition cap")
    for x in (bk, bp, d2, dp2, o1, o2):
        x.free()


# ---- several contexts, through the operator API (host/query_shim.c) ----------------------------------
# (build rows, probe rows): every owner holds >= 24 Mi build rows and receives >= 4 Mi probe keys
SHARDED = {2: (53_000_000, 10_000_000), 3: (80_000_000, 14_000_000)}
SHIM_VARS = ("ADB_SHIM_MIRROR", "ADB_SHIM_EAGER", "ADB_SHARD_MIN_ROWS", "ADB_REBALANCE_MIN", "ADB_FETCH_ROUTE_MIN")


@pytest.fixture(scope="module", params=sorted(SHARDED), ids=lambda g: f"{g}ctx")
def api(request, eng):
    """G fresh contexts in this process; they share the device on a box with fewer.  The shim
    starts contexts of its own and shuts every context down when it ends, so the module's engine
    is closed first and these tests run last."""
    from query_api import Api
    eng.close()
    with pytest.MonkeyPatch.context() as mp:
        for var in SHIM_VARS:
            mp.delenv(var, raising=False)
        a = Api()
        a.lib.adb_host_shutdown()
        assert a.lib.adb_host_init_multi(request.param) == 0, a.lib.adb_host_last_error()
        yield a
        a.lib.adb_host_shutdown()


@pytest.fixture(scope="module")
def launch_count():
    import analytical_database_b200 as adb
    lib = C.CDLL(adb.lib_path())                      # the engine libadb_query.so drives
    lib.adb_launch_count_all.restype = C.c_int64
    return lib.adb_launch_count_all


def home_of_rows(n, gpus):
    """The context each probe row lives on (query_shim.c: shards of ceil(n / G) rounded to 32)."""
    rows = ((n + gpus - 1) // gpus + 31) // 32 * 32
    return np.arange(n) // rows


def api_join(api, sides, want, what):
    R = [C.pointer(api.host_result(x)) for x in sides]
    o1, o2 = api.join("hash_join", *R)
    got1, got2 = api.tuples(o1), api.tuples(o2)
    api.drop(o1), api.drop(o2)
    assert got1.size == want[0].size, what
    check_pairs(got1, got2, want, what)


@pytest.mark.gpu
def test_sharded_owner_probe_geometry(api, launch_count, monkeypatch):
    """Every owner's default size rule picks the partitioned probe: the default launches what the
    forced partitioned form launches, more than the forced direct form; every form is exact.
    Groups of more than 8 rows on every owner are probed from other contexts, so the sharded
    expansion reads them from remote sorted build positions."""
    G = api.lib.adb_host_gpus()
    nb, n_probe = SHARDED[G]
    rng = np.random.default_rng(G)
    b = general_build(rng, nb)
    k2, p2 = probe_side(rng, n_probe, b, one_slice=False)
    b_owner, p_owner = jr.route_owner(b.keys, G), jr.route_owner(k2, G)
    assert all(jr.owner_partitioned_by_default(int(np.sum(p_owner == o)), int(np.sum(b_owner == o)))
               for o in range(G))
    long_remote = (b.counts(k2) > 8) & (p_owner != home_of_rows(n_probe, G))
    assert set(p_owner[long_remote].tolist()) == set(range(G))
    sides = (b.keys, b.pos, k2, p2)
    want = jr.hash_join(*sides)
    launches = {}
    for form in (None, "direct", "partitioned", "default"):       # the first call sizes the exchange
        if form in ("direct", "partitioned"):
            monkeypatch.setenv("ADB_JOIN_PROBE", form)
        else:
            monkeypatch.delenv("ADB_JOIN_PROBE", raising=False)
        before = launch_count()
        api_join(api, sides, want, (G, form))
        launches[form] = launch_count() - before
    assert launches["default"] == launches["partitioned"] > launches["direct"], launches


@pytest.mark.gpu
def test_sharded_pair_bound(api):
    """46 341 x 46 341 rows of one key: every context's share of the pairs is below 2^31, their sum
    is not.  The sharded join refuses it as the one-context join does, before any output exists,
    and the next join is right."""
    G = api.lib.adb_host_gpus()
    live0 = api.lib.adb_host_live_device_results()
    k, p = np.full(BOUND_ROWS, 7, np.int32), np.arange(BOUND_ROWS, dtype=np.int32)
    shares = np.bincount(home_of_rows(BOUND_ROWS, G)) * BOUND_ROWS
    assert shares.max() < 2**31 <= shares.sum() == BOUND_ROWS**2
    R = [C.pointer(api.host_result(x)) for x in (k, p, k, p)]
    with pytest.raises(RuntimeError, match="2147488281 pairs"):
        api.join("hash_join", *R)
    assert api.lib.adb_host_live_device_results() == live0
    sides = small_join(np.random.default_rng(G))
    api_join(api, sides, jr.hash_join(*sides), (G, "after the refused join"))
    assert api.lib.adb_host_live_device_results() == live0


# ---- the exchange when every stream shares one hardware work queue ---------------------------------
ONE_QUEUE_JOIN = """
import ctypes as C, sys
import numpy as np
import join_reference as jr
from query_api import Api
gpus = int(sys.argv[1])
a = Api()
assert a.lib.adb_host_init_multi(gpus) == 0, a.lib.adb_host_last_error()
rng = np.random.default_rng(gpus)
sides = [rng.integers(0, 20_000, n).astype(np.int32) for n in (70_000, 70_000, 50_000, 50_000)]
want = jr.hash_join(*sides)
for _ in range(2):
    o1, o2 = a.join("hash_join", *[C.pointer(a.host_result(x)) for x in sides])
    assert np.array_equal(a.tuples(o1), want[0]) and np.array_equal(a.tuples(o2), want[1])
    a.drop(o1), a.drop(o2)
a.lib.adb_host_shutdown()
"""


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", [2, 3])
def test_sharded_join_with_one_hardware_queue(gpus):
    """The pair exchange spin-waits on the device for every context's counts.  The contexts'
    streams may share a hardware work queue, and then nothing may wait in that queue behind a
    spinning kernel that the peers' arrival depends on.  CUDA_DEVICE_MAX_CONNECTIONS=1 puts every
    stream of a fresh process into one queue: the sharded join must still meet, the first time."""
    env = dict(os.environ, CUDA_DEVICE_MAX_CONNECTIONS="1")
    for var in SHIM_VARS + ("ADB_JOIN_PROBE", "ADB_TRACE"):
        env.pop(var, None)
    r = subprocess.run([sys.executable, "-c", ONE_QUEUE_JOIN, str(gpus)], cwd=os.path.dirname(os.path.abspath(__file__)),
                       env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=600)
    assert r.returncode == 0, r.stdout.decode()[-3000:]
