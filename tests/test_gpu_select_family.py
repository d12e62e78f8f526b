"""The select family's host protocol on one context: the kernels each entry point launches
(adb_launch_count), its answers against the oracle, and what a refused call does to the pending
select (adb_select_generation, and whether the pending count can still be emitted).  The launch
counts are those of the engine at the time this test was written; a change to the select
family's host code must leave every one of them as it is."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
I32MAX = 2**31 - 1
INVALID = -3
LO, HI = -1000, 5000

# kernels launched by one call, at n = 0 and n = 50 001 (h_count / h_agg passed unless "no_h")
LAUNCHES = {
    "select_scan": (1, 3),
    "select_count": (1, 3),
    "select_emit": (0, 1),
    "select_count_base": (1, 1),
    "select_count_base_no_h": (0, 1),
    "emit_fetch_agg_agg_only": (2, 1),
    "emit_fetch_agg": (2, 2),
    "chain_select_fetch_agg": (1, 2),
    "chain_select_agg": (2, 2),
    "emit_fetch_agg_exchange_agg_only": (3, 1),
    "emit_fetch_agg_exchange": (3, 2),
    "chain_select_fetch_agg_exchange": (2, 2),
}
SIZES = [0, 50_001]


@pytest.fixture(scope="module")
def eng():
    from analytical_database_b200 import Engine
    e = Engine(0)
    yield e
    e.close()


class Case:
    """One select column, one fetch column, the bounds, the device buffers and the expected answers."""

    def __init__(self, eng, port, rng, n):
        from analytical_database_b200.engine import _AggStruct
        self.eng, self.port, self.n, self.size_index = eng, port, n, SIZES.index(n)
        self.sel = rng.integers(-n // 2 - 1, n // 2 + 1, n).astype(np.int32)
        self.fet = rng.integers(I32MAX - 10000, I32MAX, n, dtype=np.int64).astype(np.int32)
        self.ds, self.df = eng.upload(self.sel), eng.upload(self.fet)
        self.pos, self.val = eng.alloc_i32(n), eng.alloc_i32(n)
        self.dcnt, self.dagg, self.dout = eng.alloc(8), eng.alloc(64), eng.alloc(64)
        self.blo, self.bhi = C.c_int32(LO), C.c_int32(HI)
        self.exp_pos = port.select_scan(self.sel, LO, HI)
        self.exp_val = port.fetch(self.fet, self.exp_pos)
        self.h, self.a = C.c_int64(-1), _AggStruct()

    @property
    def bounds(self):
        return C.byref(self.blo), C.byref(self.bhi)

    def launches(self, name, fn):
        before = self.eng.launch_count()
        status = fn()
        got = self.eng.launch_count() - before
        assert status == 0, (name, self.eng.lib.adb_last_error())
        assert got == LAUNCHES[name][self.size_index], (name, self.n, got)

    def count(self):
        return int(self.dcnt.to_host(1, np.int64)[0])

    def check_lists(self):
        k = self.exp_pos.size
        assert np.array_equal(self.pos.to_host(k), self.exp_pos)
        assert np.array_equal(self.val.to_host(k), self.exp_val)

    def check_agg(self, a):
        v = self.exp_val
        assert (a.sum, a.count) == (self.port.sum(v), v.size)
        if v.size:
            assert (a.min, a.max) == (self.port.min(v), self.port.max(v))
        else:
            assert (a.min, a.max) == (I32MAX, -I32MAX - 1)


@pytest.mark.parametrize("n", SIZES)
def test_launches_and_answers(eng, port, rng, n):
    c, lib = Case(eng, port, rng, n), eng.lib
    lo, hi = c.bounds
    k = c.exp_pos.size

    c.launches("select_scan", lambda: lib.adb_select_scan(c.ds.i32(), n, lo, hi, 0, c.pos.i32(), c.dcnt.i64(),
                                                          C.byref(c.h)))
    assert c.h.value == k and c.count() == k
    assert np.array_equal(c.pos.to_host(k), c.exp_pos)

    c.launches("select_count", lambda: lib.adb_select_count(c.ds.i32(), n, None, lo, hi, c.dcnt.i64(), C.byref(c.h)))
    assert c.h.value == k and c.count() == k
    c.launches("select_emit", lambda: lib.adb_select_emit(None, 7, c.pos.i32()))
    assert np.array_equal(c.pos.to_host(k), c.exp_pos + 7)

    c.launches("select_count_base_no_h", lambda: lib.adb_select_count_base(c.ds.i32(), n, lo, hi, 0, c.dcnt.i64(), None))
    assert c.count() == k
    c.launches("select_count_base", lambda: lib.adb_select_count_base(c.ds.i32(), n, lo, hi, 0, None, C.byref(c.h)))
    assert c.h.value == k
    c.launches("emit_fetch_agg_agg_only", lambda: lib.adb_select_emit_fetch_agg(
        c.df.i32(), None, None, eng.agg_ptr(c.dagg), C.byref(c.a)))
    c.check_agg(c.a)
    c.launches("emit_fetch_agg", lambda: lib.adb_select_emit_fetch_agg(
        c.df.i32(), c.pos.i32(), c.val.i32(), eng.agg_ptr(c.dagg), C.byref(c.a)))
    c.check_agg(c.a)
    c.check_lists()

    c.launches("chain_select_fetch_agg", lambda: lib.adb_chain_select_fetch_agg(
        c.ds.i32(), c.df.i32(), n, lo, hi, c.pos.i32(), c.val.i32(), c.dcnt.i64(), eng.agg_ptr(c.dagg)))
    assert c.count() == k
    c.check_agg(eng.read_agg(c.dagg))
    c.check_lists()

    c.launches("chain_select_agg", lambda: lib.adb_chain_select_agg(
        c.ds.i32(), c.df.i32(), n, lo, hi, c.dcnt.i64(), eng.agg_ptr(c.dagg), C.byref(c.a)))
    assert c.count() == k
    c.check_agg(c.a)
    assert (c.a.sum, k) == port.chain_select_fetch_sum(c.sel, c.fet, LO, HI)


@pytest.mark.parametrize("n", SIZES)
def test_exchange_launches_and_answers(eng, port, rng, n):
    """The fused exchange forms on a group of one context: the table-wide aggregate is this
    context's."""
    c, lib = Case(eng, port, rng, n), eng.lib
    lo, hi = c.bounds
    assert lib.adb_peer_connect_local(1) == 0, lib.adb_last_error()

    assert lib.adb_select_count_base(c.ds.i32(), n, lo, hi, 0, None, C.byref(c.h)) == 0
    c.launches("emit_fetch_agg_exchange_agg_only", lambda: lib.adb_select_emit_fetch_agg_exchange(
        c.df.i32(), None, None, eng.agg_ptr(c.dagg), eng.agg_ptr(c.dout), C.byref(c.a)))
    c.check_agg(c.a)
    c.launches("emit_fetch_agg_exchange", lambda: lib.adb_select_emit_fetch_agg_exchange(
        c.df.i32(), c.pos.i32(), c.val.i32(), eng.agg_ptr(c.dagg), eng.agg_ptr(c.dout), C.byref(c.a)))
    c.check_agg(c.a)
    c.check_agg(eng.read_agg(c.dout))
    c.check_lists()

    c.launches("chain_select_fetch_agg_exchange", lambda: lib.adb_chain_select_fetch_agg_exchange(
        c.ds.i32(), c.df.i32(), n, lo, hi, c.pos.i32(), c.val.i32(), c.dcnt.i64(), eng.agg_ptr(c.dagg), 1,
        eng.agg_ptr(c.dout)))
    assert c.count() == c.exp_pos.size
    c.check_agg(eng.read_agg(c.dagg))
    c.check_agg(eng.read_agg(c.dout))
    c.check_lists()


# refused call -> does it drop the pending count (bump the generation, refuse the next emit)?
REFUSALS = {
    "select_scan_null_d_count": False,
    "chain_select_agg_null_d_agg": False,
    "select_count_negative_n": True,
    "emit_fetch_agg_null_d_agg": False,
}


@pytest.mark.parametrize("refusal", sorted(REFUSALS))
def test_refusal_and_the_pending_select(eng, port, rng, refusal):
    n = SIZES[1]
    c, lib = Case(eng, port, rng, n), eng.lib
    lo, hi = c.bounds
    refuse = {
        "select_scan_null_d_count": lambda: lib.adb_select_scan(c.ds.i32(), n, lo, hi, 0, c.pos.i32(), None, None),
        "chain_select_agg_null_d_agg": lambda: lib.adb_chain_select_agg(c.ds.i32(), c.df.i32(), n, lo, hi,
                                                                        c.dcnt.i64(), None, None),
        "select_count_negative_n": lambda: lib.adb_select_count(c.ds.i32(), -1, None, lo, hi, None, None),
        "emit_fetch_agg_null_d_agg": lambda: lib.adb_select_emit_fetch_agg(c.df.i32(), c.pos.i32(), c.val.i32(),
                                                                           None, None),
    }[refusal]
    assert lib.adb_select_count_base(c.ds.i32(), n, lo, hi, 0, None, C.byref(c.h)) == 0
    gen = lib.adb_select_generation()
    assert refuse() == INVALID
    dropped = REFUSALS[refusal]
    assert lib.adb_select_generation() == gen + (1 if dropped else 0)
    status = lib.adb_select_emit(None, 0, c.pos.i32())
    if dropped:
        assert status == INVALID
    else:
        assert status == 0 and lib.adb_select_generation() == gen + 1
        assert np.array_equal(c.pos.to_host(c.h.value), c.exp_pos)
