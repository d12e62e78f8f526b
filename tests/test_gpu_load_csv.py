"""Bulk load through the operator-API host: adb_host_load_csv_count / adb_host_load_csv_emit.

The text is cut into one piece per engine context at line boundaries; every context parses its
piece, the host carries the last values of every column from piece to piece, and the rows land in
the shim's row-range shards.  Run with 1-4 contexts (more contexts than devices share a device).
The oracle is port.csv_parse, the C restatement of load_db's ingest loop
(src/db_manager.c:304-318) that tests/test_csv_load.py pins against the reference server."""
import ctypes as C
import glob
import json
import os

import numpy as np
import pytest

from query_api import Api, Column

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
LOAD = os.path.join(HERE, "golden", "load")
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(LOAD, "*.csv")))
TOKENS = ["0", "7", "-7", "+7", " 42", "\t-3", "12abc", "abc", "", "--5", "- 5", "007", "4 ", "2147483647",
          "2147483648", "-2147483648", "-2147483649", "99999999999", "9223372036854775807",
          "9223372036854775808", "-9223372036854775809", "18446744073709551616", "1.5", "2e3", "0x10",
          "\v4", "\f5", "\r6", "5\r"]


# include/adb_load_api.h
LOAD_HOOKS = {
    "adb_host_load_csv_count": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_size_t)]),
    "adb_host_load_csv_emit": (C.c_int, [C.POINTER(C.POINTER(Column)), C.c_int]),
}


def bind_load_hooks(lib):
    for name, (res, args) in LOAD_HOOKS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


@pytest.fixture(scope="module", params=[1, 2, 3, 4], ids=["1ctx", "2ctx", "3ctx", "4ctx"])
def api(request):
    a = Api()
    bind_load_hooks(a.lib)
    assert a.lib.adb_host_init_multi(request.param) == 0, a.lib.adb_host_last_error()
    a.G = request.param
    yield a
    a.lib.adb_host_shutdown()


class LoadError(RuntimeError):
    pass


class Table:
    """A table's columns as the catalog holds them: numpy arrays behind query_api.Column."""

    def __init__(self, n_cols, old=None, minmax=(0, 0)):
        self.arrays = [np.array(o, dtype=np.int32) for o in old] if old else [np.zeros(0, np.int32)] * n_cols
        self.cols = []
        for j, a in enumerate(self.arrays):
            c = Column()
            c.name = b"col%d" % (j + 1)
            c.data = a.ctypes.data_as(C.POINTER(C.c_int))
            c.row_count = a.size
            c.min, c.max = minmax if not a.size else (int(a.min()), int(a.max()))
            self.cols.append(c)

    def ptrs(self):
        return (C.POINTER(Column) * len(self.cols))(*[C.pointer(c) for c in self.cols])

    def grow(self, extra):
        """What load_db does before the emit: room for row_count + extra rows."""
        for j, c in enumerate(self.cols):
            a = np.zeros(c.row_count + extra, dtype=np.int32)
            a[:c.row_count] = self.arrays[j][:c.row_count]
            self.arrays[j] = a
            c.data = a.ctypes.data_as(C.POINTER(C.c_int))

    def data(self):
        n = self.cols[0].row_count
        return np.stack([a[:n] for a in self.arrays])


def count(api, text, n_cols, skip=1):
    rows = C.c_size_t(0)
    if api.lib.adb_host_load_csv_count(text, len(text), skip, n_cols, C.byref(rows)) != 0:
        raise LoadError(api.lib.adb_host_last_error().decode())
    return rows.value


def emit(api, table, n_cols=None):
    if api.lib.adb_host_load_csv_emit(table.ptrs(), len(table.cols) if n_cols is None else n_cols) != 0:
        raise LoadError(api.lib.adb_host_last_error().decode())


def load(api, table, text, skip=1):
    rows = count(api, text, len(table.cols), skip)
    table.grow(rows)
    emit(api, table)
    return rows


def cut_points(text, G, skip=1):
    """The documented cut rule: piece g > 0 starts right after the first '\\n' at or after byte
    g*len/G of the text after the skipped lines."""
    off = 0
    for _ in range(skip):
        k = text.find(b"\n", off)
        off = len(text) if k < 0 else k + 1
    n = len(text) - off
    out = []
    for g in range(1, G):
        k = text.find(b"\n", off + g * n // G)
        out.append(len(text) if k < 0 else k + 1)
    return out


def folded(exp, minmax):
    """insert_row's fold of the new rows into the column's min / max."""
    if exp.shape[1] == 0:
        return [minmax] * exp.shape[0]
    return [(min(minmax[0], int(r.min())), max(minmax[1], int(r.max()))) for r in exp]


def check_load(api, port, text, n_cols, skip=1, minmax=(0, 0)):
    exp = port.csv_parse(text, n_cols, skip)
    t = Table(n_cols, minmax=minmax)
    rows = load(api, t, text, skip)
    assert rows == exp.shape[1]
    got = t.data()
    assert got.shape == exp.shape and np.array_equal(got, exp)
    for c, (mn, mx) in zip(t.cols, folded(exp, minmax)):
        assert c.row_count == rows and (c.min, c.max) == (mn, mx)
    return t, exp


def random_text(rng, rows, n_cols, tidy, final_newline=None):
    lines = ["db1.t." + ",db1.t.".join(f"c{i}" for i in range(n_cols))]
    for r in range(rows):
        if tidy:
            toks = [str(int(x)) for x in rng.integers(-2**31, 2**31 - 1, n_cols)]
        else:
            k = n_cols if r == 0 else int(rng.integers(0, n_cols + 3))     # short / long rows after the first
            toks = [TOKENS[int(i)] for i in rng.integers(0, len(TOKENS), k)]
        lines.append(",".join(toks))
    nl = bool(rng.integers(0, 2)) if final_newline is None else final_newline
    return ("\n".join(lines) + ("\n" if nl else "")).encode()


@pytest.mark.parametrize("name", CASES)
def test_golden_files(api, port, name):
    with open(os.path.join(LOAD, name + ".csv"), "rb") as f:
        text = f.read()
    with open(os.path.join(LOAD, name + ".cols.json")) as f:
        exp = json.load(f)
    t, got = check_load(api, port, text, exp["n_cols"], minmax=(2**31 - 1, -2**31))
    ref = np.array(exp["columns"], dtype=np.int64).astype(np.int32).reshape(exp["n_cols"], -1)
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("tidy", [True, False])
@pytest.mark.parametrize("rows,n_cols", [(0, 1), (1, 1), (2, 3), (3, 4), (255, 2), (257, 7), (5000, 4), (70001, 5)])
def test_random_text(api, port, rng, rows, n_cols, tidy):
    for final_newline in (True, False):
        check_load(api, port, random_text(rng, rows, n_cols, tidy, final_newline), n_cols)


def test_carry_chains_through_every_piece(api, port, rng):
    """Every row after the first is short: the first row's values reach every piece."""
    n = 4000
    lines = [b"h", b"11,-22,33,44"] + [b"%d" % v for v in rng.integers(-50, 50, n)]
    text = b"\n".join(lines) + b"\n"
    t, exp = check_load(api, port, text, 4)
    assert np.all(exp[1] == -22) and np.all(exp[3] == 44)
    for at in cut_points(text, api.G):                  # every cut falls before a short row
        assert text[at:text.find(b"\n", at)].count(b",") == 0 and at < len(text)


def test_carry_from_an_earlier_piece_and_a_column_no_row_has(api, port, rng):
    """Column 3 of a 4-column table: no row has it (0 everywhere).  Column 2: only rows in the
    first piece have it, so later pieces start with short rows that inherit across the cut."""
    n = 6000
    full = [b"%d,%d,%d" % tuple(rng.integers(-9, 9, 3)) for _ in range(n // 8)]
    short = [b"%d,%d" % tuple(rng.integers(-9, 9, 2)) for _ in range(n - n // 8)]
    text = b"\n".join([b"h"] + full + short) + b"\n"
    t, exp = check_load(api, port, text, 4)
    assert np.all(exp[3] == 0) and np.all(exp[2][n // 8:] == exp[2][n // 8 - 1])
    for at in cut_points(text, api.G):
        assert text[at:text.find(b"\n", at)].count(b",") == 1     # the piece starts with a short row


def test_linear_fill_of_20m_short_rows(api, port, rng):
    """20 M lines of two fields into three columns: every row is short.  The backward walk the
    fill replaced took time quadratic in the rows here."""
    block = rng.integers(-10**6, 10**6, (4096, 2))
    lines = b"".join(b"%d,%d\n" % (a, b) for a, b in block)
    text = b"h\n" + lines * (20_000_000 // 4096) + lines[:lines.index(b"\n") + 1] * (20_000_000 % 4096)
    check_load(api, port, text, 3)


def test_the_device_copy_is_the_loaded_one(api, port, rng):
    n = 300_017
    cols = [rng.integers(-1000, 1000, n), rng.integers(0, 50_000, n), rng.permutation(n)]
    text = ("h\n" + "\n".join("%d,%d,%d" % r for r in zip(*cols)) + "\n").encode()
    t, exp = check_load(api, port, text, 3)
    for a in t.arrays:                                  # the host copy is no longer what the shards hold
        a[:] = -7
    from oracle import oracle
    cpu = oracle.port()
    s = api.select_column(t.cols[0], -100, 250)
    f = api.fetch_column(t.cols[1], s)
    epos = cpu.select_scan(exp[0], -100, 250)
    assert np.array_equal(api.tuples(s), epos)
    a = api.sum_result(f)
    assert int(api.tuples(a)[0]) == cpu.sum(cpu.fetch(exp[1], epos))
    for r in (s, f, a):
        api.drop(r)
    lows, highs = [-500, 0, 990], [-400, 300, 1000]
    res = api.shared_select(t.cols[0], lows, highs)
    for r, e in zip(res, cpu.shared_select(exp[0], lows, highs)):
        assert np.array_equal(api.tuples(r), e)
        api.drop(r)
    # an unclustered index built from the installed shards
    t.cols[2].has_index = True
    ptrs = t.ptrs()
    assert api.lib.adb_host_index_build(ptrs, 3, 2) == 0, api.lib.adb_host_last_error()
    ev, ep = cpu.index_sort(exp[2])
    ix = t.cols[2].index.contents
    assert np.array_equal(np.ctypeslib.as_array(ix.values, shape=(n,)), ev)
    s = api.select_column(t.cols[2], 1000, 5000)
    e, undefined = cpu.select_sorted_index(ev, ep, 1000, 5000)
    assert not undefined and np.array_equal(api.tuples(s), e)
    api.drop(s)


def test_append_to_a_table_that_holds_rows(api, port, rng):
    old = [rng.integers(-10, 10, 1234).astype(np.int32) for _ in range(3)]
    t = Table(3, old)
    text = random_text(rng, 5000, 3, tidy=False)
    exp = port.csv_parse(text, 3)
    before = [(c.min, c.max) for c in t.cols]
    rows = load(api, t, text)
    assert rows == exp.shape[1]
    want = np.concatenate([np.stack(old), exp], axis=1)
    assert np.array_equal(t.data(), want)
    for c, (mn, mx), e in zip(t.cols, before, exp):
        assert (c.min, c.max) == (min(mn, int(e.min())), max(mx, int(e.max())))
        assert c.row_count == 1234 + rows
    from oracle import oracle
    cpu = oracle.port()
    s = api.select_column(t.cols[0], -5, 5)
    f = api.fetch_column(t.cols[2], s)
    epos = cpu.select_scan(want[0], -5, 5)
    assert np.array_equal(api.tuples(s), epos) and np.array_equal(api.tuples(f), want[2][epos])
    api.drop(s), api.drop(f)


def test_errors_leave_the_columns_untouched(api, port, rng):
    lines = [b"%d,%d" % tuple(rng.integers(0, 99, 2)) for _ in range(4000)]
    mid = len(lines) * (api.G // 2 * 2 + 1) // (2 * api.G)        # inside the middle piece
    bad = b"\n".join([b"h"] + lines[:mid] + [b"1," * 600] + lines[mid:]) + b"\n"
    old = [np.arange(10, dtype=np.int32), np.arange(10, 20, dtype=np.int32)]
    t = Table(2, old)
    with pytest.raises(LoadError, match="1023"):
        count(api, bad, 2)
    with pytest.raises(LoadError, match="no pending"):
        emit(api, t)
    assert np.array_equal(t.data(), np.stack(old)) and t.cols[0].row_count == 10
    good = b"\n".join([b"h"] + lines) + b"\n"
    rows = count(api, good, 2)
    t.grow(rows)
    with pytest.raises(LoadError, match="columns"):
        emit(api, t, n_cols=1)                          # n_cols differs from the count's
    rows = count(api, good, 2)
    t.cols[1].row_count = 9                             # columns of unequal length
    with pytest.raises(LoadError, match="equally long"):
        emit(api, t)
    t.cols[1].row_count = 10
    assert np.array_equal(t.data(), np.stack(old)) and (t.cols[0].min, t.cols[0].max) == (0, 9)
    with pytest.raises(LoadError):
        count(api, good, 255)
    # a second count replaces the first: the emit writes the second text
    other = b"h\n5,6\n7\n"
    count(api, good, 2)
    rows = count(api, other, 2)
    assert rows == 2
    t.grow(rows)
    emit(api, t)
    assert np.array_equal(t.data(), np.concatenate([np.stack(old), port.csv_parse(other, 2)], axis=1))
    # and a good load after all of it
    check_load(api, port, good, 2)


def test_large_text_through_the_staged_upload(api, port):
    """About 280 MB of text, 4 columns, over 4 contexts: every piece is at least 64 MB, so each
    goes through the staged (pinned, multi-lane) upload."""
    if api.G != 4:
        pytest.skip("run once, at 4 contexts")
    rng = np.random.default_rng(11)
    rows = 8_500_000
    cols = [rng.integers(-2**31, 2**31 - 1, rows).astype(np.int32) for _ in range(2)]
    cols += [rng.integers(0, 100, rows).astype(np.int32), np.arange(rows, dtype=np.int32)]
    import pandas as pd
    text = ("a,b,c,d\n" + pd.DataFrame(dict(zip("abcd", cols))).to_csv(index=False, header=False)).encode()
    starts = [text.index(b"\n") + 1] + cut_points(text, 4) + [len(text)]
    assert min(e - b for b, e in zip(starts, starts[1:])) >= 64 << 20
    t = Table(4, minmax=(2**31 - 1, -2**31))
    assert load(api, t, text) == rows
    for got, c in zip(t.data(), cols):
        assert np.array_equal(got, c)
    assert [(c.min, c.max) for c in t.cols] == [(int(c.min()), int(c.max())) for c in cols]


@pytest.mark.parametrize("pieces", [1, 2, 5, 13])
def test_engine_piece_parse_carry_and_fill(api, port, rng, pieces):
    """At the C-ABI on one context: the text split at line boundaries, each piece parsed with
    adb_csv_parse_piece, the carry resolved on the host, adb_csv_fill; the concatenation equals
    adb_csv_parse of the whole text and the oracle."""
    from analytical_database_b200 import Engine
    eng = Engine(0)                                     # the shim's context 0 (adb_init is idempotent)
    n_cols = 5
    text = random_text(rng, 20_000, n_cols, tidy=False)
    body = text[text.index(b"\n") + 1:]
    exp = port.csv_parse(text, n_cols)
    whole = eng.csv_load(body, n_cols, 0)
    got_whole = np.stack([c.to_host(whole[1]) for c in whole[0]])
    for c in whole[0]:
        c.free()
    assert np.array_equal(got_whole, exp)
    cuts = sorted(set(int(x) for x in rng.integers(0, len(body), pieces - 1)))
    starts = [0] + [body.find(b"\n", c) + 1 if body.find(b"\n", c) >= 0 else len(body) for c in cuts] + [len(body)]
    carry = np.zeros(n_cols, np.int32)
    out = []
    I32 = C.POINTER(C.c_int32)
    for b, e in zip(starts[:-1], starts[1:]):
        piece = body[b:e]
        d_text = eng.upload(np.frombuffer(piece, np.uint8)) if piece else eng.alloc(16)
        rows = C.c_int64(0)
        eng._ck(eng.lib.adb_csv_index(d_text.void(), len(piece), 0, C.byref(rows)))
        cols = [eng.alloc_i32(rows.value) for _ in range(n_cols)]
        ptrs = (C.c_void_p * n_cols)(*[c.ptr for c in cols])
        last, has, short = np.zeros(n_cols, np.int32), np.zeros(n_cols, np.int32), C.c_int32(0)
        eng._ck(eng.lib.adb_csv_parse_piece(n_cols, ptrs, last.ctypes.data_as(I32), has.ctypes.data_as(I32),
                                            C.byref(short)))
        eng._ck(eng.lib.adb_csv_fill(carry.ctypes.data_as(I32)))
        if rows.value:
            out.append(np.stack([c.to_host(rows.value) for c in cols]))
        carry = np.where(has != 0, last, carry).astype(np.int32)
        eng.sync()
        for c in cols + [d_text]:
            c.free()
    got = np.concatenate(out, axis=1) if out else np.zeros((n_cols, 0), np.int32)
    assert np.array_equal(got, exp)
