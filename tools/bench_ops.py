#!/usr/bin/env python
"""Per-operator timings at the BASELINE.json config sizes (development tool; bench.py is
the contract).  python tools/bench_ops.py [shared|index|join|load|all] [--scale 1.0]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import analytical_database_b200 as adb  # noqa: E402


def timed(eng, fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    eng.sync()
    ms = []
    for _ in range(reps):
        eng.timer_start()
        fn()
        ms.append(eng.timer_stop())
    return float(np.median(ms)), float(min(ms))


def bench_shared(eng, scale):
    n, q = int(100_000_000 * scale), 100
    col = eng.synth_uniform(n, 42, 0, 0, n)
    rng = np.random.default_rng(42)
    lows = rng.integers(0, n - n // 1000, q).astype(np.int32)
    highs = (lows + n // 1000).astype(np.int32)
    out = {}

    def run():
        res = eng.shared_select(col, n, lows, highs)
        for b, _ in res:
            b.free()
        return res
    med, best = timed(eng, run)
    hits = sum(c for _, c in run())
    out = {"rows": n, "queries": q, "hits": hits, "ms": med, "best_ms": best,
           "rows_per_s": n / (med * 1e-3), "pred_evals_per_s": n * q / (med * 1e-3),
           "alg_gbs": (4 * n + 4 * hits) / (med * 1e-3) / 1e9}
    # the same batch into one slab (no per-result allocation): query i's list at slab + i * stride
    stride = 2 * (n // 1000) + 4096
    slab = eng.alloc_i32(q * stride)
    cnts = (C.c_int64 * q)()
    lo_p = lows.ctypes.data_as(C.POINTER(C.c_int32))
    hi_p = highs.ctypes.data_as(C.POINTER(C.c_int32))
    ptrs = (C.c_void_p * q)(*[slab.ptr + 4 * stride * i for i in range(q)])

    def run_slab():
        eng._ck(eng.lib.adb_shared_select_count(col.i32(), n, lo_p, hi_p, q, cnts))
        eng._ck(eng.lib.adb_shared_select_emit(ptrs, stride))
    med_s, best_s = timed(eng, run_slab)
    assert sum(cnts) == hits
    out["slab_ms"] = med_s
    out["slab_best_ms"] = best_s
    out["slab_rows_per_s"] = n / (med_s * 1e-3)
    slab.free()
    # unbatched: the same 100 selects one by one
    def run_seq():
        for i in range(q):
            p, c = eng.select_exact(col, n, int(lows[i]), int(highs[i]))
            p.free()
    med2, _ = timed(eng, run_seq, reps=3, warm=1)
    out["unbatched_ms"] = med2
    col.free()
    return out


def bench_index(eng, scale):
    n = int(500_000_000 * scale)
    key = eng.synth_uniform(n, 7, 0, 0, 1 << 31 - 1)
    pay = eng.synth_uniform(n, 8, 0, 0, 10000)
    t0 = time.perf_counter()
    vals, poss = eng.index_sort(key, n)
    eng.sync()
    build_s = time.perf_counter() - t0
    med_b, _ = timed(eng, lambda: [b.free() for b in eng.index_sort(key, n)], reps=2, warm=1)
    ix = eng.index_create(vals, poss, n, True)
    out = {"rows": n, "index_sort_ms": med_b, "first_build_s": build_s,
           "sort_mkeys_per_s": n / (med_b * 1e-3) / 1e6}
    for sel in (0.0002, 0.01, 0.1):
        lo = 1 << 20
        hi = lo + int((1 << 31) * sel)
        for tree in (False, True):
            def run():
                p, c = eng.select_index_exact(ix, lo, hi, use_btree=tree)
                f = eng.fetch(pay, p, c)
                p.free(); f.free()
                return c
            med, best = timed(eng, run)
            c = run()
            out[f"sel{sel}_{'btree' if tree else 'sorted'}"] = {
                "hits": c, "ms": med, "best_ms": best, "alg_gbs": 16.0 * c / (med * 1e-3) / 1e9}
        def run_scan():
            p, c = eng.select_exact(key, n, lo, hi)
            f = eng.fetch(pay, p, c)
            p.free(); f.free()
        med, _ = timed(eng, run_scan, reps=3, warm=1)
        out[f"sel{sel}_scan_ms"] = med
    eng.index_destroy(ix)
    for b in (key, pay, vals, poss):
        b.free()
    return out


def bench_sort_only(eng, scale):
    n = int(500_000_000 * scale)
    key = eng.synth_uniform(n, 7, 0, 0, 1 << 31 - 1)
    med, best = timed(eng, lambda: [b.free() for b in eng.index_sort(key, n)], reps=2, warm=1)
    key.free()
    return {"rows": n, "index_sort_ms": med, "sort_mkeys_per_s": n / (med * 1e-3) / 1e6}


def bench_join(eng, scale, cases=((0.8, 0.15), (0.15, 0.15), (1.0, 1.0))):
    n = int(100_000_000 * scale)
    out = {}
    k1 = eng.synth_uniform(n, 11, 0, 1, n)
    k2 = eng.synth_uniform(n, 12, 0, 1, n)
    f1 = eng.synth_uniform(n, 13, 0, 0, 1000)
    f2 = eng.synth_uniform(n, 14, 0, 0, 1000)
    for s1, s2 in cases:
        p1, c1 = eng.select_exact(f1, n, None, int(1000 * s1))
        p2, c2 = eng.select_exact(f2, n, None, int(1000 * s2))
        v1 = eng.fetch(k1, p1, c1)
        v2 = eng.fetch(k2, p2, c2)
        # parse.c:798-813: the larger side is column_one (build)
        if c2 > c1:
            (v1, p1, c1), (v2, p2, c2) = (v2, p2, c2), (v1, p1, c1)
        def run():
            o1, o2, m = eng.join(v1, p1, c1, v2, p2, c2)
            o1.free(); o2.free()
            return m
        med, best = timed(eng, run, reps=3, warm=1)
        m = run()
        out[f"prefilter_{s1}_{s2}"] = {
            "build": c1, "probe": c2, "matches": m, "ms": med, "best_ms": best,
            "tuples_per_s": (c1 + c2) / (med * 1e-3),
            "alg_gbs": (8.0 * (c1 + c2) + 8.0 * m) / (med * 1e-3) / 1e9}
        for b in (p1, p2, v1, v2):
            b.free()
    return out


def bench_load(eng, scale):
    """SURVEY.md 8f rank 1: CSV text -> columns.  The milestone-1 table shape (4 int columns,
    milestone1.py:115-119) at 4 M rows; host text -> HBM columns, staged upload included.
    CPU leg: the oracle's restatement of load_db's ingest loop on the same bytes."""
    import pandas as pd
    import time as _t
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle import oracle
    rows = int(4_000_000 * scale)
    rng = np.random.default_rng(42)
    df = pd.DataFrame({"a": rng.integers(-rows // 2, rows // 2, rows), "b": rng.integers(-rows // 2, rows // 2, rows),
                       "c": rng.integers(0, 100, rows), "d": rng.integers(2**31 - 10000, 2**31, rows)})
    text = ("db1.tbl2.col1,db1.tbl2.col2,db1.tbl2.col3,db1.tbl2.col4\n" +
            df.to_csv(index=False, header=False)).encode()
    a = np.frombuffer(text, dtype=np.uint8)

    def run():
        cols, r = eng.csv_load(a, 4)
        for c in cols:
            c.free()
        return r
    med, best = timed(eng, run, reps=3, warm=1)
    d_text = eng.upload(a)

    def run_dev():
        cols, r = eng.csv_load(a.size, 4, d_text=d_text)
        for c in cols:
            c.free()
    med_d, _ = timed(eng, run_dev, reps=5, warm=1)
    d_text.free()
    cols, r = eng.csv_load(a, 4)
    ok = all(np.array_equal(c.to_host(r), df[k].to_numpy().astype(np.int32)) for c, k in zip(cols, "abcd"))
    for c in cols:
        c.free()
    t0 = _t.perf_counter()
    ref = oracle.port().csv_parse(text, 4)
    cpu_s = _t.perf_counter() - t0
    ok = ok and all(np.array_equal(ref[i], df[k].to_numpy().astype(np.int32)) for i, k in enumerate("abcd"))
    return {"rows": rows, "text_bytes": len(text), "parity": bool(ok),
            "host_text_to_hbm_columns_ms": med, "best_ms": best, "text_gbs": len(text) / (med * 1e-3) / 1e9,
            "rows_per_s": rows / (med * 1e-3),
            "device_text_to_columns_ms": med_d, "device_text_gbs": len(text) / (med_d * 1e-3) / 1e9,
            "cpu_port_s": cpu_s, "cpu_port_text_gbs": len(text) / cpu_s / 1e9}


def bench_print(eng, scale):
    """SURVEY.md 8f rank 2: print of a long INT result.  Device formatting + text download
    against download + the reference's sprintf loop (the oracle's restatement of
    query.c:262-269; the reference itself corrupts its heap on wide values, A8)."""
    import time as _t
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle import oracle
    n = int(50_000_000 * scale)
    d = eng.synth_uniform(n, 5, 0, -500_000, 1_000_000)
    nb = C.c_int64(0)

    def kernels():
        eng._ck(eng.lib.adb_format_i32_count(d.i32(), n, C.byref(nb)))
        t = eng.alloc(nb.value)
        eng._ck(eng.lib.adb_format_i32_emit(t.void()))
        t.free()
    med_k, _ = timed(eng, kernels, reps=5, warm=2)
    # the call print makes: count, emit, download the text into a host buffer (already touched:
    # a server reuses its reply buffer; a fresh one costs a page fault per 4 KB on any path)
    host_text = np.zeros(nb.value, dtype=np.uint8)
    e2e = []
    for _ in range(3):
        t0 = _t.perf_counter()
        eng._ck(eng.lib.adb_format_i32_count(d.i32(), n, C.byref(nb)))
        t = eng.alloc(nb.value)
        eng._ck(eng.lib.adb_format_i32_emit(t.void()))
        eng._ck(eng.lib.adb_download(host_text.ctypes.data_as(C.c_void_p), t.void(), nb.value))
        t.free()
        e2e.append(_t.perf_counter() - t0)
    e2e_s = min(e2e)
    text = host_text.tobytes()
    m = min(n, 5_000_000)
    host = d.to_host(m)
    t0 = _t.perf_counter()
    ref = oracle.port().print_i32(host)
    cpu_s = (_t.perf_counter() - t0) * n / m
    ok = text[:len(ref)] == ref if m < n else text == ref
    d.free()
    return {"values": n, "text_bytes": len(text), "parity_prefix": bool(ok), "device_format_ms": med_k,
            "device_format_gvalues_per_s": n / (med_k * 1e-3) / 1e9,
            "print_to_host_text_ms": e2e_s * 1e3, "cpu_port_ms_extrapolated": cpu_s * 1e3,
            "cpu_sample_values": m}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("what", nargs="?", default="all")
    ap.add_argument("--scale", type=float, default=1.0)
    a = ap.parse_args()
    eng = adb.Engine(0)
    res = {}
    if a.what in ("shared", "all"):
        res["shared_scan"] = bench_shared(eng, a.scale)
    if a.what in ("index", "all"):
        res["index"] = bench_index(eng, a.scale)
    if a.what == "sort":
        res["sort"] = bench_sort_only(eng, a.scale)
    if a.what == "join11":
        res["join"] = bench_join(eng, a.scale, ((1.0, 1.0),))
    if a.what in ("join", "all"):
        res["join"] = bench_join(eng, a.scale)
    if a.what in ("print", "all"):
        res["print"] = bench_print(eng, a.scale)
    if a.what in ("load", "all"):
        res["load"] = bench_load(eng, a.scale)
    print(json.dumps(res, indent=1))
    eng.close()


if __name__ == "__main__":
    main()
