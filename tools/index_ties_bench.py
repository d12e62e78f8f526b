"""adb_index_sort (stable radix sort) against adb_index_sort_ref_ties (the reference quicksort's
tie order) on one GPU, CUDA events around each call, and the reference's own CPU sort where it
finishes.  Writes profiles/r03_index_ties.json (or --out).

Columns: 500 M unique keys (config 3's indexed column, a permutation of 0..n-1), and 100 M keys
uniform over [0, 2^20), uniform over [0, 1000) and zipf(1.3).  Per column: the median of
--reps timed calls of each sort after one warm-up call, the ref-ties sort's levels (ADB_TRACE)
and kernel launches, and -- on the first 10 M rows, when the quicksort's cost (quadratic in the
length of a run of equal keys) allows -- the oracle's CPU time and a bit-exact check against it.

    python tools/index_ties_bench.py [--reps 5] [--scale 1.0] [--out profiles/r03_index_ties.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import analytical_database_b200 as adb  # noqa: E402
from oracle import oracle  # noqa: E402

ORACLE_ROWS = 10_000_000
ORACLE_MAX_COST = 2e10            # sum over runs of equal keys of len^2 / 2: the quicksort's swaps


def timed(eng, fn, reps):
    fn()
    eng.sync()
    out = []
    for _ in range(reps):
        eng.timer_start()
        fn()
        out.append(eng.timer_stop())
    return float(np.median(out)), out


def traced_levels(eng, fn):
    """Run fn with ADB_TRACE set and return the level count the engine prints to stderr."""
    os.environ["ADB_TRACE"] = "1"
    with tempfile.TemporaryFile() as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
            eng.sync()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["ADB_TRACE"]
        f.seek(0)
        text = f.read().decode(errors="replace")
    for line in text.splitlines():
        if line.startswith("index_sort_ref_ties:"):
            return int(line.split()[1])
    return 0                                              # no key repeats: no level ran


def column(eng, kind, n):
    if kind == "unique":
        mul, add = 387_420_489, 123_456_789
        d = eng.alloc_i32(n)
        eng._ck(eng.lib.adb_synth_affine(d.i32(), n, 0, mul, add, n))
        return d
    if kind == "uniform_2^20":
        return eng.synth_uniform(n, 11, 0, 0, 1 << 20)
    if kind == "uniform_1000":
        return eng.synth_uniform(n, 12, 0, 0, 1000)
    if kind == "zipf":
        rng = np.random.default_rng(13)
        return eng.upload(np.minimum(rng.zipf(1.3, n), 1 << 30).astype(np.int32))
    raise AssertionError(kind)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0, help="multiply every column's length")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_index_ties.json"))
    args = ap.parse_args()
    eng = adb.Engine(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    port = oracle.reference("O2") or oracle.port()
    rows = []
    for kind, n in (("unique", 500_000_000), ("uniform_2^20", 100_000_000), ("uniform_1000", 100_000_000),
                    ("zipf", 100_000_000)):
        n = max(1, int(n * args.scale))
        d = column(eng, kind, n)
        va, pa, vb, pb = (eng.alloc_i32(n) for _ in range(4))
        stable = lambda: eng._ck(eng.lib.adb_index_sort(d.i32(), n, va.i32(), pa.i32()))      # noqa: E731
        ties = lambda: eng._ck(eng.lib.adb_index_sort_ref_ties(d.i32(), n, vb.i32(), pb.i32()))  # noqa: E731
        t_stable, all_stable = timed(eng, stable, args.reps)
        t_ties, all_ties = timed(eng, ties, args.reps)
        l0 = eng.launch_count()
        levels = traced_levels(eng, ties)
        launches = eng.launch_count() - l0
        assert np.array_equal(va.to_host(n), vb.to_host(n)), "values differ from adb_index_sort's"
        row = {"column": kind, "rows": n, "index_sort_ms": t_stable, "index_sort_ref_ties_ms": t_ties,
               "ratio": t_ties / t_stable, "index_sort_ms_all": all_stable, "index_sort_ref_ties_ms_all": all_ties,
               "levels": levels, "launches": launches}
        # the reference's own sort on a prefix, where it finishes
        m = min(n, ORACLE_ROWS)
        host = d.to_host(m)
        _, counts = np.unique(host, return_counts=True)
        cost = float((counts.astype(np.float64) ** 2).sum() / 2)
        if cost <= ORACLE_MAX_COST:
            dp = eng.upload(host)
            vp, pp = eng.alloc_i32(m), eng.alloc_i32(m)
            eng._ck(eng.lib.adb_index_sort_ref_ties(dp.i32(), m, vp.i32(), pp.i32()))
            t0 = time.perf_counter()
            ev, ep = port.index_sort(host)
            row["oracle_rows"], row["oracle_cpu_s"] = m, time.perf_counter() - t0
            row["oracle_equal"] = bool(np.array_equal(vp.to_host(m), ev) and
                                       np.array_equal(pp.to_host(m), ep.astype(np.int32)))
            for b in (dp, vp, pp):
                b.free()
        else:
            row["oracle_rows"], row["oracle_cpu_s"] = m, None
            row["oracle_skipped"] = f"quadratic: ~{cost:.2g} swaps on the first {m} rows"
        print(json.dumps(row), flush=True)
        rows.append(row)
        for b in (d, va, pa, vb, pb):
            b.free()
    out = {"gpu": gpu, "oracle": "reference" if oracle.reference("O2") else "port", "reps": args.reps,
           "timing": "CUDA events around one call, median; inputs >= 400 MB (beyond L2)", "results": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
