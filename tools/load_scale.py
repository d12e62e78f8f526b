"""Bulk load at G = 1, 2, 4, 8 engine contexts through the operator-API host's load hooks
(adb_host_load_csv_count + adb_host_load_csv_emit), against the single-context path the hooks
replace (adb_upload + adb_csv_index + adb_csv_parse + adb_download per column) and the oracle's
CPU ingest loop (load_db, src/db_manager.c:304-318) on a slice of the same text.

Input: a seeded 4-column CSV of about 1 GB, generated in memory (a block of 1 M random rows,
repeated; far above L2 and the 64 MB staging threshold).  Every run's columns are compared with
the generated values.  Writes profiles/r03_load_scale.json (or --out) with the device name, the
power limit and the device count read in the same process; with fewer devices than contexts the
contexts share devices (and their host links).

    python tools/load_scale.py [--gb 1.0] [--reps 3] [--out profiles/r03_load_scale.json]
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ["ADB_SHIM_PROFILE"] = "1"          # per-phase wall time, read back from adb_host_profile_dump

import analytical_database_b200 as adb  # noqa: E402
import query_api as q  # noqa: E402
from test_gpu_load_csv import bind_load_hooks  # noqa: E402

PHASES = {"load: upload": "upload", "load: index+parse": "index_parse", "load: fill": "fill",
          "load: re-cut": "recut", "load: aggregate": "aggregate", "load: download": "download"}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    name, power = out[0].split(", ")
    return {"device": name, "power_limit": power, "device_count": len(out)}


def make_text(gb, seed=2026):
    import pandas as pd
    rng = np.random.default_rng(seed)
    n = 1_000_000
    block = [rng.integers(-2**31, 2**31 - 1, n), rng.integers(-2**31, 2**31 - 1, n),
             rng.integers(0, 100, n), rng.integers(0, 1_000_000, n)]
    body = pd.DataFrame(dict(zip("abcd", block))).to_csv(index=False, header=False).encode()
    reps = max(1, int(np.ceil(gb * 1e9 / len(body))))
    text = b"db1.tbl.a,db1.tbl.b,db1.tbl.c,db1.tbl.d\n" + body * reps
    return text, [np.tile(np.asarray(b, dtype=np.int32), reps) for b in block]


def profile_phases(lib):
    """adb_host_profile_dump prints to stderr: catch it in a file."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            lib.adb_host_profile_dump()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read()
    out = {}
    for line in text.splitlines():
        for label, key in PHASES.items():
            m = re.match(r"\[adb shim profile\] " + re.escape(label) + r"\s+(\d+)\s+([\d.]+)", line)
            if m:
                out[key] = float(m.group(2)) / int(m.group(1)) / 1e3       # ms per call
    return out


def run_hooks(G, text, truth, reps):
    lib = bind_load_hooks(q.load())
    assert lib.adb_host_init_multi(G) == 0, lib.adb_host_last_error()
    n_cols = len(truth)
    times, parity = [], True
    for it in range(reps + 1):                                      # one warm-up
        arrays = [np.zeros(0, np.int32)] * n_cols
        cols = (q.Column * n_cols)()
        ptrs = (C.POINTER(q.Column) * n_cols)(*[C.pointer(cols[j]) for j in range(n_cols)])
        rows = C.c_size_t(0)
        t0 = time.perf_counter()
        assert lib.adb_host_load_csv_count(text, len(text), 1, n_cols, C.byref(rows)) == 0, lib.adb_host_last_error()
        t1 = time.perf_counter()
        arrays = [np.empty(rows.value, np.int32) for _ in range(n_cols)]   # the catalog grows its columns
        for j in range(n_cols):
            cols[j].data = arrays[j].ctypes.data_as(C.POINTER(C.c_int))
        t2 = time.perf_counter()
        assert lib.adb_host_load_csv_emit(ptrs, n_cols) == 0, lib.adb_host_last_error()
        t3 = time.perf_counter()
        if it == 0:
            profile_phases(lib)                                     # drop the warm-up's phases
        else:
            times.append((t1 - t0) + (t3 - t2))
        parity &= all(np.array_equal(a, t) for a, t in zip(arrays, truth))
        for j in range(n_cols):
            lib.adb_host_column_invalidate(C.pointer(cols[j]))      # free the installed shards
    phases = profile_phases(lib)
    lib.adb_host_shutdown()
    return times, phases, parity


def run_single_context(text, truth, reps):
    """The path INTEGRATION.md documented before the hooks: one context, whole file."""
    eng = adb.Engine(0)
    a = np.frombuffer(text, dtype=np.uint8)
    n_cols = len(truth)
    times, parity = [], True
    for it in range(reps + 1):
        t0 = time.perf_counter()
        cols, rows = eng.csv_load(a, n_cols, 1)                     # adb_upload + adb_csv_index + adb_csv_parse
        host = [c.to_host(rows) for c in cols]                      # adb_download per column
        t1 = time.perf_counter()
        for c in cols:
            c.free()
        if it:
            times.append(t1 - t0)
        parity &= all(np.array_equal(h, t) for h, t in zip(host, truth))
    eng.close()
    return times, parity


def run_cpu_oracle(text, slice_bytes=64 << 20):
    from oracle import oracle
    port = oracle.port()
    cut = text.index(b"\n", slice_bytes) + 1
    piece = text[:cut]
    t0 = time.perf_counter()
    rows = port.csv_parse(piece, 4).shape[1]
    dt = time.perf_counter() - t0
    return {"slice_bytes": len(piece), "slice_rows": rows, "slice_s": dt,
            "gbps": len(piece) / dt / 1e9, "scaled_s": dt * len(text) / len(piece)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_load_scale.json"))
    args = ap.parse_args()
    info = gpu_info()
    text, truth = make_text(args.gb)
    rows = int(truth[0].size)
    res = {**info, "text_bytes": len(text), "rows": rows, "columns": len(truth), "reps": args.reps,
           "timing": "host wall clock of count + emit (each ends synchronised), median of reps after one warm-up; "
                     "phases: mean wall time per call from the shim's ADB_SHIM_PROFILE counters"}
    times, parity = run_single_context(text, truth, args.reps)
    med = float(np.median(times))
    res["single_context"] = {"wall_s": med, "gbps": len(text) / med / 1e9, "rows_per_s": rows / med, "parity": parity}
    print("single context", res["single_context"], flush=True)
    res["cpu_oracle"] = run_cpu_oracle(text)
    print("cpu oracle", res["cpu_oracle"], flush=True)
    res["runs"] = []
    for G in [int(x) for x in args.gpus.split(",")]:
        times, phases, parity = run_hooks(G, text, truth, args.reps)
        med = float(np.median(times))
        r = {"G": G, "wall_s": med, "wall_all_s": times, "gbps": len(text) / med / 1e9, "rows_per_s": rows / med,
             "phases_ms": phases, "speedup_vs_single_context": res["single_context"]["wall_s"] / med, "parity": parity}
        res["runs"].append(r)
        print(json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    ok = res["single_context"]["parity"] and all(r["parity"] for r in res["runs"])
    print("parity", "ok" if ok else "FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
