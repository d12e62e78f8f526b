"""adb_host_index_build of BASELINE config 3's indexed column (500 M unique keys, a permutation of
0..n-1 held in row-sharded device buffers) at G = 1, 2, 4 and 8 contexts, unclustered and
clustered (one host-resident sibling column permuted into index order), with the shim's
per-phase wall times (ADB_SHIM_PROFILE=1).  Contexts beyond the device count share devices, so on
a one-GPU box the record shows correctness and the phase split, not multi-GPU speed.

Every (tree, G, kind) runs in a subprocess of its own against the libraries of --tree (default:
this checkout), so two checkouts -- a parent commit and a branch -- can be compared in one run:

    python tools/index_build_scale.py --tree /path/parent --label parent --tree . --label branch \\
        --out profiles/r03_index_build_scale.json

Per run: the median of --reps timed builds after one warm-up build, every build checked against
the closed form of the permutation on three windows of the catalog arrays.
"""
import argparse
import ctypes as C
import json
import os
import re
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, MUL, ADD = 500_000_000, 387_420_489, 123_456_789


def worker(tree, G, kind, n, reps):
    sys.path[:0] = [tree, os.path.join(tree, "tests")]
    import analytical_database_b200 as adb
    import query_api as q
    api = q.Api()
    assert api.lib.adb_host_init_multi(G) == 0, api.lib.adb_host_last_error()
    eng = adb.Engine(0)
    S = ((n + G - 1) // G + 31) // 32 * 32
    mul, add = (MUL, ADD) if n == N else (7, 3)         # --rows other than config 3's: n must not divide by 7
    ptrs, bufs = (C.c_void_p * G)(), []
    for g in range(G):
        eng._ck(eng.lib.adb_ctx_select(g))
        cnt = max(1, min(S, n - g * S))
        b = eng.alloc_i32(cnt)
        eng._ck(eng.lib.adb_synth_affine(b.i32(), cnt, g * S, mul, add, n))
        eng.sync()
        bufs.append(b)
        ptrs[g] = b.ptr
    eng._ck(eng.lib.adb_ctx_select(0))
    inv = pow(mul, -1, n)
    key = q.Column()
    key.name, key.row_count, key.has_index = b"key", n, True
    key.clustered = kind == "clustered"
    assert api.lib.adb_host_column_adopt_shards(C.byref(key), ptrs, S) == 0, api.lib.adb_host_last_error()
    cols = [key]
    if kind == "clustered":
        sib_data = np.arange(n, dtype=np.int32)
        sib = q.Column()
        sib.name, sib.row_count = b"sib", n
        sib.data = sib_data.ctypes.data_as(C.POINTER(C.c_int))
        cols.append(sib)
    arr = (C.POINTER(q.Column) * len(cols))(*[C.pointer(c) for c in cols])
    times = []
    for rep in range(reps + 1):
        if key.index:
            ix = key.index.contents
            for ptr in (ix.values, ix.positions, key.index):
                q._libc.free(C.cast(ptr, C.c_void_p))
            key.index = None
        if rep == 1:
            api.lib.adb_host_profile_dump()                     # drop the warm-up build's phases
        t0 = time.perf_counter()
        assert api.lib.adb_host_index_build(arr, len(cols), 0) == 0, api.lib.adb_host_last_error()
        times.append(time.perf_counter() - t0)
        hv = np.ctypeslib.as_array(key.index.contents.values, shape=(n,))
        hp = np.ctypeslib.as_array(key.index.contents.positions, shape=(n,))
        w = min(1 << 18, n)
        for a0 in (0, n // 3, n - w):
            vs = np.arange(a0, a0 + w, dtype=np.int64)
            assert np.array_equal(hv[a0:a0 + w], vs.astype(np.int32))
            exp = vs if kind == "clustered" else (vs - add) % n * inv % n
            assert np.array_equal(hp[a0:a0 + w], exp.astype(np.uint64))
    sys.stderr.flush()
    print(json.dumps({"build_s": times[1:], "warmup_s": times[0]}), flush=True)
    api.lib.adb_host_profile_dump()                             # the timed builds' phases, to stderr
    api.lib.adb_host_shutdown()


def parse_profile(text, reps):
    phases = {}
    for line in text.splitlines():
        m = re.match(r"\[adb shim profile\] (index: .+?)\s+(\d+)\s+([\d.]+)\s+([\d.]+)$", line)
        if m:
            phases[m.group(1)] = round(float(m.group(3)) / 1e6 / reps, 4)        # seconds per build
    return phases


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return {"devices": len(out), "device": out[0].split(",")[0].strip() if out else None,
                "power_limit": out[0].split(",")[1].strip() if out else None}
    except (OSError, subprocess.SubprocessError):
        return {"devices": None, "device": None, "power_limit": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", action="append", default=[])
    ap.add_argument("--label", action="append", default=[])
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--rows", type=int, default=N)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", nargs=3, metavar=("TREE", "G", "KIND"))
    a = ap.parse_args()
    if a.worker:
        worker(a.worker[0], int(a.worker[1]), a.worker[2], a.rows, a.reps)
        return
    trees = a.tree or [ROOT]
    labels = a.label or [os.path.basename(os.path.abspath(t)) for t in trees]
    record = {"rows": a.rows, "reps": a.reps, **device_info(), "runs": []}
    env = dict(os.environ, ADB_SHIM_PROFILE="1")
    # alternate the trees inside every (G, kind) so that both see the same machine state
    for G in a.gpus:
        for kind in ("unclustered", "clustered"):
            for tree, label in zip(trees, labels):
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--rows", str(a.rows), "--reps",
                                    str(a.reps), "--worker", os.path.abspath(tree), str(G), kind],
                                   capture_output=True, text=True, env=env)
                run = {"tree": label, "G": G, "kind": kind, "ok": p.returncode == 0}
                if p.returncode == 0:
                    res = json.loads(p.stdout.strip().splitlines()[-1])
                    run["build_s_median"] = round(statistics.median(res["build_s"]), 4)
                    run["build_s"] = [round(t, 4) for t in res["build_s"]]
                    run["warmup_s"] = round(res["warmup_s"], 4)
                    run["phases_s"] = parse_profile(p.stderr, a.reps)
                else:
                    run["error"] = (p.stderr or p.stdout)[-2000:]
                print(json.dumps(run), flush=True)
                record["runs"].append(run)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(record, f, indent=1)


if __name__ == "__main__":
    main()
