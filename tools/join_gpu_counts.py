"""BASELINE config 4 (hash join of two 100 M-row tables) through the operator API's hash_join at
G = 1 .. 8 engine contexts, one subprocess per G, all in one command.

Every G runs bench.api_join: the 2 M-row join first, element for element against the oracle (it
stops on a difference), then the timed 100 M x 100 M joins with prefilters 0.8 / 0.15 and
1.0 / 1.0.  Writes profiles/r03_join_gpu_counts.json (or --out) with the ms per G and the device
name, power limit and device count read in the same process.  With fewer devices than contexts
the contexts share devices.

    python tools/join_gpu_counts.py [--gpus 1,2,3,4,5,6,7,8] [--out profiles/r03_join_gpu_counts.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PREFILTERS = ("prefilter_0.8_0.15", "prefilter_1.0_1.0")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    name, power = out[0].split(", ")
    return {"device": name, "power_limit": power, "device_count": len(out)}


def run_one(G):
    """One G in this process: the host with G contexts, then bench.api_join."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import analytical_database_b200 as adb
    import bench
    import query_api as q
    eng = adb.Engine(0)
    api = q.Api()
    assert api.lib.adb_host_init_multi(G) == 0, api.lib.adb_host_last_error()

    def sync_all():
        for g in range(G):
            eng.lib.adb_ctx_select(g)
            eng.sync()
        eng.lib.adb_ctx_select(0)
    cases = bench.api_join(eng, api, q, G, sync_all)
    api.lib.adb_host_shutdown()
    print(json.dumps({"G": G, **gpu_info(), "cases": cases}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,3,4,5,6,7,8")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_join_gpu_counts.json"))
    ap.add_argument("--one", type=int, help=argparse.SUPPRESS)      # the per-G subprocess
    args = ap.parse_args()
    if args.one:
        run_one(args.one)
        return 0
    res = {**gpu_info(), "timing": "bench.api_join: host wall clock of hash_join between device synchronises, "
                                   "best of the last 3 of 4 calls", "runs": []}
    ok = True
    for G in [int(x) for x in args.gpus.split(",")]:
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", str(G)], capture_output=True, text=True)
        line = next((x for x in reversed(p.stdout.splitlines()) if x.startswith("{")), None)
        if p.returncode or line is None:
            ok = False
            res["runs"].append({"G": G, "error": (p.stdout + p.stderr)[-2000:]})
            print(f"G={G} failed:\n{(p.stdout + p.stderr)[-2000:]}", flush=True)
            continue
        r = json.loads(line)
        run = {"G": G, "parity": r["cases"]["parity"], "parity_detail": r["cases"]["parity_detail"],
               "device": r["device"], "power_limit": r["power_limit"], "device_count": r["device_count"],
               **{k: r["cases"][k] for k in PREFILTERS}}
        res["runs"].append(run)
        print(f"G={G}: " + ", ".join(f"{k} {run[k]['ms']:.2f} ms" for k in PREFILTERS), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
