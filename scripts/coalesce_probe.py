"""Concurrent single-query searches of one index, the application's traffic (threaded Flask server, one
`index.search(q.reshape(1, -1), k)` per request): T threads each issue numpy searches of their own seeded queries for a fixed
time.  One JSON line per (rows, k, T): queries per second, p50 / p99 latency per call, and the index's coalesce_stats()
moves (groups, grouped queries, int8 batch passes) when the build has them.  fp32 storage, synthetic unit-norm rows.

    python scripts/coalesce_probe.py [--rows 10000,1000000,10000000] [--threads 1,2,4,8,16,32] [--seconds 2]
                                     [--tree DIR]   (import the package from another checkout, e.g. the parent commit's)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ap = argparse.ArgumentParser()
ap.add_argument("--rows", default="10000,1000000,10000000")
ap.add_argument("--d", type=int, default=512)
ap.add_argument("--ks", default="12,48")
ap.add_argument("--threads", default="1,2,4,8,16,32")
ap.add_argument("--seconds", type=float, default=2.0)
ap.add_argument("--tree", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--label", default="")
ap.add_argument("--out", default=None)
a = ap.parse_args()
sys.path.insert(0, os.path.abspath(a.tree))

import numpy as np  # noqa: E402

import evo_ssearch_b200 as evs  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


out = open(a.out, "a") if a.out else None


def emit(rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        out.write(line + "\n")
        out.flush()


def stats(idx):
    return idx.coalesce_stats() if hasattr(idx, "coalesce_stats") else (0, 0, 0)


emit({"gpu": gpu_info(), "tree": os.path.abspath(a.tree), "label": a.label})
d = a.d
qsrc = evs.IndexFlatIP(d)
qsrc.add_synthetic(32 * 64, seed=4242)
Q = qsrc.reconstruct_n(0, 32 * 64).reshape(32, 64, d)  # thread t searches Q[t, i % 64]
for rows in [int(r) for r in a.rows.split(",")]:
    idx = evs.IndexFlatIP(d)
    idx.add_synthetic(rows, seed=0)
    for k in [int(x) for x in a.ks.split(",")]:
        for T in [int(x) for x in a.threads.split(",")]:
            for t in range(T):  # warm-up: every thread's buffers
                idx.search(Q[t, :1], k)
            lat = [[] for _ in range(T)]
            go = threading.Barrier(T + 1)
            stop = [0.0]

            def worker(t):
                qs = [np.ascontiguousarray(Q[t, i:i + 1]) for i in range(64)]
                go.wait()
                i = 0
                while True:
                    t0 = time.perf_counter()
                    if t0 >= stop[0]:
                        break
                    idx.search(qs[i % 64], k)
                    lat[t].append(time.perf_counter() - t0)
                    i += 1

            ths = [threading.Thread(target=worker, args=(t,)) for t in range(T)]
            for th in ths:
                th.start()
            s0 = stats(idx)
            stop[0] = time.perf_counter() + a.seconds
            t_start = time.perf_counter()
            go.wait()
            for th in ths:
                th.join()
            wall = time.perf_counter() - t_start
            s1 = stats(idx)
            allv = np.array([v for L in lat for v in L])
            emit({"label": a.label, "rows": rows, "k": k, "threads": T, "queries": int(allv.size),
                  "qps": round(allv.size / wall, 1), "p50_ms": round(1e3 * float(np.percentile(allv, 50)), 4),
                  "p99_ms": round(1e3 * float(np.percentile(allv, 99)), 4),
                  "groups": s1[0] - s0[0], "grouped_queries": s1[1] - s0[1], "i8_batch_passes": s1[2] - s0[2]})
    del idx
