"""Single-query search of an fp32 index from its int8 scan copy (option "scan_shadow") against the fp32 scan, one JSON line
per (rows, arm): time per search (CUDA events around `--iters` back-to-back searches of different queries), the bytes the
search reads (int8 codes and row scales plus the fp32 rows of the candidates it re-scored exactly) and their rate against
7.7 TB/s, the bound E of the first query, the distribution of the candidate count |C| over `--queries` queries and the
searches that needed more than one re-score round.

    python scripts/shadow_probe.py --rows 10000000 1250000 --out shadow_probe.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import evo_ssearch_b200 as evs  # noqa: E402

HBM_PEAK = 7.7e12  # bytes/s, HGX B200 data sheet (one GPU)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else ""
    except Exception:
        return ""


def probe(n, d, k, shadow, queries, iters, seed=5):
    import torch
    evs.set_option("scan_shadow", shadow)  # before the add: the fp32 arm builds no copy
    idx = evs.IndexFlatIP(d)
    idx.add_synthetic(n, seed=seed)
    rng = np.random.default_rng(1)
    q = rng.standard_normal((max(queries, iters), d)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    qt = torch.from_numpy(q).cuda()
    Dd = torch.empty((1, k), dtype=torch.float32, device="cuda")
    Id = torch.empty((1, k), dtype=torch.int64, device="cuda")
    cands = []
    for i in range(queries):  # candidate counts (one host read after each search)
        idx.search(qt[i:i + 1], k, D=Dd, I=Id)
        torch.cuda.synchronize()
        cands.append(idx.shadow_stats()[2])
    for i in range(10):
        idx.search(qt[i:i + 1], k, D=Dd, I=Id)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        idx.search(qt[i:i + 1], k, D=Dd, I=Id)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    wide, emax, _ = idx.shadow_stats()
    # E of the first query (evs_scan.cuh: shadow_bound_i8)
    q0 = q[0]
    sq = np.float32(np.abs(q0).max() / np.float32(32639))
    qh = float(sq) * np.clip(np.rint((q0 / sq).astype(np.float32)), -32639, 32639).astype(np.float64)
    dq, qhn, nx = np.linalg.norm(q0.astype(np.float64) - qh), np.linalg.norm(qh), idx.max_row_norm * (1 + 2.0**-7)
    E = dq * nx + qhn * emax + 2.0**-22 * qhn * (nx + emax)
    mean_c = float(np.mean(cands)) if shadow else 0.0
    nbytes = (n * d + n * 4 if shadow else n * d * 4) + mean_c * d * 4
    out = {"rows": n, "d": d, "k": k, "scan_shadow": shadow, "ms_per_search": ms, "bytes_per_search": nbytes,
           "tb_s": nbytes / ms / 1e9, "frac_hbm_peak": nbytes / (ms * 1e-3) / HBM_PEAK, "emax": emax,
           "E_first_query": E if shadow else None, "wide_searches": wide, "queries": queries}
    if shadow:
        c = np.asarray(cands)
        out["candidates"] = {"min": int(c.min()), "p50": float(np.percentile(c, 50)), "p90": float(np.percentile(c, 90)),
                             "p99": float(np.percentile(c, 99)), "max": int(c.max()), "mean": mean_c}
    del idx
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[10_000_000, 1_250_000])
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--k", type=int, default=48)
    ap.add_argument("--queries", type=int, default=200)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shadow-min-rows", type=int, default=0, help="routing cut of the copy's path (0: every size above small_max_rows)")
    a = ap.parse_args()
    evs.set_option("shadow_min_rows", a.shadow_min_rows)
    info = gpu_info()
    lines = []
    for n in a.rows:
        for shadow in (1, 0, 1, 0):
            r = probe(n, a.dim, a.k, shadow, a.queries if shadow else 0, a.iters)
            r["gpu"] = info
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
