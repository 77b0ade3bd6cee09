"""Single-query search of an fp32 index from its int8 scan copy (option "scan_shadow") against the fp32 scan, one JSON line
per (rows, arm): time per search (CUDA events around `--iters` back-to-back searches of different queries), the bytes the
search reads (int8 codes and row scales plus the fp32 rows of the candidates it re-scored exactly) and their rate against
7.7 TB/s, the bound E of the first query, the distribution of the candidate count |C| over `--queries` queries and the
searches that needed more than one re-score round.  A separate pass with option "scan_clock" on (its searches are not
timed) reads the per-CTA %globaltimer stamps: the scan loop's time (first CTA start to last loop end) and rate, and the
phases of the last CTA's tail.

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
    clocks = scan_clock_pass(idx, qt, k, (n * d + n * 4) if shadow else n * d * 4)
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
    out.update(clocks)
    if shadow:
        c = np.asarray(cands)
        out["candidates"] = {"min": int(c.min()), "p50": float(np.percentile(c, 50)), "p90": float(np.percentile(c, 90)),
                             "p99": float(np.percentile(c, 99)), "max": int(c.max()), "mean": mean_c}
    del idx
    torch.cuda.empty_cache()
    return out


def scan_clock_pass(idx, qt, k, scan_bytes, searches=16):
    """Medians over `searches` searches of the loop time (first CTA start to the last CTA's loop end), the loop's rate over
    the bytes it streams, and the tail: last loop end -> the last CTA holds its ticket -> pool read -> the best KP ranked
    -> re-scored (the final ranking starts) -> results written (evs_scan.cuh: scan_pool_kernel).  Searches of the int8
    copy also split "ranked -> written" at the finalise stamps 5-7 (finalize stamps 2 -> 5 -> 6 -> 3 -> 7 -> 4):
      ranked_to_c_gathered_us      the window C read from the pool (its rows sent to L2 as they join);
      c_gathered_to_c_rescored_us  C re-scored once (with the re-score rounds first when C holds more than 1024 keys).
                                   Before C was re-scored in one pass: the rounds of 256 only;
      c_rescored_to_rank_start_us  the ranked members restricted to canonical scores >= b.  Before: the final re-score of
                                   the kept k and the last round's keys;
      rank_start_to_c_ranked_us    ranks by counting, results stored;
      c_ranked_to_written_us       padding, the guard."""
    evs.set_option("scan_clock", 1)
    rec = {"loop_us": [], "end_spread_us": [], "loop_end_to_ticket_us": [], "ticket_to_pool_read_us": [],
           "pool_read_to_ranked_us": [], "ranked_to_rescored_us": [], "rescored_to_written_us": [], "kernel_us": []}
    window = {"ranked_to_c_gathered_us": [], "c_gathered_to_c_rescored_us": [], "c_rescored_to_rank_start_us": [],
              "rank_start_to_c_ranked_us": [], "c_ranked_to_written_us": []}
    try:
        for i in range(searches):
            idx.search(qt[i:i + 1], k)
            c = idx.scan_clocks().astype(np.int64)
            st, fs = idx.last_cta_stamps.astype(np.int64), idx.finalize_stamps.astype(np.int64)
            t0, end = c[:, 0].min(), c[:, 1].max()
            for name, v in (("loop_us", end - t0), ("end_spread_us", end - c[:, 1].min()), ("loop_end_to_ticket_us", st[0] - end),
                            ("ticket_to_pool_read_us", fs[0] - st[0]), ("pool_read_to_ranked_us", fs[2] - fs[0]),
                            ("ranked_to_rescored_us", fs[3] - fs[2]), ("rescored_to_written_us", fs[4] - fs[3]),
                            ("kernel_us", fs[4] - t0)):
                rec[name].append(v / 1e3)
            if fs[5] and fs[6]:  # the int8 copy's window stamps
                for name, v in (("ranked_to_c_gathered_us", fs[5] - fs[2]), ("c_gathered_to_c_rescored_us", fs[6] - fs[5]),
                                ("c_rescored_to_rank_start_us", fs[3] - fs[6]), ("rank_start_to_c_ranked_us", fs[7] - fs[3]),
                                ("c_ranked_to_written_us", fs[4] - fs[7])):
                    window[name].append(v / 1e3)
    finally:
        evs.set_option("scan_clock", 0)
    if window["ranked_to_c_gathered_us"]:
        rec.update(window)
    out = {name: round(float(np.median(v)), 2) for name, v in rec.items()}
    out["loop_tb_s"] = round(scan_bytes / (out["loop_us"] * 1e-6) / 1e12, 3)
    return {"scan_clock": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[10_000_000, 1_250_000])
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--k", type=int, default=48)
    ap.add_argument("--queries", type=int, default=200)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shadow-min-rows", type=int, default=0, help="routing cut of the copy's path (0: every size above small_max_rows)")
    ap.add_argument("--ctas-per-sm", type=int, default=0, help="option ctas_per_sm (0: the planned default)")
    ap.add_argument("--chunk-groups", type=int, default=0, help="option scan_chunk_groups (0: the default)")
    ap.add_argument("--arms", type=int, nargs="+", default=[1, 0, 1, 0], help="scan_shadow of each pass, in order")
    a = ap.parse_args()
    evs.set_option("shadow_min_rows", a.shadow_min_rows)
    evs.set_option("ctas_per_sm", a.ctas_per_sm)
    if a.chunk_groups:
        evs.set_option("scan_chunk_groups", a.chunk_groups)
    info = gpu_info()
    lines = []
    for n in a.rows:
        for shadow in a.arms:
            r = probe(n, a.dim, a.k, shadow, a.queries if shadow else 0, a.iters)
            r.update(gpu=info, ctas_per_sm=evs.get_option("ctas_per_sm"), scan_chunk_groups=evs.get_option("scan_chunk_groups"))
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
