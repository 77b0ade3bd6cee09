"""Large-k search (option max_k, k > 112): time per search, split into the score scan and the rest, the scan loop's read rate
and the candidate count |C|, beside the same build's k = 112 search and its k = 48 single-query search over the fp32 rows
(scan_shadow = 0).  One JSON line per (rows, storage, nq, k).  Device API (CUDA tensors), CUDA events on the current
stream; synthetic unit-norm rows, so every size larger than the 126 MB L2 is read from HBM.

    python scripts/large_k_probe.py [--rows 10000,1000000,10000000] [--out large_k_probe.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import evo_ssearch_b200 as evs  # noqa: E402


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="10000,1000000,10000000")
    ap.add_argument("--d", type=int, default=512)
    ap.add_argument("--storages", default="f32,bf16")
    ap.add_argument("--nqs", default="1,16")
    ap.add_argument("--ks", default="113,512,2048")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    evs.set_option("max_k", 2048)
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    emit({"gpu": gpu_info(), "torch": torch.__version__})
    d = a.d
    for n in [int(v) for v in a.rows.split(",")]:
        for storage in a.storages.split(","):
            idx = evs.IndexFlatIP(d, storage=storage)
            idx.add_synthetic(n, seed=1)
            ks = [int(v) for v in a.ks.split(",")] + ([200] if n <= 10000 else [])
            for nq in [int(v) for v in a.nqs.split(",")]:
                q = torch.randn(nq, d, device="cuda")
                q /= q.norm(dim=1, keepdim=True)
                iters = 50 if n * nq <= 10_000_000 else 10
                ref112 = timed(lambda: idx.search(q, 112), iters)
                evs.set_option("scan_shadow", 0)
                ref48 = timed(lambda: idx.search(q, 48), iters)
                evs.set_option("scan_shadow", 1)
                for k in ks:
                    ms = timed(lambda: idx.search(q, k), iters)
                    scan = idx.time_scan(q, k, iters=iters)
                    qpp = 4  # max_queries_per_pass(512): every pass reads the fp32 rows once
                    passes = -(-nq // qpp)
                    _, cand = idx.large_k_stats()
                    emit({"rows": n, "d": d, "storage": storage, "nq": nq, "k": k, "ms": round(ms, 4), "scan_ms": round(scan, 4),
                          "rest_ms": round(ms - scan, 4), "scan_TBps": round(n * d * 4 * passes / (scan * 1e-3) / 1e12, 3),
                          "candidates": cand, "k112_ms": round(ref112, 4), "k48_fp32_scan_ms": round(ref48, 4),
                          "ratio_vs_k112": round(ms / ref112, 3), "ratio_vs_k48_fp32": round(ms / ref48, 3)})
            del idx
            torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
