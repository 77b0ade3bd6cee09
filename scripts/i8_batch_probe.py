"""Batches of 1..16 queries (k = 48): ms per search through the exact batch search of the int8 copy (the route of 2..4
queries) against the single-tf32 tensor-core scan of the same batch (option scan_shadow = 0 for that leg: the copy is
dropped, so the batch takes the tensor-core path), and nq = 1 through the single-query search.  Also the bytes the int8
passes read (codes and scales) and their rate, the bound E of the first query (recomputed here from the copy's e_max with
the formula of DESIGN.md section 2) and the window |C| (largest over the queries).
Device API (CUDA tensors), CUDA events; synthetic unit-norm rows, larger than the 126 MB L2, so every pass reads HBM.

    python scripts/i8_batch_probe.py [--rows 1250000,10000000] [--out i8_batch_probe.jsonl]
"""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import evo_ssearch_b200 as evs  # noqa: E402

I8_QMAX = 127 * 256 + 127


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


def bound_e(q, max_norm, emax):
    """E of DESIGN.md section 2 for one query (fp32 query codes as the kernels derive them; fp64 sums)."""
    q = q.astype(np.float32)
    sq = np.float32(np.abs(q).max()) / np.float32(I8_QMAX)
    c = np.clip(np.rint(q / sq), -I8_QMAX, I8_QMAX) if sq > 0 else np.zeros_like(q)
    qh = np.float64(sq) * c.astype(np.float64)
    dq = math.sqrt(float(((q.astype(np.float64) - qh) ** 2).sum())) * (1 + 2 ** -20)
    qn = math.sqrt(float((qh ** 2).sum())) * (1 + 2 ** -20)
    nx = float(max_norm) * (1 + 2 ** -7)
    return (dq * nx + qn * emax + 2 ** -22 * qn * (nx + emax)) * (1 + 2 ** -20) + 2 ** -117


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="1250000,10000000")
    ap.add_argument("--d", type=int, default=512)
    ap.add_argument("--k", type=int, default=48)
    ap.add_argument("--nqs", default="1,2,3,4,5,6,7,8,9,10,11,12,13,14,15,16")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    emit({"gpu": gpu_info(), "torch": torch.__version__})
    d, k = a.d, a.k
    qi = evs.IndexFlatIP(d)
    qi.add_synthetic(16, seed=777)
    qh = qi.reconstruct_n(0, 16)
    q = torch.from_numpy(qh).cuda()
    for rows in [int(r) for r in a.rows.split(",")]:
        idx = evs.IndexFlatIP(d)
        idx.add_synthetic(rows, seed=11)
        emax = idx.shadow_stats()[1]
        E = bound_e(qh[0], idx.max_row_norm, emax)
        evs.set_option("scan_shadow", 0)  # the reference: no copy, so batches take the tensor-core scan of the fp32 rows
        ref = evs.IndexFlatIP(d)
        ref.add_synthetic(rows, seed=11)
        evs.set_option("scan_shadow", 1)
        for nq in [int(x) for x in a.nqs.split(",")]:
            qb = q[:nq].contiguous()
            p0 = idx.coalesce_stats()[2]
            ms = timed(lambda: idx.search(qb, k), a.iters)
            passes = (idx.coalesce_stats()[2] - p0) / (a.iters + 1)
            D, I = idx.search(qb, k)
            cand = idx.shadow_stats()[2]
            rec = {"rows": rows, "d": d, "k": k, "nq": nq, "route": "int8" if passes else ("single" if nq == 1 else "other"),
                   "ms": round(ms, 4), "us_per_query": round(1000 * ms / nq, 2), "passes": passes}
            if passes:
                nbytes = passes * rows * (d + 4)
                rec.update({"read_GB": round(nbytes / 1e9, 3), "read_TBps": round(nbytes / (ms * 1e-3) / 1e12, 2),
                            "E_q0": E, "window_max": cand})
            if nq >= 2:
                rec["tf32_ms"] = round(timed(lambda: ref.search(qb, k), a.iters), 4)
                D2, I2 = ref.search(qb, k)
                rec["same_as_tf32"] = bool(torch.equal(D, D2) and torch.equal(I, I2))
            emit(rec)
        del idx, ref
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
