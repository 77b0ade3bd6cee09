#!/usr/bin/env python
"""bench.py -- flat inner-product top-k queries/sec at 10M x 512, k = 48 (BASELINE.json `metric`).

    python bench.py [--gpus N --steps K --warmup W]            the CUDA path (one process per GPU)
    python bench.py --impl reference [...]                     the CPU reference arm (oracle port, ALL rows)
    python bench.py [...] --dump-outputs DIR                   also write the last timed step's (D, I) under DIR

A "step" is ONE search call: a batch of `--nq` queries (default 1 -- what the app issues,
oldapp.py:2005, and the case the north_star's roofline target names) scored against all rows, top-48
selected, results delivered.  The database is synthetic (counter-based unit-norm rows, seed 0) and is
row-sharded over the N ranks (total work fixed -> "strong" scaling); each step uses a different query.
The database (20.48 GB fp32) is far larger than the 126 MB L2, so no L2 flush is needed between steps.

One JSON line is printed by rank 0:
  value     whole-job queries/s with queries already resident in HBM, device-timed with CUDA events
            between barrier + synchronize, max over ranks
  e2e       the same through the public host API (numpy in, numpy out): pinned H2D of the query and D2H
            of (D, I) inside the timed region
  roofline  the scan kernel: algorithmic bytes per launch / its mean duration (CUDA events recorded by
            libevs around every scan launch inside the timed region) against the measured HBM peak
  parity    answers, not speed: host API == device API on the last step's query; self-match property at full size (a query
            equal to database row r must return r first with score ~1); at N > 1 rank 0 ALSO holds the unsharded database
            and the sharded (D, I) must equal the single-GPU (D, I) bit for bit
  configs   the other BASELINE configurations that fit this launch (C1 latency, C2, C3 at N = 1; C4 at N >= 2; C5 at N = 8)
  cpu_baseline  the CPU oracle (a labelled port of faiss-cpu's flat-IP scan; faiss itself is not
            installable here) timed on this box's host cores on a bounded row sample
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "flat-IP top-k queries/sec @10M x 512 k=48"
UNIT = "queries/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="evs", choices=["evs", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--nq", type=int, default=1)
    ap.add_argument("--k", type=int, default=48)
    ap.add_argument("--storage", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--variant", type=int, default=0, help="scan kernel: 0 auto, 1 direct loads, 2 bulk-async ring")
    ap.add_argument("--cpu-rows", type=int, default=2_000_000, help="row sample for the cpu_baseline leg of the CUDA arm")
    ap.add_argument("--ref-rows", type=int, default=0, help="rows the reference arm scans per step (0 = all of --rows)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how shard partials meet -- peer-store exchange kernels over NVLink, or NCCL all-gather + merge")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configurations reported under 'configs'")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity block (N > 1: the unsharded copy on rank 0)")
    ap.add_argument("--tc-min-nq", type=int, default=None, help="override the library's tensor-core threshold (experiments)")
    ap.add_argument("--set", action="append", default=[], metavar="NAME=VALUE", help="evs.set_option before the run (experiments)")
    ap.add_argument("--extra", action="store_true", help="also time query batches 1/4/16/64 (reported under 'extra')")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the (D, I) the last timed step returned as DIR/D.npy and DIR/I.npy, to compare builds output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs:
        os.makedirs(a.dump_outputs, exist_ok=True)  # an unwritable DIR fails before the run, not after it
    return a


def workload_name(a) -> str:
    return f"{a.rows}x{a.dim} {a.storage} flat-IP, nq={a.nq}, k={a.k}"


# ------------------------------------------------------------------------------------------------
# clocks during the timed region: NVML polled in-process every few milliseconds (the timed region of the metric is
# 10-60 ms long: nvidia-smi's 100 ms loop sees nothing of it); nvidia-smi is the fallback
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
               ("hw_power_brake_slowdown", 0x80))

    def __init__(self, gpu_index: int, period_s: float = 0.004):
        self.gpu, self.period = gpu_index, period_s
        self.sm, self.power, self.reasons = [], [], set()
        self.max_sm = None
        self._stop = threading.Event()
        self._thread = None
        self.source = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            # torch may see a permuted / masked device list: map through CUDA_VISIBLE_DEVICES when it is a plain list
            phys = self.gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis and all(p.strip().isdigit() for p in vis.split(",")):
                phys = int(vis.split(",")[self.gpu])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.source = f"NVML in-process, {self.period * 1e3:.0f} ms period"
        except Exception:  # noqa: BLE001
            self.nvml = None
            self.source = "nvidia-smi -lms 100 (NVML unavailable)"
        self._thread = threading.Thread(target=self._poll_nvml if self.nvml else self._poll_smi, daemon=True)
        self._thread.start()

    def _poll_nvml(self):
        n = self.nvml
        while not self._stop.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.power.append(n.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                try:
                    r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001 - older binding name
                    r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in self.REASONS:
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def _poll_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                     "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.source = "unavailable"
            return
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        os.set_blocking(proc.stdout.fileno(), False)
        buf = ""
        while not self._stop.is_set():
            try:
                chunk = proc.stdout.read()
            except Exception:  # noqa: BLE001
                chunk = None
            if chunk:
                buf += chunk
                *lines, buf = buf.split("\n")
                for ln in lines:
                    f = [x.strip() for x in ln.split(",")]
                    if len(f) < 7:
                        continue
                    try:
                        self.sm.append(float(f[0]))
                        self.max_sm = max(self.max_sm or 0.0, float(f[1]))
                        self.power.append(float(f[2]))
                    except ValueError:
                        continue
                    for nm, v in zip(names, f[3:7]):
                        if v.lower().startswith("active"):
                            self.reasons.add(nm)
            self._stop.wait(0.05)
        proc.terminate()

    def stop(self) -> dict:
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=5)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_sm,
                "power_w_max": max(self.power) if self.power else None, "samples": len(self.sm),
                "reasons": sorted(self.reasons), "source": self.source}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_peak_tflops():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["bf16_tflops"]), float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, D, I) -> None:
    """One search's answer as .npy files: D float32 [nq, k] and I as float64 (ids are exact below 2^53).  An answer larger
    than 64 MB is cut to a fixed, seeded sample of its queries, whose row numbers go to rows.npy."""
    D = np.asarray(D, dtype=np.float32)
    I = np.asarray(I).astype(np.float64)
    nq, k = D.shape
    keep = (DUMP_LIMIT_BYTES - 4096) // (k * 12 + 8)  # 4 + 8 bytes per result, 8 per row number, room for three headers
    rows_path = os.path.join(out_dir, "rows.npy")
    if nq > keep:
        rows = np.sort(np.random.default_rng(0).choice(nq, keep, replace=False))
        D, I = D[rows], I[rows]
        np.save(rows_path, rows.astype(np.float64))
    elif os.path.exists(rows_path):
        os.remove(rows_path)  # left by an earlier, sampled dump
    np.save(os.path.join(out_dir, "D.npy"), D)
    np.save(os.path.join(out_dir, "I.npy"), I)


def scan_arithmetic(evs, storage: str, nq: int, rows_per_gpu: int, dim: int) -> str:
    """Which arithmetic scans a batch (mirrors plan_path in evs_api.cu); the final ranking is always the fp64 re-score."""
    tcmin = evs.get_option("tc_min_nq")
    if not (tcmin > 0 and nq >= tcmin and rows_per_gpu >= 65536):
        return ("bf16 rows, " if storage == "bf16" else "") + "fp32 CUDA-core GEMV (FFMA), fp32 accumulate"
    if storage == "bf16":
        return "bf16 tensor-core scan (tcgen05.mma kind::f16), fp32 accumulate"
    if evs.get_option("x3") and nq <= evs.get_option("x3_max_nq") and dim * 4 % 128 == 0 and dim <= 768:
        return "3xTF32 tensor-core scan (tcgen05.mma kind::tf32, hi/lo split operands, 3 MMAs per K step), fp32 accumulate"
    return ("single-tf32 tensor-core scan (tcgen05.mma kind::tf32) + on-device certification against the rigorous truncation bound "
            "+ fp32 GEMV re-run of uncertified queries")


def device_timed(torch, dev, fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def config_legs_single(evs, torch, dev, k):
    """BASELINE configs 1, 2 and 3 on this GPU.  C1 (the reference's own scale) is a latency leg: microseconds per
    query through the host API and on the device.  C2 / C3 are device-timed (CUDA events on torch's stream around
    back-to-back IndexFlatIP.search calls with device-resident queries) and carry their own roofline: HBM for the
    streaming cases, dense bf16 tensor throughput for the 4096-query batch."""
    hbm_peak, _ = measured_peak_gbs()
    tf_burst, tf_sust, tf_src = measured_peak_tflops()
    out = []

    def queries(d, nq, seed=1):
        qi = evs.IndexFlatIP(d, device=dev.index)
        qi.add_synthetic(nq, seed=seed)
        return qi.reconstruct_n(0, nq)

    # ---- C1: 10k x 512, 1 query, k = 12 (what the application really runs) ----
    idx = evs.IndexFlatIP(512, device=dev.index)
    idx.add_synthetic(10_000, seed=0)
    qh = queries(512, 64)
    qd = torch.from_numpy(qh).to(dev)
    for i in range(20):
        idx.search(qh[i % 64:i % 64 + 1], 12)
    t0 = time.perf_counter()
    reps = 2000
    for i in range(reps):
        idx.search(qh[i % 64:i % 64 + 1], 12)
    host_us = (time.perf_counter() - t0) / reps * 1e6
    l0 = evs.kernel_launches()
    q1 = qd[:1].contiguous()
    Dd = torch.empty((1, 12), dtype=torch.float32, device=dev)  # outputs allocated once: the loop must stay ahead of a 16 us kernel
    Id = torch.empty((1, 12), dtype=torch.int64, device=dev)
    dev_us = device_timed(torch, dev, lambda: idx.search(q1, 12, D=Dd, I=Id), 2000, 50) * 1e3
    launches = (evs.kernel_launches() - l0) / 2050
    out.append({"config": "C1: 10000x512 f32, nq=1, k=12", "e2e_us_per_query": host_us, "e2e_queries_per_s": 1e6 / host_us,
                "device_us_per_query": dev_us, "kernel_launches_per_query": launches,
                "note": "e2e = IndexFlatIP.search(numpy) -> numpy: ONE kernel (small-shard scan + fused finalise) with the query in "
                        "its parameter block, results written to mapped pinned memory, completion word polled; device = "
                        "back-to-back searches of a device-resident query into preallocated outputs, CUDA events"})
    del idx

    for tag, rows, d, storage, nqs in (("C2", 1_000_000, 512, "f32", (1, 16)), ("C3", 1_000_000, 512, "bf16", (4096,))):
        idx = evs.IndexFlatIP(d, device=dev.index, storage=storage)
        idx.reserve(rows)
        idx.add_synthetic(rows, seed=0)
        esz = 2 if storage == "bf16" else 4
        for nq in nqs:
            xq = torch.from_numpy(queries(d, nq)).to(dev)
            ms = device_timed(torch, dev, lambda: idx.search(xq, k), 50 if nq <= 64 else 5)
            scan_ms = idx.time_scan(xq, k, iters=20 if nq <= 64 else 3)
            rec = {"config": f"{tag}: {rows}x{d} {storage}, nq={nq}, k={k}", "ms_per_search": ms, "queries_per_s": nq / ms * 1e3,
                   "scan_ms": scan_ms, "scan_arithmetic": scan_arithmetic(evs, storage, nq, rows, d)}
            if nq <= 64:
                alg = rows * d * esz + nq * d * 4 + nq * k * 12
                ach = alg / (scan_ms * 1e-3) / 1e9
                rec["roofline"] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                                   "frac_whole_search": alg / (ms * 1e-3) / 1e9 / hbm_peak}
                if storage == "f32" and nq > 1:
                    # the same batch on the fp32 CUDA-core GEMV (4 queries per database pass at d = 512), for the record
                    old = evs.get_option("tc_min_nq")
                    evs.set_option("tc_min_nq", 0)
                    gms = device_timed(torch, dev, lambda: idx.search(xq, k), 20)
                    evs.set_option("tc_min_nq", old)
                    rec["fp32_gemv_ms_per_search"] = gms
                    rec["fp32_gemv_queries_per_s"] = nq / gms * 1e3
                    rec["guard"] = dict(zip(("device_reruns", "uncertified"), idx.guard_stats()))
                    rec["guard"]["searches"] = 50 + 3 + 21
                    # ... and on the 3xTF32 split scan (fp32-class scan scores from the tensor cores, option "x3")
                    oldx = evs.get_option("x3")
                    evs.set_option("x3", 1)
                    if idx.tc_x3_max_queries() >= nq:
                        rec["x3_ms_per_search"] = device_timed(torch, dev, lambda: idx.search(xq, k), 20)
                        rec["x3_scan_ms"] = idx.time_scan(xq, k, iters=20)
                    evs.set_option("x3", oldx)
            else:
                flops = 2.0 * nq * rows * d
                ach = flops / (scan_ms * 1e-3) / 1e12
                rec["roofline"] = {"bound": "tensor", "achieved": ach, "peak": tf_burst, "unit": "TFLOP/s", "frac": ach / tf_burst,
                                   "frac_of_sustained": ach / tf_sust, "peak_source": tf_src,
                                   "frac_whole_search": flops / (ms * 1e-3) / 1e12 / tf_burst,
                                   "kernel": "evs::tc2_scan_kernel (tcgen05.mma cta_group::2) incl. threshold pre-pass, tau0, gather"}
                rec["tc_fallbacks"] = evs.get_option("tc_fallbacks")
            out.append(rec)
        del idx
    return out


def config_legs_sharded(evs, torch, dist, dev, world, rank, a, barrier, max_over_ranks):
    """BASELINE configs 4 (10M x 768 over 2/4/8 GPUs, 1 and 1024 queries) and -- at 8 GPUs -- 5 (100M x 512 bf16, 1 and 16
    queries): device-timed like the metric (CUDA events between barriers, max over ranks), with the per-GPU roofline."""
    hbm_peak, _ = measured_peak_gbs()
    tf_burst, _, _ = measured_peak_tflops()
    legs = [("C4", 10_000_000, 768, "f32", 1, 40), ("C4", 10_000_000, 768, "bf16", 1024, 10)]
    if world >= 8:
        legs += [("C5", 100_000_000, 512, "bf16", 1, 40), ("C5", 100_000_000, 512, "bf16", 16, 20)]
    out = []
    cur = None
    index = None
    for tag, rows, d, storage, nq, steps in legs:
        if cur != (rows, d, storage):
            del index
            torch.cuda.empty_cache()
            index = evs.ShardedIndexFlatIP(d, device=dev.index, storage=storage, exchange=a.exchange,
                                           exchange_max_nq=1024, exchange_max_k=a.k)
            index.add_synthetic(rows, seed=0)
            cur = (rows, d, storage)
        lo, hi = evs.shard_bounds(rows, world, rank)
        qi = evs.IndexFlatIP(d, device=dev.index)
        qi.add_synthetic(8 * nq, seed=1)
        qd = torch.from_numpy(qi.reconstruct_n(0, 8 * nq).reshape(8, nq, d)).to(dev)
        del qi
        for i in range(3):
            index.search_tensor(qd[i % 8], a.k)
        index.local.scan_profile()
        evs.set_option("profile_scans", 1)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            index.search_tensor(qd[i % 8], a.k)
        e1.record()
        barrier()
        evs.set_option("profile_scans", 0)
        ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        n_prof, scan_sum = index.local.scan_profile()
        scan_ms = scan_sum / max(n_prof, 1)
        esz = 2 if storage == "bf16" else 4
        rec = {"config": f"{tag}: {rows}x{d} {storage} over {world} GPUs, nq={nq}, k={a.k}", "ms_per_search": ms,
               "queries_per_s": nq / ms * 1e3, "scan_ms_rank0": scan_ms, "rows_per_gpu": hi - lo,
               "scan_arithmetic": scan_arithmetic(evs, storage, nq, hi - lo, d)}
        if nq <= 64:
            alg = (hi - lo) * d * esz + nq * d * 4 + nq * a.k * 12
            ach = alg / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
            rec["roofline"] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                               "frac_of_nominal_8TBs": ach / 8000.0,
                               "frac_whole_search": alg / (ms * 1e-3) / 1e9 / hbm_peak, "per": "GPU (rank 0)"}
        else:
            flops = 2.0 * nq * (hi - lo) * d
            ach = flops / (scan_ms * 1e-3) / 1e12 if scan_ms > 0 else 0.0
            rec["roofline"] = {"bound": "tensor", "achieved": ach, "peak": tf_burst, "unit": "TFLOP/s", "frac": ach / tf_burst,
                               "frac_whole_search": flops / (ms * 1e-3) / 1e12 / tf_burst, "per": "GPU (rank 0)"}
        # answers at full size (no single GPU holds these databases): a query equal to database row r -- regenerated from its
        # global id -- must return r first with score ~1, scores descending; probes fall into different shards
        ok_self = True
        probes = [0, rows // 7, rows // 2 + 3, (rows * 6) // 7, rows - 1]
        for r in probes:
            pi = evs.IndexFlatIP(d, device=dev.index)
            pi.id_base = r
            pi.add_synthetic(1, seed=0)
            qrow = np.repeat(pi.reconstruct_n(0, 1), min(nq, 16), axis=0)
            del pi
            Dp, Ip = index.search(qrow, a.k)
            tol = 1e-5 if storage == "f32" else 1e-2  # the re-score is fp64 over the fp32 master rows either way
            ok_self = ok_self and bool((Ip[:, 0] == r).all()) and abs(float(Dp[0, 0]) - 1.0) < tol and bool((np.diff(Dp.astype(np.float64), axis=1) <= 0).all())
        rec["self_match_at_full_size"] = bool(ok_self)
        rec["self_match_rows"] = probes
        out.append(rec)
    del index
    torch.cuda.empty_cache()
    return out


def ncu_traffic_per_launch(a, world):
    """dram bytes per scan launch from the committed ncu capture of this same workload, else None."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(p):
        return None
    try:
        for rec in json.load(open(p)):
            if (rec["rows_per_gpu"], rec["dim"], rec["storage"], rec["nq"]) == (-(-a.rows // world), a.dim, a.storage, a.nq):
                return rec["dram_bytes_per_launch"]
    except Exception:  # noqa: BLE001
        return None
    return None


# ------------------------------------------------------------------------------------------------
# CPU legs (oracle = test infrastructure; used here only as the timed baseline)
# ------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Threads the CPU legs use: every core this process may run on.  (torchrun exports OMP_NUM_THREADS=1 to its
    workers, which would silently turn the all-cores baseline into a single-thread one.)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_baseline(a, seconds_budget: float = 12.0) -> dict:
    import oracle
    cores = host_threads()
    rows = min(a.rows, a.cpu_rows)
    xb = oracle.synth_fill(rows, a.dim, seed=0, nthreads=cores)
    xq = oracle.synth_fill(max(a.nq, 8), a.dim, seed=1)
    scale = rows / a.rows  # a flat scan is linear in rows: q/s at the full size = q/s on the sample * rows/full

    def run(fn, min_reps=3):
        fn(0)
        t0 = time.perf_counter()
        reps = 0
        while reps < min_reps or time.perf_counter() - t0 < seconds_budget / 2:
            fn(reps)
            reps += 1
            if reps >= 2000:
                break
        return reps * a.nq / (time.perf_counter() - t0)

    def q(i):
        return np.roll(xq, i, axis=0)[:a.nq]

    all_qps = run(lambda i: oracle.allcores_search(q(i), xb, a.k, nthreads=cores))
    seq_qps = run(lambda i: oracle.faiss_seq_search(q(i), xb, a.k, simd=True, nthreads=cores))
    return {
        "value": all_qps * scale, "unit": UNIT, "cores": cores, "kind": "port",
        "sample": f"{rows} of {a.rows} rows x {a.dim}, nq={a.nq}, k={a.k}; q/s scaled by {scale:g} (flat scan is linear in rows); "
                  f"all-cores row-split scan of the oracle port (faiss-cpu not installable); the reference ARM (--impl reference) "
                  f"scans all rows",
        "faiss_threading_value": seq_qps * scale,
        "faiss_threading_note": "same port with faiss's own threading (parallel over queries only: one thread scans "
                                "the database for a single query)",
    }


def run_reference(a) -> int:
    """The CPU reference arm: the oracle port of faiss-cpu IndexFlatIP on this box's host cores, on the SAME workload --
    every step scans all --rows rows (no sampling, no scaling)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle
    cores = host_threads()
    rows = a.ref_rows if a.ref_rows > 0 else a.rows
    rows = min(rows, a.rows)
    t_fill = time.perf_counter()
    xb = oracle.synth_fill(rows, a.dim, seed=0, nthreads=cores)
    t_fill = time.perf_counter() - t_fill
    xq = oracle.synth_fill(64, a.dim, seed=1)
    scale = rows / a.rows

    def step(i):
        qs = np.roll(xq, -i, axis=0)[:a.nq]
        return oracle.allcores_search(qs, xb, a.k, nthreads=cores)

    for i in range(a.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(a.steps):
        D_last, I_last = step(a.warmup + i)
    dt = time.perf_counter() - t0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, D_last, I_last)
    qps = a.steps * a.nq / dt * scale
    # faiss's own threading for the same call, for the record (short)
    t1 = time.perf_counter()
    reps = 0
    while reps < 2 or time.perf_counter() - t1 < 3.0:
        oracle.faiss_seq_search(np.roll(xq, -reps, axis=0)[:a.nq], xb, a.k, simd=True, nthreads=cores)
        reps += 1
    seq_qps = reps * a.nq / (time.perf_counter() - t1) * scale
    if rows == a.rows:
        sample = (f"each step scans ALL {a.rows} rows x {a.dim} (nq={a.nq}, k={a.k}) with all {cores} host threads "
                  f"(rows split across threads); no sampling, no scaling")
    else:
        sample = (f"each step scans {rows} of {a.rows} rows x {a.dim} (nq={a.nq}, k={a.k}) with all {cores} host threads; "
                  f"q/s scaled by {scale:g} (--ref-rows)")
    line = {
        "impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3 / scale, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "rows": a.rows, "dim": a.dim, "nq": a.nq, "k": a.k,
                   "rows_scanned_per_step": rows, "build_s": round(t_fill, 2),
                   "engine": "oracle port of faiss-cpu IndexFlatIP (faiss not installable in this image)"},
        "cpu_baseline": {"value": qps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "faiss_threading_value": seq_qps},
        "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# the CUDA arm
# ------------------------------------------------------------------------------------------------
def run_evs(a) -> int:
    import torch
    import torch.distributed as dist
    import evo_ssearch_b200 as evs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        print(f"warning: --gpus {a.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    if evs.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device; the evs arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    evs.set_option("scan_variant", a.variant)
    if a.tc_min_nq is not None:
        evs.set_option("tc_min_nq", a.tc_min_nq)
    for kv in a.set:
        name, val = kv.split("=")
        evs.set_option(name, int(val))
    index = evs.ShardedIndexFlatIP(a.dim, device=local_rank, storage=a.storage, exchange=a.exchange,
                                   exchange_max_nq=max(64, a.nq), exchange_max_k=a.k)
    t_build = time.perf_counter()
    index.add_synthetic(a.rows, seed=0)
    barrier()
    t_build = time.perf_counter() - t_build
    lo, hi = evs.shard_bounds(a.rows, world, rank)

    # query pool: counter-based unit-norm queries (seed 1), identical on every rank
    pool = 64
    qidx = evs.IndexFlatIP(a.dim, device=local_rank)
    qidx.add_synthetic(pool * a.nq, seed=1)
    q_host = qidx.reconstruct_n(0, pool * a.nq).reshape(pool, a.nq, a.dim)
    del qidx
    q_dev = torch.from_numpy(q_host).to(dev)

    def timed_device(nq_pool, steps, warmup, profile=False):
        for i in range(warmup):
            index.search_tensor(nq_pool[i % pool], a.k)
        if profile:
            index.local.scan_profile()
            evs.set_option("profile_scans", 1)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = evs.kernel_launches()
        e0.record()
        for i in range(steps):
            D, I = index.search_tensor(nq_pool[(warmup + i) % pool], a.k)
        e1.record()
        barrier()
        launches = evs.kernel_launches() - l0
        evs.set_option("profile_scans", 0)
        ms = max_over_ranks(e0.elapsed_time(e1))
        return ms, launches, (D, I)

    # ---- value: device-resident queries, device-timed ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.02)
    # A single query (k <= 48) is ONE kernel launch per search and per rank (scan + selection + finalise [+ exchange + merge]):
    # the kernel's mean duration is then the timed region divided by the steps -- CUDA events on the launching stream at
    # the region's ends, nothing between the launches (a per-launch event pair would break the programmatic overlap of
    # consecutive searches: +9 us per step at 8 ranks).  Other batches keep libevs' per-launch event pairs around the scan.
    one_launch = a.nq == 1 and a.k <= 48 and evs.get_option("fuse_finalize") == 1 and (world == 1 or a.exchange == "peer")
    ms_total, launches, (D_last, I_last) = timed_device(q_dev, a.steps, a.warmup, profile=not one_launch)
    n_prof, scan_ms_sum = index.local.scan_profile()
    one_launch = one_launch and launches == a.steps
    if one_launch:
        n_prof, scan_ms_sum = a.steps, ms_total
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and a.dump_outputs:  # every rank holds the same merged (D, I)
        dump_outputs(a.dump_outputs, D_last.cpu().numpy(), I_last.cpu().numpy())
    value = a.steps * a.nq / (ms_total * 1e-3)
    events_check = None
    if one_launch:  # cross-check: the same kernel with libevs' own event pair around every launch (a short extra pass)
        ms_ev, _, _ = timed_device(q_dev, min(a.steps, 50), 3, profile=True)
        n_ev, sum_ev = index.local.scan_profile()
        events_check = {"kernel_ms_between_per_launch_events": sum_ev / max(n_ev, 1), "ms_per_step_with_those_events": ms_ev / min(a.steps, 50)}

    # ---- e2e: public host API, numpy in / numpy out ----
    def host_step(i):
        return index.search(q_host[i % pool], a.k)

    for i in range(a.warmup):
        host_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(a.steps):
        Dh, Ih = host_step(a.warmup + i)
    torch.cuda.synchronize(dev)
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e = {"value": a.steps * a.nq / e2e_s, "unit": UNIT, "ms_per_step": e2e_s / a.steps * 1e3,
           "h2d_bytes_per_step": a.nq * a.dim * 4, "d2h_bytes_per_step": a.nq * a.k * 12,
           "api": "IndexFlatIP.search(numpy) -> numpy via evs_index_search" if world == 1
                  else ("ShardedIndexFlatIP.search(numpy) -> numpy (H2D, scan, NCCL all-gather, merge, D2H)" if a.exchange == "nccl"
                        else "ShardedIndexFlatIP.search(numpy) -> numpy via evs_index_search_exchange (H2D, scan + fused finalise + peer stores, merge, D2H)")}

    # ---- parity: answers, not speed ----
    parity = {"host_equals_device_result": bool(np.array_equal(Ih, I_last.cpu().numpy()) and np.array_equal(Dh, D_last.cpu().numpy()))}
    if not a.no_parity:
        # (1) self-match at full size: the query IS database row r (regenerated from its global id) -> r first, score ~ 1
        probe_rows = [0, a.rows // 7, a.rows // 2 + 3, (a.rows * 6) // 7, a.rows - 1]
        ok_self = True
        for r in probe_rows:
            pi = evs.IndexFlatIP(a.dim, device=local_rank)
            pi.id_base = r
            pi.add_synthetic(1, seed=0)
            qrow = pi.reconstruct_n(0, 1)
            del pi
            Dp, Ip = index.search(qrow, a.k)
            ok_self = ok_self and int(Ip[0, 0]) == r and abs(float(Dp[0, 0]) - 1.0) < 1e-5 and bool((np.diff(Dp[0].astype(np.float64)) <= 0).all())
        parity["self_match_at_full_size"] = bool(ok_self)
        parity["self_match_rows"] = probe_rows
        # (2) N > 1: rank 0 also holds the whole database on its GPU; sharded (D, I) == single-GPU (D, I), bit for bit
        if world > 1:
            nchk = min(8, pool)
            sharded = [index.search(q_host[i], a.k) for i in range(nchk)]
            same = True
            if rank == 0:
                single = evs.IndexFlatIP(a.dim, device=local_rank, storage=a.storage)
                single.reserve(a.rows)
                single.add_synthetic(a.rows, seed=0)
                for i in range(nchk):
                    Ds, Is = single.search(q_host[i], a.k)
                    same = same and bool(np.array_equal(Is, sharded[i][1]) and np.array_equal(Ds, sharded[i][0]))
                del single
                torch.cuda.empty_cache()
            t = torch.tensor([1 if same else 0], device=dev)
            dist.broadcast(t, src=0)
            parity["sharded_equals_single_gpu"] = bool(int(t.item()) == 1)
            parity["sharded_equals_single_gpu_queries"] = nchk
            if index._px is not None:
                failed, searches = index._px.status()
                parity["exchange_failures"] = int(failed)
        parity["guard"] = dict(zip(("device_reruns", "uncertified"), index.local.guard_stats()))

    # ---- roofline of the dominant kernel (the scan) ----
    rows_local = hi - lo
    esz = 2 if a.storage == "bf16" else 4
    alg_bytes = rows_local * a.dim * esz + a.nq * a.dim * 4 + a.nq * a.k * 12  # SURVEY.md 8(d), per GPU per launch
    peak, peak_src = measured_peak_gbs()
    scan_ms = scan_ms_sum / max(n_prof, 1)
    tcmin = evs.get_option("tc_min_nq")
    # database passes per search: one with the tensor-core scan, else <= 4 queries per GEMV pass at d = 512
    tc = tcmin > 0 and a.nq >= tcmin and rows_local >= 65536
    passes = (-(-a.nq // 16) if (a.storage == "f32" and a.nq <= 32 and evs.get_option("x3")) else 1) if tc else -(-a.nq // 4)
    achieved = alg_bytes * passes / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
    achieved_alg = alg_bytes / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
    fused = a.nq == 1 and evs.get_option("fuse_finalize") == 1
    roofline = {"bound": "hbm",
                "kernel": "evs::scan_direct_kernel (score + fused top-k' + the last CTA's finalise: ONE launch per search)" if fused
                          else "evs scan kernels (score + fused top-k')",
                "achieved": achieved_alg, "peak": peak, "unit": "GB/s", "frac": achieved_alg / peak,
                "traffic": ncu_traffic_per_launch(a, world),
                "peak_source": peak_src, "frac_of_nominal_8TBs": achieved_alg / 8000.0,
                "algorithmic_bytes_per_search_per_gpu": alg_bytes, "scan_ms_per_search": scan_ms,
                "scan_launches_per_search": passes, "searches_timed": n_prof,
                "hbm_read_rate_incl_repasses": achieved,
                "scan_arithmetic": scan_arithmetic(evs, a.storage, a.nq, rows_local, a.dim),
                "scan_share_of_step": scan_ms / (ms_total / a.steps) if ms_total > 0 else None,
                "duration_source": ("timed region / steps: one launch per step, CUDA events at the region's ends on the launching stream"
                                    if one_launch else "CUDA event pair recorded by libevs around every scan launch inside the timed region")}
    if events_check:
        roofline["cross_check"] = events_check

    extra = None
    if a.extra:
        extra = {}
        for nq in (1, 4, 16, 64):
            qd = torch.from_numpy(np.ascontiguousarray(np.resize(q_host.reshape(-1, a.dim), (pool, nq, a.dim)))).to(dev)
            ms, _, _ = timed_device(qd, max(10, a.steps // 4), 3)
            extra[f"nq{nq}"] = {"queries_per_s": max(10, a.steps // 4) * nq / (ms * 1e-3)}

    configs = None
    if not a.no_configs:
        del index
        torch.cuda.empty_cache()
        if world == 1:
            configs = config_legs_single(evs, torch, dev, a.k)
        else:
            configs = config_legs_sharded(evs, torch, dist, dev, world, rank, a, barrier, max_over_ranks)

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cpu = cpu_baseline(a)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": a.storage, "data": "synthetic",
            "config": {"workload": workload_name(a), "rows": a.rows, "dim": a.dim, "nq": a.nq, "k": a.k,
                       "storage": a.storage, "sharding": f"rows/{world}", "rows_per_gpu": rows_local,
                       "exchange": None if world == 1 else a.exchange,
                       "scan_variant": evs.get_option("scan_variant"), "tc_min_nq": evs.get_option("tc_min_nq"),
                       "fuse_finalize": evs.get_option("fuse_finalize"), "scan_dynamic": evs.get_option("scan_dynamic"),
                       "l2": "inputs larger than L2 (database >> 126 MB); a different query every step",
                       "build_s": round(t_build, 3)},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "parity": parity, "host_equals_device_result": parity["host_equals_device_result"],
        }
        if extra:
            line["extra"] = extra
        if configs:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main() -> int:
    a = parse_args()
    if a.impl == "reference":
        return run_reference(a)
    return run_evs(a)


if __name__ == "__main__":
    sys.exit(main())
