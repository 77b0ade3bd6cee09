"""Merge timing, two builds side by side: the partial merge (`merge_partials`, G sorted shard partials -> top k) for
G = 8, nq in {1, 16, 4096}, k in {12, 48, 112, 2048}, and the world-1 peer-exchange single-query search (`search_exchange`,
1M x 512 fp32, k = 48), whose one launch ends with the exchange merge.  Both package trees are loaded into this one process
(each with its own libevs.so) and timed in alternation, case by case and round by round, so that the two builds see the
same card and the same neighbours.  CUDA events on the current stream.  The partials of a merge sit in L2 when they fit
(126 MB), as they do right after the all-gather that produces them.  Prints one JSON line per (case, build, round), then
one summary line per case with the median of each build, their ratio and whether the two builds' (D, I) are byte-identical.

    python scripts/merge_timing.py --trees <old tree> <new tree> [--rounds 5] [--out merge_timing.jsonl]
"""
import argparse
import hashlib
import importlib.util
import json
import os
import statistics
import subprocess
import sys

import torch


def load_tree(tree, name):
    pkg = os.path.join(os.path.abspath(tree), "evo-ssearch_b200")
    spec = importlib.util.spec_from_file_location(name, os.path.join(pkg, "__init__.py"), submodule_search_locations=[pkg])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def timed(fn, target_s=0.2):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    iters = int(min(max(target_s * 1e3 / max(e0.elapsed_time(e1), 1e-3), 3), 2000))
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def digest(*ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(t.cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def partials(G, nq, k, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    S = torch.randn(G, nq, k, dtype=torch.float64, device="cuda", generator=g).sort(dim=2, descending=True).values
    ids = torch.randperm(G * nq * k, device="cuda", generator=g).reshape(G, nq, k)
    return S.contiguous(), ids.contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs=2, required=True, metavar=("OLD", "NEW"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--G", type=int, default=8)
    ap.add_argument("--nqs", default="1,16,4096")
    ap.add_argument("--ks", default="12,48,112,2048")
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    builds = {"old": load_tree(a.trees[0], "evs_old"), "new": load_tree(a.trees[1], "evs_new")}
    for evs in builds.values():
        evs.set_option("max_k", 2048)
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    emit({"gpu": gpu_info(), "torch": torch.__version__, "trees": a.trees})
    cases = {}  # name -> {build: fn returning (D, I)}
    for nq in [int(v) for v in a.nqs.split(",")]:
        for k in [int(v) for v in a.ks.split(",")]:
            S, ids = partials(a.G, nq, k, seed=nq * 10_000 + k)
            cases[f"merge_partials G={a.G} nq={nq} k={k}"] = {
                b: (lambda evs=evs, S=S, ids=ids, k=k: evs.merge_partials(S, ids, k)) for b, evs in builds.items()}
    d = 512
    q = torch.randn(1, d, device="cuda")
    q /= q.norm()
    keep = []  # indexes and exchanges live until the end
    fns = {}
    for b, evs in builds.items():
        idx = evs.IndexFlatIP(d, storage="f32")
        idx.add_synthetic(a.rows, seed=1)
        ex = evs.PeerExchange(torch.cuda.current_device(), 0, 1, max_nq=1, max_k=48)
        ex.connect([ex.handle()])
        keep.append((idx, ex))
        fns[b] = lambda idx=idx, ex=ex: idx.search_exchange(ex, q, 48)
    cases[f"search_exchange world=1 {a.rows}x{d} f32 nq=1 k=48"] = fns

    times = {name: {b: [] for b in builds} for name in cases}
    digests = {name: {} for name in cases}
    for rnd in range(a.rounds):
        order = list(builds) if rnd % 2 == 0 else list(builds)[::-1]
        for name, per in cases.items():
            for b in order:
                ms = timed(per[b])
                times[name][b].append(ms)
                digests[name][b] = digest(*per[b]())
                emit({"case": name, "build": b, "round": rnd, "ms": round(ms, 5)})
    for name in cases:
        med = {b: statistics.median(v) for b, v in times[name].items()}
        emit({"case": name, "old_ms": round(med["old"], 5), "new_ms": round(med["new"], 5),
              "new_over_old": round(med["new"] / med["old"], 3),
              "old_spread": [round(min(times[name]["old"]), 5), round(max(times[name]["old"]), 5)],
              "new_spread": [round(min(times[name]["new"]), 5), round(max(times[name]["new"]), 5)],
              "identical": digests[name]["old"] == digests[name]["new"]})
    if out:
        out.close()


if __name__ == "__main__":
    main()
