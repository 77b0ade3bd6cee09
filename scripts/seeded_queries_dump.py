"""Single-query searches of seeded unit queries over a seeded synthetic index, one search at a time, with what each search
left behind: (D, I), `last_margins` and `last_candidates` (|C|).  Run it with two builds and compare the two files query
by query (`--compare A.npz B.npz`): a change to the tail of the single-query search must leave all four unchanged.

    python scripts/seeded_queries_dump.py --rows 10000000 1250000 --out this.npz
    python scripts/seeded_queries_dump.py --compare parent.npz this.npz
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def dump(rows, d, k, queries, out):
    import torch
    import evo_ssearch_b200 as evs
    res = {}
    for n in rows:
        idx = evs.IndexFlatIP(d)
        idx.add_synthetic(n, seed=5)
        q = np.random.default_rng(7).standard_normal((queries, d)).astype(np.float32)
        q /= np.linalg.norm(q, axis=1, keepdims=True)
        qt = torch.from_numpy(q).cuda()
        D, I, M, C = [], [], [], []
        for i in range(queries):
            Dd, Id = idx.search(qt[i:i + 1], k)
            torch.cuda.synchronize()
            D.append(Dd.cpu().numpy())
            I.append(Id.cpu().numpy())
            M.append(idx.last_margins(1).copy())
            C.append(idx.shadow_stats()[2])
        res.update({f"D{n}": np.concatenate(D), f"I{n}": np.concatenate(I), f"M{n}": np.concatenate(M), f"C{n}": np.asarray(C)})
        del idx
        torch.cuda.empty_cache()
    np.savez(out, **res)


def compare(a, b):
    A, B = np.load(a), np.load(b)
    ok = sorted(A.files) == sorted(B.files)
    for name in sorted(A.files):
        same = name in B.files and A[name].tobytes() == B[name].tobytes()
        print(name, "identical" if same else "DIFFERENT", A[name].shape)
        ok &= same
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[10_000_000, 1_250_000])
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--k", type=int, default=48)
    ap.add_argument("--queries", type=int, default=200)
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2)
    a = ap.parse_args()
    if a.compare:
        sys.exit(0 if compare(*a.compare) else 1)
    dump(a.rows, a.dim, a.k, a.queries, a.out)


if __name__ == "__main__":
    main()
