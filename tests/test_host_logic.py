"""CPU: host-side logic that needs no device -- shard layout, limit clamp, handler post-processing,
load_index failure contract, pickle compatibility of the .clip_index side files."""
import os
import pickle

import numpy as np

import evo_ssearch_b200 as evs
from evo_ssearch_b200 import lifecycle


def test_shard_bounds_cover_and_partition():
    for n in (0, 1, 7, 8, 9, 1000, 10_000_000):
        for world in (1, 2, 3, 4, 8):
            blocks = [evs.shard_bounds(n, world, r) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == n
            for (lo, hi), (lo2, _) in zip(blocks, blocks[1:]):
                assert lo <= hi == lo2
            per = -(-n // world) if n else 0
            assert all(hi - lo <= per for lo, hi in blocks)
    assert evs.shard_bounds(10, 4, 3) == (9, 10)
    assert evs.shard_bounds(3, 8, 5) == (3, 3)  # more ranks than rows: empty shards


def test_clamp_limit_matches_reference_rule():
    # oldapp.py:1985-1990: int in [MIN_RESULTS, MAX_RESULTS] else DEFAULT_RESULTS
    assert evs.clamp_limit(12) == 12 and evs.clamp_limit("24") == 24
    assert evs.clamp_limit(3) == 3 and evs.clamp_limit(48) == 48
    assert evs.clamp_limit(2) == 12 and evs.clamp_limit(49) == 12
    assert evs.clamp_limit(None) == 12 and evs.clamp_limit("abc") == 12


class _FakeIndex:
    def __init__(self, D, I):
        self.D, self.I, self.calls = D, I, []

    def search(self, x, k):
        self.calls.append((x.shape, k))
        return self.D[:, :k], self.I[:, :k]


def test_collect_filters_and_sorts_like_the_handlers():
    paths = [f"/p/{i}.jpg" for i in range(4)]
    meta = [{"path": p, "mtime": float(m), "size": 10 + i} for i, (p, m) in enumerate(zip(paths, (5, 9, 1, 7)))]
    D = np.array([[0.9, 0.8, 0.7, -3.4e38, 0.1]], np.float32)
    I = np.array([[2, 0, 3, -1, 99]], np.int64)  # -1 padding and an out-of-range id are dropped (oldapp.py:2009)
    idx = _FakeIndex(D, I)
    res = lifecycle._collect(idx, paths, meta, np.zeros(8, np.float32), 48, "similarity")
    assert idx.calls == [((1, 8), 4)]  # k = min(limit, len(paths)) (oldapp.py:2002), query reshaped to (1, d)
    assert [r["path"] for r in res] == ["/p/2.jpg", "/p/0.jpg", "/p/3.jpg"]
    assert res[0]["filename"] == "2.jpg" and abs(res[0]["similarity"] - 0.9) < 1e-6
    assert res[0]["metadata"] == {"mtime": 1.0, "size": 12}
    res_t = lifecycle._collect(_FakeIndex(D, I), paths, meta, np.zeros(8, np.float32), 48, "time")
    assert [r["path"] for r in res_t] == ["/p/3.jpg", "/p/0.jpg", "/p/2.jpg"]  # mtime desc (oldapp.py:2043-2045)
    assert lifecycle._collect(_FakeIndex(D, I), [], None, np.zeros(8, np.float32), 12, "similarity") == []


def test_load_index_failure_contract(tmp_path):
    assert evs.load_index(tmp_path) == (None, None, None)  # no .clip_index
    ci = tmp_path / ".clip_index"
    ci.mkdir()
    assert evs.load_index(tmp_path) == (None, None, None)  # no index.faiss
    (ci / "index.faiss").write_bytes(b"garbage")
    with open(ci / "paths.pkl", "wb") as f:
        pickle.dump(["a.jpg"], f)
    assert evs.load_index(tmp_path) == (None, None, None)  # corrupt file is "not indexed" (oldapp.py:134-135)


def test_side_files_are_plain_pickles(tmp_path):
    paths = ["/x/a.jpg", "/x/b.png"]
    meta = [{"path": p, "mtime": 1.5, "size": 3} for p in paths]
    with open(tmp_path / "paths.pkl", "wb") as f:
        pickle.dump(paths, f)
    with open(tmp_path / "metadata.pkl", "wb") as f:
        pickle.dump(meta, f)
    assert pickle.load(open(tmp_path / "paths.pkl", "rb")) == paths
    assert pickle.load(open(tmp_path / "metadata.pkl", "rb"))[1]["size"] == 3
    assert evs.config.INDEX_FOLDER_NAME == os.getenv("EVOSSEARCH_INDEX_FOLDER", ".clip_index")


class _NumpyIndex:
    """Host stand-in for IndexFlatIP with the methods the lifecycle functions use (no device, no search): lets the
    planning logic of create_index / update_index -- which file keeps its row, which is embedded, in what order -- run
    on CPU.  The arithmetic paths are covered by the GPU tests."""

    def __init__(self, d, device=None, storage=None):
        self.d, self.device, self.storage = d, 0, storage or "f32"
        self.rows = np.zeros((0, d), np.float32)

    @property
    def ntotal(self):
        return self.rows.shape[0]

    def add(self, x):
        self.rows = np.concatenate([self.rows, np.asarray(x, np.float32)])

    def add_rows_from(self, src, ids):
        self.rows = np.concatenate([self.rows, src.rows[np.asarray(ids, np.int64)]])


class _CountingEncoder:
    d = 8

    def __init__(self):
        self.calls = []

    def get_image_embedding(self, image_path):
        name = os.path.basename(str(image_path))
        self.calls.append(name)
        if name.startswith("broken"):
            raise OSError("cannot identify image file")
        rng = np.random.default_rng(abs(hash((name, os.path.getsize(image_path)))) % (2 ** 32))
        v = rng.standard_normal(self.d).astype(np.float32)
        return v / np.linalg.norm(v)


def test_incremental_reindex_plan_on_cpu(tmp_path, monkeypatch):
    monkeypatch.setattr(lifecycle, "IndexFlatIP", _NumpyIndex)
    store = {}
    monkeypatch.setattr(lifecycle, "write_index", lambda index, fname: store.__setitem__(fname, index) or open(fname, "wb").close())
    monkeypatch.setattr(lifecycle, "read_index", lambda fname: store[fname])
    lifecycle.evict_index()
    for i in range(10):
        (tmp_path / f"img_{i}.jpg").write_bytes(b"x" * (i + 1))
    (tmp_path / "broken.png").write_bytes(b"b")
    (tmp_path / "notes.txt").write_bytes(b"t")
    enc = _CountingEncoder()
    index, paths, meta = lifecycle.create_index(tmp_path, enc, batch_size=4)
    assert index.ntotal == len(paths) == len(meta) == 10 and len(enc.calls) == 11
    lifecycle.save_index(index, paths, meta, tmp_path)
    # unchanged folder: only the unreadable file is retried, rows and order are kept
    enc.calls.clear()
    i1, p1, m1, st = lifecycle.update_index(tmp_path, enc)
    assert enc.calls == ["broken.png"] and st == {"kept": 10, "embedded": 0, "removed": 0, "failed": 1}
    assert p1 == paths and m1 == meta and np.array_equal(i1.rows, index.rows)
    # one deleted, one changed, two new
    os.remove(tmp_path / "img_3.jpg")
    (tmp_path / "img_5.jpg").write_bytes(b"changed!")
    (tmp_path / "new_a.jpg").write_bytes(b"a")
    (tmp_path / "new_b.webp").write_bytes(b"bb")
    enc.calls.clear()
    i2, p2, m2, st = lifecycle.update_index(tmp_path, enc, batch_size=2)
    assert sorted(enc.calls) == ["broken.png", "img_5.jpg", "new_a.jpg", "new_b.webp"]
    assert st == {"kept": 8, "embedded": 3, "removed": 1, "failed": 1}
    fresh, pf, mf = lifecycle.create_index(tmp_path, _CountingEncoder())
    assert p2 == pf and m2 == mf and np.array_equal(i2.rows, fresh.rows)  # interchangeable with a full rebuild
    lifecycle.evict_index()


def test_resident_cache_is_an_lru_with_a_byte_budget(tmp_path, monkeypatch):
    """ADVICE r1: the resident cache must not grow without bound, and its signature covers all three files."""
    from evo_ssearch_b200 import lifecycle

    class Fake:
        storage = "f32"

        def __init__(self, n, d=4):
            self.ntotal, self.d = n, d

    monkeypatch.setattr(lifecycle, "CACHE_BUDGET_BYTES", 16 * 100 * 2 + 8)  # room for two 100-row indexes of d = 4
    lifecycle.evict_index()
    ev0 = lifecycle.load_stats["evictions"]
    for name in ("a", "b", "c"):
        lifecycle._cache_put(name, ("sig",), Fake(100), [], None)
    assert list(lifecycle._cache) == ["b", "c"] and lifecycle.load_stats["evictions"] == ev0 + 1
    lifecycle._cache_put("b", ("sig2",), Fake(100), [], None)  # re-put moves to the recent end
    lifecycle._cache_put("d", ("sig",), Fake(100), [], None)
    assert list(lifecycle._cache) == ["b", "d"]
    lifecycle._cache_put("huge", ("sig",), Fake(10_000), [], None)  # larger than the budget: kept alone, never evicts itself
    assert list(lifecycle._cache) == ["huge"]
    lifecycle.evict_index()
    assert not lifecycle._cache
    # the signature changes when ANY of the three files changes
    ip = tmp_path / ".clip_index"
    ip.mkdir()
    (ip / "index.faiss").write_bytes(b"x")
    s0 = lifecycle._signature(ip)
    assert s0[0] is not None and s0[1] is None and s0[2] is None
    (ip / "paths.pkl").write_bytes(b"yy")
    s1 = lifecycle._signature(ip)
    assert s1 != s0 and s1[0] == s0[0]
    assert lifecycle._want_sharded(False) is False and lifecycle._want_sharded(None) is False  # no process group here


def test_bench_reference_arm_prints_the_contract_line(tmp_path):
    """`bench.py --impl reference` (the CPU arm the driver times beside the CUDA arm) on a small workload: ONE JSON line with the
    contract's keys, `impl: reference`, a cpu_baseline block describing the run and an e2e block equal to the line's value;
    `--dump-outputs` holds the last timed step's answer; ranks other than 0 print nothing and exit 0."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--rows", "20000", "--steps", "2", "--warmup", "1",
           "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env={**os.environ, "RANK": "0"})
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "20000" in d["cpu_baseline"]["sample"]
    assert d["config"]["workload"].startswith("20000x512 f32 flat-IP")
    import oracle
    q = np.roll(oracle.synth_fill(64, 512, seed=1), -2, axis=0)[:1]  # the last timed step is step 2 (after 1 warmup step): query 2
    Dr, Ir = oracle.allcores_search(q, oracle.synth_fill(20000, 512, seed=0), 48, nthreads=d["cpu_baseline"]["cores"])
    D, I = np.load(tmp_path / "D.npy"), np.load(tmp_path / "I.npy")
    assert D.dtype == np.float32 and I.dtype == np.float64
    assert np.array_equal(D, Dr) and np.array_equal(I, Ir)
    other = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env={**os.environ, "RANK": "1"})
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_selection_thresholds_never_drop_a_top_key():
    """The two threshold rules the single-query kernels rely on (evs_scan.cuh), restated in numpy on unique keys:
    * small-shard kernel: rows are partitioned into 128 chunks (warp index mod 128); T = the 64th largest chunk maximum.
      At least 64 keys are >= T, so none of the 64 best keys is below T;
    * pool kernel: 64 slot maxima, each the maximum of a subset of the keys published to slot (row mod 64); tau = the
      smallest slot maximum (0 while a slot is empty).  The maxima belong to 64 different rows, so again no top-64 key is
      below tau -- whatever subset of the keys has been published so far.
    Ordered, clustered and tiny inputs included: the bound must hold for any data, only the survivor count varies."""
    rng = np.random.default_rng(5)
    kp, chunks = 64, 128

    def check(keys, warps, rpg):
        n = keys.shape[0]
        top = np.sort(keys)[::-1][:kp]
        # small-shard rule: group g of rpg rows belongs to warp g mod warps, chunk = warp mod 128
        rows = np.arange(n)
        chunk = ((rows // rpg) % warps) % chunks
        cmax = np.zeros(chunks, dtype=keys.dtype)
        np.maximum.at(cmax, chunk, keys)
        nz = np.sort(cmax[cmax > 0])[::-1]
        T = nz[kp - 1] if nz.shape[0] >= kp else 0
        assert (top >= T).all()
        assert (keys >= T).sum() >= min(kp, n)
        # pool rule: an arbitrary subset of the keys has been published so far
        for frac in (0.02, 0.5, 1.0):
            pub = rng.random(n) < frac
            smax = np.zeros(kp, dtype=keys.dtype)
            np.maximum.at(smax, rows[pub] % kp, keys[pub])
            tau = smax.min()  # 0 while any slot is empty
            assert (top >= tau).all()

    for n in (1, 63, 64, 129, 1000, 10_000, 32_768):
        base = rng.permutation(n).astype(np.uint64) + 1  # unique, non-zero
        for keys in (base, np.sort(base), np.sort(base)[::-1].copy()):
            for warps, rpg in ((2368, 4), (8, 4), (296, 1), (1184, 2)):
                check(keys, warps, rpg)
    # all large keys inside a few chunks (rows of one warp)
    keys = rng.permutation(20_000).astype(np.uint64) + 1
    hot = ((np.arange(20_000) // 4) % 2368) % 128 < 3
    keys[hot] += 1_000_000
    check(keys, 2368, 4)
