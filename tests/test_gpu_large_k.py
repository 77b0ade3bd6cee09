"""GPU: exact search for 112 < k <= 2048 (option ``max_k``; DESIGN.md section 2, "Large k").  Every comparison is bit for
bit against the oracle's canonical ranking."""
import os
import zlib

import numpy as np
import pytest

import evo_ssearch_b200 as evs
import oracle

pytestmark = pytest.mark.gpu

NEG = np.float32(-np.finfo(np.float32).max)


@pytest.fixture(autouse=True)
def _max_k():
    evs.set_option("max_k", 2048)
    yield
    evs.set_option("max_k", 112)  # process-wide: the default limit must hold for every other test


def _unit(rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True).astype(np.float32)


def _index(x, storage="f32"):
    idx = evs.IndexFlatIP(x.shape[1], storage=storage)
    idx.add(x)
    return idx


def _check(idx, q, x, k, tensor=False):
    if tensor:
        import torch
        D, I = idx.search(torch.from_numpy(q).cuda(), k)
        torch.cuda.synchronize()
        D, I = D.cpu().numpy(), I.cpu().numpy()
    else:
        D, I = idx.search(q, k)
    Dr, Ir = oracle.canon_search(q, x, k)
    assert np.array_equal(I, Ir), (k, np.argwhere(I != Ir)[:5])
    assert np.array_equal(D, Dr), k
    n = x.shape[0]
    if k > n:
        assert (I[:, n:] == -1).all() and (D[:, n:] == NEG).all()
    _, cands = idx.large_k_stats()
    assert cands >= min(k, n)
    return D, I


@pytest.mark.parametrize("storage", ["f32", "bf16"])
@pytest.mark.parametrize("d", [512, 768, 100])
@pytest.mark.parametrize("n", [1, 2047, 2048, 2049, 10_000])
def test_sizes(storage, d, n):
    if storage == "bf16" and d % 128:
        pytest.skip("bf16 storage keeps dimensions that are multiples of 128")
    rng = np.random.default_rng(n + d)
    x = _unit(rng, n, d)
    q = _unit(rng, 17, d)
    idx = _index(x, storage)
    for k in (113, 500, 1024, 2048):
        _check(idx, q[:3], x, k)
    _check(idx, q, x, 2048)  # 17 queries: passes of max_queries_per_pass(d) queries
    _check(idx, q[:1], x, 500, tensor=True)


@pytest.mark.parametrize("storage", ["f32", "bf16"])
def test_300k_rows(storage):
    rng = np.random.default_rng(5)
    x = _unit(rng, 300_000, 512)
    q = _unit(rng, 17, 512)
    idx = _index(x, storage)
    for nq, k in ((1, 113), (1, 2048), (3, 1024), (17, 2048)):
        _check(idx, q[:nq], x, k)
    _check(idx, q[:3], x, 2048, tensor=True)
    s, _ = idx.large_k_stats()
    assert s >= 5


def _adversarial(kind, rng, n=20_000, d=512, k=2048):
    x = _unit(rng, n, d)
    q = _unit(rng, 1, d)
    if kind == "all equal":  # |C| = n > one shared-memory sort: the radix-select rank path
        x[:] = x[0]
    elif kind == "half tied at rank k":
        s = oracle.canon_scores(q[0], x)
        order = np.argsort(-s)
        x[order[k // 2:k // 2 + n // 2]] = x[order[k]]
    elif kind == "ascending":
        t = np.linspace(-1, 1, n, dtype=np.float32)[:, None]
        x = (t * q + (1 - np.abs(t)) * 1e-3 * x).astype(np.float32)
    elif kind == "near-duplicate burst":
        s = oracle.canon_scores(q[0], x)
        base = x[np.argsort(-s)[k]]
        burst = rng.choice(n, 3000, replace=False)
        x[burst] = base + rng.standard_normal((3000, d)).astype(np.float32) * np.float32(1e-7)
    elif kind == "scaled 1e3":
        x *= np.float32(1e3)
    elif kind == "scaled 1e-3":
        x *= np.float32(1e-3)
    elif kind == "inf element":  # every row is a candidate; the row with +inf ranks first
        x[17, 3] = np.inf
        q[0, 3] = abs(q[0, 3]) + np.float32(0.1)
    elif kind == "subnormal element":
        x[17, 3] = np.float32(1e-40)
    return x, q


@pytest.mark.parametrize("storage", ["f32", "bf16"])
@pytest.mark.parametrize("kind", ["all equal", "half tied at rank k", "ascending", "near-duplicate burst", "scaled 1e3",
                                  "scaled 1e-3", "inf element", "subnormal element"])
def test_adversarial(kind, storage):
    rng = np.random.default_rng(11)
    x, q = _adversarial(kind, rng)
    idx = _index(x, storage)
    for k in (113, 2048):
        _check(idx, q, x, k)
    if kind in ("all equal", "inf element", "subnormal element"):
        assert idx.large_k_stats()[1] == x.shape[0]  # every row was re-scored


def test_nan_rows_never_enter():
    rng = np.random.default_rng(3)
    x = _unit(rng, 5000, 512)
    x[10] = np.nan
    q = _unit(rng, 1, 512)
    D, I = _index(x).search(q, 2048)
    assert 10 not in I[0]
    ok = np.ones(5000, bool)
    ok[10] = False
    Dr, Ir = oracle.canon_search(q, x[ok], 2048)
    assert np.array_equal(I[0], np.nonzero(ok)[0][Ir[0]]) and np.array_equal(D, Dr)


@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_emulated_shards_merge_bit_for_bit(G):
    import torch
    rng = np.random.default_rng(G)
    n, d, k = 30_011, 512, 2048
    x = _unit(rng, n, d)
    q = _unit(rng, 3, d)
    D0, I0 = _index(x).search(q, k)
    qt = torch.from_numpy(q).cuda()
    bounds = [(n * g // G, n * (g + 1) // G) for g in range(G)]
    parts = []
    for lo, hi in bounds:
        sub = _index(x[lo:hi])
        sub.id_base = lo
        parts.append(sub.search_partial(qt, k))
    S = torch.stack([p[0] for p in parts])
    Iid = torch.stack([p[1] for p in parts])
    D, I = evs.merge_partials(S, Iid, k)
    torch.cuda.synchronize()
    assert np.array_equal(I.cpu().numpy(), I0) and np.array_equal(D.cpu().numpy(), D0)


def test_peer_exchange_world_one():
    import torch
    rng = np.random.default_rng(8)
    x = _unit(rng, 20_000, 512)
    q = _unit(rng, 3, 512)
    idx = _index(x)
    ex = evs.PeerExchange(idx.device, 0, 1, max_nq=4, max_k=2048)
    ex.connect([ex.handle()])
    for nq, k in ((1, 2048), (3, 500)):
        D0, I0 = idx.search(q[:nq], k)
        De, Ie = idx.search_exchange(ex, torch.from_numpy(q[:nq]).cuda(), k)
        torch.cuda.synchronize()
        assert np.array_equal(Ie.cpu().numpy(), I0) and np.array_equal(De.cpu().numpy(), D0)
        Dh, Ih = idx.search_exchange_host(ex, q[:nq], k)
        assert np.array_equal(Ih, I0) and np.array_equal(Dh, D0)
    assert ex.status() == (0, 4)
    with pytest.raises(evs.EvsError):
        evs.PeerExchange(idx.device, 0, 1, max_nq=4, max_k=2049)


class _Encoder:
    """Deterministic unit-norm embeddings of file names and texts in place of CLIP."""

    def _vec(self, key):
        return oracle.synth_fill(1, 512, seed=zlib.crc32(key.encode()))[0]

    def get_image_embedding(self, image_path):
        return self._vec("img:" + os.path.basename(str(image_path)))

    def get_text_embedding(self, text):
        return self._vec("txt:" + text)


def test_search_text_with_a_raised_result_limit(tmp_path, monkeypatch):
    enc = _Encoder()
    for i in range(700):
        (tmp_path / f"img_{i:04d}.jpg").write_bytes(b"x")
    index, paths, meta = evs.create_index(tmp_path, enc)
    evs.save_index(index, paths, meta, tmp_path)
    monkeypatch.setattr(evs.config, "MAX_RESULTS", 500)
    res = evs.search_text(tmp_path, "a cat", enc, limit=300)
    xb = np.stack([enc.get_image_embedding(p) for p in paths]).astype(np.float32)
    Dr, Ir = oracle.canon_search(enc.get_text_embedding("a cat").reshape(1, -1).astype(np.float32), xb, 300)
    assert [r["path"] for r in res] == [paths[i] for i in Ir[0]]
    assert [r["similarity"] for r in res] == [float(v) for v in Dr[0]]
    evs.evict_index()


def test_routing_of_small_k_is_unchanged():
    rng = np.random.default_rng(2)
    x = _unit(rng, 300_007, 512)
    q = _unit(rng, 3, 512)
    idx = _index(x)

    def run():
        out = []
        for nq in (1, 3):
            for k in (1, 48, 112):
                before = evs.kernel_launches()
                D, I = idx.search(q[:nq], k)
                out.append((D, I, evs.kernel_launches() - before))
        return out

    wide = run()
    evs.set_option("max_k", 112)
    default = run()
    for (D1, I1, l1), (D2, I2, l2) in zip(wide, default):
        assert np.array_equal(D1, D2) and np.array_equal(I1, I2) and l1 == l2
    with pytest.raises(evs.EvsError) as e:
        idx.search(q[:1], 113)
    assert e.value.code == -7  # EVS_ELIMIT
    for mk in (112, 2048):
        evs.set_option("max_k", mk)
        with pytest.raises(evs.EvsError) as e:
            idx.search(q[:1], 2049)
        assert e.value.code == -7


def test_time_scan_and_margins():
    import torch
    rng = np.random.default_rng(4)
    x = _unit(rng, 100_000, 512)
    q = _unit(rng, 4, 512)
    idx = _index(x)
    assert idx.time_scan(torch.from_numpy(q).cuda(), 2048, iters=3) > 0
    _check(idx, q, x, 2048)  # the timing runs left nothing behind
    m = idx.last_margins(4)
    assert (m > 0).all(), m
