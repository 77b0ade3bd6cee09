"""Exact batch search of the int8 copy (batches of 2..4 queries, k <= 112; evs_large_k.cu, lk_score_i8_kernel): every
row's int8 scan key, the k-th selected, every row within 2E of it re-scored exactly.  Results must be the oracle's bit for bit
for fp32 and bf16 storage, on every entry point, and coalesce_stats()[2] shows that the route ran."""
import numpy as np
import pytest
import torch

import evo_ssearch_b200 as evs
import oracle

pytestmark = pytest.mark.gpu
M = 4  # largest batch of the route: one pass of the score scan
KS = (1, 12, 48, 100, 112)


@pytest.fixture(autouse=True)
def _copy_path_at_every_size():
    cut, small = evs.get_option("shadow_min_rows"), evs.get_option("small_max_rows")
    evs.set_option("shadow_min_rows", 0)
    yield
    evs.set_option("shadow_min_rows", cut)
    evs.set_option("small_max_rows", small)


def unit(rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True).astype(np.float32)


def check_host(idx, q, x, k, passes):
    p0 = idx.coalesce_stats()[2]
    D, I = idx.search(q, k)
    Dr, Ir = oracle.canon_search(q, x, k)
    assert np.array_equal(I, Ir) and np.array_equal(D, Dr), (q.shape[0], k)
    assert idx.coalesce_stats()[2] - p0 == passes, (q.shape[0], k)
    assert (idx.last_margins(q.shape[0]) >= 0).all()
    return D, I


@pytest.mark.parametrize("storage", ["f32", "bf16"])
@pytest.mark.parametrize("d", [256, 512, 768, 1024])
def test_batches_equal_the_oracle(d, storage):
    rng = np.random.default_rng(d + (1 if storage == "bf16" else 0))
    x = unit(rng, 40_001, d)
    q = unit(rng, M, d)
    idx = evs.IndexFlatIP(d, storage=storage)
    idx.add(x)
    for nq in range(2, M + 1):
        for k in KS:
            check_host(idx, q[:nq], x, k, 1)
    p0 = idx.coalesce_stats()[2]
    idx.search(q[:1], 12)  # one query: the single-query search, not this route
    idx.search(np.concatenate([q, q[:1]]), 12)  # M + 1 queries: the tensor-core scan
    assert idx.coalesce_stats()[2] == p0


def test_near_tie_burst_beyond_one_sort():
    """5000 near-copies of the query, perturbed by about E: the window holds more than the 4096 candidates the rank kernel
    sorts at once, so its radix select runs."""
    d, n, m = 512, 60_000, 5000
    rng = np.random.default_rng(5)
    x = unit(rng, n, d)
    q = unit(rng, 3, d)
    E = 4e-4 / np.sqrt(d)  # the copy's bound on unit rows is ~1e-4 at d = 512: the burst straddles rank k within E
    rows = rng.choice(n, m, replace=False)
    x[rows] = q[0] + rng.standard_normal((m, d)).astype(np.float32) * np.float32(E)
    idx = evs.IndexFlatIP(d)
    idx.add(x)
    for k in (12, 112):
        check_host(idx, q, x, k, 1)
        assert idx.shadow_stats()[2] > 4096


@pytest.mark.parametrize("scale", [1e-3, 64.0])
def test_scaled_rows(scale):
    d = 512
    rng = np.random.default_rng(9)
    x = unit(rng, 40_000, d) * np.float32(scale) * rng.uniform(0.5, 1.0, (40_000, 1)).astype(np.float32)
    q = unit(rng, 4, d) * np.float32(3.0)
    idx = evs.IndexFlatIP(d)
    idx.add(x)
    for k in (1, 48, 112):
        check_host(idx, q, x, k, 1)


def test_k_beyond_ntotal():
    evs.set_option("small_max_rows", 0)  # a 50-row shard on the route
    d = 256
    rng = np.random.default_rng(12)
    x = unit(rng, 50, d)
    q = unit(rng, 3, d)
    for storage in ("f32", "bf16"):
        idx = evs.IndexFlatIP(d, storage=storage)
        idx.add(x)
        D, I = check_host(idx, q, x, 100, 1)
        assert (I[:, 50:] == -1).all() and (D[:, 50:] == -np.finfo(np.float32).max).all()


def test_device_and_partial_entry_points():
    d, n = 768, 80_000  # shards of 40 000 rows: above small_max_rows
    rng = np.random.default_rng(21)
    x = unit(rng, n, d)
    q = unit(rng, 4, d)
    idx = evs.IndexFlatIP(d)
    idx.add(x)
    qt = torch.from_numpy(q).cuda()
    for k in (12, 100):
        Dr, Ir = oracle.canon_search(q, x, k)
        p0 = idx.coalesce_stats()[2]
        D, I = idx.search(qt, k)
        assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(D.cpu().numpy(), Dr), k
        S, Ip = idx.search_partial(qt, k)
        assert np.array_equal(Ip.cpu().numpy(), Ir) and np.array_equal(S.cpu().numpy().astype(np.float32), Dr), k
        assert idx.coalesce_stats()[2] - p0 == 2
        # two row shards, each on the route, merged
        half = n // 2
        parts = []
        for lo, hi in ((0, half), (half, n)):
            sh = evs.IndexFlatIP(d)
            sh.add(x[lo:hi])
            sh.id_base = lo
            parts.append(sh.search_partial(qt, k))
            assert sh.coalesce_stats()[2] == 1
        Dm, Im = evs.merge_partials(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), k)
        assert np.array_equal(Im.cpu().numpy(), Ir) and np.array_equal(Dm.cpu().numpy(), Dr), k
