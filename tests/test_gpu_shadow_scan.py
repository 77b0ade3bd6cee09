"""Single-query searches of the bf16 scan copy (option "scan_shadow", evs_scan.cuh: scan_pool_kernel under the rounding
bound): always the oracle's bits and the fp32 scan's bits, one launch, and a copy that stays in step with the rows."""
import os

import numpy as np
import pytest

import evo_ssearch_b200 as evs
import oracle

pytestmark = pytest.mark.gpu
D = 512


@pytest.fixture(autouse=True)
def _opts():
    cut = evs.get_option("shadow_min_rows")
    evs.set_option("shadow_min_rows", 0)  # the copy's path at every size above small_max_rows
    yield
    evs.set_option("scan_shadow", 1)
    evs.set_option("shadow_min_rows", cut)


def unit(rng, n, d=D):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True).astype(np.float32)


def build(x, shadow=1, storage="f32"):
    evs.set_option("scan_shadow", shadow)
    idx = evs.IndexFlatIP(x.shape[1], storage=storage)
    idx.add(x)
    evs.set_option("scan_shadow", 1)
    return idx


def check(idx, q, x, ks=(1, 12, 48), ref=None):
    for k in ks:
        Dr, Ir = oracle.canon_search(q, x, k)
        for qi in range(q.shape[0]):
            l0 = evs.kernel_launches()
            Dd, Id = idx.search(q[qi:qi + 1], k)
            assert evs.kernel_launches() - l0 == 1
            assert np.array_equal(Id, Ir[qi:qi + 1]) and np.array_equal(Dd, Dr[qi:qi + 1]), (k, qi)
            if ref is not None:
                D0, I0 = ref.search(q[qi:qi + 1], k)
                assert np.array_equal(Id, I0) and np.array_equal(Dd, D0)
            assert idx.last_margins(1)[0] >= 0


@pytest.mark.parametrize("n", [300_000, 1_000_000])
def test_random_rows_equal_the_oracle_and_the_fp32_scan(n):
    rng = np.random.default_rng(n)
    x = unit(rng, n)
    q = unit(rng, 3)
    idx, ref = build(x), build(x, shadow=0)
    assert idx.shadow_stats()[1] > 0 and ref.shadow_stats()[1] == -1
    assert idx.shadow_stats()[2] == 0  # nothing searched yet
    check(idx, q, x, ref=ref)


def test_ordered_and_one_hot_slot_rows():
    rng = np.random.default_rng(3)
    n = 300_000
    x = unit(rng, n)
    q = unit(rng, 1)
    order = np.argsort(x @ q[0])
    hot = x.copy()
    dst = np.arange(500) * 64
    tmp = hot[dst].copy()
    hot[dst] = x[order[-500:]]
    hot[order[-500:]] = tmp
    for name, xx in {"ascending": x[order], "descending": x[order[::-1]], "one hot slot": hot}.items():
        xx = np.ascontiguousarray(xx)
        check(build(xx), q, xx, ref=build(xx, shadow=0))


@pytest.mark.parametrize("m", [300, 3000])
def test_near_tie_bursts(m):
    """m rows within 1e-4 of one another around rank k; more than 256 of them take the re-score rounds (counted)."""
    rng = np.random.default_rng(m)
    n = 300_000
    x = unit(rng, n)
    q = unit(rng, 1)
    base = x[np.argsort(x @ q[0])[-40]]
    x[rng.choice(n, m, replace=False)] = base + rng.standard_normal((m, D)).astype(np.float32) * np.float32(1e-4 / np.sqrt(D))
    idx = build(x)
    w0 = idx.shadow_stats()[0]
    check(idx, q, x, ks=(12, 48), ref=build(x, shadow=0))
    assert (idx.shadow_stats()[0] > w0) == (m > 256)


@pytest.mark.parametrize("scale", [1e-3, 1e3])
def test_large_and_small_norms(scale):
    rng = np.random.default_rng(7)
    x = unit(rng, 200_000) * np.float32(scale) * rng.uniform(0.5, 2, (200_000, 1)).astype(np.float32)
    q = unit(rng, 2) * np.float32(scale)
    check(build(x), q, x, ref=build(x, shadow=0))


def test_device_partial_and_exchange_entry_points():
    import torch
    rng = np.random.default_rng(1)
    x = unit(rng, 300_000)
    q = unit(rng, 1)
    idx = build(x)
    Dr, Ir = oracle.canon_search(q, x, 48)
    qt = torch.from_numpy(q).cuda()
    Dt, It = idx.search(qt, 48)
    torch.cuda.synchronize()
    assert np.array_equal(It.cpu().numpy(), Ir) and np.array_equal(Dt.cpu().numpy(), Dr)
    S, I = idx.search_partial(qt, 48)
    torch.cuda.synchronize()
    assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(S.cpu().numpy().astype(np.float32), Dr)
    ex = evs.PeerExchange(idx.device, 0, 1, max_nq=4, max_k=48)
    ex.connect([ex.handle()])
    De, Ie = idx.search_exchange_host(ex, q, 48)
    assert np.array_equal(Ie, Ir) and np.array_equal(De, Dr)
    De, Ie = idx.search_exchange(ex, qt, 48)
    torch.cuda.synchronize()
    assert np.array_equal(Ie.cpu().numpy(), Ir) and np.array_equal(De.cpu().numpy(), Dr)


def test_copy_stays_coherent(tmp_path):
    rng = np.random.default_rng(2)
    x = unit(rng, 400_000)
    q = unit(rng, 2)
    idx = evs.IndexFlatIP(D)
    idx.reserve(50_000)
    idx.add(x[:100_000])
    idx.add(x[100_000:250_000])  # reserve growth
    evs.set_option("scan_shadow", 0)
    idx.add(x[250_000:300_000])  # drops the copy
    assert idx.shadow_stats()[1] == -1
    check(idx, q, x[:300_000], ks=(48,))
    evs.set_option("scan_shadow", 1)
    idx.add(x[300_000:])  # builds it again over every row
    assert idx.shadow_stats()[1] > 0
    check(idx, q, x, ks=(48,))
    evs.set_option("scan_shadow", 0)  # toggled between searches: the fp32 scan, same bits
    check(idx, q, x, ks=(48,))
    evs.set_option("scan_shadow", 1)
    for st in ("bf16", "f32", "bf16", "f32"):
        idx.set_storage(st)
        check(idx, q, x, ks=(48,))
    other = evs.IndexFlatIP(D)
    rows = rng.permutation(x.shape[0])[:200_000]
    other.add_rows_from(idx, rows)
    check(other, q, x[rows], ks=(48,))
    path = os.path.join(str(tmp_path), "index.faiss")
    evs.write_index(idx, path)
    back = evs.read_index(path)
    check(back, q, x, ks=(48,))
    idx.reset()
    idx.add(x[:60_000])
    check(idx, q, x[:60_000], ks=(48,))


@pytest.mark.parametrize("kind", ["subnormal", "bf16 overflow"])
def test_special_rows_scan_the_fp32_rows(kind):
    rng = np.random.default_rng(4)
    x = unit(rng, 200_000)
    q = unit(rng, 1)
    if kind == "subnormal":
        x[17, 3] = np.float32(1e-40)
    else:
        x[17] = 0.0
        x[17, 3] = np.float32(3.3955e38)  # rounds to a bf16 infinity
        q[0, 3] = 0.0
    idx = build(x)
    check(idx, q, x, ks=(48,), ref=build(x, shadow=0))
