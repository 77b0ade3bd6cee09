"""The int8 copy's re-score window C (evs_scan.cuh, the last CTA of scan_pool_kernel<int8_t>): up to POOL_CMAX = 1024
candidates are re-scored in one pass and ranked from those scores; larger windows walk the pool in rounds of a running
exact top k.  Every case is checked bit for bit against the oracle and the fp32 scan, and `last_candidates` shows which of
the two paths it took."""
import numpy as np
import pytest

import evo_ssearch_b200 as evs
import oracle

pytestmark = pytest.mark.gpu
D = 512
N = 300_000
CMAX = 1024  # candidates re-scored in one pass


@pytest.fixture(autouse=True)
def _copy_path_at_every_size():
    cut = evs.get_option("shadow_min_rows")
    evs.set_option("shadow_min_rows", 0)
    yield
    evs.set_option("scan_shadow", 1)
    evs.set_option("shadow_min_rows", cut)


def unit(rng, n, d=D):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True).astype(np.float32)


def build(x, shadow=1):
    evs.set_option("scan_shadow", shadow)
    idx = evs.IndexFlatIP(x.shape[1])
    idx.add(x)
    evs.set_option("scan_shadow", 1)
    return idx


def check(idx, ref, q, x, k):
    Dr, Ir = oracle.canon_search(q, x, k)
    l0 = evs.kernel_launches()
    Dd, Id = idx.search(q, k)
    assert evs.kernel_launches() - l0 == 1
    assert np.array_equal(Id, Ir) and np.array_equal(Dd, Dr), k
    D0, I0 = ref.search(q, k)
    assert np.array_equal(Id, I0) and np.array_equal(Dd, D0), k
    assert idx.last_margins(1)[0] >= 0
    return idx.shadow_stats()[2]


def burst(m, seed):
    """N random unit rows, m of them replaced by near-copies of the query (within 1e-4 of one another): their scores
    (~1) lie far above every other row's (< 0.3), so the window C is exactly the burst for any k <= m."""
    rng = np.random.default_rng(seed)
    x = unit(rng, N)
    q = unit(rng, 1)
    x[rng.choice(N, m, replace=False)] = q[0] + rng.standard_normal((m, D)).astype(np.float32) * np.float32(1e-4 / np.sqrt(D))
    return x, q


@pytest.mark.parametrize("m", [CMAX - 1, CMAX, CMAX + 1, 3000])
def test_window_at_and_around_one_pass(m):
    x, q = burst(m, 70 + m)
    idx, ref = build(x), build(x, shadow=0)
    w0 = idx.shadow_stats()[0]
    for k in (1, 12, 48):
        assert check(idx, ref, q, x, k) == m  # > CMAX: the rounds; otherwise one pass
    assert idx.shadow_stats()[0] == w0 + 3  # every window held more than 256 candidates


def test_ties_at_rank_k():
    rng = np.random.default_rng(80)
    x = unit(rng, N)
    q = unit(rng, 1)
    order = np.argsort(x @ q[0])[::-1]
    for k in (1, 12, 48):
        y = x.copy()
        y[rng.choice(order[200:], 7, replace=False)] = y[order[k - 1]]  # 8 equal rows at rank k: the lowest ids win
        idx, ref = build(y), build(y, shadow=0)
        assert 8 <= check(idx, ref, q, y, k) <= CMAX


def test_all_rows_equal():
    rng = np.random.default_rng(81)
    x = np.repeat(unit(rng, 1), N, axis=0)
    q = unit(rng, 1)
    idx, ref = build(x), build(x, shadow=0)
    for k in (1, 12, 48):
        assert check(idx, ref, q, x, k) == N  # every row is in the window: the rounds


@pytest.mark.parametrize("m", [600, 3000])
def test_partial_and_exchange_entry_points(m):
    import torch
    x, q = burst(m, 90 + m)
    idx = build(x)
    qt = torch.from_numpy(q).cuda()
    for k in (1, 12, 48):
        Dr, Ir = oracle.canon_search(q, x, k)
        S, I = idx.search_partial(qt, k)
        torch.cuda.synchronize()
        assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(S.cpu().numpy().astype(np.float32), Dr), k
        assert idx.shadow_stats()[2] == m
        ex = evs.PeerExchange(idx.device, 0, 1, max_nq=4, max_k=48)
        ex.connect([ex.handle()])
        De, Ie = idx.search_exchange(ex, qt, k)
        torch.cuda.synchronize()
        assert np.array_equal(Ie.cpu().numpy(), Ir) and np.array_equal(De.cpu().numpy(), Dr), k
        assert idx.shadow_stats()[2] == m
