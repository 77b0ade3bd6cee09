"""Single-query searches of the int8 scan copy (evs_scan.cuh: scan_pool_kernel<int8_t> under shadow_bound_i8): the
oracle's bits and the fp32 scan's bits in one launch, with candidate windows below and above one re-score round."""
import numpy as np
import pytest

import evo_ssearch_b200 as evs
import oracle
from test_gpu_shadow_scan import D, _opts, build, check, unit  # noqa: F401  (_opts: the autouse option fixture)

pytestmark = pytest.mark.gpu


def test_bench_rows_at_one_million():
    x = oracle.synth_fill(1_000_000, D, seed=0)
    q = oracle.synth_fill(3, D, seed=1)
    idx, ref = build(x), build(x, shadow=0)
    assert 0 < idx.shadow_stats()[1] < 0.02
    check(idx, q, x, ref=ref)


@pytest.mark.parametrize("m", [0, 1000])
def test_windows_below_and_above_one_round(m):
    rng = np.random.default_rng(20 + m)
    n = 300_000
    x = unit(rng, n)
    q = unit(rng, 1)
    if m:
        base = x[np.argsort(x @ q[0])[-30]]
        x[rng.choice(n, m, replace=False)] = base + rng.standard_normal((m, D)).astype(np.float32) * np.float32(1e-4 / np.sqrt(D))
    idx = build(x)
    w0 = idx.shadow_stats()[0]
    check(idx, q, x, ks=(1,) if m == 0 else (48,), ref=build(x, shadow=0))
    wide, _, last = idx.shadow_stats()
    assert (last > 256) == (m > 0) and (wide > w0) == (m > 0), (m, last)


def test_dominant_element_rows():
    rng = np.random.default_rng(21)
    n = 200_000
    x = unit(rng, n) * np.float32(1e-3)
    x[np.arange(n), rng.integers(0, D, n)] = rng.choice([-1.0, 1.0], n).astype(np.float32)
    q = unit(rng, 2)
    check(build(x), q, x, ref=build(x, shadow=0))


def test_bf16_storage_searches_the_int8_copy():
    rng = np.random.default_rng(22)
    x = unit(rng, 300_000)
    q = unit(rng, 2)
    idx = build(x, shadow=0, storage="bf16")  # bf16 storage keeps the copy whatever the option says
    assert idx.shadow_stats()[1] > 0
    check(idx, q, x, ref=build(x, shadow=0))


def test_partial_and_exchange_entry_points():
    import torch
    rng = np.random.default_rng(23)
    x = unit(rng, 300_000)
    q = unit(rng, 1)
    idx = build(x)
    Dr, Ir = oracle.canon_search(q, x, 48)
    qt = torch.from_numpy(q).cuda()
    S, I = idx.search_partial(qt, 48)
    torch.cuda.synchronize()
    assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(S.cpu().numpy().astype(np.float32), Dr)
    ex = evs.PeerExchange(idx.device, 0, 1, max_nq=4, max_k=48)
    ex.connect([ex.handle()])
    De, Ie = idx.search_exchange(ex, qt, 48)
    torch.cuda.synchronize()
    assert np.array_equal(Ie.cpu().numpy(), Ir) and np.array_equal(De.cpu().numpy(), Dr)
