"""Concurrent single-query searches of one index are served in groups (evs_index_search, group commit): every caller
gets the answer of the same call made alone, bit for bit; a lone caller runs exactly as before; a malformed call fails
alone; batch and large-k callers keep their own searches while groups run.  Groups form on shards with an int8 copy of at
least shadow_min_rows rows (262 144 by default)."""
import threading

import numpy as np
import pytest

import evo_ssearch_b200 as evs
import oracle

pytestmark = pytest.mark.gpu
D = 512
THREADS = 16
ROUNDS = 12


def hammer(idx, Q, ks, extra=None):
    """THREADS threads search their own queries ROUNDS times each, released together; returns {(t, r): (D, I)}."""
    res, errs = {}, []
    go = threading.Barrier(THREADS + (1 if extra else 0))

    def worker(t):
        try:
            go.wait()
            for r in range(ROUNDS):
                res[(t, r)] = idx.search(Q[t, r:r + 1], ks[t][r])
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    ths = [threading.Thread(target=worker, args=(t,)) for t in range(THREADS)]
    if extra:
        ths.append(threading.Thread(target=lambda: (go.wait(), extra())))
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    assert not errs, errs
    return res


def queries_and_ks(seed):
    rng = np.random.default_rng(seed)
    Q = oracle.synth_fill(THREADS * ROUNDS, D, seed).reshape(THREADS, ROUNDS, D)
    ks = rng.integers(3, 49, size=(THREADS, ROUNDS))
    return Q, [[int(k) for k in row] for row in ks]


@pytest.mark.parametrize("rows,storage", [(10_000, "f32"), (300_000, "f32"), (300_000, "bf16")])
def test_concurrent_equals_sequential(rows, storage):
    idx = evs.IndexFlatIP(D, storage=storage)
    idx.add_synthetic(rows, seed=rows)
    Q, ks = queries_and_ks(rows + 1)
    alone = {(t, r): idx.search(Q[t, r:r + 1], ks[t][r]) for t in range(THREADS) for r in range(ROUNDS)}
    g0 = idx.coalesce_stats()
    grouped = False
    for _ in range(3):
        res = hammer(idx, Q, ks)
        for key, (Dd, Id) in res.items():
            assert np.array_equal(Dd, alone[key][0]) and np.array_equal(Id, alone[key][1]), (rows, storage, key)
        g1 = idx.coalesce_stats()
        grouped = grouped or (g1[1] - g0[1] > g1[0] - g0[0])
    if rows >= 300_000:  # an int8 copy above shadow_min_rows: groups run as one search, those of up to 4 on the int8 route
        assert grouped and g1[2] > g0[2], (rows, storage, g0, g1)
    else:  # the small-shard kernel: callers are searched one by one (a group would be slower)
        assert g1 == g0, (rows, storage, g0, g1)
    xb = idx.reconstruct_n(0, rows) if rows <= 10_000 else None
    if xb is not None:  # the small index against the oracle too
        for t in range(0, THREADS, 5):
            Dr, Ir = oracle.canon_search(Q[t, :1], xb, ks[t][0])
            assert np.array_equal(alone[(t, 0)][1], Ir) and np.array_equal(alone[(t, 0)][0], Dr)


@pytest.mark.parametrize("rows", [10_000, 300_000])
def test_lone_caller_is_unchanged(rows):
    idx = evs.IndexFlatIP(D)
    idx.add_synthetic(rows, seed=3)
    q = oracle.synth_fill(8, D, 4)
    idx.search(q[:1], 12)
    s0 = idx.coalesce_stats()
    for i in range(8):
        l0 = evs.kernel_launches()
        idx.search(q[i:i + 1], 12 + i)
        assert evs.kernel_launches() - l0 == 1  # the fused single-query search: one launch
    assert idx.coalesce_stats() == s0


def test_malformed_call_fails_alone_and_batches_keep_their_own_search():
    rows = 300_000
    evs.set_option("max_k", 256)
    try:
        idx = evs.IndexFlatIP(D)
        idx.add_synthetic(rows, seed=7)
        xb = idx.reconstruct_n(0, rows)
        Q, ks = queries_and_ks(8)
        alone = {(t, r): idx.search(Q[t, r:r + 1], ks[t][r]) for t in range(THREADS) for r in range(ROUNDS)}
        qb = oracle.synth_fill(20, D, 9)
        Dbr, Ibr = oracle.canon_search(qb, xb, 200)
        side = {}

        def extra():
            L = evs._lib.lib()  # a single-query call without a query buffer: fails in its own thread, before any group
            side["bad"] = L.evs_index_search(idx._h, 1, None, 12, None, None)
            side["bad_msg"] = L.evs_last_error().decode()
            side["batch"] = idx.search(qb[:6], 40)      # nq > 1: its own search
            side["large_k"] = idx.search(qb[:1], 200)   # k > 112: its own search
            side["batch_large_k"] = idx.search(qb, 200)

        res = hammer(idx, Q, ks, extra)
        for key, (Dd, Id) in res.items():
            assert np.array_equal(Dd, alone[key][0]) and np.array_equal(Id, alone[key][1]), key
        assert side["bad"] == -1 and "NULL" in side["bad_msg"], side  # EVS_EINVAL
        assert np.array_equal(side["batch"][1], Ibr[:6, :40]) and np.array_equal(side["batch"][0], Dbr[:6, :40])
        assert np.array_equal(side["large_k"][1], Ibr[:1]) and np.array_equal(side["large_k"][0], Dbr[:1])
        assert np.array_equal(side["batch_large_k"][1], Ibr) and np.array_equal(side["batch_large_k"][0], Dbr)
    finally:
        evs.set_option("max_k", 112)
