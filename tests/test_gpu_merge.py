"""GPU: the merge of sorted shard partials (``evs.merge_partials``) on synthetic partials, for k on both sides of
EVS_MAX_K (entries staged in shared memory up to 112, ranked in global memory above), bit for bit against a numpy sort
by (score desc, id asc)."""
import numpy as np
import pytest

import evo_ssearch_b200 as evs

pytestmark = pytest.mark.gpu

NEG64 = -np.finfo(np.float64).max
NEG32 = np.float32(-np.finfo(np.float32).max)


@pytest.fixture(autouse=True)
def _max_k():
    evs.set_option("max_k", 2048)
    yield
    evs.set_option("max_k", 112)  # process-wide: the default limit must hold for every other test


def _partials(rng, G, nq, k):
    """Sorted partials [G, nq, k] with padding tails of random length (empty parts included) and, per query, ties at
    rank k: entries of several parts share the score that ranks k-th in the union, with different ids."""
    S = np.full((G, nq, k), NEG64)
    I = np.full((G, nq, k), -1, np.int64)
    for q in range(nq):
        lens = rng.integers(0, k + 1, G)
        if q == 0:
            lens[:] = k  # every part full
        elif q == 1 and G > 1:
            lens[0] = 0  # an empty first part
        total = int(lens.sum())
        ids = rng.permutation(10 * total + 10)[:total].astype(np.int64)
        sc = np.round(rng.standard_normal(total), 2)  # coarse: ties everywhere
        sc[rng.random(total) < 0.05] = 0.0
        if total > k:  # plant ties at rank k across parts
            order = np.lexsort((ids, -sc))
            below = order[k:]
            sc[rng.choice(below, min(len(below), 2 * G), replace=False)] = sc[order[k - 1]]
        off = np.concatenate([[0], np.cumsum(lens)])
        for g in range(G):
            s, i = sc[off[g]:off[g + 1]], ids[off[g]:off[g + 1]]
            o = np.lexsort((i, -s))
            S[g, q, :lens[g]], I[g, q, :lens[g]] = s[o], i[o]
    return S, I


def _reference(S, I, k):
    G, nq, _ = S.shape
    D = np.full((nq, k), NEG32)
    Ir = np.full((nq, k), -1, np.int64)
    for q in range(nq):
        s, i = S[:, q].reshape(-1), I[:, q].reshape(-1)
        s, i = s[i >= 0], i[i >= 0]
        o = np.lexsort((i, -s))[:k]
        D[q, :o.size] = s[o].astype(np.float32)
        Ir[q, :o.size] = i[o]
    return D, Ir


def _merge(S, I, k):
    import torch
    D, Io = evs.merge_partials(torch.from_numpy(S).cuda(), torch.from_numpy(I).cuda(), k)
    torch.cuda.synchronize()
    return D.cpu().numpy(), Io.cpu().numpy()


@pytest.mark.parametrize("G,k", [(G, k) for k in (1, 12, 48, 112, 113, 2048) for G in (1, 3, 8)] + [(70, 12)])
def test_merge_matches_sort(G, k):
    rng = np.random.default_rng(1000 * G + k)
    S, I = _partials(rng, G, 5, k)
    D, Io = _merge(S, I, k)
    Dr, Ir = _reference(S, I, k)
    assert np.array_equal(Io, Ir), np.argwhere(Io != Ir)[:5]
    assert np.array_equal(D, Dr)


def test_merge_limits():
    rng = np.random.default_rng(7)
    for G, k in ((9, 113), (77, 112), (1000, 12)):  # more than 8 parts above EVS_MAX_K; nparts*k*24 > 200 KB below
        S, I = _partials(rng, G, 2, k)
        with pytest.raises(evs.EvsError) as e:
            _merge(S, I, k)
        assert e.value.code == -7, (G, k)  # EVS_ELIMIT
    S, I = _partials(rng, 76, 2, 112)  # 76 * 112 * 24 bytes: the largest staged merge
    D, Io = _merge(S, I, 112)
    Dr, Ir = _reference(S, I, 112)
    assert np.array_equal(Io, Ir) and np.array_equal(D, Dr)
