"""GPU (B200) parity tests proper: the CUDA path, called through the C ABI of libevs.so, against the
CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star):
  * ids and fp32 scores BIT-EXACT against the oracle's canonical ranking (CANON-32 fp64 scores,
    (score desc, id asc)) -- for every scan variant, storage precision, query batch and shard count;
  * against the faiss restatement: ids identical except exact ties and near-ties closer than the fp32
    accumulation error, scores within 1e-5 relative (tolerance written below as RTOL);
  * normalise / layout / generator kernels bit-exact against their oracle definitions, and within
    1 ulp-level tolerance of torch's own ops.
"""
import ctypes
import json
import os
import threading

import numpy as np
import pytest

import evo_ssearch_b200 as evs
import oracle
from oracle import faiss_io

pytestmark = pytest.mark.gpu

RTOL = 1e-5  # north_star: "scores within 1e-5 relative"
NEG = np.float32(-np.finfo(np.float32).max)


@pytest.fixture(autouse=True)
def _reset_options():
    yield
    for name in ("scan_variant", "tile_rows", "stages", "ctas_per_sm", "scan_clock"):
        evs.set_option(name, 0)
    evs.set_option("fuse_finalize", 1)
    evs.set_option("pool_select", 1)
    evs.set_option("scan_dynamic", 1)
    evs.set_option("scan_chunk_groups", 4)
    evs.set_option("small_max_rows", 32768)
    evs.set_option("small_fast_cap", 2048)
    evs.set_option("io_threads", 0)


def _index(xb, storage="f32", variant=0):
    evs.set_option("scan_variant", variant)
    idx = evs.IndexFlatIP(xb.shape[1], storage=storage)
    idx.add(xb)
    return idx


def _assert_canon(idx, xq, xb, k):
    D, I = idx.search(xq, k)
    Dr, Ir = oracle.canon_search(xq, xb, k)
    assert D.dtype == np.float32 and I.dtype == np.int64 and D.shape == (xq.shape[0], k)
    assert np.array_equal(I, Ir), f"ids differ: {np.argwhere(I != Ir)[:5]}"
    assert np.array_equal(D, Dr), "scores differ from the canonical fp32-rounded fp64 scores"
    return D, I


def _assert_faiss_near_tie_aware(D, I, xq, xb, k):
    """ids equal to the faiss restatement except (near-)ties; scores within RTOL."""
    Df, If = oracle.faiss_seq_search(xq, xb, k)
    valid = If >= 0
    assert np.array_equal(valid, I >= 0)
    assert np.allclose(D[valid], Df[valid], rtol=RTOL, atol=1e-7)
    eps = xb.shape[1] * 2.0 ** -24  # fp32 accumulation bound for unit-norm inputs (SURVEY.md 8c)
    for q in range(xq.shape[0]):
        for r in np.nonzero(I[q] != If[q])[0]:
            a, b = I[q, r], If[q, r]
            sa = oracle.dot_canon32(xb[a], xq[q])
            sb = oracle.dot_canon32(xb[b], xq[q])
            assert abs(sa - sb) <= eps, f"query {q} rank {r}: ids {a} vs {b} differ by {abs(sa - sb)}"


# ------------------------------------------------------------------------------------------------
def test_hand_cases(golden_dir):
    with open(os.path.join(golden_dir, "hand_cases.json")) as f:
        cases = json.load(f)
    for variant in (1, 2):
        for c in cases:
            xb = np.array(c["xb"], np.float32)
            xq = np.array(c["xq"], np.float32)
            idx = _index(xb, variant=variant)
            D, I = idx.search(xq, c["k"])
            assert I.tolist() == c["canon_I"], (c["name"], variant)
            assert np.array_equal(D, np.array(c["canon_D"], np.float32)), (c["name"], variant)


def test_c1_golden_config(golden_dir):
    """BASELINE config 1: 10k x 512, 1 query, k = 12, against the committed golden vectors."""
    with open(os.path.join(golden_dir, "c1_10k_512.json")) as f:
        g = json.load(f)
    xb = oracle.synth_fill(g["n"], g["d"], g["seed_xb"])
    xq = oracle.synth_fill(1, g["d"], g["seed_xq"])
    for variant in (1, 2):
        for storage in ("f32", "bf16"):
            idx = _index(xb, storage, variant)
            D, I = idx.search(xq, g["k"])
            assert I.tolist() == g["canon_I"], (variant, storage)
            assert [float(v).hex() for v in D[0]] == g["canon_D_f32_hex"], (variant, storage)
            assert I.tolist() == g["faiss_I"]
            Df = np.array([float.fromhex(h) for h in g["faiss_D_f32_hex"]], np.float32)
            assert np.allclose(D[0], Df, rtol=RTOL, atol=0)


@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("storage", ["f32", "bf16"])
@pytest.mark.parametrize("d", [512, 768])
def test_sweep_app_dims(variant, storage, d):
    n = 20011  # not a multiple of any tile
    xb = oracle.synth_fill(n, d, 100 + d)
    xq = oracle.synth_fill(17, d, 200 + d)
    idx = _index(xb, storage, variant)
    for nq, k in ((1, 48), (2, 12), (3, 3), (4, 48), (5, 1), (16, 48), (17, 30)):
        D, I = _assert_canon(idx, xq[:nq], xb, k)
        if storage == "f32" and nq <= 4:
            _assert_faiss_near_tie_aware(D, I, xq[:nq], xb, k)
    m = idx.last_margins(17)
    assert (m > (1e-5 if storage == "f32" else 1e-3)).all(), m.min()  # candidates cover the scan's error band


@pytest.mark.parametrize("d", [1, 45, 100, 128, 256, 384, 1024])
def test_other_dims(d):
    rng = np.random.default_rng(d)
    xb = rng.standard_normal((3001, d)).astype(np.float32)
    xq = rng.standard_normal((5, d)).astype(np.float32)
    for variant in (1, 2):
        for storage in ("f32", "bf16") if d >= 128 else ("f32",):
            idx = _index(xb, storage, variant)
            _assert_canon(idx, xq, xb, 48)
            _assert_canon(idx, xq[:1], xb, 100)


def test_small_and_edge_sizes():
    d = 512
    xq = oracle.synth_fill(3, d, 7)
    for n in (1, 2, 15, 16, 17, 47, 48, 49, 63, 64, 65, 129, 1000):
        xb = oracle.synth_fill(n, d, 1000 + n)
        for variant in (1, 2):
            idx = _index(xb, "f32", variant)
            for k in (1, 12, 48, 112):
                D, I = _assert_canon(idx, xq, xb, k)
                if k > n:
                    assert (I[:, n:] == -1).all() and (D[:, n:] == NEG).all()


def test_empty_index_and_argument_errors():
    idx = evs.IndexFlatIP(512)
    assert idx.ntotal == 0 and idx.is_trained and idx.d == 512
    D, I = idx.search(np.zeros((2, 512), np.float32), 5)
    assert (I == -1).all() and (D == NEG).all()  # faiss: all padding on an empty index
    D0, I0 = idx.search(np.zeros((0, 512), np.float32), 5)
    assert D0.shape == (0, 5) and I0.shape == (0, 5)
    with pytest.raises(AssertionError):
        idx.search(np.zeros((1, 256), np.float32), 5)  # faiss wrapper: assert d == self.d
    with pytest.raises(AssertionError):
        idx.search(np.zeros((1, 512), np.float32), 0)  # assert k > 0
    with pytest.raises(AssertionError):
        idx.add(np.zeros((3, 100), np.float32))
    with pytest.raises(evs.EvsError) as e:
        idx.search(np.zeros((1, 512), np.float32), 113)
    assert e.value.code == -7  # EVS_ELIMIT
    idx.add(np.zeros((0, 512), np.float32))
    assert idx.ntotal == 0


def test_exact_ties_and_duplicates():
    d = 512
    base = oracle.synth_fill(300, d, 5)
    xb = np.concatenate([base, base[:100], base[50:150], base])  # every row occurs 2-3 times
    xq = oracle.synth_fill(4, d, 6)
    for variant in (1, 2):
        for storage in ("f32", "bf16"):
            idx = _index(xb, storage, variant)
            for k in (1, 7, 48, 100):
                _assert_canon(idx, xq, xb, k)
    # all rows identical: canonical order is the k lowest ids
    same = np.repeat(base[:1], 5000, axis=0)
    D, I = _index(same).search(xq[:1], 48)
    assert I[0].tolist() == list(range(48)) and (D[0] == D[0, 0]).all()


def test_zero_and_nan_rows():
    d = 512
    xb = oracle.synth_fill(500, d, 8)
    xb[3] = 0.0
    xb[10] = np.nan  # what a normalised zero embedding looks like (oldapp.py:35 has no epsilon)
    xq = oracle.synth_fill(1, d, 9)
    D, I = _index(xb).search(xq, 48)
    assert 10 not in I[0]  # a NaN score never enters (faiss: heap_top < NaN is false)
    ok = np.ones(500, bool)
    ok[10] = False
    Dr, Ir = oracle.canon_search(xq, xb[ok], 48)
    remap = np.nonzero(ok)[0]
    assert np.array_equal(I[0], remap[Ir[0]]) and np.array_equal(D, Dr)


def test_incremental_add_and_reconstruct():
    d = 768
    xb = oracle.synth_fill(5000, d, 31)
    idx = evs.IndexFlatIP(d, storage="bf16")
    for lo, hi in ((0, 1), (1, 1000), (1000, 1003), (1003, 5000)):  # forces regrowth copies
        idx.add(xb[lo:hi])
    assert idx.ntotal == 5000
    assert np.array_equal(idx.reconstruct_n(0, 5000), xb)
    assert np.array_equal(idx.reconstruct(1234), xb[1234])
    _assert_canon(idx, oracle.synth_fill(2, d, 32), xb, 48)
    idx.reset()
    assert idx.ntotal == 0


def test_fp16_query_view_like_the_app():
    """oldapp.py:52/2005: on CUDA the query is an fp16 vector reshaped to (1, d); faiss casts to fp32."""
    d = 512
    xb = oracle.synth_fill(4000, d, 41)
    q16 = oracle.synth_fill(1, d, 42).astype(np.float16).reshape(-1)
    idx = _index(xb)
    D, I = idx.search(q16.reshape(1, -1), 12)
    Dr, Ir = oracle.canon_search(q16.astype(np.float32).reshape(1, -1), xb, 12)
    assert np.array_equal(I, Ir) and np.array_equal(D, Dr)


def test_device_tensor_api_matches_host_api():
    import torch
    d = 512
    xb = oracle.synth_fill(30000, d, 51)
    xq = oracle.synth_fill(6, d, 52)
    host = _index(xb)
    dev = evs.IndexFlatIP(d)
    dev.add(torch.from_numpy(xb).cuda())
    Dh, Ih = host.search(xq, 48)
    Dt, It = dev.search(torch.from_numpy(xq).cuda(), 48)
    assert Dt.is_cuda and It.dtype == torch.int64
    assert np.array_equal(Dt.cpu().numpy(), Dh) and np.array_equal(It.cpu().numpy(), Ih)
    # half-precision encoder output is widened exactly (oldapp.py:86 astype('float32'))
    xh = torch.from_numpy(xb[:1000]).cuda().half()
    h = evs.IndexFlatIP(d)
    h.add(xh)
    assert np.array_equal(h.reconstruct_n(0, 1000), xh.float().cpu().numpy())


def test_partials_and_merge_equal_single_index():
    """Row sharding emulated on one GPU: G shards -> partials -> merge kernel == one index, bit for bit."""
    import torch
    d, n, k = 512, 9001, 48
    xb = oracle.synth_fill(n, d, 61)
    xb[n - 1] = xb[0]  # exact tie across shards
    xq = oracle.synth_fill(5, d, 62)
    single = _index(xb)
    Ds, Is = single.search(xq, k)
    xq_t = torch.from_numpy(xq).cuda()
    for G in (1, 2, 3, 8):
        S, I = [], []
        for g in range(G):
            lo, hi = evs.shard_bounds(n, G, g)
            sh = evs.IndexFlatIP(d)
            sh.id_base = lo
            sh.add(xb[lo:hi])
            s, i = sh.search_partial(xq_t, k)
            S.append(s)
            I.append(i)
        D, Ifin = evs.merge_partials(torch.stack(S), torch.stack(I), k)
        assert np.array_equal(Ifin.cpu().numpy(), Is) and np.array_equal(D.cpu().numpy(), Ds), G
    # shards with fewer than k rows, and empty shards (more ranks than rows)
    tiny = xb[:5]
    Dt, It = _index(tiny).search(xq, 12)
    S, I = [], []
    for g in range(8):
        lo, hi = evs.shard_bounds(5, 8, g)
        sh = evs.IndexFlatIP(d)
        sh.id_base = lo
        if hi > lo:
            sh.add(tiny[lo:hi])
        s, i = sh.search_partial(xq_t, 12)
        S.append(s)
        I.append(i)
    D, Ifin = evs.merge_partials(torch.stack(S), torch.stack(I), 12)
    assert np.array_equal(Ifin.cpu().numpy(), It) and np.array_equal(D.cpu().numpy(), Dt)


def test_peer_exchange_single_rank_equals_search():
    """evs_exchange_* with world = 1 (the slots live on this GPU): the fused finalise -> slot -> flag ->
    merge path, the publish path (tensor-core scan, empty shard), slot-generation reuse and the limits.
    The cross-GPU case runs under torchrun in scripts/check_sharded.py (tests/test_gpu_sharded.py)."""
    import torch
    d, n, k = 512, 70_001, 48
    xb = oracle.synth_fill(n, d, 71)
    xq = oracle.synth_fill(300, d, 72)
    idx = _index(xb)
    idx.id_base = 1000
    px = evs.PeerExchange(0, 0, 1, max_nq=300, max_k=48)
    assert len(px.handle()) == 64
    xq_t = torch.from_numpy(xq).cuda()
    evs.set_option("tc_min_nq", 0)  # GEMV scan: the finalise kernel writes the slots itself
    try:
        for nq, kk in ((1, 48), (3, 12), (1, 48), (300, 48), (2, 1)):  # 300 > one finalise launch (256 queries)
            Dr, Ir = idx.search(xq[:nq], kk)
            D, I = idx.search_exchange(px, xq_t[:nq], kk)
            assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(D.cpu().numpy(), Dr), (nq, kk)
        evs.set_option("tc_min_nq", 2)  # tensor-core scan: partial staged locally, then published
        Dr, Ir = idx.search(xq[:40], 48)
        D, I = idx.search_exchange(px, xq_t[:40], 48)
        assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(D.cpu().numpy(), Dr)
        Dr, Ir = idx.search(xq[:16], 48)  # small tensor-core batch (on-chip heaps): finalise writes the slots itself
        D, I = idx.search_exchange(px, xq_t[:16], 48)
        assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(D.cpu().numpy(), Dr)
        for nq, kk in ((1, 48), (16, 12), (40, 48)):  # host entry point: staging and the one sync inside the library
            Dr, Ir = idx.search(xq[:nq], kk)
            Dh, Ih = idx.search_exchange_host(px, xq[:nq], kk)
            assert Dh.dtype == np.float32 and Ih.dtype == np.int64
            assert np.array_equal(Ih, Ir) and np.array_equal(Dh, Dr), (nq, kk)
    finally:
        evs.set_option("tc_min_nq", 2)
    empty = evs.IndexFlatIP(d)
    D, I = empty.search_exchange(px, xq_t[:2], 5)
    assert (I.cpu().numpy() == -1).all() and (D.cpu().numpy() == np.finfo(np.float32).min).all()
    timed_out, searches = px.status()
    assert not timed_out and searches == 11
    with pytest.raises(evs.EvsError):
        idx.search_exchange(px, torch.from_numpy(oracle.synth_fill(301, d, 1)).cuda(), 48)  # beyond max_nq
    px2 = evs.PeerExchange(0, 0, 2, max_nq=4, max_k=48)  # world 2, never connected
    with pytest.raises(evs.EvsError):
        idx.search_exchange(px2, xq_t[:1], 48)


def test_single_query_search_is_one_launch_whatever_the_scan_options():
    """What the app issues (oldapp.py:2005): one query.  The GEMV scan's last CTA finalises, so the whole search is ONE
    kernel launch; dealing the rows statically or dynamically, fused or not, f32 or bf16 rows gives the same bits."""
    d, n, k = 512, 300_007, 48
    q = oracle.synth_fill(3, d, 7)
    for storage in ("f32", "bf16"):
        idx = evs.IndexFlatIP(d, storage=storage)
        idx.add_synthetic(n, seed=11)
        xb = idx.reconstruct_n(0, n)
        Dr, Ir = oracle.canon_search(q, xb, k)
        for fuse, pool, dyn, chunk in ((1, 1, 0, 2), (1, 1, 1, 4), (1, 1, 1, 1), (1, 0, 2, 2), (1, 0, 2, 1), (1, 0, 2, 7), (1, 0, 0, 2), (0, 0, 0, 2)):
            evs.set_option("fuse_finalize", fuse)
            evs.set_option("pool_select", pool)  # 1: survivor pool under a global threshold (the default); 0: per-CTA lists
            evs.set_option("scan_dynamic", dyn)
            evs.set_option("scan_chunk_groups", chunk)
            for qi in range(3):
                l0 = evs.kernel_launches()
                D, I = idx.search(q[qi:qi + 1], k)
                assert evs.kernel_launches() - l0 == (1 if fuse else 2), (storage, fuse, pool, dyn, chunk)
                assert np.array_equal(I, Ir[qi:qi + 1]) and np.array_equal(D, Dr[qi:qi + 1]), (storage, fuse, pool, dyn, chunk, qi)
        evs.set_option("pool_select", 1)
        # per-CTA scan clocks (diagnostics): one record per CTA, ends after starts
        evs.set_option("fuse_finalize", 1)
        evs.set_option("scan_clock", 1)
        idx.search(q[:1], k)
        clk = idx.scan_clocks()
        evs.set_option("scan_clock", 0)
        assert clk.shape[0] >= 148 and (clk[:, 1] >= clk[:, 0]).all()


@pytest.mark.parametrize("storage", ["f32", "bf16"])
def test_pool_selection_does_not_depend_on_the_data(storage):
    """The single-query search keeps its candidates in one survivor pool under a global running threshold (scan_pool_kernel).
    Worst cases for it: rows in ASCENDING score order (every row beats everything before it: every warp keeps re-filling
    its buffer and the pool ends up holding the warps' whole buffers, far more than the last CTA holds in shared memory at a
    time, so its streaming bitonic rounds run); all high rows in ONE slot of the 64 slot maxima (rows = 0 mod 64: the
    global threshold stays low); descending order; fewer rows than slots; k' = 128 (the per-CTA-list path); consecutive
    searches (the last CTA must leave the pool zeroed).  Always the oracle's bits, and the same as the list-based paths."""
    d, k = 512, 48
    rng = np.random.default_rng(17)
    q = oracle.synth_fill(2, d, 7)
    for n in (200_003, 40_000, 63, 1):
        xb = oracle.synth_fill(n, d, 21)
        order = np.argsort(xb @ q[0])
        cases = {"ascending": xb[order], "descending": xb[order[::-1]]}
        if n > 1000:
            hot = xb.copy()  # the 500 best rows of query 0 moved to rows that are multiples of 64
            best = order[-500:]
            dst = np.arange(500) * 64
            tmp = hot[dst].copy()
            hot[dst] = xb[best]
            hot[best] = tmp
            cases["one hot slot"] = hot
        for name, x in cases.items():
            x = np.ascontiguousarray(x)
            idx = evs.IndexFlatIP(d, storage=storage)
            idx.add(x)
            for kk in (k, 1, 100):
                Dr, Ir = oracle.canon_search(q, x, kk)
                for rep in range(2):  # pool left clean by the previous search
                    for qi in range(2):
                        D, I = idx.search(q[qi:qi + 1], kk)
                        assert np.array_equal(I, Ir[qi:qi + 1]) and np.array_equal(D, Dr[qi:qi + 1]), (n, name, kk, rep, qi)
                evs.set_option("pool_select", 0)
                D0, I0 = idx.search(q[:1], kk)
                evs.set_option("pool_select", 1)
                assert np.array_equal(I0, Ir[:1]) and np.array_equal(D0, Dr[:1]), (n, name, kk)
            m = idx.last_margins(1)
            assert m[0] >= 0 or n <= 100


@pytest.mark.parametrize("storage", ["f32", "bf16"])
def test_small_shard_kernel_equals_the_oracle_and_the_pool_kernel(storage):
    """Shards of up to 32 768 rows -- the application's indexes (BASELINE config 1: 10k rows, oldapp.py:2005) -- take
    scan_small_kernel: every row's key stored by row, the threshold from 128 chunk maxima, the last CTA's keys in
    registers.  Its worst cases: more keys above the threshold than the survivor buffer holds (rows in score order, every
    row the same vector: exact ties; `small_fast_cap` 1 drives the general rounds on ordinary data too), fewer rows than
    chunks, a row count just past one register batch (10 240) and at the routing limit.  Always one launch, the oracle's
    bits, the pool kernel's bits, and a pool left clean for the next search whichever kernel runs it."""
    import torch
    d = 512
    q = oracle.synth_fill(3, d, 7)
    for n in (1, 5, 64, 129, 1000, 10_000, 10_241, 20_000, 32_768, 32_769):
        xb = oracle.synth_fill(n, d, 21)
        order = np.argsort(xb @ q[0])
        cases = {"random": xb}
        if n in (129, 10_000, 20_000):
            cases["ascending"] = xb[order]
            cases["descending"] = xb[order[::-1]]
            cases["all rows equal"] = np.repeat(xb[:1], n, axis=0)
            blocks = xb.copy()  # long runs of identical high rows: thousands of exact ties above any chunk threshold
            blocks[: n // 2] = xb[order[-1]]
            cases["half the rows tied at the top"] = blocks
        for name, x in cases.items():
            x = np.ascontiguousarray(x)
            idx = evs.IndexFlatIP(d, storage=storage)
            idx.add(x)
            for kk in (12, 48, 1):
                Dr, Ir = oracle.canon_search(q, x, kk)
                for cap in (2048, 1):
                    evs.set_option("small_fast_cap", cap)
                    for rep in range(2):
                        for qi in range(3):
                            l0 = evs.kernel_launches()
                            D, I = idx.search(q[qi:qi + 1], kk)
                            assert evs.kernel_launches() - l0 == 1
                            assert np.array_equal(I, Ir[qi:qi + 1]) and np.array_equal(D, Dr[qi:qi + 1]), (n, name, kk, cap, rep, qi)
                evs.set_option("small_fast_cap", 2048)
                evs.set_option("small_max_rows", 0)  # the pool kernel on the same handle, then the small kernel again
                D0, I0 = idx.search(q[:1], kk)
                evs.set_option("small_max_rows", 32768)
                D1, I1 = idx.search(q[:1], kk)
                assert np.array_equal(I0, Ir[:1]) and np.array_equal(D0, Dr[:1]), (n, name, kk)
                assert np.array_equal(I1, Ir[:1]) and np.array_equal(D1, Dr[:1]), (n, name, kk)
                # a numpy query travels in the kernel's parameter block; a CUDA tensor is read where it lies
                Dt, It = idx.search(torch.from_numpy(q[1:2]).cuda(), kk)
                assert np.array_equal(It.cpu().numpy(), Ir[1:2]) and np.array_equal(Dt.cpu().numpy(), Dr[1:2]), (n, name, kk)
    # NaN scores never enter (key 0), zero rows tie at 0: the contract of test_zero_and_nan_rows at 3000 rows
    x = oracle.synth_fill(3000, d, 5)
    x[7] = np.nan
    x[100:2000] = 0.0
    idx = evs.IndexFlatIP(d, storage=storage)
    idx.add(x)
    ok = np.ones(3000, bool)
    ok[7] = False
    remap = np.nonzero(ok)[0]
    Dr, Ir = oracle.canon_search(q, x[ok], 48)
    for qi in range(3):
        D, I = idx.search(q[qi:qi + 1], 48)
        assert np.array_equal(I[0], remap[Ir[qi]]) and np.array_equal(D[0], Dr[qi])


def test_back_to_back_device_searches_overlap_safely():
    """Consecutive searches enqueued on one stream without any host synchronisation: every kernel is launched with
    programmatic stream serialisation (the next search's CTAs become resident while the previous one drains and wait for
    it before they read or write anything shared: lists, ticket, chunk counter).  200 single-query searches and 60 small
    batches, all checked afterwards."""
    import torch
    d, n, k = 512, 200_003, 48
    idx = evs.IndexFlatIP(d)
    idx.add_synthetic(n, seed=13)
    xb = idx.reconstruct_n(0, n)
    q = oracle.synth_fill(40, d, 14)
    qt = torch.from_numpy(q).cuda()
    Dr, Ir = oracle.canon_search(q, xb, k)
    outs = [idx.search(qt[i % 40:i % 40 + 1], k) for i in range(200)]
    outs16 = [idx.search(qt[(i % 3) * 8:(i % 3) * 8 + 16], k) for i in range(60)]
    torch.cuda.synchronize()
    for i, (D, I) in enumerate(outs):
        j = i % 40
        assert np.array_equal(I.cpu().numpy(), Ir[j:j + 1]) and np.array_equal(D.cpu().numpy(), Dr[j:j + 1]), i
    for i, (D, I) in enumerate(outs16):
        j = (i % 3) * 8
        assert np.array_equal(I.cpu().numpy(), Ir[j:j + 16]) and np.array_equal(D.cpu().numpy(), Dr[j:j + 16]), i


def test_read_rows_is_the_shard_loader(tmp_path):
    """evs_index_read_rows reads only rows [lo, hi) of index.faiss: G shard handles loaded that way answer exactly like
    the whole file loaded on one GPU (partials + merge), ids are global, and the header-only query agrees."""
    import torch
    from evo_ssearch_b200.index import index_file_info, read_index_rows
    d, n, k = 512, 70_003, 48
    xb = oracle.synth_fill(n, d, 41)
    xq = oracle.synth_fill(5, d, 42)
    whole = _index(xb)
    path = str(tmp_path / "index.faiss")
    evs.write_index(whole, path)
    assert index_file_info(path) == (d, n)
    Ds, Is = whole.search(xq, k)
    xq_t = torch.from_numpy(xq).cuda()
    for G in (1, 3):
        S, I = [], []
        for g in range(G):
            lo, hi = evs.shard_bounds(n, G, g)
            sh, n_file = read_index_rows(path, lo, hi)
            assert n_file == n and sh.ntotal == hi - lo and sh.id_base == lo
            assert np.array_equal(sh.reconstruct_n(0, min(7, hi - lo)), xb[lo:lo + min(7, hi - lo)])
            s, i = sh.search_partial(xq_t, k)
            S.append(s)
            I.append(i)
        D, Ifin = evs.merge_partials(torch.stack(S), torch.stack(I), k)
        assert np.array_equal(Ifin.cpu().numpy(), Is) and np.array_equal(D.cpu().numpy(), Ds), G
    # every 64 MiB chunk is read by several threads over disjoint slices (option io_threads; 0 = one per hardware thread, at most
    # 16): whatever the split, the rows are the file's, and a file written again from the loaded index has the same bytes
    for threads in (1, 5, 16, 0):
        evs.set_option("io_threads", threads)
        again = evs.read_index(path)
        assert again.ntotal == n and np.array_equal(again.reconstruct_n(0, n), xb), threads
        lo, hi = 12_345, 60_001
        part, _ = read_index_rows(path, lo, hi)
        assert np.array_equal(part.reconstruct_n(0, hi - lo), xb[lo:hi]), threads
    evs.set_option("io_threads", 0)
    path2 = str(tmp_path / "index2.faiss")
    evs.write_index(again, path2)
    with open(path, "rb") as f1, open(path2, "rb") as f2:
        assert f1.read() == f2.read()
    empty, _ = read_index_rows(path, n, n)
    assert empty.ntotal == 0 and empty.id_base == n
    with pytest.raises(evs.EvsError):
        read_index_rows(path, 10, 5)


def test_set_storage_derives_and_drops_the_bf16_scan_copy():
    d, n, k = 512, 100_000, 48
    idx = evs.IndexFlatIP(d)
    idx.add_synthetic(n, seed=21)
    xb = idx.reconstruct_n(0, n)
    q = oracle.synth_fill(200, d, 22)
    Dr, Ir = oracle.canon_search(q[:8], xb, k)
    ref = evs.IndexFlatIP(d, storage="bf16")
    ref.add(xb)
    idx.set_storage("bf16")
    assert idx.storage == "bf16"
    for nq in (1, 8, 200):
        D, I = idx.search(q[:nq], k)
        D2, I2 = ref.search(q[:nq], k)
        assert np.array_equal(I, I2) and np.array_equal(D, D2), nq
        assert np.array_equal(I[:min(nq, 8)], Ir[:min(nq, 8)])
    idx.add(xb[:1000])  # the derived copy follows later adds
    assert idx.search(q[:3], k)[1].shape == (3, k)
    idx.set_storage("f32")
    assert idx.storage == "f32"
    D, I = idx.search(q[:8], k)
    Dr2, Ir2 = oracle.canon_search(q[:8], np.concatenate([xb, xb[:1000]]), k)
    assert np.array_equal(I, Ir2) and np.array_equal(D, Dr2)


def test_concurrent_search_threads():
    """The Flask dev server is threaded (oldapp.py:2258): concurrent searches on one handle."""
    d = 512
    xb = oracle.synth_fill(50000, d, 71)
    idx = _index(xb)
    qs = [oracle.synth_fill(1, d, 100 + t) for t in range(8)]
    want = [oracle.canon_search(q, xb, 48) for q in qs]
    errs = []

    def work(t):
        for _ in range(20):
            D, I = idx.search(qs[t], 48)
            if not (np.array_equal(I, want[t][1]) and np.array_equal(D, want[t][0])):
                errs.append(t)

    th = [threading.Thread(target=work, args=(t,)) for t in range(8)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs


# ------------------------------------------------------------------------------------------------
# kernels (1) of north_star: normalise and the bf16 layout kernel; the synthetic generator
# ------------------------------------------------------------------------------------------------
def test_normalize_bitexact_vs_oracle_and_close_to_torch():
    import torch
    rng = np.random.default_rng(81)
    for d in (512, 768, 45, 1):
        x = (rng.standard_normal((1000, d)) * rng.uniform(0.01, 50.0, (1000, 1))).astype(np.float32)
        want = oracle.l2_normalize(x)
        got = x.copy()
        evs.normalize_L2(got)  # host entry point (faiss.normalize_L2 signature)
        assert np.array_equal(got, want), d
        t = torch.from_numpy(x).cuda()
        ref = t / t.norm(dim=-1, keepdim=True)  # the reference's expression (oldapp.py:35)
        evs.normalize_L2(t)
        assert np.array_equal(t.cpu().numpy(), want)
        assert torch.allclose(t, ref, rtol=3e-7, atol=0)  # fp32: within 2 ulp of torch's own reduction order
    # encoder dtypes on CUDA (clip.load gives fp16): same expression evaluated in that dtype
    for dt, tol in ((torch.float16, 2e-3), (torch.bfloat16, 1.6e-2)):
        t = torch.from_numpy(rng.standard_normal((257, 512)).astype(np.float32)).cuda().to(dt)
        ref = t / t.norm(dim=-1, keepdim=True)
        evs.normalize_L2(t)
        assert torch.allclose(t.float(), ref.float(), rtol=tol, atol=tol * 1e-2)
        assert torch.allclose(t.float().norm(dim=-1), torch.ones(257, device="cuda"), atol=tol)
    z = np.zeros((2, 8), np.float32)
    evs.normalize_L2(z)
    assert np.isnan(z).all()  # no epsilon
    # The tuned fp32 kernel (rows of 128 .. 1024 values) divides with a shared reciprocal + two FMA correction steps and
    # falls back to IEEE division for rows outside [2^-60, 2^60]: bit-identical to the oracle's division either way --
    # many random mantissas, odd row counts (the kernel takes rows in pairs), signed zeros, huge / tiny / subnormal /
    # inf / NaN elements, zero rows.
    for d in (128, 256, 384, 512, 640, 768, 1024):
        n = 4001
        x = (rng.standard_normal((n, d)) * np.exp2(rng.integers(-40, 40, (n, 1)))).astype(np.float32)
        x[rng.random((n, d)) < 0.02] = 0.0
        x[rng.random((n, d)) < 0.01] = -0.0
        x[7] *= np.float32(2.0 ** 70)          # row beyond the fast range
        x[8] *= np.float32(2.0 ** -75)
        x[9, ::5] = np.float32(1e-41)          # subnormal elements
        x[10, 3] = np.float32(3e38)            # the sum of squares overflows fp32 but not fp64
        x[11, 0] = np.inf
        x[12, 1] = np.nan
        x[13] = 0.0
        x[14, 5] = np.float32(1e-30)           # one tiny element in an ordinary row
        with np.errstate(all="ignore"):
            want = oracle.l2_normalize(x)
        t = torch.from_numpy(x).cuda()
        evs.normalize_L2(t)
        got = t.cpu().numpy()
        assert np.array_equal(got.view(np.uint32)[~np.isnan(want)], want.view(np.uint32)[~np.isnan(want)]), d
        assert np.array_equal(np.isnan(got), np.isnan(want)), d


def test_bf16_layout_kernel_is_rne():
    import torch
    from evo_ssearch_b200 import _lib
    rng = np.random.default_rng(82)
    for count in (8 * 1000, 8 * 1000 + 5, 3):
        x = torch.from_numpy(rng.standard_normal(count).astype(np.float32)).cuda()
        out = torch.empty(count, dtype=torch.bfloat16, device="cuda")
        _lib.check(_lib.lib().evs_f32_to_bf16_dev(0, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                                  count, None))
        torch.cuda.synchronize()
        assert torch.equal(out, x.to(torch.bfloat16))


def test_synthetic_generator_bitexact():
    for d, n in ((512, 3000), (768, 100), (45, 77)):
        idx = evs.IndexFlatIP(d)
        idx.id_base = 12345
        idx.add_synthetic(n, seed=3)
        assert np.array_equal(idx.reconstruct_n(0, n), oracle.synth_fill(n, d, 3, row_base=12345))
        idx.add_synthetic(10, seed=3, normalize=False)  # continues the global row counter
        assert np.array_equal(idx.reconstruct_n(n, 10), oracle.synth_fill(10, d, 3, row_base=12345 + n, normalize=False))


# ------------------------------------------------------------------------------------------------
# .clip_index/index.faiss
# ------------------------------------------------------------------------------------------------
def test_index_file_bytes_and_roundtrip(golden_dir, tmp_path):
    fixture = os.path.join(golden_dir, "index_flat_3x4.faiss")
    idx = evs.read_index(fixture)
    assert (idx.d, idx.ntotal) == (4, 3)
    out = tmp_path / "index.faiss"
    evs.write_index(idx, str(out))
    assert out.read_bytes() == open(fixture, "rb").read()  # byte-exact
    xb = oracle.synth_fill(70001, 512, 91)  # payload larger than one 64 MiB staging chunk
    a = _index(xb)
    evs.write_index(a, str(out))
    assert out.stat().st_size == 45 + 4 * xb.size
    assert out.read_bytes() == faiss_io.pack_index_flat(xb)
    b = evs.read_index(str(out), storage="bf16")
    assert b.ntotal == 70001 and np.array_equal(b.reconstruct_n(0, 10), xb[:10])
    xq = oracle.synth_fill(2, 512, 92)
    _assert_canon(b, xq, xb, 48)
    with pytest.raises(evs.EvsError):
        evs.read_index(str(tmp_path / "nope.faiss"))


def test_bench_dump_is_the_last_timed_search(tmp_path):
    """`bench.py --dump-outputs DIR`: --steps searches are timed (one launch each for a single query), and DIR holds the (D, I)
    of the last one -- query (warmup + steps - 1) mod 64 of the seed-1 pool against the seed-0 database -- in the oracle's bits."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n, steps, warmup = 70_000, 5, 2
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--rows", str(n), "--steps", str(steps), "--warmup", str(warmup),
           "--no-configs", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == steps and line["gpu_launches"] == steps
    q = oracle.synth_fill(64, 512, seed=1)[(warmup + steps - 1) % 64][None]
    Dr, Ir = oracle.canon_search(q, oracle.synth_fill(n, 512, seed=0), 48)
    D, I = np.load(tmp_path / "D.npy"), np.load(tmp_path / "I.npy")
    assert D.dtype == np.float32 and I.dtype == np.float64
    assert np.array_equal(D, Dr) and np.array_equal(I, Ir)


# ------------------------------------------------------------------------------------------------
# full BASELINE sizes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("storage", ["f32", "bf16"])
def test_config2_1m_x_512_exact(storage):
    """BASELINE config 2: 1M x 512, k = 48, query batches 1 and 16 -- bit-exact against the oracle."""
    n, d, k = 1_000_000, 512, 48
    idx = evs.IndexFlatIP(d, storage=storage)
    idx.add_synthetic(n, seed=0)
    xb = oracle.synth_fill(n, d, 0)
    assert np.array_equal(idx.reconstruct_n(n - 1000, 1000), xb[-1000:])
    xq = oracle.synth_fill(16, d, 1)
    for variant in (1, 2):
        evs.set_option("scan_variant", variant)
        D1, I1 = _assert_canon(idx, xq[:1], xb, k)
        D16, I16 = _assert_canon(idx, xq, xb, k)
        assert np.array_equal(I16[0], I1[0])  # batch-size invariance
    if storage == "f32":
        _assert_faiss_near_tie_aware(D16, I16, xq, xb, k)
        assert (idx.last_margins(16) > 1e-5).all()


def test_1m_rows_against_torch_fp32_matmul_topk():
    """An independent implementation at a size the CPU oracle does not reach in seconds: torch's fp32 matmul on the
    GPU (TF32 off) + topk over 1M x 512, 64 queries.  Ids equal except pairs closer than the fp32 accumulation
    error, scores within 1e-5 relative (the north_star's tolerance); every routing (GEMV, on-chip heaps,
    thresholds + gather) gives the same bits."""
    import torch
    n, d, k, nq = 1_000_000, 512, 48, 64
    idx = evs.IndexFlatIP(d)
    idx.add_synthetic(n, seed=0)
    xq = oracle.synth_fill(nq, d, 1)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        xb_t = torch.empty((n, d), dtype=torch.float32, device="cuda")
        for c0 in range(0, n, 250_000):
            xb_t[c0:c0 + 250_000] = torch.from_numpy(idx.reconstruct_n(c0, 250_000)).cuda()
        S = torch.from_numpy(xq).cuda() @ xb_t.T
        Dt, It = torch.topk(S, k, dim=1)
        Dt, It = Dt.cpu().numpy(), It.cpu().numpy()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    results = []
    for lo, hi in ((0, 1), (1, 17), (17, 64)):  # 1 query (GEMV), 16 (on-chip heaps), 47 (thresholds + gather)
        D, I = idx.search(xq[lo:hi], k)
        results.append((D, I))
        assert np.allclose(D, Dt[lo:hi], rtol=RTOL, atol=1e-7)
        eps = d * 2.0 ** -24
        for q in range(hi - lo):
            for r in np.nonzero(I[q] != It[lo + q])[0]:
                a, b = int(I[q, r]), int(It[lo + q, r])
                sa = oracle.dot_canon32(idx.reconstruct(a), xq[lo + q])
                sb = oracle.dot_canon32(idx.reconstruct(b), xq[lo + q])
                assert abs(sa - sb) <= eps, (lo + q, r, a, b, sa, sb)
        assert (I == It[lo:hi]).mean() > 0.98
    Dall, Iall = idx.search(xq, k)  # one batch of 64: same bits as the three routings above
    assert np.array_equal(Iall, np.concatenate([r[1] for r in results]))
    assert np.array_equal(Dall, np.concatenate([r[0] for r in results]))


def test_metric_size_10m_x_512_properties():
    """10M x 512 (the metric's size): planted neighbours must come back exactly, in order, and the
    result must not depend on scan variant, storage precision or sharding."""
    import torch
    n_blocks, block, d, k = 10, 1_000_000, 512, 48
    q = oracle.synth_fill(1, d, 1)
    # 48 planted rows r_j = a_j q + sqrt(1 - a_j^2) u_j (u_j orthogonal to q): score ~ a_j >> any random score
    rng = np.random.default_rng(7)
    u = rng.standard_normal((k, d))
    u -= (u @ q[0].astype(np.float64))[:, None] * q[0]
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    a = 0.95 - 0.01 * np.arange(k)
    planted = (a[:, None] * q[0] + np.sqrt(1 - a[:, None] ** 2) * u).astype(np.float32)
    results = {}
    for storage in ("f32", "bf16"):
        idx = evs.IndexFlatIP(d, storage=storage)
        idx.reserve(n_blocks * block + k)
        want_ids = []
        for b in range(n_blocks):
            idx.add_synthetic(block, seed=0)
            sl = slice(b * 5, min(k, b * 5 + 5))
            if planted[sl].shape[0]:
                want_ids += list(range(idx.ntotal, idx.ntotal + planted[sl].shape[0]))
                idx.add(planted[sl])
        assert idx.ntotal == n_blocks * block + k
        for variant in (1, 2):
            evs.set_option("scan_variant", variant)
            D, I = idx.search(q, k)
            assert I[0].tolist() == want_ids
            want_scores = np.array([oracle.dot_canon32(planted[j], q[0]) for j in range(k)]).astype(np.float32)
            assert np.array_equal(D[0], want_scores)
            results[(storage, variant)] = (D, I)
        # below the planted rows: top-96 minus the planted = true top-48 of the random rows; check invariance
        D2, I2 = idx.search(q, 96)
        results[(storage, "k96")] = (D2, I2)
        assert (np.diff(D2[0].astype(np.float64)) <= 0).all()
        # the same query inside batches that take the tensor-core scans (one-CTA kernel, CTA-pair kernel): identical
        # answer for it, and no query of the batch may have needed the GEMV re-run (large shards pass ~9000
        # candidates per query through the gather: it must hold them)
        fb0 = evs.get_option("tc_fallbacks")
        qb = np.concatenate([q, oracle.synth_fill(299, d, 5)])
        for nqb in (16, 300):
            Db, Ib = idx.search(qb[:nqb], k)
            assert np.array_equal(Ib[:1], results[(storage, 1)][1]) and np.array_equal(Db[:1], results[(storage, 1)][0]), nqb
            assert (np.diff(Db.astype(np.float64), axis=1) <= 0).all() and (Ib >= 0).all()
        assert evs.get_option("tc_fallbacks") == fb0
        if storage == "f32":
            # sharded: 4 shards on this one GPU -> partials -> merge == unsharded
            xq_t = torch.from_numpy(q).cuda()
            rows = idx.ntotal
            S, Is = [], []
            for g in range(4):
                lo, hi = evs.shard_bounds(rows, 4, g)
                sh = evs.IndexFlatIP(d)
                sh.id_base = lo
                t = torch.empty((hi - lo, d), dtype=torch.float32, device="cuda")
                for c0 in range(lo, hi, 500_000):
                    c1 = min(hi, c0 + 500_000)
                    t[c0 - lo:c1 - lo] = torch.from_numpy(idx.reconstruct_n(c0, c1 - c0)).cuda()
                sh.add(t)
                del t
                s, i = sh.search_partial(xq_t, 96)
                S.append(s)
                Is.append(i)
                del sh
            Dm, Im = evs.merge_partials(torch.stack(S), torch.stack(Is), 96)
            assert np.array_equal(Im.cpu().numpy(), I2) and np.array_equal(Dm.cpu().numpy(), D2)
        del idx
    assert np.array_equal(results[("f32", "k96")][1], results[("bf16", "k96")][1])
    assert np.array_equal(results[("f32", "k96")][0], results[("bf16", "k96")][0])
