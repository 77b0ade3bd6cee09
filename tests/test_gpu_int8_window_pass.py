"""The int8 copy's window pass (evs_scan.cuh, scan_pool_kernel<int8_t>): the last CTA and the CTAs holding the tickets
just before it re-score the window W (every pool key within 2E of the k-th largest slot maximum) in slices, and the last CTA ranks the candidate
window C from W; a W of more than POOL_CMAX entries falls back to the pool read.  Every case is checked bit for bit against
the oracle and the fp32 scan, `last_candidates` against |C| recomputed here from the int8 scan keys, and the finalise
stamps (option "scan_clock") show which path ran."""
import numpy as np
import pytest

import evo_ssearch_b200 as evs
import oracle

pytestmark = pytest.mark.gpu
f32 = np.float32
QMAX = 127 * 256 + 127
CMAX = 1024  # entries of W


@pytest.fixture(autouse=True)
def _copy_path_at_every_size():
    cut, cps = evs.get_option("shadow_min_rows"), evs.get_option("ctas_per_sm")
    evs.set_option("shadow_min_rows", 0)
    yield
    evs.set_option("scan_shadow", 1)
    evs.set_option("shadow_min_rows", cut)
    evs.set_option("ctas_per_sm", cps)
    evs.set_option("scan_clock", 0)


def unit(rng, n, d):
    x = rng.standard_normal((n, d), dtype=f32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def build(x, shadow=1):
    evs.set_option("scan_shadow", shadow)
    idx = evs.IndexFlatIP(x.shape[1])
    idx.add(x)
    evs.set_option("scan_shadow", 1)
    return idx


def scan_scores(x, q, chunk=65536):
    """The int8 scan's scores s~ = fl(fl(I) fl(s_q s_r)) (DESIGN.md section 2): row codes rint(x / s_r), s_r = max|x| / 127,
    query codes rint(q / s_q), s_q = max|q| / 32639; I is exact in fp64 (|I| < 2^33)."""
    sq = f32(np.abs(q).max() / f32(QMAX))
    cq = np.clip(np.rint((q / sq).astype(f32)), -QMAX, QMAX).astype(np.float64)
    out = np.empty(len(x), f32)
    for i in range(0, len(x), chunk):
        xc = x[i:i + chunk]
        s = (np.abs(xc).max(1).astype(f32) / f32(127)).astype(f32)
        c = np.clip(np.rint((xc / s[:, None]).astype(f32)), -127, 127).astype(np.float64)
        out[i:i + chunk] = (c @ cq).astype(f32) * (sq * s).astype(f32)
    return out


def shadow_E(idx, q):
    """E of evs_scan.cuh shadow_bound_i8 from the index's e_max and norm estimate."""
    sq = f32(np.abs(q).max() / f32(QMAX))
    qh = float(sq) * np.clip(np.rint((q / sq).astype(f32)), -QMAX, QMAX).astype(np.float64)
    dq = np.sqrt(((q.astype(np.float64) - qh) ** 2).sum()) * (1 + 2.0**-20)
    qn = np.sqrt((qh**2).sum()) * (1 + 2.0**-20)
    nx = float(f32(idx.max_row_norm)) * (1 + 2.0**-7)
    em = float(f32(idx.shadow_stats()[1]))
    e = (dq * nx + qn * em + 2.0**-22 * qn * (nx + em)) * (1 + 2.0**-20) + 2.0**-117
    e32 = f32(e)
    return e32 if float(e32) >= e else np.nextafter(e32, f32(np.inf))


def window_size(s, k, E):
    """|C|: the rows whose scan score is >= fl_down(s~_(k) - 2E) (keys order by score, then by row: ties at s~_(k) all count)."""
    sk = np.partition(s, len(s) - k)[len(s) - k]
    twoE = f32(2) * E
    v = float(sk) - float(twoE)
    lo = f32(v)
    if float(lo) > v:
        lo = np.nextafter(lo, f32(-np.inf))
    return int((s >= lo).sum())


def check(idx, ref, q, x, k, s=None):
    Dr, Ir = oracle.canon_search(q, x, k)
    l0 = evs.kernel_launches()
    Dd, Id = idx.search(q, k)
    assert evs.kernel_launches() - l0 == 1
    assert np.array_equal(Id, Ir) and np.array_equal(Dd, Dr), k
    D0, I0 = ref.search(q, k)
    assert np.array_equal(Id, I0) and np.array_equal(Dd, D0), k
    assert idx.last_margins(1)[0] >= 0
    c = idx.shadow_stats()[2]
    if s is not None:
        assert c == window_size(s, k, shadow_E(idx, q[0])), k
    return c


def ranked_from_w(idx):
    """Whether the last search ranked C from W (finalise stamp 10), with |W| (0xffffffff: overflowed), the slices the
    helpers took and the pool's size."""
    idx.scan_clocks()
    fs = idx.finalize_stamps
    return int(fs[10]) != 0, int(fs[11]), int(fs[12]), int(fs[13])


@pytest.mark.parametrize("n", [262_147, 1_250_000])
@pytest.mark.parametrize("d", [256, 512, 1024])
def test_random_rows(n, d):
    rng = np.random.default_rng(n + d)
    x = unit(rng, n, d)
    idx, ref = build(x), build(x, shadow=0)
    for k in (48, 12, 1):  # (Gaussian rows at d = 512: W holds ~900-1150 keys, so either path may run)
        q = unit(rng, 1, d)
        check(idx, ref, q, x, k, scan_scores(x, q[0]))


@pytest.mark.parametrize("cps", [1, 2, 3])
def test_grid_and_helper_counts(cps):
    evs.set_option("ctas_per_sm", cps)
    rng = np.random.default_rng(100 + cps)
    x = unit(rng, 1_250_000, 256)  # |W| ~ 400-600
    idx, ref = build(x), build(x, shadow=0)
    evs.set_option("scan_clock", 1)
    for k in (48, 12):
        q = unit(rng, 1, 256)
        check(idx, ref, q, x, k, scan_scores(x, q[0]))
        w = ranked_from_w(idx)
        assert w[0], w
        if cps <= 2:  # (every CTA is resident: the helpers are waiting when the pass opens)
            assert w[2] > 0, w


def burst(n, m, d, seed):
    """n random unit rows, m of them near-copies of the query (within 1e-4 of one another): their scores (~1) lie far above
    every other row's, so W and C are exactly the burst."""
    rng = np.random.default_rng(seed)
    x = unit(rng, n, d)
    q = unit(rng, 1, d)
    x[rng.choice(n, m, replace=False)] = q[0] + rng.standard_normal((m, d)).astype(f32) * f32(1e-4 / np.sqrt(d))
    return x, q


@pytest.mark.parametrize("m", [CMAX - 1, CMAX, CMAX + 1])
def test_w_capacity_and_fallback(m):
    x, q = burst(300_000, m, 512, 200 + m)
    idx, ref = build(x), build(x, shadow=0)
    evs.set_option("scan_clock", 1)
    for k in (1, 48):
        assert check(idx, ref, q, x, k) == m
        w = ranked_from_w(idx)
        assert w[0] == (m <= CMAX), w


@pytest.mark.parametrize("streams", [1, 2])
def test_two_handles_back_to_back(streams):
    import torch
    rng = np.random.default_rng(300 + streams)
    xs = [unit(rng, 400_000, 512), unit(rng, 300_000, 512)]
    idxs = [build(x) for x in xs]
    qs = unit(rng, 16, 512)
    k = 48
    want = [[oracle.canon_search(qs[i:i + 1], x, k) for i in range(len(qs))] for x in xs]
    qt = torch.from_numpy(qs).cuda()
    sts = [torch.cuda.current_stream(), torch.cuda.Stream() if streams == 2 else torch.cuda.current_stream()]
    outs = [[None] * len(qs) for _ in xs]
    for i in range(len(qs)):
        for h in (0, 1):
            with torch.cuda.stream(sts[h]):
                outs[h][i] = idxs[h].search(qt[i:i + 1], k)
    torch.cuda.synchronize()
    for h in (0, 1):
        for i in range(len(qs)):
            D, I = (t.cpu().numpy() if hasattr(t, "cpu") else t for t in outs[h][i])
            assert np.array_equal(I, want[h][i][1]) and np.array_equal(D, want[h][i][0]), (h, i)
