"""CPU restatement of the exact single-query search from the int8 scan copy (evs_scan.cuh: scan_pool_kernel,
shadow_bound_i8; DESIGN.md section 2).  Row x: scale s_r = max|x_i| / 127 (fp32), codes c = rint(x / s_r) in [-127, 127].
Query q: s_q = max|q_i| / 32639 (fp32), codes c_q = rint(q / s_q), split c_q = 256 h + l into signed bytes.  The scan
score is s~ = fl(fl(I) * fl(s_q s_r)) with I = 256 sum(h c) + sum(l c) exact, and

    |q.x - s~| <= |q - q^| max|x| + |q^| e_max + 2^-22 |q^| (max|x| + e_max) + 2^-117 = E   (inflated, rounded up)

These tests check the bound on adversarial rows and queries and replay rules 1 and 2 with it."""
import numpy as np
import pytest

from test_shadow_bound import replay, unit

D = 512
QMAX = 127 * 256 + 127
f32 = np.float32


def quantise_rows(x):
    amax = np.abs(x).max(1).astype(f32)
    s = (amax / f32(127)).astype(f32)
    with np.errstate(divide="ignore", invalid="ignore"):
        c = np.where(s[:, None] > 0, np.rint((x / s[:, None]).astype(f32)), 0)
    return s, np.clip(c, -127, 127).astype(np.int8)


def quantise_query(q):
    sq = f32(np.abs(q).max() / f32(QMAX))
    c = np.clip(np.rint((q / sq).astype(f32)), -QMAX, QMAX).astype(np.int64) if sq > 0 else np.zeros(q.shape, np.int64)
    lo = ((c + 128) & 255) - 128
    hi = (c - lo) >> 8
    assert np.abs(hi).max(initial=0) <= 127 and np.abs(lo).max(initial=0) <= 128
    return sq, c, hi, lo


def scan_scores(q, s, c):
    """The kernel's arithmetic: integer dot products of the split query codes (int32 at d <= 512), one rounding to fp32,
    times the fp32 product of the scales."""
    sq, cq, hi, lo = quantise_query(q)
    ci = c.astype(np.int64)
    I = 256 * (ci @ hi) + ci @ lo
    assert np.abs(I).max() < 2**31 and np.array_equal(I, ci @ cq)
    return (I.astype(f32) * (f32(sq) * s).astype(f32)).astype(f32)


def bound(q, x, s, c):
    xh = s.astype(np.float64)[:, None] * c.astype(np.float64)
    emax = np.sqrt(((x.astype(np.float64) - xh) ** 2).sum(1)).max()
    emax = float(np.nextafter(f32(emax), f32(np.inf)))  # rounded up to fp32, as the add stores it
    max_norm = float(f32(np.sqrt((x.astype(np.float64) ** 2).sum(1)).max()) * f32(1.000001))
    sq, cq, _, _ = quantise_query(q)
    qh = float(sq) * cq.astype(np.float64)
    dq = np.sqrt(((q.astype(np.float64) - qh) ** 2).sum()) * (1 + 2.0**-20)
    qn = np.sqrt((qh**2).sum()) * (1 + 2.0**-20)
    nx = max_norm * (1 + 2.0**-7)
    e = (dq * nx + qn * emax + 2.0**-22 * qn * (nx + emax)) * (1 + 2.0**-20) + 2.0**-117
    return float(np.nextafter(f32(e), f32(np.inf)))


def rows_cases():
    rng = np.random.default_rng(5)
    x = unit(rng, 4000)
    scaled = x * f32(10.0) ** rng.uniform(-3, 3, (4000, 1)).astype(f32)
    # one dominant element: the scale is set by it, every other element rounds to code 0
    dominant = x * f32(1e-3)
    dominant[np.arange(4000), rng.integers(0, D, 4000)] = rng.choice([-1.0, 1.0], 4000)
    # every element half a quantisation step from its code, with the query's signs: the per-element errors add up
    q = unit(rng, 1)[0]
    half = np.where(rng.random((1000, D)) < 0.5, 0.5, -0.5) + rng.integers(-126, 126, (1000, D))
    half = (half * np.sign(q)).astype(f32)
    half[:, 0] = f32(127.0)  # the scale: exactly 1
    return {"random": x, "scaled": scaled, "dominant": dominant, "half step": half}, q, rng


@pytest.mark.parametrize("case", ["random", "scaled", "dominant", "half step"])
def test_scan_of_the_int8_rows_stays_within_the_bound(case):
    cases, q0, rng = rows_cases()
    x = cases[case]
    s, c = quantise_rows(x)
    # the last query: one element at the top of the 16-bit code range, the others spread over it (|I| near 2^31)
    edge = np.full(D, 0.999, f32) * np.sign(q0).astype(f32)
    for q in (q0, unit(rng, 1)[0] * f32(37.0), unit(rng, 1)[0] * f32(1e-3), edge):
        E = bound(q, x, s, c)
        true = x.astype(np.float64) @ q.astype(np.float64)
        err = np.abs(true - scan_scores(q, s, c).astype(np.float64))
        assert err.max() <= E, (case, err.max(), E)
        assert err.max() > 0.0


def test_query_codes_at_the_int32_edge():
    """|c_q| = 32639 and |c_r| = 127 in every element: |I| = 512 * 32639 * 127 just below 2^31."""
    x = np.full((2, D), 1.0, f32)
    x[1] = -1.0
    s, c = quantise_rows(x)
    q = np.full(D, 0.25, f32)
    sc = scan_scores(q, s, c)
    assert abs(512 * QMAX * 127) < 2**31
    true = x.astype(np.float64) @ q.astype(np.float64)
    assert np.abs(true - sc).max() <= bound(q, x, s, c)


def test_bound_on_gaussian_unit_rows_is_about_a_hundredth():
    rng = np.random.default_rng(9)
    x = unit(rng, 20000)
    s, c = quantise_rows(x)
    e = np.sqrt(((x.astype(np.float64) - s[:, None].astype(np.float64) * c) ** 2).sum(1))
    assert 6e-3 < e.mean() < 9e-3 and e.max() < 1.4e-2
    assert 8e-3 < bound(unit(rng, 1)[0], x, s, c) < 1.5e-2


@pytest.mark.parametrize("k", [1, 12, 48])
@pytest.mark.parametrize("layout", ["random", "ascending", "descending", "near-tie burst", "wide burst"])
def test_rules_keep_the_exact_top_k(layout, k):
    rng = np.random.default_rng(11 + k)
    n = 6000
    x = unit(rng, n)
    q = unit(rng, 1)[0]
    if layout in ("near-tie burst", "wide burst"):
        m = 300 if layout == "near-tie burst" else 1500
        base = x[np.argsort(x @ q)[-k]]
        x[rng.choice(n, m, replace=False)] = (base + rng.standard_normal((m, D)).astype(f32) * f32(1e-4 / np.sqrt(D)))
    true = x.astype(np.float64) @ q.astype(np.float64)
    if layout == "ascending":
        x, true = x[np.argsort(true)], np.sort(true)
    elif layout == "descending":
        o = np.argsort(true)[::-1]
        x, true = x[o], true[o]
    s, c = quantise_rows(x)
    sc = scan_scores(q, s, c)
    E = bound(q, x, s, c)
    assert np.abs(true - sc).max() <= E
    rows = np.arange(n)
    want = rows[np.lexsort((rows, -true))][:k]
    got, csize = replay(sc, true, E, k)
    assert np.array_equal(got, want), (layout, k)
    assert csize >= k
    if layout == "wide burst":
        assert csize > 256  # more than one re-score round of the last CTA
