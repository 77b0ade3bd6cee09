"""CPU restatement of the exact single-query search from the bf16 scan copy (evs_scan.cuh: scan_pool_kernel, DESIGN.md
section 2).  For a row x, x^ = bf16_rn(x) and s~ the fp32 scan score of x^ against the fp32 query:

    |q.x - s~| <= |q| |x - x^| + gamma_d |q| |x^| <= E = |q| (e_max + gamma_d max|x| (1 + 2^-7))   (inflated, rounded up)

Rule 1 drops a row only if s~ < t - 2E for a score t that 64 rows are known to reach; rule 2 re-scores every survivor with
s~ >= s~_(k) - 2E.  These tests check the bound against the scan's own summation order and replay both rules."""
import numpy as np
import pytest

D = 512


def bf16_rn(x):
    """fp32 -> bf16 (round to nearest even), returned as fp32 (finite inputs)."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32).reshape(np.shape(x))


def gemv_err_coef(d):
    return (d // 32 + 8) * 2.0**-24


def scan_scores(q, xh):
    """The pool kernel's fp32 order for bf16 rows (8 elements per lane and 16-byte vector): lane l, vector j holds elements
    8 (l + 32 j) .. +8; four partial sums by element index mod 4, combined (p0 + p1) + (p2 + p3), then the xor butterfly."""
    n, d = xh.shape
    nv = d // 256
    x = xh.reshape(n, nv, 32, 8).astype(np.float32)
    qq = q.reshape(nv, 32, 8).astype(np.float32)
    p = np.zeros((n, 32, 4), np.float32)
    for j in range(nv):
        for e in range(8):
            p[:, :, e & 3] = p[:, :, e & 3] + x[:, j, :, e] * qq[j, :, e]
    s = (p[:, :, 0] + p[:, :, 1]) + (p[:, :, 2] + p[:, :, 3])
    for off in (16, 8, 4, 2, 1):
        s = s + s[:, np.arange(32) ^ off]
    return s[:, 0]


def bound(q, x, xh):
    d = x.shape[1]
    emax = np.sqrt(((x.astype(np.float64) - xh) ** 2).sum(1)).max()
    emax = float(np.nextafter(np.float32(emax), np.float32(np.inf)))  # rounded up to fp32, as the add stores it
    max_norm = float(np.float32(np.sqrt((x.astype(np.float64) ** 2).sum(1)).max()) * np.float32(1.000001))
    qn = np.sqrt((q.astype(np.float64) ** 2).sum()) * (1 + 2.0**-20)
    e = qn * (emax + gemv_err_coef(d) * max_norm * (1 + 2.0**-7)) * (1 + 2.0**-20) + d * 2.0**-149
    return float(np.nextafter(np.float32(e), np.float32(np.inf)))


def unit(rng, n, d=D):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True).astype(np.float32)


def rows_cases():
    rng = np.random.default_rng(5)
    x = unit(rng, 4000)
    scaled = x * np.float32(10.0) ** rng.uniform(-3, 3, (4000, 1)).astype(np.float32)
    dominant = x * np.float32(1e-3)
    dominant[np.arange(4000), rng.integers(0, D, 4000)] = rng.choice([-1.0, 1.0], 4000)
    # elements that sit half a bf16 ulp away from their rounding (relative error close to 2^-9 everywhere), signs that
    # follow the query's so that the per-element errors add up
    q = unit(rng, 1)[0]
    mant = np.float32(1.0) + np.float32(2.0**-8) * np.float32(0.999)
    worst = (mant * np.sign(q) * np.float32(2.0) ** rng.integers(-6, 0, (1000, D))).astype(np.float32)
    return {"random": (x, rng), "scaled": (scaled, rng), "dominant": (dominant, rng), "worst rounding": (worst, rng)}, q


@pytest.mark.parametrize("case", ["random", "scaled", "dominant", "worst rounding"])
def test_scan_of_the_bf16_rows_stays_within_the_bound(case):
    cases, q0 = rows_cases()
    x, rng = cases[case]
    xh = bf16_rn(x)
    for q in (q0, unit(rng, 1)[0] * np.float32(37.0), unit(rng, 1)[0] * np.float32(1e-3)):
        E = bound(q, x, xh)
        true = x.astype(np.float64) @ q.astype(np.float64)
        err = np.abs(true - scan_scores(q, xh).astype(np.float64))
        assert err.max() <= E, (case, err.max(), E)
        assert err.max() > 0.0


def test_bound_on_unit_rows_is_about_two_thousandths():
    rng = np.random.default_rng(9)
    x = unit(rng, 20000)
    xh = bf16_rn(x)
    e = np.sqrt(((x.astype(np.float64) - xh) ** 2).sum(1))
    assert 1.4e-3 < e.mean() < 1.9e-3 and e.max() < 2.2e-3
    assert 1.5e-3 < bound(unit(rng, 1)[0], x, xh) < 2.5e-3


def floor_f32(v):
    """largest fp32 <= v"""
    f = np.float32(v)
    return float(np.nextafter(f, np.float32(-np.inf))) if float(f) > v else float(f)


def replay(s, true, E, k, nwarps=37, seed=0):
    """Rules 1 and 2 on scan scores s (fp32) and exact scores `true`: keys order (s desc, row asc), a warp's rows are
    row mod nwarps, the 64 slot maxima are row mod 64.  Returns the k rows ranked by (true desc, row asc) within C."""
    n = s.shape[0]
    rows = np.arange(n)
    key = np.lexsort((rows, -s.astype(np.float64)))  # best first
    rank = np.empty(n, np.int64)
    rank[key] = np.arange(n)
    # t: the larger of the warp's own 64th best and tau_g (smallest slot maximum): both are reached by 64 rows
    tau_g = min(s[rows % 64 == sl].max() for sl in range(min(64, n))) if n >= 64 else -np.inf
    surv = np.zeros(n, bool)
    for w in range(nwarps):
        mine = rows[rows % nwarps == w]
        sw = np.sort(s[mine])[::-1]
        t = max(sw[63] if sw.shape[0] >= 64 else -np.inf, tau_g)
        cut = floor_f32(float(t) - 2 * E) if np.isfinite(t) else -np.inf
        surv[mine] = s[mine] >= cut
    sk = s[key[k - 1]]
    assert surv[key[:k]].all()
    C = rows[surv & (s >= floor_f32(float(sk) - 2 * E))]
    best = C[np.lexsort((C, -true[C]))][:k]
    return best, C.shape[0]


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
        x[rng.choice(n, m, replace=False)] = (base + rng.standard_normal((m, D)).astype(np.float32) * np.float32(1e-4 / np.sqrt(D)))
    true = x.astype(np.float64) @ q.astype(np.float64)
    if layout == "ascending":
        x, true = x[np.argsort(true)], np.sort(true)
    elif layout == "descending":
        o = np.argsort(true)[::-1]
        x, true = x[o], true[o]
    xh = bf16_rn(x)
    s = scan_scores(q, xh)
    E = bound(q, x, xh)
    assert np.abs(true - s).max() <= E
    rows = np.arange(n)
    want = rows[np.lexsort((rows, -true))][:k]
    got, csize = replay(s, true, E, k)
    assert np.array_equal(got, want), (layout, k)
    assert csize >= k
    if layout == "wide burst":
        assert csize > 256  # more than one re-score round of the last CTA
