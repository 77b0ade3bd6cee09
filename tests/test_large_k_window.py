"""CPU: the large-k window rule (DESIGN.md section 2, "Large k") replayed in numpy, and the option that enables it.

Rule: with s_(k) the k-th largest fp32 scan score and E a bound of |scan score - exact score| for every row, every row whose
scan score is >= fl_down(s_(k) - 2E) is re-scored exactly, and the top k of those is the answer.  The replay perturbs the
exact scores adversarially by up to E -- the exact top k pushed down, every other row pushed up -- and checks that the
candidate set still holds the exact top k."""
import os
import re

import numpy as np
import pytest

import evo_ssearch_b200 as evs
from evo_ssearch_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32


def test_max_k_option():
    assert evs.get_option("max_k") == 112
    try:
        for v in (112, 113, 2048, 500):
            evs.set_option("max_k", v)
            assert evs.get_option("max_k") == v
        for bad in (111, 2049, 0, -1):
            with pytest.raises(evs.EvsError) as e:
                evs.set_option("max_k", bad)
            assert e.value.code == _lib.EVS_EINVAL
        assert evs.get_option("max_k") == 500  # a rejected value leaves the option as it was
    finally:
        evs.set_option("max_k", 112)


def test_constants_match_the_header():
    text = open(os.path.join(ROOT, "include", "evs.h")).read()
    consts = dict(re.findall(r"#define\s+(EVS_MAX_K\w*)\s+(\d+)", text))
    assert int(consts["EVS_MAX_K"]) == _lib.EVS_MAX_K == 112
    assert int(consts["EVS_MAX_K_LARGE"]) == _lib.EVS_MAX_K_LARGE == 2048


def _down(v):
    """largest fp32 <= v (v an fp64)"""
    f = f32(v)
    return f32(np.nextafter(f, f32(-np.inf))) if float(f) > v else f


def _up(v):
    f = f32(v)
    return f32(np.nextafter(f, f32(np.inf))) if float(f) < v else f


def _candidates(exact, k, E):
    """the window of the large-k path after an adversarial scan"""
    n = exact.shape[0]
    top = np.lexsort((np.arange(n), -exact))[:k]
    scan = np.array([_down(s + E) for s in exact], np.float32)  # everything else pushed up (rounded inside the bound)
    scan[top] = [_up(exact[i] - E) for i in top]                # the exact top k pushed down
    if n <= k:
        return top, np.arange(n)
    sk = np.sort(scan)[::-1][k - 1]
    cut = _down(float(sk) - 2 * E)
    return top, np.nonzero(scan >= cut)[0]


def _data(kind, n, k, rng):
    if kind == "ordered":
        return np.linspace(-1.0, 1.0, n)
    s = rng.standard_normal(n) * 0.05
    if kind == "tied":
        order = np.argsort(-s)
        s[order[k // 2:k // 2 + n // 3]] = s[order[k]]
    elif kind == "near-tie":
        order = np.argsort(-s)
        h = min(200, k // 2)
        s[order[k - h:k + h]] = s[order[k]] + rng.uniform(-1e-6, 1e-6, 2 * h)
    return s


@pytest.mark.parametrize("kind", ["ordered", "tied", "near-tie", "random"])
@pytest.mark.parametrize("k", [113, 1024, 2048])
def test_window_holds_the_exact_top_k(kind, k):
    rng = np.random.default_rng(k)
    n = 6000
    for E in (1e-7, 3e-6, 1e-4):
        exact = _data(kind, n, k, rng)
        exact = exact.astype(np.float32).astype(np.float64) * 0.999 + exact * 1e-3  # scores off the fp32 grid
        top, cand = _candidates(exact, k, E)
        assert np.isin(top, cand).all(), (kind, k, E)
        # the window is not the whole shard on ordinary data
        if kind in ("ordered", "random") and E < 1e-5:
            assert cand.shape[0] < n // 2


def test_window_fewer_rows_than_k():
    exact = np.linspace(0, 1, 100)
    top, cand = _candidates(exact, 113, 1e-6)
    assert np.isin(top, cand).all() and cand.shape[0] == 100
