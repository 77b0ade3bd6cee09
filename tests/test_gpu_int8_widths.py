"""Single-query searches of the int8 scan copy at every row width it is planned for (d = 256, 512, 768, 1024: one to four
8-byte lanes' worth of codes per row, 16-, 8- and 4-row groups): the oracle's bits and the fp32 scan's bits on random
rows, on ascending rows (every group passes the threshold, so the warp buffers compact before they append) and on a row
count that is not a multiple of any group size."""
import numpy as np
import pytest

from test_gpu_shadow_scan import _opts, build, check, unit  # noqa: F401  (_opts: the autouse option fixture)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("d", [256, 768, 1024])
def test_random_rows(d):
    rng = np.random.default_rng(40 + d)
    x = unit(rng, 300_000, d)
    q = unit(rng, 2, d)
    idx = build(x)
    assert idx.shadow_stats()[1] > 0
    check(idx, q, x, ref=build(x, shadow=0))


@pytest.mark.parametrize("d", [256, 768, 1024])
def test_ascending_rows(d):
    rng = np.random.default_rng(50 + d)
    x = unit(rng, 300_000, d)
    q = unit(rng, 1, d)
    x = np.ascontiguousarray(x[np.argsort(x @ q[0])])
    check(build(x), q, x, ks=(48,), ref=build(x, shadow=0))


@pytest.mark.parametrize("d", [256, 512, 768, 1024])
def test_row_count_off_the_group_size(d):
    rng = np.random.default_rng(60 + d)
    x = unit(rng, 262_147, d)
    q = unit(rng, 2, d)
    check(build(x), q, x, ks=(1, 48), ref=build(x, shadow=0))
