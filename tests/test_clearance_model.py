"""The numpy restatement of the obstacle clearance model (tests/clearance_model.py) against scipy's exact
Euclidean distance transform, a brute-force window search and the three cases of the cost rule."""
import math

import numpy as np
import pytest
from scipy.ndimage import distance_transform_edt

import clearance_model as cm


def _edt_cut(obstacle, radius, margin, g):
    d = distance_transform_edt(~obstacle.astype(bool)) * g
    return np.where(d > radius + margin, np.inf, d)


def _mask(shape, density, seed, border=False):
    rng = np.random.default_rng(seed)
    ob = rng.random(shape) < density
    if border:
        ob[0, rng.integers(0, shape[1])] = ob[-1, rng.integers(0, shape[1])] = True
        ob[rng.integers(0, shape[0]), 0] = ob[rng.integers(0, shape[0]), -1] = True
    ob[rng.integers(0, shape[0]), rng.integers(0, shape[1])] = True  # at least one obstacle
    return ob


# (shape, obstacle density, global_res, radius, margin): R = 0, 1, a few cells and 128, margin 0,
# sizes that are not multiples of 32
CASES = [
    ((37, 53), 0.02, 1.0, 0.0, 0.5),       # R = 0
    ((64, 96), 0.01, 1.0, 1.0, 0.0),       # R = 1, margin 0
    ((70, 130), 0.005, 0.35, 0.7, 1.5),    # R = 6, global_res != 1
    ((50, 41), 0.03, 2.5, 2.0, 5.5),       # R = 3, global_res != 1
    ((300, 290), 0.0005, 1.0, 60.0, 68.5), # R = 128
    ((33, 65), 0.2, 1.0, 2.0, 3.0),        # dense
]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_clearance_equals_scipy_edt(case, seed):
    shape, density, g, radius, margin = case
    ob = _mask(shape, density, seed, border=(seed == 2))
    d = cm.clearance(ob, radius, margin, g)
    ref = _edt_cut(ob, radius, margin, g)
    assert np.array_equal(np.isinf(d), np.isinf(ref))
    assert np.array_equal(d, ref)  # bit for bit
    assert np.all(d[ob] == 0.0)


def test_reach_128_is_the_limit():
    assert cm.reach_cells(60.0, 68.5, 1.0) == cm.MAX_CELLS
    assert cm.reach_cells(60.0, 69.0, 1.0) == cm.MAX_CELLS + 1


def test_all_obstacles_and_no_obstacles():
    ob = np.ones((20, 45), dtype=bool)
    assert np.all(cm.clearance(ob, 2.0, 3.0, 1.0) == 0.0)
    # no obstacle to measure to (scipy has none either): +inf everywhere by definition
    assert np.all(np.isinf(cm.clearance(np.zeros((20, 45), dtype=bool), 2.0, 3.0, 1.0)))


def test_squared_distance_is_the_window_minimum():
    """The separable restatement equals the brute-force minimum over the (2R+1)^2 window, including
    cells whose nearest obstacle lies outside the window (no obstacle: -1)."""
    ob = _mask((23, 31), 0.03, 9, border=True)
    for R in (0, 1, 3, 7):
        s = cm.squared_distance(ob, R)
        oj, oi = np.nonzero(ob)
        for j in range(ob.shape[0]):
            for i in range(ob.shape[1]):
                inw = (np.abs(oi - i) <= R) & (np.abs(oj - j) <= R)
                want = int(np.min((oi[inw] - i) ** 2 + (oj[inw] - j) ** 2)) if inw.any() else -1
                assert s[j, i] == want


def test_cost_rule_three_cases():
    radius, margin, penalty = 2.0, 3.0, 4.0
    d = np.array([0.0, 1.0, 2.0, 2.0000000001, 3.0, 4.999999, 5.0, 6.0, np.inf])
    c = np.linspace(0.3, 2.1, d.size)
    out = cm.ceff(c, d, radius, margin, penalty)
    for k in range(d.size):
        if d[k] <= radius:
            assert out[k] == math.inf
        elif d[k] < radius + margin:
            assert out[k] == c[k] * (1.0 + penalty * ((radius + margin - d[k]) / margin))
            assert out[k] > c[k]
        else:
            assert out[k] == c[k]
    # margin 0: lethal ring only, everything else untouched
    out0 = cm.ceff(c, d, radius, 0.0, penalty)
    assert np.array_equal(out0, np.where(d <= radius, np.inf, c))
    # radius 0: only obstacles (d = 0) are lethal
    outr = cm.ceff(c, d, 0.0, margin, penalty)
    assert outr[0] == math.inf and np.all(np.isfinite(outr[1:]))
