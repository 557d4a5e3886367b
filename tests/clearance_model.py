"""numpy restatement of the obstacle clearance model (include/dymu_cuda.h, dymu_set_obstacle_clearance),
in the expression order of the device code."""
import math

import numpy as np

MAX_CELLS = 128
_NONE = np.int64(1) << 40


def reach_cells(radius, margin, g):
    """R = floor((radius + margin) / g)."""
    return int(math.floor((radius + margin) / g))


def squared_distance(obstacle, R):
    """s: the smallest di*di + dj*dj over obstacle cells (i+di, j+dj) with |di|, |dj| <= R (cells
    outside the grid are not obstacles); -1 where there is none.  Exact integers: the minimum over the
    window is taken along the columns first, then along the rows."""
    ob = np.asarray(obstacle).astype(bool)
    ny, nx = ob.shape
    col = np.full((ny, nx), _NONE, dtype=np.int64)
    for dj in range(-R, R + 1):
        lo, hi = max(0, -dj), min(ny, ny - dj)
        if lo < hi:
            np.minimum(col[lo:hi], np.where(ob[lo + dj:hi + dj], dj * dj, _NONE), out=col[lo:hi])
    s = np.full((ny, nx), _NONE, dtype=np.int64)
    for di in range(-R, R + 1):
        lo, hi = max(0, -di), min(nx, nx - di)
        if lo < hi:
            np.minimum(s[:, lo:hi], col[:, lo + di:hi + di] + di * di, out=s[:, lo:hi])
    return np.where(s >= _NONE, -1, s)


def clearance(obstacle, radius, margin, g):
    """d = sqrt(s) * g, +inf where there is no obstacle in the window or d > radius + margin."""
    s = squared_distance(obstacle, reach_cells(radius, margin, g))
    d = np.sqrt(np.where(s < 0, 0, s).astype(np.float64)) * g
    return np.where((s < 0) | (d > radius + margin), np.inf, d)


def factor(d, radius, margin, penalty):
    """The margin factor 1.0 + penalty * ((radius + margin - d) / margin) (meaningful in the band)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return 1.0 + penalty * ((radius + margin - d) / margin)


def plain_ceff(cost, haz, traff, obstacle, g):
    """C_eff without clearance: g * cost * (2 + hazard - trafficability), +inf on obstacles."""
    with np.errstate(invalid="ignore", over="ignore"):
        c = g * cost * (2 + haz - traff)
    return np.where(np.asarray(obstacle).astype(bool), np.inf, c)


def ceff(c, d, radius, margin, penalty):
    """Clearance-adjusted C_eff from the plain one `c` and the clearance `d`: +inf for d <= radius,
    c * factor for radius < d < radius + margin, c itself (selected, not multiplied) otherwise."""
    band = (d > radius) & (d < radius + margin)
    with np.errstate(invalid="ignore", over="ignore"):
        scaled = c * factor(d, radius, margin, penalty)
    return np.where(d <= radius, np.inf, np.where(band, scaled, c))
