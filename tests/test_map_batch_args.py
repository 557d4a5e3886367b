"""cuda_api.batch_solve_maps refuses, before any native call, a cost array that does not match the
layers: the library reads and writes the contexts' ny x nx cells per map, so a wrongly shaped array
would be read past its end and the returned matrices written past theirs.  No GPU needed: the checks
only look at the layers' sizes."""
import types

import numpy as np
import pytest


def _layers(nx, ny, k=2):
    return [types.SimpleNamespace(nx=nx, ny=ny) for _ in range(k)]


@pytest.mark.parametrize("shape,sizes", [
    ((3, 41, 50), [(50, 40)] * 2), ((3, 39, 50), [(50, 40)] * 2),   # more / fewer rows than the layers
    ((3, 40, 51), [(50, 40)] * 2), ((3, 40, 49), [(50, 40)] * 2),   # more / fewer columns
    ((3, 40, 50), [(50, 40), (50, 41)]),                             # one layer of another size
    ((40, 50), [(50, 40)] * 2),                                      # not a stack of maps
])
def test_shape_must_match_every_layer(pkg, shape, sizes):
    layers = [types.SimpleNamespace(nx=nx, ny=ny) for nx, ny in sizes]
    with pytest.raises(ValueError):
        pkg.cuda_api.batch_solve_maps(layers, np.ones(shape), [(1, 1)] * 3, total_cost=True)


def test_one_goal_and_one_start_per_map(pkg):
    costs = np.ones((3, 40, 50))
    with pytest.raises(ValueError):
        pkg.cuda_api.batch_solve_maps(_layers(50, 40), costs, [(1, 1)] * 2)
    with pytest.raises(ValueError):
        pkg.cuda_api.batch_solve_maps(_layers(50, 40), costs, [(1, 1)] * 3, starts=[(2.0, 2.0)] * 4)
