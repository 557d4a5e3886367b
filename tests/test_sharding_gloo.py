"""N > 1 host logic on the CPU: world_size-2/3 gloo runs of the domain-decomposition driver
(planning-path_planning_b200/sharding.py) with a numpy strip solver standing in for the GPU;
the assembled map must equal the oracle's single-grid solve."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _eikonal(Tx, Ty, C):
    d = Tx - Ty
    with np.errstate(invalid="ignore"):
        two = np.abs(d) < C
        arg = np.where(two, 2 * (C * C) - d * d, 1.0)
        return np.where(two, (Tx + Ty + np.sqrt(arg)) / 2, np.minimum(Tx, Ty) + C)


class NumpyStrip:
    """Same interface as sharding.CudaStrip; Jacobi fixed point of G.cpp:500-546 in numpy."""

    def __init__(self, layout, cost_own_rows):
        self.layout = layout
        cost = layout.local_cost(cost_own_rows)
        self.C = np.where(cost > 0, 1.0 * cost * (2 + 0.0 - 1.0), np.inf)
        self.T = np.full(cost.shape, np.inf)

    def _relax(self, max_sweeps):
        """Returns True if it stopped at the sweep budget with changes still happening."""
        T, C = self.T, self.C
        sweeps = 0
        while True:
            if sweeps >= max_sweeps:
                return True
            sweeps += 1
            P = np.pad(T, 1, constant_values=np.inf)
            Tx = np.minimum(P[1:-1, :-2], P[1:-1, 2:])
            Ty = np.minimum(P[:-2, 1:-1], P[2:, 1:-1])
            with np.errstate(invalid="ignore"):
                Tn = _eikonal(Tx, Ty, C)
            better = np.isfinite(C) & (Tn < T)
            if not better.any():
                return False
            T[better] = Tn[better]

    # a "phase" is one Jacobi sweep here
    def start(self, goal_global, phases):
        gi, gj = goal_global
        self.T[...] = np.inf
        if self.layout.owns(gj):
            self.T[self.layout.local_row(gj), gi] = 0.0
            return self._relax(phases)
        return False

    def boundary_rows(self):
        lay = self.layout
        return (torch.from_numpy(self.T[lay.first_own].copy()),
                torch.from_numpy(self.T[lay.last_own].copy()))

    def absorb(self, from_above, from_below):
        ranges, key = [], np.inf
        for row, src in ((0, from_above), (self.layout.ny_local - 1, from_below)):
            if src is None:
                continue
            v = src.numpy()
            m = v < self.T[row]
            if m.any():
                self.T[row][m] = v[m]
                ranges.append((row, row + 1))
                key = min(key, float(v[m].min()))
        return ranges, key

    def advance(self, ranges, key, phases):
        assert (not ranges) or np.isfinite(key)
        return self._relax(phases)

    def own_rows(self):
        lay = self.layout
        return self.T[lay.first_own:lay.last_own + 1]


def _worker(rank, world, port, cost, goal, out_dir, phases):
    sys.path.insert(0, ROOT)
    import dymu_b200
    sh = dymu_b200.load().sharding
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lay = sh.StripLayout(cost.shape[0], world, rank, align=8)
    strip = NumpyStrip(lay, cost[lay.r0:lay.r1])
    comm = sh.TorchComm(rank, world, torch.device("cpu"))
    rounds = sh.dd_solve_pipelined(strip, comm, goal, phases_per_round=phases)
    np.save(os.path.join(out_dir, "T_%d.npy" % rank), strip.own_rows())
    np.save(os.path.join(out_dir, "rounds_%d.npy" % rank), np.array([rounds, lay.r0, lay.r1]))
    dist.destroy_process_group()


# 10**6 phases per round: a budget no strip exhausts, so every strip converges before it trades rows
@pytest.mark.parametrize("world,port,phases", [(2, 29611, 10**6), (3, 29612, 10**6),
                                               (2, 29613, 7), (3, 29614, 7)])
def test_domain_decomposition_matches_single_grid(pkg, oracle_mod, tmp_path, world, port, phases):
    ny, nx = 72, 56
    cost = pkg.synthetic.smooth_cost_map(ny, nx, seed=5, obstacle_fraction=0.05)
    ob = cost <= 0
    gi, gj = pkg.synthetic.free_interior_cell_near(ob, 40, 12)   # goal inside the first strip
    mp.spawn(_worker, args=(world, port, cost, (gi, gj), str(tmp_path), phases), nprocs=world,
             join=True)
    parts = [np.load(tmp_path / ("T_%d.npy" % r)) for r in range(world)]
    T = np.vstack(parts)
    po = oracle_mod.Port(1.0, 1.5, 2.0, 1)
    po.initGlobalLayer(1.0, 0.1, nx, ny)
    po.setCostMap(cost)
    assert po.setGoal(gi, gj) and po.computeEntireTotalCostMap()
    To = po.plane("total_cost")
    assert np.array_equal(np.isinf(T), np.isinf(To))
    fin = np.isfinite(To) & (To > 0)
    assert np.max(np.abs(T[fin] - To[fin]) / To[fin]) <= 1e-12
    rounds = [int(np.load(tmp_path / ("rounds_%d.npy" % r))[0]) for r in range(world)]
    assert len(set(rounds)) == 1 and rounds[0] >= world   # every rank leaves the loop together


def test_partition_helpers(pkg):
    sh = pkg.sharding
    for n, w in ((1024, 8), (10, 3), (7, 8)):
        got = [list(sh.shard_queries(n, w, r)) for r in range(w)]
        assert sum(got, []) == list(range(n))
        assert max(len(g) for g in got) - min(len(g) for g in got) <= 1
    for ny, w in ((16384, 8), (4096, 4), (1000, 3), (96, 2)):
        cuts = [sh.strip_rows(ny, w, r) for r in range(w)]
        assert cuts[0][0] == 0 and cuts[-1][1] == ny
        for a, b in zip(cuts, cuts[1:]):
            assert a[1] == b[0] and a[1] % 32 == 0
        assert all(hi > lo for lo, hi in cuts)
