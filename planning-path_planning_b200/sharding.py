"""Multi-GPU partitioning of the total-cost propagation (SURVEY.md section 8e).

Two cases shard naturally:

* independent goal queries / maps -- ``shard_queries``: block assignment of queries to
  ranks, no data-path collective (each rank holds the read-only cost planes);
* one very large grid -- row-strip domain decomposition (``strip_rows`` +
  ``dd_solve_pipelined``): each rank owns a contiguous band of rows plus one ghost row per
  interior side.  Every round, a rank advances its strip by a bounded number of solver
  phases (``dymu_solve_start`` / ``dymu_solve_advance`` keep the pending work on the
  device), boundary rows are exchanged with the two neighbours (point-to-point) and a
  1-word all-reduce decides termination.  A neighbour starts as soon as the wave front
  crosses the cut instead of after the whole strip behind it has converged.  Ghost rows
  carry C_eff = +inf, so they are never updated locally and act as Dirichlet data; values
  only ever decrease, so the iteration converges to the single-grid fixed point.

The driver is written against two small interfaces so that the very same control flow runs
on GPUs (``CudaStrip`` + torch.distributed/NCCL) and in the CPU test-suite (a numpy strip
solver + gloo).
"""
import numpy as np


def shard_queries(n_queries, world, rank):
    """Contiguous block of query indices owned by `rank` (sizes differ by at most one)."""
    base, extra = divmod(n_queries, world)
    lo = rank * base + min(rank, extra)
    return range(lo, lo + base + (1 if rank < extra else 0))


def strip_rows(ny, world, rank, align=32):
    """Rows [r0, r1) of the global grid owned by `rank`; interior cuts are multiples of
    `align` (the solver tile) so that no tile straddles two ranks."""
    cuts = [0]
    for k in range(1, world):
        c = int(round(k * ny / float(world) / align)) * align
        cuts.append(min(max(c, cuts[-1] + align), ny - align * (world - k)))
    cuts.append(ny)
    return cuts[rank], cuts[rank + 1]


class StripLayout:
    """Index arithmetic of one strip: global rows [r0, r1) plus ghost rows."""

    def __init__(self, ny, world, rank, align=32):
        self.world, self.rank = world, rank
        self.r0, self.r1 = strip_rows(ny, world, rank, align)
        self.ghost_top = 1 if rank > 0 else 0
        self.ghost_bottom = 1 if rank < world - 1 else 0
        self.ny_local = (self.r1 - self.r0) + self.ghost_top + self.ghost_bottom

    def local_row(self, global_row):
        return global_row - self.r0 + self.ghost_top

    @property
    def first_own(self):
        return self.ghost_top

    @property
    def last_own(self):
        return self.ghost_top + (self.r1 - self.r0) - 1

    def owns(self, global_row):
        return self.r0 <= global_row < self.r1

    def local_cost(self, cost_global_rows):
        """Cost plane of the strip: own rows of the global cost map, ghost rows = 0 (cost <= 0
        marks an obstacle => C_eff = +inf => never a propagation target)."""
        nx = cost_global_rows.shape[1]
        out = np.zeros((self.ny_local, nx), dtype=np.float64)
        out[self.first_own:self.last_own + 1] = cost_global_rows
        return out


class TorchComm:
    """Neighbour exchange + termination vote over torch.distributed (nccl or gloo)."""

    def __init__(self, rank, world, device):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.world, self.device = rank, world, device

    def exchange(self, top_row, bottom_row):
        """Sends my first own row up and my last own row down; returns (row from the rank
        above, row from the rank below), None where there is no neighbour."""
        torch, dist = self.torch, self.dist
        ops, from_above, from_below = [], None, None
        if self.rank > 0:
            from_above = torch.empty_like(top_row)
            ops.append(dist.P2POp(dist.isend, top_row, self.rank - 1))
            ops.append(dist.P2POp(dist.irecv, from_above, self.rank - 1))
        if self.rank < self.world - 1:
            from_below = torch.empty_like(bottom_row)
            ops.append(dist.P2POp(dist.isend, bottom_row, self.rank + 1))
            ops.append(dist.P2POp(dist.irecv, from_below, self.rank + 1))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
            # NCCL completes on torch's stream; the library reads the rows on its own stream
            if self.device.type == "cuda":
                torch.cuda.synchronize(self.device)
        return from_above, from_below

    def any(self, flag):
        t = self.torch.tensor([1 if flag else 0], dtype=self.torch.int32, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return int(t.item()) > 0


class CudaStrip:
    """One rank's strip on its GPU, on top of the C ABI (include/dymu_cuda.h)."""

    def __init__(self, cuda_api, layout, nx, cost_own_rows, device_index, torch):
        self.layout, self.nx, self.torch = layout, nx, torch
        self.dev = cuda_api.DeviceLayer(nx, layout.ny_local, 1.0, 0.1, device=device_index)
        self.dev.set_cost_map(layout.local_cost(cost_own_rows))
        self.device = torch.device("cuda", device_index)
        self._row = {k: torch.empty(nx, dtype=torch.float64, device=self.device) for k in "tb"}
        self.stats = []

    def boundary_rows(self):
        lay = self.layout
        self.dev.export_rows(lay.first_own, 1, self._row["t"].data_ptr(), True)
        self.dev.export_rows(lay.last_own, 1, self._row["b"].data_ptr(), True)
        return self._row["t"], self._row["b"]

    def start(self, goal_global, phases):
        """Initial local solve of at most `phases` solver phases: the rank owning the goal seeds
        it, the others start at +inf.  Returns True while work is pending on the device."""
        gi, gj = goal_global
        if self.layout.owns(gj):
            st = self.dev.solve_start((gi, self.layout.local_row(gj)), phases)
            self.stats.append(st)
            return not st["converged"]
        self.dev.reset_total_cost()
        return False

    def absorb(self, from_above, from_below):
        """Min-merges neighbour rows into the ghost rows.  Returns the row ranges to wake and
        the smallest value a ghost row was lowered to: the priority the woken tiles get among
        the pending ones."""
        lay, ranges, key = self.layout, [], float("inf")
        if from_above is not None:
            ch, lo = self.dev.import_rows_min_key(0, 1, from_above.data_ptr(), True)
            if ch:
                ranges.append((0, 2))
                key = min(key, lo)
        if from_below is not None:
            ch, lo = self.dev.import_rows_min_key(lay.ny_local - 1, 1, from_below.data_ptr(), True)
            if ch:
                ranges.append((lay.ny_local - 2, lay.ny_local))
                key = min(key, lo)
        return ranges, key

    def advance(self, ranges, key, phases):
        st = self.dev.solve_advance(ranges, key if ranges else 0.0, phases)
        self.stats.append(st)
        return not st["converged"]

    def own_rows(self):
        lay = self.layout
        T = self.dev.download_total_cost()
        return T[lay.first_own:lay.last_own + 1]


def dd_solve_pipelined(strip, comm, goal_global, phases_per_round=16, max_rounds=1000000):
    """Domain-decomposed solve with bounded work per exchange round: every rank runs at most
    `phases_per_round` solver phases, trades boundary rows, merges what it received into its
    pending work, and the loop ends when no rank has pending work or fresh halo values.
    Returns the number of rounds."""
    import time
    lap = {"advance": 0.0, "export": 0.0, "exchange": 0.0, "absorb": 0.0, "vote": 0.0}

    def timed(name, fn, *a):
        t0 = time.perf_counter()
        out = fn(*a)
        lap[name] += time.perf_counter() - t0
        return out

    pending = timed("advance", strip.start, goal_global, phases_per_round)
    rounds = 0
    while rounds < max_rounds:
        top, bottom = timed("export", strip.boundary_rows)
        from_above, from_below = timed("exchange", comm.exchange, top, bottom)
        ranges, key = timed("absorb", strip.absorb, from_above, from_below)
        rounds += 1
        if not timed("vote", comm.any, bool(ranges) or pending):
            break
        pending = timed("advance", strip.advance, ranges, key, phases_per_round)
    strip.laps = lap
    return rounds


def dd_solve_lockstep(strips, goal_global, phases_per_round=16, max_rounds=1000000):
    """dd_solve_pipelined with all strips in ONE process (k logical shards on one device, or
    several devices driven by one host thread): rows are handed over directly instead of
    through torch.distributed.  Returns the number of exchange rounds."""
    pending = [s.start(goal_global, phases_per_round) for s in strips]
    rounds = 0
    while rounds < max_rounds:
        rows = [tuple(r.clone() for r in s.boundary_rows()) for s in strips]
        rounds += 1
        todo = []
        for k, s in enumerate(strips):
            from_above = rows[k - 1][1] if k > 0 else None
            from_below = rows[k + 1][0] if k + 1 < len(strips) else None
            todo.append(s.absorb(from_above, from_below))
        if not any(pending) and not any(r for r, _ in todo):
            break
        pending = [s.advance(r, key, phases_per_round) for s, (r, key) in zip(strips, todo)]
    return rounds
