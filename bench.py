#!/usr/bin/env python
"""bench.py -- DyMu total-cost propagation on B200: one JSON line per run.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on and the largest
that is meant for one GPU): a 4096x4096 synthetic Mars-like DEM (seeded fBm + craters),
cost map built by the device cost-map pipeline (computeCostMap), one goal at the free
interior cell nearest the centre.

A "step" = one plan = full total-cost-map solve (computeEntireTotalCostMap equivalent:
reset + tile-FIM kernel) + gradient-descent path extraction from a fixed start.

  value  : plans/s with the cost planes already resident in HBM (device time, CUDA events
           on the library's stream, max over ranks).  ms_per_step is BASELINE's "ms per
           4096^2 total-cost-map solve" (+ path).
  e2e    : the same through the drop-in class (DyMuPathPlanner in libdymu_b200.so) with HOST
           buffers inside the timed region: H2D of the cost plane (setCostMap), solve, path,
           D2H of the total-cost matrix (getTotalCostMatrix) every step.  e2e_cabi is the same
           work issued directly against the C ABI of include/dymu_cuda.h.
  sub-objects config2_repair / queries2048 / dd16384: the other BASELINE configs, measured in
           the same run (see their docstrings).
  N > 1  : one process per GPU (torchrun); every rank plans on its own copy of the map
           with its own goal -- independent queries, no data-path collective ("weak").

--impl reference times the UNMODIFIED reference (oracle/_ref) on the host cores.

--dump-outputs DIR writes, after the timed steps, what the last step of the headline arm handed
its caller: DIR/total_cost.npy (the total-cost matrix, -1 where unreached as getTotalCostMatrix
delivers it; float64, rows and columns taken with a fixed stride so that it stays under 48 MB:
every 2nd at 4096^2) and DIR/path.npy (the waypoints, float64).  The inputs depend on --size and --seed only, so two
builds run with the same arguments can be compared array for array.  Compare with a tolerance:
the solver's update order varies between runs, and so do the last bits (two runs of one build
on a B200 differed by at most 3.6e-15 relative on the total cost and 1e-11 on the waypoints,
with the same unreached cells).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: leave no __pycache__ in it

METRIC = "plans_per_s"
UNIT = "plans/s"
CELL_SWEEP_BYTES = 24   # per cell of an activated tile: read T, read C_eff, write T (fp64)
SOLVE_BYTES_PER_CELL = 16  # lower bound per solve: read C_eff once, write T once


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="all",
                    help="comma list of plan4096 (BASELINE configs[2], the headline metric/value), config2 "
                         "(configs[1]: 1000^2 + local repair, both approaches, reference beside it), "
                         "queries2048 (configs[3]: 1024 goal queries on a 2048^2 map, sharded over the "
                         "ranks), dd16384 (configs[4]: one 16384^2 grid, domain-decomposed for N >= 2); "
                         "default all -- the sub-benchmarks are reported as sub-objects of the one line")
    ap.add_argument("--dd-size", type=int, default=16384)
    ap.add_argument("--dd-phases", type=int, default=32)
    ap.add_argument("--queries", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed plan4096 step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and (a.impl != "b200" or (a.workload != "all" and "plan4096" not in a.workload.split(","))):
        ap.error("--dump-outputs needs the b200 plan4096 workload")
    return a


def dist_env():
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
            int(os.environ.get("WORLD_SIZE", "1")))


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_workload(pkg, n, seed):
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(n, n, seed=seed)
    lut, slopes, locs = syn.default_lut()
    return elev, terr, lut, slopes, locs


# ---------------------------------------------------------------------------------------
# reference arm
# ---------------------------------------------------------------------------------------
def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return 0
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dymu_b200
    import oracle
    pkg = dymu_b200.load()
    n = args.size
    elev, terr, lut, slopes, locs = build_workload(pkg, n, args.seed)
    # bounded sample: the reference's vector narrow band scales ~x16 per doubling
    # (BASELINE.md: 12.6 s @1000^2, 3152 s @4096^2), so each step solves the central crop
    # whose single-thread time fits the budget
    budget_s = max(2.0, 150.0 / max(1, args.steps + args.warmup))
    crop = int(1000.0 * (budget_s / 14.0) ** 0.25)
    crop = max(256, min(1024, crop, n))
    lo = (n - crop) // 2
    e_c = np.ascontiguousarray(elev[lo:lo + crop, lo:lo + crop])
    t_c = np.ascontiguousarray(terr[lo:lo + crop, lo:lo + crop])
    use_ref = oracle.have_reference()
    cores = min(os.cpu_count() or 1, 32)
    if use_ref:
        lib = oracle.reference()
        make = lambda: lib.DyMuPathPlanner(1.0, 1.5, 2.0, 1)
        kind = "reference"
    else:
        make = lambda: oracle.Port(1.0, 1.5, 2.0, 1)
        kind = "port"
    planners, goals = [], []
    rng = np.random.default_rng(args.seed + 1)
    for c in range(cores):
        p = make()
        p.initGlobalLayer(1.0, 0.1, crop, crop)
        p.computeCostMap(lut, slopes, locs, e_c, t_c)
        ob = p.node_field(4) if hasattr(p, "node_field") else p.plane("isObstacle")
        gi, gj = pkg.synthetic.free_interior_cell_near(
            ob, crop // 2 + int(rng.integers(-crop // 8, crop // 8 + 1)),
            crop // 2 + int(rng.integers(-crop // 8, crop // 8 + 1)))
        si, sj = pkg.synthetic.free_interior_cell_near(ob, crop // 8, crop // 8)
        assert p.setGoal(gi, gj)
        planners.append((p, si, sj))

    def one(p, si, sj):
        p.computeEntireTotalCostMap()
        p.getPath(float(si), float(sj))

    def step():
        ts = [threading.Thread(target=one, args=t) for t in planners]
        for t in ts:
            t.start()
        for t in ts:
            t.join()

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    ms_per_step = dt / args.steps * 1e3
    frac = (crop * crop) / float(n * n)
    value = cores * frac / (dt / args.steps)
    sample = ("%d threads, each one full solve + path on the central %dx%d crop (%.4f of the "
              "%dx%d cells) per step; value = crop-fraction plans/s, i.e. assumes time linear in "
              "cells, which flatters the reference (its narrow-band scan scales ~x16 per "
              "doubling: 3152 s measured for one 4096^2 solve in BASELINE.md)"
              % (cores, crop, crop, frac, n, n))
    # same configuration, different container: the pinned C port of the reference's update with a
    # binary heap instead of the reference's linear narrow-band scan, full map, one core
    same_config = None
    try:
        q = oracle.Port(1.0, 1.5, 2.0, 1)
        q.initGlobalLayer(1.0, 0.1, n, n)
        q.computeCostMap(lut, slopes, locs, elev, terr)
        g2 = pkg.synthetic.free_interior_cell_near(q.plane("isObstacle"), n // 2, n // 2)
        q.setGoal(*g2)
        t1 = time.perf_counter()
        q.computeEntireTotalCostMap(heap=True)
        q.getPath(float(n // 8), float(n // 8))
        dt_full = time.perf_counter() - t1
        q.close()
        same_config = {"seconds_per_plan": dt_full, "plans_per_s_per_core": 1.0 / dt_full, "cores": 1,
                       "kind": "port (oracle/dymu_oracle.c, heap-ordered; the unmodified reference needs "
                               "3152 s for this solve, BASELINE.md)"}
    except Exception as e:
        same_config = {"error": str(e)}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "configs[2]: %dx%d synthetic Mars-like DEM cost map, FMM total-cost "
                               "solve + path, 1 goal" % (n, n), "seed": args.seed,
                   "reference_sample_crop": crop},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "same_config_full_map": same_config,
    }
    print(json.dumps(line))
    return 0


def cpu_baseline_leg(pkg, elev, terr, lut, slopes, locs, n):
    """Reference (oracle/_ref) or port, 1 thread, bounded sample (~15 s): central 1024^2 crop."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    crop = min(1024, n)
    lo = (n - crop) // 2
    e_c = np.ascontiguousarray(elev[lo:lo + crop, lo:lo + crop])
    t_c = np.ascontiguousarray(terr[lo:lo + crop, lo:lo + crop])
    if oracle.have_reference():
        p = oracle.reference().DyMuPathPlanner(1.0, 1.5, 2.0, 1)
        kind = "reference"
    else:
        p = oracle.Port(1.0, 1.5, 2.0, 1)
        kind = "port"
    p.initGlobalLayer(1.0, 0.1, crop, crop)
    p.computeCostMap(lut, slopes, locs, e_c, t_c)
    ob = p.node_field(4) if hasattr(p, "node_field") else p.plane("isObstacle")
    gi, gj = pkg.synthetic.free_interior_cell_near(ob, crop // 2, crop // 2)
    p.setGoal(gi, gj)
    t0 = time.perf_counter()
    p.computeEntireTotalCostMap()
    p.getPath(float(crop // 8), float(crop // 8))
    dt = time.perf_counter() - t0
    frac = (crop * crop) / float(n * n)
    # the C port with a heap (not the reference's algorithmic complexity) on the full map
    fast = None
    try:
        q = oracle.Port(1.0, 1.5, 2.0, 1)
        q.initGlobalLayer(1.0, 0.1, n, n)
        q.computeCostMap(lut, slopes, locs, elev, terr)
        g2 = pkg.synthetic.free_interior_cell_near(q.plane("isObstacle"), n // 2, n // 2)
        q.setGoal(*g2)
        t1 = time.perf_counter()
        q.computeEntireTotalCostMap(heap=True)
        fast = time.perf_counter() - t1
        q.close()
    except Exception:
        fast = None
    return {
        "value": frac / dt, "unit": UNIT, "cores": 1, "kind": kind,
        "sample": ("1 thread, one full solve + path on the central %dx%d crop (%.4f of the cells) "
                   "in %.2f s; value = crop-fraction plans/s (linear-in-cells extrapolation, "
                   "optimistic for the reference)" % (crop, crop, frac, dt)),
        "sample_seconds": dt,
        "heap_port_full_map_seconds": fast,
    }


# ---------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------
NCU_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r2_k_fim_traffic.json")


def _ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_fim launch on this workload from the
    committed `ncu --set full` capture of this round (profiles/), with its capture date -- kept
    beside the figure derived live from the kernel's own counters."""
    try:
        with open(NCU_TRAFFIC_FILE) as f:
            d = json.load(f)
        return {"dram_bytes_per_launch": float(d["dram_bytes_per_launch"]), "captured": d.get("captured"),
                "source": os.path.relpath(NCU_TRAFFIC_FILE, ROOT)}
    except (OSError, KeyError, ValueError):
        return None


_ALL_CORES = None


def unpin():
    """Back to every core of the box (rank 0 before it drives all GPUs from one process)."""
    try:
        if _ALL_CORES:
            os.sched_setaffinity(0, _ALL_CORES)
    except (AttributeError, OSError):
        pass


def pin_rank(local_rank, world):
    """Give every rank its own slice of the host cores before it allocates pinned buffers, so that
    first-touch places them next to the cores that drive this GPU's copies."""
    global _ALL_CORES
    try:
        cores = sorted(os.sched_getaffinity(0))
        _ALL_CORES = cores
        per = max(1, len(cores) // max(1, world))
        mine = cores[local_rank * per:(local_rank + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return [mine[0], mine[-1]]
    except (AttributeError, OSError):
        return None


class Dist:
    def __init__(self):
        import torch
        self.torch = torch
        self.rank, self.local_rank, self.world = dist_env()
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the B200 arm has no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        self.on = self.world > 1
        if self.on:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group(backend="nccl", device_id=torch.device("cuda", self.local_rank))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.on:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def host_barrier(self, name):
        """Barrier on the rendezvous store, without a GPU kernel: ranks that wait here leave their
        GPU idle (an NCCL barrier would keep a spinning kernel on it), so rank 0 may meanwhile drive
        all GPUs of the box from its own process (dymu_dd_solve)."""
        self.torch.cuda.synchronize()
        if not self.on:
            return
        store = self.dist.distributed_c10d._get_default_store()
        key = "bench_host_barrier_" + name
        store.add(key, 1)
        t0 = time.perf_counter()
        while store.add(key, 0) < self.world:
            if time.perf_counter() - t0 > 900.0:
                raise RuntimeError("bench.py: rank %d waited 15 min at host barrier %s" % (self.rank, name))
            time.sleep(0.002)

    def max(self, values):
        if not self.on:
            return [float(v) for v in values]
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def gather(self, values):
        """per-rank lists of floats -> list (rank order) on every rank"""
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        if not self.on:
            return [[float(v) for v in t]]
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [[float(v) for v in o] for o in out]

    def close(self):
        if self.on:
            self.dist.destroy_process_group()


def headline_plan4096(args, D, pkg, affinity):
    """configs[2]: the line's metric/value/e2e/roofline."""
    torch = D.torch
    rank, world = D.rank, D.world
    n = args.size
    elev, terr, lut, slopes, locs = build_workload(pkg, n, args.seed)
    dev = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1, device=D.local_rank)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    ob = dev.download_plane_u8("obstacle")
    syn = pkg.synthetic
    rng = np.random.default_rng(args.seed + 17 * rank)
    if rank == 0:
        goal = syn.free_interior_cell_near(ob, n // 2, n // 2)
    else:  # independent query per rank
        goal = syn.free_interior_cell_near(ob, int(rng.uniform(0.3, 0.7) * n),
                                           int(rng.uniform(0.3, 0.7) * n))
    start = syn.free_interior_cell_near(ob, n // 8, n // 8)
    tile, pitch, rows = dev.geometry()

    retries = {"resident": 0, "cabi": 0, "class": 0}

    def guarded(what, fn):
        """A plan that fails (the solver reports its own defects, e.g. a grid barrier that timed out)
        is logged, counted and run again inside the timed region, at most three times per arm: the
        other ranks are waiting in a collective and must not be left there."""
        try:
            return fn()
        except (RuntimeError, AssertionError) as e:
            retries[what] += 1
            print("[bench] rank %d: %s plan failed (%s), running it again" % (rank, what, e), file=sys.stderr,
                  flush=True)
            if retries[what] > 3:
                raise
            # the conservative variants for the rest of the run: streamed solves cut by phase count
            # instead of on the copy engine's word, the matrix copied after the solve
            os.environ["DYMU_STREAM_PHASES"] = "40"
            if what == "cabi":
                dev.set_total_cost_export(None)
            return fn()

    def plan():
        st = dev.solve_total_cost([goal])
        wps, status = dev.extract_global_path(float(start[0]), float(start[1]), 0.4, goal[0],
                                              goal[1])
        return st, wps, status

    # ---- resident-input arm -----------------------------------------------------------
    for _ in range(args.warmup):
        st, wps, status = guarded("resident", plan)
    reached = dev.count_reached()
    assert reached >= 0.90 * n * n, "goal is walled in: only %.3f of the map reached" % (
        reached / float(n * n))
    sampler = ClockSampler(D.local_rank)
    D.barrier()
    if rank == 0:
        sampler.start()
    launches0 = dev.launches
    kernel_ms, tiles, updates, outers, written = [], [], [], [], []
    dev.event_record(0)
    for _ in range(args.steps):
        st, wps, status = guarded("resident", plan)
        kernel_ms.append(st["kernel_ms"])
        tiles.append(st["tile_activations"])
        updates.append(st["cell_updates"])
        outers.append(st["outer_iterations"])
        written.append(st["cells_written"])
    dev.event_record(1)
    total_ms = dev.event_elapsed_ms(0, 1)
    launches = dev.launches - launches0
    D.barrier()
    clocks = sampler.stop() if rank == 0 else None
    nwp = len(wps)
    outputs = None
    if args.dump_outputs and rank == 0:
        stride = 1
        while ((n + stride - 1) // stride) ** 2 * 8 > 48 << 20:
            stride += 1
        T = dev.download_total_cost(xform=pkg.cuda_api.XFORM_INF_TO_MINUS1)
        outputs = {"total_cost": np.ascontiguousarray(T[::stride, ::stride]), "path": wps}

    # ---- end-to-end, C ABI: host buffers in, host matrix out, every step ----------------
    cost_host = torch.empty((n, n), dtype=torch.float64).pin_memory()
    # the host-side input of a plan is the cost map a caller would hand to setCostMap: obstacles
    # carry cost <= 0 (getGlobalCostMatrix convention, G.cpp:815-829), so it is self-contained
    dev.download_plane("cost", xform=pkg.cuda_api.XFORM_EFFECTIVE_COST, out=cost_host.numpy())
    t_host = torch.empty((n, n), dtype=torch.float64).pin_memory()

    # the matrix is page-locked: the solve kernel stores each tile into it as soon as the front
    # is past the tile (dymu_set_total_cost_export), download_*_begin/_end then have nothing to copy
    direct = dev.set_total_cost_export(t_host.numpy(), xform=pkg.cuda_api.XFORM_INF_TO_MINUS1)
    def plan_cabi():
        st_ = dev.plan_streamed(cost_host.numpy(), goal)
        dev.download_total_cost_begin(t_host.numpy(), xform=pkg.cuda_api.XFORM_INF_TO_MINUS1)
        dev.extract_global_path(float(start[0]), float(start[1]), 0.4, goal[0], goal[1])
        dev.download_total_cost_end()
        return st_

    for _ in range(min(2, args.warmup)):
        guarded("cabi", plan_cabi)
    D.barrier()
    dev.event_record(2)
    for _ in range(args.steps):
        st_cabi = guarded("cabi", plan_cabi)
    dev.event_record(3)
    dev.set_total_cost_export(None)
    cabi_ms = dev.event_elapsed_ms(2, 3)
    D.barrier()
    t_check = t_host.numpy().copy() if rank == 0 else None
    # copy rates of this rank's host link, all ranks copying at the same time (what the e2e step
    # has to hide; on one GPU this is the rate of the link alone)
    D.barrier()
    dev.event_record(4)
    dev.upload_plane("cost", cost_host.numpy())
    dev.event_record(5)
    dev.download_total_cost(out=t_host.numpy())
    dev.event_record(6)
    h2d_gbs = n * n * 8 / (dev.event_elapsed_ms(4, 5) * 1e-3) / 1e9
    d2h_gbs = n * n * 8 / (dev.event_elapsed_ms(5, 6) * 1e-3) / 1e9
    dev.close()

    # ---- end-to-end, through the drop-in class (the call a user of the reference makes) ----
    # DyMuPathPlanner::setCostMap(const double*, ld) -> computeEntireTotalCostMap() -> getPath()
    # -> getTotalCostMatrix(double*, ld) via libdymu_b200.so
    pl = pkg.DyMuPathPlanner(1.0, 1.5, 2.0, pkg.planner_api.SWEEPING)
    assert pl.initGlobalLayer(1.0, 0.1, n, n), "initGlobalLayer failed"
    assert pl.setCostMapFlat(cost_host.numpy())
    assert pl.setGoal(float(goal[0]), float(goal[1]))
    assert pl.setTotalCostMatrixTarget(t_host.numpy())

    def plan_class():
        ok = pl.setCostMapFlat(cost_host.numpy())
        ok = ok and pl.computeEntireTotalCostMap()
        path = pl.getPath(float(start[0]), float(start[1]))
        ok = ok and pl.getTotalCostMatrixFlat(t_host.numpy())
        assert ok
        return len(path)

    for _ in range(max(1, min(2, args.warmup))):
        nwp_class = guarded("class", plan_class)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        nwp_class = guarded("class", plan_class)
    torch.cuda.synchronize()
    class_ms = (time.perf_counter() - t0) * 1e3
    D.barrier()
    if rank == 0:
        # the class delivered the same matrix as the C-ABI arm (inf -> -1 in both); getPath appends
        # the goal waypoint (G.cpp:589-611), the raw C-ABI path does not
        with np.errstate(invalid="ignore"):
            same = np.array_equal(t_check < 0, t_host.numpy() < 0)
        assert same and abs(nwp_class - nwp) <= 1, ("class e2e arm disagrees with the C-ABI arm: unreached mask equal "
                                           "%s (%d vs %d cells), waypoints %d vs %d"
                                           % (same, int((t_check < 0).sum()), int((t_host.numpy() < 0).sum()),
                                              nwp_class, nwp))
    pl.setTotalCostMatrixTarget(None)
    pl.close()

    total_ms, cabi_ms, class_ms = D.max([total_ms, cabi_ms, class_ms])
    rates = D.gather([h2d_gbs, d2h_gbs])
    if rank != 0:
        return None
    ms_per_step = total_ms / args.steps
    value = world * 1e3 / ms_per_step
    peak, peak_src = measured_peak()
    k_ms = statistics.mean(kernel_ms)
    # SURVEY.md section 8(d): (i) 24 B per cell update (read C_eff, read T, write T) x the cell
    # updates one launch performs -- the figure `achieved` is built from; (ii) 16 B per reached
    # cell per solve, the lower bound.
    algo_bytes = statistics.mean(updates) * CELL_SWEEP_BYTES
    achieved = algo_bytes / (k_ms * 1e-3) / 1e9
    solve_bytes = SOLVE_BYTES_PER_CELL * reached
    # live DRAM-side figure from the kernel's own counters: every activation stages T, C_eff and
    # the 4 x 32 halo cells of its tile, and stores back the cells that changed.  This is what
    # crosses between L2 and the SMs -- an upper bound of the DRAM traffic (part of it hits in
    # the 126 MB L2); the ncu capture of this round sits beside it.
    staged = statistics.mean(tiles) * (2 * tile * tile + 4 * tile) * 8
    stored = statistics.mean(written) * 8
    ncu = _ncu_traffic()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": "configs[2]: %dx%d synthetic Mars-like DEM cost map (device computeCostMap), "
                        "isotropic upwind FMM total-cost solve + gradient-descent path, 1 goal per "
                        "GPU" % (n, n),
            "seed": args.seed, "tile": tile, "obstacle_fraction": float(ob.mean()),
            "reached_fraction": reached / float(n * n), "waypoints": nwp,
            "l2": "inputs larger than L2 (each fp64 plane %.0f MB > 126 MB L2)" % (n * n * 8 / 1e6),
            "parallelism": "1 independent plan per GPU, no collective",
            "streamed_solve_cut": ("after %s / 2 x %s phases (DYMU_STREAM_PHASES)"
                                   % ((os.environ["DYMU_STREAM_PHASES"],) * 2)
                                   if os.environ.get("DYMU_STREAM_PHASES") else
                                   "when the copy engine reports the next part of the cost map"),
            "rank_core_affinity": affinity,
        },
        "solve_ms_per_4096_map": k_ms,
        "solve_kernel_ms": k_ms,
        "gcell_updates_per_s": statistics.mean(updates) / (k_ms * 1e-3) / 1e9,
        "updates_per_cell": statistics.mean(updates) / float(n * n),
        "activations_per_tile": statistics.mean(tiles) / float((pitch // tile) * (rows // tile)),
        "outer_iterations": statistics.mean(outers),
        "roofline": {
            "bound": "hbm", "kernel": "k_fim<%d,0> (tile FIM sweep)" % tile,
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": (ncu or {}).get("dram_bytes_per_launch"),
            "traffic_ncu": ncu,
            "traffic_live": {"bytes": staged + stored, "staged_bytes": staged, "stored_bytes": stored,
                             "gbs": (staged + stored) / (k_ms * 1e-3) / 1e9,
                             "definition": "tile activations x (2 x %d^2 + 4 x %d) x 8 B staged + cells "
                                           "written back x 8 B, both counted by the kernel in this run; "
                                           "L2<->SM bytes, an upper bound of the DRAM bytes" % (tile, tile)},
            "dram_frac": (((ncu or {}).get("dram_bytes_per_launch") or (staged + stored))
                          / (k_ms * 1e-3) / 1e9 / peak),
            "peak_source": peak_src,
            "algorithmic_bytes_per_launch": algo_bytes,
            "definition": "SURVEY 8(d)(i): cell updates x 24 B (read C_eff, read T, write T) / kernel "
                          "time.  The updates of an activated tile run in shared memory, so `frac` "
                          "measures on-chip stencil work, not HBM use: `dram_frac` (measured DRAM bytes "
                          "/ time / peak) is the honest HBM figure and it is < 1 %% -- the solve is "
                          "bounded by dependency latency (DESIGN.md section 5)",
            "solve_level": {"bytes": solve_bytes,
                            "achieved": solve_bytes / (k_ms * 1e-3) / 1e9,
                            "frac": solve_bytes / (k_ms * 1e-3) / 1e9 / peak,
                            "definition": "SURVEY 8(d)(ii): 16 B x reached cells / solve time "
                                          "(lower bound: 41 us at peak)"},
        },
        "e2e": {"value": world * 1e3 / (class_ms / args.steps), "unit": UNIT,
                "ms_per_step": class_ms / args.steps,
                "h2d_bytes_per_step": n * n * 8, "d2h_bytes_per_step": n * n * 8 + nwp * 32,
                "plans_run_again_after_a_solver_error": retries["class"],
                "api": "DyMuPathPlanner::setCostMap(const double*, ld) -> computeEntireTotalCostMap() -> "
                       "getPath() -> getTotalCostMatrix(double*, ld) through libdymu_b200.so, pinned "
                       "host buffers (the cost map is uploaded while the solve starts, the matrix is stored "
                       "by the solve kernel tile by tile), wall clock around the synchronous calls (max "
                       "over ranks)"},
        "e2e_cabi": {"value": world * 1e3 / (cabi_ms / args.steps), "unit": UNIT,
                     "ms_per_step": cabi_ms / args.steps,
                     "plans_run_again_after_a_solver_error": retries["cabi"],
                     "api": "dymu_set_total_cost_export + dymu_plan_streamed + dymu_download_total_cost_begin/"
                            "_end + dymu_extract_global_path (include/dymu_cuda.h), CUDA events",
                     "matrix_delivery": {"direct": bool(direct),
                                         "tiles_stored_during_solve": st_cabi["tiles_delivered_early"],
                                         "tiles_stored_after_last_phase": st_cabi["tiles_delivered_late"],
                                         "solve_kernel_ms": st_cabi["kernel_ms"]}},
        "link_gbs_per_rank": [{"h2d": r[0], "d2h": r[1]} for r in rates],
        "gpu_launches": int(launches),
        "plans_run_again_after_a_solver_error": retries["resident"],
        "clocks": clocks,
    }
    return line, (elev, terr, lut, slopes, locs), outputs


def dump_outputs(out_dir, outputs):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def stencil_leg(args, D, pkg):
    """the streaming (HBM-bound) stencil kernels of the same path, timed once each"""
    n = args.size
    peak, _ = measured_peak()
    try:
        dev = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1, device=D.local_rank)
        dev.set_cost_map(np.ones((n, n)))
        tile, pitch, rows = dev.geometry()
        sm = dev.time_stencils()
        dev.close()
        cells, pcells = float(n * n), float(pitch * rows)
        spec = [("k_fill_f64 (total-cost reset)", sm[0], 8 * cells),
                ("k_ceff (C_eff build)", sm[1], 33 * pcells),
                ("k_readback (inf -> -1)", sm[2], 16 * cells),
                ("k_set_cost_map (obstacle mask)", sm[3], 8 * cells)]
        return {nm: {"ms": ms_, "algorithmic_bytes": b, "gbs": b / (ms_ * 1e-3) / 1e9,
                     "frac_of_measured_peak": b / (ms_ * 1e-3) / 1e9 / peak}
                for nm, ms_, b in spec if ms_ > 0}
    except Exception as e:  # informational
        return {"error": str(e)}


def config2_repair(args, D, pkg):
    """configs[1]: 1000x1000 global layer + local repair after injected obstacles, both repairing
    approaches, through DyMuPathPlanner; the UNMODIFIED reference is timed beside it in the same
    process on identical calls (rank 0 only: the local layer does not shard -- replicas only)."""
    if D.rank != 0:
        return None
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import scenarios as sc
    syn = pkg.synthetic
    n = 1000
    out = {"workload": "configs[1]: 1000x1000 Mars-like map, goal (800,800), start (200,200), "
                       "computeTotalCostMap + getPath, 120x120 px frame with an obstacle disc on path[10] "
                       "+ 3 random discs (seed 7), computeLocalPlanning", "approaches": {}}
    ref_lib = None
    if not args.no_cpu_baseline:
        try:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import oracle
            ref_lib = oracle.reference() if oracle.have_reference() else None
        except Exception:
            ref_lib = None
    for approach, name in ((pkg.planner_api.SWEEPING, "SWEEPING"), (pkg.planner_api.CONSERVATIVE, "CONSERVATIVE")):
        rec = {}
        reps = 5
        t_rep, traj = [], None
        for _ in range(reps):        # a repair changes the planner's state: fresh planner per run
            p = sc.make_planner(pkg.DyMuPathPlanner, approach, n, n)
            g = sc.global_scenario(p, syn, n, n, seed=args.seed)
            c = g["path"][0, :2]
            img = _config2_frame(syn, g["path"], 7)
            t0 = time.perf_counter()
            repaired, traj, _ = p.computeLocalPlanning(c[0], c[1], img, 0.1)
            t_rep.append((time.perf_counter() - t0) * 1e3)
            ridx = p.getReconnectingIndex()
            p.close()
        rec["b200"] = {"repair_ms": statistics.median(t_rep), "repair_ms_all": t_rep, "repaired": bool(repaired),
                       "trajectory_waypoints": int(len(traj)), "reconnecting_index": int(ridx)}
        if ref_lib is not None:
            p = sc.make_planner(ref_lib.DyMuPathPlanner, approach, n, n)
            t0 = time.perf_counter()
            g = sc.global_scenario(p, syn, n, n, seed=args.seed)
            t_global_ref = time.perf_counter() - t0
            c = g["path"][0, :2]
            img = _config2_frame(syn, g["path"], 7)
            t0 = time.perf_counter()
            repaired_r, traj_r, _ = p.computeLocalPlanning(c[0], c[1], img, 0.1)
            t_ref = (time.perf_counter() - t0) * 1e3
            rec["reference"] = {"repair_ms": t_ref, "repaired": bool(repaired_r),
                                "trajectory_waypoints": int(len(traj_r)),
                                "reconnecting_index": int(p.getReconnectingIndex()),
                                "global_setup_s": t_global_ref, "cores": 1, "kind": "reference"}
            rec["speedup_vs_reference"] = t_ref / rec["b200"]["repair_ms"]
            same = (traj_r.shape == traj.shape and float(np.max(np.abs(traj_r[:, :2] - traj[:, :2]))) <= 1e-3
                    and rec["reference"]["reconnecting_index"] == rec["b200"]["reconnecting_index"])
            rec["same_trajectory_as_reference"] = bool(same)
            p.close()
        out["approaches"][name] = rec
    return out


def _config2_frame(syn, path, seed):
    c = path[0, :2]
    d = path[min(10, len(path) - 2), :2]
    rng = np.random.default_rng(seed)
    discs = [(d[0], d[1], 0.8)]
    discs += [(c[0] + rng.uniform(-4, 4), c[1] + rng.uniform(-4, 4), rng.uniform(0.2, 0.5)) for _ in range(3)]
    return syn.obstacle_frame(120, 120, 0.1, c, discs)


def queries2048(args, D, pkg):
    """configs[3]: `--queries` independent goal queries (full solve + path each) on one shared
    2048x2048 map, block-sharded over the ranks (no data-path collective), `--batch` goals per
    launch.  Strong scaling: the total work is fixed."""
    syn, sh = pkg.synthetic, pkg.sharding
    n = 2048
    elev, terr, lut, slopes, locs = build_workload(pkg, n, args.seed)
    dev = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1, device=D.local_rank)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    ob = dev.download_plane_u8("obstacle")
    rng_g, rng_s = np.random.default_rng(11), np.random.default_rng(13)
    goals = [syn.free_interior_cell_near(ob, int(rng_g.uniform(0.03, 0.97) * n),
                                         int(rng_g.uniform(0.03, 0.97) * n)) for _ in range(args.queries)]
    starts = [syn.free_interior_cell_near(ob, int(rng_s.uniform(0.03, 0.97) * n),
                                          int(rng_s.uniform(0.03, 0.97) * n)) for _ in range(args.queries)]
    mine = list(sh.shard_queries(args.queries, D.world, D.rank))
    B = max(1, min(args.batch, len(mine)))
    dev.reserve_slots(B)

    def run(idx_all):
        nwp, kms = 0, 0.0
        for lo in range(0, len(idx_all), B):
            idx = idx_all[lo:lo + B]
            st = dev.solve_total_cost([goals[q] for q in idx])
            kms += st["kernel_ms"]
            paths, _ = dev.extract_global_path_batch(
                list(range(len(idx))), [[float(starts[q][0]), float(starts[q][1])] for q in idx], 0.4,
                [goals[q] for q in idx], cap=1 << 14)
            nwp += sum(len(w) for w in paths)
        return nwp, kms

    run(mine[:B])                      # warm-up: one batch
    D.barrier()
    launches0 = dev.launches
    dev.event_record(0)
    nwp, kms = run(mine)
    dev.event_record(1)
    ms = dev.event_elapsed_ms(0, 1)
    launches = dev.launches - launches0
    dev.close()
    ms, kms = D.max([ms, kms])
    if D.rank != 0:
        return None
    return {"workload": "configs[3]: %d independent goal queries (solve + path) on one shared 2048x2048 "
                        "map, %d goals per launch, block-sharded over %d GPU(s)" % (args.queries, B, D.world),
            "plans_per_s": args.queries / (ms * 1e-3), "ms_total": ms, "max_rank_solve_kernel_ms": kms,
            "queries": args.queries, "n_gpus": D.world, "scaling": "strong", "gpu_launches_rank0": int(launches),
            "waypoints_rank0": int(nwp)}


def dd16384(args, D, pkg):
    """configs[4]: one 16384x16384 grid (periodic 4096^2 fBm cost tile, goal near the centre).
    1 GPU: the plain single-grid solve (scaling base).  N >= 2: row strips, one per rank, halo rows
    exchanged between bounded bursts of solver phases (sharding.dd_solve_pipelined); every rank
    then solves the whole grid alone and checks its strip against it (`verified`)."""
    torch = D.torch
    sh, api, syn = pkg.sharding, pkg.cuda_api, pkg.synthetic
    n, base = args.dd_size, min(4096, args.dd_size)
    tile = syn.smooth_cost_map(base, base, seed=args.seed, obstacle_fraction=0.03)   # periodic (FFT fBm)
    reps = n // base
    g0 = syn.free_interior_cell_near(tile <= 0, base // 2, base // 2)
    goal = (g0[0] + (reps // 2) * base, g0[1] + (reps // 2) * base)
    whole = api.DeviceLayer(n, n, device=D.local_rank)
    whole.set_cost_map(np.tile(tile, (reps, reps)))
    whole.solve_total_cost([goal])                                   # warm-up
    st1 = whole.solve_total_cost([goal])
    single_ms = st1["kernel_ms"]
    rec = {"workload": "configs[4]: %dx%d single grid, goal near the centre" % (n, n), "n_gpus": D.world,
           "single_gpu_solve_ms": None, "strips": None}
    if D.world == 1:
        whole.close()
        rec["single_gpu_solve_ms"] = single_ms
        rec["updates_per_cell"] = st1["cell_updates"] / float(n * n)
        return rec
    lay = sh.StripLayout(n, D.world, D.rank)
    rows = np.arange(lay.r0, lay.r1) % base
    strip = sh.CudaStrip(api, lay, n, np.tile(tile[rows], (1, reps)), D.local_rank, torch)
    comm = sh.TorchComm(D.rank, D.world, torch.device("cuda", D.local_rank))
    times, rounds, kms = [], 0, 0.0
    for _ in range(2):
        n0 = len(strip.stats)
        D.barrier()
        t0 = time.perf_counter()
        rounds = sh.dd_solve_pipelined(strip, comm, goal, args.dd_phases)
        torch.cuda.synchronize()
        D.barrier()
        times.append((time.perf_counter() - t0) * 1e3)
        kms = sum(s["kernel_ms"] for s in strip.stats[n0:])
    T_whole = whole.download_total_cost()
    T1 = T_whole[lay.r0:lay.r1]
    Tk = strip.own_rows()
    fin = np.isfinite(T1) & (T1 > 0)
    err = float(np.max(np.abs(Tk[fin] - T1[fin]) / T1[fin])) if fin.any() else 0.0
    good = 1.0 if (np.array_equal(np.isinf(Tk), np.isinf(T1)) and err <= 1e-12) else 0.0
    whole.close()
    strip.dev.close()
    wall, kmax, single, neg_good, errmax = D.max([min(times), kms, single_ms, -good, err])
    D.host_barrier("dd_torch_done")
    # the same decomposition behind ONE C-ABI call: rank 0 drives all N GPUs (one host thread per
    # strip, boundary rows copied GPU to GPU) while the other ranks wait
    cabi = None
    if D.rank == 0:
        try:
            layers, cuts = [], [0]
            for r in range(D.world):
                lr = sh.StripLayout(n, D.world, r)
                d = api.DeviceLayer(n, lr.ny_local, 1.0, 0.1, device=r)
                rr = np.arange(lr.r0, lr.r1) % base
                d.set_cost_map(lr.local_cost(np.tile(tile[rr], (1, reps))))
                layers.append((d, lr))
                cuts.append(lr.r1)
            unpin()   # one host thread per strip: they need a core each
            api.dd_solve([d for d, _ in layers], cuts, goal, args.dd_phases)      # warm-up
            sweep = {}
            for ph in sorted({8, 16, args.dd_phases}):
                sweep[ph] = min((api.dd_solve([d for d, _ in layers], cuts, goal, ph) for _ in range(2)),
                                key=lambda q: q["wall_ms"])
            best_ph = min(sweep, key=lambda ph: sweep[ph]["wall_ms"])
            best = sweep[best_ph]
            Tc = np.vstack([d.download_total_cost()[lr.first_own:lr.last_own + 1] for d, lr in layers])
            finw = np.isfinite(T_whole) & (T_whole > 0)
            errc = float(np.max(np.abs(Tc[finw] - T_whole[finw]) / T_whole[finw]))
            cabi = {"wall_ms": best["wall_ms"], "max_rank_kernel_ms": best["max_kernel_ms"],
                    "sum_kernel_ms": best["sum_kernel_ms"], "exchange_rounds": best["rounds"],
                    "phases_per_round": best_ph,
                    "wall_ms_by_phases_per_round": {str(ph): sweep[ph]["wall_ms"] for ph in sweep},
                    "verified": bool(np.array_equal(np.isinf(Tc), np.isinf(T_whole)) and errc <= 1e-12),
                    "max_rel_err_vs_single_grid": errc,
                    "updates_per_cell": best["cell_updates"] / float(n * n),
                    "driver": "dymu_dd_solve (include/dymu_cuda.h): one process, one host thread per strip, "
                              "cudaMemcpyPeerAsync rows, host barrier per round"}
            for d, _ in layers:
                d.close()
        except Exception as e:
            cabi = {"error": "%s: %s" % (type(e).__name__, e)}
    D.host_barrier("dd_cabi_done")
    if D.rank != 0:
        return None
    rec["single_gpu_solve_ms"] = single
    rec["strips"] = cabi
    rec["strips_torch"] = {"wall_ms": wall, "max_rank_kernel_ms": kmax, "exchange_rounds": rounds,
                           "phases_per_round": args.dd_phases, "verified": bool(neg_good == -1.0),
                           "max_rel_err_vs_single_grid": errmax,
                           "driver": "sharding.dd_solve_pipelined: one rank per GPU, torch.distributed (NCCL) "
                                     "point-to-point rows, all-reduce vote per round"}
    return rec


class Watchdog:
    """A leg that does not come back (a deadlocked kernel, a rank that died inside a collective) must
    not take the whole line with it: when a leg overruns its allowance, rank 0 prints the line as far
    as it got, marked `incomplete`, and every rank leaves (ctypes calls release the GIL, so this
    thread runs while the main thread is stuck in one)."""
    ALLOWANCE = {"plan4096": 300.0, "config2_repair": 180.0, "queries2048": 420.0, "dd16384": 240.0}

    def __init__(self, rank):
        import threading
        self.rank, self.leg, self.t0, self.line = rank, None, 0.0, None
        self.lock = threading.Lock()
        t = threading.Thread(target=self._run, daemon=True)
        t.start()

    def enter(self, leg):
        with self.lock:
            self.leg, self.t0 = leg, time.perf_counter()
        print("[bench] rank %d: %s ..." % (self.rank, leg), file=sys.stderr, flush=True)

    def leave(self):
        with self.lock:
            if self.leg:
                print("[bench] rank %d: %s done in %.1f s" % (self.rank, self.leg, time.perf_counter() - self.t0),
                      file=sys.stderr, flush=True)
            self.leg = None

    def _run(self):
        while True:
            time.sleep(1.0)
            with self.lock:
                leg, t0, line = self.leg, self.t0, self.line
            if leg and time.perf_counter() - t0 > self.ALLOWANCE.get(leg, 300.0):
                msg = "leg %s did not return within %.0f s on rank %d" % (leg, self.ALLOWANCE.get(leg, 300.0),
                                                                           self.rank)
                print("[bench] " + msg + ": giving up", file=sys.stderr, flush=True)
                if self.rank == 0 and line is not None:
                    line = dict(line)
                    line["incomplete"] = msg
                    print(json.dumps(line), flush=True)
                    os._exit(0)
                os._exit(0 if self.rank != 0 else 3)


def run_b200(args):
    import dymu_b200
    D = Dist()
    dog = Watchdog(D.rank)
    if D.world > 1:
        # The hand-back of a streamed solve on the copy engine's word was re-verified on one GPU only
        # after its race was fixed (DESIGN.md section 7); with several ranks the launches of a
        # streamed solve are cut by phase count, the variant every multi-GPU line so far was taken with.
        os.environ.setdefault("DYMU_STREAM_PHASES", "40")
    affinity = pin_rank(D.local_rank, D.world)
    pkg = dymu_b200.load()
    want = set(args.workload.split(",")) if args.workload != "all" else {"plan4096", "config2", "queries2048",
                                                                        "dd16384"}
    line, maps = None, None
    if "plan4096" in want:
        dog.enter("plan4096")
        res = headline_plan4096(args, D, pkg, affinity)
        dog.leave()
        if D.rank == 0:
            line, maps, outputs = res
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, outputs)
            line["stencils"] = stencil_leg(args, D, pkg)
            if not args.no_cpu_baseline and D.world == 1:
                line["cpu_baseline"] = cpu_baseline_leg(pkg, *maps, args.size)
    elif D.rank == 0:
        line = {"metric": METRIC, "unit": UNIT, "n_gpus": D.world, "note": "sub-benchmarks only"}
    extra = {}
    for name, fn in (("config2_repair", config2_repair), ("queries2048", queries2048), ("dd16384", dd16384)):
        key = {"config2_repair": "config2", "queries2048": "queries2048", "dd16384": "dd16384"}[name]
        if key not in want:
            continue
        t0 = time.perf_counter()
        if D.rank == 0 and line is not None:
            dog.line = dict(line, **extra)
        dog.enter(name)
        try:
            rec = fn(args, D, pkg)
        except Exception as e:  # a sub-benchmark must not take the headline line down with it
            rec = {"error": "%s: %s" % (type(e).__name__, e)}
        D.host_barrier("after_" + name)
        dog.leave()
        if D.rank == 0 and rec is not None:
            rec["bench_seconds"] = time.perf_counter() - t0
            extra[name] = rec
    if D.rank == 0:
        line.update(extra)
        print(json.dumps(line))
    D.close()
    return 0


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        sys.exit(run_reference(a))
    sys.exit(run_b200(a))
