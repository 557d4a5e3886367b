"""Developer probe: throughput of map batches under obstacle clearance and slope anisotropy
(dymu_set_maps_clearance / dymu_set_maps_anisotropy with dymu_solve_maps).

    python scripts/probe_map_terrain.py [--runs R] [--out DIR]

The workloads of scripts/probe_maps.py (seeded synthetic.smooth_cost_map maps, seed 1000 + q): 64 maps at
2048^2 and 256 maps at 1024^2, on a synthetic.mars_dem elevation (seed 7), three settings: clearance
(radius 1, margin 2, penalty 1.5, global_res 1), anisotropy (the table of DESIGN.md section 10) and both.
Arms, run in alternation R times per setting:
  1. solo: one fresh context per map with the same settings (elevation, dymu_set_cost_map, the
     clearance and the table set before timing), dymu_solve_total_cost timed alone -- it includes the
     context's C_eff / clearance / directional-cost refresh the new map needs;
  2. dymu_set_maps + dymu_solve_maps with 16, 32 and 64 maps per launch on one context, the solve timed
     alone -- it includes the adjusted-plane rebuild of the maps just set, the factor planes and the band.
Per arm: maps/s for the solve (host wall clock around calls that end in a synchronise), and the solver's
kernel ms, phases, tile activations summed over the launches, and cell updates per map cell.
The new passes are timed with torch.profiler (CUPTI kernel durations) over one 64-map solve with both
settings on, each as a rate over the bytes it must move:
  k_map_clear_cols   8 B of plain C_eff read twice (plus the 2R-row overlap of the strips), 2 B of gcol
                     written and 1 B read per cell and map
  k_map_clear_rows   1 B gcol + 8 B plain C_eff read, 8 B adjusted C_eff written per cell and map
  k_dirfactor        8 B elevation read, 32 B factors written per cell (once per solve)
  k_map_band         8 B of C_q per cell and map, the 32 B of factors per cell once
The card name and power limit are read in the same run.  The JSON summary goes to DIR/probe_map_terrain.json."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import dymu_b200  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--runs", type=int, default=3)
ap.add_argument("--out", default=".")
args = ap.parse_args()

import torch  # noqa: E402

card = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as e:  # the number is still reported, with what could not be read
    power = "unknown (%s)" % e
print("card: %s, power limit %s" % (card, power), flush=True)

pkg = dymu_b200.load()
api, syn = pkg.cuda_api, pkg.synthetic
CLEAR = (1.0, 2.0, 1.5)
TABLE = ([-20.0, -5.0, 0.0, 10.0, 25.0], [0.6, 0.8, 1.0, 1.8, 3.5])
SETTINGS = {"clearance": (CLEAR, None), "anisotropy": (None, TABLE), "both": (CLEAR, TABLE)}
HBM_GBS = 6546.0  # the bandwidth the other stencils are quoted against (DESIGN.md section 6)


def workload(n, m):
    costs = np.stack([syn.smooth_cost_map(n, n, seed=1000 + q) for q in range(m)])
    rng = np.random.default_rng(n + m)
    goals = []
    for q in range(m):
        ob = costs[q] <= 0
        goals.append(syn.free_interior_cell_near(ob, int(rng.uniform(0.1, 0.9) * n), int(rng.uniform(0.1, 0.9) * n)))
    return costs, goals


def work(stats_list, cells):
    return {"kernel_ms": float(sum(s["kernel_ms"] for s in stats_list)),
            "phases": int(sum(s["outer_iterations"] for s in stats_list)),
            "tile_activations": int(sum(s["tile_activations"] for s in stats_list)),
            "updates_per_map_cell": float(sum(s["cell_updates"] for s in stats_list)) / cells}


def solo_layers(n, costs, elev, clear, table):
    layers = []
    for q in range(len(costs)):
        d = api.DeviceLayer(n, n, 1.0, 0.1)
        d.upload_plane("elevation", elev)
        if clear:
            d.set_obstacle_clearance(*clear)
        if table:
            d.set_anisotropy(*table)
        layers.append(d)
    return layers


def arm_solo(layers, costs, goals):
    t_solve, st = 0.0, []
    for q, d in enumerate(layers):
        d.set_cost_map(costs[q])
        d.synchronize()
        t0 = time.perf_counter()
        st.append(d.solve_total_cost([goals[q]]))
        t_solve += time.perf_counter() - t0
    return t_solve, st


def arm_batch(d, costs, goals, per):
    t_solve, st = 0.0, []
    for q0 in range(0, len(goals), per):
        k = min(per, len(goals) - q0)
        d.set_maps(costs[q0:q0 + k])
        t0 = time.perf_counter()
        st.append(d.solve_maps(goals[q0:q0 + k]))
        t_solve += time.perf_counter() - t0
    return t_solve, st


def pass_rates(d, n, costs, goals):
    """CUPTI durations of the new passes in one 64-map solve with both settings on."""
    m = 64
    d.set_maps(costs[:m])
    d.solve_maps(goals[:m])   # warm
    _, pitch, rows = d.geometry()
    pcells = float(pitch * rows)
    R = int(np.floor((CLEAR[0] + CLEAR[1]) / 1.0))
    bytes_per = {"k_map_clear_cols": m * pcells * (16.0 * (1 + 2.0 * R / 256) + 3.0),
                 "k_map_clear_rows": m * pcells * 17.0,
                 "k_dirfactor": pcells * 40.0,
                 "k_map_band": m * pcells * 8.0 + pcells * 32.0}
    out = {}
    for _ in range(3):
        d.set_maps(costs[:m])
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            d.solve_maps(goals[:m])
            torch.cuda.synchronize()
        for ev in prof.events():
            for name in bytes_per:
                if name in ev.name:
                    us = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
                    out.setdefault(name, []).append(us / 1e3)
    res = {}
    for name, ms_list in out.items():
        # one launch per pass and solve here (64 maps fit one launch); median over the repetitions
        t = float(np.median(ms_list))
        gbs = bytes_per[name] / 1e9 / (t / 1e3)
        res[name] = {"ms": t, "GB_per_s": gbs, "share_of_6546": gbs / HBM_GBS}
    return res


results = {"card": card, "power_limit": power, "runs": args.runs, "workloads": []}
for n, m in ((2048, 64), (1024, 256)):
    costs, goals = workload(n, m)
    elev, _ = syn.mars_dem(n, n, seed=7)
    cells = float(n * n) * m   # the updates are reported per cell of a map
    rec = {"n": n, "maps": m, "settings": {}}
    layers = {}
    for name, (clear, table) in SETTINGS.items():
        solo = solo_layers(n, costs, elev, clear, table)
        one = api.DeviceLayer(n, n, 1.0, 0.1)
        one.upload_plane("elevation", elev)
        if clear:
            one.set_maps_clearance(*clear)
        if table:
            one.set_maps_anisotropy(*table)
        one.reserve_maps(64)
        arm_solo(solo[:2], costs[:2], goals[:2])          # warm-up of every shape
        for per in (16, 32, 64):
            arm_batch(one, costs[:per], goals[:per], per)
        layers[name] = (solo, one)
        rec["settings"][name] = {"solo": [], "batch": {str(p): [] for p in (16, 32, 64)}}
    for r in range(args.runs):
        for name in SETTINGS:                             # the arms alternate within a run
            solo, one = layers[name]
            s = rec["settings"][name]
            ts, st = arm_solo(solo, costs, goals)
            s["solo"].append({"maps_per_s_solve": m / ts, "launches": len(st), **work(st, cells)})
            for per in (16, 32, 64):
                ts, st = arm_batch(one, costs, goals, per)
                s["batch"][str(per)].append({"maps_per_s_solve": m / ts, "launches": len(st), **work(st, cells)})
            print(json.dumps({"n": n, "run": r, "setting": name, "solo": s["solo"][-1],
                              "batch": {p: v[-1] for p, v in s["batch"].items()}}), flush=True)
    rec["passes"] = pass_rates(layers["both"][1], n, costs, goals)
    print(json.dumps({"n": n, "passes": rec["passes"]}), flush=True)
    results["workloads"].append(rec)
    for solo, one in layers.values():
        for d in solo + [one]:
            d.close()

os.makedirs(args.out, exist_ok=True)
with open(os.path.join(args.out, "probe_map_terrain.json"), "w") as f:
    json.dump(results, f, indent=1)
print("card: %s, power limit %s" % (card, power))
