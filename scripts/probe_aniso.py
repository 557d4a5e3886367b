"""Developer probe: cost of the slope-anisotropic solve on the 4096^2 benchmark map.

    python scripts/probe_aniso.py [n] [--runs R] [--out DIR]

Two contexts on the same map and goal (bench.py's generator and seed, goal nearest the centre,
start nearest (n // 8, n // 8)), one isotropic and one with the table below, solved in
alternation R times each.  Per run: solve kernel ms (CUDA events around the cooperative launch),
phases, tile activations, updates per cell; path kernel ms and waypoint count.  k_dircost: its
device time from torch.profiler over 20 rebuilds, and the bandwidth of its 48 B per cell (elevation
and C_eff read, four planes written).  The card name and power limit are read in the same run.
The JSON summary goes to DIR/probe_aniso.json (default: the current directory)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import dymu_b200  # noqa: E402

TABLE = ([-20.0, -5.0, 0.0, 10.0, 25.0], [0.6, 0.8, 1.0, 1.8, 3.5])

ap = argparse.ArgumentParser()
ap.add_argument("n", type=int, nargs="?", default=4096)
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
syn = pkg.synthetic
n = args.n
elev, terr = syn.mars_dem(n, n, seed=20261018)
lut, slopes, locs = syn.default_lut()
devs = {}
for name in ("iso", "aniso"):
    d = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    d.compute_cost_map(lut, slopes, len(locs), elev, terr)
    if name == "aniso":
        d.set_anisotropy(*TABLE)
    devs[name] = d
ob = devs["iso"].download_plane_u8("obstacle")
goal = syn.free_interior_cell_near(ob, n // 2, n // 2)
start = syn.free_interior_cell_near(ob, n // 8, n // 8)
free = int(np.count_nonzero(ob == 0))

rows = {"iso": [], "aniso": []}
for name, d in devs.items():  # warm-up of both kernels and paths
    d.solve_total_cost([goal])
    d.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal)
for r in range(args.runs):
    for name in ("iso", "aniso") if r % 2 == 0 else ("aniso", "iso"):
        d = devs[name]
        st = d.solve_total_cost([goal])
        d.event_record(0)
        wps, status = d.extract_global_path(float(start[0]), float(start[1]), 0.4, *goal)
        d.event_record(1)
        row = dict(solve_ms=st["kernel_ms"], phases=st["outer_iterations"], activations=st["tile_activations"],
                   updates_per_cell=st["cell_updates"] / free, path_ms=d.event_elapsed_ms(0, 1),
                   waypoints=len(wps), path_status=status, converged=st["converged"])
        rows[name].append(row)
        print(name, json.dumps(row), flush=True)

# k_dircost alone: every set_anisotropy on a clean C_eff rebuilds the four planes
from torch.profiler import ProfilerActivity, profile  # noqa: E402

d = devs["aniso"]
reps = 20
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(reps):
        d.set_anisotropy(*TABLE)
    d.synchronize()
us = [e.device_time for e in prof.events() if "k_dircost" in e.name]
_, pitch, prow = d.geometry()
cells = pitch * prow
dircost_ms = float(np.median(us)) / 1e3 if us else float("nan")
gbs = 48.0 * cells / (dircost_ms * 1e-3) / 1e9 if us else float("nan")
print("k_dircost: %d launches, median %.3f ms, %.0f GB/s (48 B per padded cell, %d cells)"
      % (len(us), dircost_ms, gbs, cells), flush=True)

summary = {"card": card, "power_limit": power, "n": n, "goal": goal, "start": start, "table": TABLE,
           "runs": rows, "k_dircost_ms": dircost_ms, "k_dircost_gbs": gbs, "k_dircost_launches": len(us)}
for name in rows:
    for key in ("solve_ms", "path_ms", "phases", "activations", "updates_per_cell", "waypoints"):
        summary["%s_%s_mean" % (name, key)] = float(np.mean([r[key] for r in rows[name]]))
os.makedirs(args.out, exist_ok=True)
with open(os.path.join(args.out, "probe_aniso.json"), "w") as f:
    json.dump(summary, f, indent=1)
print(json.dumps({k: v for k, v in summary.items() if k.endswith("_mean")}), flush=True)
