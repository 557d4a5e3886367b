"""Developer probe: cost of obstacle clearance on the 4096^2 benchmark map.

    python scripts/probe_clearance.py [n] [--runs R] [--out DIR]

Map, goal and start as in scripts/probe_aniso.py (bench.py's generator and seed).
  * Clearance build: for R = 4, 32 and 128 cells (radius + margin = R + 0.5 m, radius = margin),
    20 rebuilds each (every dymu_set_obstacle_clearance followed by a C_eff refresh runs both passes,
    the row pass fused with C_eff); device time of k_clear_cols and k_clear_rows from torch.profiler.
  * C_eff-only refresh (hazard changed, obstacles did not): k_ceff_clear, 20 refreshes.
  * Solve: four contexts -- clearance off / on (radius 2, margin 6, penalty 4), each isotropic and
    with the slope-anisotropy table of probe_aniso.py -- solved in alternation R times: solve kernel
    ms (CUDA events), phases, tile activations.
Bytes per padded cell each pass must move are stated beside its rate.  The card name and power limit
are read in the same run.  The JSON summary goes to DIR/probe_clearance.json."""
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
RMP = (2.0, 6.0, 4.0)

ap = argparse.ArgumentParser()
ap.add_argument("n", type=int, nargs="?", default=4096)
ap.add_argument("--runs", type=int, default=3)
ap.add_argument("--out", default=".")
args = ap.parse_args()

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

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


def layer(clear, aniso):
    d = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    d.compute_cost_map(lut, slopes, len(locs), elev, terr)
    if clear:
        d.set_obstacle_clearance(*RMP)
    if aniso:
        d.set_anisotropy(*TABLE)
    return d


def kernel_ms(prof, name):
    us = [e.device_time for e in prof.events() if name in e.name]
    return (float(np.median(us)) / 1e3 if us else float("nan")), len(us)


summary = {"card": card, "power_limit": power, "n": n, "clearance": RMP, "table": TABLE}
d = layer(True, False)
_, pitch, prow = d.geometry()
cells = pitch * prow
reps = 20
d.download_plane("ceff")  # warm-up
for R in (4, 32, 128):
    reach = R + 0.5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            d.set_obstacle_clearance(reach / 2, reach / 2, 1.0)
            d.download_plane("ceff")
        d.synchronize()
    cols_ms, nc = kernel_ms(prof, "k_clear_cols")
    rows_ms, nr = kernel_ms(prof, "k_clear_rows")
    # column pass: the obstacle bytes twice with the 2R overlap of its 256-row strips, gcol written twice
    # and read once; fused row pass: gcol (and its halo) + cost, hazard, trafficability, obstacle read,
    # clearance and C_eff written
    cols_b = 2.0 * (1 + 2.0 * R / 256) + 3.0
    rows_b = 1.0 + 2.0 * R / 256 + 25.0 + 16.0
    row = dict(R=R, cols_ms=cols_ms, rows_ms=rows_ms, build_ms=cols_ms + rows_ms, launches=(nc, nr),
               cols_bytes_per_cell=cols_b, rows_bytes_per_cell=rows_b,
               cols_gbs=cols_b * cells / (cols_ms * 1e-3) / 1e9, rows_gbs=rows_b * cells / (rows_ms * 1e-3) / 1e9)
    summary["build_R%d" % R] = row
    print("build", json.dumps(row), flush=True)

d.set_obstacle_clearance(*RMP)
d.download_plane("ceff")
haz = d.read_rect("hazard_density", 10, 10, 1, 1)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for k in range(reps):
        d.write_rect("hazard_density", 10, 10, haz + (k % 2) * 0.01)
        d.download_plane("ceff")
    d.synchronize()
ms, nk = kernel_ms(prof, "k_ceff_clear")
summary["ceff_only"] = dict(ms=ms, launches=nk, bytes_per_cell=41.0, gbs=41.0 * cells / (ms * 1e-3) / 1e9)
print("k_ceff_clear", json.dumps(summary["ceff_only"]), flush=True)
del d

devs = {"off": layer(False, False), "on": layer(True, False), "off_aniso": layer(False, True),
        "on_aniso": layer(True, True)}
ob = devs["off"].download_plane_u8("obstacle")
blocked = ob.astype(bool) | (devs["on"].download_plane("clearance") <= RMP[0])
goal = syn.free_interior_cell_near(blocked, n // 2, n // 2)
summary["goal"] = goal
rows = {k: [] for k in devs}
for d in devs.values():  # warm-up
    d.solve_total_cost([goal])
order = list(devs)
for r in range(args.runs):
    for name in (order if r % 2 == 0 else order[::-1]):
        st = devs[name].solve_total_cost([goal])
        row = dict(solve_ms=st["kernel_ms"], phases=st["outer_iterations"], activations=st["tile_activations"],
                   converged=st["converged"])
        rows[name].append(row)
        print(name, json.dumps(row), flush=True)
summary["runs"] = rows
for name in rows:
    for key in ("solve_ms", "phases", "activations"):
        summary["%s_%s_mean" % (name, key)] = float(np.mean([r[key] for r in rows[name]]))
os.makedirs(args.out, exist_ok=True)
with open(os.path.join(args.out, "probe_clearance.json"), "w") as f:
    json.dump(summary, f, indent=1)
print(json.dumps({k: v for k, v in summary.items() if k.endswith("_mean")}), flush=True)
