"""Developer probe: throughput of batches of independent cost maps (dymu_solve_maps).

    python scripts/probe_maps.py [--runs R] [--out DIR]

Two workloads of seeded synthetic.smooth_cost_map maps (seed 1000 + q, goals and starts from a seeded
generator): 64 maps at 2048^2 and 256 maps at 1024^2.  Three arms, run in alternation R times:
  1. solo: one map at a time, dymu_set_cost_map + dymu_solve_total_cost (+ dymu_extract_global_path),
     the upload (set_cost_map and a synchronise) and the solve (with its C_eff refresh) timed apart.
     Each map has a context of its own, created before timing (setCostMap only ever adds obstacles,
     so one context reused for different maps would solve the union of their obstacles);
  2. dymu_set_maps + dymu_solve_maps with 16, 32 and 64 maps per launch on one context (+ one
     dymu_extract_global_path_batch per launch);
  3. dymu_batch_solve_maps over every visible GPU, 64 maps per launch (with and without paths).
Per arm: maps/s for the solve alone (not measured for arm 3, one call does everything), with the
upload, and with the path (host wall clock around calls that end in a
synchronise), and the solver's kernel ms, phases, tile activations and cell updates per cell summed
over the launches, beside the sums over the solo solves.  k_map_ceff: dymu_set_maps from one torch
CUDA tensor holding every map (device input, no staging), CUDA events on the context's stream around
the call (the kernel plus a 24 B/map statistics read-back), 8 B read + 8 B written per cell.
The card name and power limit are read in the same run.  The JSON summary goes to DIR/probe_maps.json."""
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
n_gpu = torch.cuda.device_count()
print("card: %s, power limit %s, %d GPU(s)" % (card, power, n_gpu), flush=True)

pkg = dymu_b200.load()
api, syn = pkg.cuda_api, pkg.synthetic
TAU, CAP = 0.4, 1 << 14
HBM_GBS = 6546.0  # the bandwidth the other stencils are quoted against (DESIGN.md section 6)


def workload(n, m):
    costs = np.stack([syn.smooth_cost_map(n, n, seed=1000 + q) for q in range(m)])
    rng = np.random.default_rng(n + m)
    goals, starts = [], []
    for q in range(m):
        ob = costs[q] <= 0
        goals.append(syn.free_interior_cell_near(ob, int(rng.uniform(0.1, 0.9) * n), int(rng.uniform(0.1, 0.9) * n)))
        starts.append(syn.free_interior_cell_near(ob, int(rng.uniform(0.1, 0.9) * n), int(rng.uniform(0.1, 0.9) * n)))
    return costs, goals, starts


def work(stats_list, cells):
    return {"kernel_ms": float(sum(s["kernel_ms"] for s in stats_list)),
            "phases": int(sum(s["outer_iterations"] for s in stats_list)),
            "tile_activations": int(sum(s["tile_activations"] for s in stats_list)),
            "updates_per_cell": float(sum(s["cell_updates"] for s in stats_list)) / cells}


def arm_solo(layers, costs, goals, starts):
    m = len(goals)
    t_set = t_solve = t_path = 0.0
    st = []
    for q in range(m):
        d = layers[q]
        t0 = time.perf_counter()
        d.set_cost_map(costs[q])
        d.synchronize()
        t1 = time.perf_counter()
        st.append(d.solve_total_cost([goals[q]]))  # includes the C_eff refresh the new map needs
        t2 = time.perf_counter()
        d.extract_global_path(float(starts[q][0]), float(starts[q][1]), TAU, goals[q][0], goals[q][1], cap=CAP)
        t3 = time.perf_counter()
        t_set += t1 - t0
        t_solve += t2 - t1
        t_path += t3 - t2
    return t_set, t_solve, t_path, st


def arm_batch(d, costs, goals, starts, per):
    m = len(goals)
    t_set = t_solve = t_path = 0.0
    st = []
    for q0 in range(0, m, per):
        k = min(per, m - q0)
        t0 = time.perf_counter()
        d.set_maps(costs[q0:q0 + k])
        t1 = time.perf_counter()
        st.append(d.solve_maps(goals[q0:q0 + k]))
        t2 = time.perf_counter()
        d.extract_global_path_batch(list(range(k)), [(float(i), float(j)) for i, j in starts[q0:q0 + k]], TAU,
                                    goals[q0:q0 + k], cap=CAP)
        t3 = time.perf_counter()
        t_set += t1 - t0
        t_solve += t2 - t1
        t_path += t3 - t2
    return t_set, t_solve, t_path, st


def arm_multi(layers, costs, goals, starts):
    t0 = time.perf_counter()
    api.batch_solve_maps(layers, costs, goals)
    t1 = time.perf_counter()
    api.batch_solve_maps(layers, costs, goals, starts=starts, tau=TAU, cap=CAP)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def map_ceff_rate(d, costs):
    m, n = costs.shape[0], costs.shape[1]
    dev = torch.from_numpy(costs).to("cuda:0")
    torch.cuda.synchronize()
    _, pitch, rows = d.geometry()
    ms = []
    for _ in range(6):
        d.event_record(0)
        d.set_maps_device(dev.data_ptr(), m, n, n * n)
        d.event_record(1)
        ms.append(d.event_elapsed_ms(0, 1))
    t = float(np.median(ms[1:]))
    gbytes = m * (n * n + pitch * rows) * 8 / 1e9
    return {"maps": m, "ms": t, "GB_per_s": gbytes / (t / 1e3), "share_of_6546": gbytes / (t / 1e3) / HBM_GBS}


results = {"card": card, "power_limit": power, "gpus": n_gpu, "runs": args.runs, "workloads": []}
for n, m in ((2048, 64), (1024, 256)):
    costs, goals, starts = workload(n, m)
    cells = float(n * n)
    solo_layers = [api.DeviceLayer(n, n, 1.0, 0.1) for _ in range(m)]
    one = api.DeviceLayer(n, n, 1.0, 0.1)
    one.reserve_maps(64)
    multi = []
    for k in range(n_gpu):
        layer = api.DeviceLayer(n, n, 1.0, 0.1, device=k)
        layer.reserve_maps(64)
        multi.append(layer)
    # warm-up of every shape
    arm_solo(solo_layers[:2], costs[:2], goals[:2], starts[:2])
    for per in (16, 32, 64):
        arm_batch(one, costs[:per], goals[:per], starts[:per], per)
    arm_multi(multi, costs[:64], goals[:64], starts[:64])
    rec = {"n": n, "maps": m, "solo": [], "batch": {str(p): [] for p in (16, 32, 64)}, "multi": []}
    for r in range(args.runs):
        tset, ts, tp, st = arm_solo(solo_layers, costs, goals, starts)
        rec["solo"].append({"maps_per_s_solve": m / ts, "maps_per_s_set_solve": m / (tset + ts),
                            "maps_per_s_set_solve_path": m / (tset + ts + tp), **work(st, cells)})
        for per in (16, 32, 64):
            tset, ts, tp, st = arm_batch(one, costs, goals, starts, per)
            rec["batch"][str(per)].append({"maps_per_s_solve": m / ts, "maps_per_s_set_solve": m / (tset + ts),
                                           "maps_per_s_set_solve_path": m / (tset + ts + tp),
                                           "launches": len(st), **work(st, cells)})
        t_nopath, t_path = arm_multi(multi, costs, goals, starts)
        rec["multi"].append({"maps_per_s_set_solve": m / t_nopath, "maps_per_s_set_solve_path": m / t_path})
        print(json.dumps({"n": n, "run": r, "solo": rec["solo"][-1],
                          "batch": {p: v[-1] for p, v in rec["batch"].items()}, "multi": rec["multi"][-1]}),
              flush=True)
    rec["k_map_ceff"] = map_ceff_rate(one, costs[:64])
    print(json.dumps({"n": n, "k_map_ceff": rec["k_map_ceff"]}), flush=True)
    results["workloads"].append(rec)
    for layer in solo_layers + [one] + multi:
        layer.close()

os.makedirs(args.out, exist_ok=True)
with open(os.path.join(args.out, "probe_maps.json"), "w") as f:
    json.dump(results, f, indent=1)
print("card: %s, power limit %s" % (card, power))
