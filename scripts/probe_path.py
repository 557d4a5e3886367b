"""Developer probe: time of the global path extraction alone on the 4096^2 benchmark map.

    python scripts/probe_path.py [n] [--start S]

The start defaults to the free cell nearest (n // 16, n // 16); bench.py starts at n // 8.
With a DYMU_PATH_PROFILE=1 build the library also prints, per call, the walker's cycles
spent walking, the cycles spent waiting for or doing window reloads, and the reload count."""
import argparse, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("DYMU_TRACE_CALLS", "1")
import dymu_b200
ap = argparse.ArgumentParser()
ap.add_argument("n", type=int, nargs="?", default=4096)
ap.add_argument("--start", type=int, default=None, help="start cell (S, S); default n // 16")
args = ap.parse_args()
pkg = dymu_b200.load(); syn = pkg.synthetic
n = args.n
s0 = n // 16 if args.start is None else args.start
elev, terr = syn.mars_dem(n, n, seed=20261018)
lut, slopes, locs = syn.default_lut()
dev = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
ob = dev.download_plane_u8("obstacle")
goal = syn.free_interior_cell_near(ob, n // 2, n // 2)
start = syn.free_interior_cell_near(ob, s0, s0)
dev.solve_total_cost([goal])
for rep in range(4):
    dev.event_record(0)
    wps, status = dev.extract_global_path(float(start[0]), float(start[1]), 0.4, goal[0], goal[1])
    dev.event_record(1); dev.synchronize()
    print("path: %d waypoints, status %d, %.3f ms (%.1f ns/step)" % (len(wps), status, dev.event_elapsed_ms(0, 1),
          dev.event_elapsed_ms(0, 1) * 1e6 / max(len(wps), 1)), flush=True)
