"""ctypes binding of include/dymu_cuda.h (libdymu_cuda.so).

Thin and explicit: one Python method per C entry point, numpy arrays in and out.
There is no CPU fallback; ``DeviceLayer`` raises if the library is missing or no
CUDA device can be opened.
"""
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CUDA_SO = os.path.join(HERE, "libdymu_cuda.so")

OK = 0
PLANE = {"elevation": 0, "slope": 1, "raw_cost": 2, "cost": 3, "hazard_density": 4,
         "trafficability": 5, "total_cost": 6, "ceff": 7,
         # directional costs of the anisotropic solve (read-only, only while it is on)
         "dircost_xm": 8, "dircost_xp": 9, "dircost_ym": 10, "dircost_yp": 11,
         # distance to the nearest obstacle (read-only, only while obstacle clearance is on)
         "clearance": 12}
PLANE_U8 = {"obstacle": 0, "locmode": 1}
XFORM_NONE, XFORM_INF_TO_MINUS1, XFORM_EFFECTIVE_COST = 0, 1, 2
LPLANE = {"risk": 0, "deviation": 1, "total_cost": 2}
LPLANE_U8 = {"obstacle": 0, "state": 1}

_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)


class DdStats(C.Structure):
    _fields_ = [("rounds", C.c_uint32), ("converged", C.c_uint32), ("wall_ms", C.c_float),
                ("max_kernel_ms", C.c_float), ("sum_kernel_ms", C.c_float), ("reserved_", C.c_uint32),
                ("tile_activations", C.c_uint64), ("cell_updates", C.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved_"}


class SolveStats(C.Structure):
    _fields_ = [("outer_iterations", C.c_uint32), ("converged", C.c_uint32),
                ("tile_activations", C.c_uint64), ("cell_updates", C.c_uint64),
                ("cells_reached", C.c_uint64), ("tiles_deferred", C.c_uint64), ("inner_iterations", C.c_uint64), ("kernel_ms", C.c_float), ("reset_ms", C.c_float),
                ("goal_obstacle", C.c_uint32), ("tiles_delivered_early", C.c_uint32),
                ("cells_written", C.c_uint64),
                ("tiles_delivered_late", C.c_uint32), ("reserved_", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved_"}


_SIG = {
    "dymu_create": (C.c_int, [C.c_int, C.c_uint32, C.c_uint32, C.c_double, C.c_double,
                              C.POINTER(C.c_void_p)]),
    "dymu_destroy": (C.c_int, [C.c_void_p]),
    "dymu_last_error": (C.c_char_p, [C.c_void_p]),
    "dymu_stream": (C.c_void_p, [C.c_void_p]),
    "dymu_synchronize": (C.c_int, [C.c_void_p]),
    "dymu_launch_count": (C.c_uint64, [C.c_void_p]),
    "dymu_event_record": (C.c_int, [C.c_void_p, C.c_int]),
    "dymu_event_elapsed_ms": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "dymu_selftest_sqrt": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), _dp]),
    "dymu_time_stencils": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "dymu_geometry": (C.c_int, [C.c_void_p, _u32p, _u32p, _u32p]),
    "dymu_upload_plane": (C.c_int, [C.c_void_p, C.c_int, _dp, C.c_size_t]),
    "dymu_download_plane": (C.c_int, [C.c_void_p, C.c_int, _dp, C.c_size_t, C.c_int]),
    "dymu_download_plane_u8": (C.c_int, [C.c_void_p, C.c_int, _u8p, C.c_size_t]),
    "dymu_read_rect": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                                 C.c_uint32, _dp]),
    "dymu_write_rect": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                                  C.c_uint32, _dp]),
    "dymu_read_rect_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                                    C.c_uint32, _u8p]),
    "dymu_plane_device_ptr": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p),
                                        C.POINTER(C.c_size_t)]),
    "dymu_dd_solve": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint32, _u32p, C.c_uint32, C.c_uint32, C.c_uint32,
                                C.POINTER(DdStats)]),
    "dymu_batch_solve": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, _u32p, _u32p, _dp, C.c_double,
                                   _dp, C.c_uint32, _u32p, C.POINTER(C.c_int32), C.POINTER(C.c_float)]),
    "dymu_reserve_maps": (C.c_int, [C.c_void_p, C.c_uint32]),
    "dymu_set_maps": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int]),
    "dymu_solve_maps": (C.c_int, [C.c_void_p, C.c_uint32, _u32p, _u32p, C.POINTER(SolveStats)]),
    "dymu_batch_solve_maps": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, _dp, C.c_size_t, C.c_size_t,
                                        _u32p, _u32p, _dp, C.c_double, _dp, C.c_uint32, _u32p,
                                        C.POINTER(C.c_int32), _dp, C.c_size_t, C.POINTER(C.c_float)]),
    "dymu_set_maps_clearance": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double]),
    "dymu_set_maps_anisotropy": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int]),
    "dymu_local_reshape": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int64, C.c_int64]),
    "dymu_solve_incremental": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(SolveStats),
                                         C.POINTER(C.c_uint64)]),
    "dymu_set_cost_map_begin": (C.c_int, [C.c_void_p, _dp, C.c_size_t, C.c_uint32]),
    "dymu_set_cost_map": (C.c_int, [C.c_void_p, _dp, C.c_size_t]),
    "dymu_compute_cost_map": (C.c_int, [C.c_void_p, _dp, C.c_int, _dp, C.c_int, C.c_int, _dp,
                                        C.c_size_t, _dp, C.c_size_t]),
    "dymu_upload_terrain": (C.c_int, [C.c_void_p, _dp, C.c_size_t]),
    "dymu_reserve_slots": (C.c_int, [C.c_void_p, C.c_uint32]),
    "dymu_set_anisotropy": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int]),
    "dymu_set_obstacle_clearance": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double]),
    "dymu_solve_total_cost": (C.c_int, [C.c_void_p, C.c_uint32, _u32p, _u32p,
                                        C.POINTER(SolveStats)]),
    "dymu_solve_start": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(SolveStats)]),
    "dymu_solve_advance": (C.c_int, [C.c_void_p, _u32p, C.c_uint32, C.c_double, C.c_uint32,
                                     C.POINTER(SolveStats)]),
    "dymu_plan_streamed": (C.c_int, [C.c_void_p, _dp, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32,
                                     C.POINTER(SolveStats)]),
    "dymu_reset_total_cost": (C.c_int, [C.c_void_p]),
    "dymu_export_rows": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int]),
    "dymu_import_rows_min_key": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                           C.c_int, C.POINTER(C.c_int), _dp]),
    "dymu_count_reached": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64)]),
    "dymu_stop_threshold": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, _dp]),
    "dymu_download_total_cost": (C.c_int, [C.c_void_p, C.c_uint32, _dp, C.c_size_t, C.c_int]),
    "dymu_download_total_cost_begin": (C.c_int, [C.c_void_p, C.c_uint32, _dp, C.c_size_t, C.c_int]),
    "dymu_download_total_cost_end": (C.c_int, [C.c_void_p]),
    "dymu_set_total_cost_export": (C.c_int, [C.c_void_p, _dp, C.c_size_t, C.c_int, C.POINTER(C.c_int)]),
    "dymu_read_cells": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, _u32p, C.c_uint32, _dp]),
    "dymu_read_node": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _dp]),
    "dymu_count_leq": (C.c_int, [C.c_void_p, C.c_uint32, C.c_double, C.POINTER(C.c_uint64)]),
    "dymu_extract_global_path": (C.c_int, [C.c_void_p, C.c_uint32, C.c_double, C.c_double,
                                           C.c_double, C.c_uint32, C.c_uint32, _dp, C.c_uint32,
                                           _u32p, C.POINTER(C.c_int)]),
    "dymu_extract_global_path_batch": (C.c_int, [C.c_void_p, C.c_uint32, _u32p, _dp, C.c_double, _u32p,
                                                 _dp, C.c_uint32, _u32p, C.POINTER(C.c_int)]),
    "dymu_local_create": (C.c_int, [C.c_void_p, C.c_uint32]),
    "dymu_local_anchor": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64]),
    "dymu_local_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _u32p,
                                  _u32p]),
    "dymu_local_read_rect": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                                       C.c_uint32, _dp]),
    "dymu_local_read_rect_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                                          C.c_uint32, _u8p]),
    "dymu_local_ingest": (C.c_int, [C.c_void_p, _u8p, C.c_uint32, C.c_uint32, C.c_uint32,
                                    C.c_uint32, C.c_double, C.c_double, C.c_double, _u32p,
                                    C.c_uint32, _u32p]),
    "dymu_local_blocking": (C.c_int, [C.c_void_p, _u32p, C.c_uint32, _dp, C.c_uint32, C.c_double,
                                      _u32p, _u32p, C.POINTER(C.c_int)]),
    "dymu_local_expand_risk": (C.c_int, [C.c_void_p, C.c_double, C.POINTER(SolveStats)]),
    "dymu_local_propagate": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double,
                                       C.c_double, C.c_double, C.c_double, C.POINTER(C.c_int64),
                                       _u32p, C.POINTER(C.c_uint64)]),
    "dymu_local_extract_path": (C.c_int, [C.c_void_p, C.c_int64, C.c_double, C.c_double,
                                          C.c_double, C.c_double, _dp, C.c_uint32, _u32p,
                                          C.POINTER(C.c_int)]),
    "dymu_local_read_entered": (C.c_int, [C.c_void_p, _u8p, C.c_int]),
    "dymu_local_sample_risk": (C.c_int, [C.c_void_p, _dp, C.c_uint32, _dp]),
    "dymu_local_cell_of": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.POINTER(C.c_int64)]),
}

CUDA_SYMBOLS = tuple(_SIG)
_LIB = None


def load_library():
    """Loads libdymu_cuda.so (RTLD_GLOBAL so libdymu_b200.so resolves against it)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(CUDA_SO):
            raise RuntimeError("libdymu_cuda.so is not built: run "
                               "`python planning-path_planning_b200/build.py` (no CPU fallback)")
        lib = C.CDLL(CUDA_SO, mode=C.RTLD_GLOBAL)
        for name, (res, args) in _SIG.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _LIB = lib
    return _LIB


class DymuError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("dymu_cuda error %d: %s" % (code, text))
        self.code = code


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class DeviceLayer:
    """One dymu_ctx: the global layer of a DyMu planner resident on one GPU."""

    def __init__(self, nx, ny, global_res=1.0, local_res=0.1, device=-1):
        self._l = load_library()
        self._h = C.c_void_p()
        self.nx, self.ny = int(nx), int(ny)
        rc = self._l.dymu_create(device, self.nx, self.ny, global_res, local_res,
                                 C.byref(self._h))
        if rc != OK:
            text = self._l.dymu_last_error(self._h).decode() if self._h else "no CUDA device"
            if self._h:
                self._l.dymu_destroy(self._h)
                self._h = C.c_void_p()
            raise DymuError(rc, text)

    def _chk(self, rc):
        if rc != OK:
            raise DymuError(rc, self._l.dymu_last_error(self._h).decode())

    def close(self):
        if self._h:
            self._l.dymu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # context
    @property
    def stream(self):
        return self._l.dymu_stream(self._h)

    def synchronize(self):
        self._chk(self._l.dymu_synchronize(self._h))

    @property
    def launches(self):
        return int(self._l.dymu_launch_count(self._h))

    def event_record(self, which):
        self._chk(self._l.dymu_event_record(self._h, which))

    def event_elapsed_ms(self, a, b):
        ms = C.c_float()
        self._chk(self._l.dymu_event_elapsed_ms(self._h, a, b, C.byref(ms)))
        return ms.value

    def selftest_sqrt(self, n, seed=1):
        bad, first = C.c_uint64(), C.c_double()
        self._chk(self._l.dymu_selftest_sqrt(self._h, n, seed, C.byref(bad), C.byref(first)))
        return int(bad.value), first.value

    def time_stencils(self):
        ms = (C.c_float * 6)()
        self._chk(self._l.dymu_time_stencils(self._h, ms))
        return [float(v) for v in ms]

    def geometry(self):
        t, p, r = C.c_uint32(), C.c_uint32(), C.c_uint32()
        self._chk(self._l.dymu_geometry(self._h, C.byref(t), C.byref(p), C.byref(r)))
        return t.value, p.value, r.value

    # planes
    def upload_plane(self, name, host):
        a = _f64(host)
        self._chk(self._l.dymu_upload_plane(self._h, PLANE[name], a.ctypes.data_as(_dp),
                                            a.shape[1]))

    def download_plane(self, name, xform=XFORM_NONE, out=None):
        if out is None:
            out = np.empty((self.ny, self.nx), dtype=np.float64)
        self._chk(self._l.dymu_download_plane(self._h, PLANE[name], out.ctypes.data_as(_dp),
                                              out.shape[1], xform))
        return out

    def download_plane_u8(self, name):
        out = np.empty((self.ny, self.nx), dtype=np.uint8)
        self._chk(self._l.dymu_download_plane_u8(self._h, PLANE_U8[name],
                                                 out.ctypes.data_as(_u8p), self.nx))
        return out

    def read_rect(self, name, i0, j0, w, h):
        out = np.empty((h, w), dtype=np.float64)
        self._chk(self._l.dymu_read_rect(self._h, PLANE[name], i0, j0, w, h,
                                         out.ctypes.data_as(_dp)))
        return out

    def write_rect(self, name, i0, j0, values):
        a = _f64(values)
        self._chk(self._l.dymu_write_rect(self._h, PLANE[name], i0, j0, a.shape[1], a.shape[0],
                                          a.ctypes.data_as(_dp)))

    def plane_device_ptr(self, name):
        p, pitch = C.c_void_p(), C.c_size_t()
        self._chk(self._l.dymu_plane_device_ptr(self._h, PLANE[name], C.byref(p), C.byref(pitch)))
        return p.value, pitch.value

    # cost map
    def set_cost_map(self, cost=None):
        if cost is None:
            self._chk(self._l.dymu_set_cost_map(self._h, None, 0))
        else:
            a = _f64(cost)
            self._chk(self._l.dymu_set_cost_map(self._h, a.ctypes.data_as(_dp), a.shape[1]))

    def compute_cost_map(self, lut, slopes, n_locs, elevation=None, terrain=None):
        lut, slopes = _f64(lut), _f64(slopes)
        e = _f64(elevation) if elevation is not None else None
        t = _f64(terrain) if terrain is not None else None
        self._chk(self._l.dymu_compute_cost_map(
            self._h, lut.ctypes.data_as(_dp), lut.size, slopes.ctypes.data_as(_dp), slopes.size,
            n_locs, e.ctypes.data_as(_dp) if e is not None else None,
            e.shape[1] if e is not None else 0,
            t.ctypes.data_as(_dp) if t is not None else None, t.shape[1] if t is not None else 0))

    def set_anisotropy(self, theta_deg, factors):
        """Slope anisotropy: f(theta) piecewise linear in the table (theta in degrees, strictly
        ascending, positive = uphill; factors finite > 0); empty tables switch it off."""
        t, f = _f64(theta_deg).ravel(), _f64(factors).ravel()
        if t.size != f.size:
            raise ValueError("theta_deg and factors differ in length")
        self._chk(self._l.dymu_set_anisotropy(self._h, t.ctypes.data_as(_dp), f.ctypes.data_as(_dp), t.size))

    def set_obstacle_clearance(self, radius, margin, penalty):
        """Obstacle clearance (metres): C_eff = +inf within `radius` of an obstacle, scaled by
        1 + penalty * (radius + margin - d) / margin up to radius + margin; (0, 0, 0) switches it off."""
        self._chk(self._l.dymu_set_obstacle_clearance(self._h, float(radius), float(margin), float(penalty)))

    # solve
    def reserve_slots(self, n):
        self._chk(self._l.dymu_reserve_slots(self._h, n))

    def solve_total_cost(self, goals):
        """goals: iterable of (i, j).  Returns the aggregate SolveStats as a dict."""
        g = np.asarray(list(goals), dtype=np.uint32).reshape(-1, 2)
        gi, gj = np.ascontiguousarray(g[:, 0]), np.ascontiguousarray(g[:, 1])
        st = SolveStats()
        self._chk(self._l.dymu_solve_total_cost(self._h, g.shape[0], gi.ctypes.data_as(_u32p),
                                                gj.ctypes.data_as(_u32p), C.byref(st)))
        return st.as_dict()

    # map batches (map q <-> total-cost slot q; read the slots with the slot-based calls)
    def reserve_maps(self, n):
        """n cost-term planes, one per total-cost slot (grows the slots to n); 0 frees them."""
        self._chk(self._l.dymu_reserve_maps(self._h, int(n)))

    def set_maps(self, costs, first=0):
        """Maps [first, first+n) from a numpy (n, ny, nx) (or (ny, nx)) array of costs."""
        a = _f64(costs)
        a = a.reshape((-1,) + a.shape[-2:])
        if a.shape[1:] != (self.ny, self.nx):
            raise ValueError("expected maps of shape (%d, %d)" % (self.ny, self.nx))
        self._chk(self._l.dymu_set_maps(self._h, int(first), a.shape[0], C.c_void_p(a.ctypes.data),
                                        a.shape[2], a.shape[1] * a.shape[2], 0))

    def set_maps_device(self, ptr, n, ld, map_stride, first=0):
        """Maps [first, first+n) from device memory of this GPU (e.g. a torch CUDA tensor's data_ptr(),
        after the stream that wrote it was synchronised); ld, map_stride in doubles."""
        self._chk(self._l.dymu_set_maps(self._h, int(first), int(n), C.c_void_p(ptr), int(ld), int(map_stride), 1))

    def solve_maps(self, goals):
        """goals[q] = (i, j) of map q, solved into slot q in one launch.  Returns the aggregate SolveStats."""
        g = np.asarray(list(goals), dtype=np.uint32).reshape(-1, 2)
        gi, gj = np.ascontiguousarray(g[:, 0]), np.ascontiguousarray(g[:, 1])
        st = SolveStats()
        self._chk(self._l.dymu_solve_maps(self._h, g.shape[0], gi.ctypes.data_as(_u32p), gj.ctypes.data_as(_u32p),
                                          C.byref(st)))
        return st.as_dict()

    def set_maps_clearance(self, radius, margin, penalty):
        """Obstacle clearance of every map solve of this layer (the obstacles of map q are its cells with
        cost <= 0); parameters as set_obstacle_clearance, (0, 0, 0) switches it off."""
        self._chk(self._l.dymu_set_maps_clearance(self._h, float(radius), float(margin), float(penalty)))

    def set_maps_anisotropy(self, theta_deg, factors):
        """Slope anisotropy of every map solve of this layer, on the layer's elevation plane; table as
        set_anisotropy, empty tables switch it off."""
        t, f = _f64(theta_deg).ravel(), _f64(factors).ravel()
        if t.size != f.size:
            raise ValueError("theta_deg and factors differ in length")
        self._chk(self._l.dymu_set_maps_anisotropy(self._h, t.ctypes.data_as(_dp), f.ctypes.data_as(_dp), t.size))

    def solve_incremental(self, goal):
        """Re-solve after small changes of cost / hazard_density / trafficability.  Returns
        (stats, cells invalidated or None when a full solve ran)."""
        st, inv = SolveStats(), C.c_uint64()
        self._chk(self._l.dymu_solve_incremental(self._h, int(goal[0]), int(goal[1]), C.byref(st), C.byref(inv)))
        return st.as_dict(), (None if inv.value == 2 ** 64 - 1 else int(inv.value))

    def solve_start(self, goal, max_phases):
        """Seed the goal and run at most max_phases solver phases; stats['converged'] == 0 means
        work is pending on the device (continue with solve_advance)."""
        st = SolveStats()
        self._chk(self._l.dymu_solve_start(self._h, int(goal[0]), int(goal[1]), int(max_phases), C.byref(st)))
        return st.as_dict()

    def solve_advance(self, ranges, seed_key, max_phases):
        r = np.ascontiguousarray(list(ranges), dtype=np.uint32).reshape(-1, 2)
        st = SolveStats()
        self._chk(self._l.dymu_solve_advance(self._h, r.ctypes.data_as(_u32p), r.shape[0], float(seed_key),
                                             int(max_phases), C.byref(st)))
        return st.as_dict()

    def _host_plane(self, a):
        """The caller's buffer itself (it is read after the call returns, so never a copy)."""
        if (not isinstance(a, np.ndarray) or a.dtype != np.float64 or not a.flags.c_contiguous
                or a.shape != (self.ny, self.nx)):
            raise ValueError("expected a C-contiguous float64 array of shape (%d, %d)" % (self.ny, self.nx))
        return a

    def set_cost_map_begin(self, cost_host, first_row):
        """set_cost_map without waiting for the copy (dymu_set_cost_map_begin)."""
        cost_host = self._host_plane(cost_host)
        self._chk(self._l.dymu_set_cost_map_begin(self._h, cost_host.ctypes.data_as(_dp), cost_host.shape[1],
                                                  int(first_row)))

    def plan_streamed(self, cost_host, goal, first_phases=0):
        """set_cost_map(cost_host) + solve_total_cost([goal]) with the upload overlapped with the
        solve (cost_host: C-contiguous float64 [ny, nx], pinned for a truly asynchronous copy)."""
        cost_host = self._host_plane(cost_host)
        st = SolveStats()
        self._chk(self._l.dymu_plan_streamed(self._h, cost_host.ctypes.data_as(_dp), cost_host.shape[1],
                                             int(goal[0]), int(goal[1]), int(first_phases), C.byref(st)))
        return st.as_dict()

    def reset_total_cost(self):
        self._chk(self._l.dymu_reset_total_cost(self._h))

    def export_rows(self, j0, n_rows, dst_ptr, device_ptr, slot=0):
        self._chk(self._l.dymu_export_rows(self._h, slot, j0, n_rows, C.c_void_p(dst_ptr),
                                           int(device_ptr)))

    def import_rows_min_key(self, j0, n_rows, src_ptr, device_ptr, slot=0):
        """-> (changed, smallest value that replaced a larger one or +inf)."""
        ch = C.c_int()
        lo = C.c_double()
        self._chk(self._l.dymu_import_rows_min_key(self._h, slot, j0, n_rows, C.c_void_p(src_ptr),
                                                   int(device_ptr), C.byref(ch), C.byref(lo)))
        return bool(ch.value), float(lo.value)

    def count_reached(self, slot=0):
        n = C.c_uint64()
        self._chk(self._l.dymu_count_reached(self._h, slot, C.byref(n)))
        return int(n.value)

    def read_node(self, i, j):
        out = np.empty(10, dtype=np.float64)
        self._chk(self._l.dymu_read_node(self._h, i, j, out.ctypes.data_as(_dp)))
        return out

    def count_leq(self, threshold, slot=0):
        n = C.c_uint64()
        self._chk(self._l.dymu_count_leq(self._h, slot, threshold, C.byref(n)))
        return int(n.value)

    def stop_threshold(self, start_i, start_j, slot=0):
        t = C.c_double()
        self._chk(self._l.dymu_stop_threshold(self._h, slot, start_i, start_j, C.byref(t)))
        return t.value

    def download_total_cost(self, slot=0, xform=XFORM_NONE, out=None):
        if out is None:
            out = np.empty((self.ny, self.nx), dtype=np.float64)
        self._chk(self._l.dymu_download_total_cost(self._h, slot, out.ctypes.data_as(_dp),
                                                   out.shape[1], xform))
        return out

    def download_total_cost_begin(self, out, slot=0, xform=XFORM_NONE):
        """Start the read-back on the copy stream; `out` (pinned for a truly asynchronous copy)
        is valid after download_total_cost_end()."""
        self._chk(self._l.dymu_download_total_cost_begin(self._h, slot, out.ctypes.data_as(_dp),
                                                         out.shape[1], xform))

    def set_total_cost_export(self, out, xform=XFORM_NONE):
        """Direct delivery: full single-goal solves store the total-cost matrix into `out` (a pinned,
        C-contiguous float64 array, e.g. the numpy view of a torch pinned tensor) while they run.
        Returns False when `out` is not page-locked (nothing is set up then); None switches it off."""
        direct = C.c_int(0)
        if out is None:
            self._chk(self._l.dymu_set_total_cost_export(self._h, None, 0, xform, C.byref(direct)))
            return False
        self._chk(self._l.dymu_set_total_cost_export(self._h, out.ctypes.data_as(_dp), out.shape[1], xform,
                                                     C.byref(direct)))
        return bool(direct.value)

    def download_total_cost_end(self):
        self._chk(self._l.dymu_download_total_cost_end(self._h))

    def read_cells(self, name, cells, slot=0):
        idx = np.ascontiguousarray(cells, dtype=np.uint32)
        out = np.empty(idx.size, dtype=np.float64)
        self._chk(self._l.dymu_read_cells(self._h, PLANE[name], slot, idx.ctypes.data_as(_u32p),
                                          idx.size, out.ctypes.data_as(_dp)))
        return out

    def extract_global_path(self, x0, y0, tau, goal_i, goal_j, slot=0, cap=1 << 18):
        """Returns ((n,5) array of x, y, z, dCostX, dCostY, status)."""
        out = np.empty((cap, 5), dtype=np.float64)
        n, status = C.c_uint32(), C.c_int()
        self._chk(self._l.dymu_extract_global_path(self._h, slot, x0, y0, tau, goal_i, goal_j,
                                                   out.ctypes.data_as(_dp), cap, C.byref(n),
                                                   C.byref(status)))
        return out[:n.value].copy(), status.value

    def extract_global_path_batch(self, slots, starts_xy, tau, goals_ij, cap=1 << 15):
        """One launch for many queries.  Returns (list of (n_q,5) arrays, list of status)."""
        sl = np.ascontiguousarray(slots, dtype=np.uint32)
        xy = _f64(starts_xy).reshape(-1, 2)
        g = np.ascontiguousarray(goals_ij, dtype=np.uint32).reshape(-1, 2)
        n = sl.size
        out = np.empty((n, cap, 5), dtype=np.float64)
        n_out = np.zeros(n, dtype=np.uint32)
        status = np.zeros(n, dtype=np.int32)
        self._chk(self._l.dymu_extract_global_path_batch(
            self._h, n, sl.ctypes.data_as(_u32p), xy.ctypes.data_as(_dp), tau, g.ctypes.data_as(_u32p),
            out.ctypes.data_as(_dp), cap, n_out.ctypes.data_as(_u32p),
            status.ctypes.data_as(C.POINTER(C.c_int))))
        return [out[q, :n_out[q]].copy() for q in range(n)], [int(v) for v in status]

    # local layer
    def local_create(self, wg):
        self._chk(self._l.dymu_local_create(self._h, wg))

    def local_anchor(self, gx0, gy0):
        self._chk(self._l.dymu_local_anchor(self._h, gx0, gy0))

    def local_info(self):
        gx0, gy0, wg, r = C.c_int64(), C.c_int64(), C.c_uint32(), C.c_uint32()
        self._chk(self._l.dymu_local_info(self._h, C.byref(gx0), C.byref(gy0), C.byref(wg),
                                          C.byref(r)))
        return gx0.value, gy0.value, wg.value, r.value

    def local_read(self, name, x0=0, y0=0, w=None, h=None):
        _, _, wg, r = self.local_info()
        w = wg * r - x0 if w is None else w
        h = wg * r - y0 if h is None else h
        if name in LPLANE:
            out = np.empty((h, w), dtype=np.float64)
            self._chk(self._l.dymu_local_read_rect(self._h, LPLANE[name], x0, y0, w, h,
                                                   out.ctypes.data_as(_dp)))
        else:
            key = {"isObstacle": "obstacle"}.get(name, name)
            out = np.empty((h, w), dtype=np.uint8)
            self._chk(self._l.dymu_local_read_rect_u8(self._h, LPLANE_U8[key], x0, y0, w, h,
                                                      out.ctypes.data_as(_u8p)))
        return out

    def local_ingest(self, image, res, rover_x, rover_y):
        img = np.ascontiguousarray(image, dtype=np.uint8)
        h, w = img.shape
        cap = w * h
        cells = np.empty(cap, dtype=np.uint32)
        n = C.c_uint32()
        self._chk(self._l.dymu_local_ingest(self._h, img.ctypes.data_as(_u8p), w, h, w, 1, res,
                                            rover_x, rover_y, cells.ctypes.data_as(_u32p), cap,
                                            C.byref(n)))
        return cells[:n.value].copy()

    def local_blocking(self, cells, path_xy, risk_distance, min_index, max_index):
        c = np.ascontiguousarray(cells, dtype=np.uint32)
        p = _f64(path_xy)
        mn, mx, b = C.c_uint32(min_index), C.c_uint32(max_index), C.c_int()
        self._chk(self._l.dymu_local_blocking(self._h, c.ctypes.data_as(_u32p), c.size,
                                              p.ctypes.data_as(_dp), p.shape[0], risk_distance,
                                              C.byref(mn), C.byref(mx), C.byref(b)))
        return mn.value, mx.value, bool(b.value)

    def local_expand_risk(self, risk_distance):
        st = SolveStats()
        self._chk(self._l.dymu_local_expand_risk(self._h, risk_distance, C.byref(st)))
        return st.as_dict()

    def local_propagate(self, approach, start, overtake, t_overtake, risk_ratio):
        end, status, closed = C.c_int64(), C.c_uint32(), C.c_uint64()
        self._chk(self._l.dymu_local_propagate(self._h, approach, start[0], start[1], overtake[0],
                                               overtake[1], t_overtake, risk_ratio, C.byref(end),
                                               C.byref(status), C.byref(closed)))
        return end.value, status.value, closed.value

    def local_extract_path(self, end_cell, start, offset=(0.0, 0.0), cap=1 << 16):
        out = np.empty((cap, 6), dtype=np.float64)
        n, status = C.c_uint32(), C.c_int()
        self._chk(self._l.dymu_local_extract_path(self._h, end_cell, start[0], start[1], offset[0],
                                                  offset[1], out.ctypes.data_as(_dp), cap,
                                                  C.byref(n), C.byref(status)))
        return out[:n.value].copy(), status.value

    def local_read_entered(self, clear=False):
        _, _, wg, _ = self.local_info()
        out = np.empty((wg, wg), dtype=np.uint8)
        self._chk(self._l.dymu_local_read_entered(self._h, out.ctypes.data_as(_u8p), int(clear)))
        return out

    def local_sample_risk(self, xy):
        a = _f64(xy)
        out = np.empty(a.shape[0], dtype=np.float64)
        self._chk(self._l.dymu_local_sample_risk(self._h, a.ctypes.data_as(_dp), a.shape[0],
                                                 out.ctypes.data_as(_dp)))
        return out

    def local_cell_of(self, x, y):
        c = C.c_int64()
        self._chk(self._l.dymu_local_cell_of(self._h, x, y, C.byref(c)))
        return c.value


# ---- several contexts behind one call (include/dymu_cuda.h, "several GPUs behind one call") ----
def _ctx_array(layers):
    arr = (C.c_void_p * len(layers))()
    for k, d in enumerate(layers):
        arr[k] = d._h
    return arr


def dd_solve(layers, cuts, goal, phases_per_round=32):
    """dymu_dd_solve: `layers[k]` is the DeviceLayer of strip k (own rows [cuts[k], cuts[k+1]) plus
    ghost rows, cost map set), `goal` = (i, j) in grid coordinates.  Returns the statistics dict."""
    lib = load_library()
    c = np.ascontiguousarray(cuts, dtype=np.uint32)
    if c.size != len(layers) + 1:
        raise ValueError("cuts must hold len(layers) + 1 rows")
    st = DdStats()
    rc = lib.dymu_dd_solve(_ctx_array(layers), len(layers), c.ctypes.data_as(_u32p), int(goal[0]), int(goal[1]),
                           int(phases_per_round), C.byref(st))
    if rc != 0:
        texts = [lib.dymu_last_error(d._h).decode() for d in layers]
        raise DymuError(rc, "; ".join(t for t in texts if t))
    return st.as_dict()


def batch_solve(layers, goals, starts=None, tau=0.4, cap=1 << 14):
    """dymu_batch_solve: the goal queries are dealt out over `layers` (one context per GPU, same cost
    map, reserve_slots() goals per launch).  Returns (paths or None, per-context wall ms)."""
    lib = load_library()
    g = np.ascontiguousarray(goals, dtype=np.uint32).reshape(-1, 2)
    gi, gj = np.ascontiguousarray(g[:, 0]), np.ascontiguousarray(g[:, 1])
    n = g.shape[0]
    ms = np.zeros(len(layers), dtype=np.float32)
    if starts is None:
        rc = lib.dymu_batch_solve(_ctx_array(layers), len(layers), n, gi.ctypes.data_as(_u32p),
                                  gj.ctypes.data_as(_u32p), None, float(tau), None, 0, None, None,
                                  ms.ctypes.data_as(C.POINTER(C.c_float)))
        paths = None
    else:
        xy = np.ascontiguousarray(starts, dtype=np.float64).reshape(n, 2)
        out = np.empty((n, cap, 5), dtype=np.float64)
        ln = np.zeros(n, dtype=np.uint32)
        stt = np.zeros(n, dtype=np.int32)
        rc = lib.dymu_batch_solve(_ctx_array(layers), len(layers), n, gi.ctypes.data_as(_u32p),
                                  gj.ctypes.data_as(_u32p), xy.ctypes.data_as(_dp), float(tau),
                                  out.ctypes.data_as(_dp), int(cap), ln.ctypes.data_as(_u32p),
                                  stt.ctypes.data_as(C.POINTER(C.c_int32)), ms.ctypes.data_as(C.POINTER(C.c_float)))
        paths = [(out[q, :ln[q]].copy(), int(stt[q])) for q in range(n)]
    if rc != 0:
        texts = [lib.dymu_last_error(d._h).decode() for d in layers]
        raise DymuError(rc, "; ".join(t for t in texts if t))
    return paths, ms


def batch_solve_maps(layers, costs, goals, starts=None, tau=0.4, cap=1 << 14, total_cost=False):
    """dymu_batch_solve_maps: map q of `costs` (numpy (n, ny, nx)) toward goals[q], dealt out over
    `layers` (same size, reserve_maps() maps per launch each).  Returns (paths or None, total-cost
    matrices (n, ny, nx) or None, per-context wall ms)."""
    lib = load_library()
    a = _f64(costs)
    if a.ndim != 3:
        raise ValueError("costs must be an (n, ny, nx) array of maps")
    n, ny, nx = a.shape
    # the library reads and writes ny rows of nx cells per map, with ny and nx taken from the contexts
    for d in layers:
        if (d.ny, d.nx) != (ny, nx):
            raise ValueError("maps of shape (%d, %d) for a layer of shape (%d, %d)" % (ny, nx, d.ny, d.nx))
    g = np.ascontiguousarray(goals, dtype=np.uint32).reshape(-1, 2)
    if g.shape[0] != n:
        raise ValueError("one goal per map")
    gi, gj = np.ascontiguousarray(g[:, 0]), np.ascontiguousarray(g[:, 1])
    ms = np.zeros(len(layers), dtype=np.float32)
    xy = out = ln = stt = None
    if starts is not None:
        xy = np.ascontiguousarray(starts, dtype=np.float64)
        if xy.size != 2 * n:
            raise ValueError("one start (x, y) per map")
        xy = xy.reshape(n, 2)
        out = np.empty((n, cap, 5), dtype=np.float64)
        ln = np.zeros(n, dtype=np.uint32)
        stt = np.zeros(n, dtype=np.int32)
    T = np.empty((n, ny, nx), dtype=np.float64) if total_cost else None
    rc = lib.dymu_batch_solve_maps(
        _ctx_array(layers), len(layers), n, a.ctypes.data_as(_dp), nx, ny * nx, gi.ctypes.data_as(_u32p),
        gj.ctypes.data_as(_u32p), xy.ctypes.data_as(_dp) if xy is not None else None, float(tau),
        out.ctypes.data_as(_dp) if out is not None else None, int(cap) if out is not None else 0,
        ln.ctypes.data_as(_u32p) if ln is not None else None,
        stt.ctypes.data_as(C.POINTER(C.c_int32)) if stt is not None else None,
        T.ctypes.data_as(_dp) if T is not None else None, nx, ms.ctypes.data_as(C.POINTER(C.c_float)))
    if rc != 0:
        texts = [lib.dymu_last_error(d._h).decode() for d in layers]
        raise DymuError(rc, "; ".join(t for t in texts if t))
    paths = [(out[q, :ln[q]].copy(), int(stt[q])) for q in range(n)] if out is not None else None
    return paths, T, ms
