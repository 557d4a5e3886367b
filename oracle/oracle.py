"""Python access to the parity oracle (TEST INFRASTRUCTURE ONLY).

Two checkers live under oracle/:

* ``reference()`` -- the UNMODIFIED reference sources compiled into
  ``oracle/_ref/libdymu_ref.so`` (oracle/Makefile, target ``ref``), driven
  through the flat C API of include/dymu_planner_c.h.  Present wherever the
  snapshot was built with /root/reference available (the .so travels to the GPU
  box; the sources do not).
* ``Port`` -- the plain-C restatement ``oracle/dymu_oracle.c`` compiled into
  ``oracle/libdymu_oracle.so`` (target ``port``), pinned against the reference
  by tests/test_oracle_vs_reference.py and tests/golden/.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs may import this module.
"""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(HERE, "_ref", "libdymu_ref.so")
PORT_SO = os.path.join(HERE, "libdymu_oracle.so")

CONSERVATIVE, SWEEPING = 0, 1
_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)


def build(ref=True, port=True):
    """Compile the checkers (building the checker is not using it)."""
    targets = []
    if port:
        targets.append("port")
    # the unmodified reference sources: /root/reference unless DYMU_REFERENCE names another checkout
    reference = os.environ.get("DYMU_REFERENCE", "/root/reference")
    if ref and os.path.isdir(os.path.join(reference, "src")):
        targets += ["ref", "REFERENCE=" + os.path.abspath(reference)]
    if targets:
        subprocess.run(["make", "-C", HERE] + targets, check=True, stdout=subprocess.DEVNULL)


def have_reference():
    return os.path.exists(REF_SO)


def reference():
    """PlannerLib bound to the compiled unmodified reference."""
    import importlib.util
    api = os.path.join(os.path.dirname(HERE), "planning-path_planning_b200", "planner_api.py")
    spec = importlib.util.spec_from_file_location("_dymu_planner_api_for_oracle", api)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.PlannerLib(REF_SO)


def _load_port():
    if not os.path.exists(PORT_SO):
        build(ref=False, port=True)
    lib = C.CDLL(PORT_SO)
    sig = {
        "orc_create": (C.c_void_p, [C.c_double, C.c_double, C.c_double, C.c_int]),
        "orc_destroy": (None, [C.c_void_p]),
        "orc_init_global_layer": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_uint32,
                                            C.c_uint32, C.c_double, C.c_double]),
        "orc_set_cost_map": (C.c_int, [C.c_void_p, _dp, C.c_uint32, C.c_uint32]),
        "orc_compute_cost_map": (C.c_int, [C.c_void_p, _dp, C.c_int, _dp, C.c_int, C.c_int, _dp,
                                           _dp]),
        "orc_set_goal": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double]),
        "orc_compute_entire_total_cost_map": (C.c_int, [C.c_void_p]),
        "orc_compute_total_cost_map": (C.c_int, [C.c_void_p, C.c_double, C.c_double]),
        "orc_solve_heap": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64]),
        "orc_fixed_point_violations": (C.c_uint64, [C.c_void_p, _dp, C.c_double]),
        "orc_compute_global_path": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double,
                                              C.c_int64]),
        "orc_get_total_cost": (C.c_double, [C.c_void_p, C.c_double, C.c_double]),
        "orc_compute_local_planning": (C.c_int, [C.c_void_p, C.c_double, C.c_double, _u8p, C.c_int,
                                                 C.c_int, C.c_double]),
        "orc_expand_risk": (None, [C.c_void_p]),
        "orc_get_path": (C.c_int64, [C.c_void_p, C.c_double, C.c_double, _dp, C.c_int64]),
        "orc_get_local_matrix": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp]),
        "orc_local_propagation": (C.c_int64, [C.c_void_p, C.c_double, C.c_double, C.c_double,
                                              C.c_double]),
        "orc_plane": (_dp, [C.c_void_p, C.c_int]),
        "orc_plane_u8": (_u8p, [C.c_void_p, C.c_int]),
        "orc_terrain": (C.POINTER(C.c_uint32), [C.c_void_p]),
        "orc_locmode": (C.POINTER(C.c_int32), [C.c_void_p]),
        "orc_local_plane": (_dp, [C.c_void_p, C.c_int]),
        "orc_local_plane_u8": (_u8p, [C.c_void_p, C.c_int]),
        "orc_local_dim": (C.c_uint64, [C.c_void_p, C.c_int]),
        "orc_path_size": (C.c_size_t, [C.c_void_p]),
        "orc_path_data": (_dp, [C.c_void_p]),
        "orc_set_path": (None, [C.c_void_p, _dp, C.c_size_t]),
        "orc_counter": (C.c_uint64, [C.c_void_p, C.c_int]),
        "orc_reconnecting_index": (C.c_int, [C.c_void_p]),
        "orc_propagated_count": (C.c_size_t, [C.c_void_p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


_PORT = None


def _port():
    global _PORT
    if _PORT is None:
        _PORT = _load_port()
    return _PORT


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Port:
    """The plain-C restatement, with the reference's method names."""

    PLANES = {"elevation": 0, "slope": 1, "raw_cost": 2, "cost": 3, "hazard_density": 4,
              "trafficability": 5, "total_cost": 6}
    PLANES_U8 = {"isObstacle": 0, "state": 1, "hasLocalMap": 2}

    def __init__(self, risk_distance, reconnect_distance, risk_ratio, approach):
        self._l = _port()
        self._h = self._l.orc_create(risk_distance, reconnect_distance, risk_ratio, int(approach))
        self.nx = self.ny = 0

    def close(self):
        if self._h:
            self._l.orc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def initGlobalLayer(self, globalres, localres, num_nodes_X, num_nodes_Y, offset=(0.0, 0.0)):
        self.nx, self.ny = int(num_nodes_X), int(num_nodes_Y)
        self.r = int(globalres / localres)
        return bool(self._l.orc_init_global_layer(self._h, globalres, localres, self.nx, self.ny,
                                                  offset[0], offset[1]))

    def setCostMap(self, cost_map):
        m = _f64(cost_map)
        return bool(self._l.orc_set_cost_map(self._h, m.ctypes.data_as(_dp), m.shape[0],
                                             m.shape[1]))

    def computeCostMap(self, cost_data, slope_values, locomotionModes, elevation, terrainMap):
        lut, sl, e, t = _f64(cost_data), _f64(slope_values), _f64(elevation), _f64(terrainMap)
        return bool(self._l.orc_compute_cost_map(
            self._h, lut.ctypes.data_as(_dp), lut.size, sl.ctypes.data_as(_dp), sl.size,
            len(locomotionModes), e.ctypes.data_as(_dp), t.ctypes.data_as(_dp)))

    def setGoal(self, x, y, heading=0.0):
        return bool(self._l.orc_set_goal(self._h, x, y, heading))

    def computeEntireTotalCostMap(self, heap=False):
        if heap:
            return bool(self._l.orc_solve_heap(self._h, -1, -1))
        return bool(self._l.orc_compute_entire_total_cost_map(self._h))

    def computeTotalCostMap(self, x, y):
        return bool(self._l.orc_compute_total_cost_map(self._h, x, y))

    def computeGlobalPath(self, x, y, heading=0.0, max_steps=10 ** 8):
        return int(self._l.orc_compute_global_path(self._h, x, y, heading, max_steps))

    @property
    def current_path(self):
        n = self._l.orc_path_size(self._h)
        if n == 0:
            return np.empty((0, 4))
        return np.ctypeslib.as_array(self._l.orc_path_data(self._h), shape=(n, 4)).copy()

    @current_path.setter
    def current_path(self, xyzh):
        a = _f64(xyzh)
        self._l.orc_set_path(self._h, a.ctypes.data_as(_dp), a.shape[0])

    def getPath(self, x, y):
        cap = 1 << 20
        buf = np.empty((cap, 4))
        n = self._l.orc_get_path(self._h, x, y, buf.ctypes.data_as(_dp), cap)
        return buf[:n].copy()

    def getTotalCost(self, x, y):
        return float(self._l.orc_get_total_cost(self._h, x, y))

    def plane(self, name):
        """Copy of a globalNode field plane (inf kept)."""
        if name in self.PLANES:
            p = self._l.orc_plane(self._h, self.PLANES[name])
            return np.ctypeslib.as_array(p, shape=(self.ny, self.nx)).copy()
        if name in self.PLANES_U8:
            p = self._l.orc_plane_u8(self._h, self.PLANES_U8[name])
            return np.ctypeslib.as_array(p, shape=(self.ny, self.nx)).copy()
        if name == "terrain":
            return np.ctypeslib.as_array(self._l.orc_terrain(self._h),
                                         shape=(self.ny, self.nx)).copy()
        if name == "locmode":
            return np.ctypeslib.as_array(self._l.orc_locmode(self._h),
                                         shape=(self.ny, self.nx)).copy()
        raise KeyError(name)

    def set_plane(self, name, values):
        p = self._l.orc_plane(self._h, self.PLANES[name])
        np.ctypeslib.as_array(p, shape=(self.ny, self.nx))[...] = values

    # DYMU_NODE_* of include/dymu_planner_c.h (fields 1-6 pinned against the reference's taps by
    # tests/test_golden_cpu.py)
    NODE_FIELDS = ("elevation", "slope", "raw_cost", "cost", "isObstacle", "state", "hasLocalMap",
                   "terrain", "total_cost")

    def node_field(self, field):
        return self.plane(self.NODE_FIELDS[field]).astype(np.float64)

    def getTotalCostMatrix(self):
        T = self.plane("total_cost")
        T[np.isinf(T)] = -1.0
        return T

    # the flat-buffer calls of include/dymu_planner_c.h as the C view of the reference makes them
    # (capi/planner_capi.cpp:442-480): by value through setCostMap / getTotalCostMatrix
    def setCostMapFlat(self, cost_map):
        return self.setCostMap(cost_map)

    def setTotalCostMatrixTarget(self, out):
        return True

    def getTotalCostMatrixFlat(self, out):
        out[...] = self.getTotalCostMatrix()
        return True

    def getGlobalCostMatrix(self):
        c = self.plane("cost") * (2 + self.plane("hazard_density") - self.plane("trafficability"))
        c[self.plane("isObstacle") != 0] = -1.0
        return c

    def getHazardDensityMatrix(self):
        return self.plane("hazard_density")

    def getTrafficabilityMatrix(self):
        return self.plane("trafficability")

    def fixed_point_violations(self, T, rel_tol=0.0):
        a = _f64(T)
        return int(self._l.orc_fixed_point_violations(self._h, a.ctypes.data_as(_dp), rel_tol))

    # local layer
    def computeLocalPlanning(self, x, y, image, res):
        img = np.ascontiguousarray(image, dtype=np.uint8)
        ok = self._l.orc_compute_local_planning(self._h, x, y, img.ctypes.data_as(_u8p),
                                                img.shape[1], img.shape[0], res)
        return bool(ok), (self.current_path if ok else np.empty((0, 4))), 0.0

    def local_plane(self, name):
        lnx = self._l.orc_local_dim(self._h, 0)
        lny = self._l.orc_local_dim(self._h, 1)
        if name in ("risk", "deviation", "total_cost"):
            p = self._l.orc_local_plane(self._h, ("risk", "deviation", "total_cost").index(name))
        else:
            p = self._l.orc_local_plane_u8(self._h, ("isObstacle", "state").index(name))
        return np.ctypeslib.as_array(p, shape=(lny, lnx)).copy()

    def _local(self, kind, x, y):
        side = 21 * self.r
        out = np.empty((side, side))
        self._l.orc_get_local_matrix(self._h, kind, x, y, out.ctypes.data_as(_dp))
        return out

    def getRiskMatrix(self, x, y):
        return self._local(0, x, y)

    def getDeviationMatrix(self, x, y):
        return self._local(1, x, y)

    def getReconnectingIndex(self):
        return int(self._l.orc_reconnecting_index(self._h))

    def counters(self):
        return {"pops": int(self._l.orc_counter(self._h, 0)),
                "updates": int(self._l.orc_counter(self._h, 1))}
