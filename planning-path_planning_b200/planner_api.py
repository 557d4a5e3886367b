"""ctypes view of include/dymu_planner_c.h.

The same class drives any shared library that implements that header:
``libdymu_b200.so`` (this repository's drop-in DyMuPathPlanner on top of the
CUDA C-ABI) or, in the test-suite only, the compiled unmodified reference.  Method names mirror the reference class
(``/root/reference/src/DyMu.hpp:471-608``) so that parity tests read like
calls on ``PathPlanning_lib::DyMuPathPlanner``.
"""
import ctypes as C
import numpy as np

CONSERVATIVE = 0
SWEEPING = 1

MAT_TOTAL_COST, MAT_GLOBAL_COST, MAT_HAZARD_DENSITY, MAT_TRAFFICABILITY = 0, 1, 2, 3
LOCAL_RISK, LOCAL_DEVIATION = 0, 1
(NODE_ELEVATION, NODE_SLOPE, NODE_RAW_COST, NODE_COST, NODE_IS_OBSTACLE, NODE_STATE,
 NODE_HAS_LOCAL_MAP, NODE_TERRAIN, NODE_TOTAL_COST_RAW) = range(9)

_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)

_SIGNATURES = {
    "dymu_planner_impl": (C.c_char_p, []),
    "dymu_planner_create": (C.c_void_p, [C.c_double, C.c_double, C.c_double, C.c_int]),
    "dymu_planner_destroy": (None, [C.c_void_p]),
    "dymu_planner_init_global_layer": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_uint,
                                                 C.c_uint, C.c_double, C.c_double]),
    "dymu_planner_set_cost_map": (C.c_int, [C.c_void_p, _dp, C.c_uint, C.c_uint]),
    "dymu_planner_compute_cost_map": (C.c_int, [C.c_void_p, _dp, C.c_int, _dp, C.c_int, C.c_char_p,
                                                _dp, _dp, C.c_uint, C.c_uint]),
    "dymu_planner_set_goal": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double]),
    "dymu_planner_compute_total_cost_map": (C.c_int, [C.c_void_p, C.c_double, C.c_double]),
    "dymu_planner_compute_entire_total_cost_map": (C.c_int, [C.c_void_p]),
    "dymu_planner_get_path": (C.c_int, [C.c_void_p, C.c_double, C.c_double, _dp, C.c_int]),
    "dymu_planner_compute_global_path": (C.c_int, [C.c_void_p, C.c_double, C.c_double]),
    "dymu_planner_get_current_path": (C.c_int, [C.c_void_p, _dp, C.c_int]),
    "dymu_planner_get_matrix": (C.c_int, [C.c_void_p, C.c_int, _dp]),
    "dymu_planner_get_total_cost": (C.c_double, [C.c_void_p, C.c_double, C.c_double]),
    "dymu_planner_get_locomotion_mode": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_char_p,
                                                   C.c_int]),
    "dymu_planner_compute_local_planning": (C.c_int, [C.c_void_p, C.c_double, C.c_double, _u8p,
                                                      C.c_int, C.c_int, C.c_double, _dp, C.c_int,
                                                      C.POINTER(C.c_int), _dp]),
    "dymu_planner_get_local_matrix": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, _dp,
                                                C.c_int]),
    "dymu_planner_get_reconnecting_index": (C.c_int, [C.c_void_p]),
    "dymu_planner_get_remaining_total_cost": (C.c_double, [C.c_void_p]),
    "dymu_planner_get_node_field": (C.c_int, [C.c_void_p, C.c_int, _dp]),
    "dymu_planner_cora_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, C.c_int]),
    "dymu_planner_get_terrain": (C.c_int, [C.c_void_p, C.c_double, C.c_double]),
    "dymu_planner_fill_terrain_info": (C.c_int, [C.c_void_p, C.c_int, _dp, C.c_int]),
    "dymu_planner_update_cost": (C.c_int, [C.c_void_p, _dp, C.c_int]),
    "dymu_planner_compute_cost_ratio": (C.c_int, [C.c_void_p, _dp, C.c_int]),
    "dymu_planner_recompute_cost_map": (C.c_int, [C.c_void_p]),
    "dymu_planner_gradient_node": (C.c_int, [C.c_void_p, C.c_uint, C.c_uint, _dp, _dp]),
    "dymu_planner_next_global_waypoint": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double, _dp]),
    "dymu_planner_propagate_global_node": (C.c_int, [C.c_void_p, C.c_uint, C.c_uint, _dp]),
    "dymu_planner_set_cost_map_flat": (C.c_int, [C.c_void_p, _dp, C.c_uint]),
    "dymu_planner_set_total_cost_target": (C.c_int, [C.c_void_p, _dp, C.c_uint]),
    "dymu_planner_get_total_cost_matrix_flat": (C.c_int, [C.c_void_p, _dp, C.c_uint]),
    "dymu_planner_last_call_seconds": (C.c_double, [C.c_void_p]),
    "dymu_planner_set_slope_anisotropy": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int]),
    "dymu_planner_set_obstacle_clearance": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double]),
}

PLANNER_SYMBOLS = tuple(_SIGNATURES)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(_dp)


class PlannerLib:
    """A loaded shared library exporting the dymu_planner_* entry points."""

    def __init__(self, path, mode=C.RTLD_LOCAL):
        self.path = str(path)
        self.lib = C.CDLL(self.path, mode=mode)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(self.lib, name)
            fn.restype = res
            fn.argtypes = args

    @property
    def impl(self):
        return self.lib.dymu_planner_impl().decode()

    def DyMuPathPlanner(self, risk_distance, reconnect_distance, risk_ratio, approach):
        return Planner(self, risk_distance, reconnect_distance, risk_ratio, approach)


class Planner:
    """Mirror of PathPlanning_lib::DyMuPathPlanner over the flat C API."""

    MAX_PATH = 1 << 20

    def __init__(self, plib, risk_distance, reconnect_distance, risk_ratio, approach):
        self._l = plib.lib
        self._h = self._l.dymu_planner_create(risk_distance, reconnect_distance, risk_ratio,
                                              int(approach))
        if not self._h:
            raise RuntimeError("dymu_planner_create failed")
        self.nx = self.ny = 0

    def close(self):
        if self._h:
            self._l.dymu_planner_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # --- global layer -------------------------------------------------
    def initGlobalLayer(self, globalres, localres, num_nodes_X, num_nodes_Y, offset=(0.0, 0.0)):
        self.nx, self.ny = int(num_nodes_X), int(num_nodes_Y)
        return bool(self._l.dymu_planner_init_global_layer(
            self._h, globalres, localres, self.nx, self.ny, offset[0], offset[1]))

    def setCostMap(self, cost_map):
        m = _f64(cost_map)
        return bool(self._l.dymu_planner_set_cost_map(self._h, _ptr(m), m.shape[0], m.shape[1]))

    @staticmethod
    def _flat(a, ny, nx):
        """float64 [ny, nx] array with contiguous rows, used in place (never copied: the callee may
        read or write it after the call returns)."""
        if (not isinstance(a, np.ndarray) or a.dtype != np.float64 or a.ndim != 2 or a.shape != (ny, nx)
                or a.strides[1] != 8 or a.strides[0] % 8 or a.strides[0] < 8 * nx):
            raise ValueError("expected a float64 array of shape (%d, %d) with contiguous rows" % (ny, nx))
        return a, a.strides[0] // 8

    def gradientNode(self, i, j):
        """(dnx, dny) of global node (i, j), or None when it does not exist."""
        a, b = C.c_double(), C.c_double()
        if self._l.dymu_planner_gradient_node(self._h, int(i), int(j), C.byref(a), C.byref(b)) != 1:
            return None
        return a.value, b.value

    def computeNextGlobalWaypoint(self, x, y, tau):
        """(next x, next y, heading, z of the input waypoint)."""
        out = np.zeros(4)
        self._l.dymu_planner_next_global_waypoint(self._h, x, y, tau, _ptr(out))
        return out

    def propagateGlobalNode(self, i, j):
        t = C.c_double()
        if self._l.dymu_planner_propagate_global_node(self._h, int(i), int(j), C.byref(t)) != 1:
            return None
        return t.value

    def setCostMapFlat(self, cost_map):
        """setCostMap(const double*, ld) of the drop-in: no nesting, and with a goal in place the
        upload is streamed behind the next computeEntireTotalCostMap() -- `cost_map` must stay
        unchanged until that call returns (pinned memory makes the copy asynchronous)."""
        m, ld = self._flat(cost_map, self.ny, self.nx)
        return bool(self._l.dymu_planner_set_cost_map_flat(self._h, _ptr(m), ld))

    def setTotalCostMatrixTarget(self, out):
        """Deliver the total-cost matrix into `out` right after every solve (None = off)."""
        if out is None:
            self._target = None
            return bool(self._l.dymu_planner_set_total_cost_target(self._h, None, 0))
        m, ld = self._flat(out, self.ny, self.nx)
        self._target = m  # keep the buffer alive while the planner writes into it
        return bool(self._l.dymu_planner_set_total_cost_target(self._h, _ptr(m), ld))

    def getTotalCostMatrixFlat(self, out):
        m, ld = self._flat(out, self.ny, self.nx)
        return bool(self._l.dymu_planner_get_total_cost_matrix_flat(self._h, _ptr(m), ld))

    def computeCostMap(self, cost_data, slope_values, locomotionModes, elevation, terrainMap):
        lut, sl = _f64(cost_data), _f64(slope_values)
        e, t = _f64(elevation), _f64(terrainMap)
        return bool(self._l.dymu_planner_compute_cost_map(
            self._h, _ptr(lut), lut.size, _ptr(sl), sl.size, ",".join(locomotionModes).encode(),
            _ptr(e), _ptr(t), e.shape[0], e.shape[1]))

    def setGoal(self, x, y, heading=0.0):
        return bool(self._l.dymu_planner_set_goal(self._h, x, y, heading))

    def computeTotalCostMap(self, x, y):
        return bool(self._l.dymu_planner_compute_total_cost_map(self._h, x, y))

    def setSlopeAnisotropy(self, slope_angles_deg, factors):
        """Extension of the B200 drop-in (the reference build returns -1, reported as False)."""
        a, f = _f64(slope_angles_deg).ravel(), _f64(factors).ravel()
        if a.size != f.size:
            return False
        return self._l.dymu_planner_set_slope_anisotropy(self._h, _ptr(a), _ptr(f), a.size) == 1

    def setObstacleClearance(self, radius, margin, penalty):
        """Extension of the B200 drop-in: lethal radius and penalised margin around obstacles (metres);
        (0, 0, 0) switches it off.  The reference build returns -1, reported as False."""
        return self._l.dymu_planner_set_obstacle_clearance(self._h, float(radius), float(margin),
                                                           float(penalty)) == 1

    def computeEntireTotalCostMap(self):
        return bool(self._l.dymu_planner_compute_entire_total_cost_map(self._h))

    def _path(self, fn, *args):
        cap = 1 << 15   # a second call would compute the path again
        while True:
            buf = np.empty((cap, 4), dtype=np.float64)
            n = fn(self._h, *args, _ptr(buf), cap)
            if n < 0:
                raise RuntimeError("path call failed (%d)" % n)
            if n <= cap:
                return buf[:n].copy()
            if cap >= self.MAX_PATH:
                raise RuntimeError("path longer than MAX_PATH")
            cap = min(self.MAX_PATH, max(2 * cap, n))
            # NOTE: getPath has side effects (evaluatePath); callers needing an
            # exact single call should pre-size via current_path afterwards.
            fn = self._l.dymu_planner_get_current_path
            args = ()

    def getPath(self, x, y):
        """(n,4) array of x, y, z, heading (world frame)."""
        return self._path(self._l.dymu_planner_get_path, x, y)

    def computeGlobalPath(self, x, y):
        return bool(self._l.dymu_planner_compute_global_path(self._h, x, y))

    @property
    def current_path(self):
        return self._path(self._l.dymu_planner_get_current_path)

    def _matrix(self, kind):
        out = np.empty((self.ny, self.nx), dtype=np.float64)
        r = self._l.dymu_planner_get_matrix(self._h, kind, _ptr(out))
        if r != 1:
            raise RuntimeError("get_matrix(%d) failed (%d)" % (kind, r))
        return out

    def getTotalCostMatrix(self):
        return self._matrix(MAT_TOTAL_COST)

    def getGlobalCostMatrix(self):
        return self._matrix(MAT_GLOBAL_COST)

    def getHazardDensityMatrix(self):
        return self._matrix(MAT_HAZARD_DENSITY)

    def getTrafficabilityMatrix(self):
        return self._matrix(MAT_TRAFFICABILITY)

    def getTotalCost(self, x, y):
        return float(self._l.dymu_planner_get_total_cost(self._h, x, y))

    def getLocomotionMode(self, x, y):
        buf = C.create_string_buffer(256)
        n = self._l.dymu_planner_get_locomotion_mode(self._h, x, y, buf, 256)
        if n < 0:
            raise RuntimeError("getLocomotionMode failed")
        return buf.value.decode()

    # --- local layer ----------------------------------------------------
    def computeLocalPlanning(self, x, y, image, res):
        """Returns (repaired: bool, trajectory (n,4), localTime seconds)."""
        img = np.ascontiguousarray(image, dtype=np.uint8)
        h, w = img.shape
        cap = 1 << 16
        buf = np.empty((cap, 4), dtype=np.float64)
        n = C.c_int(0)
        t = C.c_double(0.0)
        ok = self._l.dymu_planner_compute_local_planning(
            self._h, x, y, img.ctypes.data_as(_u8p), w, h, res, _ptr(buf), cap, C.byref(n),
            C.byref(t))
        if ok < 0:
            raise RuntimeError("computeLocalPlanning failed")
        if n.value > cap:
            raise RuntimeError("trajectory longer than buffer")
        return bool(ok), buf[:n.value].copy(), t.value

    def _local(self, kind, x, y):
        cap = 1024 * 1024
        out = np.empty(cap, dtype=np.float64)
        side = self._l.dymu_planner_get_local_matrix(self._h, kind, x, y, _ptr(out), cap)
        if side < 0 or side * side > cap:
            raise RuntimeError("get_local_matrix failed (%d)" % side)
        return out[:side * side].reshape(side, side).copy()

    def getRiskMatrix(self, x, y):
        return self._local(LOCAL_RISK, x, y)

    def getDeviationMatrix(self, x, y):
        return self._local(LOCAL_DEVIATION, x, y)

    def getReconnectingIndex(self):
        return int(self._l.dymu_planner_get_reconnecting_index(self._h))

    @property
    def remaining_total_cost(self):
        return float(self._l.dymu_planner_get_remaining_total_cost(self._h))

    # --- CoRa: cost ratio updating after traverse (G.cpp:895-1038) ----------
    def initCoRaMethod(self, num_terrains, num_criteria, weights):
        w = _f64(weights)
        return self._l.dymu_planner_cora_init(self._h, num_terrains, num_criteria, _ptr(w), w.size) == 1

    def getTerrain(self, x, y):
        return int(self._l.dymu_planner_get_terrain(self._h, x, y))

    def fillTerrainInfo(self, terrain_id, data):
        d = _f64(data)
        return self._l.dymu_planner_fill_terrain_info(self._h, terrain_id, _ptr(d), d.size) == 1

    def updateCost(self, cap=4096):
        out = np.empty(cap, dtype=np.float64)
        n = self._l.dymu_planner_update_cost(self._h, _ptr(out), cap)
        if n < 0 or n > cap:
            raise RuntimeError("update_cost failed (%d)" % n)
        return out[:n].copy()

    def computeCostRatio(self, cap=64):
        out = np.empty(cap, dtype=np.float64)
        n = self._l.dymu_planner_compute_cost_ratio(self._h, _ptr(out), cap)
        if n < 0 or n > cap:
            raise RuntimeError("compute_cost_ratio failed (%d)" % n)
        return out[:n].copy()

    def recomputeCostMap(self):
        """computeCostMap again with the planner's current cost_lutable and the maps of the
        previous call (kept on the host by the reference build, in HBM by the B200 build)."""
        return self._l.dymu_planner_recompute_cost_map(self._h) == 1

    # --- diagnostics ------------------------------------------------------
    def node_field(self, field):
        out = np.empty((self.ny, self.nx), dtype=np.float64)
        r = self._l.dymu_planner_get_node_field(self._h, field, _ptr(out))
        if r != 1:
            raise RuntimeError("get_node_field(%d) failed (%d)" % (field, r))
        return out

    @property
    def last_call_seconds(self):
        return float(self._l.dymu_planner_last_call_seconds(self._h))
