"""ctypes view of the slope-anisotropic restatement (oracle/dymu_oracle_aniso.c); test infrastructure only.

The library is compiled on first use, with the flags of the isotropic restatement (oracle/Makefile:
no FMA contraction), into oracle/_aniso/ or, where the tree is read-only, a temporary directory.
Dense [ny, nx] planes; the directional costs are a [4, ny, nx] array in the order i-1, i+1, j-1, j+1.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "dymu_oracle_aniso.c")
DEPS = (SRC, os.path.join(HERE, "dymu_oracle.c"), os.path.join(HERE, "dymu_oracle_local.inc"))
CC = "/usr/bin/gcc"  # not $CC: see oracle/Makefile
CFLAGS = ["-O2", "-std=c11", "-fPIC", "-Wall", "-Wextra", "-ffp-contract=off"]

_dp = C.POINTER(C.c_double)
_LIB = None


def _build():
    out_dir = os.path.join(HERE, "_aniso")
    try:
        os.makedirs(out_dir, exist_ok=True)
        if not os.access(out_dir, os.W_OK):
            raise PermissionError(out_dir)
    except OSError:
        out_dir = tempfile.mkdtemp(prefix="dymu_oracle_aniso_")
    so = os.path.join(out_dir, "libdymu_oracle_aniso.so")
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in DEPS):
        subprocess.run([CC] + CFLAGS + ["-shared", SRC, "-o", so, "-lm"], check=True,
                       stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return so


def _lib():
    global _LIB
    if _LIB is None:
        lib = C.CDLL(_build())
        sig = {
            "orc_aniso_dircost": (None, [_dp, _dp, C.c_uint32, C.c_uint32, C.c_double, _dp, _dp, C.c_int, _dp]),
            "orc_aniso_march": (C.c_int, [_dp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, _dp]),
            "orc_aniso_improvable": (C.c_uint64, [_dp, _dp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                                  C.c_double]),
            "orc_aniso_path": (C.c_uint32, [_dp, _dp, _dp, C.c_uint32, C.c_uint32, C.c_double, C.c_double,
                                            C.c_double, C.c_double, C.c_uint32, C.c_uint32, _dp, C.c_uint32,
                                            C.POINTER(C.c_int)]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _LIB = lib
    return _LIB


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def aniso_dircost(elevation, ceff, gres, theta_deg, factors):
    """Directional costs a(x->m) from elevation, C_eff (+inf = impassable) and the factor table."""
    e, c = _f64(elevation), _f64(ceff)
    t, f = _f64(theta_deg).ravel(), _f64(factors).ravel()
    ny, nx = e.shape
    A = np.empty((4, ny, nx), dtype=np.float64)
    _lib().orc_aniso_dircost(e.ctypes.data_as(_dp), c.ctypes.data_as(_dp), nx, ny, gres,
                             t.ctypes.data_as(_dp), f.ctypes.data_as(_dp), t.size, A.ctypes.data_as(_dp))
    return A


def aniso_march(A, goal):
    """Heap-ordered march of the anisotropic update from T(goal) = 0; +inf where unreached."""
    A = _f64(A)
    _, ny, nx = A.shape
    T = np.empty((ny, nx), dtype=np.float64)
    _lib().orc_aniso_march(A.ctypes.data_as(_dp), nx, ny, int(goal[0]), int(goal[1]), T.ctypes.data_as(_dp))
    return T


def aniso_improvable(A, T, goal, rel_tol=0.0):
    """Number of cells (goal excluded) whose update would lower T by more than rel_tol * T."""
    A, T = _f64(A), _f64(T)
    _, ny, nx = A.shape
    return int(_lib().orc_aniso_improvable(A.ctypes.data_as(_dp), T.ctypes.data_as(_dp), nx, ny,
                                           int(goal[0]), int(goal[1]), rel_tol))


def aniso_path(A, T, elevation, gres, start_xy, tau, goal, cap=1 << 16):
    """The descent of dymu_extract_global_path on the anisotropic node vectors: ([n, 5]
    waypoints {x, y, z, dCostX, dCostY}, status)."""
    A, T, e = _f64(A), _f64(T), _f64(elevation)
    _, ny, nx = A.shape
    out = np.empty((cap, 5), dtype=np.float64)
    st = C.c_int()
    n = _lib().orc_aniso_path(A.ctypes.data_as(_dp), T.ctypes.data_as(_dp), e.ctypes.data_as(_dp), nx, ny, gres,
                              float(start_xy[0]), float(start_xy[1]), tau, int(goal[0]), int(goal[1]),
                              out.ctypes.data_as(_dp), cap, C.byref(st))
    return out[:n].copy(), st.value
