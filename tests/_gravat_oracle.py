"""The checker of `sph_gravity_at` (TEST INFRASTRUCTURE): oracle/sph_oracle.cpp compiled unchanged together with one
entry point, tests/_gravat_oracle.cpp, into a library in the temporary directory.  Not a test module.

`GravAtOracle` is an oracle.oracle.Oracle on that library (upload, evaluate, accel_parts, conserved ... as usual) with
`gravity_at(points, h=None)`: the dict of the nine columns for the tree of the last evaluation."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.oracle import Oracle
from summersph_b200._abi import SphParams

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "_gravat_oracle.cpp"), os.path.join(ROOT, "oracle", "sph_oracle.cpp"), os.path.join(ROOT, "include", "sph_b200.h")]
FLAGS = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-std=c++17", "-fopenmp", "-shared"]      # oracle/Makefile's
COLS = ("phi_gas", "gx_gas", "gy_gas", "gz_gas", "phi_sink", "gx_sink", "gy_sink", "gz_sink", "accepted")
_LIB = None


def build():
    dig = hashlib.sha256()
    for s in SOURCES:
        with open(s, "rb") as f:
            dig.update(f.read())
    so = os.path.join(tempfile.gettempdir(), f"sph_gravat_oracle_{os.getuid()}_{dig.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"
        tmp = f"{so}.{os.getpid()}"
        subprocess.check_call([cxx] + FLAGS + ["-o", tmp, SOURCES[0]])
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.orc_create.restype = C.c_void_p
        L.orc_create.argtypes = [C.POINTER(SphParams), C.c_int]
        L.orc_lookup_grav_kernel.restype = C.c_double
        L.orc_lookup_grav_kernel.argtypes = [C.c_void_p, C.c_double, C.c_double]
        L.orc_G.restype = C.c_double
        L.orc_download_neighbours.restype = C.c_int64
        L.orc_kick.argtypes = [C.c_void_p, C.c_double]
        L.orc_drift.argtypes = [C.c_void_p, C.c_double]
        L.orc_gravity_at.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 5
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class GravAtOracle(Oracle):
    def __init__(self, params: SphParams, threads=1):
        self.params = params
        self._l = lib()
        self._c = C.c_void_p(self._l.orc_create(C.byref(params), int(threads)))

    def gravity_at(self, points, h=None):
        pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
        m = len(pts)
        cols = [np.ascontiguousarray(pts[:, k]) for k in range(3)]
        hh = None if h is None else np.ascontiguousarray(np.broadcast_to(np.asarray(h, dtype=np.float64), (m,)))
        out = np.zeros(len(COLS) * m)
        self._l.orc_gravity_at(self._c, m, *[_p(c) for c in cols], _p(hh), _p(out))
        return {k: out[i * m:(i + 1) * m] for i, k in enumerate(COLS)}
