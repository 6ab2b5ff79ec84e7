"""RRT::grow_tree (rrt.rs:102-181) restated in C++ over the oracle (tests/rrt_oracle.cpp) -- TEST INFRASTRUCTURE.

The Python mirror (tests/rrt_mirror.py) is too slow to be the reference for batches of long trees; this restatement is, and
tests/test_rrt_oracle_cpu.py pins it to the mirror bit for bit.  It is compiled on first use together with oracle/porrt_oracle.cpp,
with oracle/Makefile's flags, into a cache directory under the system's temporary directory (never into the repository), and takes
the map and goal handles of pyoracle's GridMap and SquareGoal."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SOURCES = [os.path.join(_HERE, "rrt_oracle.cpp"), os.path.join(_ORACLE, "porrt_oracle.cpp")]
_HEADERS = [os.path.join(_ORACLE, "porrt_oracle.hpp")]
# oracle/Makefile's flags: -ffp-contract=off keeps the f64 arithmetic bit-exact with the reference
_CXX = os.environ.get("ORACLE_CXX", "/usr/bin/g++")
_FLAGS = ["-std=c++17", "-O3", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-fopenmp", "-Wall", "-Wextra",
          "-fvisibility=hidden", "-shared"]
_LIB = None
vp, i64, u64, f64 = C.c_void_p, C.c_int64, C.c_uint64, C.c_double


def build():
    """-> path of the compiled library; rebuilt when a source, the header or the flags change"""
    h = hashlib.sha256(" ".join([_CXX] + _FLAGS).encode())
    for f in _SOURCES + _HEADERS:
        with open(f, "rb") as fh:
            h.update(fh.read())
    d = os.path.join(tempfile.gettempdir(), "porrt_rrt_oracle_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    so = os.path.join(d, "librrt_oracle_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(so):
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.run([_CXX] + _FLAGS + ["-o", tmp] + _SOURCES, check=True, capture_output=True)
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        for name, res, args in (("orc_rrt_new", vp, [vp, vp, vp, u64]), ("orc_rrt_free", None, [vp]),
                                ("orc_rrt_grow_tree", C.c_int, [vp, vp, vp, f64, f64, u64, u64, vp]),
                                ("orc_rrt_export", None, [vp, vp, vp, vp, vp])):
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _LIB = L
    return _LIB


class RRT:
    """rrt.rs RRT on `gridmap` (a pyoracle.GridMap) with ContinuousSampler seed `seed`; tree() -> (states[V, 2], parent[V],
    dist_from_root[V], final ids)"""

    def __init__(self, gridmap, low, up, seed=0):
        self.map = gridmap                  # keeps the map handle alive
        self.h = lib().orc_rrt_new(gridmap.h, O.P(O.f64a(low)), O.P(O.f64a(up)), seed)
        self.sizes = np.zeros(3, np.int64)

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_rrt_free(self.h)
            self.h = None

    def grow_tree(self, start, goal, max_step, search_radius, n_iter_min, n_iter_max):
        """goal: a pyoracle.SquareGoal.  -> 0 with a final node, 1 without, < -1 the panic code of the check that panicked (at
        iteration n_it())"""
        self._goal = goal
        return lib().orc_rrt_grow_tree(self.h, O.P(O.f64a(start)), goal.h, max_step, search_radius, n_iter_min, n_iter_max,
                                       O.P(self.sizes))

    def n_it(self):
        return int(self.sizes[2])

    def tree(self):
        V, F = int(self.sizes[0]), int(self.sizes[1])
        xy, par, dist, fin = np.empty((V, 2)), np.empty(V, np.int64), np.empty(V), np.empty(F, np.int64)
        lib().orc_rrt_export(self.h, O.P(xy), O.P(par), O.P(dist), O.P(fin))
        return xy, par, dist, fin
