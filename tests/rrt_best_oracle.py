"""get_best_solution + get_path_to (rrt.rs:183-193, :48-60) restated in C++ (tests/rrt_best_oracle.cpp) over a tree that
tests/rrt_oracle.py grew -- TEST INFRASTRUCTURE, the CPU baseline of scripts/rrt_query_batch_bench.py.  Compiled on first use, like
tests/rrt_oracle.py and with its compiler and flags, into a cache directory under the system's temporary directory."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import pyoracle as O
import rrt_oracle as RO

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = [os.path.join(_HERE, "rrt_best_oracle.cpp"), os.path.join(os.path.dirname(_HERE), "oracle", "porrt_oracle.cpp")]
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        h = hashlib.sha256(" ".join([RO._CXX] + RO._FLAGS).encode())
        for f in _SOURCES + RO._HEADERS:
            with open(f, "rb") as fh:
                h.update(fh.read())
        d = os.path.join(tempfile.gettempdir(), "porrt_rrt_oracle_%d" % os.getuid())
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "librrt_best_oracle_%s.so" % h.hexdigest()[:16])
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.run([RO._CXX] + RO._FLAGS + ["-o", tmp] + _SOURCES, check=True, capture_output=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.orc_rrt_best_path.restype = C.c_double
        L.orc_rrt_best_path.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        _LIB = L
    return _LIB


def best_path(tree):
    """tree: rrt_oracle.RRT.tree()'s (states, parent, dist, finals) -> (path[L, 2] root first, cost), or None without a final"""
    xy, parent, _, finals = (np.ascontiguousarray(a) for a in tree)
    path, out = np.empty((max(len(xy), 1), 2)), np.zeros(2, np.int64)
    cost = lib().orc_rrt_best_path(O.P(xy), O.P(parent), len(xy), O.P(finals), len(finals), O.P(path), O.P(out))
    return None if out[0] < 0 else (path[:out[1]].copy(), cost)
