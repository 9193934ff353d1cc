"""The reference's inlier graph for problems too large for orc_build_graph_bits (which materialises the n(n-1)/2 TIMs):
tests/cpp/graph_fused_oracle.cc, compiled on first use into a temporary directory with the oracle's compiler flags.
TEST INFRASTRUCTURE ONLY."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle_lib as orc

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "graph_fused_oracle.cc")
_fn = None


def _lib():
    global _fn
    if _fn is not None:
        return _fn
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    tmp = tempfile.mkdtemp(prefix="graph_fused_oracle_")
    atexit.register(shutil.rmtree, tmp, True)
    so = os.path.join(tmp, "libgraph_fused_oracle.so")
    # the flags of oracle/Makefile: -O3, OpenMP, no FP contraction
    subprocess.check_call([cxx, "-O3", "-DNDEBUG", "-fopenmp", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared",
                           "-o", so, SRC])
    f = C.CDLL(so).graph_bits_fused
    f.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, C.c_double, C.c_double,
                  C.POINTER(C.c_uint64), C.c_int, C.POINTER(C.c_int32)]
    f.restype = C.c_int64
    _fn = f
    return f


def build_graph_bits_fused(src, dst, nb, cbar2=1.0, want_bits=True):
    """(bits (n, ceil(n/64)) uint64 or None, degrees (n,) int32, edge count)."""
    s, d = orc.as_pts(src), orc.as_pts(dst)
    n = s.shape[0]
    W = (n + 63) // 64
    bits = np.zeros((n, W), dtype=np.uint64) if want_bits else None
    deg = np.zeros(n, dtype=np.int32)
    e = _lib()(orc._dp(s), orc._dp(d), n, nb, cbar2, bits.ctypes.data_as(C.POINTER(C.c_uint64)) if want_bits else None,
               W, deg.ctypes.data_as(C.POINTER(C.c_int32)))
    return bits, deg, int(e)
