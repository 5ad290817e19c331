"""ctypes wrapper of surface_oracle.c (test infrastructure): the literal T at every grid point.

The library is compiled on first use into a temporary directory, so the tests need nothing built in the
tree beyond what ``__graft_entry__.build()`` makes.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'surface_oracle.c')
_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix='surface_oracle_')
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, 'libsurface_oracle.so')
        subprocess.run(['gcc', '-O2', '-fPIC', '-fopenmp', '-Wall', '-Wextra', '-std=c11', '-shared', '-o', so, _SRC,
                        '-lm'], check=True)
        L = C.CDLL(so)
        L.oracle_surface.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                     C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_int32]
        _lib = L
    return _lib


def surface(genpos, cls, G, SP, A, t, lo, hi, n_x, n_a, n_threads=0):
    """-> (S [n, n_A, n_x, n_a] float64, nsA [n, n_A] int32); SP is [n_x*n_a, n_classes]."""
    genpos = np.ascontiguousarray(genpos, np.float64)
    cls = np.ascontiguousarray(cls, np.int32)
    G = np.ascontiguousarray(G, np.float64)
    SP = np.ascontiguousarray(SP, np.float64)
    A = np.ascontiguousarray(A, np.float64)
    t = np.ascontiguousarray(t, np.float64)
    lo = np.ascontiguousarray(lo, np.int64)
    hi = np.ascontiguousarray(hi, np.int64)
    n = len(t)
    S = np.empty((n, len(A), n_x, n_a))
    ns = np.zeros((n, len(A)), np.int32)

    def p(a):
        return a.ctypes.data_as(C.c_void_p)

    rc = lib().oracle_surface(len(genpos), p(genpos), p(cls), len(G), p(G), p(SP), SP.shape[0], len(A), p(A), n,
                              p(t), p(lo), p(hi), p(S), p(ns), int(n_threads))
    if rc != 0:
        raise MemoryError('oracle_surface failed')
    return S, ns


def problem_surface(prob, t, lo, hi):
    """``surface`` of a native.ScanProblem."""
    return surface(prob.genpos, prob.cls, prob.G, prob.SP, prob.A, t, lo, hi, prob.n_x, prob.n_a)
