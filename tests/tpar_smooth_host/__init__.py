"""TEST-ONLY: the time-parallel RTS smoother (csrc/kf_tpar_smooth.cuh) compiled for the host.

``run`` emulates the CTA's fold, suffix scan and checked walk with ``nchunks`` chunks and a chosen scan tree (see
tpar_smooth_host.cpp), so the smoothing elements and their combination can be checked against the oracle without a
GPU.  ``sequential`` runs the sequential smoother of kf_smooth.cuh the same way.  Not part of the product.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "pymc_statespace_b200", "csrc")
_LIB = None


def build():
    """Compiles tpar_smooth_host.cpp into a temporary directory (the source tree is left untouched)."""
    global _LIB
    if _LIB is None:
        out = os.path.join(tempfile.mkdtemp(prefix="kfb_tpar_smooth_host_"), "tpar_smooth_host.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-I", CSRC,
                               os.path.join(HERE, "tpar_smooth_host.cpp"), "-o", out])
        _LIB = ctypes.CDLL(out)
    return _LIB


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _prep(T, R, Q, fs, fc):
    f8 = lambda x: np.ascontiguousarray(np.asarray(x, dtype=np.float64))  # noqa: E731
    T, R, Q, fs, fc = map(f8, (T, R, Q, fs, fc))
    C = f8(R @ Q @ R.T)
    n, m = fc.shape[0], fc.shape[-1]
    return T, C, f8(fs.reshape(n, m)), fc, n, m


def run(T, R, Q, fs, fc, nchunks=8, tree=1, seed=1, tol=1e-10):
    """Returns (smoothed_states [n,m,1], smoothed_covs [n,m,m], fallback): fallback = 1 if the walk disagreed with the
    scan and the unit was re-run by the sequential recursion."""
    lib = build()
    T, C, fs, fc, n, m = _prep(T, R, Q, fs, fc)
    ss, sc = np.zeros((n, m)), np.zeros((n, m, m))
    fb = np.zeros(1, dtype=np.int32)
    rc = lib.tpar_smooth_host_run(m, n, _p(T), _p(C), _p(fs), _p(fc), _p(ss), _p(sc), int(nchunks), int(tree),
                                  ctypes.c_uint(seed), ctypes.c_double(tol), _p(fb))
    if rc != 0:
        raise RuntimeError(f"tpar_smooth_host_run rc={rc}")
    return ss[..., None], sc, int(fb[0])


def sequential(T, R, Q, fs, fc):
    lib = build()
    T, C, fs, fc, n, m = _prep(T, R, Q, fs, fc)
    ss, sc = np.zeros((n, m)), np.zeros((n, m, m))
    if lib.tpar_smooth_host_sequential(m, n, _p(T), _p(C), _p(fs), _p(fc), _p(ss), _p(sc)) != 0:
        raise RuntimeError("tpar_smooth_host_sequential")
    return ss[..., None], sc
