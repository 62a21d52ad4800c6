"""TEST-ONLY: the reduced ARMA kernels of kf_p1.cuh compiled for the host, one unit, with the adjoint instantiation the
kernels would pick for the requested cotangents (p1ctape_host.cpp).  Never imported by ``pymc_statespace_b200``."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SO = os.path.join(HERE, "_p1ctape_host.so")
CSRC = os.path.join(ROOT, "pymc_statespace_b200", "csrc")


def build():
    src = os.path.join(HERE, "p1ctape_host.cpp")
    deps = [src] + [os.path.join(CSRC, f) for f in ("kf_core.cuh", "kf_p1.cuh")]
    if not os.path.exists(SO) or any(os.path.getmtime(f) > os.path.getmtime(SO) for f in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-I", CSRC, src,
                               "-o", SO])
    return ctypes.CDLL(SO)


def run(y, a0, P0, T, C, c, d, g_ll_obs=None, want_cd=True):
    """Loglik, info and the cotangents of a0, P0, T, C (and c, d when want_cd) of one unit with Z = e0, H = 0, a
    companion T and complete data (the reduced recursion).  Cotangent of every ll_t: 1, plus g_ll_obs[t] if given."""
    lib = build()
    f8 = lambda x: np.ascontiguousarray(np.asarray(x, dtype=np.float64))  # noqa: E731
    y, a0, P0, T, C, c, d = map(f8, (np.ravel(y), np.ravel(a0), P0, T, C, np.ravel(c), np.ravel(d)))
    n, m = y.shape[0], T.shape[0]
    glo = None if g_ll_obs is None else f8(g_ll_obs)
    p = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    loglik, info = np.zeros(1), np.zeros(1, dtype=np.int32)
    g = {"a0": np.zeros(m), "P0": np.zeros((m, m)), "T": np.zeros((m, m)), "C": np.zeros((m, m))}
    if want_cd:
        g["c"], g["d"] = np.zeros(m), np.zeros(1)
    rc = lib.p1ctape_run(m, n, p(y), p(a0), p(P0), p(T), p(C), p(c), p(d), ctypes.c_double(float(np.log(2 * np.pi))),
                         p(glo), p(loglik), p(info), p(g["a0"]), p(g["P0"]), p(g["T"]), p(g["C"]), p(g.get("c")),
                         p(g.get("d")))
    if rc != 0:
        raise RuntimeError(f"p1ctape_run rc={rc}")
    return float(loglik[0]), int(info[0]), g
