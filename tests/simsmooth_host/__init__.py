"""TEST-ONLY: the simulation smoother of csrc/kf_simsmooth.cuh compiled for the host (simsmooth_host.cpp).  ``run``
takes the same arguments and layouts as kfb_simulation_smoother for n_draws x n_series units.  Not part of the product."""
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
    """Compiles simsmooth_host.cpp into a temporary directory (the source tree is left untouched)."""
    global _LIB
    if _LIB is None:
        out = os.path.join(tempfile.mkdtemp(prefix="kfb_simsmooth_host_"), "simsmooth_host.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-I", CSRC,
                               os.path.join(HERE, "simsmooth_host.cpp"), "-o", out])
        _LIB = ctypes.CDLL(out)
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def is_static(m, p, r):
    return bool(build().simsmooth_host_is_static(m, p, r))


def run(y, mats, pc, spu, z_init, z_state, z_obs, n_draws=1, n_series=1, force_dyn=False):
    """y [n, p] or [n_series, n, p]; mats: dict of a0 P0 T Z R H Q c d, each shared (base shape) or [n_draws, ...];
    pc [U, n+1, m, m].  Returns (states [S, n, m], info [U])."""
    lib = build()
    f8 = lambda x: None if x is None else np.ascontiguousarray(np.asarray(x, dtype=np.float64))  # noqa: E731
    y = f8(y)
    T = f8(mats["T"])
    m = T.shape[-1]
    p = f8(mats["Z"]).shape[-2]
    r = f8(mats["R"]).shape[-1]
    n = y.shape[-2]
    base = {"a0": (m,), "P0": (m, m), "T": (m, m), "Z": (p, m), "R": (m, r), "H": (p, p), "Q": (r, r), "c": (m,),
            "d": (p,)}
    args = []
    for k in ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d"):
        v = f8(mats.get(k))
        size = int(np.prod(base[k]))
        if v is None:
            args += [None, 0]
            continue
        bs = size if v.size == n_draws * size and n_draws > 1 else 0
        args += [_p(v), bs]
        mats[k] = v  # keep alive
    U = n_draws * n_series
    S = U * spu
    lanes = (S + 31) // 32 * 32
    states = np.zeros((S, n, m))
    info = np.zeros(U, dtype=np.int32)
    gain = np.zeros(U * n * (m * p + p * p))
    fac = np.zeros(U * (2 * m * m + m * r + p * p + r * r))
    uscr = np.zeros(n * lanes * p)
    rscr = np.zeros(max(n - 1, 1) * lanes * m)
    ustat = np.zeros(U, dtype=np.int32)
    pc, z_init, z_state, z_obs = f8(pc), f8(z_init), f8(z_state), f8(z_obs)
    rc = lib.simsmooth_host_run(
        ctypes.c_longlong(n_draws), ctypes.c_longlong(n_series), ctypes.c_longlong(spu), n, m, p, r, _p(y),
        ctypes.c_longlong(n * p if y.ndim == 3 else 0), *[a if i % 2 == 0 else ctypes.c_longlong(a) for i, a in enumerate(args)],
        _p(pc), _p(z_init), _p(z_state), _p(z_obs), _p(states), _p(info), _p(gain), _p(fac), _p(uscr), _p(rscr),
        _p(ustat), int(force_dyn))
    if rc != 0:
        raise RuntimeError(f"simsmooth_host_run rc={rc}")
    return states, info
