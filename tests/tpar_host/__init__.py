"""TEST-ONLY: the time-parallel filter and adjoint (csrc/kf_tpar.cuh) compiled for the host.

``run`` emulates the CTA's blocked scans with ``nchunks`` chunks and a chosen scan tree (see tpar_host.cpp), so the
combination operators can be checked against the oracle without a GPU.  Not part of the product.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

from tests import hostsim

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "pymc_statespace_b200", "csrc")
LOG_2PI = float(np.log(2 * np.pi))
_LIB = None


def build():
    """Compiles tpar_host.cpp into a temporary directory (the source tree is left untouched)."""
    global _LIB
    if _LIB is None:
        out = os.path.join(tempfile.mkdtemp(prefix="kfb_tpar_host_"), "tpar_host.so")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-I", CSRC,
                               os.path.join(HERE, "tpar_host.cpp"), "-o", out])
        _LIB = ctypes.CDLL(out)
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def run(kind, data, a0, P0, T, Z, R, H, Q, c=None, d=None, strict=True, nchunks=8, tree=1, seed=1, do_bwd=True,
        g_loglik=None, g_ll_obs=None):
    """Returns (outputs6 in the oracle's order, grads dict or None, info, walk): walk = 0 scan, 1 sequential walk because
    an element was undefined, 2 sequential walk because the scan failed the consistency check."""
    lib = build()
    f8 = lambda x: np.ascontiguousarray(np.asarray(x, dtype=np.float64))  # noqa: E731
    data, a0, P0, T, Z, R, H, Q = map(f8, (data, a0, P0, T, Z, R, H, Q))
    n, p = data.shape[0], data.shape[1]
    assert p == 1
    m = T.shape[-1]
    c = None if c is None else f8(c)
    d = None if d is None else f8(d)
    tv = lambda x: x is not None and x.ndim == 3  # noqa: E731
    if tv(R) or tv(Q):
        Rt = R if tv(R) else np.broadcast_to(R, (n,) + R.shape)
        Qt = Q if tv(Q) else np.broadcast_to(Q, (n,) + Q.shape)
        C = f8(np.einsum("tij,tjk,tlk->til", Rt, Qt, Rt))
    else:
        C = f8(R @ Q @ R.T)
    ts = np.array([m * m * tv(T), m * tv(Z), tv(H), m * m * (C.ndim == 3), m * tv(c), tv(d)], dtype=np.int64)
    if kind == "standard":
        ll_const, d_sign = (LOG_2PI if strict else LOG_2PI), 1.0
    elif kind == "single":
        ll_const, d_sign = LOG_2PI, (-1.0 if strict else 1.0)
    elif kind == "cholesky":
        ll_const, d_sign = LOG_2PI, 1.0
    else:
        raise ValueError(kind)
    loglik, ll_obs = np.zeros(1), np.zeros(n)
    fs, ps = np.zeros((n, m, 1)), np.zeros((n + 1, m, 1))
    fc, pc = np.zeros((n, m, m)), np.zeros((n + 1, m, m))
    info, seq = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32)
    g = dict(a0=np.zeros((m, 1)), P0=np.zeros((m, m)), T=np.zeros(T.shape), Z=np.zeros(Z.shape), H=np.zeros(H.shape),
             C=np.zeros(C.shape), c=np.zeros((n, m, 1) if tv(c) else (m, 1)), d=np.zeros((n, 1, 1) if tv(d) else (1, 1)))
    gl = None if g_loglik is None else f8(np.atleast_1d(g_loglik))
    glo = None if g_ll_obs is None else f8(g_ll_obs)
    rc = lib.tpar_host_run(m, n, _p(data), _p(a0), _p(P0), _p(T), _p(Z), _p(H), _p(C), _p(c), _p(d), _p(ts),
                           ctypes.c_double(ll_const), ctypes.c_double(d_sign), int(nchunks), int(tree),
                           ctypes.c_uint(seed), _p(loglik), _p(ll_obs), _p(fs), _p(ps), _p(fc), _p(pc), _p(info),
                           _p(seq), int(do_bwd), _p(gl), _p(glo),
                           *[_p(g[k]) for k in ("a0", "P0", "T", "Z", "H", "C", "c", "d")])
    if rc != 0:
        raise RuntimeError(f"tpar_host_run rc={rc}")
    outs = [fs, ps, fc, pc, float(loglik[0]), ll_obs]
    grads = None
    if do_bwd:
        g["Pss"], g["Gss"] = None, None
        grads = hostsim.chain_to_inputs(kind, g, T, Z, R, H, Q, C, None, None)
    return outs, grads, int(info[0]), int(seq[0])
