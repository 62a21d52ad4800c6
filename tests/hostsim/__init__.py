"""TEST-ONLY: run the device step programs (csrc/kf_core.cuh) compiled for the host.

Lets the Kalman/adjoint math be checked against the oracle in the GPU-less build container.
Not part of the product; never imported by ``pymc_statespace_b200``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import scipy.linalg

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SO = os.path.join(HERE, "_hostsim.so")
LOG_2PI = float(np.log(2 * np.pi))

MK = {"standard": 0, "single": 0, "cholesky": 0, "univariate": 1, "steady_state": 2}


def build(force=False):
    src = os.path.join(HERE, "hostsim.cpp")
    deps = [src] + [os.path.join(ROOT, "pymc_statespace_b200", "csrc", f) for f in ("kf_core.cuh", "kf_ctx.cuh", "kf_dare.cuh", "kf_pred.cuh", "kf_smooth.cuh", "kf_p1.cuh", "kf_run.cuh")]
    if force or not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(
            ["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas",
             "-I", os.path.join(ROOT, "pymc_statespace_b200", "csrc"), src, "-o", SO]
        )
    return ctypes.CDLL(SO)


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def run(kind, data, a0, P0, T, Z, R, H, Q, c=None, d=None, strict=True, static_dims=False, do_bwd=True,
        g_loglik=None, g_ll_obs=None, full=True, pred=False, skip=(), p1=False, z_unit0=False, h_zero=False,
        t_companion=False, no_missing=False):
    """Returns (outputs6, grads dict or None, info).  ``skip``: cotangents NOT requested (null pointers, left zero)."""
    lib = build()
    f8 = lambda x: np.ascontiguousarray(np.asarray(x, dtype=np.float64))  # noqa: E731
    data, a0, P0, T, Z, R, H, Q = map(f8, (data, a0, P0, T, Z, R, H, Q))
    n, p = data.shape[0], data.shape[1]
    m, r = T.shape[-1], R.shape[-1]
    c = None if c is None else f8(c)
    d = None if d is None else f8(d)
    tv = lambda x: x is not None and x.ndim == 3  # noqa: E731
    # C = R Q R^T (time varying if R or Q is)
    if tv(R) or tv(Q):
        Rt = R if tv(R) else np.broadcast_to(R, (n,) + R.shape)
        Qt = Q if tv(Q) else np.broadcast_to(Q, (n,) + Q.shape)
        C = f8(np.einsum("tij,tjk,tlk->til", Rt, Qt, Rt))
    else:
        C = f8(R @ Q @ R.T)
    ts = np.array([m * m * tv(T), p * m * tv(Z), p * p * tv(H), m * m * (C.ndim == 3), m * tv(c), p * tv(d)],
                  dtype=np.int64)
    mk = MK[kind]
    if kind == "cholesky" and p > 1 and strict and static_dims:
        raise ValueError("MK_CHOLS has no thread-per-unit instantiation")
    if kind == "standard":
        ll_const, d_sign = (LOG_2PI if strict else p * LOG_2PI), 1.0
    elif kind == "single":
        ll_const, d_sign = LOG_2PI, (-1.0 if strict else 1.0)
    elif kind == "cholesky":
        if p > 1 and strict:
            mk = 3  # MK_CHOLS: the as-coded filter (SURVEY A.2-Q4)
        ll_const, d_sign = p * LOG_2PI, 1.0
    elif kind == "steady_state":
        ll_const, d_sign = (LOG_2PI if strict else p * LOG_2PI), (0.0 if strict else 1.0)
    else:
        ll_const, d_sign = 0.0, 1.0
    Pss = Gss = None
    if kind == "steady_state":
        Pss = f8(scipy.linalg.solve_discrete_are(T.T, Z.T, C, H))
        Gss = f8(np.linalg.inv(Z @ Pss @ Z.T + H))
    loglik = np.zeros(1)
    ll_obs = np.zeros(n) if full else None
    fs, ps = np.zeros((n, m, 1)), np.zeros((n + 1, m, 1))
    fc, pc = np.zeros((n, m, m)), np.zeros((n + 1, m, m))
    info = np.zeros(1, dtype=np.int32)
    g = None
    if do_bwd:
        g = dict(a0=np.zeros((m, 1)), P0=np.zeros((m, m)), T=np.zeros(T.shape), Z=np.zeros(Z.shape), H=np.zeros(H.shape),
                 C=np.zeros(C.shape), c=np.zeros((n, m, 1) if tv(c) else (m, 1)), d=np.zeros((n, p, 1) if tv(d) else (p, 1)),
                 Pss=np.zeros((m, m)), Gss=np.zeros((p, p)))
    gl = None if g_loglik is None else f8(np.atleast_1d(g_loglik))
    glo = None if g_ll_obs is None else f8(g_ll_obs)
    rc = lib.hostsim_run(
        mk, m, p, n, _p(data), _p(a0), _p(P0), _p(T), _p(Z), _p(H), _p(C), _p(c), _p(d), _p(Pss), _p(Gss), _p(ts),
        ctypes.c_double(ll_const), ctypes.c_double(d_sign), int(static_dims) | (2 if pred else 0) | (4 * int(p1)) | (16 if z_unit0 else 0) | (32 if h_zero else 0) | (64 if t_companion else 0) | (128 if no_missing else 0), _p(loglik), _p(ll_obs), _p(fs), _p(ps),
        _p(fc), _p(pc), _p(info), int(do_bwd), _p(gl), _p(glo),
        *([None if k in skip else _p(g[k]) for k in ("a0", "P0", "T", "Z", "H", "C", "c", "d", "Pss", "Gss")]
          if do_bwd else [None] * 10),
    )
    if rc != 0:
        raise RuntimeError(f"hostsim_run rc={rc}")
    outs = [fs, ps, fc, pc, float(loglik[0]), ll_obs]
    grads = None
    if do_bwd:
        grads = chain_to_inputs(kind, g, T, Z, R, H, Q, C, Pss, Gss)
    return outs, grads, int(info[0])


def chain_to_inputs(kind, g, T, Z, R, H, Q, C, Pss, Gss):
    """numpy epilogue: C-bar -> (R-bar, Q-bar); steady state: (Pss-bar, Gss-bar) -> DARE adjoint
    (reference utils/pytensor_scipy.py:39-60)."""
    out = {k: g[k].copy() for k in ("a0", "P0", "T", "Z", "H", "c", "d")}
    Cb = g["C"].copy()
    if kind == "steady_state":
        Fb = -Gss.T @ g["Gss"] @ Gss.T
        Xb = g["Pss"] + Z.T @ Fb @ Z
        out["Z"] += Fb @ Z @ Pss.T + Fb.T @ Z @ Pss
        out["H"] += Fb
        A_, B_ = T.T, Z.T
        K = np.linalg.solve(H + B_.T @ Pss @ B_, B_.T @ Pss @ A_)
        At = A_ - B_ @ K
        S = scipy.linalg.solve_discrete_lyapunov(At, 0.5 * (Xb + Xb.T), method="bilinear")
        out["T"] += (2 * Pss @ At @ S).T
        out["Z"] += (-2 * Pss @ At @ S @ K.T).T
        Cb = Cb + S
        out["H"] += K @ S @ K.T
    if R.ndim == 3 or Q.ndim == 3:
        n = Cb.shape[0]
        Rt = R if R.ndim == 3 else np.broadcast_to(R, (n,) + R.shape)
        Qt = Q if Q.ndim == 3 else np.broadcast_to(Q, (n,) + Q.shape)
        Rb = np.einsum("tij,tjk,tlk->til", Cb, Rt, Qt) + np.einsum("tji,tjk,tkl->til", Cb, Rt, Qt)
        Qb = np.einsum("tji,tjk,tkl->til", Rt, Cb, Rt)
        out["R"] = Rb if R.ndim == 3 else Rb.sum(0)
        out["Q"] = Qb if Q.ndim == 3 else Qb.sum(0)
    else:
        out["R"] = Cb @ R @ Q.T + Cb.T @ R @ Q
        out["Q"] = R.T @ Cb @ R
    return out
