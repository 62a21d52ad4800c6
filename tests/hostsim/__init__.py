"""TEST-ONLY: the device code of csrc/ compiled for the host, so that the Kalman / adjoint math can be checked against the
oracle without a GPU.  One library is built from the .cpp files here:

* hostsim.cpp - the sequential filters and adjoints (kf_core.cuh, kf_pred.cuh, kf_p1.cuh), the DARE and the RTS smoother;
* tpar.cpp - the time-parallel filter, adjoint and smoother (kf_tpar.cuh, kf_tpar_smooth.cuh) with emulated CTA scans;
* draws.cpp - the simulation smoother, forecast paths, impulse responses and conditional forecasts (kf_simsmooth.cuh,
  kf_forecast.cuh, kf_condfc.cuh); its Python entry points are in ``tests.hostsim.draws``.

The filter entry points take the C ABI's filter kind and KFB_FLAG_* bits and apply the library's own rules to them
(kf_run.cuh); the entry points of draws.cpp take the C ABI's own arguments and build the kernels' arguments and
workspace with the library's builders (kf_draws_run.cuh).  Not part of the product; never imported by
``pymc_statespace_b200``.
"""
from __future__ import annotations

import ctypes
import glob
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import scipy.linalg

from pymc_statespace_b200._lib import (FILTER_KIND, KFB_FLAG_CORRECTED, KFB_FLAG_H_ZERO, KFB_FLAG_NO_MISSING,
                                       KFB_FLAG_T_COMPANION, KFB_FLAG_Z_UNIT0)

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "pymc_statespace_b200", "csrc")
SOURCES = sorted(glob.glob(os.path.join(HERE, "*.cpp")))
COMPILE = ["g++", "-O1", "-std=c++17", "-fPIC", "-Wno-unknown-pragmas", "-I", CSRC, "-c"]
LINK = ["g++", "-shared"]
_LIB = None


def _digest():
    """Hash of the compile and link commands and of every file the library can be built from."""
    h = hashlib.sha256(repr((COMPILE, LINK)).encode())
    files = list(SOURCES)
    for top in (CSRC, os.path.join(ROOT, "include")):
        files += [os.path.join(d, f) for d, _, fs in os.walk(top) for f in fs]
    for f in sorted(files):
        h.update(os.path.relpath(f, ROOT).encode() + b"\0")
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:24]


def build():
    """Compiles each .cpp here to an object (in parallel), links them into one library in a per-user cache directory
    outside the source tree, named by _digest(), and loads it once per process.  A library of that name is reused."""
    global _LIB
    if _LIB is None:
        cache = os.path.join(tempfile.gettempdir(), f"kfb_hostsim_{os.getuid()}")
        so = os.path.join(cache, f"hostsim_{_digest()}.so")
        if not os.path.exists(so):
            os.makedirs(cache, exist_ok=True)
            with tempfile.TemporaryDirectory(dir=cache) as tmp:
                objs = [os.path.join(tmp, os.path.basename(s)[:-4] + ".o") for s in SOURCES]
                procs = [subprocess.Popen(COMPILE + [s, "-o", o]) for s, o in zip(SOURCES, objs)]
                if any([p.wait() for p in procs]):
                    raise RuntimeError("g++ failed on the host build of the kernels")
                subprocess.check_call(LINK + objs + ["-o", os.path.join(tmp, "hostsim.so")])
                os.replace(os.path.join(tmp, "hostsim.so"), so)  # atomic: concurrent sessions see all or nothing
        _LIB = ctypes.CDLL(so)
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def f8(x):
    return None if x is None else np.ascontiguousarray(np.asarray(x, dtype=np.float64))


def _system(data, a0, P0, T, Z, R, H, Q, c, d, full, do_bwd):
    """One unit's inputs as the filter entry points take them (C = R Q R^T, time strides of T, Z, H, C, c, d) and
    zeroed outputs, per-step outputs if ``full``, and cotangents of the kernels' inputs if ``do_bwd``."""
    data, a0, P0, T, Z, R, H, Q, c, d = map(f8, (data, a0, P0, T, Z, R, H, Q, c, d))
    n, p = data.shape[0], data.shape[1]
    m = T.shape[-1]
    tv = lambda x: x is not None and x.ndim == 3  # noqa: E731
    if tv(R) or tv(Q):  # C is time varying if R or Q is
        Rt = R if tv(R) else np.broadcast_to(R, (n,) + R.shape)
        Qt = Q if tv(Q) else np.broadcast_to(Q, (n,) + Q.shape)
        C = f8(np.einsum("tij,tjk,tlk->til", Rt, Qt, Rt))
    else:
        C = f8(R @ Q @ R.T)
    ts = np.array([m * m * tv(T), p * m * tv(Z), p * p * tv(H), m * m * (C.ndim == 3), m * tv(c), p * tv(d)],
                  dtype=np.int64)
    g = None
    if do_bwd:
        g = dict(a0=np.zeros((m, 1)), P0=np.zeros((m, m)), T=np.zeros(T.shape), Z=np.zeros(Z.shape), H=np.zeros(H.shape),
                 C=np.zeros(C.shape), c=np.zeros((n, m, 1) if tv(c) else (m, 1)), d=np.zeros((n, p, 1) if tv(d) else (p, 1)),
                 Pss=np.zeros((m, m)), Gss=np.zeros((p, p)))
    return dict(n=n, m=m, p=p, y=data, a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q, C=C, c=c, d=d, ts=ts, g=g,
                loglik=np.zeros(1), ll_obs=np.zeros(n) if full else None, fs=np.zeros((n, m, 1)),
                ps=np.zeros((n + 1, m, 1)), fc=np.zeros((n, m, m)), pc=np.zeros((n + 1, m, m)),
                info=np.zeros(1, dtype=np.int32))


def _inputs(s):
    return [_p(s[k]) for k in ("y", "a0", "P0", "T", "Z", "H", "C", "c", "d")]


def _outputs(s):
    return [_p(s[k]) for k in ("loglik", "ll_obs", "fs", "ps", "fc", "pc", "info")]


def _results(s):
    return [s["fs"], s["ps"], s["fc"], s["pc"], float(s["loglik"][0]), s["ll_obs"]]


def _cotangent_seeds(g_loglik, g_ll_obs):
    return _p(None if g_loglik is None else f8(np.atleast_1d(g_loglik))), _p(f8(g_ll_obs))


def _flags(strict, z_unit0=False, h_zero=False, t_companion=False, no_missing=False):
    return ((0 if strict else KFB_FLAG_CORRECTED) | (KFB_FLAG_Z_UNIT0 if z_unit0 else 0) | (KFB_FLAG_H_ZERO if h_zero else 0)
            | (KFB_FLAG_T_COMPANION if t_companion else 0) | (KFB_FLAG_NO_MISSING if no_missing else 0))


def run(kind, data, a0, P0, T, Z, R, H, Q, c=None, d=None, strict=True, static_dims=False, do_bwd=True,
        g_loglik=None, g_ll_obs=None, full=True, pred=False, skip=(), p1=False, z_unit0=False, h_zero=False,
        t_companion=False, no_missing=False):
    """Returns (outputs6, grads dict or None, info).  ``skip``: cotangents NOT requested (null pointers, left zero).
    Choices of the tests: ``static_dims`` runs the thread-per-unit instantiations (else the run-time-dims context),
    ``pred`` the one-step-predictor programs (else the two-stage reference programs), ``p1`` the k_endog = 1 kernels of
    kf_p1.cuh (2: the generic forward, then their adjoint)."""
    lib = build()
    s = _system(data, a0, P0, T, Z, R, H, Q, c, d, full, do_bwd)
    Pss = Gss = None
    if kind == "steady_state":  # the kernels take the DARE solution as an input
        Pss = f8(scipy.linalg.solve_discrete_are(s["T"].T, s["Z"].T, s["C"], s["H"]))
        Gss = f8(np.linalg.inv(s["Z"] @ Pss @ s["Z"].T + s["H"]))
    g = s["g"]
    rc = lib.hostsim_run(
        FILTER_KIND[kind], _flags(strict, z_unit0, h_zero, t_companion, no_missing), s["m"], s["p"], s["n"],
        *_inputs(s), _p(Pss), _p(Gss), _p(s["ts"]), int(static_dims), int(pred), int(p1), *_outputs(s), int(do_bwd),
        *_cotangent_seeds(g_loglik, g_ll_obs),
        *([None if k in skip else _p(g[k]) for k in ("a0", "P0", "T", "Z", "H", "C", "c", "d", "Pss", "Gss")]
          if do_bwd else [None] * 10),
    )
    if rc != 0:
        raise RuntimeError(f"hostsim_run rc={rc}")
    grads = chain_to_inputs(kind, g, s["T"], s["Z"], s["R"], s["H"], s["Q"], s["C"], Pss, Gss) if do_bwd else None
    return _results(s), grads, int(s["info"][0])


def tpar_run(kind, data, a0, P0, T, Z, R, H, Q, c=None, d=None, strict=True, nchunks=8, tree=1, seed=1, do_bwd=True,
             g_loglik=None, g_ll_obs=None):
    """The time-parallel filter and adjoint (k_endog = 1) with ``nchunks`` chunks and scan tree ``tree`` (tpar.cpp).
    Returns (outputs6 in the oracle's order, grads dict or None, info, walk): walk = 0 scan, 1 sequential walk because
    an element was undefined, 2 sequential walk because the scan failed the consistency check."""
    lib = build()
    s = _system(data, a0, P0, T, Z, R, H, Q, c, d, True, True)
    g, seq = s["g"], np.zeros(1, dtype=np.int32)
    rc = lib.tpar_host_run(FILTER_KIND[kind], _flags(strict), s["m"], s["n"], *_inputs(s), _p(s["ts"]), int(nchunks),
                           int(tree), ctypes.c_uint(seed), *_outputs(s), _p(seq), int(do_bwd),
                           *_cotangent_seeds(g_loglik, g_ll_obs), *[_p(g[k]) for k in ("a0", "P0", "T", "Z", "H", "C", "c", "d")])
    if rc != 0:
        raise RuntimeError(f"tpar_host_run rc={rc}")
    grads = chain_to_inputs(kind, g, s["T"], s["Z"], s["R"], s["H"], s["Q"], s["C"], None, None) if do_bwd else None
    return _results(s), grads, int(s["info"][0]), int(seq[0])


def _smooth_prep(T, R, Q, fs, fc):
    T, R, Q, fs, fc = map(f8, (T, R, Q, fs, fc))
    n, m = fc.shape[0], fc.shape[-1]
    return T, f8(R @ Q @ R.T), f8(fs.reshape(n, m)), fc, n, m


def tpar_smooth(T, R, Q, fs, fc, nchunks=8, tree=1, seed=1, tol=1e-10):
    """The time-parallel RTS smoother (tpar.cpp).  Returns (smoothed_states [n,m,1], smoothed_covs [n,m,m], fallback):
    fallback = 1 if the walk disagreed with the scan and the unit was re-run by the sequential recursion."""
    lib = build()
    T, C, fs, fc, n, m = _smooth_prep(T, R, Q, fs, fc)
    ss, sc = np.zeros((n, m)), np.zeros((n, m, m))
    fb = np.zeros(1, dtype=np.int32)
    rc = lib.tpar_host_smooth_run(m, n, _p(T), _p(C), _p(fs), _p(fc), _p(ss), _p(sc), int(nchunks), int(tree),
                                  ctypes.c_uint(seed), ctypes.c_double(tol), _p(fb))
    if rc != 0:
        raise RuntimeError(f"tpar_host_smooth_run rc={rc}")
    return ss[..., None], sc, int(fb[0])


def smoother(T, R, Q, fs, fc, static_dims=False):
    """The sequential RTS smoother of kf_smooth.cuh: in the run-time-dims context, or with ``static_dims`` in the
    thread-per-unit context TX<M> of k_states 1..4.  Returns (smoothed_states [n,m,1], smoothed_covs [n,m,m])."""
    lib = build()
    T, C, fs, fc, n, m = _smooth_prep(T, R, Q, fs, fc)
    ss, sc = np.zeros((n, m)), np.zeros((n, m, m))
    entry = lib.tpar_host_smooth_sequential if static_dims else lib.hostsim_smoother
    if entry(n, m, _p(T), _p(C), _p(fs), _p(fc), _p(ss), _p(sc)) != 0:
        raise RuntimeError("host smoother")
    return ss[..., None], sc


def dare(T, Z, H, C, gPss, gGss):
    """The DARE solve and its adjoint (kf_dare.cuh, run-time dims).  Returns (Pss, Gss, dict of T, Z, H, C cotangents)
    for the cotangents gPss, gGss of P_ss and F^-1 = (Z P_ss Z^T + H)^-1."""
    lib = build()
    T, Z, H, C, gPss, gGss = map(f8, (T, Z, H, C, gPss, gGss))
    m, p = T.shape[0], Z.shape[0]
    Pss, Gss = np.zeros((m, m)), np.zeros((p, p))
    g = dict(T=np.zeros((m, m)), Z=np.zeros((p, m)), H=np.zeros((p, p)), C=np.zeros((m, m)))
    rc = lib.hostsim_dare(m, p, _p(T), _p(Z), _p(H), _p(C), _p(Pss), _p(Gss), 1, _p(gPss), _p(gGss),
                          *[_p(g[k]) for k in ("T", "Z", "H", "C")])
    if rc != 0:
        raise RuntimeError(f"hostsim_dare rc={rc}")
    return Pss, Gss, g


def simsmooth_is_static(m, p, r):
    """True if (m, p, r) has a compile-time instantiation of the simulation smoother."""
    return bool(build().draws_host_is_static(m, p, r))


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
