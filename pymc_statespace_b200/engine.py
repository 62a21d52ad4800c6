"""Batched Kalman log-likelihood (+ adjoint) on one B200: thin host layer over ``libkfb200.so``.

torch is used for device memory, streams and (in ``dist.py``) NCCL only; all arithmetic happens in the
hand-written CUDA kernels behind the C ABI (``include/kfb200.h``).

Replaces the scan at reference ``pymc_statespace/filters/kalman_filter.py:152-159`` and PyTensor's
autodiff of it, for a whole batch of (parameter draw x series) units per launch.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Iterable, Optional

import torch

from . import _lib
from ._lib import (FILTER_KIND, KFB_FLAG_CORRECTED, KFB_FLAG_FORCE_COOP, KFB_FLAG_GENERIC_ADJOINT, KFB_FLAG_H_ZERO,
                   KFB_FLAG_NO_MISSING, KFB_FLAG_T_COMPANION, KFB_FLAG_TIME_PARALLEL, KFB_FLAG_Z_UNIT0, KfbCotangents, KfbDesc, KfbGrads, KfbInputs,
                   KfbOutputs, check, load)

MATRIX_NAMES = ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")
TV_NAMES = ("T", "Z", "R", "H", "Q", "c", "d")
OUTPUT_NAMES = ("filtered_states", "predicted_states", "filtered_covs", "predicted_covs", "loglik", "ll_obs")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class KalmanNumericalError(RuntimeError):
    """Per-unit numerical failure (non-PD innovation covariance or partially missing row)."""


class BatchedKalman:
    """One problem geometry (filter kind, n, m, p, r, #draws, #series) bound to a device.

    Inputs to ``forward`` are float64 CUDA tensors.  For each of a0,P0,T,Z,R,H,Q,c,d the layout is
    inferred from ``ndim`` relative to the base shape (a0:[m], P0:[m,m], T:[m,m], Z:[p,m], R:[m,r],
    H:[p,p], Q:[r,r], c:[m], d:[p]; trailing singleton column of a0/c/d as in the reference is accepted):
    base = shared by all draws; base+1 = one per draw ``[B,...]``; names listed in ``time_varying`` carry
    an extra time axis right before the matrix axes (``[n,...]`` or ``[B,n,...]``), i.e. time-first as in
    reference ``filters/utilities.py:9-14``.  ``y`` is ``[n,p]`` (shared) or ``[S,n,p]`` (one per series).

    ``time_parallel=True`` asks for the time-parallel kernels (one CTA per unit, scans over time: faster with few units
    and long series, see DESIGN.md section 8).  They exist for k_endog = 1, k_states <= 4 and the standard / single /
    cholesky filters; any other geometry runs the sequential kernels exactly as without the option.
    ``time_parallel_active`` says which path runs.
    """

    def __init__(self, kind: str, n: int, m: int, p: int, r: int, n_draws: int, n_series: int = 1,
                 strict_reference: bool = True, time_varying: Iterable[str] = (), device="cuda",
                 force_coop: bool = False, generic_adjoint: bool = False, z_unit0: bool = False, h_zero: bool = False,
                 pad_odd: bool = True, t_companion: bool = False, no_missing: bool = False, time_parallel: bool = False):
        kind = kind.lower()
        if kind not in FILTER_KIND:
            raise NotImplementedError("The following are valid filter types: " + ", ".join(FILTER_KIND))
        self.lib = load()
        self.kind, self.n, self.m, self.p, self.r = kind, int(n), int(m), int(p), int(r)
        self.n_draws, self.n_series = int(n_draws), int(n_series)
        self.units = self.n_draws * self.n_series
        self.strict_reference = bool(strict_reference)
        self.time_varying = frozenset(time_varying)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("pymc_statespace_b200 runs on CUDA devices only (no CPU fallback)")
        self.flags = ((0 if strict_reference else KFB_FLAG_CORRECTED) | (KFB_FLAG_FORCE_COOP if force_coop else 0)
                      | (KFB_FLAG_GENERIC_ADJOINT if generic_adjoint else 0)  # the last two: testing / A-B timing only
                      # structure promises (k_endog = 1): Z = [1, 0, ..], H = 0 - verified per unit by the forward kernel
                      | (KFB_FLAG_Z_UNIT0 if z_unit0 else 0) | (KFB_FLAG_H_ZERO if (h_zero and z_unit0) else 0)
                      # + T in companion form (only column 0 carries parameters): columns >= 1 of the T gradient come back 0
                      | (KFB_FLAG_T_COMPANION if (t_companion and h_zero and z_unit0) else 0)
                      # + no NaN in y: with all four the tape holds only what varies from step to step
                      | (KFB_FLAG_NO_MISSING if (no_missing and t_companion and h_zero and z_unit0) else 0))
        self.time_parallel = bool(time_parallel)
        if self.time_parallel and kind in ("standard", "single", "cholesky") and self.p == 1 and self.m <= 4:
            self.flags |= KFB_FLAG_TIME_PARALLEL
        self._base = {"a0": (m,), "P0": (m, m), "T": (m, m), "Z": (p, m), "R": (m, r), "H": (p, p), "Q": (r, r),
                      "c": (m,), "d": (p,)}
        self._desc = None
        self._inputs = None
        self._held = None
        self._ws = None
        self._saved = False
        # Odd k_states in 9..31 have no fused kernels of their own: the loglik (+ gradient) hot path runs the same model
        # embedded in k_states + 1 states (the extra state has zero rows / columns everywhere, stays identically zero and
        # adds only zeros to every product - exact, cf. models.pad_spec) on the tensor-core row kernels.
        self._inner = None
        self._via_inner = False
        if (pad_odd and not force_coop and m % 2 == 1 and 9 <= m <= 31 and p == 1 and not self.time_varying
                and self.n_series == 1 and kind in ("standard", "single", "cholesky", "steady_state")):
            self._inner = BatchedKalman(kind, n, m + 1, p, r, n_draws, n_series, strict_reference, (), device,
                                        generic_adjoint=generic_adjoint, pad_odd=False)

    @property
    def time_parallel_active(self) -> bool:
        """True if forward / backward run the time-parallel kernels (``time_parallel=True`` on a geometry that has them)."""
        return bool(self.flags & KFB_FLAG_TIME_PARALLEL)

    # ------------------------------------------------------------------ helpers
    def _canon(self, name, t):
        if t is None:
            return None, 0, 0
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64):
            raise TypeError(f"{name}: expected a float64 CUDA tensor")
        base = self._base[name]
        if name in ("a0", "c", "d") and t.ndim >= 2 and t.shape[-1] == 1 and t.shape[-2] == base[0]:
            t = t[..., 0]
        nb = len(base)
        tv = name in self.time_varying
        if tuple(t.shape[-nb:]) != base:
            raise ValueError(f"{name}: trailing shape {tuple(t.shape[-nb:])} != {base}")
        lead = tuple(t.shape[:-nb])
        size = 1
        for s in base:
            size *= s
        want_tv = (self.n,) if tv else ()
        if lead == want_tv:
            bs = 0
        elif lead == (self.n_draws,) + want_tv:
            bs = size * (self.n if tv else 1)
        else:
            raise ValueError(f"{name}: leading shape {lead} is neither {want_tv} nor {(self.n_draws,) + want_tv}")
        return t.contiguous(), bs, (size if tv else 0)

    def _make_desc(self, strides):
        d = KfbDesc()
        d.filter_kind, d.flags = FILTER_KIND[self.kind], self.flags
        d.n_draws, d.n_series = self.n_draws, self.n_series
        d.n, d.m, d.p, d.r = self.n, self.m, self.p, self.r
        for k, (bs, ts) in strides.items():
            setattr(d, k + "_bs", bs)
            if k in TV_NAMES:
                setattr(d, k + "_ts", ts)
        return d

    # ------------------------------------------------------------------ forward
    def forward(self, y, a0, P0, T, Z, R, H, Q, c=None, d=None, outputs=("loglik",), save_for_backward=False,
                check_info=False, out: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """``out``: optional caller-owned result buffers (name -> contiguous tensor of the documented shape, "info"
        included); anything not given is allocated.  Lets a captured CUDA graph write straight into a staging buffer."""
        self._via_inner = self._inner is not None and set(outputs) <= {"loglik"} and y.ndim <= 3 and y.shape[0] == self.n
        if self._via_inner:
            return self._inner.forward(y, *self._pad_inputs(a0, P0, T, Z, R, H, Q, c), d=d, outputs=outputs,
                                       save_for_backward=save_for_backward, check_info=check_info, out=out)
        if y.ndim >= 2 and y.shape[-1] == 1 and y.shape[-2] == self.p and y.ndim in (3, 4) and y.shape[-3] == self.n:
            y = y[..., 0]  # reference layout data[n,p,1]
        if not (y.is_cuda and y.dtype == torch.float64):
            raise TypeError("y: expected a float64 CUDA tensor")
        if tuple(y.shape) == (self.n, self.p):
            if self.n_series != 1:
                raise ValueError("y has no series axis but n_series > 1")
            y_bs = 0
        elif tuple(y.shape) == (self.n_series, self.n, self.p):
            y_bs = self.n * self.p
        else:
            raise ValueError(f"y: shape {tuple(y.shape)} is neither {(self.n, self.p)} nor "
                             f"{(self.n_series, self.n, self.p)}")
        y = y.contiguous()
        held, strides = {"y": y}, {"y": (y_bs, 0)}
        for name, t in zip(MATRIX_NAMES, (a0, P0, T, Z, R, H, Q, c, d)):
            tt, bs, ts = self._canon(name, t)
            held[name], strides[name] = tt, (bs, ts)
        desc = self._make_desc(strides)
        nbytes = ctypes.c_size_t(0)
        check(self.lib.kfb_workspace_bytes(ctypes.byref(desc), int(save_for_backward), ctypes.byref(nbytes)),
              "kfb_workspace_bytes")
        if self._ws is None or self._ws.numel() < nbytes.value:
            self._ws = None
            self._ws = torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=self.device)
        U, n, m, p = self.units, self.n, self.m, self.p
        shapes = {"loglik": (U,), "ll_obs": (U, n), "filtered_states": (U, n, m), "predicted_states": (U, n + 1, m),
                  "filtered_covs": (U, n, m, m), "predicted_covs": (U, n + 1, m, m)}
        given, out = (out or {}), {}
        for k in outputs:
            if k not in shapes:
                raise KeyError(k)
            out[k] = self._buffer(given.get(k), shapes[k], torch.float64, k)
        out["info"] = self._buffer(given.get("info"), (U,), torch.int32, "info")
        ins = KfbInputs(*[_ptr(held[k]) for k in ("y",) + MATRIX_NAMES])
        outs = KfbOutputs(*[_ptr(out.get(k)) for k in ("loglik", "ll_obs", "filtered_states", "predicted_states",
                                                        "filtered_covs", "predicted_covs", "info")])
        with torch.cuda.device(self.device):
            check(self.lib.kfb_forward(ctypes.byref(desc), ctypes.byref(ins), ctypes.byref(outs), _ptr(self._ws),
                                       self._ws.numel(), int(save_for_backward), _stream_ptr(self.device)),
                  "kfb_forward")
        self._desc, self._inputs, self._held, self._saved = desc, ins, held, bool(save_for_backward)
        if check_info:
            self.raise_on_info(out["info"])
        return out

    def _pad_inputs(self, a0, P0, T, Z, R, H, Q, c):
        from torch.nn.functional import pad

        m = self.m

        def vec(t):  # [.., m] or [.., m, 1]
            if t is None:
                return None
            return pad(t, (0, 0, 0, 1)) if (t.ndim >= 2 and t.shape[-1] == 1 and t.shape[-2] == m) else pad(t, (0, 1))

        return (vec(a0), pad(P0, (0, 1, 0, 1)), pad(T, (0, 1, 0, 1)), pad(Z, (0, 1)), pad(R, (0, 0, 0, 1)), H, Q, vec(c))

    def _buffer(self, t, shape, dtype, name):
        if t is None:
            return torch.empty(shape, dtype=dtype, device=self.device)
        if not (t.is_cuda and t.dtype == dtype and t.is_contiguous() and t.numel() == int(torch.Size(shape).numel())):
            raise TypeError(f"{name}: expected a contiguous {dtype} CUDA buffer of {tuple(shape)}")
        return t.view(shape)

    @staticmethod
    def raise_on_info(info: torch.Tensor):
        bad = torch.nonzero(info != 0)
        if bad.numel():
            u = int(bad[0, 0])
            code = int(info[u])
            if code == _lib.KFB_INFO_BAD_STRUCTURE:
                raise KalmanNumericalError(f"unit {u}: z_unit0 / h_zero was promised but Z != [1, 0, ..] or H != 0")
            if code == _lib.KFB_INFO_DARE_FAILED:
                raise KalmanNumericalError(f"unit {u}: the steady-state covariance (DARE) did not converge")
            if code == _lib.KFB_INFO_NOT_STATIONARY:
                raise KalmanNumericalError(f"unit {u}: T is not stationary, no stationary initial covariance exists")
            if code > 0:
                raise KalmanNumericalError(f"unit {u}: innovation covariance F_t not positive definite at step {code - 1}")
            raise KalmanNumericalError(
                f"unit {u}: y[{-code - 1}] is partially missing; only filter_type='univariate' supports partial rows "
                "(the reference raises LinAlgError here)")

    # ------------------------------------------------------------------ backward
    def backward(self, g_loglik: Optional[torch.Tensor] = None, g_ll_obs: Optional[torch.Tensor] = None,
                 wrt: Iterable[str] = MATRIX_NAMES, out: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """Per-unit gradients of  sum_u (g_loglik[u] * loglik[u] + sum_t g_ll_obs[u,t] * ll_obs[u,t]).
        ``out``: optional caller-owned gradient buffers (see ``forward``)."""
        if self._via_inner:
            m, wrt = self.m, tuple(wrt)
            g = self._inner.backward(g_loglik, g_ll_obs, wrt)
            cut = {"a0": lambda t: t[:, :m], "c": lambda t: t[:, :m], "P0": lambda t: t[:, :m, :m], "T": lambda t: t[:, :m, :m],
                   "Z": lambda t: t[:, :, :m], "R": lambda t: t[:, :m, :]}
            res = {}
            for k in wrt:
                t = cut[k](g[k]) if k in cut else g[k]
                buf = (out or {}).get(k)
                if buf is not None:
                    buf = self._buffer(buf, t.shape, torch.float64, k)
                    buf.copy_(t)
                    res[k] = buf
                else:
                    res[k] = t.contiguous()
            return res
        if not self._saved:
            raise RuntimeError("backward() needs a preceding forward(..., save_for_backward=True)")
        U, n = self.units, self.n
        shapes = dict(self._base)
        grads = {}
        for k in wrt:
            if k not in shapes:
                raise KeyError(k)
            lead = (U, n) if k in self.time_varying else (U,)
            grads[k] = self._buffer((out or {}).get(k), lead + shapes[k], torch.float64, k)
        for name, t in (("g_loglik", g_loglik), ("g_ll_obs", g_ll_obs)):
            if t is not None and not (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
                raise TypeError(f"{name}: expected a contiguous float64 CUDA tensor")
        if g_loglik is not None and tuple(g_loglik.shape) != (U,):
            raise ValueError("g_loglik must have shape [units]")
        if g_ll_obs is not None and tuple(g_ll_obs.shape) != (U, n):
            raise ValueError("g_ll_obs must have shape [units, n]")
        cot = KfbCotangents(_ptr(g_loglik), _ptr(g_ll_obs))
        g = KfbGrads(*[_ptr(grads.get(k)) for k in MATRIX_NAMES])
        with torch.cuda.device(self.device):
            check(self.lib.kfb_backward(ctypes.byref(self._desc), ctypes.byref(self._inputs), ctypes.byref(cot),
                                        ctypes.byref(g), _ptr(self._ws), self._ws.numel(), _stream_ptr(self.device)),
                  "kfb_backward")
        return grads


TIME_PARALLEL_SMOOTHER_MAX_STATES = 4  # kfb_smoother_ex with KFB_FLAG_TIME_PARALLEL covers k_states 1..4


def smoother_workspace_numel(n_draws: int, m: int) -> int:
    """float64 elements of the workspace rts_smoother needs (R Q R^T per draw; enough whether or not R, Q are shared)."""
    return max(n_draws, 1) * m * m


def rts_smoother(T, R, Q, filtered_states, filtered_covs, n_series: int = 1, time_parallel: bool = False, out=None,
                 workspace=None):
    """Batched RTS smoother (reference filters/kalman_smoother.py:56-104; SURVEY section 8(f) row f2).
    T:[B,m,m]|[m,m], R:[B,m,r]|[m,r], Q:[B,r,r]|[r,r] static; filtered_states [U,n,m], filtered_covs [U,n,m,m]
    (outputs of BatchedKalman.forward).  Returns (smoothed_states [U,n,m], smoothed_covs [U,n,m,m]).

    ``time_parallel=True`` runs the time-parallel kernel (one CTA per unit, a scan over time; faster for few units over
    long series) for k_states <= 4; at larger k_states the sequential kernel runs, as BatchedKalman falls back.
    ``out=(ss, sc)`` and ``workspace`` (float64, ``smoother_workspace_numel(n_draws, m)`` elements) may be preallocated, so
    that a CUDA graph can capture the call without allocating."""
    lib = load()
    fs, fc = filtered_states.contiguous(), filtered_covs.contiguous()
    U, n, m = fs.shape
    r = R.shape[-1]
    T, R, Q = T.contiguous(), R.contiguous(), Q.contiguous()
    n_draws = U // n_series
    for name, t, nd in (("T", T, 2), ("R", R, 2), ("Q", Q, 2)):
        if t.ndim == nd + 1 and t.shape[0] != n_draws:
            raise ValueError(f"{name}: leading dimension {t.shape[0]} != n_draws {n_draws}")
    if out is None:
        ss, sc = torch.empty_like(fs), torch.empty_like(fc)
    else:
        ss, sc = out
        if ss.shape != fs.shape or sc.shape != fc.shape or not (ss.is_contiguous() and sc.is_contiguous()):
            raise ValueError("out: contiguous tensors of the shapes of filtered_states and filtered_covs")
    ws = workspace
    if ws is None:
        ws = torch.empty(smoother_workspace_numel(n_draws, m), dtype=torch.float64, device=fs.device)
    flags = KFB_FLAG_TIME_PARALLEL if time_parallel and m <= TIME_PARALLEL_SMOOTHER_MAX_STATES else 0
    with torch.cuda.device(fs.device):
        check(lib.kfb_smoother_ex(n_draws, n_series, n, m, r, _ptr(T), m * m if T.ndim == 3 else 0, _ptr(R),
                                  m * r if R.ndim == 3 else 0, _ptr(Q), r * r if Q.ndim == 3 else 0, _ptr(fs), _ptr(fc),
                                  _ptr(ss), _ptr(sc), _ptr(ws), ws.numel() * 8, flags, _stream_ptr(fs.device)),
              "kfb_smoother_ex")
    return ss, sc


def lyapunov_forward(A: torch.Tensor, R: torch.Tensor, Q: torch.Tensor):
    """X = A X A^T + R Q R^T per draw (reference models/SARIMAX.py:100-107).  A:[B,m,m], R:[B,m,r]|[m,r],
    Q:[B,r,r]|[r,r].  Returns (X[B,m,m], info[B])."""
    lib = load()
    B, m = A.shape[0], A.shape[-1]
    r = R.shape[-1]
    A, R, Q = A.contiguous(), R.contiguous(), Q.contiguous()
    X = torch.empty((B, m, m), dtype=torch.float64, device=A.device)
    info = torch.empty((B,), dtype=torch.int32, device=A.device)
    with torch.cuda.device(A.device):
        check(lib.kfb_lyapunov_forward(B, m, r, _ptr(A), m * m, _ptr(R), m * r if R.ndim == 3 else 0, _ptr(Q),
                                       r * r if Q.ndim == 3 else 0, _ptr(X), _ptr(info), _stream_ptr(A.device)),
              "kfb_lyapunov_forward")
    return X, info


def lyapunov_backward(A, R, Q, X, Xbar, Abar, Rbar, Qbar):
    """Accumulates (+=) into Abar[B,m,m], Rbar[B,m,r], Qbar[B,r,r] (any may be None)."""
    lib = load()
    B, m = A.shape[0], A.shape[-1]
    r = R.shape[-1]
    A, R, Q, X, Xbar = (t.contiguous() for t in (A, R, Q, X, Xbar))
    with torch.cuda.device(A.device):
        check(lib.kfb_lyapunov_backward(B, m, r, _ptr(A), m * m, _ptr(R), m * r if R.ndim == 3 else 0, _ptr(Q),
                                        r * r if Q.ndim == 3 else 0, _ptr(X), _ptr(Xbar), _ptr(Abar), _ptr(Rbar),
                                        _ptr(Qbar), _stream_ptr(A.device)),
              "kfb_lyapunov_backward")


def fp64_peak_tflops(device="cuda", iters=4096, repeats=5, distinct_operands=False, warps_per_smsp=16):
    """Measured FP64 FMA throughput (TFLOP/s) of this GPU: the "FP64 roofline" denominator.
    ``distinct_operands=True``: every FMA reads three different registers (no operand reuse)."""
    lib = load()
    fn = lib.kfb_fp64_peak_distinct if distinct_operands else lib.kfb_fp64_peak
    dev = torch.device(device)
    sink = torch.zeros(8, dtype=torch.float64, device=dev)
    flops = ctypes.c_double(0)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    best = 0.0
    with torch.cuda.device(dev):
        for i in range(repeats + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            blocks = max(1, (sms * 4 * warps_per_smsp * 32) // 256)
            check(fn(iters, blocks, 256, _ptr(sink), ctypes.byref(flops), _stream_ptr(dev)), "kfb_fp64_peak")
            e1.record()
            e1.synchronize()
            if i:
                best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best
