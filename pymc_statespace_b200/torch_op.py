"""Eager / autograd entry for ONE model in the reference's shapes (used by ``filters.py``).

``log_likelihood`` and ``ll_obs`` are differentiable wrt (a0, P0, T, Z, R, H, Q, c, d) through the adjoint kernel;
the filtered / predicted moments are returned detached (the reference only ever differentiates the
``pm.Potential("log_likelihood")`` term, ``pymc_statespace/core/statespace.py:174``).
"""
from __future__ import annotations

import numpy as np
import torch

from .engine import MATRIX_NAMES, BatchedKalman

_OUT = ("filtered_states", "predicted_states", "filtered_covs", "predicted_covs", "loglik", "ll_obs")


def _raise_info(info: int):
    from ._lib import KFB_INFO_DARE_FAILED

    if info == KFB_INFO_DARE_FAILED:
        raise np.linalg.LinAlgError("the steady-state covariance could not be computed: the discrete algebraic Riccati "
                                    "equation has no stabilising solution for these matrices (scipy's solve_discrete_are "
                                    "raises LinAlgError at this point in the reference)")
    if info > 0:
        raise np.linalg.LinAlgError(
            f"innovation covariance F_t is not positive definite at step {info - 1} "
            "(scipy's solve(assume_a='pos') / cholesky raise LinAlgError at this point in the reference)")
    raise np.linalg.LinAlgError(
        f"y[{-info - 1}] is partially missing: the masked F_t is singular (the reference raises LinAlgError here, "
        "SURVEY.md A.2-Q2); use filter_type='univariate' for partially observed rows")


class _KalmanFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, bk, y, present, *mats):
        full = dict(zip(present, mats))
        args = [full.get(k) for k in MATRIX_NAMES]
        needs = [k for k, t in full.items() if t.requires_grad]
        out = bk.forward(y, *[None if a is None else a.detach()[None] for a in args], outputs=_OUT,
                         save_for_backward=bool(needs))
        info = int(out["info"][0])
        if info != 0:
            _raise_info(info)
        ctx.bk, ctx.present, ctx.needs = bk, present, needs
        ctx.shapes = {k: t.shape for k, t in full.items()}
        res = tuple(out[k][0] for k in _OUT)
        ctx.mark_non_differentiable(*res[:4])
        return res

    @staticmethod
    def backward(ctx, g_fs, g_ps, g_fc, g_pc, g_ll, g_llobs):
        bk = ctx.bk
        dev = bk.device
        gl = torch.zeros(1, dtype=torch.float64, device=dev) if g_ll is None else g_ll.reshape(1).contiguous()
        glo = None if g_llobs is None else g_llobs.reshape(1, bk.n).contiguous()
        grads = bk.backward(g_loglik=gl, g_ll_obs=glo, wrt=ctx.needs)
        res = []
        for k in ctx.present:
            res.append(grads[k][0].reshape(ctx.shapes[k]) if k in ctx.needs else None)
        return (None, None, None, *res)


_BK_CACHE = {}


def _evaluator(flt, n, m, p, r, tv, device):
    """One BatchedKalman (and its workspace) per problem geometry: PyMC calls the Op once per leapfrog step with the
    same shapes, so the evaluator and its device buffers are built once (ADVICE r1)."""
    tpar = bool(getattr(flt, "time_parallel", False))
    key = (flt.kind, n, m, p, r, bool(flt.strict_reference), tpar, tuple(tv), str(device))
    bk = _BK_CACHE.get(key)
    if bk is None:
        if len(_BK_CACHE) > 64:
            _BK_CACHE.clear()
        bk = _BK_CACHE[key] = BatchedKalman(flt.kind, n, m, p, r, n_draws=1, strict_reference=flt.strict_reference,
                                            time_varying=tv, device=device, time_parallel=tpar)
    return bk


def kalman_logp_grads(flt, data, mats, g_loglik=1.0, g_ll_obs=None):
    """What the gradient Op needs and nothing more: ONE loglik-only forward pass (hot-path kernels, tape saved) + the
    adjoint kernel.  ``mats``: name -> float64 CUDA tensor in the reference's shapes (a0[m,1], P0[m,m], ..., optional c, d).
    Returns (loglik 0-d tensor, {name: cotangent with the input's shape}) for
    ``g_loglik * loglik + sum_t g_ll_obs[t] * ll_obs[t]``."""
    full = {k: mats.get(k) for k in MATRIX_NAMES}
    n, m, p, r, tv = flt._validate(data, *[full[k] for k in MATRIX_NAMES])
    bk = _evaluator(flt, n, m, p, r, tv, data.device)
    present = tuple(k for k in MATRIX_NAMES if full[k] is not None)
    out = bk.forward(data[..., 0].contiguous(), *[None if full[k] is None else full[k].detach()[None] for k in MATRIX_NAMES],
                     outputs=("loglik",), save_for_backward=True)
    info = int(out["info"][0])
    if info != 0:
        _raise_info(info)
    dev = data.device
    gl = torch.as_tensor(g_loglik, dtype=torch.float64, device=dev).reshape(1).contiguous()
    glo = None if g_ll_obs is None else torch.as_tensor(g_ll_obs, dtype=torch.float64, device=dev).reshape(1, n).contiguous()
    grads = bk.backward(g_loglik=gl, g_ll_obs=glo, wrt=present)
    return out["loglik"][0], {k: grads[k][0].reshape(full[k].shape) for k in present}


def kalman_filter_torch(flt, data, a0, P0, T, Z, R, H, Q, c=None, d=None):
    """data[n,p,1], a0[m,1], ... float64 CUDA tensors -> the reference's 6-list (torch tensors)."""
    n, m, p, r, tv = flt._validate(data, a0, P0, T, Z, R, H, Q, c, d)
    bk = _evaluator(flt, n, m, p, r, tv, data.device)
    full = {"a0": a0, "P0": P0, "T": T, "Z": Z, "R": R, "H": H, "Q": Q, "c": c, "d": d}
    present = tuple(k for k in MATRIX_NAMES if full[k] is not None)
    fs, ps, fc, pc, ll, llo = _KalmanFn.apply(bk, data[..., 0].contiguous(), present, *[full[k] for k in present])
    return [fs[..., None], ps[..., None], fc, pc, ll, llo]
