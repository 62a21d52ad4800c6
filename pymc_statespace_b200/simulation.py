"""Batched simulation helpers on the GPU (SURVEY.md section 8(f) row f4; not on the logp/grad path).

Mirrors reference ``pymc_statespace/utils/simulation.py`` (numba): ``simulate_statespace`` (:29-62),
``unconditional_simulations`` (:65-79) and ``conditional_simulation`` (:17-26).  ``simulation_smoother`` goes beyond the
reference: joint draws of the whole state path from p(x_0..x_{n-1} | y, theta) (Durbin & Koopman 2002), where
``conditional_simulation`` draws every time step on its own from the smoothed marginal.  The reference draws its normals from
NumPy's global RNG inside numba, so its trajectories are not reproducible from outside; here the standard-normal draws
come from ``torch.randn`` on the device (or are passed in, which makes the result exactly checkable) and the CUDA kernels
are deterministic transforms of them.
"""
from __future__ import annotations

from typing import Optional

import ctypes

import torch

from ._lib import check, load
from .engine import BatchedKalman, _ptr, _stream_ptr


def _bs(t, base_ndim, size):
    return size if t.ndim == base_ndim + 1 else 0


def simulate_statespace(T, Z, R, H, Q, n_steps: int, x0=None, n_simulations: int = 1, z_state=None, z_obs=None,
                        generator: Optional[torch.Generator] = None):
    """T:[B,m,m]|[m,m] ... float64 CUDA tensors.  Returns (states[B*S,n,m], obs[B*S,n,p]) for S = n_simulations
    trajectories per draw (``unconditional_simulations`` ordering: draw-major)."""
    lib = load()
    dev = T.device
    m, p, r = T.shape[-1], Z.shape[-2], R.shape[-1]
    B = max([t.shape[0] for t, nd in ((T, 2), (Z, 2), (R, 2), (H, 2), (Q, 2)) if t.ndim == nd + 1] + [1])
    S = B * n_simulations
    T, Z, R, H, Q = (t.contiguous() for t in (T, Z, R, H, Q))
    if z_state is None:
        z_state = torch.randn((S, n_steps, r), dtype=torch.float64, device=dev, generator=generator)
    if z_obs is None:
        z_obs = torch.randn((S, n_steps, p), dtype=torch.float64, device=dev, generator=generator)
    z_state, z_obs = z_state.contiguous(), z_obs.contiguous()
    if tuple(z_state.shape) != (S, n_steps, r) or tuple(z_obs.shape) != (S, n_steps, p):
        raise ValueError("z_state / z_obs must have shapes [B*S, n, k_posdef] / [B*S, n, k_endog]")
    x0c = None if x0 is None else x0.reshape(-1, m).contiguous()
    states = torch.empty((S, n_steps, m), dtype=torch.float64, device=dev)
    obs = torch.empty((S, n_steps, p), dtype=torch.float64, device=dev)
    info = torch.zeros(S, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_simulate(B, n_simulations, n_steps, m, p, r, _ptr(T), _bs(T, 2, m * m), _ptr(Z), _bs(Z, 2, p * m),
                               _ptr(R), _bs(R, 2, m * r), _ptr(H), _bs(H, 2, p * p), _ptr(Q), _bs(Q, 2, r * r), _ptr(x0c),
                               0 if x0c is None or x0c.shape[0] == 1 else m, _ptr(z_state), _ptr(z_obs), _ptr(states),
                               _ptr(obs), _ptr(info), _stream_ptr(dev)), "kfb_simulate")
    if int(info.sum()) != 0:
        raise RuntimeError("simulate_statespace: Q or H is not positive definite for some draw")
    return states, obs


def conditional_simulation(mus, covs, n_simulations: int = 100, z=None, jitter=None,
                           generator: Optional[torch.Generator] = None):
    """mus[U,n,k], covs[U,n,k,k] (filtered / predicted / smoothed moments) -> simulations[U*S,n,k]:
    each time block is an independent draw mu_t + chol(cov_t + jitter I) z (reference :8-26; the reference's jitter is
    uniform(1e-12, 1e-8) per trajectory)."""
    lib = load()
    dev = mus.device
    U, n, k = mus.shape
    S = U * n_simulations
    if z is None:
        z = torch.randn((S, n, k), dtype=torch.float64, device=dev, generator=generator)
    if jitter is None:
        jitter = 1e-12 + (1e-8 - 1e-12) * torch.rand(S, dtype=torch.float64, device=dev, generator=generator)
    mus, covs, z, jitter = mus.contiguous(), covs.contiguous(), z.contiguous(), jitter.contiguous()
    out = torch.empty((S, n, k), dtype=torch.float64, device=dev)
    info = torch.zeros(S, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_mvn_draws(U, n_simulations, n, k, _ptr(mus), _ptr(covs), _ptr(z), _ptr(jitter), _ptr(out), _ptr(info),
                                _stream_ptr(dev)), "kfb_mvn_draws")
    if int(info.sum()) != 0:
        raise RuntimeError("conditional_simulation: a covariance block is not positive definite")
    return out


_BASE_NDIM = {"a0": 1, "P0": 2, "T": 2, "Z": 2, "R": 2, "H": 2, "Q": 2, "c": 1, "d": 1}


def _simulation_smoother(kalman: BatchedKalman, y, mats, n_simulations, z_init, z_state, z_obs, generator):
    """kfb_forward (predicted covariances) then kfb_simulation_smoother on ``kalman``'s geometry.  Returns
    (states [U*S, n, m], info [U]) without raising on a non-zero info."""
    lib = load()
    dev = kalman.device
    n, m, p, r, U = kalman.n, kalman.m, kalman.p, kalman.r, kalman.units
    S = U * n_simulations
    pc = kalman.forward(y, *[mats.get(k) for k in ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")],
                        outputs=("predicted_covs",))["predicted_covs"]
    f64 = dict(dtype=torch.float64, device=dev)
    z_init = torch.randn((S, m), generator=generator, **f64) if z_init is None else z_init
    z_state = torch.randn((max(n - 1, 0), S, r), generator=generator, **f64) if z_state is None else z_state
    z_obs = torch.randn((n, S, p), generator=generator, **f64) if z_obs is None else z_obs
    for name, t, shape in (("z_init", z_init, (S, m)), ("z_state", z_state, (max(n - 1, 0), S, r)),
                           ("z_obs", z_obs, (n, S, p))):
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64 and tuple(t.shape) == shape):
            raise ValueError(f"{name}: expected a float64 CUDA tensor of shape {shape} (time-major normals)")
    z_init, z_state, z_obs = z_init.contiguous(), z_state.contiguous(), z_obs.contiguous()
    desc = kalman._desc
    nbytes = ctypes.c_size_t(0)
    check(lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(desc), n_simulations, ctypes.byref(nbytes)),
          "kfb_simulation_smoother_workspace_bytes")
    ws = torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=dev)
    states = torch.empty((S, n, m), **f64)
    info = torch.empty(U, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_simulation_smoother(ctypes.byref(desc), ctypes.byref(kalman._inputs), _ptr(pc), n_simulations,
                                          _ptr(z_init), _ptr(z_state) if n > 1 else None, _ptr(z_obs), _ptr(states),
                                          _ptr(info), _ptr(ws), ws.numel(), _stream_ptr(dev)), "kfb_simulation_smoother")
    return states, info


def simulation_smoother(y, a0, P0, T, Z, R, H, Q, c=None, d=None, n_simulations: int = 1, z_init=None, z_state=None,
                        z_obs=None, generator: Optional[torch.Generator] = None):
    """Joint draws of the state paths x_0..x_{n-1} from p(x | y, theta) (Durbin & Koopman 2002, mean correction;
    include/kfb200.h states the model and the recursion).

    Float64 CUDA tensors; each matrix is shared (a0 [m], P0 [m, m], T [m, m], Z [p, m], R [m, r], H [p, p], Q [r, r],
    c [m], d [p]) or one per draw with a leading [B] axis, as in ``BatchedKalman``.  y is [n, p] or [n_series, n, p]
    (NaN = missing; a row must be all observed or all missing).  Units are draw-major (u = draw * n_series + series) and
    so are the simulations (s = u * n_simulations + k).  Normals may be given, time-major: z_init [S, m], z_state
    [n-1, S, r], z_obs [n, S, p] for S = U * n_simulations; otherwise they are drawn with ``torch.randn``.
    Returns states [S, n, m].  Raises RuntimeError if some unit fails (F_t not positive definite, a partly missing row,
    P0 / Q / H not positive semi-definite) and NotImplementedError for time-varying matrices."""
    mats = {"a0": a0, "P0": P0, "T": T, "Z": Z, "R": R, "H": H, "Q": Q, "c": c, "d": d}
    for k, t in mats.items():
        if t is not None and k in ("a0", "c", "d") and t.ndim >= 2 and t.shape[-1] == 1:
            mats[k] = t = t[..., 0]
        if t is not None and t.ndim > _BASE_NDIM[k] + 1:
            raise NotImplementedError("simulation_smoother: time-varying matrices are not supported")
    if y.ndim == 3 and y.shape[-1] == 1 and y.shape[-2] == Z.shape[-2]:
        y = y[..., 0]  # reference layout [n, p, 1]
    n_series = 1 if y.ndim == 2 else y.shape[0]
    m, p, r = T.shape[-1], Z.shape[-2], R.shape[-1]
    B = max([t.shape[0] for k, t in mats.items() if t is not None and t.ndim == _BASE_NDIM[k] + 1] + [1])
    kalman = BatchedKalman("standard", y.shape[-2], m, p, r, n_draws=B, n_series=n_series, strict_reference=False,
                           device=T.device)
    states, info = _simulation_smoother(kalman, y, mats, int(n_simulations), z_init, z_state, z_obs, generator)
    bad = torch.nonzero(info != 0)
    if bad.numel():
        u = int(bad[0, 0])
        raise RuntimeError(f"simulation_smoother: unit {u} failed with info {int(info[u])} (codes in include/kfb200.h)")
    return states
