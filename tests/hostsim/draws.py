"""TEST-ONLY: Python entry points of draws.cpp, the per-draw sampling calls of csrc/ compiled for the host: the
simulation smoother, forecast paths, impulse responses and conditional forecasts.  Each takes its C ABI call's
arguments as a ``KfbDesc`` / ``KfbInputs`` pair built here.  draws.cpp is linked into the one host library that
``tests.hostsim.build()`` makes from the .cpp files of this directory.  Not part of the product."""
from __future__ import annotations

import ctypes

import numpy as np

from pymc_statespace_b200._lib import KfbDesc, KfbInputs
from tests.hostsim import _p, build, f8


def _request(mats, n_draws, n_series=1, n=0, y=None):
    """(KfbDesc, KfbInputs, arrays to keep alive) of a static-matrix request: ``mats`` holds any of a0 P0 T Z R H Q c d,
    each shared (base shape) or [n_draws, ...]; y [n, p] shared by the series or [n_series, n, p]."""
    m, p, r = f8(mats["T"]).shape[-1], f8(mats["Z"]).shape[-2], f8(mats["R"]).shape[-1]
    base = {"a0": m, "P0": m * m, "T": m * m, "Z": p * m, "R": m * r, "H": p * p, "Q": r * r, "c": m, "d": p}
    desc, ins, keep = KfbDesc(n_draws=n_draws, n_series=n_series, n=n, m=m, p=p, r=r), KfbInputs(), []
    for k, v in dict(mats, y=y).items():
        v = f8(v)
        if v is None:
            continue
        if k == "y":
            bs = n * p if v.ndim == 3 else 0
        else:
            bs = base[k] if v.size == n_draws * base[k] and n_draws > 1 else 0
        setattr(desc, k + "_bs", bs)
        setattr(ins, k, _p(v))
        keep.append(v)
    return desc, ins, keep


def simsmooth(y, mats, pc, spu, z_init, z_state, z_obs, n_draws=1, n_series=1, force_dyn=False):
    """The simulation smoother with the arguments and layouts of kfb_simulation_smoother for n_draws x n_series units.
    y [n, p] or [n_series, n, p]; mats: dict of a0 P0 T Z R H Q c d, each shared (base shape) or [n_draws, ...];
    pc [U, n+1, m, m].  Returns (states [S, n, m], info [U])."""
    y = f8(y)
    n = y.shape[-2]
    desc, ins, keep = _request(mats, n_draws, n_series, n, y)
    U = n_draws * n_series
    states = np.zeros((U * spu, n, desc.m))
    info = np.zeros(U, dtype=np.int32)
    pc, z_init, z_state, z_obs = f8(pc), f8(z_init), f8(z_state), f8(z_obs)
    rc = build().draws_host_simulation_smoother(ctypes.byref(desc), ctypes.byref(ins), _p(pc), ctypes.c_longlong(spu),
                                                _p(z_init), _p(z_state), _p(z_obs), _p(states), _p(info),
                                                int(force_dyn), None)
    if rc != 0:
        raise RuntimeError(f"draws_host_simulation_smoother rc={rc}")
    return states, info


def forecast_paths(mats, mean, cov, spu, z_init, z_state, z_obs, n_draws=1, n_series=1, force_dyn=False,
                   want=("states", "obs")):
    """The forecast paths with the arguments and layouts of kfb_forecast_paths for n_draws x n_series units: mats holds
    T Z R H Q c d, each shared or [n_draws, ...]; mean [U, m], cov [U, m, m]; time-major normals.
    Returns (states [H, S, m] or None, obs [H, S, p] or None, info [U], used_static)."""
    desc, ins, keep = _request(mats, n_draws, n_series)
    z_init, z_state, z_obs, mean, cov = map(f8, (z_init, z_state, z_obs, mean, cov))
    H = z_obs.shape[0]
    S = n_draws * n_series * spu
    states = np.zeros((H, S, desc.m)) if "states" in want else None
    obs = np.zeros((H, S, desc.p)) if "obs" in want else None
    info, used = np.full(n_draws * n_series, -99, dtype=np.int32), np.zeros(1, dtype=np.int32)
    rc = build().draws_host_forecast_paths(ctypes.byref(desc), ctypes.byref(ins), _p(mean), _p(cov), H,
                                           ctypes.c_longlong(spu), _p(z_init), _p(z_state) if H > 1 else None,
                                           _p(z_obs), _p(states), _p(obs), _p(info), int(force_dyn), _p(used))
    if rc != 0:
        raise RuntimeError(f"draws_host_forecast_paths rc={rc}")
    return states, obs, info, bool(used[0])


def impulse_response(mats, horizon, shock, n_draws=1, force_dyn=False):
    """The impulse responses with the arguments of kfb_impulse_response: mats holds T Z R Q, each shared or
    [n_draws, ...].  Returns (states [n_draws, H, m, r], obs [n_draws, H, p, r], info [n_draws], used_static)."""
    desc, ins, keep = _request(mats, n_draws)
    states, obs = np.zeros((n_draws, horizon, desc.m, desc.r)), np.zeros((n_draws, horizon, desc.p, desc.r))
    info, used = np.full(n_draws, -99, dtype=np.int32), np.zeros(1, dtype=np.int32)
    rc = build().draws_host_impulse_response(ctypes.byref(desc), ctypes.byref(ins), int(horizon), int(shock),
                                             _p(states), _p(obs), _p(info), int(force_dyn), _p(used))
    if rc != 0:
        raise RuntimeError(f"draws_host_impulse_response rc={rc}")
    return states, obs, info, bool(used[0])


def conditional_forecast(mats, mean, cov, cond, spu=0, z_init=None, z_state=None, z_obs=None, n=0, n_draws=1,
                         n_series=1, force_dyn=False, want=("states", "obs")):
    """The conditional forecast with the arguments and layouts of kfb_conditional_forecast for n_draws x n_series
    units: mats holds T Z R H Q c d, each shared or [n_draws, ...]; mean [U, m], cov [U, m, m]; cond [H, p] shared or
    [U, H, p]; time-major normals if spu > 0.  Returns (moments dict of state_mean [U, H, m], state_cov, obs_mean,
    obs_cov; states [H, S, m] or None, obs [H, S, p] or None, info [U], used_static)."""
    desc, ins, keep = _request(mats, n_draws, n_series, int(n))
    m, p = desc.m, desc.p
    mean, cov, cond = map(f8, (mean, cov, cond))
    H = cond.shape[-2]
    U = n_draws * n_series
    S = U * spu
    mom = {"state_mean": np.zeros((U, H, m)), "state_cov": np.zeros((U, H, m, m)), "obs_mean": np.zeros((U, H, p)),
           "obs_cov": np.zeros((U, H, p, p))}
    states = np.zeros((H, S, m)) if spu and "states" in want else None
    obs = np.zeros((H, S, p)) if spu and "obs" in want else None
    z_init, z_state, z_obs = map(f8, (z_init, z_state, z_obs))
    info, used = np.full(U, -99, dtype=np.int32), np.zeros(1, dtype=np.int32)
    rc = build().draws_host_conditional_forecast(
        ctypes.byref(desc), ctypes.byref(ins), _p(mean), _p(cov), H, _p(cond),
        ctypes.c_longlong(H * p if cond.ndim == 3 else 0), ctypes.c_longlong(spu), _p(z_init),
        _p(z_state) if H > 1 else None, _p(z_obs),
        *[_p(mom[k]) for k in ("state_mean", "state_cov", "obs_mean", "obs_cov")], _p(states), _p(obs), _p(info),
        int(force_dyn), _p(used))
    if rc != 0:
        raise RuntimeError(f"draws_host_conditional_forecast rc={rc}")
    return mom, states, obs, info, bool(used[0])
