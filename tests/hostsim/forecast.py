"""TEST-ONLY: Python entry points of forecast.cpp, the forecast paths and impulse responses of csrc/kf_forecast.cuh compiled
for the host.  forecast.cpp is linked into the one host library that ``tests.hostsim.build()`` makes from the .cpp files
of this directory; this module only adds the ctypes wrappers.  Not part of the product."""
from __future__ import annotations

import ctypes

import numpy as np

from tests.hostsim import _p, build, f8


def _batched(mats, base, n_draws):
    """ctypes arguments (pointer, batch stride) of each matrix in ``base``: shared (base shape) or [n_draws, ...]."""
    args = []
    for k, shape in base.items():
        v = f8(mats.get(k))
        if v is None:
            args += [None, ctypes.c_longlong(0)]
            continue
        size = int(np.prod(shape))
        args += [_p(v), ctypes.c_longlong(size if v.size == n_draws * size and n_draws > 1 else 0)]
        mats[k] = v  # keep alive
    return args


def forecast_paths(mats, mean, cov, spu, z_init, z_state, z_obs, n_draws=1, n_series=1, force_dyn=False,
                   want=("states", "obs")):
    """The forecast paths (forecast.cpp) with the arguments and layouts of kfb_forecast_paths for n_draws x n_series
    units: mats holds T Z R H Q c d, each shared or [n_draws, ...]; mean [U, m], cov [U, m, m]; time-major normals.
    Returns (states [H, S, m] or None, obs [H, S, p] or None, info [U], used_static)."""
    lib = build()
    mats = dict(mats)
    m, p, r = f8(mats["T"]).shape[-1], f8(mats["Z"]).shape[-2], f8(mats["R"]).shape[-1]
    z_init, z_state, z_obs, mean, cov = map(f8, (z_init, z_state, z_obs, mean, cov))
    H = z_obs.shape[0]
    U = n_draws * n_series
    base = {"T": (m, m), "Z": (p, m), "R": (m, r), "H": (p, p), "Q": (r, r), "c": (m,), "d": (p,)}
    states = np.zeros((H, U * spu, m)) if "states" in want else None
    obs = np.zeros((H, U * spu, p)) if "obs" in want else None
    info, used = np.full(U, -99, dtype=np.int32), np.zeros(1, dtype=np.int32)
    rc = lib.forecast_host_run(ctypes.c_longlong(n_draws), ctypes.c_longlong(n_series), ctypes.c_longlong(spu), H, m, p,
                               r, *_batched(mats, base, n_draws), _p(mean), _p(cov), _p(z_init),
                               _p(z_state) if H > 1 else None, _p(z_obs), _p(states), _p(obs), _p(info), int(force_dyn),
                               _p(used))
    if rc != 0:
        raise RuntimeError(f"forecast_host_run rc={rc}")
    return states, obs, info, bool(used[0])


def impulse_response(mats, horizon, shock, n_draws=1, force_dyn=False):
    """The impulse responses (forecast.cpp) with the arguments of kfb_impulse_response: mats holds T Z R Q, each shared
    or [n_draws, ...].  Returns (states [n_draws, H, m, r], obs [n_draws, H, p, r], info [n_draws], used_static)."""
    lib = build()
    mats = dict(mats)
    m, p, r = f8(mats["T"]).shape[-1], f8(mats["Z"]).shape[-2], f8(mats["R"]).shape[-1]
    base = {"T": (m, m), "Z": (p, m), "R": (m, r), "Q": (r, r)}
    states, obs = np.zeros((n_draws, horizon, m, r)), np.zeros((n_draws, horizon, p, r))
    info, used = np.full(n_draws, -99, dtype=np.int32), np.zeros(1, dtype=np.int32)
    rc = lib.forecast_host_irf(ctypes.c_longlong(n_draws), int(horizon), m, p, r, int(shock),
                               *_batched(mats, base, n_draws), _p(states), _p(obs), _p(info), int(force_dyn), _p(used))
    if rc != 0:
        raise RuntimeError(f"forecast_host_irf rc={rc}")
    return states, obs, info, bool(used[0])
