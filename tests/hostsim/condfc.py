"""TEST-ONLY: Python entry point of condfc.cpp, the conditional forecasts of csrc/kf_condfc.cuh compiled for the host.
condfc.cpp is linked into the one host library that ``tests.hostsim.build()`` makes from the .cpp files of this
directory; this module only adds the ctypes wrapper.  Not part of the product."""
from __future__ import annotations

import ctypes

import numpy as np

from tests.hostsim import _p, build, f8
from tests.hostsim.forecast import _batched


def conditional_forecast(mats, mean, cov, cond, spu=0, z_init=None, z_state=None, z_obs=None, n=0, n_draws=1,
                         n_series=1, force_dyn=False, want=("states", "obs")):
    """The conditional forecast (condfc.cpp) with the arguments and layouts of kfb_conditional_forecast for
    n_draws x n_series units: mats holds T Z R H Q c d, each shared or [n_draws, ...]; mean [U, m], cov [U, m, m];
    cond [H, p] shared or [U, H, p]; time-major normals if spu > 0.  Returns (moments dict of state_mean [U, H, m],
    state_cov, obs_mean, obs_cov; states [H, S, m] or None, obs [H, S, p] or None, info [U], used_static)."""
    lib = build()
    mats = dict(mats)
    m, p, r = f8(mats["T"]).shape[-1], f8(mats["Z"]).shape[-2], f8(mats["R"]).shape[-1]
    mean, cov, cond = map(f8, (mean, cov, cond))
    H = cond.shape[-2]
    U = n_draws * n_series
    S = U * spu
    base = {"T": (m, m), "Z": (p, m), "R": (m, r), "H": (p, p), "Q": (r, r), "c": (m,), "d": (p,)}
    mom = {"state_mean": np.zeros((U, H, m)), "state_cov": np.zeros((U, H, m, m)), "obs_mean": np.zeros((U, H, p)),
           "obs_cov": np.zeros((U, H, p, p))}
    states = np.zeros((H, S, m)) if spu and "states" in want else None
    obs = np.zeros((H, S, p)) if spu and "obs" in want else None
    z_init, z_state, z_obs = map(f8, (z_init, z_state, z_obs))
    info, used = np.full(U, -99, dtype=np.int32), np.zeros(1, dtype=np.int32)
    rc = lib.condfc_host_run(ctypes.c_longlong(n_draws), ctypes.c_longlong(n_series), ctypes.c_longlong(spu), int(n), H,
                             m, p, r, *_batched(mats, base, n_draws), _p(mean), _p(cov), _p(cond),
                             ctypes.c_longlong(H * p if cond.ndim == 3 else 0), _p(z_init),
                             _p(z_state) if H > 1 else None, _p(z_obs),
                             *[_p(mom[k]) for k in ("state_mean", "state_cov", "obs_mean", "obs_cov")], _p(states),
                             _p(obs), _p(info), int(force_dyn), _p(used))
    if rc != 0:
        raise RuntimeError(f"condfc_host_run rc={rc}")
    return mom, states, obs, info, bool(used[0])
