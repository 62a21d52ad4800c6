"""TEST-ONLY: Python entry points for data with partly observed rows: the masked filter of csrc/ compiled for the host
(partial.cpp) and the host simulation smoother of draws.cpp with desc.flags set (KFB_FLAG_PARTIAL_ROWS).  Requests are
built by ``tests.hostsim.draws``.  Not part of the product."""
from __future__ import annotations

import ctypes

import numpy as np

from tests.hostsim import _p, build, f8
from tests.hostsim.draws import _request


def masked_filter(y, mats, n_draws=1, n_series=1, force_dyn=False, want=("states", "covs")):
    """The masked filter with the arguments and layouts of kfb_masked_filter for n_draws x n_series units: y [n, p] or
    [n_series, n, p]; mats: dict of a0 P0 T Z R H Q c d, each shared or [n_draws, ...].  Returns (predicted_states
    [U, n+1, m] or None, predicted_covs [U, n+1, m, m] or None, info [U], used_static)."""
    y = f8(y)
    n = y.shape[-2]
    desc, ins, keep = _request(mats, n_draws, n_series, n, y)
    U, m = n_draws * n_series, desc.m
    ps = np.zeros((U, n + 1, m)) if "states" in want else None
    pc = np.zeros((U, n + 1, m, m)) if "covs" in want else None
    info, used = np.full(U, -99, dtype=np.int32), np.zeros(1, dtype=np.int32)
    rc = build().partial_host_masked_filter(ctypes.byref(desc), ctypes.byref(ins), _p(ps), _p(pc), _p(info),
                                            int(force_dyn), _p(used))
    if rc != 0:
        raise RuntimeError(f"partial_host_masked_filter rc={rc}")
    return ps, pc, info, bool(used[0])


def simsmooth(y, mats, pc, spu, z_init, z_state, z_obs, n_draws=1, n_series=1, force_dyn=False, flags=0):
    """``tests.hostsim.draws.simsmooth`` with ``flags`` in desc.flags (e.g. KFB_FLAG_PARTIAL_ROWS).
    Returns (states [S, n, m], info [U])."""
    y = f8(y)
    n = y.shape[-2]
    desc, ins, keep = _request(mats, n_draws, n_series, n, y)
    desc.flags = flags
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
