"""Forecasts from the end of the sample and impulse responses, restated in numpy, and the dense joint law of the future
they sample from.

Model (the filters', as in oracle/simsmooth.py): y_t = Z x_t + d + eps_t, eps_t ~ N(0, H); x_{t+1} = T x_t + c + R eta_t,
eta_t ~ N(0, Q); static matrices.  The data are y_0..y_{n-1}; a forecast of horizon H covers times n..n+H-1 (index h is
time n + h).  Column vectors a0, c, d may be given as [k] or [k, 1].
"""
from __future__ import annotations

import numpy as np

from . import kalman_numpy as kn
from .simsmooth import _col, dense_state_posterior, psd_factor


def _extended(y, horizon):
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    return np.concatenate([y, np.full((horizon, y.shape[1]), np.nan)])


def forecast_paths(start_mean, start_cov, T, Z, R, H, Q, c, d, z_init, z_state, z_obs):
    """The loop of kfb_forecast_paths, literally, for S simulations started at N(start_mean, start_cov) and fed the
    normals z_init [S, m], z_state [H-1, S, r], z_obs [H, S, p] (time-major, as the kernel takes them).
    Returns (states [S, H, m], obs [S, H, p], info) with info 0 or "not_psd" (NaN paths)."""
    T, Z, R, H, Q = (np.asarray(x, dtype=np.float64) for x in (T, Z, R, H, Q))
    m, p = T.shape[0], Z.shape[0]
    a, c, d = _col(start_mean, m), _col(c, m), _col(d, p)
    S, hor = z_init.shape[0], z_obs.shape[0]
    SP, okp = psd_factor(start_cov)
    SQ, okq = psd_factor(Q)
    SH, okh = psd_factor(H)
    if not (okp and okq and okh) or np.isnan(a).any():
        return np.full((S, hor, m), np.nan), np.full((S, hor, p), np.nan), "not_psd"
    states, obs = np.empty((S, hor, m)), np.empty((S, hor, p))
    for s in range(S):
        x = a + SP @ z_init[s]
        for h in range(hor):
            states[s, h] = x
            obs[s, h] = Z @ x + d + SH @ z_obs[h, s]
            if h < hor - 1:
                x = T @ x + c + (R @ SQ) @ z_state[h, s]
    return states, obs, 0


def forecast_moments(y, a0, P0, T, Z, R, H, Q, c=None, d=None, horizon=1):
    """The corrected standard filter (oracle.kalman_numpy) on y plus ``horizon`` NaN rows: its predicted moments
    n..n+H-1 and the observation moments Z a + d, Z P Z^T + H.  Returns a dict of state_mean [H, m], state_cov
    [H, m, m], obs_mean [H, p], obs_cov [H, p, p]; the start of the paths is (state_mean[0], state_cov[0])."""
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    n = y.shape[0]
    T, Z, R, H, Q, P0 = (np.asarray(x, dtype=np.float64) for x in (T, Z, R, H, Q, P0))
    m, p = T.shape[0], Z.shape[0]
    cc = None if c is None else _col(c, m)[:, None]
    dd = None if d is None else _col(d, p)[:, None]
    _, ps, _, pc, _, _ = kn.kalman_filter("standard", _extended(y, horizon)[..., None], _col(a0, m)[:, None], P0, T, Z,
                                          R, H, Q, cc, dd, strict_reference=False)
    a, P = ps[n:n + horizon, :, 0], pc[n:n + horizon]
    return {"state_mean": a, "state_cov": P, "obs_mean": a @ Z.T + _col(d, p),
            "obs_cov": np.einsum("ij,hjk,lk->hil", Z, P, Z) + H}


def dense_forecast_law(y, a0, P0, T, Z, R, H, Q, c=None, d=None, horizon=1):
    """The joint law of x_n..x_{n+H-1} and y_n..y_{n+H-1} given y, by dense joint-Gaussian algebra only
    (oracle.simsmooth.dense_state_posterior on y plus H NaN rows, last H state blocks); shares no recursion with any
    filter.  Returns (state_mean [H, m], state_cov [H m, H m], obs_mean [H, p], obs_cov [H p, H p]); cross-horizon
    blocks included, row index h m + i.  The observations are G x + d + noise with G = I (x) Z, so their covariance is
    G Sxx G^T + I (x) H."""
    T, Z, H = (np.asarray(x, dtype=np.float64) for x in (T, Z, H))
    m, p = T.shape[0], Z.shape[0]
    mu, Sxx = dense_state_posterior(_extended(y, horizon), a0, P0, T, Z, R, H, Q, c, d)
    mu, Sxx = mu[-horizon:], Sxx[-horizon * m:, -horizon * m:]
    G = np.kron(np.eye(horizon), Z)
    return mu, Sxx, mu @ Z.T + _col(d, p), G @ Sxx @ G.T + np.kron(np.eye(horizon), H)


def impulse_responses(T, Z, R, Q, horizon, shock="cholesky"):
    """Column j of horizon h: T^h R S e_j (states [H, m, r]) and Z T^h R S e_j (obs [H, p, r]), from literal powers of
    T; S = I ("unit"), diag(sqrt(diag Q)) ("std") or psd_factor(Q) ("cholesky")."""
    T, Z, R, Q = (np.asarray(x, dtype=np.float64) for x in (T, Z, R, Q))
    S = {"unit": lambda: np.eye(Q.shape[0]), "std": lambda: np.diag(np.sqrt(np.diag(Q))),
         "cholesky": lambda: psd_factor(Q)[0]}[shock]()
    states = np.stack([np.linalg.matrix_power(T, h) @ R @ S for h in range(horizon)])
    return states, np.einsum("ij,hjk->hik", Z, states)
