"""Conditional forecasts from the end of the sample restated in numpy, and the dense joint law they sample from.

Model (the filters', as in oracle/forecast.py): y_t = Z x_t + d + eps_t, eps_t ~ N(0, H); x_{t+1} = T x_t + c + R eta_t,
eta_t ~ N(0, Q); static matrices.  The data are y_0..y_{n-1}; window index h is time n + h.  cond [H, p] holds the known
values of y_{n+h} (NaN = free).  Everything is conditioned on y and on every non-NaN entry of cond.  Column vectors
a0, c, d may be given as [k] or [k, 1].
"""
from __future__ import annotations

import numpy as np

from .simsmooth import _col, dense_state_posterior, psd_factor


def _ginv_psd(A):
    """W^T W with W the inverse of psd_factor(A) on its non-zero pivots and 0 elsewhere: a generalised inverse of A."""
    L, _ = psd_factor(A)
    J = np.flatnonzero(np.diag(L) != 0.0)
    W = np.zeros_like(L)
    if J.size:
        W[np.ix_(J, J)] = np.linalg.inv(L[np.ix_(J, J)])
    return W.T @ W


def window(start_mean, start_cov, T, Z, R, H, Q, c, d, cond, n=0):
    """Step 1, literally: the masked filter over the window, the fast state smoother backwards and the observation
    moments.  Returns (moments dict of state_mean [H, m], state_cov [H, m, m], obs_mean [H, p], obs_cov [H, p, p],
    tape list of (K, Fi, G) per step, info) with info 0, n + h + 1 (F_o not positive definite at step h) or "not_psd"."""
    T, Z, R, H, Q = (np.asarray(x, dtype=np.float64) for x in (T, Z, R, H, Q))
    cond = np.asarray(cond, dtype=np.float64)
    m, p = T.shape[0], Z.shape[0]
    hor = cond.shape[0]
    c, d = _col(c, m), _col(d, p)
    a, P = _col(start_mean, m), np.asarray(start_cov, dtype=np.float64)
    nan = {"state_mean": np.full((hor, m), np.nan), "state_cov": np.full((hor, m, m), np.nan),
           "obs_mean": np.full((hor, p), np.nan), "obs_cov": np.full((hor, p, p), np.nan)}
    if not (psd_factor(P)[1] and psd_factor(Q)[1] and psd_factor(H)[1]) or np.isnan(a).any():
        return nan, None, "not_psd"
    C = R @ Q @ R.T
    steps = []
    for h in range(hor):
        o = ~np.isnan(cond[h])
        Fi = np.zeros((p, p))
        K = np.zeros((m, p))
        u = np.zeros(p)
        v = np.zeros(p)
        if o.any():
            F = (Z @ P @ Z.T + H)[np.ix_(o, o)]
            if not np.all(np.linalg.eigvalsh(F) > 0):
                return nan, None, n + h + 1
            Fi[np.ix_(o, o)] = np.linalg.inv(F)
            K = T @ P @ Z.T @ Fi
            v[o] = (cond[h] - Z @ a - d)[o]
            u = Fi @ v
        G = np.zeros((p, p))
        if o.any() and (~o).any():
            Hoo = np.where(np.outer(o, o), H, 0.0)
            G[np.ix_(~o, o)] = (H @ _ginv_psd(Hoo))[np.ix_(~o, o)]
        steps.append((a, P, K, Fi, G, u, o))
        L = T - K @ Z
        a = T @ a + c + K @ v
        P = T @ P @ L.T + C
        P = 0.5 * (P + P.T)
    out = {k: np.empty_like(v) for k, v in nan.items()}
    r, N = np.zeros(m), np.zeros((m, m))
    for h in range(hor - 1, -1, -1):
        a, P, K, Fi, G, u, o = steps[h]
        L = T - K @ Z
        r = Z.T @ (u - K.T @ r) + T.T @ r
        N = Z.T @ Fi @ Z + L.T @ N @ L
        xm, V = a + P @ r, P - P @ N @ P
        out["state_mean"][h], out["state_cov"][h] = xm, 0.5 * (V + V.T)
        D = np.where(o[:, None], 0.0, Z - G @ Z)
        ym = Z @ xm + d
        ym = np.where(o, cond[h], ym + G @ np.where(o, cond[h] - ym, 0.0))
        Oc = D @ V @ D.T + H - G @ H
        Oc[o, :] = 0.0
        Oc[:, o] = 0.0
        out["obs_mean"][h], out["obs_cov"][h] = ym, 0.5 * (Oc + Oc.T)
    return out, [(K, Fi, G) for (_, _, K, Fi, G, _, _) in steps], 0


def conditional_paths(start_mean, start_cov, T, Z, R, H, Q, c, d, cond, z_init, z_state, z_obs, n=0):
    """Step 2, literally: the mean correction over the window for S simulations fed the normals z_init [S, m],
    z_state [H-1, S, r], z_obs [H, S, p] (time-major, as the kernel takes them).  Returns (states [S, H, m],
    obs [S, H, p], info) with info as in ``window`` (NaN paths on failure)."""
    T, Z, R, H, Q = (np.asarray(x, dtype=np.float64) for x in (T, Z, R, H, Q))
    cond = np.asarray(cond, dtype=np.float64)
    m, p = T.shape[0], Z.shape[0]
    hor, S = cond.shape[0], z_init.shape[0]
    _, tape, info = window(start_mean, start_cov, T, Z, R, H, Q, c, d, cond, n)
    if info != 0:
        return np.full((S, hor, m), np.nan), np.full((S, hor, p), np.nan), info
    a0, c, d = _col(start_mean, m), _col(c, m), _col(d, p)
    P0 = np.asarray(start_cov, dtype=np.float64)
    SP, SQ, SH = psd_factor(P0)[0], psd_factor(Q)[0], psd_factor(H)[0]
    C = R @ Q @ R.T
    o = ~np.isnan(cond)
    states, obs = np.empty((S, hor, m)), np.empty((S, hor, p))
    for s in range(S):
        xp, eps = np.empty((hor, m)), np.empty((hor, p))
        xp[0] = a0 + SP @ z_init[s]
        for h in range(hor):
            eps[h] = SH @ z_obs[h, s]
            if h + 1 < hor:
                xp[h + 1] = T @ xp[h] + c + R @ (SQ @ z_state[h, s])
        ys = np.where(o, cond - (xp @ Z.T + d + eps), 0.0)
        a = np.zeros(m)
        us = []
        for h in range(hor):
            K, Fi, _ = tape[h]
            v = np.where(o[h], ys[h] - Z @ a, 0.0)
            us.append(Fi @ v)
            a = T @ a + K @ v
        r = np.zeros(m)
        rs = np.zeros((hor, m))  # rs[h] = r_{h-1}
        for h in range(hor - 1, -1, -1):
            K = tape[h][0]
            r = Z.T @ (us[h] - K.T @ r) + T.T @ r
            rs[h] = r
        xh = P0 @ rs[0]
        for h in range(hor):
            xt = xp[h] + xh
            states[s, h] = xt
            G = tape[h][2]
            yt = Z @ xt + d + eps[h]
            obs[s, h] = np.where(o[h], cond[h], yt + G @ np.where(o[h], cond[h] - yt, 0.0))
            if h + 1 < hor:
                xh = T @ xh + C @ rs[h + 1]
    return states, obs, 0


def dense_conditional_forecast_law(y, a0, P0, T, Z, R, H, Q, c=None, d=None, cond=None):
    """The joint law of (x_n..x_{n+H-1}, y_n..y_{n+H-1}) given y and the non-NaN entries of cond [H, p], by dense
    joint-Gaussian algebra only: dense_state_posterior's prior of the states over n + H steps and the observations of
    every (time, entry), then one conditioning on every observed entry of y and cond.  Shares no recursion with any
    filter.  Returns (mean [H m + H p], cov [H m + H p, H m + H p]) of the vector (x window, y window), each h-major
    (conditioned entries: mean cond, variance 0 to rounding)."""
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    cond = np.asarray(cond, dtype=np.float64)
    T, Z, H = (np.asarray(x, dtype=np.float64) for x in (T, Z, H))
    n, p = y.shape
    m, hor = T.shape[0], cond.shape[0]
    N = n + hor
    # prior of x_0..x_{N-1}: dense_state_posterior with nothing observed
    mux, Sxx = dense_state_posterior(np.full((N, p), np.nan), a0, P0, T, Z, R, H, Q, c, d)
    mux = mux.reshape(-1)
    G = np.kron(np.eye(N), Z)
    muy = G @ mux + np.tile(_col(d, p), N)
    Syy = G @ Sxx @ G.T + np.kron(np.eye(N), H)
    mu = np.concatenate([mux, muy])
    S = np.block([[Sxx, Sxx @ G.T], [G @ Sxx, Syy]])
    yall = np.concatenate([y, cond]).reshape(-1)
    obs = N * m + np.flatnonzero(~np.isnan(yall))
    keep = np.concatenate([np.arange(n * m, N * m), N * m + n * p + np.arange(hor * p)])
    if obs.size:
        Soo = S[np.ix_(obs, obs)]
        Sko = S[np.ix_(keep, obs)]
        W = np.linalg.solve(Soo, Sko.T).T
        mean = mu[keep] + W @ (yall[obs - N * m] - mu[obs])
        cov = S[np.ix_(keep, keep)] - W @ Sko.T
    else:
        mean, cov = mu[keep], S[np.ix_(keep, keep)]
    return mean, 0.5 * (cov + cov.T)
