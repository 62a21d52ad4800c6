"""Simulation smoother restated in numpy (Durbin & Koopman, "A simple and efficient simulation smoother for state space
time series analysis", Biometrika 89(3), 2002; the fast state smoother of Durbin & Koopman's book, section 4.6.2), and
the dense joint posterior of the states it samples from.

Model (the one the filters evaluate): x_0 ~ N(a0, P0); y_t = Z x_t + d + eps_t, eps_t ~ N(0, H), t = 0..n-1;
x_{t+1} = T x_t + c + R eta_t, eta_t ~ N(0, Q), t = 0..n-2.  Static matrices; a row of y is either fully observed or
fully missing (NaN).  Column vectors a0, c, d may be given as [k] or [k, 1].
"""
from __future__ import annotations

import numpy as np

PSD_RTOL = 1e-10


def psd_factor(A):
    """Lower L with L L^T = A for a positive SEMI-definite A.  A pivot at or below PSD_RTOL times the largest diagonal
    entry is taken as zero and its column is zeroed; a pivot below -PSD_RTOL times it (or NaN) is an error.
    Returns (L, ok)."""
    A = np.asarray(A, dtype=np.float64)
    n = A.shape[0]
    L = np.zeros((n, n))
    dmax = max(0.0, float(np.max(np.diag(A)))) if not np.isnan(np.diag(A)).any() else np.nan
    tol = PSD_RTOL * dmax
    ok = True
    for j in range(n):
        dj = A[j, j] - L[j, :j] @ L[j, :j]
        if dj > tol:
            L[j, j] = np.sqrt(dj)
            L[j + 1:, j] = (A[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
        else:
            ok = ok and bool(dj >= -tol)
    return L, ok


def _col(v, k):
    return np.zeros(k) if v is None else np.asarray(v, dtype=np.float64).reshape(k)


def predicted_covs(y, P0, T, Z, R, H, Q):
    """P_t = Cov(x_t | y_0..y_{t-1}) for t = 0..n (the standard filter's predicted covariances)."""
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    C = R @ Q @ R.T
    P = [np.asarray(P0, dtype=np.float64)]
    for t in range(y.shape[0]):
        Pt = P[-1]
        if np.isnan(y[t]).all():
            P.append(T @ Pt @ T.T + C)
            continue
        F = Z @ Pt @ Z.T + H
        K = T @ Pt @ Z.T @ np.linalg.inv(F)
        P.append(T @ Pt @ (T - K @ Z).T + C)
    return np.stack(P)


def simulation_smoother(y, a0, P0, T, Z, R, H, Q, c=None, d=None, z_init=None, z_state=None, z_obs=None, P=None):
    """The five steps, literally, for S simulations of one unit fed the normals z_init[S, m], z_state[n-1, S, r],
    z_obs[n, S, p] (time-major, as the kernels take them).  ``P``: predicted covariances [n+1, m, m] (default: computed
    here).  Returns (states[S, n, m], info) with info 0, t+1 (F_t not PD), -(t+1) (row t partly missing) or "not_psd"."""
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    T, Z, R, H, Q, P0 = (np.asarray(x, dtype=np.float64) for x in (T, Z, R, H, Q, P0))
    n, p = y.shape
    m, r = T.shape[0], R.shape[1]
    a0, c, d = _col(a0, m), _col(c, m), _col(d, p)
    S = z_init.shape[0]
    SP0, ok0 = psd_factor(P0)
    SQ, okq = psd_factor(Q)
    SH, okh = psd_factor(H)
    if not (ok0 and okq and okh):
        return np.full((S, n, m), np.nan), "not_psd"
    P = predicted_covs(y, P0, T, Z, R, H, Q) if P is None else P
    C = R @ Q @ R.T
    Ks, Finvs, miss = [], [], []
    for t in range(n):
        nm = int(np.isnan(y[t]).sum())
        if 0 < nm < p:
            return np.full((S, n, m), np.nan), -(t + 1)
        miss.append(nm == p)
        if nm == p:
            Ks.append(np.zeros((m, p)))
            Finvs.append(np.zeros((p, p)))
            continue
        F = Z @ P[t] @ Z.T + H
        if not np.all(np.linalg.eigvalsh(F) > 0):
            return np.full((S, n, m), np.nan), t + 1
        Fi = np.linalg.inv(F)
        Ks.append(T @ P[t] @ Z.T @ Fi)
        Finvs.append(Fi)
    out = np.empty((S, n, m))
    for s in range(S):
        # 1. unconditional draw
        xp = np.empty((n, m))
        yp = np.empty((n, p))
        xp[0] = a0 + SP0 @ z_init[s]
        for t in range(n):
            yp[t] = Z @ xp[t] + d + SH @ z_obs[t, s]
            if t + 1 < n:
                xp[t + 1] = T @ xp[t] + c + R @ (SQ @ z_state[t, s])
        ys = y - yp
        # 2. zero-mean predictor recursion on y*
        a = np.zeros(m)
        v = np.zeros((n, p))
        for t in range(n):
            if not miss[t]:
                v[t] = ys[t] - Z @ a
            a = T @ a + Ks[t] @ v[t]
        # 3. backward pass
        rr = np.zeros(m)
        rs = np.zeros((n, m))  # rs[t] = r_{t-1}
        for t in range(n - 1, -1, -1):
            Lt = T - Ks[t] @ Z
            rr = Z.T @ Finvs[t] @ v[t] + Lt.T @ rr
            rs[t] = rr
        # 4. forward pass: xhat_0 = P0 r_{-1}, xhat_{t+1} = T xhat_t + C r_t
        xh = P0 @ rs[0]
        for t in range(n):
            out[s, t] = xp[t] + xh
            if t + 1 < n:
                xh = T @ xh + C @ rs[t + 1]
    return out, 0


def dense_state_posterior(y, a0, P0, T, Z, R, H, Q, c=None, d=None):
    """E[x_0..x_{n-1} | y] as [n, m] and Cov as [n m, n m] (row index t m + i), by dense joint-Gaussian algebra only:
    the prior moments of (x, y) from powers of T, then one conditioning on every observed entry of y.  Shares no
    recursion with any filter or smoother.  Small cases only."""
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    T, Z, R, H, Q, P0 = (np.asarray(x, dtype=np.float64) for x in (T, Z, R, H, Q, P0))
    n, p = y.shape
    m = T.shape[0]
    a0, c, d = _col(a0, m), _col(c, m), _col(d, p)
    C = R @ Q @ R.T
    mu, V = [a0], [P0]
    for _ in range(n - 1):
        mu.append(T @ mu[-1] + c)
        V.append(T @ V[-1] @ T.T + C)
    Tp = [np.eye(m)]
    for _ in range(n):
        Tp.append(T @ Tp[-1])
    Sxx = np.empty((n * m, n * m))
    for t in range(n):
        for s in range(n):  # Cov(x_t, x_s)
            Sxx[t * m:(t + 1) * m, s * m:(s + 1) * m] = Tp[t - s] @ V[s] if t >= s else (Tp[s - t] @ V[t]).T
    mux = np.concatenate(mu)
    obs = [(t, i) for t in range(n) for i in range(p) if not np.isnan(y[t, i])]
    if not obs:
        return mux.reshape(n, m), Sxx
    G = np.zeros((len(obs), n * m))  # y_obs = G x + d + noise
    for k, (t, i) in enumerate(obs):
        G[k, t * m:(t + 1) * m] = Z[i]
    Hn = np.array([[H[i, j] if t == s else 0.0 for (s, j) in obs] for (t, i) in obs])
    Syy = G @ Sxx @ G.T + Hn
    Sxy = Sxx @ G.T
    resid = np.array([y[t, i] - Z[i] @ mu[t] - d[i] for (t, i) in obs])
    W = np.linalg.solve(Syy, Sxy.T).T
    return (mux + W @ resid).reshape(n, m), Sxx - W @ Sxy.T
