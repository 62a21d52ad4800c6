"""The exact filter over data with partly observed rows (kfb_masked_filter), restated literally in numpy.

Model as in oracle/simsmooth.py: y_t = Z x_t + d + eps_t, eps_t ~ N(0, H); x_{t+1} = T x_t + c + R eta_t,
eta_t ~ N(0, Q); static matrices.  At step t the observed set o of y_t is selected with index arrays (Z[o], H[o][:, o]),
not with the kernels' masked p x p form, so the two share only the algebra.
"""
from __future__ import annotations

import numpy as np

from .simsmooth import _col, dense_state_posterior


def masked_filter(y, a0, P0, T, Z, R, H, Q, c=None, d=None):
    """Predicted moments a_t = E[x_t | y_0..y_{t-1}], P_t = Cov(x_t | y_0..y_{t-1}) for t = 0..n, conditioned on the
    observed (non-NaN) entries only.  Returns (a [n+1, m], P [n+1, m, m], info): info 0, or t+1 if F_o is not positive
    definite at step t (a and P are then NaN)."""
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    T, Z, R, H, Q, P = (np.asarray(x, dtype=np.float64) for x in (T, Z, R, H, Q, P0))
    n, m, p = y.shape[0], T.shape[0], Z.shape[0]
    a, c, d = _col(a0, m), _col(c, m), _col(d, p)
    C = R @ Q @ R.T
    out_a, out_P = [a], [P]
    for t in range(n):
        o = np.flatnonzero(~np.isnan(y[t]))
        if o.size:
            Zo = Z[o]
            F = Zo @ P @ Zo.T + H[np.ix_(o, o)]
            try:
                np.linalg.cholesky(F)
            except np.linalg.LinAlgError:
                return np.full((n + 1, m), np.nan), np.full((n + 1, m, m), np.nan), t + 1
            K = T @ P @ Zo.T @ np.linalg.inv(F)
            a = T @ a + c + K @ (y[t, o] - Zo @ a - d[o])
            P = T @ P @ (T - K @ Zo).T + C
        else:
            a = T @ a + c
            P = T @ P @ T.T + C
        P = 0.5 * (P + P.T)
        out_a.append(a)
        out_P.append(P)
    return np.stack(out_a), np.stack(out_P), 0


def dense_predicted(y, a0, P0, T, Z, R, H, Q, c=None, d=None):
    """The same moments by dense joint-Gaussian algebra only (dense_state_posterior of y_0..y_{t-1} over t + 1 steps,
    its last block), sharing no recursion with any filter.  Returns (a [n+1, m], P [n+1, m, m])."""
    y = np.asarray(y, dtype=np.float64).reshape(len(y), -1)
    n, p = y.shape
    m = np.asarray(T).shape[0]
    a, P = [], []
    for t in range(n + 1):
        yt = np.concatenate([y[:t], np.full((1, p), np.nan)])
        mu, S = dense_state_posterior(yt, a0, P0, T, Z, R, H, Q, c, d)
        a.append(mu[-1])
        P.append(S[-m:, -m:])
    return np.stack(a), np.stack(P)
