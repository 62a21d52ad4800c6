"""CPU checks of the simulation smoother: the numpy restatement (oracle/simsmooth.py) pins itself against dense
joint-Gaussian algebra through the affine map from normals to paths, the host build of the kernels' KFB_HD code
(tests/hostsim) equals the restatement, and the C ABI validates its arguments without a device."""
import ctypes

import numpy as np
import pytest
import scipy.linalg

from oracle import kalman_numpy as kn
from oracle import simsmooth as oss
from tests.helpers import nile_inputs, random_system

N_SMALL = 12


# ---------------------------------------------------------------------------------------------------- shared helpers
def unit_basis(n, m, p, r):
    """Normals for 1 + N simulations of one unit: the zero vector, then every unit vector e_k of the N = m + (n-1) r + n p
    normals a path consumes.  Returns (z_init [S, m], z_state [n-1, S, r], z_obs [n, S, p])."""
    N = m + (n - 1) * r + n * p
    E = np.concatenate([np.zeros((1, N)), np.eye(N)])
    S = N + 1
    z_init = E[:, :m].copy()
    z_state = E[:, m:m + (n - 1) * r].reshape(S, n - 1, r).transpose(1, 0, 2).copy()
    z_obs = E[:, m + (n - 1) * r:].reshape(S, n, p).transpose(1, 0, 2).copy()
    return z_init, z_state, z_obs


def random_normals(rng, S, n, m, p, r):
    return rng.normal(size=(S, m)), rng.normal(size=(max(n - 1, 0), S, r)), rng.normal(size=(n, S, p))


def check_joint(paths, mean, cov, rtol):
    """paths [1 + N, n, m] from unit_basis: path 0 is the mean; the differences span the covariance.  Tolerances are
    relative to the largest entry, or to 1 where that is smaller (a fully observed state has a posterior covariance of
    rounding size)."""
    x0 = paths[0].reshape(-1)
    M = paths[1:].reshape(paths.shape[0] - 1, -1) - x0
    scale_mu = np.abs(mean).max() + 1.0
    assert np.abs(x0 - mean.reshape(-1)).max() <= rtol * scale_mu
    scale = max(np.abs(cov).max(), 1.0)
    assert np.abs(M.T @ M - cov).max() <= rtol * scale
    return M.T @ M


def arma11(rho, theta, sigma2=0.7, n=N_SMALL, seed=3):
    T = np.array([[rho, 1.0], [0.0, 0.0]])
    R = np.array([[1.0], [theta]])
    Q = np.array([[sigma2]])
    P0 = scipy.linalg.solve_discrete_lyapunov(T, R @ Q @ R.T)
    P0 = 0.5 * (P0 + P0.T)
    y = np.random.default_rng(seed).normal(size=(n, 1, 1))
    return y, np.zeros((2, 1)), P0, T, np.array([[1.0, 0.0]]), R, np.zeros((1, 1)), Q


def cases():
    """(name, y, a0, P0, T, Z, R, H, Q, c, d, rtol)"""
    out = []
    rng = np.random.default_rng(7)
    for m in range(1, 5):
        for p in range(1, 4):
            r = 1 + (m + p) % m
            y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, r, N_SMALL)
            y[[0, 5, N_SMALL - 1]] = np.nan  # whole rows: first and last included
            c = rng.normal(size=(m, 1)) if (m + p) % 2 else None
            d = rng.normal(size=(p, 1)) if (m + p) % 2 else None
            out.append((f"random_m{m}_p{p}_r{r}", y, a0, P0, T, Z, R, H, Q, c, d, 1e-10))
    out.append(("arma11_H0",) + arma11(0.6, 0.3) + (None, None, 1e-10))
    out.append(("arma11_theta0_singular_P0",) + arma11(0.6, 0.0) + (None, None, 1e-10))
    out.append(("arma11_theta_minus_rho",) + arma11(0.5, -0.5) + (None, None, 1e-10))
    for n in (1, 2):
        y, a0, P0, T, Z, R, H, Q = random_system(rng, 2, 1, 2, n)
        out.append((f"n{n}", y, a0, P0, T, Z, R, H, Q, None, None, 1e-10))
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 3, 2, 2, 4)
    y[:] = np.nan
    out.append(("all_missing", y, a0, P0, T, Z, R, H, Q, None, None, 1e-10))
    return out


CASES = cases()
IDS = [c[0] for c in CASES]


def mats_of(case):
    _, y, a0, P0, T, Z, R, H, Q, c, d, _ = case
    return dict(a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q, c=c, d=d)


# ---------------------------------------------------------------------------------------------------- oracle pins itself
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_oracle_joint_law_matches_dense_posterior(case):
    name, y, a0, P0, T, Z, R, H, Q, c, d, rtol = case
    n, p, m, r = y.shape[0], Z.shape[0], T.shape[0], R.shape[1]
    zi, zs, zo = unit_basis(n, m, p, r)
    paths, info = oss.simulation_smoother(y, a0, P0, T, Z, R, H, Q, c, d, zi, zs, zo)
    assert info == 0
    mean, cov = oss.dense_state_posterior(y, a0, P0, T, Z, R, H, Q, c, d)
    MM = check_joint(paths, mean, cov, rtol)
    if c is None and d is None and not np.isnan(y).all() and H.any():
        # the marginal blocks are the RTS smoother's covariances (not with H = 0: its gain takes the pseudo-inverse of a
        # singular predicted covariance there, good to ~1e-6 only)
        fs, _, fc, _, _, _ = kn.kalman_filter("standard", y, a0, P0, T, Z, R, H, Q, strict_reference=False)
        _, sc = kn.kalman_smoother(T, R, Q, fs, fc)
        for t in range(n):
            blk = MM[t * m:(t + 1) * m, t * m:(t + 1) * m]
            assert np.abs(blk - sc[t]).max() <= 1e-9 * (np.abs(sc).max() + 1.0), (name, t)


def test_oracle_nile_diffuse_p0():
    """Nile, P0 = 1e6 I.  The dense solve conditions a 1e6-scale prior on 100 observations and keeps only about six
    significant digits here (its mean is 2e-6 relative off the RTS smoother's, which the recursion matches to 3e-10), so
    the tolerance is 2e-5 relative."""
    y, a0, P0, T, Z, R, H, Q = nile_inputs()
    n, m, p, r = y.shape[0], 2, 1, 2
    zi, zs, zo = unit_basis(n, m, p, r)
    paths, info = oss.simulation_smoother(y, a0, P0, T, Z, R, H, Q, None, None, zi, zs, zo)
    assert info == 0
    mean, cov = oss.dense_state_posterior(y, a0, P0, T, Z, R, H, Q)
    check_joint(paths, mean, cov, 2e-5)


def test_marginal_draws_fail_the_cross_time_check():
    """Draws from the smoothed marginals (what conditional_simulation does) have the right diagonal blocks and the wrong
    cross-time blocks: the check above tells joint from marginal."""
    case = CASES[IDS.index("random_m2_p1_r2")] if "random_m2_p1_r2" in IDS else CASES[3]
    _, y, a0, P0, T, Z, R, H, Q, c, d, _ = case
    n, m = y.shape[0], T.shape[0]
    mean, cov = oss.dense_state_posterior(y, a0, P0, T, Z, R, H, Q, c, d)
    # the affine map of the marginal sampler: x_t = mean_t + chol(Sigma_tt) z_t with z_t independent over t
    N = n * m
    paths = np.empty((N + 1, n, m))
    paths[0] = mean
    E = np.eye(N)
    for k in range(N):
        for t in range(n):
            blk = cov[t * m:(t + 1) * m, t * m:(t + 1) * m]
            paths[k + 1, t] = mean[t] + np.linalg.cholesky(blk) @ E[k, t * m:(t + 1) * m]
    M = paths[1:].reshape(N, -1) - paths[0].reshape(-1)
    MM = M.T @ M
    for t in range(n):  # marginals agree
        sl = slice(t * m, (t + 1) * m)
        assert np.abs(MM[sl, sl] - cov[sl, sl]).max() <= 1e-10 * np.abs(cov).max()
    with pytest.raises(AssertionError):
        check_joint(paths, mean, cov, 1e-10)


def test_oracle_factor_rule():
    L, ok = oss.psd_factor(np.zeros((2, 2)))
    assert ok and not L.any()
    A = np.array([[2.0, 1.0], [1.0, 0.5]])  # rank 1
    L, ok = oss.psd_factor(A)
    assert ok and np.abs(L @ L.T - A).max() < 1e-14 and L[1, 1] == 0.0
    _, ok = oss.psd_factor(np.array([[1.0, 0.0], [0.0, -0.1]]))
    assert not ok


# ---------------------------------------------------------------------------------------------------- host build
@pytest.mark.parametrize("force_dyn", [False, True], ids=["instantiation", "runtime_dims"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_host_build_equals_oracle(case, force_dyn):
    from tests.hostsim.draws import simsmooth

    name, y, a0, P0, T, Z, R, H, Q, c, d, _ = case
    n, p, m, r = y.shape[0], Z.shape[0], T.shape[0], R.shape[1]
    rng = np.random.default_rng(11)
    S = 5
    zi, zs, zo = random_normals(rng, S, n, m, p, r)
    pc = oss.predicted_covs(y, P0, T, Z, R, H, Q)
    want, info = oss.simulation_smoother(y, a0, P0, T, Z, R, H, Q, c, d, zi, zs, zo, P=pc)
    assert info == 0
    got, hinfo = simsmooth(y[..., 0], mats_of(case), pc[None], S, zi, zs.reshape(-1), zo, force_dyn=force_dyn)
    assert (hinfo == 0).all()
    assert np.abs(got - want).max() <= 1e-13 * (np.abs(want).max() + 1.0), name


def test_host_build_nile():
    from tests.hostsim.draws import simsmooth

    y, a0, P0, T, Z, R, H, Q = nile_inputs(n_missing=5)
    rng = np.random.default_rng(2)
    S, n = 4, y.shape[0]
    zi, zs, zo = random_normals(rng, S, n, 2, 1, 2)
    pc = oss.predicted_covs(y, P0, T, Z, R, H, Q)
    want, _ = oss.simulation_smoother(y, a0, P0, T, Z, R, H, Q, None, None, zi, zs, zo, P=pc)
    got, info = simsmooth(y[..., 0], dict(a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q), pc[None], S, zi, zs, zo)
    assert (info == 0).all()
    # P0 = 1e6 I: xhat_0 = P0 r_{-1} scales the rounding of r_{-1} (different F^-1 and summation orders) by 1e6
    assert np.abs(got - want).max() <= 1e-8 * np.abs(want).max()


def test_host_build_info_codes():
    from tests.hostsim.draws import simsmooth
    from pymc_statespace_b200._lib import KFB_INFO_NOT_PSD

    rng = np.random.default_rng(5)
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 2, 2, 2, 6)
    zi, zs, zo = random_normals(rng, 2, 6, 2, 2, 2)
    pc = oss.predicted_covs(y, P0, T, Z, R, H, Q)
    mats = dict(a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q)
    yp = y.copy()
    yp[3, 1] = np.nan  # partly missing row 3
    got, info = simsmooth(yp[..., 0], dict(mats), pc[None], 2, zi, zs, zo)
    assert info[0] == -4 and np.isnan(got).all()
    got, info = simsmooth(y[..., 0], dict(mats, Q=-Q), pc[None], 2, zi, zs, zo)
    assert info[0] == KFB_INFO_NOT_PSD and np.isnan(got).all()
    pc_bad = pc.copy()
    pc_bad[2] = -10 * np.eye(2)  # F_2 = Z P_2 Z^T + H not PD
    got, info = simsmooth(y[..., 0], dict(mats), pc_bad[None], 2, zi, zs, zo)
    assert info[0] == 3 and np.isnan(got).all()


def test_instantiation_choice():
    from tests import hostsim

    for m in range(1, 5):
        for p in range(1, 4):
            assert hostsim.simsmooth_is_static(m, p, 1) and hostsim.simsmooth_is_static(m, p, m)
    assert not hostsim.simsmooth_is_static(2, 1, 3) and not hostsim.simsmooth_is_static(5, 1, 1) and not hostsim.simsmooth_is_static(13, 1, 3)
    assert not hostsim.simsmooth_is_static(2, 4, 1)


# ---------------------------------------------------------------------------------------------------- C ABI
def _desc(n_draws=3, n_series=2, n=50, m=2, p=1, r=1):
    from pymc_statespace_b200 import _lib

    d = _lib.KfbDesc()
    d.n_draws, d.n_series, d.n, d.m, d.p, d.r = n_draws, n_series, n, m, p, r
    return d


def _round(b):
    return (b + 255) // 256 * 256


def test_cabi_workspace_rule():
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    nb = ctypes.c_size_t(0)
    for (nd, ns, n, m, p, r, spu) in ((3, 2, 50, 2, 1, 1, 7), (1, 1, 1, 13, 1, 3, 64), (4, 1, 10, 3, 2, 2, 1)):
        d = _desc(nd, ns, n, m, p, r)
        assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(d), spu, ctypes.byref(nb)) == _lib.KFB_OK
        U = nd * ns
        S32 = (U * spu + 31) // 32 * 32
        want = (_round(8 * U * n * (m * p + p * p)) + _round(8 * U * (2 * m * m + m * r + p * p + r * r))
                + _round(8 * n * S32 * p) + _round(8 * (n - 1) * S32 * m) + _round(4 * U))
        assert nb.value == want


def test_cabi_argument_validation():
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    nb = ctypes.c_size_t(0)
    d = _desc()
    assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(d), 0, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    assert lib.kfb_simulation_smoother_workspace_bytes(None, 4, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(d), 4, None) == _lib.KFB_ERR_INVALID_ARG
    for k in ("n", "m", "p", "r", "n_draws", "n_series"):
        bad = _desc()
        setattr(bad, k, 0)
        assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(bad), 4, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    for k in ("T", "Z", "R", "H", "Q", "c", "d"):
        tv = _desc()
        setattr(tv, k + "_ts", 4)
        assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(tv), 4, ctypes.byref(nb)) == _lib.KFB_ERR_UNSUPPORTED
        ins = _lib.KfbInputs()
        assert lib.kfb_simulation_smoother(ctypes.byref(tv), ctypes.byref(ins), None, 4, None, None, None, None, None, None,
                                           0, None) == _lib.KFB_ERR_UNSUPPORTED
    big = _desc(m=33)
    assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(big), 4, ctypes.byref(nb)) == _lib.KFB_ERR_UNSUPPORTED
    # null pointers (checked before any device work)
    ins = _lib.KfbInputs()
    assert lib.kfb_simulation_smoother(ctypes.byref(d), ctypes.byref(ins), None, 4, None, None, None, None, None, None, 0,
                                       None) == _lib.KFB_ERR_INVALID_ARG
    assert lib.kfb_simulation_smoother(ctypes.byref(d), None, None, 4, None, None, None, None, None, None, 0,
                                       None) == _lib.KFB_ERR_INVALID_ARG
