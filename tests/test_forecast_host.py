"""CPU checks of the forecasts from the end of the sample and the impulse responses: the numpy restatement
(oracle/forecast.py) pins itself against dense joint-Gaussian algebra through the affine map from normals to paths, the
host build of the kernels' KFB_HD code (tests/hostsim/draws.cpp) equals the restatement, and the C ABI validates its
arguments without a device."""
import ctypes

import numpy as np
import pytest

from oracle import forecast as ofc
from tests.helpers import random_system
from tests.test_simulation_smoother_host import arma11, check_joint, random_normals, unit_basis


def local_linear_trend(n=10, n_missing_tail=3, seed=4):
    rng = np.random.default_rng(seed)
    y = np.cumsum(rng.normal(size=n))[:, None, None]
    y[n - n_missing_tail:] = np.nan  # missing rows at the end of the sample
    T = np.array([[1.0, 1.0], [0.0, 1.0]])
    return y, np.zeros((2, 1)), np.eye(2), T, np.array([[1.0, 0.0]]), np.eye(2), np.array([[0.8]]), np.diag([0.5, 0.01])


def cases():
    """(name, y, a0, P0, T, Z, R, H, Q, c, d, horizon)"""
    rng = np.random.default_rng(17)
    out = []
    for (m, p, r) in ((2, 1, 2), (4, 3, 4)):
        y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, r, 8)
        y[3] = np.nan
        out.append((f"random_m{m}_p{p}_r{r}", y, a0, P0, T, Z, R, H, Q, rng.normal(size=(m, 1)), rng.normal(size=(p, 1)),
                    5))
    out.append(("arma11_H0",) + arma11(0.6, 0.3) + (None, None, 6))  # P_n of rank < k_states
    out.append(("local_linear_trend_missing_tail",) + local_linear_trend() + (None, None, 4))
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 3, 2, 2, 1)
    out.append(("n1", y, a0, P0, T, Z, R, H, Q, rng.normal(size=(3, 1)), None, 4))
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 2, 2, 1, 6)
    out.append(("horizon1", y, a0, P0, T, Z, R, H, Q, None, rng.normal(size=(2, 1)), 1))
    return out


CASES = cases()
IDS = [c[0] for c in CASES]


def _start(case):
    _, y, a0, P0, T, Z, R, H, Q, c, d, hor = case
    mom = ofc.forecast_moments(y, a0, P0, T, Z, R, H, Q, c, d, horizon=hor)
    return mom, mom["state_mean"][0], mom["state_cov"][0]


# ---------------------------------------------------------------------------------------------------- oracle pins itself
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_oracle_joint_law_matches_dense_forecast_law(case):
    name, y, a0, P0, T, Z, R, H, Q, c, d, hor = case
    m, p, r = T.shape[0], Z.shape[0], R.shape[1]
    _, a, P = _start(case)
    zi, zs, zo = unit_basis(hor, m, p, r)
    states, obs, info = ofc.forecast_paths(a, P, T, Z, R, H, Q, c, d, zi, zs, zo)
    assert info == 0
    xm, xc, ym, yc = ofc.dense_forecast_law(y, a0, P0, T, Z, R, H, Q, c, d, horizon=hor)
    check_joint(states, xm, xc, 1e-10)
    check_joint(obs, ym, yc, 1e-10)


def test_marginal_draws_fail_the_cross_horizon_check():
    """Horizon-by-horizon draws from the forecast marginals have the right diagonal blocks and the wrong cross-horizon
    blocks: the check above tells joint from marginal."""
    _, y, a0, P0, T, Z, R, H, Q, c, d, hor = CASES[0]
    m = T.shape[0]
    xm, xc, _, _ = ofc.dense_forecast_law(y, a0, P0, T, Z, R, H, Q, c, d, horizon=hor)
    N = hor * m
    paths = np.empty((N + 1, hor, m))
    paths[0] = xm
    E = np.eye(N)
    for k in range(N):
        for h in range(hor):
            blk = xc[h * m:(h + 1) * m, h * m:(h + 1) * m]
            paths[k + 1, h] = xm[h] + np.linalg.cholesky(blk) @ E[k, h * m:(h + 1) * m]
    M = paths[1:].reshape(N, -1) - paths[0].reshape(-1)
    MM = M.T @ M
    for h in range(hor):  # marginals agree
        sl = slice(h * m, (h + 1) * m)
        assert np.abs(MM[sl, sl] - xc[sl, sl]).max() <= 1e-10 * np.abs(xc).max()
    with pytest.raises(AssertionError):
        check_joint(paths, xm, xc, 1e-10)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_forecast_moments_equal_dense_diagonal_blocks(case):
    name, y, a0, P0, T, Z, R, H, Q, c, d, hor = case
    m, p = T.shape[0], Z.shape[0]
    mom, _, _ = _start(case)
    xm, xc, ym, yc = ofc.dense_forecast_law(y, a0, P0, T, Z, R, H, Q, c, d, horizon=hor)
    for got, want, k in ((mom["state_mean"], xm, None), (mom["obs_mean"], ym, None), (mom["state_cov"], xc, m),
                         (mom["obs_cov"], yc, p)):
        if k is not None:
            want = np.stack([want[h * k:(h + 1) * k, h * k:(h + 1) * k] for h in range(hor)])
        assert np.abs(got - want).max() <= 1e-12 * (np.abs(want).max() + 1.0), name


# ---------------------------------------------------------------------------------------------------- impulse responses
def test_oracle_impulse_responses_closed_forms():
    phi, theta, hor = 0.7, 0.4, 12
    _, _, _, T, Z, R, _, Q = arma11(phi, theta)
    _, obs = ofc.impulse_responses(T, Z, R, Q, hor, "unit")
    psi = np.array([1.0] + [(phi + theta) * phi ** (h - 1) for h in range(1, hor)])
    assert np.abs(obs[:, 0, 0] - psi).max() <= 1e-14
    A = np.array([[0.5, 0.1, 0.0], [-0.2, 0.3, 0.2], [0.1, 0.0, 0.4]])
    L = np.array([[1.0, 0.0, 0.0], [0.3, 0.8, 0.0], [-0.2, 0.1, 0.5]])
    Qv = L @ L.T
    for shock, S in (("unit", np.eye(3)), ("std", np.diag(np.sqrt(np.diag(Qv)))), ("cholesky", L)):
        states, obs = ofc.impulse_responses(A, np.eye(3), np.eye(3), Qv, hor, shock)
        want = np.stack([np.linalg.matrix_power(A, h) @ S for h in range(hor)])
        assert np.abs(states - want).max() <= 1e-14 and np.abs(obs - want).max() <= 1e-14
    one = np.ones((1, 1))
    states, obs = ofc.impulse_responses(one, one, one, 0.3 * one, hor, "unit")
    assert (states == 1.0).all() and (obs == 1.0).all()


# ---------------------------------------------------------------------------------------------------- host build
GEOMS = [(m, p, r) for m in range(1, 5) for p in range(1, 4) for r in sorted({1, m})] + [(5, 1, 2), (3, 4, 2), (2, 1, 3)]


def _batched_system(rng, m, p, r, n_draws):
    systems = [random_system(rng, m, p, r, 2) for _ in range(n_draws)]
    st = lambda i: np.stack([s[i] for s in systems])  # noqa: E731
    T, Z, R, H, Q = st(3), st(4), st(5), st(6), st(7)
    return dict(T=T, Z=Z, R=R, H=H, Q=Q, c=rng.normal(size=(n_draws, m)), d=rng.normal(size=(n_draws, p)))


def _oracle_paths(mats, mean, cov, spu, zi, zs, zo, n_draws, n_series):
    hor = zo.shape[0]
    m, p = mats["T"].shape[-1], mats["Z"].shape[-2]
    S = n_draws * n_series * spu
    states, obs = np.empty((hor, S, m)), np.empty((hor, S, p))
    infos = []
    for u in range(n_draws * n_series):
        b = u // n_series
        sl = slice(u * spu, (u + 1) * spu)
        mb = {k: v[b] for k, v in mats.items()}
        xs, ys, info = ofc.forecast_paths(mean[u], cov[u], mb["T"], mb["Z"], mb["R"], mb["H"], mb["Q"], mb["c"], mb["d"],
                                          zi[sl], zs[:, sl], zo[:, sl])
        states[:, sl], obs[:, sl] = xs.transpose(1, 0, 2), ys.transpose(1, 0, 2)
        infos.append(info)
    return states, obs, infos


def _starts(rng, U, m):
    A = rng.normal(size=(U, m, m))
    return rng.normal(size=(U, m)), A @ A.transpose(0, 2, 1) + 0.1 * np.eye(m)


@pytest.mark.parametrize("force_dyn", [False, True], ids=["instantiation", "runtime_dims"])
@pytest.mark.parametrize("geom", GEOMS, ids=[f"m{m}_p{p}_r{r}" for (m, p, r) in GEOMS])
def test_host_build_equals_oracle(geom, force_dyn):
    from tests import hostsim
    from tests.hostsim import draws as hfc

    m, p, r = geom
    rng = np.random.default_rng(100 * m + 10 * p + r)
    nD, NS, spu, hor = 3, 2, 37, 6
    mats = _batched_system(rng, m, p, r, nD)
    mean, cov = _starts(rng, nD * NS, m)
    zi, zs, zo = random_normals(rng, nD * NS * spu, hor, m, p, r)
    want_x, want_y, infos = _oracle_paths(mats, mean, cov, spu, zi, zs, zo, nD, NS)
    assert all(i == 0 for i in infos)
    x, y, info, used_static = hfc.forecast_paths(mats, mean, cov, spu, zi, zs, zo, n_draws=nD, n_series=NS,
                                                     force_dyn=force_dyn)
    assert (info == 0).all()
    assert used_static == (not force_dyn and hostsim.simsmooth_is_static(m, p, r))
    assert np.abs(x - want_x).max() <= 1e-13 * (np.abs(want_x).max() + 1.0)
    assert np.abs(y - want_y).max() <= 1e-13 * (np.abs(want_y).max() + 1.0)
    # either output alone gives the same bits
    x1, y1, _, _ = hfc.forecast_paths(mats, mean, cov, spu, zi, zs, zo, nD, NS, force_dyn, want=("states",))
    x2, y2, _, _ = hfc.forecast_paths(mats, mean, cov, spu, zi, zs, zo, nD, NS, force_dyn, want=("obs",))
    assert y1 is None and x2 is None and np.array_equal(x1, x) and np.array_equal(y2, y)


def test_host_build_horizon1_shared_matrices():
    from tests.hostsim import draws as hfc

    rng = np.random.default_rng(6)
    _, _, _, T, Z, R, H, Q = random_system(rng, 2, 1, 2, 2)
    mats = dict(T=T, Z=Z, R=R, H=H, Q=Q)
    mean, cov = _starts(rng, 1, 2)
    zi, _, zo = random_normals(rng, 5, 1, 2, 1, 2)
    x, y, info, _ = hfc.forecast_paths(mats, mean, cov, 5, zi, None, zo)
    wx, wy, winfo = ofc.forecast_paths(mean[0], cov[0], T, Z, R, H, Q, None, None, zi, np.zeros((0, 5, 2)), zo)
    assert winfo == 0 and (info == 0).all()
    assert np.abs(x[0] - wx[:, 0]).max() <= 1e-13 * np.abs(wx).max()
    assert np.abs(y[0] - wy[:, 0]).max() <= 1e-13 * np.abs(wy).max()


@pytest.mark.parametrize("force_dyn", [False, True], ids=["instantiation", "runtime_dims"])
def test_host_build_info_codes(force_dyn):
    from pymc_statespace_b200._lib import KFB_INFO_NOT_PSD
    from tests.hostsim import draws as hfc

    rng = np.random.default_rng(8)
    nD, NS, spu, hor, m, p, r = 3, 2, 4, 5, 2, 2, 2
    mats = _batched_system(rng, m, p, r, nD)
    mats["Q"][1] = -mats["Q"][1]  # draw 1: Q not PSD -> units 2, 3
    mean, cov = _starts(rng, nD * NS, m)
    cov[4] = np.array([[1.0, 0.0], [0.0, -0.5]])  # unit 4: start covariance not PSD
    mean[5, 1] = np.nan  # unit 5: NaN start
    zi, zs, zo = random_normals(rng, nD * NS * spu, hor, m, p, r)
    x, y, info, _ = hfc.forecast_paths(mats, mean, cov, spu, zi, zs, zo, nD, NS, force_dyn)
    assert list(info) == [0, 0, KFB_INFO_NOT_PSD, KFB_INFO_NOT_PSD, KFB_INFO_NOT_PSD, KFB_INFO_NOT_PSD]
    good = slice(0, 2 * spu)
    assert np.isfinite(x[:, good]).all() and np.isfinite(y[:, good]).all()
    assert np.isnan(x[:, 2 * spu:]).all() and np.isnan(y[:, 2 * spu:]).all()
    _, _, infos = _oracle_paths(mats, mean, cov, spu, zi, zs, zo, nD, NS)
    assert infos == [0, 0] + ["not_psd"] * 4


@pytest.mark.parametrize("force_dyn", [False, True], ids=["instantiation", "runtime_dims"])
@pytest.mark.parametrize("geom", GEOMS, ids=[f"m{m}_p{p}_r{r}" for (m, p, r) in GEOMS])
def test_host_build_impulse_responses_equal_oracle(geom, force_dyn):
    from pymc_statespace_b200._lib import SHOCK_KIND
    from tests import hostsim
    from tests.hostsim import draws as hfc

    m, p, r = geom
    rng = np.random.default_rng(7 + m + p + r)
    nD, hor = 3, 7
    mats = _batched_system(rng, m, p, r, nD)
    for shock, code in SHOCK_KIND.items():
        x, y, info, used_static = hfc.impulse_response(mats, hor, code, n_draws=nD, force_dyn=force_dyn)
        assert (info == 0).all() and used_static == (not force_dyn and hostsim.simsmooth_is_static(m, p, r))
        for b in range(nD):
            wx, wy = ofc.impulse_responses(mats["T"][b], mats["Z"][b], mats["R"][b], mats["Q"][b], hor, shock)
            assert np.abs(x[b] - wx).max() <= 1e-13 * (np.abs(wx).max() + 1.0), (shock, b)
            assert np.abs(y[b] - wy).max() <= 1e-13 * (np.abs(wy).max() + 1.0), (shock, b)


def test_host_build_impulse_responses_closed_forms_and_info():
    from pymc_statespace_b200._lib import KFB_INFO_NOT_PSD, SHOCK_KIND
    from tests.hostsim import draws as hfc

    phi, theta, hor = -0.6, 0.25, 15
    _, _, _, T, Z, R, _, Q = arma11(phi, theta)
    _, y, info, _ = hfc.impulse_response(dict(T=T, Z=Z, R=R, Q=Q), hor, SHOCK_KIND["unit"])
    psi = np.array([1.0] + [(phi + theta) * phi ** (h - 1) for h in range(1, hor)])
    assert info[0] == 0 and np.abs(y[0, :, 0, 0] - psi).max() <= 1e-14
    one = np.ones((1, 1))
    x, y, _, _ = hfc.impulse_response(dict(T=one, Z=one, R=one, Q=one), hor, SHOCK_KIND["unit"])
    assert (x == 1.0).all() and (y == 1.0).all()
    rng = np.random.default_rng(3)
    mats = _batched_system(rng, 3, 1, 2, 2)
    mats["Q"][1] = -mats["Q"][1]
    for shock, code in SHOCK_KIND.items():
        x, y, info, _ = hfc.impulse_response(mats, 4, code, n_draws=2)
        assert info[0] == 0 and np.isfinite(x[0]).all() and np.isfinite(y[0]).all()
        if shock == "unit":  # S = I does not read Q
            assert info[1] == 0 and np.isfinite(x[1]).all()
        else:
            assert info[1] == KFB_INFO_NOT_PSD and np.isnan(x[1]).all() and np.isnan(y[1]).all()


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
    for (nd, ns, m, p, r, spu) in ((3, 2, 2, 1, 1, 7), (1, 1, 13, 1, 3, 64), (4, 1, 3, 2, 2, 1), (2, 3, 32, 32, 32, 5)):
        d = _desc(nd, ns, 0, m, p, r)  # desc->n is not read
        assert lib.kfb_forecast_paths_workspace_bytes(ctypes.byref(d), spu, ctypes.byref(nb)) == _lib.KFB_OK
        U = nd * ns
        assert nb.value == _round(8 * U * (m * m + m * r + p * p + r * r)) + _round(4 * U)


def test_cabi_argument_validation():
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    nb = ctypes.c_size_t(0)
    d = _desc()
    fw = lib.kfb_forecast_paths_workspace_bytes
    assert fw(ctypes.byref(d), 0, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    assert fw(None, 4, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    assert fw(ctypes.byref(d), 4, None) == _lib.KFB_ERR_INVALID_ARG
    for k in ("m", "p", "r", "n_draws", "n_series"):
        bad = _desc()
        setattr(bad, k, 0)
        assert fw(ctypes.byref(bad), 4, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    ins = _lib.KfbInputs()
    for k in ("T", "Z", "R", "H", "Q", "c", "d"):
        tv = _desc()
        setattr(tv, k + "_ts", 4)
        assert fw(ctypes.byref(tv), 4, ctypes.byref(nb)) == _lib.KFB_ERR_UNSUPPORTED
        assert lib.kfb_forecast_paths(ctypes.byref(tv), ctypes.byref(ins), None, None, 3, 4, None, None, None, None, None,
                                      None, None, 0, None) == _lib.KFB_ERR_UNSUPPORTED
        assert lib.kfb_impulse_response(ctypes.byref(tv), ctypes.byref(ins), 3, 0, None, None, None,
                                        None) == _lib.KFB_ERR_UNSUPPORTED
    for k in ("m", "p", "r"):
        big = _desc(**{k: 33})
        assert fw(ctypes.byref(big), 4, ctypes.byref(nb)) == _lib.KFB_ERR_UNSUPPORTED
        assert lib.kfb_impulse_response(ctypes.byref(big), ctypes.byref(ins), 3, 0, None, None, None,
                                        None) == _lib.KFB_ERR_UNSUPPORTED
    # null pointers, horizon < 1, both outputs NULL, bad shock, small workspace (all checked before any device work)
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below is refused first
    full = _lib.KfbInputs(*([fake] * 8 + [None, None]))
    fp = lib.kfb_forecast_paths

    def paths(ins_, mean=fake, cov=fake, hor=3, spu=4, zi=fake, zs=fake, zo=fake, xs=fake, ys=fake, info=fake, ws=None,
              nbytes=0):
        return fp(ctypes.byref(d), ins_ if ins_ is None else ctypes.byref(ins_), mean, cov, hor, spu, zi, zs, zo, xs, ys,
                  info, ws, nbytes, None)

    assert paths(None) == _lib.KFB_ERR_INVALID_ARG
    assert paths(ins) == _lib.KFB_ERR_INVALID_ARG
    for kw in (dict(mean=None), dict(cov=None), dict(zi=None), dict(zs=None), dict(zo=None), dict(info=None),
               dict(xs=None, ys=None), dict(hor=0), dict(spu=0)):
        assert paths(full, **kw) == _lib.KFB_ERR_INVALID_ARG, kw
    assert fw(ctypes.byref(d), 4, ctypes.byref(nb)) == _lib.KFB_OK
    assert paths(full) == _lib.KFB_ERR_WORKSPACE
    assert paths(full, ws=fake, nbytes=nb.value - 1) == _lib.KFB_ERR_WORKSPACE
    ir = lib.kfb_impulse_response
    assert ir(ctypes.byref(d), ctypes.byref(full), 3, 3, fake, fake, fake, None) == _lib.KFB_ERR_INVALID_ARG
    assert ir(ctypes.byref(d), ctypes.byref(full), 3, -1, fake, fake, fake, None) == _lib.KFB_ERR_INVALID_ARG
    assert ir(ctypes.byref(d), ctypes.byref(full), 0, 0, fake, fake, fake, None) == _lib.KFB_ERR_INVALID_ARG
    assert ir(ctypes.byref(d), ctypes.byref(full), 3, 0, None, None, fake, None) == _lib.KFB_ERR_INVALID_ARG
    assert ir(ctypes.byref(d), ctypes.byref(full), 3, 0, fake, fake, None, None) == _lib.KFB_ERR_INVALID_ARG
    assert ir(ctypes.byref(d), ctypes.byref(ins), 3, 0, fake, fake, fake, None) == _lib.KFB_ERR_INVALID_ARG
    assert ir(None, ctypes.byref(full), 3, 0, fake, fake, fake, None) == _lib.KFB_ERR_INVALID_ARG
