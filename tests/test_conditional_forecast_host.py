"""CPU checks of the conditional forecasts: the numpy restatement (oracle/condforecast.py) and the host build of the
kernels' KFB_HD code (tests/hostsim/condfc.cpp) pin themselves against dense joint-Gaussian algebra through the affine
map from normals to paths, the host build equals the restatement on every instantiation, and the C ABI validates its
arguments without a device."""
import ctypes

import numpy as np
import pytest

from oracle import condforecast as ocf
from oracle import forecast as ofc
from tests.helpers import random_system
from tests.test_forecast_host import GEOMS, _batched_system, _starts
from tests.test_simulation_smoother_host import arma11, check_joint, random_normals, unit_basis


def _cond(hor, p, entries):
    cond = np.full((hor, p), np.nan)
    for (h, i, v) in entries:
        cond[h, i] = v
    return cond


def cases():
    """(name, y, a0, P0, T, Z, R, H, Q, c, d, cond)"""
    rng = np.random.default_rng(23)
    out = []
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 3, 2, 2, 8, diag_H=True)
    c, d = rng.normal(size=3), rng.normal(size=2)
    out.append(("full_rows", y, a0, P0, T, Z, R, H, Q, c, d, _cond(5, 2, [(0, 0, 0.3), (0, 1, -0.2), (3, 0, 1.1),
                                                                         (3, 1, 0.4)])))
    out.append(("single_entries", y, a0, P0, T, Z, R, H, Q, c, d, _cond(5, 2, [(0, 1, 0.5), (2, 0, -0.7), (4, 1, 0.2)])))
    out.append(("later_horizons_only", y, a0, P0, T, Z, R, H, Q, c, d, _cond(6, 2, [(4, 0, 0.9), (5, 0, 1.2)])))
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 4, 3, 2, 7)  # H not diagonal
    c, d = rng.normal(size=4), rng.normal(size=3)
    out.append(("nondiag_H", y, a0, P0, T, Z, R, H, Q, c, d, _cond(4, 3, [(0, 0, 0.1), (1, 1, -0.4), (1, 2, 0.6),
                                                                          (3, 0, 0.2), (3, 2, -0.1)])))
    Hs = H.copy()
    Hs[0, :] = Hs[:, 0] = 0.0  # a singular H: the generalised inverse's zero pivot
    out.append(("singular_nondiag_H", y, a0, P0, T, Z, R, Hs, Q, c, d, _cond(4, 3, [(0, 0, 0.1), (1, 0, 0.3),
                                                                                    (1, 1, -0.4), (2, 2, 0.5)])))
    out.append(("arma11_H0",) + arma11(0.6, 0.3) + (None, None, _cond(6, 1, [(1, 0, 0.8), (4, 0, -0.5)])))
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 3, 2, 3, 6)
    out.append(("H0_p2_single_entries", y, a0, P0, T, Z, R, 0.0 * H, Q, None, None,
                _cond(4, 2, [(0, 0, 0.2), (2, 1, 0.3), (3, 0, -0.1)])))
    return out


CASES = cases()
IDS = [c[0] for c in CASES]


def _start(y, a0, P0, T, Z, R, H, Q, c, d):
    mom = ofc.forecast_moments(y, a0, P0, T, Z, R, H, Q, c, d, horizon=1)
    return mom["state_mean"][0], mom["state_cov"][0]


def _mats(T, Z, R, H, Q, c, d):
    return dict(T=T, Z=Z, R=R, H=H, Q=Q, c=c, d=d)


def joint(states, obs):
    """[S, H, m] and [S, H, p] paths -> [S, 1, H m + H p]: the vector of dense_conditional_forecast_law per path."""
    S = states.shape[0]
    return np.concatenate([states.reshape(S, -1), obs.reshape(S, -1)], axis=1)[:, None, :]


def _host(case, spu, zi, zs, zo, force_dyn=False):
    from tests.hostsim import condfc as hcf

    _, y, a0, P0, T, Z, R, H, Q, c, d, cond = case
    a, P = _start(y, a0, P0, T, Z, R, H, Q, c, d)
    mom, x, yy, info, _ = hcf.conditional_forecast(_mats(T, Z, R, H, Q, c, d), a[None], P[None], cond, spu, zi, zs, zo,
                                                   n=len(y), force_dyn=force_dyn)
    return mom, (None if x is None else x.transpose(1, 0, 2)), (None if yy is None else yy.transpose(1, 0, 2)), info


# ---------------------------------------------------------------------------------------------------- joint law
@pytest.mark.parametrize("force_dyn", [False, True], ids=["instantiation", "runtime_dims"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_joint_law_matches_dense_conditional_law(case, force_dyn):
    """Zero and unit-vector normals: the affine map from normals to (states, observations) paths has the dense law's
    mean and full covariance, cross-horizon and state-observation blocks included, for the restatement and the host
    build."""
    name, y, a0, P0, T, Z, R, H, Q, c, d, cond = case
    m, p, r, hor = T.shape[0], Z.shape[0], R.shape[1], cond.shape[0]
    zi, zs, zo = unit_basis(hor, m, p, r)
    mean, cov = ocf.dense_conditional_forecast_law(y, a0, P0, T, Z, R, H, Q, c, d, cond)
    a, P = _start(y, a0, P0, T, Z, R, H, Q, c, d)
    xs, ys, info = ocf.conditional_paths(a, P, T, Z, R, H, Q, c, d, cond, zi, zs, zo, n=len(y))
    assert info == 0
    check_joint(joint(xs, ys), mean, cov, 1e-10)
    _, hx, hy, hinfo = _host(case, zi.shape[0], zi, zs, zo, force_dyn)
    assert (hinfo == 0).all()
    check_joint(joint(hx, hy), mean, cov, 1e-10)
    o = ~np.isnan(cond)
    assert (hy[:, o] == cond[o]).all()  # conditioned entries are the condition, bit for bit


def test_overwritten_unconditional_paths_fail_the_check():
    """Unconditional forecast paths with the known entries overwritten have the wrong law: the states and the other
    series do not respond to the condition."""
    name, y, a0, P0, T, Z, R, H, Q, c, d, cond = CASES[1]
    m, p, r, hor = T.shape[0], Z.shape[0], R.shape[1], cond.shape[0]
    zi, zs, zo = unit_basis(hor, m, p, r)
    a, P = _start(y, a0, P0, T, Z, R, H, Q, c, d)
    xs, ys, _ = ofc.forecast_paths(a, P, T, Z, R, H, Q, c, d, zi, zs, zo)
    o = ~np.isnan(cond)
    ys[:, o] = cond[o]
    mean, cov = ocf.dense_conditional_forecast_law(y, a0, P0, T, Z, R, H, Q, c, d, cond)
    with pytest.raises(AssertionError):
        check_joint(joint(xs, ys), mean, cov, 1e-10)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_moments_match_dense_law(case):
    name, y, a0, P0, T, Z, R, H, Q, c, d, cond = case
    m, p, hor = T.shape[0], Z.shape[0], cond.shape[0]
    mean, cov = ocf.dense_conditional_forecast_law(y, a0, P0, T, Z, R, H, Q, c, d, cond)
    a, P = _start(y, a0, P0, T, Z, R, H, Q, c, d)
    want = {"state_mean": mean[:hor * m].reshape(hor, m), "obs_mean": mean[hor * m:].reshape(hor, p),
            "state_cov": np.stack([cov[h * m:(h + 1) * m, h * m:(h + 1) * m] for h in range(hor)]),
            "obs_cov": np.stack([cov[hor * m + h * p:hor * m + (h + 1) * p, hor * m + h * p:hor * m + (h + 1) * p]
                                 for h in range(hor)])}
    got, _, info = ocf.window(a, P, T, Z, R, H, Q, c, d, cond, n=len(y))
    hmom, _, _, hinfo = _host(case, 0, None, None, None)
    assert info == 0 and (hinfo == 0).all()
    o = ~np.isnan(cond)
    assert (hmom["obs_mean"][0][o] == cond[o]).all()
    assert (hmom["obs_cov"][0][:, :, :][np.broadcast_to(o[:, :, None], (hor, p, p))] == 0.0).all()
    for k, v in want.items():
        scale = max(np.abs(v).max(), 1.0)
        assert np.abs(got[k] - v).max() <= 1e-10 * scale, (name, k)
        assert np.abs(hmom[k][0] - v).max() <= 1e-10 * scale, (name, k)


@pytest.mark.parametrize("force_dyn", [False, True], ids=["instantiation", "runtime_dims"])
def test_all_nan_conditions_reproduce_forecast(force_dyn):
    """No condition: the moments are forecast's (to rounding) and the paths are the forecast paths bit for bit."""
    from tests.hostsim import forecast as hfc

    name, y, a0, P0, T, Z, R, H, Q, c, d, _ = CASES[3]
    m, p, r, hor, spu = T.shape[0], Z.shape[0], R.shape[1], 6, 37
    cond = np.full((hor, p), np.nan)
    zi, zs, zo = random_normals(np.random.default_rng(5), spu, hor, m, p, r)
    mom, x, yy, info = _host(CASES[3][:-1] + (cond,), spu, zi, zs, zo, force_dyn)
    a, P = _start(y, a0, P0, T, Z, R, H, Q, c, d)
    fx, fy, finfo, _ = hfc.forecast_paths(_mats(T, Z, R, H, Q, c, d), a[None], P[None], spu, zi, zs, zo,
                                          force_dyn=force_dyn)
    assert (info == 0).all() and (finfo == 0).all()
    assert np.array_equal(x, fx.transpose(1, 0, 2)) and np.array_equal(yy, fy.transpose(1, 0, 2))
    want = ofc.forecast_moments(y, a0, P0, T, Z, R, H, Q, c, d, horizon=hor)
    for k, v in want.items():
        assert np.abs(mom[k][0] - v).max() <= 1e-12 * (np.abs(v).max() + 1.0), k


# ---------------------------------------------------------------------------------------------------- host build
def _oracle_units(mats, mean, cov, cond, spu, zi, zs, zo, n_draws, n_series, n):
    hor = cond.shape[-2]
    m, p = mats["T"].shape[-1], mats["Z"].shape[-2]
    U = n_draws * n_series
    S = U * spu
    states, obs = np.empty((hor, S, m)), np.empty((hor, S, p))
    moms, infos = [], []
    for u in range(U):
        b = u // n_series
        sl = slice(u * spu, (u + 1) * spu)
        mb = {k: v[b] for k, v in mats.items()}
        cu = cond if cond.ndim == 2 else cond[u]
        args = (mean[u], cov[u], mb["T"], mb["Z"], mb["R"], mb["H"], mb["Q"], mb["c"], mb["d"], cu)
        mom, _, info = ocf.window(*args, n=n)
        xs, ys, _ = ocf.conditional_paths(*args, zi[sl], zs[:, sl], zo[:, sl], n=n)
        states[:, sl], obs[:, sl] = xs.transpose(1, 0, 2), ys.transpose(1, 0, 2)
        moms.append(mom)
        infos.append(info)
    return moms, states, obs, infos


def _random_cond(rng, U, hor, p, per_unit):
    cond = rng.normal(size=(U, hor, p) if per_unit else (hor, p))
    cond[rng.random(cond.shape) < 0.6] = np.nan
    return cond


@pytest.mark.parametrize("force_dyn", [False, True], ids=["instantiation", "runtime_dims"])
@pytest.mark.parametrize("geom", GEOMS, ids=[f"m{m}_p{p}_r{r}" for (m, p, r) in GEOMS])
def test_host_build_equals_oracle(geom, force_dyn):
    from tests import hostsim
    from tests.hostsim import condfc as hcf

    m, p, r = geom
    rng = np.random.default_rng(300 + 100 * m + 10 * p + r)
    nD, NS, spu, hor, n = 3, 2, 37, 6, 20
    mats = _batched_system(rng, m, p, r, nD)
    mean, cov = _starts(rng, nD * NS, m)
    zi, zs, zo = random_normals(rng, nD * NS * spu, hor, m, p, r)
    for per_unit in (False, True):
        cond = _random_cond(rng, nD * NS, hor, p, per_unit)
        moms, want_x, want_y, infos = _oracle_units(mats, mean, cov, cond, spu, zi, zs, zo, nD, NS, n)
        assert all(i == 0 for i in infos)
        mom, x, y, info, used_static = hcf.conditional_forecast(mats, mean, cov, cond, spu, zi, zs, zo, n=n,
                                                                n_draws=nD, n_series=NS, force_dyn=force_dyn)
        assert (info == 0).all()
        assert used_static == (not force_dyn and hostsim.simsmooth_is_static(m, p, r))
        assert np.abs(x - want_x).max() <= 1e-12 * (np.abs(want_x).max() + 1.0)
        assert np.abs(y - want_y).max() <= 1e-12 * (np.abs(want_y).max() + 1.0)
        for k in moms[0]:
            want = np.stack([mo[k] for mo in moms])
            assert np.abs(mom[k] - want).max() <= 1e-12 * (np.abs(want).max() + 1.0), k
        # either output alone, and moments only, give the same bits
        m1, x1, y1, _, _ = hcf.conditional_forecast(mats, mean, cov, cond, spu, zi, zs, zo, n, nD, NS, force_dyn,
                                                    want=("states",))
        _, x2, y2, _, _ = hcf.conditional_forecast(mats, mean, cov, cond, spu, zi, zs, zo, n, nD, NS, force_dyn,
                                                   want=("obs",))
        m3, x3, _, _, _ = hcf.conditional_forecast(mats, mean, cov, cond, 0, n=n, n_draws=nD, n_series=NS,
                                                   force_dyn=force_dyn)
        assert y1 is None and x2 is None and x3 is None
        assert np.array_equal(x1, x) and np.array_equal(y2, y)
        assert all(np.array_equal(m1[k], mom[k]) and np.array_equal(m3[k], mom[k]) for k in mom)


@pytest.mark.parametrize("force_dyn", [False, True], ids=["instantiation", "runtime_dims"])
def test_host_build_info_codes(force_dyn):
    from pymc_statespace_b200._lib import KFB_INFO_NOT_PSD
    from tests.hostsim import condfc as hcf

    rng = np.random.default_rng(8)
    nD, NS, spu, hor, m, p, r, n = 4, 2, 3, 5, 2, 2, 2, 50
    mats = _batched_system(rng, m, p, r, nD)
    mats["Q"][1] = -mats["Q"][1]  # draw 1: Q not PSD -> units 2, 3
    mats["Z"][2] = np.array([[1.0, 0.0], [1.0, 0.0]])  # draw 2: both series see x_0 alone ...
    mats["H"][2] = np.zeros((2, 2))  # ... without noise: conditioning both at h = 3 is singular
    mean, cov = _starts(rng, nD * NS, m)
    cov[6] = np.array([[1.0, 0.0], [0.0, -0.5]])  # unit 6: start covariance not PSD
    mean[7, 1] = np.nan  # unit 7: NaN start
    cond = np.full((nD * NS, hor, p), np.nan)
    cond[:, 1, 0] = 0.3
    cond[:, 3] = [0.4, 0.5]
    zi, zs, zo = random_normals(rng, nD * NS * spu, hor, m, p, r)
    mom, x, y, info, _ = hcf.conditional_forecast(mats, mean, cov, cond, spu, zi, zs, zo, n=n, n_draws=nD, n_series=NS,
                                                  force_dyn=force_dyn)
    want = [0, 0, KFB_INFO_NOT_PSD, KFB_INFO_NOT_PSD, n + 3 + 1, n + 3 + 1, KFB_INFO_NOT_PSD, KFB_INFO_NOT_PSD]
    assert list(info) == want
    good, bad = slice(0, 2 * spu), slice(2 * spu, None)
    assert np.isfinite(x[:, good]).all() and np.isfinite(y[:, good]).all()
    assert np.isnan(x[:, bad]).all() and np.isnan(y[:, bad]).all()
    for k, v in mom.items():
        assert np.isfinite(v[:2]).all() and np.isnan(v[2:]).all(), k
    _, _, _, infos = _oracle_units(mats, mean, cov, cond, spu, zi, zs, zo, nD, NS, n)
    assert infos == [0, 0, "not_psd", "not_psd", n + 4, n + 4, "not_psd", "not_psd"]


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
    for (nd, ns, m, p, r, hor, spu) in ((3, 2, 2, 1, 1, 5, 7), (1, 1, 13, 1, 3, 24, 64), (4, 1, 3, 2, 2, 1, 1),
                                        (2, 3, 32, 32, 32, 3, 5), (2, 1, 3, 3, 3, 8, 0)):
        d = _desc(nd, ns, 100, m, p, r)
        assert lib.kfb_conditional_forecast_workspace_bytes(ctypes.byref(d), hor, spu, ctypes.byref(nb)) == _lib.KFB_OK
        U = nd * ns
        S32 = (U * spu + 31) // 32 * 32
        want = (_round(8 * U * hor * (m * p + 2 * p * p + p + m + m * m)) + _round(8 * U * (2 * m * m + m * r + p * p + r * r))
                + _round(8 * U * (3 * m * m + 2 * m * p + 4 * p * p)) + _round(4 * U) + _round(8 * hor * S32 * p)
                + _round(8 * (hor - 1) * S32 * m))
        assert nb.value == want


def test_cabi_argument_validation():
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    nb = ctypes.c_size_t(0)
    d = _desc()
    fw = lib.kfb_conditional_forecast_workspace_bytes
    assert fw(ctypes.byref(d), 4, -1, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    assert fw(ctypes.byref(d), 0, 4, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    assert fw(None, 4, 4, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    assert fw(ctypes.byref(d), 4, 4, None) == _lib.KFB_ERR_INVALID_ARG
    for k in ("m", "p", "r", "n_draws", "n_series"):
        bad = _desc()
        setattr(bad, k, 0)
        assert fw(ctypes.byref(bad), 4, 4, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    neg = _desc(n=-1)
    assert fw(ctypes.byref(neg), 4, 4, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    ins = _lib.KfbInputs()
    fc = lib.kfb_conditional_forecast
    for k in ("T", "Z", "R", "H", "Q", "c", "d"):
        tv = _desc()
        setattr(tv, k + "_ts", 4)
        assert fw(ctypes.byref(tv), 4, 4, ctypes.byref(nb)) == _lib.KFB_ERR_UNSUPPORTED
        assert fc(ctypes.byref(tv), ctypes.byref(ins), None, None, 3, None, 0, 4, None, None, None, None, None, None,
                  None, None, None, None, None, 0, None) == _lib.KFB_ERR_UNSUPPORTED
    for k in ("m", "p", "r"):
        big = _desc(**{k: 33})
        assert fw(ctypes.byref(big), 4, 4, ctypes.byref(nb)) == _lib.KFB_ERR_UNSUPPORTED
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below is refused first
    full = _lib.KfbInputs(*([fake] * 8 + [None, None]))

    def call(ins_, mean=fake, cov=fake, hor=3, cond=fake, cbs=0, spu=4, zi=fake, zs=fake, zo=fake, xs=fake, ys=fake,
             info=fake, ws=None, nbytes=0):
        return fc(ctypes.byref(d), ins_ if ins_ is None else ctypes.byref(ins_), mean, cov, hor, cond, cbs, spu, zi, zs,
                  zo, None, None, None, None, xs, ys, info, ws, nbytes, None)

    assert call(None) == _lib.KFB_ERR_INVALID_ARG
    assert call(ins) == _lib.KFB_ERR_INVALID_ARG
    for kw in (dict(mean=None), dict(cov=None), dict(cond=None), dict(cbs=-1), dict(zi=None), dict(zs=None),
               dict(zo=None), dict(info=None), dict(xs=None, ys=None), dict(hor=0), dict(spu=-1)):
        assert call(full, **kw) == _lib.KFB_ERR_INVALID_ARG, kw
    # moments only: no normal or path pointer is needed
    assert call(full, spu=0, zi=None, zs=None, zo=None, xs=None, ys=None) == _lib.KFB_ERR_WORKSPACE
    assert call(full, zs=None, hor=1) == _lib.KFB_ERR_WORKSPACE  # H = 1 reads no z_state
    assert fw(ctypes.byref(d), 3, 4, ctypes.byref(nb)) == _lib.KFB_OK
    assert call(full) == _lib.KFB_ERR_WORKSPACE
    assert call(full, ws=fake, nbytes=nb.value - 1) == _lib.KFB_ERR_WORKSPACE
