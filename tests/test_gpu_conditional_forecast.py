"""Conditional forecasts on the GPU (kfb_conditional_forecast via simulation.conditional_forecast and
KalmanLogp.conditional_forecast) against the numpy restatement (oracle/condforecast.py) fed the same normals, against
the unconditional forecast paths, and against the simulation smoother run on the sample extended by the conditions."""
import numpy as np
import pytest
import torch

from oracle import condforecast as ocf
from oracle import forecast as ofc
from pymc_statespace_b200 import _lib
from tests.helpers import random_system
from tests.test_conditional_forecast_host import CASES, IDS, joint
from tests.test_forecast_host import GEOMS
from tests.test_simulation_smoother_host import check_joint, random_normals, unit_basis

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x):
    return None if x is None else torch.as_tensor(np.asarray(x, dtype=np.float64), device=DEV)


def _np(d):
    return {k: v.cpu().numpy() for k, v in d.items()}


def _condfc(y, a0, P0, T, Z, R, H, Q, c, d, cond, spu=0, zi=None, zs=None, zo=None):
    from pymc_statespace_b200.simulation import conditional_forecast

    return _np(conditional_forecast(_t(y[..., 0] if y.ndim == 3 else y), _t(a0), _t(P0), _t(T), _t(Z), _t(R), _t(H),
                                    _t(Q), _t(c), _t(d), conditions=_t(cond), n_simulations=spu, z_init=_t(zi),
                                    z_state=_t(zs), z_obs=_t(zo)))


def _start(y, a0, P0, T, Z, R, H, Q, c, d):
    mom = ofc.forecast_moments(y, a0, P0, T, Z, R, H, Q, c, d, horizon=1)
    return mom["state_mean"][0], mom["state_cov"][0]


def _close(got, want, tol, what=None):
    assert np.abs(got - want).max() <= tol * (np.abs(want).max() + 1.0), what


GEOMS_GPU = GEOMS + [(6, 3, 3), (7, 2, 3), (13, 1, 3)]


@pytest.mark.parametrize("geom", GEOMS_GPU, ids=[f"m{m}_p{p}_r{r}" for (m, p, r) in GEOMS_GPU])
def test_equals_oracle_on_the_same_normals(geom):
    m, p, r = geom
    rng = np.random.default_rng(70 + 9 * m + 3 * p + r)
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, r, 12)
    y[[2, 11]] = np.nan
    c, d = rng.normal(size=m), rng.normal(size=p)
    hor, S = 9, 37  # more than one warp, not a multiple of 32
    cond = rng.normal(size=(hor, p))
    cond[rng.random(cond.shape) < 0.6] = np.nan
    zi, zs, zo = random_normals(np.random.default_rng(3), S, hor, m, p, r)
    got = _condfc(y, a0, P0, T, Z, R, H, Q, c, d, cond, S, zi, zs, zo)
    a, P = _start(y, a0, P0, T, Z, R, H, Q, c, d)
    mom, _, info = ocf.window(a, P, T, Z, R, H, Q, c, d, cond, n=len(y))
    wx, wy, _ = ocf.conditional_paths(a, P, T, Z, R, H, Q, c, d, cond, zi, zs, zo, n=len(y))
    assert info == 0
    _close(got["state_paths"], wx, 1e-10)
    _close(got["obs_paths"], wy, 1e-10)
    o = ~np.isnan(cond)
    assert (got["obs_paths"][:, o] == cond[o]).all()
    for k, v in mom.items():
        _close(got[k][0], v, 1e-10, k)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_joint_law_matches_dense_conditional_law(case):
    name, y, a0, P0, T, Z, R, H, Q, c, d, cond = case
    m, p, r, hor = T.shape[0], Z.shape[0], R.shape[1], cond.shape[0]
    zi, zs, zo = unit_basis(hor, m, p, r)
    got = _condfc(y, a0, P0, T, Z, R, H, Q, c, d, cond, zi.shape[0], zi, zs, zo)
    mean, cov = ocf.dense_conditional_forecast_law(y, a0, P0, T, Z, R, H, Q, c, d, cond)
    check_joint(joint(got["state_paths"], got["obs_paths"]), mean, cov, 1e-10)


@pytest.mark.parametrize("per_unit", [False, True], ids=["shared_conditions", "per_unit_conditions"])
def test_batched_draws_series_and_simulations(per_unit):
    from pymc_statespace_b200.simulation import conditional_forecast

    rng = np.random.default_rng(8)
    B, NS, spu, n, m, p, r, hor = 3, 2, 5, 15, 3, 2, 2, 8
    systems = [random_system(rng, m, p, r, n) for _ in range(B)]
    ys = np.stack([random_system(rng, m, p, r, n)[0][..., 0] for _ in range(NS)])
    ys[1, 4] = np.nan
    st = lambda i: np.stack([s[i] for s in systems])  # noqa: E731
    a0, P0, T, Z, R, H, Q = (st(i) for i in range(1, 8))
    c, d = rng.normal(size=(B, m)), rng.normal(size=(B, p))
    U, S = B * NS, B * NS * spu
    cond = rng.normal(size=(U, hor, p) if per_unit else (hor, p))
    cond[rng.random(cond.shape) < 0.5] = np.nan
    zi, zs, zo = random_normals(rng, S, hor, m, p, r)
    got = _np(conditional_forecast(_t(ys), _t(a0[..., 0]), _t(P0), _t(T), _t(Z), _t(R), _t(H), _t(Q), _t(c), _t(d),
                                   conditions=_t(cond), n_simulations=spu, z_init=_t(zi), z_state=_t(zs),
                                   z_obs=_t(zo)))
    assert got["state_mean"].shape == (U, hor, m) and got["obs_paths"].shape == (S, hor, p)
    for u in range(U):
        b, se = divmod(u, NS)
        sl = slice(u * spu, (u + 1) * spu)
        a, P = _start(ys[se], a0[b], P0[b], T[b], Z[b], R[b], H[b], Q[b], c[b], d[b])
        args = (a, P, T[b], Z[b], R[b], H[b], Q[b], c[b], d[b], cond[u] if per_unit else cond)
        mom, _, info = ocf.window(*args, n=n)
        wx, wy, _ = ocf.conditional_paths(*args, zi[sl], zs[:, sl], zo[:, sl], n=n)
        assert info == 0
        for k, v in mom.items():
            _close(got[k][u], v, 1e-10, (u, k))
        _close(got["state_paths"][sl], wx, 1e-10, u)
        _close(got["obs_paths"][sl], wy, 1e-10, u)


def test_all_nan_conditions_give_the_forecast_paths():
    """No condition: r = 0 throughout and the paths are kfb_forecast_paths' on the same normals, bit for bit (the same
    KFB_HD functions in the same order, and x+ + 0 = x+).  The moments come from another recursion (the window filter
    instead of the filter over n + H rows) and agree to rounding."""
    from pymc_statespace_b200.simulation import conditional_forecast, forecast

    for (m, p, r) in ((2, 1, 1), (3, 3, 2), (7, 2, 3)):
        rng = np.random.default_rng(m + p + r)
        y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, r, 30)
        args = [_t(v) for v in (y[..., 0], a0, P0, T, Z, R, H, Q)]
        hor, S = 11, 300
        zi, zs, zo = (_t(z) for z in random_normals(rng, S, hor, m, p, r))
        cond = torch.full((hor, p), float("nan"), dtype=torch.float64, device=DEV)
        got = conditional_forecast(*args, conditions=cond, n_simulations=S, z_init=zi, z_state=zs, z_obs=zo)
        want = forecast(*args, horizon=hor, n_simulations=S, z_init=zi, z_state=zs, z_obs=zo)
        assert set(got) == set(want)
        assert torch.equal(got["state_paths"], want["state_paths"]), (m, p, r)
        assert torch.equal(got["obs_paths"], want["obs_paths"]), (m, p, r)
        for k in ("state_mean", "state_cov", "obs_mean", "obs_cov"):
            _close(got[k].cpu().numpy(), want[k].cpu().numpy(), 1e-12, k)


def _law(paths):
    """Mean and covariance of the affine map from unit-basis normals to paths [1 + N, ...] (flattened per path)."""
    x0 = paths[0].reshape(-1)
    M = paths[1:].reshape(paths.shape[0] - 1, -1) - x0
    return x0, M.T @ M


def test_fully_conditioned_rows_match_the_simulation_smoother():
    """Every entry of the window conditioned: the states' joint law is the simulation smoother's on [y; cond] over
    its last H time steps."""
    from pymc_statespace_b200.simulation import simulation_smoother

    rng = np.random.default_rng(31)
    m, p, r, n, hor = 3, 2, 2, 10, 4
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, r, n)
    c, d = rng.normal(size=m), rng.normal(size=p)
    cond = rng.normal(size=(hor, p))
    zi, zs, zo = unit_basis(hor, m, p, r)
    got = _condfc(y, a0, P0, T, Z, R, H, Q, c, d, cond, zi.shape[0], zi, zs, zo)
    mean, cov = _law(got["state_paths"])
    yx = np.concatenate([y[..., 0], cond])
    N = n + hor
    bi, bs, bo = unit_basis(N, m, p, r)
    ss = simulation_smoother(_t(yx), _t(a0), _t(P0), _t(T), _t(Z), _t(R), _t(H), _t(Q), _t(c), _t(d),
                             n_simulations=bi.shape[0], z_init=_t(bi), z_state=_t(bs), z_obs=_t(bo)).cpu().numpy()
    smean, scov = _law(ss)
    k = slice(n * m, N * m)
    _close(mean, smean[k], 1e-10)
    assert np.abs(cov - scov[k, k]).max() <= 1e-10 * max(np.abs(scov[k, k]).max(), 1.0)
    _close(got["state_mean"][0].reshape(-1), smean[k], 1e-10)


def test_info_codes_and_nan_outputs():
    from pymc_statespace_b200.engine import BatchedKalman
    from pymc_statespace_b200.simulation import _conditional_forecast, conditional_forecast

    rng = np.random.default_rng(9)
    B, n, m, p, r, spu, hor = 4, 10, 2, 2, 2, 3, 6
    systems = [random_system(rng, m, p, r, n) for _ in range(B)]
    y = systems[0][0][..., 0].copy()
    y[1:] = np.nan  # only row 0 observed
    st = lambda i: np.stack([s[i] for s in systems])  # noqa: E731
    a0, P0, T, Z, R, H, Q = (st(i) for i in range(1, 8))
    Q[1] = -Q[1]  # not PSD
    # draw 2: state 1 is 0 after the first step (row 1 of T and R zero), so P_n has an exactly zero row and column 1,
    # and series 1 observes it without noise: conditioning series 1 at h = 2 gives F_11 = 0 exactly
    T[2], Z[2], R[2], H[2] = np.diag([0.5, 0.0]), np.eye(2), np.diag([1.0, 0.0]), np.diag([0.3, 0.0])
    H[3] = -1000 * np.eye(2)  # F_0 not positive definite in the sample
    cond = np.full((hor, p), np.nan)
    cond[2] = [0.1, 0.2]
    mats = {k: _t(v) for k, v in dict(a0=a0[..., 0], P0=P0, T=T, Z=Z, R=R, H=H, Q=Q).items()}
    kal = BatchedKalman("standard", n, m, p, r, n_draws=B, strict_reference=False, device=DEV)
    res, finfo, winfo = _conditional_forecast(kal, _t(y), mats, _t(cond), spu, None, None, None, None)
    finfo, winfo = finfo.cpu().numpy(), winfo.cpu().numpy()
    assert finfo[0] == 0 and finfo[2] == 0 and finfo[3] == 1
    assert winfo[0] == 0 and winfo[1] == _lib.KFB_INFO_NOT_PSD and winfo[2] == n + 2 + 1
    x = res["state_paths"].cpu().numpy().reshape(B, spu, hor, m)
    assert np.isfinite(x[0]).all() and np.isnan(x[1:3]).all()
    for k in ("state_mean", "state_cov", "obs_mean", "obs_cov"):
        v = res[k].cpu().numpy()
        assert np.isfinite(v[0]).all() and np.isnan(v[1:3]).all(), k
    with pytest.raises(RuntimeError):
        conditional_forecast(_t(y), *[mats[k] for k in ("a0", "P0", "T", "Z", "R", "H", "Q")], conditions=_t(cond),
                             n_simulations=2)
    with pytest.raises(ValueError):
        conditional_forecast(_t(y), *[mats[k] for k in ("a0", "P0", "T", "Z", "R", "H", "Q")],
                             conditions=_t(np.zeros((hor, p + 1))))


def test_two_runs_identical_bits():
    from pymc_statespace_b200.simulation import conditional_forecast

    rng = np.random.default_rng(4)
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 3, 2, 2, 200)
    args = [_t(v) for v in (y[..., 0], a0, P0, T, Z, R, H, Q)]
    cond = rng.normal(size=(50, 2))
    cond[rng.random(cond.shape) < 0.7] = np.nan
    g = torch.Generator(device=DEV)
    out = []
    for _ in range(2):
        g.manual_seed(5)
        out.append(conditional_forecast(*args, conditions=_t(cond), n_simulations=300, generator=g))
    for k in out[0]:
        assert torch.equal(out[0][k], out[1][k]), k


# ---------------------------------------------------------------------------------------------------- theta level
def _varmax10_k3(B, n, rng):
    from pymc_statespace_b200.models import varmax_spec

    k = 3
    spec = varmax_spec(k, (1, 0), stationary_initialization=True, measurement_error=True)
    L = np.tril(rng.normal(0.0, 0.1, (B, k, k)), -1) + np.eye(k) * 0.5
    theta = np.concatenate([rng.normal(0, 0.1, (B, k)), rng.uniform(-0.3, 0.3, (B, k * k)),
                            (L @ L.transpose(0, 2, 1)).reshape(B, -1), np.exp(rng.normal(-1.0, 0.2, (B, k)))], axis=1)
    y = rng.normal(size=(n, k))
    y[[3, 17]] = np.nan
    return spec, y, theta


def _own_states(model, mats):
    m0 = model.k_states_model
    if model.spec.k_states == m0:
        return mats
    return {k: (v[..., :m0, :m0] if k in ("P0", "T") else v[..., :m0] if k in ("a0", "c", "Z") else
                v[..., :m0, :] if k == "R" else v) for k, v in mats.items()}


@pytest.mark.parametrize("name", ["arma11", "varmax10_k3", "varmax20_k3", "trend_seasonal12_padded"])
def test_kalman_logp_conditional_forecast(name):
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import varmax20_workload
    from tests.test_gpu_simulation_smoother import _theta_workloads

    if name == "varmax20_k3":
        spec, y, theta = varmax20_workload(6, 40)
    elif name == "varmax10_k3":
        spec, y, theta = _varmax10_k3(6, 40, np.random.default_rng(2))
    else:
        spec, y, theta = _theta_workloads()[name]
    B, n = theta.shape[0], y.shape[0]
    theta = theta.copy()
    if name == "arma11":
        theta[B - 1, 3] = 1.3  # not stationary: no stationary P0
    model = KalmanLogp(spec, y, n_draws=B, filter_type="standard", device=DEV)
    th = torch.as_tensor(theta, device=DEV)
    m0, p, r = model.k_states_model, spec.k_endog, spec.k_posdef
    spu, hor = 3, 7
    S = B * spu
    cond = np.full((hor, p), np.nan)
    cond[:4, 0] = np.linspace(-0.5, 0.5, 4)  # series 0 conditioned over the first four steps
    g = torch.Generator(device=DEV)
    g.manual_seed(1)
    zi = torch.randn((S, m0), dtype=torch.float64, device=DEV, generator=g)
    zs = torch.randn((hor - 1, S, r), dtype=torch.float64, device=DEV, generator=g)
    zo = torch.randn((hor, S, p), dtype=torch.float64, device=DEV, generator=g)
    got = _np(model.conditional_forecast(th, _t(cond), spu, z_init=zi, z_state=zs, z_obs=zo))
    assert got["state_mean"].shape == (B, hor, m0) and got["state_paths"].shape == (S, hor, m0)
    mats = {k: v.cpu().numpy() for k, v in _own_states(model, model.system_matrices(th)).items()}
    zi, zs, zo = zi.cpu().numpy(), zs.cpu().numpy(), zo.cpu().numpy()
    yy = np.asarray(y, dtype=np.float64).reshape(n, p)
    o = ~np.isnan(cond)
    for b in range(B):
        mb = {k: (v[b] if v.ndim == (1 if k in ("a0", "c", "d") else 2) + 1 else v) for k, v in mats.items()}
        sl = slice(b * spu, (b + 1) * spu)
        if name == "arma11" and b == B - 1:
            assert got["info"][b] == _lib.KFB_INFO_NOT_STATIONARY
            assert all(np.isnan(got[k][b]).all() for k in ("state_mean", "state_cov", "obs_mean", "obs_cov"))
            assert np.isnan(got["state_paths"][sl]).all() and np.isnan(got["obs_paths"][sl]).all()
            continue
        assert got["info"][b] == 0, b
        a, P = _start(yy, mb["a0"], mb["P0"], mb["T"], mb["Z"], mb["R"], mb["H"], mb["Q"], mb["c"], mb["d"])
        args = (a, P, mb["T"], mb["Z"], mb["R"], mb["H"], mb["Q"], mb["c"], mb["d"], cond)
        mom, _, info = ocf.window(*args, n=n)
        wx, wy, _ = ocf.conditional_paths(*args, zi[sl], zs[:, sl], zo[:, sl], n=n)
        assert info == 0
        for k, v in mom.items():
            _close(got[k][b], v, 1e-9, (name, b, k))
        _close(got["state_paths"][sl], wx, 1e-9, (name, b))
        _close(got["obs_paths"][sl], wy, 1e-9, (name, b))
        assert (got["obs_paths"][sl][:, o] == cond[o]).all()
    # moments only, per-draw conditions, and draws generated inside
    mo = model.conditional_forecast(th, _t(cond))
    assert "state_paths" not in mo and torch.equal(mo["info"].cpu(), torch.as_tensor(got["info"]))
    per = model.conditional_forecast(th, _t(np.broadcast_to(cond, (B, hor, p)).copy()))
    for k in ("state_mean", "obs_mean"):
        assert torch.equal(torch.nan_to_num(per[k]), torch.nan_to_num(mo[k])), k
    assert model.conditional_forecast(th, _t(cond), 2)["obs_paths"].shape == (B * 2, hor, p)
