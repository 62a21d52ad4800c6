"""Forecasts and impulse responses on the GPU (kfb_forecast_paths / kfb_impulse_response via simulation.forecast,
simulation.impulse_responses and KalmanLogp.forecast / impulse_responses) against the numpy restatement
(oracle/forecast.py) fed the same normals, and the paths' joint law against the dense law of the future."""
import numpy as np
import pytest
import torch

from oracle import forecast as ofc
from pymc_statespace_b200 import _lib
from tests.helpers import random_system
from tests.test_forecast_host import CASES, GEOMS, IDS, _batched_system, arma11, local_linear_trend
from tests.test_simulation_smoother_host import check_joint, random_normals, unit_basis

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x):
    return None if x is None else torch.as_tensor(np.asarray(x, dtype=np.float64), device=DEV)


def _np(d):
    return {k: v.cpu().numpy() for k, v in d.items()}


def _forecast(y, a0, P0, T, Z, R, H, Q, c, d, hor, spu=0, zi=None, zs=None, zo=None):
    from pymc_statespace_b200.simulation import forecast

    return _np(forecast(_t(y[..., 0] if y.ndim == 3 else y), _t(a0), _t(P0), _t(T), _t(Z), _t(R), _t(H), _t(Q), _t(c),
                        _t(d), horizon=hor, n_simulations=spu, z_init=_t(zi), z_state=_t(zs), z_obs=_t(zo)))


def _geom_case(m, p, r):
    rng = np.random.default_rng(40 + 9 * m + 3 * p + r)
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, r, 12)
    y[[2, 11]] = np.nan
    return y, a0, P0, T, Z, R, H, Q, rng.normal(size=(m, 1)), rng.normal(size=(p, 1))


@pytest.mark.parametrize("geom", GEOMS + [(7, 2, 3), (13, 1, 3)], ids=[f"m{m}_p{p}_r{r}" for (m, p, r) in
                                                                        GEOMS + [(7, 2, 3), (13, 1, 3)]])
def test_paths_equal_oracle_on_the_same_normals(geom):
    m, p, r = geom
    y, a0, P0, T, Z, R, H, Q, c, d = _geom_case(m, p, r)
    hor, S = 9, 37  # more than one warp, not a multiple of 32
    zi, zs, zo = random_normals(np.random.default_rng(3), S, hor, m, p, r)
    got = _forecast(y, a0, P0, T, Z, R, H, Q, c, d, hor, S, zi, zs, zo)
    mom = ofc.forecast_moments(y, a0, P0, T, Z, R, H, Q, c, d, horizon=hor)
    wx, wy, info = ofc.forecast_paths(mom["state_mean"][0], mom["state_cov"][0], T, Z, R, H, Q, c, d, zi, zs, zo)
    assert info == 0
    assert np.abs(got["state_paths"] - wx).max() <= 1e-10 * (np.abs(wx).max() + 1.0)
    assert np.abs(got["obs_paths"] - wy).max() <= 1e-10 * (np.abs(wy).max() + 1.0)
    for k in ("state_mean", "state_cov", "obs_mean", "obs_cov"):
        assert np.abs(got[k][0] - mom[k]).max() <= 1e-10 * (np.abs(mom[k]).max() + 1.0), k


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_joint_law_matches_dense_forecast_law(case):
    name, y, a0, P0, T, Z, R, H, Q, c, d, hor = case
    m, p, r = T.shape[0], Z.shape[0], R.shape[1]
    zi, zs, zo = unit_basis(hor, m, p, r)
    got = _forecast(y, a0, P0, T, Z, R, H, Q, c, d, hor, zi.shape[0], zi, zs, zo)
    xm, xc, ym, yc = ofc.dense_forecast_law(y, a0, P0, T, Z, R, H, Q, c, d, horizon=hor)
    check_joint(got["state_paths"], xm, xc, 1e-10)
    check_joint(got["obs_paths"], ym, yc, 1e-10)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_moments_equal_oracle_filter(case):
    name, y, a0, P0, T, Z, R, H, Q, c, d, hor = case
    got = _forecast(y, a0, P0, T, Z, R, H, Q, c, d, hor)
    assert "state_paths" not in got
    want = ofc.forecast_moments(y, a0, P0, T, Z, R, H, Q, c, d, horizon=hor)
    for k, v in want.items():
        assert np.abs(got[k][0] - v).max() <= 1e-10 * (np.abs(v).max() + 1.0), (name, k)


def test_batched_draws_series_and_simulations():
    """Per-draw matrices, n_series > 1 and several paths per unit: every unit equals the oracle on its normals."""
    from pymc_statespace_b200.simulation import forecast

    rng = np.random.default_rng(8)
    B, NS, spu, n, m, p, r, hor = 3, 2, 5, 15, 3, 2, 2, 8
    systems = [random_system(rng, m, p, r, n) for _ in range(B)]
    ys = np.stack([random_system(rng, m, p, r, n)[0][..., 0] for _ in range(NS)])
    ys[1, 4] = np.nan
    st = lambda i: np.stack([s[i] for s in systems])  # noqa: E731
    a0, P0, T, Z, R, H, Q = (st(i) for i in range(1, 8))
    c, d = rng.normal(size=(B, m)), rng.normal(size=(B, p))
    U, S = B * NS, B * NS * spu
    zi, zs, zo = random_normals(rng, S, hor, m, p, r)
    got = _np(forecast(_t(ys), _t(a0[..., 0]), _t(P0), _t(T), _t(Z), _t(R), _t(H), _t(Q), _t(c), _t(d), horizon=hor,
                       n_simulations=spu, z_init=_t(zi), z_state=_t(zs), z_obs=_t(zo)))
    assert got["state_mean"].shape == (U, hor, m) and got["obs_paths"].shape == (S, hor, p)
    for u in range(U):
        b, se = divmod(u, NS)
        sl = slice(u * spu, (u + 1) * spu)
        mom = ofc.forecast_moments(ys[se], a0[b], P0[b], T[b], Z[b], R[b], H[b], Q[b], c[b], d[b], horizon=hor)
        for k, v in mom.items():
            assert np.abs(got[k][u] - v).max() <= 1e-10 * (np.abs(v).max() + 1.0), (u, k)
        wx, wy, info = ofc.forecast_paths(mom["state_mean"][0], mom["state_cov"][0], T[b], Z[b], R[b], H[b], Q[b], c[b],
                                          d[b], zi[sl], zs[:, sl], zo[:, sl])
        assert info == 0
        assert np.abs(got["state_paths"][sl] - wx).max() <= 1e-10 * (np.abs(wx).max() + 1.0), u
        assert np.abs(got["obs_paths"][sl] - wy).max() <= 1e-10 * (np.abs(wy).max() + 1.0), u


def test_info_codes_nan_paths_and_one_output():
    from pymc_statespace_b200.engine import BatchedKalman
    from pymc_statespace_b200.simulation import _forecast, forecast

    rng = np.random.default_rng(9)
    B, n, m, p, r, spu, hor = 4, 10, 2, 2, 2, 3, 6
    systems = [random_system(rng, m, p, r, n) for _ in range(B)]
    y = systems[0][0][..., 0]
    st = lambda i: np.stack([s[i] for s in systems])  # noqa: E731
    a0, P0, T, Z, R, H, Q = (st(i) for i in range(1, 8))
    Q[2] = -Q[2]  # not PSD
    H[3] = -1000 * np.eye(2)  # F_0 not positive definite
    mats = {k: _t(v) for k, v in dict(a0=a0[..., 0], P0=P0, T=T, Z=Z, R=R, H=H, Q=Q).items()}
    kal = BatchedKalman("standard", n + hor, m, p, r, n_draws=B, strict_reference=False, device=DEV)
    res, finfo, pinfo = _forecast(kal, _t(y), mats, hor, spu, None, None, None, None)
    finfo, pinfo = finfo.cpu().numpy(), pinfo.cpu().numpy()
    # draw 2's negative Q also makes the forward fail at some step; its paths report the factor failure
    assert finfo[0] == 0 and finfo[1] == 0 and finfo[2] > 0 and finfo[3] == 1
    assert list(pinfo[:3]) == [0, 0, _lib.KFB_INFO_NOT_PSD]
    x = res["state_paths"].cpu().numpy().reshape(B, spu, hor, m)
    assert np.isfinite(x[:2]).all() and np.isnan(x[2]).all()
    with pytest.raises(RuntimeError):
        forecast(_t(y), *[mats[k] for k in ("a0", "P0", "T", "Z", "R", "H", "Q")], horizon=hor, n_simulations=2)


def test_two_runs_identical_bits():
    from pymc_statespace_b200.simulation import forecast

    y, a0, P0, T, Z, R, H, Q = local_linear_trend(n=200, n_missing_tail=2)
    args = [_t(v) for v in (y[..., 0], a0, P0, T, Z, R, H, Q)]
    g = torch.Generator(device=DEV)
    out = []
    for _ in range(2):
        g.manual_seed(5)
        out.append(forecast(*args, horizon=50, n_simulations=300, generator=g))
    for k in out[0]:
        assert torch.equal(out[0][k], out[1][k]), k


# ---------------------------------------------------------------------------------------------------- impulse responses
@pytest.mark.parametrize("geom", GEOMS + [(7, 2, 3)], ids=[f"m{m}_p{p}_r{r}" for (m, p, r) in GEOMS + [(7, 2, 3)]])
def test_impulse_responses_equal_oracle(geom):
    from pymc_statespace_b200.simulation import impulse_responses

    m, p, r = geom
    nD, hor = 3, 11
    mats = _batched_system(np.random.default_rng(m * 31 + p * 7 + r), m, p, r, nD)
    for shock in ("unit", "std", "cholesky"):
        x, y = impulse_responses(_t(mats["T"]), _t(mats["Z"]), _t(mats["R"]), _t(mats["Q"]), hor, shock)
        x, y = x.cpu().numpy(), y.cpu().numpy()
        for b in range(nD):
            wx, wy = ofc.impulse_responses(mats["T"][b], mats["Z"][b], mats["R"][b], mats["Q"][b], hor, shock)
            assert np.abs(x[b] - wx).max() <= 1e-13 * (np.abs(wx).max() + 1.0), (shock, b)
            assert np.abs(y[b] - wy).max() <= 1e-13 * (np.abs(wy).max() + 1.0), (shock, b)


def test_impulse_responses_closed_forms():
    from pymc_statespace_b200.simulation import impulse_responses

    phi, theta, hor = 0.7, -0.3, 20
    _, _, _, T, Z, R, _, Q = arma11(phi, theta)
    _, y = impulse_responses(_t(T), _t(Z), _t(R), _t(Q), hor, "unit")
    psi = np.array([1.0] + [(phi + theta) * phi ** (h - 1) for h in range(1, hor)])
    assert np.abs(y.cpu().numpy()[0, :, 0, 0] - psi).max() <= 1e-14
    A = np.array([[0.5, 0.1, 0.0], [-0.2, 0.3, 0.2], [0.1, 0.0, 0.4]])
    L = np.array([[1.0, 0.0, 0.0], [0.3, 0.8, 0.0], [-0.2, 0.1, 0.5]])
    for shock, S in (("unit", np.eye(3)), ("std", np.diag(np.sqrt(np.diag(L @ L.T)))), ("cholesky", L)):
        x, y = impulse_responses(_t(A), _t(np.eye(3)), _t(np.eye(3)), _t(L @ L.T), hor, shock)
        want = np.stack([np.linalg.matrix_power(A, h) @ S for h in range(hor)])
        assert np.abs(x.cpu().numpy()[0] - want).max() <= 1e-14 and np.abs(y.cpu().numpy()[0] - want).max() <= 1e-14
    one = torch.ones((1, 1), dtype=torch.float64, device=DEV)
    x, y = impulse_responses(one, one, one, one, hor, "unit")
    assert bool((x == 1.0).all()) and bool((y == 1.0).all())
    with pytest.raises(RuntimeError):
        impulse_responses(one, one, one, -one, hor, "cholesky")
    with pytest.raises(ValueError):
        impulse_responses(one, one, one, one, hor, "sideways")


# ---------------------------------------------------------------------------------------------------- theta level
def _workloads():
    from tests.test_gpu_simulation_smoother import _theta_workloads

    return _theta_workloads()


def _own_states(model, mats):
    m0 = model.k_states_model
    if model.spec.k_states == m0:
        return mats
    return {k: (v[..., :m0, :m0] if k in ("P0", "T") else v[..., :m0] if k in ("a0", "c", "Z") else
                v[..., :m0, :] if k == "R" else v) for k, v in mats.items()}


@pytest.mark.parametrize("name", ["arma11", "local_linear_trend", "varmax10_k2", "trend_seasonal12_padded",
                                  "varmax20_k3"])
def test_kalman_logp_forecast(name):
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import varmax20_workload

    if name == "varmax20_k3":
        spec, y, theta = varmax20_workload(6, 40)
    else:
        spec, y, theta = _workloads()[name]
    B, n = theta.shape[0], y.shape[0]
    theta = theta.copy()
    if name == "arma11":
        theta[B - 1, 3] = 1.3  # not stationary: no stationary P0
    model = KalmanLogp(spec, y, n_draws=B, filter_type="standard", device=DEV)
    th = torch.as_tensor(theta, device=DEV)
    m0, p, r = model.k_states_model, spec.k_endog, spec.k_posdef
    spu, hor = 3, 7
    S = B * spu
    g = torch.Generator(device=DEV)
    g.manual_seed(1)
    zi = torch.randn((S, m0), dtype=torch.float64, device=DEV, generator=g)
    zs = torch.randn((hor - 1, S, r), dtype=torch.float64, device=DEV, generator=g)
    zo = torch.randn((hor, S, p), dtype=torch.float64, device=DEV, generator=g)
    got = _np(model.forecast(th, hor, spu, z_init=zi, z_state=zs, z_obs=zo))
    assert got["state_mean"].shape == (B, hor, m0) and got["state_paths"].shape == (S, hor, m0)
    mats = {k: v.cpu().numpy() for k, v in _own_states(model, model.system_matrices(th)).items()}
    zi, zs, zo = zi.cpu().numpy(), zs.cpu().numpy(), zo.cpu().numpy()
    yy = np.asarray(y, dtype=np.float64).reshape(n, p)
    for b in range(B):
        mb = {k: (v[b] if v.ndim == (1 if k in ("a0", "c", "d") else 2) + 1 else v) for k, v in mats.items()}
        sl = slice(b * spu, (b + 1) * spu)
        if name == "arma11" and b == B - 1:
            assert got["info"][b] == _lib.KFB_INFO_NOT_STATIONARY
            assert all(np.isnan(got[k][b]).all() for k in ("state_mean", "state_cov", "obs_mean", "obs_cov"))
            assert np.isnan(got["state_paths"][sl]).all() and np.isnan(got["obs_paths"][sl]).all()
            continue
        assert got["info"][b] == 0, b
        mom = ofc.forecast_moments(yy, mb["a0"], mb["P0"], mb["T"], mb["Z"], mb["R"], mb["H"], mb["Q"], mb["c"],
                                   mb["d"], horizon=hor)
        for k, v in mom.items():
            assert np.abs(got[k][b] - v).max() <= 1e-9 * (np.abs(v).max() + 1.0), (name, b, k)
        wx, wy, info = ofc.forecast_paths(mom["state_mean"][0], mom["state_cov"][0], mb["T"], mb["Z"], mb["R"],
                                          mb["H"], mb["Q"], mb["c"], mb["d"], zi[sl], zs[:, sl], zo[:, sl])
        assert info == 0
        assert np.abs(got["state_paths"][sl] - wx).max() <= 1e-9 * (np.abs(wx).max() + 1.0), (name, b)
        assert np.abs(got["obs_paths"][sl] - wy).max() <= 1e-9 * (np.abs(wy).max() + 1.0), (name, b)
    # moments only, and draws generated inside
    mo = model.forecast(th, hor)
    assert "state_paths" not in mo and torch.equal(mo["info"].cpu(), torch.as_tensor(got["info"]))
    assert model.forecast(th, hor, 2)["obs_paths"].shape == (B * 2, hor, p)


def test_kalman_logp_impulse_responses_varmax_orthogonalised():
    from pymc_statespace_b200.logp import KalmanLogp

    spec, y, theta = _workloads()["varmax10_k2"]
    B = theta.shape[0]
    model = KalmanLogp(spec, y, n_draws=B, device=DEV)
    th = torch.as_tensor(theta, device=DEV)
    hor = 12
    out = {k: v.cpu().numpy() for k, v in model.impulse_responses(th, hor, "cholesky").items()}
    assert (out["info"] == 0).all()
    mats = {k: v.cpu().numpy() for k, v in model.system_matrices(th).items()}
    for b in range(B):
        mb = {k: (v[b] if v.ndim == 3 else v) for k, v in mats.items() if k in ("T", "Z", "R", "Q")}
        # VAR(1): T = A, R = I, Z = I: the orthogonalised responses are A^h chol(Q)
        L = np.linalg.cholesky(mb["Q"])
        want = np.stack([np.linalg.matrix_power(mb["T"], h) @ mb["R"] @ L for h in range(hor)])
        assert np.abs(out["states"][b] - want).max() <= 1e-13 * (np.abs(want).max() + 1.0)
        wx, wy = ofc.impulse_responses(mb["T"], mb["Z"], mb["R"], mb["Q"], hor, "cholesky")
        assert np.abs(out["obs"][b] - wy).max() <= 1e-13 * (np.abs(wy).max() + 1.0)
    spec, y, theta = _workloads()["trend_seasonal12_padded"]
    model = KalmanLogp(spec, y, n_draws=theta.shape[0], device=DEV)
    out = model.impulse_responses(torch.as_tensor(theta, device=DEV), 5, "std")
    assert out["states"].shape == (theta.shape[0], 5, 13, 3) and out["obs"].shape == (theta.shape[0], 5, 1, 3)
