"""The per-draw calls on data with partly observed rows, on the GPU: kfb_masked_filter for every instantiation and the
run-time dims against the host build of the same code, the simulation smoother with KFB_FLAG_PARTIAL_ROWS for batched
draws, series and simulations, bitwise reruns, and KalmanLogp.sample_states / forecast / conditional_forecast on a
VARMAX(1,0) with measurement error whose sample has scattered partly observed rows and a ragged last two rows."""
import numpy as np
import pytest
import torch

from oracle import condforecast as ocf
from oracle import forecast as ofc
from oracle import masked as oms
from pymc_statespace_b200._lib import KFB_FLAG_CORRECTED, KFB_FLAG_PARTIAL_ROWS
from tests.helpers import random_system
from tests.hostsim import draws, partial
from tests.test_gpu_conditional_forecast import _close, _np, _t, _varmax10_k3
from tests.test_partial_rows_host import ragged, system
from tests.test_simulation_smoother_host import random_normals

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N = 10
KEYS = ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")
GEOMS = [(m, p) for m in range(1, 5) for p in range(1, 4)] + [(6, 3), (7, 2)]


def _kalman(y, mats, n_draws=1, n_series=1):
    from pymc_statespace_b200.engine import BatchedKalman

    m, p, r = mats["T"].shape[-1], mats["Z"].shape[-2], mats["R"].shape[-1]
    return BatchedKalman("standard", y.shape[-2], m, p, r, n_draws=n_draws, n_series=n_series,
                         strict_reference=False, device=DEV)


@pytest.mark.parametrize("m,p", GEOMS, ids=[f"m{m}_p{p}" for m, p in GEOMS])
def test_masked_filter_equals_host_build(m, p):
    mats, y = system(m, p)
    y = y[..., 0]
    out = _kalman(y, mats).masked_filter(_t(y), *[_t(mats[k]) for k in KEYS])
    ps, pc, info, _ = partial.masked_filter(y, mats)
    assert int(out["info"][0]) == 0 and info[0] == 0
    _close(out["predicted_states"].cpu().numpy(), ps, 1e-12)
    _close(out["predicted_covs"].cpu().numpy(), pc, 1e-12)
    a, P, _ = oms.masked_filter(y, *[mats[k] for k in KEYS])
    _close(out["predicted_covs"][0].cpu().numpy(), P, 1e-10)


def test_masked_filter_info_and_nan_outputs():
    rng = np.random.default_rng(2)
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 2, 2, 1, N)
    Z[0] = 0.0
    H = np.diag([0.0, 1.0])
    y[:3, 0] = np.nan
    y[3, 1] = np.nan
    mats = dict(a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q, c=None, d=None)
    out = _kalman(y[..., 0], mats).masked_filter(_t(y[..., 0]), *[_t(mats[k]) for k in KEYS])
    assert int(out["info"][0]) == 4
    assert torch.isnan(out["predicted_states"]).all() and torch.isnan(out["predicted_covs"]).all()


def _smoother_case(nd=3, ns=2, m=3, p=3, spu=37, seed=4):
    rng = np.random.default_rng(seed)
    mats, _ = system(m, p)
    mats["T"] = np.stack([mats["T"] * s for s in np.linspace(0.5, 1.5, nd)])
    mats["H"] = np.stack([mats["H"] * s for s in np.linspace(1.0, 2.0, nd)])
    ys = np.stack([ragged(rng, rng.normal(size=(N, p, 1)), rows=rows)[..., 0]
                   for rows in ((0, 2, 7, N - 1), (1, 5, N - 2, N - 1))][:ns])
    S = nd * ns * spu
    return mats, ys, S, random_normals(np.random.default_rng(seed + 1), S, N, m, p, mats["R"].shape[1])


def test_simulation_smoother_batched_equals_host_build():
    from pymc_statespace_b200.simulation import simulation_smoother

    nd, ns, spu = 3, 2, 37
    mats, ys, S, (zi, zs, zo) = _smoother_case(nd, ns, spu=spu)
    got = simulation_smoother(_t(ys), *[_t(mats[k]) for k in KEYS], n_simulations=spu, z_init=_t(zi),
                              z_state=_t(zs), z_obs=_t(zo)).cpu().numpy()
    _, pc, info, _ = partial.masked_filter(ys, mats, n_draws=nd, n_series=ns)
    want, sinfo = partial.simsmooth(ys, mats, pc, spu, zi, zs, zo, n_draws=nd, n_series=ns,
                                    flags=KFB_FLAG_PARTIAL_ROWS | KFB_FLAG_CORRECTED)
    assert (info == 0).all() and (sinfo == 0).all() and np.isfinite(got).all()
    _close(got, want, 1e-10)


@pytest.mark.parametrize("m,p", [(2, 2), (4, 3), (6, 3)])
def test_simulation_smoother_instances_equal_host_build(m, p):
    from pymc_statespace_b200.simulation import simulation_smoother

    mats, y = system(m, p)
    y = y[..., 0]
    spu = 5
    zi, zs, zo = random_normals(np.random.default_rng(8), spu, N, m, p, mats["R"].shape[1])
    got = simulation_smoother(_t(y), *[_t(mats[k]) for k in KEYS], n_simulations=spu, z_init=_t(zi), z_state=_t(zs),
                              z_obs=_t(zo)).cpu().numpy()
    _, pc, _, _ = partial.masked_filter(y, mats)
    want, info = partial.simsmooth(y, mats, pc, spu, zi, zs, zo, flags=KFB_FLAG_PARTIAL_ROWS)
    assert info[0] == 0
    _close(got, want, 1e-10)


def test_two_runs_identical_bits():
    from pymc_statespace_b200.simulation import conditional_forecast, forecast, simulation_smoother

    mats, ys, S, (zi, zs, zo) = _smoother_case(3, 2, spu=37)
    args = [_t(mats[k]) for k in KEYS]
    a = [simulation_smoother(_t(ys), *args, n_simulations=37, z_init=_t(zi), z_state=_t(zs), z_obs=_t(zo))
         for _ in range(2)]
    assert torch.equal(a[0], a[1])
    f = [forecast(_t(ys), *args, horizon=4) for _ in range(2)]
    cond = np.full((4, 3), np.nan)
    cond[0, 1] = 0.3
    g = [conditional_forecast(_t(ys), *args, conditions=_t(cond)) for _ in range(2)]
    for x, y_ in (f, g):
        for k in x:
            assert torch.equal(x[k], y_[k]), k


# ---------------------------------------------------------------------------------------------------- theta level
def _ragged_varmax(B=6, n=40):
    spec, y, theta = _varmax10_k3(B, n, np.random.default_rng(2))
    rng = np.random.default_rng(12)
    for t in rng.choice(n - 2, 4, replace=False):  # scattered partly observed rows
        y[t, rng.integers(0, 3)] = np.nan
    y[n - 2, 2] = np.nan  # the ragged edge: series 2 one step behind, series 1 and 2 two steps
    y[n - 1, 1:] = np.nan
    return spec, y, theta


def _draw_mats(model, th, b):
    mats = {k: v.cpu().numpy() for k, v in model.system_matrices(th).items()}
    return {k: (v[b] if v.ndim == (1 if k in ("a0", "c", "d") else 2) + 1 else v) for k, v in mats.items()}


def test_kalman_logp_sample_states_forecast_conditional_forecast():
    from pymc_statespace_b200.logp import KalmanLogp

    spec, y, theta = _ragged_varmax()
    B, n, p = theta.shape[0], y.shape[0], 3
    model = KalmanLogp(spec, y, n_draws=B, filter_type="univariate", device=DEV)
    th = torch.as_tensor(theta, device=DEV)
    m, r, spu, hor = spec.k_states, spec.k_posdef, 4, 5
    S = B * spu
    gen = torch.Generator(device=DEV)
    gen.manual_seed(3)
    zi = torch.randn((S, m), dtype=torch.float64, device=DEV, generator=gen)
    zs = torch.randn((n - 1, S, r), dtype=torch.float64, device=DEV, generator=gen)
    zo = torch.randn((n, S, p), dtype=torch.float64, device=DEV, generator=gen)
    states = model.sample_states(th, spu, z_init=zi, z_state=zs, z_obs=zo).cpu().numpy()
    assert (model.sample_states_info == 0).all() and np.isfinite(states).all()
    fc = _np(model.forecast(th, hor))
    cond = np.full((hor, p), np.nan)
    cond[0, 0] = 0.2
    cond[2, 1:] = (-0.1, 0.4)
    cf = _np(model.conditional_forecast(th, _t(cond), 3))
    for res in (fc, cf):
        assert (res["info"] == 0).all()
        assert all(np.isfinite(v).all() for k, v in res.items() if k != "info")
    zi, zs, zo = zi.cpu().numpy(), zs.cpu().numpy(), zo.cpu().numpy()
    for b in (0, 3, B - 1):
        mb = _draw_mats(model, th, b)
        args = [mb[k] for k in KEYS]
        sl = slice(b * spu, (b + 1) * spu)
        _, pc, _ = oms.masked_filter(y, *args)
        want, info = partial.simsmooth(y, mb, pc[None], spu, zi[sl], zs[:, sl], zo[:, sl], flags=KFB_FLAG_PARTIAL_ROWS)
        assert info[0] == 0
        _close(states[sl], want, 1e-9, ("sample_states", b))
        mu, Sxx, muy, Syy = ofc.dense_forecast_law(y, *args, horizon=hor)
        _close(fc["state_mean"][b], mu, 1e-8, ("forecast", b))
        _close(fc["obs_cov"][b], np.stack([Syy[h * p:(h + 1) * p, h * p:(h + 1) * p] for h in range(hor)]), 1e-8)
        mean, _ = ocf.dense_conditional_forecast_law(y, *args, cond=cond)
        _close(cf["state_mean"][b].reshape(-1), mean[:hor * m], 1e-8, ("conditional_forecast", b))
        _close(cf["obs_mean"][b].reshape(-1), mean[hor * m:], 1e-8, ("conditional_forecast", b))
