"""The simulation smoother on the GPU (kfb_simulation_smoother via simulation.simulation_smoother and
KalmanLogp.sample_states) against the numpy restatement (oracle/simsmooth.py) fed the same normals, and its joint law
against the dense posterior."""
import numpy as np
import pytest
import torch

from oracle import simsmooth as oss
from pymc_statespace_b200 import _lib
from tests.helpers import nile_inputs, random_system
from tests.test_simulation_smoother_host import CASES, IDS, check_joint, random_normals, unit_basis

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x):
    return None if x is None else torch.as_tensor(np.asarray(x, dtype=np.float64), device=DEV)


def _run(y, a0, P0, T, Z, R, H, Q, c, d, zi, zs, zo, spu):
    from pymc_statespace_b200.simulation import simulation_smoother

    out = simulation_smoother(_t(y[..., 0]), _t(a0), _t(P0), _t(T), _t(Z), _t(R), _t(H), _t(Q), _t(c), _t(d),
                              n_simulations=spu, z_init=_t(zi), z_state=_t(zs), z_obs=_t(zo))
    return out.cpu().numpy()


def _extra_cases():
    """Geometries of the run-time-dims path (k_states > 4, k_endog > 3, k_posdef > k_states) and the Nile fixture."""
    rng = np.random.default_rng(21)
    out = []
    for (m, p, r) in ((5, 1, 2), (3, 4, 2), (2, 1, 3), (7, 2, 3)):
        y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, r, 12)
        y[[0, 11]] = np.nan
        out.append((f"runtime_m{m}_p{p}_r{r}", y, a0, P0, T, Z, R, H, Q, None, None, 1e-10))
    y, a0, P0, T, Z, R, H, Q = nile_inputs(n_missing=5)
    out.append(("nile", y, a0, P0, T, Z, R, H, Q, None, None, 1e-7))
    return out


ALL = CASES + _extra_cases()


@pytest.mark.parametrize("case", ALL, ids=[c[0] for c in ALL])
def test_equals_oracle_on_the_same_normals(case):
    name, y, a0, P0, T, Z, R, H, Q, c, d, rtol = case
    n, p, m, r = y.shape[0], Z.shape[0], T.shape[0], R.shape[1]
    S = 37  # more than one warp, not a multiple of 32
    zi, zs, zo = random_normals(np.random.default_rng(3), S, n, m, p, r)
    got = _run(y, a0, P0, T, Z, R, H, Q, c, d, zi, zs, zo, S)
    want, info = oss.simulation_smoother(y, a0, P0, T, Z, R, H, Q, c, d, zi, zs, zo)
    assert info == 0
    assert np.abs(got - want).max() <= rtol * (np.abs(want).max() + 1.0), name


@pytest.mark.parametrize("name", ["random_m2_p1_r2", "random_m4_p3_r4", "arma11_theta0_singular_P0", "n1",
                                  "runtime_m5_p1_r2"])
def test_joint_law_matches_dense_posterior(name):
    case = ALL[[c[0] for c in ALL].index(name)]
    _, y, a0, P0, T, Z, R, H, Q, c, d, _ = case
    n, p, m, r = y.shape[0], Z.shape[0], T.shape[0], R.shape[1]
    zi, zs, zo = unit_basis(n, m, p, r)
    paths = _run(y, a0, P0, T, Z, R, H, Q, c, d, zi, zs, zo, zi.shape[0])
    mean, cov = oss.dense_state_posterior(y, a0, P0, T, Z, R, H, Q, c, d)
    check_joint(paths, mean, cov, 1e-10)


def test_batched_draws_series_and_simulations():
    """Per-draw matrices, n_series > 1 and sims_per_unit > 1: every unit equals the oracle on its slice of normals."""
    from pymc_statespace_b200.simulation import simulation_smoother

    rng = np.random.default_rng(8)
    B, NS, spu, n, m, p, r = 3, 2, 5, 20, 3, 2, 2
    systems = [random_system(rng, m, p, r, n) for _ in range(B)]
    ys = np.stack([random_system(rng, m, p, r, n)[0][..., 0] for _ in range(NS)])
    ys[1, 4] = np.nan
    st = lambda i: np.stack([s[i] for s in systems])  # noqa: E731
    a0, P0, T, Z, R, H, Q = (st(i) for i in range(1, 8))
    c = rng.normal(size=(B, m))
    U, S = B * NS, B * NS * spu
    zi, zs, zo = random_normals(rng, S, n, m, p, r)
    got = simulation_smoother(_t(ys), _t(a0[..., 0]), _t(P0), _t(T), _t(Z), _t(R), _t(H), _t(Q), _t(c),
                              n_simulations=spu, z_init=_t(zi), z_state=_t(zs), z_obs=_t(zo)).cpu().numpy()
    for u in range(U):
        b, se = divmod(u, NS)
        sl = slice(u * spu, (u + 1) * spu)
        want, info = oss.simulation_smoother(ys[se][..., None], a0[b], P0[b], T[b], Z[b], R[b], H[b], Q[b], c[b], None,
                                             zi[sl], zs[:, sl], zo[:, sl])
        assert info == 0
        assert np.abs(got[sl] - want).max() <= 1e-10 * (np.abs(want).max() + 1.0), u


def test_info_codes_and_nan_paths():
    from pymc_statespace_b200.engine import BatchedKalman
    from pymc_statespace_b200.simulation import _simulation_smoother, simulation_smoother

    rng = np.random.default_rng(9)
    B, n, m, p, r, spu = 4, 10, 2, 2, 2, 3
    systems = [random_system(rng, m, p, r, n) for _ in range(B)]
    y = systems[0][0][..., 0]
    st = lambda i: np.stack([s[i] for s in systems])  # noqa: E731
    a0, P0, T, Z, R, H, Q = (st(i) for i in range(1, 8))
    Z[1] = 0.0
    H[1] = 0.0  # F_0 = 0: not positive definite at t = 0
    Q[2] = -Q[2]  # not PSD
    mats = {k: _t(v) for k, v in dict(a0=a0[..., 0], P0=P0, T=T, Z=Z, R=R, H=H, Q=Q).items()}
    kal = BatchedKalman("standard", n, m, p, r, n_draws=B, strict_reference=False, device=DEV)
    states, info = _simulation_smoother(kal, _t(y), mats, spu, None, None, None, None)
    states, info = states.cpu().numpy().reshape(B, spu, n, m), info.cpu().numpy()
    assert list(info) == [0, 1, _lib.KFB_INFO_NOT_PSD, 0]
    assert np.isfinite(states[[0, 3]]).all() and np.isnan(states[[1, 2]]).all()
    yp = y.copy()
    yp[6, 0] = np.nan  # partly missing row 6
    states, info = _simulation_smoother(kal, _t(yp), mats, spu, None, None, None, None)
    assert list(info.cpu().numpy()) == [-7, 1, _lib.KFB_INFO_NOT_PSD, -7]
    assert torch.isnan(states).all()
    with pytest.raises(RuntimeError):
        simulation_smoother(_t(y), *[mats[k] for k in ("a0", "P0", "T", "Z", "R", "H", "Q")])


def test_two_runs_identical_bits():
    from pymc_statespace_b200.simulation import simulation_smoother

    y, a0, P0, T, Z, R, H, Q = nile_inputs(n_missing=3)
    args = [_t(v) for v in (y[..., 0], a0, P0, T, Z, R, H, Q)]
    g = torch.Generator(device=DEV)
    g.manual_seed(5)
    x1 = simulation_smoother(*args, n_simulations=100, generator=g)
    g.manual_seed(5)
    x2 = simulation_smoother(*args, n_simulations=100, generator=g)
    assert torch.equal(x1, x2)


def test_time_varying_is_not_implemented():
    from pymc_statespace_b200.simulation import simulation_smoother

    y, a0, P0, T, Z, R, H, Q = nile_inputs()
    args = [_t(v) for v in (y[..., 0], a0, P0, T, Z, R, H, Q)]
    args[3] = args[3].expand(3, y.shape[0], 2, 2)
    with pytest.raises(NotImplementedError):
        simulation_smoother(*args)


# ---------------------------------------------------------------------------------------------------- theta level
def _varmax10(B, n, rng):
    from pymc_statespace_b200.models import varmax_spec

    spec = varmax_spec(2, (1, 0), stationary_initialization=True, measurement_error=True)
    theta = np.concatenate([rng.normal(0, 0.1, (B, 2)), rng.uniform(-0.4, 0.4, (B, 4)),
                            np.tile([0.5, 0.1, 0.1, 0.4], (B, 1)), np.exp(rng.normal(-1.0, 0.2, (B, 2)))], axis=1)
    y = rng.normal(size=(n, 2))
    y[[3, 17]] = np.nan
    return spec, y, theta


def _theta_workloads():
    from pymc_statespace_b200.models import local_level_spec
    from pymc_statespace_b200.synthetic import arma11_workload, trend_seasonal_workload

    rng = np.random.default_rng(12)
    B, n = 8, 60
    out = {"arma11": arma11_workload(B, n)}
    llt = local_level_spec()
    th = np.tile([0.0, 0.0, 1.0, 0.0, 0.0, 1.0, 0.8, 0.5, 0.01], (B, 1))
    th[:, 6:] *= np.exp(rng.normal(0, 0.2, (B, 3)))
    out["local_linear_trend"] = (llt, np.cumsum(rng.normal(size=n))[:, None], th)
    out["varmax10_k2"] = _varmax10(B, n, rng)
    spec, y, theta = trend_seasonal_workload(B, n, period=12)  # 13 states: embedded in 14 (padded spec)
    out["trend_seasonal12_padded"] = (spec, y, theta)
    return out


@pytest.mark.parametrize("name", ["arma11", "local_linear_trend", "varmax10_k2", "trend_seasonal12_padded"])
def test_sample_states_theta_level(name):
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.simulation import simulation_smoother

    spec, y, theta = _theta_workloads()[name]
    B, n = theta.shape[0], y.shape[0]
    model = KalmanLogp(spec, y, n_draws=B, filter_type="standard", device=DEV)
    th = torch.as_tensor(theta, device=DEV)
    m0, p, r = model.k_states_model, spec.k_endog, spec.k_posdef
    spu = 3
    S = B * spu
    zeros = [torch.zeros(s, dtype=torch.float64, device=DEV) for s in ((S, m0), (n - 1, S, r), (n, S, p))]
    x0 = model.sample_states(th, spu, z_init=zeros[0], z_state=zeros[1], z_obs=zeros[2])
    assert int((model.sample_states_info != 0).sum()) == 0
    ss, _, _ = model.smooth(th)
    mean = x0.view(B, spu, n, m0)
    for k in range(spu):
        err = (mean[:, k] - ss[..., 0] if ss.ndim == 4 else mean[:, k] - ss).abs().max().item()
        # smooth() is the reference RTS smoother (pseudo-inverse gain; with H = 0 its predicted covariances are singular)
        assert err <= 1e-6 * (ss.abs().max().item() + 1.0), (name, err)
    g = torch.Generator(device=DEV)
    g.manual_seed(1)
    zi = torch.randn((S, m0), dtype=torch.float64, device=DEV, generator=g)
    zs = torch.randn((n - 1, S, r), dtype=torch.float64, device=DEV, generator=g)
    zo = torch.randn((n, S, p), dtype=torch.float64, device=DEV, generator=g)
    got = model.sample_states(th, spu, z_init=zi, z_state=zs, z_obs=zo)
    mats = model.system_matrices(th)
    if model.spec.k_states != m0:  # the matrix-level call on the model's own states
        mats = {k: (v[..., :m0, :m0] if k in ("P0", "T") else v[..., :m0] if k in ("a0", "c", "Z") else
                    v[..., :m0, :] if k == "R" else v) for k, v in mats.items()}
    want = simulation_smoother(model.y, mats["a0"], mats["P0"], mats["T"], mats["Z"], mats["R"], mats["H"], mats["Q"],
                               mats["c"], mats["d"], n_simulations=spu, z_init=zi, z_state=zs, z_obs=zo)
    assert (got - want).abs().max().item() <= 1e-10 * (want.abs().max().item() + 1.0)
