"""CPU checks of the per-draw calls on data with partly observed rows: the masked filter (kfb_masked_filter) against
its literal numpy restatement and the dense conditional moments (oracle/masked.py), against the corrected standard and
univariate filters where those apply, and the simulation smoother with KFB_FLAG_PARTIAL_ROWS, forecasts and
conditional forecasts from its output against dense joint-Gaussian laws.  The kernels' own code runs through the host
build (tests/hostsim)."""
import ctypes

import numpy as np
import pytest

from oracle import condforecast as ocf
from oracle import forecast as ofc
from oracle import masked as oms
from oracle import simsmooth as oss
from pymc_statespace_b200._lib import KFB_FLAG_CORRECTED, KFB_FLAG_PARTIAL_ROWS
from tests import hostsim
from tests.helpers import random_system
from tests.hostsim import draws, partial
from tests.test_conditional_forecast_host import _desc, _round
from tests.test_simulation_smoother_host import check_joint, unit_basis

N = 10


def ragged(rng, y, rows=(0, 3, 6, N - 2, N - 1)):
    """y [n, p, 1] with one random entry of each of ``rows`` set to NaN (partly observed rows: the first and the
    ragged last two included) and row 4 fully missing."""
    y = y.copy()
    p = y.shape[1]
    for t in rows:
        y[t, rng.integers(0, p)] = np.nan
    y[4] = np.nan
    return y


def system(m, p, seed=0, n=N, c_d=True):
    rng = np.random.default_rng(100 * m + 10 * p + seed)
    r = 1 + (m + p) % m
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, r, n)  # non-diagonal H
    if p > 1:
        y = ragged(rng, y)
    c = rng.normal(size=(m, 1)) if c_d else None
    d = rng.normal(size=(p, 1)) if c_d else None
    return dict(a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q, c=c, d=d), y


GEOMS = [(m, p) for m in range(1, 5) for p in range(1, 4)]


def oracle_args(mats):
    return [mats[k] for k in ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")]


# ----------------------------------------------------------------------------------------------------- masked filter
@pytest.mark.parametrize("force_dyn", [False, True])
@pytest.mark.parametrize("m,p", GEOMS)
def test_masked_filter_matches_restatement_and_dense(m, p, force_dyn):
    mats, y = system(m, p)
    ps, pc, info, used = partial.masked_filter(y[..., 0], mats, force_dyn=force_dyn)
    assert used == (not force_dyn) and info[0] == 0
    a, P, oinfo = oms.masked_filter(y, *oracle_args(mats))
    assert oinfo == 0
    np.testing.assert_allclose(ps[0], a, rtol=1e-11, atol=1e-11 * np.abs(a).max())
    np.testing.assert_allclose(pc[0], P, rtol=1e-11, atol=1e-11 * np.abs(P).max())
    da, dP = oms.dense_predicted(y, *oracle_args(mats))
    np.testing.assert_allclose(ps[0], da, rtol=1e-9, atol=1e-9 * np.abs(da).max())
    np.testing.assert_allclose(pc[0], dP, rtol=1e-9, atol=1e-9 * np.abs(dP).max())


@pytest.mark.parametrize("kind", ["singular", "zero"])
def test_masked_filter_singular_and_zero_H(kind):
    rng = np.random.default_rng(5)
    m, p = 3, 2
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, 2, N)
    H = np.zeros((p, p)) if kind == "zero" else np.full((p, p), 0.8)  # rank 1
    y = ragged(rng, y)
    mats = dict(a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q, c=None, d=None)
    ps, pc, info, _ = partial.masked_filter(y[..., 0], mats)
    assert info[0] == 0
    da, dP = oms.dense_predicted(y, *oracle_args(mats))
    np.testing.assert_allclose(ps[0], da, rtol=1e-8, atol=1e-8 * np.abs(da).max())
    np.testing.assert_allclose(pc[0], dP, rtol=1e-8, atol=1e-8 * np.abs(dP).max())


def test_masked_filter_batched_draws_and_series():
    """n_draws = 3 with per-draw T and H, n_series = 2 with different NaN patterns per series; either output alone."""
    rng = np.random.default_rng(11)
    m, p, nd, ns = 2, 3, 3, 2
    mats, _ = system(m, p)
    mats["T"] = np.stack([mats["T"] * s for s in (0.5, 1.0, 1.5)])
    mats["H"] = np.stack([mats["H"] * s for s in (1.0, 2.0, 0.5)])
    ys = np.stack([ragged(rng, rng.normal(size=(N, p, 1)), rows=rows)[..., 0]
                   for rows in ((0, 2, 7), (1, 5, N - 1))])
    ps, pc, info, _ = partial.masked_filter(ys, mats, n_draws=nd, n_series=ns)
    assert (info == 0).all()
    for u in range(nd * ns):
        dr, se = divmod(u, ns)
        mu = dict(mats, T=mats["T"][dr], H=mats["H"][dr])
        a, P, _ = oms.masked_filter(ys[se], *oracle_args(mu))
        np.testing.assert_allclose(ps[u], a, rtol=1e-11, atol=1e-12)
        np.testing.assert_allclose(pc[u], P, rtol=1e-11, atol=1e-12)
    ps2, _, _, _ = partial.masked_filter(ys, mats, n_draws=nd, n_series=ns, want=("states",))
    _, pc2, _, _ = partial.masked_filter(ys, mats, n_draws=nd, n_series=ns, want=("covs",))
    assert np.array_equal(ps2, ps) and np.array_equal(pc2, pc)


@pytest.mark.parametrize("m,p", [(2, 1), (3, 2), (4, 3)])
def test_masked_filter_complete_rows_match_standard_filter(m, p):
    mats, y = system(m, p)
    y = np.nan_to_num(y, nan=0.25)
    y[4] = np.nan  # whole missing rows are the standard filter's own
    ps, pc, info, _ = partial.masked_filter(y[..., 0], mats)
    out, _, sinfo = hostsim.run("standard", y, *oracle_args(mats), strict=False, do_bwd=False)
    assert info[0] == 0 and sinfo == 0
    np.testing.assert_allclose(ps[0], out[1][..., 0], rtol=1e-12, atol=1e-12 * np.abs(ps).max())
    np.testing.assert_allclose(pc[0], out[3], rtol=1e-12, atol=1e-12 * np.abs(pc).max())


@pytest.mark.parametrize("m,p", [(2, 2), (3, 3), (4, 2)])
def test_masked_filter_diagonal_H_matches_univariate_filter(m, p):
    mats, y = system(m, p)
    mats["H"] = np.diag(np.diag(mats["H"]))
    ps, pc, info, _ = partial.masked_filter(y[..., 0], mats)
    out, _, uinfo = hostsim.run("univariate", y, *oracle_args(mats), strict=False, do_bwd=False)
    assert info[0] == 0 and uinfo == 0
    np.testing.assert_allclose(ps[0], out[1][..., 0], rtol=1e-10, atol=1e-10 * np.abs(ps).max())
    np.testing.assert_allclose(pc[0], out[3], rtol=1e-10, atol=1e-10 * np.abs(pc).max())


@pytest.mark.parametrize("force_dyn", [False, True])
def test_masked_filter_info_at_partial_row(force_dyn):
    """Entry 0 is observed without noise and not loaded on the states: F_o is 0 at the first row that observes it."""
    rng = np.random.default_rng(2)
    m, p = 2, 2
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, 1, N)
    Z[0] = 0.0
    H = np.diag([0.0, 1.0])
    y[:3, 0] = np.nan  # rows 0..2 observe entry 1 only
    y[3, 1] = np.nan   # row 3 observes entry 0 only
    mats = dict(a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q, c=None, d=None)
    ps, pc, info, _ = partial.masked_filter(y[..., 0], mats, force_dyn=force_dyn)
    assert info[0] == 4 and oms.masked_filter(y, *oracle_args(mats))[2] == 4
    assert np.isnan(ps).all() and np.isnan(pc).all()


# ------------------------------------------------------------------------------------ simulation smoother, flag set
def _smooth(y, mats, pc, flags, force_dyn=False):
    n, m, p, r = y.shape[0], mats["T"].shape[0], mats["Z"].shape[0], mats["R"].shape[1]
    zi, zs, zo = unit_basis(n, m, p, r)
    return partial.simsmooth(y, mats, pc[None], zi.shape[0], zi, zs, zo, force_dyn=force_dyn, flags=flags)


@pytest.mark.parametrize("force_dyn", [False, True])
@pytest.mark.parametrize("m,p", [(1, 2), (2, 2), (2, 3), (3, 2), (4, 3)])
def test_simulation_smoother_joint_law_with_partial_rows(m, p, force_dyn):
    mats, y = system(m, p)
    y = y[..., 0]
    _, pc, info, _ = partial.masked_filter(y, mats)
    states, sinfo = _smooth(y, mats, pc[0], KFB_FLAG_PARTIAL_ROWS | KFB_FLAG_CORRECTED, force_dyn)
    assert info[0] == 0 and sinfo[0] == 0
    mean, cov = oss.dense_state_posterior(y, *oracle_args(mats))
    check_joint(states, mean, cov, 1e-10)
    # a baseline that treats every partly observed row as missing has another law
    yb = y.copy()
    yb[np.isnan(yb).any(axis=1)] = np.nan
    _, pcb, _, _ = partial.masked_filter(yb, mats)
    base, _ = _smooth(yb, mats, pcb[0], 0)
    with pytest.raises(AssertionError):
        check_joint(base, mean, cov, 1e-10)


def test_simulation_smoother_flag_without_partial_rows_is_bitwise_same():
    rng = np.random.default_rng(9)
    m, p = 3, 2
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, p, 2, N, n_missing=2)
    mats = dict(a0=a0, P0=P0, T=T, Z=Z, R=R, H=H, Q=Q, c=rng.normal(size=m), d=rng.normal(size=p))
    pc = oss.predicted_covs(y, P0, T, Z, R, H, Q)
    zi, zs, zo = rng.normal(size=(7, m)), rng.normal(size=(N - 1, 7, 2)), rng.normal(size=(N, 7, p))
    for force_dyn in (False, True):
        a, ia = draws.simsmooth(y[..., 0], mats, pc[None], 7, zi, zs, zo, force_dyn=force_dyn)
        b, ib = partial.simsmooth(y[..., 0], mats, pc[None], 7, zi, zs, zo, force_dyn=force_dyn,
                                  flags=KFB_FLAG_PARTIAL_ROWS)
        assert np.array_equal(a, b) and (ia == 0).all() and (ib == 0).all()


def test_simulation_smoother_partial_row_without_flag_still_refused():
    mats, y = system(2, 2)
    _, pc, _, _ = partial.masked_filter(y[..., 0], mats)
    states, info = _smooth(y[..., 0], mats, pc[0], 0)
    assert info[0] == -1 and np.isnan(states).all()  # row 0 is partly observed


# ------------------------------------------------------------------------------- forecasts from the ragged edge
@pytest.mark.parametrize("m,p", [(2, 2), (3, 3)])
def test_forecast_from_ragged_edge_matches_dense_law(m, p):
    hor = 3
    mats, y = system(m, p)
    yx = np.concatenate([y[..., 0], np.full((hor, p), np.nan)])
    ps, pc, info, _ = partial.masked_filter(yx, mats)
    assert info[0] == 0
    mu, Sxx, muy, Syy = ofc.dense_forecast_law(y, *oracle_args(mats), horizon=hor)
    np.testing.assert_allclose(ps[0, N:N + hor], mu, rtol=1e-9, atol=1e-9 * np.abs(mu).max())
    r = mats["R"].shape[1]
    zi, zs, zo = unit_basis(hor, m, p, r)
    S = zi.shape[0]
    states, obs, finfo, _ = draws.forecast_paths(mats, ps[:, N], pc[:, N], S, zi, zs, zo)
    assert finfo[0] == 0
    check_joint(states.transpose(1, 0, 2), mu, Sxx, 1e-10)
    check_joint(obs.transpose(1, 0, 2), muy, Syy, 1e-10)


@pytest.mark.parametrize("force_dyn", [False, True])
def test_conditional_forecast_from_ragged_edge_matches_dense_law(force_dyn):
    m, p, hor = 3, 3, 3
    mats, y = system(m, p)
    cond = np.full((hor, p), np.nan)
    cond[0, 1] = 0.4
    cond[2, [0, 2]] = (-0.3, 1.1)
    ps, pc, info, _ = partial.masked_filter(y[..., 0], mats)
    r = mats["R"].shape[1]
    zi, zs, zo = unit_basis(hor, m, p, r)
    S = zi.shape[0]
    mom, states, obs, cinfo, _ = draws.conditional_forecast(mats, ps[:, N], pc[:, N], cond, S, zi, zs, zo, n=N,
                                                            force_dyn=force_dyn)
    assert info[0] == 0 and cinfo[0] == 0
    mean, cov = ocf.dense_conditional_forecast_law(y, *oracle_args(mats), cond=cond)
    k = hor * m
    tol = 1e-9 * (np.abs(mean).max() + 1)
    assert np.abs(mom["state_mean"][0].reshape(-1) - mean[:k]).max() <= tol
    assert np.abs(mom["obs_mean"][0].reshape(-1) - mean[k:]).max() <= tol
    paths = np.concatenate([states.transpose(1, 0, 2).reshape(S, -1), obs.transpose(1, 0, 2).reshape(S, -1)], axis=1)
    check_joint(paths[:, None, :], mean, cov, 1e-10)


# ------------------------------------------------------------------------------------------------------------ C ABI
def test_cabi_masked_filter_workspace_rule():
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    nb = ctypes.c_size_t(0)
    for (nd, ns, m, p, r) in ((3, 2, 2, 1, 1), (1, 1, 13, 1, 3), (4, 1, 3, 2, 2), (2, 3, 32, 32, 32)):
        d = _desc(nd, ns, 100, m, p, r)
        assert lib.kfb_masked_filter_workspace_bytes(ctypes.byref(d), ctypes.byref(nb)) == _lib.KFB_OK
        assert nb.value == _round(8 * nd * ns * (5 * m * m + 2 * m * p + 3 * p * p))


def test_cabi_masked_filter_argument_validation():
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    nb = ctypes.c_size_t(0)
    fw, f = lib.kfb_masked_filter_workspace_bytes, lib.kfb_masked_filter
    d = _desc()
    assert fw(None, ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    assert fw(ctypes.byref(d), None) == _lib.KFB_ERR_INVALID_ARG
    for k in ("m", "p", "r", "n_draws", "n_series", "n"):
        bad = _desc()
        setattr(bad, k, 0)
        assert fw(ctypes.byref(bad), ctypes.byref(nb)) == _lib.KFB_ERR_INVALID_ARG
    for k in ("T", "Z", "R", "H", "Q", "c", "d"):
        tv = _desc()
        setattr(tv, k + "_ts", 4)
        assert fw(ctypes.byref(tv), ctypes.byref(nb)) == _lib.KFB_ERR_UNSUPPORTED
    for k in ("m", "p", "r"):
        assert fw(ctypes.byref(_desc(**{k: 33})), ctypes.byref(nb)) == _lib.KFB_ERR_UNSUPPORTED
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below is refused first
    full = _lib.KfbInputs(*([fake] * 8 + [None, None]))

    def call(ins, ps=fake, pc=fake, info=fake, ws=None, nbytes=0):
        return f(ctypes.byref(d), ins if ins is None else ctypes.byref(ins), ps, pc, info, ws, nbytes, None)

    assert call(None) == _lib.KFB_ERR_INVALID_ARG
    for i in range(8):  # y a0 P0 T Z R H Q are required
        ins = _lib.KfbInputs(*([fake] * 8 + [None, None]))
        setattr(ins, ("y", "a0", "P0", "T", "Z", "R", "H", "Q")[i], None)
        assert call(ins) == _lib.KFB_ERR_INVALID_ARG
    assert call(full, ps=None, pc=None) == _lib.KFB_ERR_INVALID_ARG
    assert call(full, info=None) == _lib.KFB_ERR_INVALID_ARG
    assert call(full, ps=None) == _lib.KFB_ERR_WORKSPACE
    assert fw(ctypes.byref(d), ctypes.byref(nb)) == _lib.KFB_OK
    assert call(full, ws=fake, nbytes=nb.value - 1) == _lib.KFB_ERR_WORKSPACE


def test_cabi_simulation_smoother_flag_keeps_request_rules():
    """KFB_FLAG_PARTIAL_ROWS (and any other flag) changes neither the workspace nor the argument checks."""
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    a, b = ctypes.c_size_t(0), ctypes.c_size_t(0)
    d = _desc()
    assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(d), 5, ctypes.byref(a)) == _lib.KFB_OK
    d.flags = KFB_FLAG_PARTIAL_ROWS | KFB_FLAG_CORRECTED | 0x8000
    assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(d), 5, ctypes.byref(b)) == _lib.KFB_OK
    assert a.value == b.value
    tv = _desc()
    tv.flags, tv.T_ts = KFB_FLAG_PARTIAL_ROWS, 4
    assert lib.kfb_simulation_smoother_workspace_bytes(ctypes.byref(tv), 5, ctypes.byref(b)) == _lib.KFB_ERR_UNSUPPORTED
