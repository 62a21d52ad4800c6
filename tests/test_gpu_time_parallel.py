"""Time-parallel kernels (BatchedKalman(time_parallel=True), KFB_FLAG_TIME_PARALLEL) on the GPU.

Parity with the oracle (all six outputs, all nine cotangents), known answers that share no recursion (dense Gaussian
density and its autograd, the Nile fixture), agreement with the sequential kernels at batch sizes 1..64 and at theta
level, a 65,536-step series, determinism and info codes, the fall-back to the sequential kernels outside the
time-parallel geometry, and the seam / Op pair with the filter attribute set.
"""
import importlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from oracle import kalman_numpy as kn
from oracle import kalman_torch as kt
from tests.helpers import GOLDEN, nile_inputs, random_system, rel_err

pytestmark = pytest.mark.gpu

RTOL = 1e-8
OUT = ("filtered_states", "predicted_states", "filtered_covs", "predicted_covs", "loglik", "ll_obs")
NAMES = ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")


def _dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device="cuda")


def run(kind, args, c=None, d=None, strict=True, time_varying=(), g_ll_obs=None, time_parallel=True, bwd=True):
    """One unit through BatchedKalman; (outputs in the oracle's shapes, grads, info, time_parallel_active)."""
    from pymc_statespace_b200 import BatchedKalman

    y, a0, P0, T, Z, R, H, Q = args
    n, p = y.shape[0], y.shape[1]
    m, r = T.shape[-1], R.shape[-1]
    bk = BatchedKalman(kind, n, m, p, r, n_draws=1, strict_reference=strict, time_varying=time_varying,
                       time_parallel=time_parallel)
    ins = {k: None if v is None else _dev(np.asarray(v, dtype=float)[None])
           for k, v in zip(NAMES, (a0, P0, T, Z, R, H, Q, c, d))}
    out = bk.forward(_dev(y[..., 0]), **ins, outputs=OUT, save_for_backward=bwd)
    res = [out["filtered_states"][0].cpu().numpy()[..., None], out["predicted_states"][0].cpu().numpy()[..., None],
           out["filtered_covs"][0].cpu().numpy(), out["predicted_covs"][0].cpu().numpy(),
           float(out["loglik"][0]), out["ll_obs"][0].cpu().numpy()]
    info = int(out["info"][0])
    grads = None
    if bwd:
        gl = None if g_ll_obs is None else _dev(np.zeros(1))
        glo = None if g_ll_obs is None else _dev(np.asarray(g_ll_obs)[None])
        grads = {k: v[0].cpu().numpy() for k, v in bk.backward(g_loglik=gl, g_ll_obs=glo).items()}
        for k in ("a0", "c", "d"):
            grads[k] = grads[k][..., None]
    return res, grads, info, bk.time_parallel_active


def check(kind, args, c=None, d=None, strict=True, time_varying=(), g_ll_obs=None, rtol=RTOL, grad_rtol=RTOL):
    ref = kn.kalman_filter(kind, *args, c=c, d=d, strict_reference=strict)
    res, g, info, active = run(kind, args, c, d, strict, time_varying, g_ll_obs)
    assert active and info == 0
    for name, a, b in zip(OUT, res, ref):
        assert rel_err(a, b) < rtol, (kind, name, rel_err(a, b))
    _, gref = kt.loglik_and_grads(kind, *args, c=c, d=d, strict_reference=strict, g_ll_obs=g_ll_obs)
    for k in gref:
        scale = max(np.abs(gref[k]).max(), 1e-12 * max(np.abs(v).max() for v in gref.values()))
        assert np.abs(g[k] - gref[k]).max() / scale < grad_rtol, (kind, k, np.abs(g[k] - gref[k]).max() / scale)


def _missing(y, n):
    y = y.copy()
    if n >= 4:
        y[[0, n // 3, n // 2, n - 1]] = np.nan  # first and last included
    elif n == 3:
        y[[0, 2]] = np.nan
    return y


# ---------------------------------------------------------------------------------------------- 1. parity
@pytest.mark.parametrize("n", [1, 2, 3, 31, 1000, 4097])
@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_parity_with_oracle(m, n):
    rng = np.random.default_rng(10 * m + n)
    args = random_system(rng, m, 1, 2, n)
    c, d = rng.normal(size=(m, 1)), rng.normal(size=(1, 1))
    check("standard", args, c, d)
    check("standard", (_missing(args[0], n),) + args[1:], c, d, strict=False,
          g_ll_obs=rng.normal(size=n) if n > 2 else None)


@pytest.mark.parametrize("kind", ["standard", "single", "cholesky"])
@pytest.mark.parametrize("strict", [True, False])
def test_filter_kinds_missing_rows_nonsymmetric_P0(kind, strict):
    rng = np.random.default_rng(3)
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 3, 1, 2, 300, n_missing=20)
    P0 = P0 + 0.3 * rng.normal(size=P0.shape)
    args = (_missing(y, 300), a0, P0, T, Z, R, H, Q)
    check(kind, args, rng.normal(size=(3, 1)), rng.normal(size=(1, 1)), strict=strict)
    check(kind, args, None, rng.normal(size=(1, 1)), strict=strict, g_ll_obs=rng.normal(size=300))


def test_time_varying_matrices():
    rng = np.random.default_rng(4)
    n, m = 200, 3
    systems = [random_system(rng, m, 1, 2, n, n_missing=10) for _ in range(n)]
    y, a0, P0 = systems[0][:3]
    T, Z, R, H, Q = (np.stack([s[i] for s in systems]) for i in range(3, 8))
    c, d = rng.normal(size=(n, m, 1)), rng.normal(size=(n, 1, 1))
    check("standard", (_missing(y, n), a0, P0, T, Z, R, H, Q), c, d, time_varying=("T", "Z", "R", "H", "Q", "c", "d"))
    check("single", (y, a0, P0, T, Z[0], R, H[0], Q), None, d[0], strict=False, time_varying=("T", "R", "Q"),
          g_ll_obs=rng.normal(size=n))


# ---------------------------------------------------------------------------------------------- 2. known answers
def test_loglik_against_dense_density_and_arma21_gradient_against_dense_autograd():
    from oracle import models as om
    from pymc_statespace_b200.synthetic import simulate_arma

    y = simulate_arma(60, (0.5, -0.2), (0.3,), 1.0, seed=3)[:, None, None]
    a0, P0, T, Z, R, H, Q = (x.detach().numpy() for x in om.arma_matrices(
        torch.tensor([0.1, -0.2, 0.8, 0.5, -0.2, 0.3], dtype=torch.float64), (2, 1), True))
    args = (y, a0.reshape(-1, 1), P0, T, Z, R, H, Q)
    res, g, info, active = run("standard", args)
    assert active and info == 0
    dense = kn.dense_gaussian_loglik(*args)
    assert abs(res[4] - dense) < 1e-10 * abs(dense)
    # The dense density reads the symmetric inputs P0, H, Q in another entry-wise gauge than the recursion (it sees them
    # through their symmetric parts in another order), so their symmetric parts are compared, as in test_oracle_pins /
    # test_hostsim_math; the recursion's full-matrix gauge is pinned against the restated filter right after.
    _, gd = kt.dense_loglik_and_grads(*args)
    _, gr = kt.loglik_and_grads("standard", *args)
    sym = lambda k, x: 0.5 * (x + x.T) if k in ("P0", "H", "Q") else x  # noqa: E731
    for k in gd:
        got = g[k].reshape(np.shape(gd[k]))
        scale = max(np.abs(gd[k]).max(), 1e-12)
        assert np.abs(sym(k, got) - sym(k, gd[k])).max() / scale < 1e-8, k
        assert np.abs(got - gr[k]).max() / max(np.abs(gr[k]).max(), 1e-12) < 1e-8, k


@pytest.mark.parametrize("n_missing", [0, 5])
def test_nile_fixture(n_missing):
    """Loglik against the 40-digit dense density at 1e-10; gradients against the oracle at 1e-6 (P0 = 1e6 I)."""
    gold = json.load(open(os.path.join(GOLDEN, "nile_dense_loglik.json")))[str(n_missing)]["loglik"]
    args = nile_inputs(n_missing)
    res, g, info, active = run("standard", args)
    assert active and info == 0 and abs(res[4] - gold) < 1e-10 * abs(gold), (res[4], gold)
    _, gref = kt.loglik_and_grads("standard", *args)
    for k in gref:
        scale = max(np.abs(gref[k]).max(), 1e-12 * max(np.abs(v).max() for v in gref.values()))
        assert np.abs(g[k] - gref[k]).max() / scale < 1e-6, k


# ---------------------------------------------------------------------------------------------- 3. vs sequential
def _batch(spec_name, B, n, seed=0):
    from oracle import models as om

    rng = np.random.default_rng(seed)
    if spec_name == "arma11":
        from pymc_statespace_b200.synthetic import simulate_arma

        y = simulate_arma(n, (0.6,), (0.3,), 1.0, seed=seed)[:, None]
        mats = [om.arma_matrices(torch.tensor([*rng.normal(size=2), np.exp(rng.normal(0, .3)), rng.uniform(-.9, .9),
                                               rng.normal(0, .5)], dtype=torch.float64), (1, 1), True) for _ in range(B)]
        a0, P0, T, Z, R, H, Q = (np.stack([mm[i].detach().numpy() for mm in mats]) for i in range(7))
        a0 = a0.reshape(B, -1)
        Z, H = Z[0], H[0]
    else:  # local linear trend
        y = np.cumsum(np.cumsum(rng.normal(size=n)) * 0.1 + rng.normal(size=n))[:, None]
        T, Z, R = np.array([[1.0, 1.0], [0.0, 1.0]]), np.array([[1.0, 0.0]]), np.eye(2)
        Q = np.stack([np.diag(np.exp(rng.normal(size=2)) * [0.5, 0.01]) for _ in range(B)])
        H = np.exp(rng.normal(size=(B, 1, 1)))
        a0, P0 = rng.normal(size=(B, 2)), np.stack([np.eye(2) * 10.0] * B)
    y[rng.choice(n, 7, replace=False)] = np.nan
    return y, a0, P0, T, Z, R, H, Q


def _both(y, a0, P0, T, Z, R, H, Q, B, gl=None, glo=None):
    from pymc_statespace_b200 import BatchedKalman

    n, m, r = y.shape[0], P0.shape[-1], R.shape[-1]
    res = {}
    for tp in (False, True):
        bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, time_parallel=tp)
        out = bk.forward(_dev(y), _dev(a0), _dev(P0), _dev(T), _dev(Z), _dev(R), _dev(H), _dev(Q), outputs=OUT,
                         save_for_backward=True)
        g = bk.backward(g_loglik=gl, g_ll_obs=glo)
        res[tp] = ({k: v.cpu().numpy() for k, v in out.items()}, {k: v.cpu().numpy() for k, v in g.items()})
        assert bk.time_parallel_active == tp
    return res


@pytest.mark.parametrize("model", ["arma11", "llt"])
@pytest.mark.parametrize("B", [1, 7, 64])
def test_agrees_with_sequential_kernels(model, B):
    n = 1000
    args = _batch(model, B, n, seed=B)
    rng = np.random.default_rng(B)
    for gl, glo in ((None, None), (_dev(rng.normal(size=B)), _dev(rng.normal(size=(B, n))))):
        res = _both(*args, B, gl, glo)
        (os_, gs), (op, gp) = res[False], res[True]
        assert (os_["info"] == 0).all() and (op["info"] == op["info"]).all() and (op["info"] == 0).all()
        for k in OUT:
            assert rel_err(op[k], os_[k]) < RTOL, (k, rel_err(op[k], os_[k]))
        for k in gs:
            for b in range(B):
                scale = max(np.abs(gs[k][b]).max(), 1e-12)
                assert np.abs(gp[k][b] - gs[k][b]).max() / scale < RTOL, (k, b)


@pytest.mark.parametrize("spec_name", ["arma11", "local_level"])
def test_theta_level_logp_and_grad(spec_name):
    from pymc_statespace_b200 import models
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import arma11_workload

    if spec_name == "arma11":
        spec, y, theta = arma11_workload(16, 500, seed=2)
    else:
        spec = models.local_level_spec()
        rng = np.random.default_rng(5)
        y = np.cumsum(rng.normal(size=500))[:, None]
        theta = np.concatenate([rng.normal(size=(16, 2)), np.tile([3.0, 0.1, 0.1, 2.0], (16, 1)),
                                np.exp(rng.normal(size=(16, 3)))], axis=1)
    th = _dev(theta)
    seq = KalmanLogp(spec, y, n_draws=16)
    tpar = KalmanLogp(spec, y, n_draws=16, time_parallel=True)
    assert tpar.kalman.time_parallel_active and not seq.kalman.time_parallel_active
    assert tpar.clone_for(4).kalman.time_parallel_active
    lp0, g0 = (t.cpu().numpy() for t in seq.logp_and_grad(th))
    lp1, g1 = (t.cpu().numpy() for t in tpar.logp_and_grad(th))
    assert (tpar.info == 0).all()
    assert rel_err(lp1, lp0) < RTOL
    for b in range(16):
        assert np.abs(g1[b] - g0[b]).max() <= RTOL * np.abs(g0[b]).max(), b


# ---------------------------------------------------------------------------------------------- 4. long series
def test_long_series():
    n = 65536
    y, a0, P0, T, Z, R, H, Q = _batch("arma11", 1, n, seed=11)
    res = _both(y, a0, P0, T, Z, R, H, Q, 1)
    (os_, gs), (op, gp) = res[False], res[True]
    assert np.isfinite(op["loglik"]).all() and op["info"][0] == 0
    assert rel_err(op["loglik"], os_["loglik"]) < 1e-10
    for k in OUT:
        assert rel_err(op[k], os_[k]) < RTOL, k
    for k in gs:
        assert np.isfinite(gp[k]).all()
        assert rel_err(gp[k], gs[k]) < RTOL, (k, rel_err(gp[k], gs[k]))


# ---------------------------------------------------------------------------------------------- 5. determinism, status
def test_bitwise_deterministic():
    y, a0, P0, T, Z, R, H, Q = _batch("llt", 4, 3000, seed=1)
    r1 = _both(y, a0, P0, T, Z, R, H, Q, 4)[True]
    r2 = _both(y, a0, P0, T, Z, R, H, Q, 4)[True]
    for a, b in ((r1[0], r2[0]), (r1[1], r2[1])):
        for k in a:
            assert np.array_equal(a[k], b[k], equal_nan=True), k


def test_info_codes_and_undefined_elements():
    rng = np.random.default_rng(8)
    # Z P0 Z^T + H = 0: F_0 = 0 -> info 1, loglik NaN on both paths
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 2, 1, 1, 50)
    args = (y, a0, np.diag([0.0, 1.0]), T, np.array([[1.0, 0.0]]), R, np.zeros((1, 1)), Q)
    r_seq = run("standard", args, time_parallel=False, bwd=False)
    r_tp = run("standard", args, bwd=False)
    assert r_seq[2] == r_tp[2] == 1 and np.isnan(r_tp[0][4])
    # Z C Z^T + H = 0 at every step: no parallel element; the unit takes the sequential walk inside its CTA
    y = rng.normal(size=(400, 1, 1))
    y[[3, 200]] = np.nan
    args = (y, rng.normal(size=(2, 1)), np.eye(2), np.array([[0.5, 0.8], [0.0, 0.3]]), np.array([[1.0, 0.0]]),
            np.array([[0.0], [1.0]]), np.zeros((1, 1)), np.eye(1))
    check("standard", args)
    r_seq, r_tp = run("standard", args, time_parallel=False), run("standard", args)
    assert r_seq[2] == r_tp[2] == 0
    for a, b in zip(r_tp[0], r_seq[0]):
        assert rel_err(a, b) < 1e-10
    for k in r_seq[1]:
        assert rel_err(r_tp[1][k], r_seq[1][k]) < 1e-8, k


# ---------------------------------------------------------------------------------------------- 6. fall-back
@pytest.mark.parametrize("case", ["univariate", "steady_state", "m6p3"])
def test_unsupported_geometry_runs_the_sequential_kernels(case):
    rng = np.random.default_rng(9)
    if case == "m6p3":
        args, kind = random_system(rng, 6, 3, 2, 80, n_missing=4), "standard"
    else:
        args, kind = random_system(rng, 2, 1, 1, 80, n_missing=0 if case == "steady_state" else 4), case
    r0 = run(kind, args, time_parallel=False)
    r1 = run(kind, args, time_parallel=True)
    assert not r1[3] and not r0[3] and r0[2] == r1[2]
    for a, b in zip(r0[0], r1[0]):
        assert np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)
    for k in r0[1]:
        assert np.array_equal(r0[1][k], r1[1][k]), k


# ---------------------------------------------------------------------------------------------- 7. seam and Op pair
def test_seam_numpy_in_and_out():
    from pymc_statespace_b200.filters import FILTER_FACTORY
    from pymc_statespace_b200.seam import filter_numpy, logp_grads_numpy, seam_graph

    rng = np.random.default_rng(21)
    args = random_system(rng, 2, 1, 2, 500, n_missing=6)
    d = rng.normal(size=(1, 1))
    flt = FILTER_FACTORY["standard"]()
    assert flt.time_parallel is False
    flt.time_parallel = True
    outs = filter_numpy(flt, *args, d=d)
    ref = kn.kalman_filter("standard", *args, d=d)
    for a, b in zip(outs, ref):
        assert rel_err(a, b) < RTOL
    names = ("data",) + NAMES[:7] + ("d",)
    arrays = dict(zip(names, list(args) + [d]))
    w = rng.normal(size=500)
    _, g1 = kt.loglik_and_grads("standard", *args, d=d)
    _, g2 = kt.loglik_and_grads("standard", *args, d=d, g_ll_obs=w)
    for gl, glo in ((1.0, None), (0.5, w)):
        ll, g = logp_grads_numpy(flt, arrays, g_loglik=gl, g_ll_obs=glo)
        assert abs(ll - ref[4]) < RTOL * abs(ref[4])
        for k in g:
            want = gl * g1[k] + (0.0 if glo is None else g2[k])
            assert rel_err(g[k], np.asarray(want).reshape(g[k].shape)) < RTOL, k
    assert seam_graph(flt, arrays, "grad").bk.time_parallel_active
    flt.time_parallel = False
    assert not seam_graph(flt, arrays, "grad").bk.time_parallel_active


SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fake_pytensor")


@pytest.fixture()
def shim_tp():
    """pymc_statespace_b200.pytensor_op re-imported against the stand-in pytensor; restored afterwards."""
    sys.path.insert(0, SHIM)
    for k in [k for k in sys.modules if k == "pytensor" or k.startswith("pytensor.")]:
        del sys.modules[k]
    import pymc_statespace_b200.pytensor_op as pop

    pop = importlib.reload(pop)
    assert pop.HAVE_PYTENSOR
    import pytensor

    yield pop, pytensor
    sys.path.remove(SHIM)
    for k in [k for k in sys.modules if k == "pytensor" or k.startswith("pytensor.")]:
        del sys.modules[k]
    importlib.reload(pop)


def test_op_pair_with_time_parallel_attribute(shim_tp):
    pop, pytensor = shim_tp
    import pytensor.tensor as pt

    from pymc_statespace_b200.filters import FILTER_FACTORY

    assert pop.KalmanFilterOp("standard", True, True, False) == pop.KalmanFilterOp("standard", True, True, False, False)
    assert pop.KalmanFilterOp("standard", True, True, False) != pop.KalmanFilterOp("standard", True, True, False, True)
    rng = np.random.default_rng(31)
    m, n = 3, 120
    args = list(random_system(rng, m, 1, 2, n, n_missing=5))
    c = rng.normal(size=(m, 1))
    names = ["data", "a0", "P0", "T", "Z", "R", "H", "Q", "c"]
    ins = [pt.dtensor3(k) if k == "data" else pt.dmatrix(k) for k in names]
    flt = FILTER_FACTORY["standard"]()
    flt.time_parallel = True
    outs = flt.build_graph(*ins[:8], c=ins[8])
    assert outs[4].owner.op.time_parallel
    grads = pytensor.grad(outs[4], ins)
    f = pytensor.function(ins, list(outs) + list(grads[1:]))
    res = f(*(args + [c]))
    ref = kn.kalman_filter("standard", *args, c=c)
    for a, b in zip(res[:6], ref):
        assert rel_err(a, b) < RTOL
    _, gref = kt.loglik_and_grads("standard", *args, c=c)
    for name, got in zip(names[1:], res[6:]):
        scale = max(np.abs(gref[name]).max(), 1e-12)
        assert np.abs(got - gref[name]).max() / scale < RTOL, name
