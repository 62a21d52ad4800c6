"""The device step programs (csrc/kf_core.cuh) compiled for the HOST and checked against the oracle.
This is how the Kalman / adjoint math is verified in the GPU-less build container; the GPU tests repeat the
same comparisons through the real kernels.  (tests/hostsim is test infrastructure, not a product path.)"""
import numpy as np
import pytest

from oracle import kalman_numpy as kn
from oracle import kalman_torch as kt
from tests import hostsim
from tests.helpers import nile_inputs, random_system, rel_err


def _check(kind, args, c=None, d=None, strict=True, static=False, w=None, tol=1e-9):
    ref = kn.kalman_filter(kind, *args, c=c, d=d, strict_reference=strict)
    outs, g, info = hostsim.run(kind, *args, c=c, d=d, strict=strict, static_dims=static, g_ll_obs=w,
                                g_loglik=(0.0 if w is not None else None))
    assert info == 0
    for a, b in zip(outs, ref):
        assert rel_err(a, b) < tol
    _, gt = kt.loglik_and_grads(kind, *args, c=c, d=d, strict_reference=strict, g_ll_obs=w)
    for k in gt:
        assert rel_err(g[k], gt[k]) < tol or np.abs(g[k] - gt[k]).max() < 1e-13, (kind, k)


@pytest.mark.parametrize("static", [True, False], ids=["ThreadCtx", "CoopCtx"])
@pytest.mark.parametrize("dims", [(1, 1, 1), (2, 1, 1), (3, 2, 2), (4, 3, 2)])
@pytest.mark.parametrize("kind", ["standard", "univariate"])
def test_forward_and_adjoint(kind, dims, static):
    m, p, r = dims
    rng = np.random.default_rng(m * 10 + p)
    args = random_system(rng, m, p, r, 25, n_missing=2)
    c, d = rng.normal(size=(m, 1)), rng.normal(size=(p, 1))
    _check(kind, args, c, d, True, static)
    _check(kind, args, c, d, False, static, w=rng.normal(size=25))


@pytest.mark.parametrize("static", [True, False], ids=["ThreadCtx", "CoopCtx"])
def test_single_cholesky_p1_and_steady_state(static):
    rng = np.random.default_rng(2)
    args = random_system(rng, 3, 1, 2, 30, n_missing=3)
    d = rng.normal(size=(1, 1))
    _check("single", args, None, d, True, static)
    _check("cholesky", args, None, d, True, static)
    args = random_system(rng, 4, 2, 2, 30)
    _check("steady_state", args, None, rng.normal(size=(2, 1)), True, static, tol=1e-8)
    _check("steady_state", args, None, rng.normal(size=(2, 1)), False, static, tol=1e-8)


def test_time_varying_and_partial_missing():
    rng = np.random.default_rng(1)
    n, m, p, r = 12, 3, 2, 2
    systems = [random_system(rng, m, p, r, n) for _ in range(n)]
    y, a0, P0 = systems[0][:3]
    T, Z, R, H, Q = (np.stack([s[i] for s in systems]) for i in range(3, 8))
    _check("standard", (y, a0, P0, T, Z, R, H, Q), rng.normal(size=(n, m, 1)), rng.normal(size=(n, p, 1)))
    args = random_system(rng, 4, 3, 2, 30, n_missing=2, partial=True, diag_H=True)
    _check("univariate", args)
    _, _, info = hostsim.run("standard", *args, do_bwd=False)
    assert info < 0


def test_deferred_log_matches_per_step_log():
    args = nile_inputs(5)
    ref = kn.kalman_filter("standard", *args)[4]
    outs, _, _ = hostsim.run("standard", *args, static_dims=True, full=False, do_bwd=False)
    assert abs(outs[4] - ref) < 1e-12 * abs(ref)


@pytest.mark.parametrize("dims", [(4, 2, 2), (6, 3, 3), (3, 3, 1)])
def test_as_coded_cholesky_filter_multivariate(dims):
    # SURVEY A.2-Q4: bug-compatible CholeskyFilter for k_endog > 1 (cooperative kernels only)
    m, p, r = dims
    rng = np.random.default_rng(m + p)
    args = random_system(rng, m, p, r, 25, n_missing=2)
    _check("cholesky", args, rng.normal(size=(m, 1)), rng.normal(size=(p, 1)), True, False, tol=1e-8)


def test_dare_solver_and_adjoint_on_host():
    import scipy.linalg
    import torch

    from pymc_statespace_b200.models import arma_spec, trend_seasonal_spec

    def run(T, Z, H, C, grad_tol):
        m, p = T.shape[0], Z.shape[0]
        T, Z, H, C = [np.ascontiguousarray(v, dtype=float) for v in (T, Z, H, C)]
        gP, gG = np.random.default_rng(0).normal(size=(m, m)), np.random.default_rng(1).normal(size=(p, p))
        Pss, Gss, gs = hostsim.dare(T, Z, H, C, gP, gG)  # raises unless the solve succeeds
        gT, gZ, gH, gC = (gs[k] for k in ("T", "Z", "H", "C"))
        ref = scipy.linalg.solve_discrete_are(T.T, Z.T, C, H)
        assert rel_err(Pss, ref) < 1e-12
        ts = [torch.tensor(v, requires_grad=True) for v in (T, Z, H, C)]
        X = kt.solve_discrete_are(ts[0].T, ts[1].T, ts[3], ts[2])
        G = torch.linalg.inv(ts[1] @ X @ ts[1].T + ts[2])
        ((X * torch.tensor(gP)).sum() + (G * torch.tensor(gG)).sum()).backward()
        if grad_tol:
            for a, b in zip((gT, gZ, gH, gC), ts):
                assert rel_err(a, b.grad.numpy()) < grad_tol

    rng = np.random.default_rng(3)
    m, p, r = 4, 2, 2
    T, Z, R = rng.normal(size=(m, m)) * 0.4, rng.normal(size=(p, m)), rng.normal(size=(m, r))
    A = rng.normal(size=(p, p))
    run(T, Z, A @ A.T + 0.1 * np.eye(p), R @ R.T, 1e-10)
    mats = arma_spec((1, 1)).matrices(np.array([0, 0, 1.3, 0.7, 0.4]))  # H = 0: exact observation
    run(mats["T"], mats["Z"], mats["H"], mats["R"] @ mats["Q"] @ mats["R"].T, None)
    mats = trend_seasonal_spec(29).matrices(np.array([0.1, 0.01, 0.05, 0.5]))  # k_states = 30, unit roots
    run(mats["T"], mats["Z"], mats["H"], mats["R"] @ mats["Q"] @ mats["R"].T, 1e-9)
    run(np.array([[1.0, 1.0], [0.0, 1.0]]), np.array([[1.0, 0.0]]), np.array([[0.8]]), np.diag([0.5, 0.01]), 1e-10)


@pytest.mark.parametrize("static", [True, False], ids=["ThreadCtx", "CoopCtx"])
@pytest.mark.parametrize("dims", [(1, 1, 1), (2, 1, 1), (3, 2, 2), (4, 3, 2)])
def test_predictor_form_hot_path(dims, static):
    """kf_pred.cuh: loglik-only forward + adjoint in one-step-predictor form (what the GPU hot path runs)."""
    m, p, r = dims
    rng = np.random.default_rng(m * 13 + p)
    args = random_system(rng, m, p, r, 25, n_missing=2)
    c, d = rng.normal(size=(m, 1)), rng.normal(size=(p, 1))
    for kind, strict, w in (("standard", True, None), ("standard", False, rng.normal(size=25))) + (
            (("single", True, None), ("cholesky", True, None)) if p == 1 else ()):
        ref = kn.kalman_filter(kind, *args, c=c, d=d, strict_reference=strict)
        outs, g, info = hostsim.run(kind, *args, c=c, d=d, strict=strict, static_dims=static, full=False, pred=True,
                                    g_ll_obs=w, g_loglik=(0.0 if w is not None else None))
        assert info == 0 and abs(outs[4] - ref[4]) < 1e-12 * abs(ref[4])
        _, gt = kt.loglik_and_grads(kind, *args, c=c, d=d, strict_reference=strict, g_ll_obs=w)
        for k in gt:
            assert rel_err(g[k], gt[k]) < 1e-9 or np.abs(g[k] - gt[k]).max() < 1e-13, (kind, k)


@pytest.mark.parametrize("static", [True, False], ids=["ThreadCtx", "CoopCtx"])
def test_predictor_form_without_T_and_Z_cotangents(static):
    """Structural models have constant T and Z: with T-bar / Z-bar not requested the adjoint drops the dense
    Lb = Ps L (P + P^T) product (kf_pred.cuh need_Lb).  Every other cotangent must be unchanged."""
    rng = np.random.default_rng(5)
    args = random_system(rng, 4, 2, 2, 20, n_missing=2)
    c, d = rng.normal(size=(4, 1)), rng.normal(size=(2, 1))
    for kind in ("standard", "steady_state"):
        kw = dict(c=c, d=d) if kind == "standard" else {}
        _, g_all, _ = hostsim.run(kind, *args, static_dims=static, full=False, pred=True, **kw)
        _, g_few, _ = hostsim.run(kind, *args, static_dims=static, full=False, pred=True, skip=("T", "Z"), **kw)
        _, gt = kt.loglik_and_grads(kind, *args, **kw)
        for k in gt:
            if k in ("T", "Z"):
                continue
            if kind == "steady_state" and k in ("R", "Q", "H"):
                continue  # the DARE epilogue (numpy, in hostsim) folds T-bar / Z-bar contributions into these
            assert rel_err(g_few[k], g_all[k]) < 1e-12 or np.abs(g_few[k] - g_all[k]).max() < 1e-14, (kind, k)
            assert rel_err(g_few[k], gt[k]) < 1e-8 or np.abs(g_few[k] - gt[k]).max() < 1e-13, (kind, k)


def test_predictor_form_steady_state_and_time_varying():
    rng = np.random.default_rng(77)
    args = random_system(rng, 4, 2, 2, 30)
    for static in (True, False):
        ref = kn.kalman_filter("steady_state", *args)
        outs, g, _ = hostsim.run("steady_state", *args, static_dims=static, full=False, pred=True)
        assert abs(outs[4] - ref[4]) < 1e-11 * abs(ref[4])
        _, gt = kt.loglik_and_grads("steady_state", *args)
        for k in gt:
            assert rel_err(g[k], gt[k]) < 1e-8 or np.abs(g[k] - gt[k]).max() < 1e-13, k
    n, m, p, r = 12, 3, 2, 2
    S = [random_system(rng, m, p, r, n) for _ in range(n)]
    y, a0, P0 = S[0][:3]
    T, Z, R, H, Q = (np.stack([s[i] for s in S]) for i in range(3, 8))
    c, d = rng.normal(size=(n, m, 1)), rng.normal(size=(n, p, 1))
    ref = kn.kalman_filter("standard", y, a0, P0, T, Z, R, H, Q, c=c, d=d)
    outs, g, _ = hostsim.run("standard", y, a0, P0, T, Z, R, H, Q, c=c, d=d, full=False, pred=True)
    assert abs(outs[4] - ref[4]) < 1e-12 * abs(ref[4])
    _, gt = kt.loglik_and_grads("standard", y, a0, P0, T, Z, R, H, Q, c=c, d=d)
    for k in gt:
        assert rel_err(g[k], gt[k]) < 1e-9, k


def test_rts_smoother_on_host():
    rng = np.random.default_rng(0)
    from tests.helpers import make_test_inputs

    for args, skip in ((nile_inputs(0), 5), (make_test_inputs(1, 5, 1, 10), 0),
                       (make_test_inputs(1, 5, 2, 10, missing_data=1), 0), (random_system(rng, 6, 3, 3, 30, n_missing=2), 0)):
        o = kn.kalman_filter("standard", *args)
        T, R, Q = (np.ascontiguousarray(args[i]) for i in (3, 5, 7))
        fs = o[0][..., 0]
        ss, sc = hostsim.smoother(T, R, Q, o[0], o[2])
        ss = ss[..., 0]
        rs, rc = kn.kalman_smoother(T, R, Q, o[0], o[2])
        assert rel_err(ss, rs[..., 0]) < 1e-10
        # reference tests/test_kalman_filter.py:236-238: the first few smoothed covariances of the P0 = 1e6 fixture are
        # ill-conditioned (pinv of cond ~3e6 followed by a 1e6-sized cancellation) and are skipped there as well
        assert rel_err(sc[skip:], rc[skip:]) < 1e-10
        np.testing.assert_allclose(ss[-1], fs[-1])


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_short_form_adjoint(m):
    """kf_p1.cuh: symmetric short-form adjoint for t >= 1 + literal Joseph-form adjoint at t = 0 (k_endog = 1).
    Must reproduce torch-autograd of the literal restatement for every cotangent, including the entry-wise gauge of
    P0-bar for a NON-symmetric P0 (BayesianARMA with stationary_initialization=False writes P0 = theta.reshape)."""
    rng = np.random.default_rng(100 + m)
    for n, n_missing, asym in ((25, 3, False), (25, 0, True), (2, 0, True), (1, 0, False), (3, 1, True)):
        args = list(random_system(rng, m, 1, min(m, 2), n, n_missing=n_missing))
        if asym:
            args[2] = args[2] + 0.05 * rng.normal(size=(m, m))
        c, d = rng.normal(size=(m, 1)), rng.normal(size=(1, 1))
        for kind, strict, w, skip in (("standard", True, None, ()), ("standard", True, None, ("Z",)),
                                      ("single", True, None, ()), ("cholesky", False, rng.normal(size=n), ()),
                                      ("standard", False, rng.normal(size=n), ("Z", "H"))):
            ref = kn.kalman_filter(kind, *args, c=c, d=d, strict_reference=strict)
            outs, g, info = hostsim.run(kind, *args, c=c, d=d, strict=strict, static_dims=True, full=False, pred=True,
                                        p1=True, g_ll_obs=w, g_loglik=(0.0 if w is not None else None), skip=skip)
            assert info == 0 and abs(outs[4] - ref[4]) < 1e-12 * abs(ref[4])
            _, gt = kt.loglik_and_grads(kind, *args, c=c, d=d, strict_reference=strict, g_ll_obs=w)
            for k in gt:
                if k in skip:
                    continue
                assert rel_err(g[k], gt[k]) < 1e-9 or np.abs(g[k] - gt[k]).max() < 1e-13, (kind, n, k, g[k], gt[k])


def test_p1_short_form_adjoint_nile_fixture():
    """Diffuse start (P0 = 1e6 I): the reverse sweep loses ~9 digits to cancellation in its first steps whatever the
    formula (d logp / d P0 ~ 5e-7 next to T-bar ~ 2e6); the GPU tests hold every kernel to 1e-6 on this fixture.  The
    specialised adjoint drops two terms of the gain cotangent that cancel algebraically (kf_p1.cuh), which costs
    correlation with the forward pass's rounding: P0-bar 3e-7 here instead of 1e-9, everything else <= 3e-11."""
    for n_missing in (0, 5):
        args = nile_inputs(n_missing)
        outs, g, info = hostsim.run("standard", *args, static_dims=True, full=False, pred=True, p1=True)
        _, gt = kt.loglik_and_grads("standard", *args)
        for k in gt:
            assert rel_err(g[k], gt[k]) < (1e-6 if k == "P0" else 1e-10), (k, g[k], gt[k])


@pytest.mark.parametrize("static", [True, False], ids=["ThreadCtx", "CoopCtx"])
def test_non_symmetric_P0_multivariate_matches_reference_triangle_use(static):
    """ADVICE r1 (medium): BayesianVARMAX(stationary_initialization=False) hands the filter P0 = theta.reshape(m, m),
    which NUTS makes non-symmetric, so F_0 = Z P0 Z^T + H is non-symmetric.  The reference's StandardFilter then inverts
    the UPPER triangle (LAPACK posv, scipy default lower=False, kalman_filter.py:267-269) and takes log det of the FULL
    matrix (:281).  The kernels mirror both (ldl_inverse / lu_pivots); the oracle restates the reference's SciPy calls."""
    rng = np.random.default_rng(17)
    for (m, p, r) in ((3, 2, 2), (4, 3, 2)):
        args = list(random_system(rng, m, p, r, 12, n_missing=1))
        args[2] = args[2] + 0.1 * rng.normal(size=(m, m))
        for pred in (False, True):
            for strict in (True, False):
                ref = kn.kalman_filter("standard", *args, strict_reference=strict)
                outs, _, info = hostsim.run("standard", *args, strict=strict, static_dims=static, full=not pred, pred=pred,
                                            do_bwd=False)
                assert info == 0 and abs(outs[4] - ref[4]) < 1e-12 * abs(ref[4]), (m, p, pred, strict, outs[4], ref[4])
                if not pred:
                    for a, b in zip(outs[:4], ref[:4]):
                        assert rel_err(a, b) < 1e-11


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_structure_flags_give_identical_values(m):
    """KFB_FLAG_Z_UNIT0 / KFB_FLAG_H_ZERO: with Z = [1, 0, ..] (and H = 0) promised, the products with the known ones and
    zeros are not issued.  Values and cotangents must equal the unflagged kernels' (same operations on the remaining
    terms) and the oracle's; a false promise is reported, not silently used."""
    rng = np.random.default_rng(300 + m)
    for h_zero in (False, True):
        for n, n_missing in ((25, 3), (2, 0), (1, 0)):
            args = list(random_system(rng, m, 1, min(m, 2), n, n_missing=n_missing))
            args[4] = np.eye(m)[:1].copy()                       # Z = e_0
            if h_zero:
                args[6] = np.zeros((1, 1))
            args[2] = args[2] + 0.05 * rng.normal(size=(m, m))   # non-symmetric P0 (t = 0 runs the literal adjoint)
            c, d = rng.normal(size=(m, 1)), rng.normal(size=(1, 1))
            for w in (None, rng.normal(size=n)):
                kw = dict(c=c, d=d, static_dims=True, full=False, pred=True, p1=True, g_ll_obs=w,
                          g_loglik=(0.0 if w is not None else None), skip=("Z", "H"))
                o0, g0, i0 = hostsim.run("standard", *args, **kw)
                o1, g1, i1 = hostsim.run("standard", *args, z_unit0=True, h_zero=h_zero, **kw)
                assert i0 == 0 and i1 == 0 and abs(o1[4] - o0[4]) <= 1e-14 * abs(o0[4])
                _, gt = kt.loglik_and_grads("standard", *args, c=c, d=d, g_ll_obs=w)
                for k in gt:
                    if k in ("Z", "H"):
                        continue
                    assert rel_err(g1[k], g0[k]) < 1e-13 or np.abs(g1[k] - g0[k]).max() < 1e-14, (k, n, h_zero)
                    assert rel_err(g1[k], gt[k]) < 1e-9 or np.abs(g1[k] - gt[k]).max() < 1e-13, (k, n, h_zero)
    # a false promise: Z is not the unit vector / H is not zero
    args = list(random_system(rng, m, 1, 1, 6))
    _, _, info = hostsim.run("standard", *args, static_dims=True, full=False, pred=True, p1=True, z_unit0=True, do_bwd=False)
    assert info == 0x40000003
    args[4] = np.eye(m)[:1].copy()
    _, _, info = hostsim.run("standard", *args, static_dims=True, full=False, pred=True, p1=True, z_unit0=True, h_zero=True,
                             do_bwd=False)
    assert info == 0x40000003


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_companion_T_and_compressed_tape_on_host(m):
    """The device math of the two ARMA-family promises of round 2, compiled for the host (kf_p1.cuh, ZU = 2 / 3):
    KFB_FLAG_T_COMPANION (T = [t | e_0 .. e_{m-2}]: products with the unit columns not issued, only column 0 of T-bar) and,
    on complete data, the compressed tape (P_t = C + blockdiag(B_t, 0): a_t and the leading block of P_t only).  Same
    loglik and cotangents as the kernels with Z = e0 / H = 0 alone and as torch-autograd of the oracle; a T that is not a
    companion matrix, or a missing observation under the no-missing promise, is reported."""
    rng = np.random.default_rng(600 + m)
    for n, n_missing in ((25, 0), (25, 3), (2, 0), (1, 0)):
        args = list(random_system(rng, m, 1, 1, n, n_missing=n_missing))
        args[4] = np.eye(m)[:1].copy()                       # Z = e_0
        args[6] = np.zeros((1, 1))                           # H = 0
        Tc = np.zeros((m, m))
        Tc[:, 1:] = np.eye(m)[:, :m - 1]
        Tc[:, 0] = rng.uniform(-0.5, 0.5, size=m) / np.arange(1, m + 1)
        args[3] = Tc
        args[2] = args[2] + 0.05 * rng.normal(size=(m, m))   # non-symmetric P0
        c, d = rng.normal(size=(m, 1)), rng.normal(size=(1, 1))
        for w in (None, rng.normal(size=n)):
            kw = dict(c=c, d=d, static_dims=True, full=False, pred=True, p1=True, g_ll_obs=w,
                      g_loglik=(0.0 if w is not None else None), skip=("Z", "H"), z_unit0=True, h_zero=True)
            o0, g0, i0 = hostsim.run("standard", *args, **kw)
            variants = [dict(t_companion=True)] + ([dict(t_companion=True, no_missing=True)] if n_missing == 0 else [])
            _, gt = kt.loglik_and_grads("standard", *args, c=c, d=d, g_ll_obs=w)
            for extra in variants:
                o1, g1, i1 = hostsim.run("standard", *args, **kw, **extra)
                assert i0 == 0 and i1 == 0 and abs(o1[4] - o0[4]) <= 1e-13 * abs(o0[4]), (extra, n)
                for k in gt:
                    if k in ("Z", "H"):
                        continue
                    a, b, t = g1[k], g0[k], gt[k]
                    if k == "T":  # only the first column of a companion T carries parameters
                        assert m == 1 or np.abs(np.asarray(a).reshape(m, m)[:, 1:]).max() == 0.0
                        a, b, t = (np.asarray(v).reshape(m, m)[:, 0] for v in (a, b, t))
                    assert rel_err(a, b) < 1e-11 or np.abs(a - b).max() < 1e-13, (k, n, extra)
                    assert rel_err(a, t) < 1e-9 or np.abs(a - t).max() < 1e-13, (k, n, extra)
    # false promises
    args = list(random_system(rng, m, 1, 1, 6))
    args[4], args[6] = np.eye(m)[:1].copy(), np.zeros((1, 1))
    kw = dict(static_dims=True, full=False, pred=True, p1=True, z_unit0=True, h_zero=True, do_bwd=False)
    if m >= 2:  # a random T is not a companion matrix
        _, _, info = hostsim.run("standard", *args, t_companion=True, **kw)
        assert info == 0x40000003
    Tc = np.zeros((m, m))
    Tc[:, 1:] = np.eye(m)[:, :m - 1]
    Tc[:, 0] = 0.3 / np.arange(1, m + 1)
    args[3] = Tc
    args[0] = args[0].copy()
    args[0][3] = np.nan
    _, _, info = hostsim.run("standard", *args, t_companion=True, no_missing=True, **kw)
    assert info == 0x40000003
    _, _, info = hostsim.run("standard", *args, t_companion=True, **kw)
    assert info == 0


@pytest.mark.parametrize("m", [1, 2, 3])
def test_device_math_gradient_equals_autograd_of_dense_density(m):
    """The device step programs against an answer that shares nothing with them: torch-autograd of the dense
    multivariate-normal log-density of the stacked sample (oracle.kalman_torch.dense_gaussian_loglik) - not the restated
    recursion, not a hand-written adjoint.  Generic thread-per-unit math (all nine cotangents, missing rows, k_endog 1 and
    2) and the ARMA-family reduced recursion of kf_p1.cuh (Z = e0, H = 0, companion T, complete data)."""
    rng = np.random.default_rng(800 + m)
    sym = lambda k, g: 0.5 * (g + g.T) if k in ("P0", "H", "Q") else g  # noqa: E731
    for p in (1, 2)[:m]:  # thread-per-unit instantiations exist for k_endog <= k_states
        args = random_system(rng, m, p, min(m, 2), 16, n_missing=2)
        c, d = rng.normal(size=(m, 1)), rng.normal(size=(p, 1))
        ll, gd = kt.dense_loglik_and_grads(*args, c=c, d=d)
        outs, g, info = hostsim.run("standard", *args, c=c, d=d, strict=False, static_dims=True)
        assert info == 0 and abs(outs[4] - ll) < 1e-11 * abs(ll)
        for k in gd:
            a, b = sym(k, np.asarray(g[k]).reshape(gd[k].shape)), sym(k, gd[k])
            assert rel_err(a, b) < 1e-9 or np.abs(a - b).max() < 1e-13, (p, k)
    # ARMA family: the four structure promises -> reduced recursion, 16-byte tape entries at k_states 2
    args = list(random_system(rng, m, 1, 1, 20))
    args[4], args[6] = np.eye(m)[:1].copy(), np.zeros((1, 1))
    Tc = np.zeros((m, m))
    Tc[:, 1:] = np.eye(m)[:, :m - 1]
    Tc[:, 0] = rng.uniform(-0.5, 0.5, size=m) / np.arange(1, m + 1)
    args[3] = Tc
    ll, gd = kt.dense_loglik_and_grads(*args)
    outs, g, info = hostsim.run("standard", *args, static_dims=True, full=False, pred=True, p1=True, skip=("Z", "H"),
                                z_unit0=True, h_zero=True, t_companion=True, no_missing=True)
    assert info == 0 and abs(outs[4] - ll) < 1e-11 * abs(ll)
    for k in ("a0", "P0", "T", "R", "Q"):
        a, b = sym(k, np.asarray(g[k]).reshape(gd[k].shape)), sym(k, gd[k])
        if k == "T":
            a, b = a[:, 0], b[:, 0]
        assert rel_err(a, b) < 1e-9 or np.abs(a - b).max() < 1e-13, ("reduced", k)


def test_device_math_moments_and_smoother_equal_dense_conditional_moments():
    """Full-output device math (filtered / predicted moments) and the device RTS smoother, compiled for the host, against
    the dense conditional moments of the joint Gaussian (oracle.kalman_numpy.dense_gaussian_state_moments) - a known answer
    that shares no recursion with them."""
    rng = np.random.default_rng(77)
    for (m, p, r), static in (((2, 1, 1), True), ((3, 2, 2), True), ((4, 3, 2), False)):
        n = 10
        args = random_system(rng, m, p, r, n, n_missing=2)
        d = rng.normal(size=(p, 1))
        cond = kn.dense_gaussian_state_moments(*args, d=d)
        outs, _, info = hostsim.run("standard", *args, d=d, strict=False, static_dims=static, do_bwd=False)
        assert info == 0
        fs, ps, fc, pc = outs[:4]
        for t in range(n):
            for (got_a, got_P), (a, P) in (((fs[t], fc[t]), cond(t, t)), ((ps[t + 1], pc[t + 1]), cond(t + 1, t))):
                assert rel_err(got_a, a) < 1e-10 and rel_err(got_P, P) < 1e-10, (m, t)
        ss, sc = hostsim.smoother(args[3], args[5], args[7], fs, fc)
        ss = ss[..., 0]
        for t in range(n):
            a, P = cond(t, n - 1)
            assert rel_err(ss[t], a[:, 0]) < 1e-10 and rel_err(sc[t], P) < 1e-10, (m, t)


@pytest.mark.parametrize("static", [True, False], ids=["ThreadCtx", "CoopCtx"])
def test_device_math_time_varying_loglik_equals_dense_density(static):
    """Row f3 on the device math: time-varying T, Z, R, H, Q, c, d against the dense density of the stacked sample."""
    rng = np.random.default_rng(11)
    n, m, p, r = 12, 3, 2, 2
    systems = [random_system(rng, m, p, r, n, n_missing=2) for _ in range(n)]
    y, a0, P0 = systems[0][:3]
    T, Z, R, H, Q = (np.stack([s[i] for s in systems]) for i in range(3, 8))
    c, d = rng.normal(size=(n, m, 1)), rng.normal(size=(n, p, 1))
    dense = kn.dense_gaussian_loglik_time_varying(y, a0, P0, T, Z, R, H, Q, c, d)
    outs, _, info = hostsim.run("standard", y, a0, P0, T, Z, R, H, Q, c=c, d=d, strict=False, static_dims=static, do_bwd=False)
    assert info == 0 and abs(outs[4] - dense) < 1e-10 * abs(dense)
    # all six outputs and every cotangent of the time-varying instantiation against the oracle (strict and corrected)
    _check("standard", (y, a0, P0, T, Z, R, H, Q), c, d, True, static)
    _check("standard", (y, a0, P0, T, Z, R, H, Q), c, d, False, static, w=rng.normal(size=n))


def test_device_math_steady_state_gradient_equals_dense_density_at_the_riccati_fixed_point():
    """Steady-state device math (forward + adjoint incl. the P_ss / F^-1 cotangents chained through the DARE adjoint)
    against autograd of [unrolled Riccati iteration -> dense density started at P_ss] - no shared recursion or adjoint."""
    import torch

    rng = np.random.default_rng(21)
    sym = lambda k, a: 0.5 * (a + a.T) if k in ("H", "Q") else a  # noqa: E731
    for (m, p, r), static in (((2, 1, 1), True), ((4, 2, 2), True), ((4, 3, 2), False)):
        args = list(random_system(rng, m, p, r, 14))
        names = ("a0", "P0", "T", "Z", "R", "H", "Q")
        ins = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in zip(names, args[1:])}
        T, Z, R, H, Q = (ins[k] for k in ("T", "Z", "R", "H", "Q"))
        lld = kt.dense_gaussian_loglik(args[0], ins["a0"], kt.dare_by_riccati_iteration(T, Z, R @ Q @ R.T, H), T, Z, R, H, Q)
        gs = dict(zip(names, torch.autograd.grad(lld, [ins[k] for k in names], allow_unused=True)))
        outs, g, info = hostsim.run("steady_state", *args, strict=False, static_dims=static)
        assert info == 0 and abs(outs[4] - float(lld.detach())) < 1e-10 * abs(outs[4])
        for k in ("a0", "T", "Z", "R", "H", "Q"):
            a, b = sym(k, np.asarray(g[k]).reshape(gs[k].shape)), sym(k, gs[k].numpy())
            assert rel_err(a, b) < 1e-7, (m, k)  # 1e-7: the tolerance of every steady-state gradient test (DESIGN section 2)
