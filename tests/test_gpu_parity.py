"""GPU parity: CUDA kernels (through the C ABI) vs the CPU oracle on identical seeded inputs.

Tolerance: rtol 1e-8 in float64 (BASELINE.json north_star) on logp, per-step ll, filtered / predicted
moments and every gradient.  Sizes are small enough for the per-step Python oracle to finish in seconds.
"""
import numpy as np
import pytest
import torch

from oracle import kalman_numpy as kn
from oracle import kalman_torch as kt
from tests.helpers import make_test_inputs, nile_inputs, random_system, rel_err

pytestmark = pytest.mark.gpu

RTOL = 1e-8
ALL_OUT = ("filtered_states", "predicted_states", "filtered_covs", "predicted_covs", "loglik", "ll_obs")


def _dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device="cuda")


def run_single(kind, args, c=None, d=None, strict=True, force_coop=False, time_varying=(), bwd=True, g_ll_obs=None):
    """One unit through BatchedKalman; returns (outs, grads) as numpy in reference shapes."""
    from pymc_statespace_b200 import BatchedKalman

    y, a0, P0, T, Z, R, H, Q = args
    n, p = y.shape[0], y.shape[1]
    m, r = T.shape[-1], R.shape[-1]
    bk = BatchedKalman(kind, n, m, p, r, n_draws=1, strict_reference=strict, force_coop=force_coop,
                       time_varying=time_varying)

    def prep(name, x):
        if x is None:
            return None
        x = np.asarray(x, dtype=float)
        return _dev(x[None]) if name not in () else _dev(x)

    ins = {k: prep(k, v) for k, v in zip(("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d"), (a0, P0, T, Z, R, H, Q, c, d))}
    out = bk.forward(_dev(y[..., 0]), **ins, outputs=ALL_OUT, save_for_backward=bwd)
    torch.cuda.synchronize()
    res = [out["filtered_states"][0].cpu().numpy()[..., None], out["predicted_states"][0].cpu().numpy()[..., None],
           out["filtered_covs"][0].cpu().numpy(), out["predicted_covs"][0].cpu().numpy(),
           float(out["loglik"][0]), out["ll_obs"][0].cpu().numpy()]
    info = int(out["info"][0])
    grads = None
    if bwd:
        gl = None if g_ll_obs is None else _dev(np.zeros(1))
        glo = None if g_ll_obs is None else _dev(np.asarray(g_ll_obs)[None])
        g = bk.backward(g_loglik=gl, g_ll_obs=glo)
        torch.cuda.synchronize()
        grads = {k: v[0].cpu().numpy() for k, v in g.items()}
        for k in ("a0", "c", "d"):
            grads[k] = grads[k][..., None]
    return res, grads, info


def check_against_oracle(kind, args, c=None, d=None, strict=True, force_coop=False, time_varying=(), g_ll_obs=None,
                         rtol=RTOL, grad_rtol=RTOL):
    ref = kn.kalman_filter(kind, *args, c=c, d=d, strict_reference=strict)
    res, grads, info = run_single(kind, args, c, d, strict, force_coop, time_varying, True, g_ll_obs)
    assert info == 0
    for name, a, b in zip(ALL_OUT, res, ref):
        assert rel_err(a, b) < rtol, (kind, name, rel_err(a, b))
    _, gref = kt.loglik_and_grads(kind, *args, c=c, d=d, strict_reference=strict, g_ll_obs=g_ll_obs)
    for k in gref:
        scale = max(np.abs(gref[k]).max(), 1e-12 * max(np.abs(v).max() for v in gref.values()))
        assert np.abs(grads[k] - gref[k]).max() / scale < grad_rtol, (kind, k, np.abs(grads[k] - gref[k]).max() / scale)


KINDS_P1 = ["standard", "cholesky", "single", "univariate"]


@pytest.mark.parametrize("force_coop", [False, True], ids=["thread", "coop"])
@pytest.mark.parametrize("kind", KINDS_P1)
@pytest.mark.parametrize("n_missing", [0, 5])
def test_nile_local_linear_trend(kind, n_missing, force_coop):
    # the fixture of reference tests/test_kalman_filter.py:226-241 (m=2, p=1, P0 = 1e6 I)
    # Forward moments / logp: rtol 1e-8.  Gradients: P0 = 1e6 I makes the first updates cancel ~6 digits
    # (P - K K^T F in the univariate filter), so oracle and kernel - both float64, different rounding order -
    # agree to ~1e-7 on the tiny dlogp/dP0 entries; the reference's own tolerance on this fixture is
    # rtol = atol = 1e-7 (tests/test_kalman_filter.py:241).
    check_against_oracle(kind, nile_inputs(n_missing), force_coop=force_coop, grad_rtol=1e-6)


@pytest.mark.parametrize("force_coop", [False, True], ids=["thread", "coop"])
@pytest.mark.parametrize("kind", ["standard", "univariate"])
@pytest.mark.parametrize("dims", [(1, 1, 1), (2, 1, 1), (2, 2, 1), (3, 2, 2), (3, 3, 3), (4, 1, 2), (4, 3, 2)],
                         ids=lambda d: "m%dp%dr%d" % d)
def test_random_systems_with_intercepts(kind, dims, force_coop):
    m, p, r = dims
    rng = np.random.default_rng(100 * m + 10 * p + r)
    args = random_system(rng, m, p, r, 40, n_missing=4)
    c, d = rng.normal(size=(m, 1)), rng.normal(size=(p, 1))
    check_against_oracle(kind, args, c, d, strict=True, force_coop=force_coop)
    check_against_oracle(kind, args, c, d, strict=False, force_coop=force_coop,
                         g_ll_obs=rng.normal(size=40))


@pytest.mark.parametrize("dims", [(6, 3, 3), (5, 5, 1), (9, 2, 4)], ids=lambda d: "m%dp%dr%d" % d)
@pytest.mark.parametrize("kind", ["standard", "univariate"])
def test_larger_systems_coop(kind, dims):
    m, p, r = dims
    rng = np.random.default_rng(7 + m)
    args = random_system(rng, m, p, r, 30, n_missing=3, scale_T=0.25)
    check_against_oracle(kind, args)


def test_cta_per_unit_mode():
    # arena too large for 4 warps per SM -> one CTA per unit
    m, p, r = 30, 1, 3
    rng = np.random.default_rng(3)
    args = random_system(rng, m, p, r, 12, n_missing=1, scale_T=0.1)
    check_against_oracle("standard", args)
    check_against_oracle("univariate", args)


def test_univariate_partial_missing():
    rng = np.random.default_rng(11)
    args = random_system(rng, 4, 3, 2, 40, n_missing=3, partial=True, diag_H=True)
    check_against_oracle("univariate", args, force_coop=False)
    check_against_oracle("univariate", args, force_coop=True)


def test_partial_missing_flags_info_in_standard():
    rng = np.random.default_rng(12)
    args = list(random_system(rng, 3, 2, 2, 20))
    args[0][7, 1] = np.nan
    res, _, info = run_single("standard", args, bwd=False)
    assert info == -(7 + 1) and np.isnan(res[4])


def test_time_varying_matrices():
    # reference tests/test_kalman_filter.py:102-156 (shapes only there; values here)
    rng = np.random.default_rng(5)
    n, m, p, r = 12, 3, 2, 2
    sys_t = [random_system(rng, m, p, r, n) for _ in range(n)]
    y, a0, P0 = sys_t[0][:3]
    T, Z, R, H, Q = (np.stack([s[i] for s in sys_t]) for i in range(3, 8))
    c, d = rng.normal(size=(n, m, 1)), rng.normal(size=(n, p, 1))
    for force_coop in (False, True):  # thread-per-unit kernels with per-step reloads (ThreadCtx<M,P,true>) / generic cooperative
        check_against_oracle("standard", (y, a0, P0, T, Z, R, H, Q), c, d, force_coop=force_coop,
                             time_varying=("T", "Z", "R", "H", "Q", "c", "d"))
        # only some matrices time varying
        check_against_oracle("standard", (y, a0, P0, T, sys_t[0][4], sys_t[0][5], H, sys_t[0][7]), force_coop=force_coop,
                             time_varying=("T", "H"))
    # k_endog = 1 (the specialised static kernels must NOT be picked) with missing rows and a per-step ll cotangent
    n, m, p, r = 15, 2, 1, 1
    sys_t = [random_system(rng, m, p, r, n, n_missing=2) for _ in range(n)]
    y, a0, P0 = sys_t[0][:3]
    T, Q = (np.stack([s[i] for s in sys_t]) for i in (3, 7))
    check_against_oracle("standard", (y, a0, P0, T, sys_t[0][4], sys_t[0][5], sys_t[0][6], Q), time_varying=("T", "Q"),
                         g_ll_obs=rng.normal(size=n))


@pytest.mark.parametrize("p,m,r,n", [(1, 1, 1, 10), (1, 2, 2, 10), (1, 5, 2, 10), (1, 5, 1, 10), (5, 5, 1, 10)])
@pytest.mark.parametrize("kind", ["standard", "univariate"])
def test_reference_shape_fixtures(kind, p, m, r, n):
    # make_test_inputs of reference tests/utilities/test_helpers.py:62-76 incl. missing data (:192-209)
    for missing in (None, 1):
        args = make_test_inputs(p, m, r, n, missing_data=missing)
        ref = kn.kalman_filter(kind, *args)
        res, _, info = run_single(kind, args, bwd=False)
        assert info == 0
        for name, a, b in zip(ALL_OUT, res, ref):
            assert np.asarray(a).shape == np.asarray(b).shape
            assert not np.any(np.isnan(a))
            assert rel_err(a, b) < RTOL, (name, rel_err(a, b))


def test_batched_draws_and_series_match_unit_runs():
    from pymc_statespace_b200 import BatchedKalman

    rng = np.random.default_rng(21)
    B, S, n, m, p, r = 37, 3, 50, 2, 1, 1
    systems = [random_system(rng, m, p, r, n) for _ in range(B)]
    ys = np.stack([random_system(rng, m, p, r, n, n_missing=3)[0][..., 0] for _ in range(S)])
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    bk = BatchedKalman("standard", n, m, p, r, n_draws=B, n_series=S)
    out = bk.forward(_dev(ys), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7),
                     outputs=("loglik",), save_for_backward=True)
    g = bk.backward()
    ll = out["loglik"].cpu().numpy().reshape(B, S)
    gT = g["T"].cpu().numpy().reshape(B, S, m, m)
    for b in (0, 17, 36):
        for s in range(S):
            args = (ys[s][..., None],) + tuple(systems[b][1:])
            ref = kn.kalman_filter("standard", *args)[4]
            assert abs(ll[b, s] - ref) < RTOL * abs(ref)
            _, gref = kt.loglik_and_grads("standard", *args)
            assert rel_err(gT[b, s], gref["T"]) < RTOL


def test_lyapunov_forward_backward():
    import scipy.linalg

    from pymc_statespace_b200 import lyapunov_backward, lyapunov_forward

    rng = np.random.default_rng(4)
    B, m, r = 33, 5, 2
    A = rng.normal(size=(B, m, m))
    A *= (rng.uniform(0.2, 0.97, size=B) / np.abs(np.linalg.eigvals(A)).max(axis=1))[:, None, None]
    R = rng.normal(size=(B, m, r))
    L = rng.normal(size=(B, r, r))
    Q = L @ L.transpose(0, 2, 1) + 0.1 * np.eye(r)
    X, info = lyapunov_forward(_dev(A), _dev(R), _dev(Q))
    assert int(info.abs().sum()) == 0
    Xn = X.cpu().numpy()
    for b in range(B):
        ref = scipy.linalg.solve_discrete_lyapunov(A[b], R[b] @ Q[b] @ R[b].T, method="bilinear")
        assert rel_err(Xn[b], ref) < RTOL
    Xbar = rng.normal(size=(B, m, m))
    Ab, Rb, Qb = (torch.zeros_like(_dev(x)) for x in (A, R, Q))
    lyapunov_backward(_dev(A), _dev(R), _dev(Q), X, _dev(Xbar), Ab, Rb, Qb)
    for b in (0, 5, 32):
        At, Rt, Qt = (torch.tensor(x[b], requires_grad=True) for x in (A, R, Q))
        Xt = kt.solve_discrete_lyapunov(At, Rt @ Qt @ Rt.T)
        (Xt * torch.tensor(Xbar[b])).sum().backward()
        assert rel_err(Ab[b].cpu().numpy(), At.grad.numpy()) < 1e-7
        assert rel_err(Rb[b].cpu().numpy(), Rt.grad.numpy()) < 1e-7
        assert rel_err(Qb[b].cpu().numpy(), Qt.grad.numpy()) < 1e-7


@pytest.mark.parametrize("force_coop", [False, True], ids=["thread", "coop"])
@pytest.mark.parametrize("strict", [True, False])
@pytest.mark.parametrize("dims", [(2, 1, 1), (4, 2, 2)], ids=lambda d: "m%dp%dr%d" % d)
def test_steady_state_filter(dims, strict, force_coop):
    # SteadyStateFilter: on-GPU DARE (Riccati + Newton-Hewer) + fixed-gain recursion + DARE adjoint
    m, p, r = dims
    rng = np.random.default_rng(40 + m)
    args = random_system(rng, m, p, r, 30)
    d = rng.normal(size=(p, 1))
    check_against_oracle("steady_state", args, None, d, strict=strict, force_coop=force_coop, rtol=1e-8, grad_rtol=1e-7)


def test_steady_state_nile_and_trend_seasonal():
    from pymc_statespace_b200.models import trend_seasonal_spec

    check_against_oracle("steady_state", nile_inputs(0), grad_rtol=1e-6)
    mats = trend_seasonal_spec(29).matrices(np.array([0.1, 0.01, 0.05, 0.5]))
    rng = np.random.default_rng(0)
    y = rng.normal(size=(40, 1, 1))
    args = (y, mats["a0"], mats["P0"], mats["T"], mats["Z"], mats["R"], mats["H"], mats["Q"])
    check_against_oracle("steady_state", args, rtol=1e-8, grad_rtol=1e-6)


@pytest.mark.parametrize("dims", [(4, 2, 2), (6, 3, 3)], ids=lambda d: "m%dp%dr%d" % d)
def test_as_coded_cholesky_filter_multivariate(dims):
    # SURVEY A.2-Q4: CholeskyFilter as coded (second triangular solve reads only diag(L)) for k_endog > 1
    m, p, r = dims
    rng = np.random.default_rng(60 + m)
    args = random_system(rng, m, p, r, 30, n_missing=3)
    check_against_oracle("cholesky", args, rng.normal(size=(m, 1)), rng.normal(size=(p, 1)), strict=True)


@pytest.mark.parametrize("dims", [(5, 1, 2), (6, 3, 3), (7, 2, 3), (8, 3, 2)], ids=lambda d: "m%dp%dr%d" % d)
@pytest.mark.parametrize("kind", ["standard", "univariate", "steady_state"])
def test_subwarp_static_kernels(kind, dims):
    """CoopCtxT<M,P,8>: 8 lanes per unit, 4 units per warp, compile-time dims (k_states 5..8)."""
    m, p, r = dims
    rng = np.random.default_rng(90 + 10 * m + p)
    miss = 0 if kind == "steady_state" else 3
    args = random_system(rng, m, p, r, 30, n_missing=miss, scale_T=0.25)
    c, d = rng.normal(size=(m, 1)), rng.normal(size=(p, 1))
    check_against_oracle(kind, args, c, d, grad_rtol=1e-7 if kind == "steady_state" else RTOL)
    # and the generic cooperative kernels give the same numbers
    check_against_oracle(kind, args, c, d, force_coop=True, grad_rtol=1e-7 if kind == "steady_state" else RTOL)


def test_subwarp_kernels_many_units_not_multiple_of_group():
    # 37 units: the last warp holds a partial set of 8-lane groups (active-mask sync)
    from pymc_statespace_b200 import BatchedKalman

    rng = np.random.default_rng(5)
    B, n, m, p, r = 37, 25, 6, 3, 3
    systems = [random_system(rng, m, p, r, n, scale_T=0.25) for _ in range(B)]
    y = random_system(rng, m, p, r, n, n_missing=3)[0]
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    for kind in ("standard", "univariate"):
        bk = BatchedKalman(kind, n, m, p, r, n_draws=B)
        out = bk.forward(_dev(y[..., 0]), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7),
                         outputs=("loglik",), save_for_backward=True)
        g = bk.backward()
        ll = out["loglik"].cpu().numpy()
        for b in (0, 31, 32, 36):
            args = (y,) + tuple(systems[b][1:])
            ref, gref = kt.loglik_and_grads(kind, *args)
            assert abs(ll[b] - ref) < RTOL * abs(ref)
            assert rel_err(g["T"][b].cpu().numpy(), gref["T"]) < RTOL
            assert rel_err(g["Q"][b].cpu().numpy(), gref["Q"]) < RTOL


@pytest.mark.parametrize("wrt", [("a0", "P0", "T", "R", "H", "Q", "c", "d"), ("a0", "P0", "R", "H", "Q", "c", "d"), ("H", "Q")],
                         ids=["with_Tbar", "no_Tbar", "HQ_only"])
@pytest.mark.parametrize("dims", [(5, 1, 2), (5, 3, 2), (6, 2, 3), (6, 3, 3), (7, 3, 2), (8, 1, 1), (8, 3, 3), (30, 1, 3),
                                  (18, 1, 2), (20, 1, 1), (22, 1, 3), (24, 1, 2), (26, 1, 2), (28, 1, 3), (32, 1, 2),
                                  (10, 1, 2), (12, 1, 3), (14, 1, 1), (16, 1, 2)],
                         ids=lambda d: "m%dp%dr%d" % d)
def test_fused_row_kernels_hot_path(dims, wrt):
    """The theta-level hot path of mid-size / large systems: loglik-only forward + adjoint WITHOUT Z-bar go through the
    fused row kernels (kf_rows.cuh: 4 lanes x 2 rows, k_states 5..8; kf_rowsD.cuh: warp per unit, k_states 10..32), with and
    without T-bar (separate instantiations / code paths).  13 units: partial last warp; shared y with missing rows."""
    from pymc_statespace_b200 import BatchedKalman

    m, p, r = dims
    rng = np.random.default_rng(1000 + 10 * m + p)
    B, n = 13, 24
    systems = [random_system(rng, m, p, r, n, scale_T=0.25 if m < 10 else 0.1) for _ in range(B)]
    y = random_system(rng, m, p, r, n, n_missing=3)[0]
    cs, ds = rng.normal(size=(B, m)), rng.normal(size=(B, p))
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    bk = BatchedKalman("standard", n, m, p, r, n_draws=B)
    out = bk.forward(_dev(y[..., 0]), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7),
                     c=_dev(cs), d=_dev(ds), outputs=("loglik",), save_for_backward=True)
    w = rng.normal(size=B)
    g = bk.backward(g_loglik=_dev(w), wrt=wrt)
    assert int(out["info"].abs().max()) == 0
    ll = out["loglik"].cpu().numpy()
    for b in (0, 7, 8, 12):
        args = (y,) + tuple(systems[b][1:])
        ref, gref = kt.loglik_and_grads("standard", *args, c=cs[b][:, None], d=ds[b][:, None])
        assert abs(ll[b] - ref) < RTOL * abs(ref)
        for k in wrt:
            got = g[k][b].cpu().numpy().reshape(gref[k].shape)
            scale = max(np.abs(gref[k]).max(), 1e-12)
            assert np.abs(got - w[b] * gref[k]).max() / (abs(w[b]) * scale) < RTOL, (k, b)
    # cotangent on the per-step log-likelihoods instead (g_loglik = 0): the same kernels with lb = g_ll_obs[u, t]
    wt = rng.normal(size=(B, n))
    g2 = bk.backward(g_loglik=_dev(np.zeros(B)), g_ll_obs=_dev(wt), wrt=wrt)
    for b in (0, 12):
        args = (y,) + tuple(systems[b][1:])
        _, gref = kt.loglik_and_grads("standard", *args, c=cs[b][:, None], d=ds[b][:, None], g_ll_obs=wt[b])
        for k in wrt:
            got = g2[k][b].cpu().numpy().reshape(gref[k].shape)
            scale = max(np.abs(gref[k]).max(), 1e-12)
            assert np.abs(got - gref[k]).max() / scale < RTOL, ("g_ll_obs", k, b)


@pytest.mark.parametrize("wrt", [("a0", "T", "R", "H", "Q", "c", "d"), ("R", "H", "Q")], ids=["with_Tbar", "no_Tbar"])
@pytest.mark.parametrize("dims", [(30, 1, 3), (6, 3, 3), (5, 1, 2), (8, 2, 2), (18, 1, 2), (24, 1, 3), (10, 1, 2), (16, 1, 3)],
                         ids=lambda d: "m%dp%dr%d" % d)
def test_fused_row_kernels_steady_state(dims, wrt):
    """SteadyStateFilter through the fused row kernels (MK_STEADY instantiations of kf_rows.cuh for k_states 5..8 and of the
    tensor-core kf_rowsD.cuh for k_states = 30) + DARE kernels; no Z-bar."""
    from pymc_statespace_b200 import BatchedKalman

    m, p, r = dims
    rng = np.random.default_rng(77 + m)
    B, n = 11, 20
    systems = [random_system(rng, m, p, r, n, scale_T=0.1 if m >= 10 else 0.25) for _ in range(B)]
    y = systems[0][0]
    cs, ds = rng.normal(size=(B, m)), rng.normal(size=(B, p))
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    bk = BatchedKalman("steady_state", n, m, p, r, n_draws=B)
    out = bk.forward(_dev(y[..., 0]), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7),
                     c=_dev(cs), d=_dev(ds), outputs=("loglik",), save_for_backward=True)
    g = bk.backward(wrt=wrt)
    assert int(out["info"].abs().max()) == 0
    ll = out["loglik"].cpu().numpy()
    for b in (0, 10):
        args = (y,) + tuple(systems[b][1:])
        ref, gref = kt.loglik_and_grads("steady_state", *args, c=cs[b][:, None], d=ds[b][:, None])
        assert abs(ll[b] - ref) < RTOL * abs(ref)
        for k in wrt:
            got = g[k][b].cpu().numpy().reshape(gref[k].shape)
            scale = max(np.abs(gref[k]).max(), 1e-12)
            assert np.abs(got - gref[k]).max() / scale < 1e-7, (k, b)  # DARE adjoint: 1e-7 as in the other steady tests


@pytest.mark.parametrize("n", [1, 2])
@pytest.mark.parametrize("dims", [(6, 3, 3), (30, 1, 3), (12, 1, 2)], ids=lambda d: "m%dp%dr%d" % d)
def test_fused_row_kernels_very_short_series(dims, n):
    """n = 1: no tape at all; n = 2: a single tape entry (the prefetch / double-buffer edge cases of the fused kernels)."""
    from pymc_statespace_b200 import BatchedKalman

    m, p, r = dims
    rng = np.random.default_rng(300 + m + n)
    B = 3
    systems = [random_system(rng, m, p, r, n, scale_T=0.1 if m >= 10 else 0.25) for _ in range(B)]
    y = systems[0][0]
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    for kind in ("standard", "steady_state"):
        bk = BatchedKalman(kind, n, m, p, r, n_draws=B)
        out = bk.forward(_dev(y[..., 0]), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7),
                         outputs=("loglik",), save_for_backward=True)
        wrt = ("a0", "P0", "T", "R", "H", "Q") if kind == "standard" else ("a0", "T", "R", "H", "Q")
        g = bk.backward(wrt=wrt)
        ll = out["loglik"].cpu().numpy()
        for b in range(B):
            ref, gref = kt.loglik_and_grads(kind, y, *systems[b][1:])
            assert abs(ll[b] - ref) < RTOL * abs(ref)
            for k in wrt:
                got = g[k][b].cpu().numpy().reshape(gref[k].shape)
                scale = max(np.abs(gref[k]).max(), 1e-12)
                assert np.abs(got - gref[k]).max() / scale < (1e-7 if kind == "steady_state" else RTOL), (kind, k, b)


@pytest.mark.parametrize("force_coop", [False, True], ids=["thread", "coop"])
@pytest.mark.parametrize("n", [1, 2, 3])
def test_very_short_series(n, force_coop):
    # n = 1: no tape at all; n = 2: one tape entry; the ring read-ahead must not run past the start
    rng = np.random.default_rng(n)
    for kind, (m, p, r) in (("standard", (2, 1, 1)), ("univariate", (3, 2, 2)), ("steady_state", (2, 1, 1))):
        args = random_system(rng, m, p, r, n)
        check_against_oracle(kind, args, force_coop=force_coop, grad_rtol=1e-7 if kind == "steady_state" else RTOL)


def test_all_rows_missing_and_first_last_missing():
    rng = np.random.default_rng(2)
    args = list(random_system(rng, 2, 1, 1, 12))
    y = args[0].copy()
    y[[0, 11]] = np.nan
    args[0] = y
    for kind in ("standard", "univariate", "single"):
        check_against_oracle(kind, args)
    args[0] = np.full_like(y, np.nan)
    res, grads, info = run_single("standard", args)
    ref = kn.kalman_filter("standard", *args)
    assert info == 0 and res[4] == 0.0 and ref[4] == 0.0
    for a, b in zip(res[:4], ref[:4]):
        assert rel_err(a, b) < RTOL
    assert all(np.all(np.isfinite(g)) for g in grads.values())


def test_more_observables_than_states_and_wide_p():
    # k_endog > k_states and k_endog = 5 have no compile-time instantiation: generic cooperative kernels
    rng = np.random.default_rng(9)
    for (m, p, r) in ((1, 2, 1), (2, 5, 2), (3, 4, 1)):
        args = random_system(rng, m, p, r, 20, n_missing=2)
        check_against_oracle("standard", args)
        check_against_oracle("univariate", args)


def test_units_not_multiple_of_block_and_per_series_y():
    from pymc_statespace_b200 import BatchedKalman

    rng = np.random.default_rng(33)
    B, S, n, m, p, r = 67, 2, 30, 2, 1, 1  # 134 units: 2 full 64-thread CTAs + 6 threads
    systems = [random_system(rng, m, p, r, n) for _ in range(B)]
    ys = np.stack([random_system(rng, m, p, r, n, n_missing=2)[0][..., 0] for _ in range(S)])
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    for force in (False, True):
        bk = BatchedKalman("standard", n, m, p, r, n_draws=B, n_series=S, force_coop=force)
        out = bk.forward(_dev(ys), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7),
                         outputs=("loglik",), save_for_backward=True)
        g = bk.backward(wrt=("T", "a0"))
        ll = out["loglik"].cpu().numpy().reshape(B, S)
        for b, s in ((0, 0), (66, 1), (31, 1)):
            args = (ys[s][..., None],) + tuple(systems[b][1:])
            ref, gref = kt.loglik_and_grads("standard", *args)
            assert abs(ll[b, s] - ref) < RTOL * abs(ref)
            assert rel_err(g["T"].cpu().numpy().reshape(B, S, m, m)[b, s], gref["T"]) < RTOL


def test_invalid_requests_raise():
    from pymc_statespace_b200 import BatchedKalman
    from pymc_statespace_b200._lib import KfbError

    bk = BatchedKalman("standard", 10, 2, 1, 1, n_draws=4)
    z = lambda *s: torch.zeros(*s, dtype=torch.float64, device="cuda")  # noqa: E731
    with pytest.raises(ValueError):
        bk.forward(z(10, 1), z(3, 2), z(4, 2, 2), z(2, 2), z(1, 2), z(2, 1), z(1, 1), z(1, 1))  # a0 batch 3 != 4
    with pytest.raises(TypeError):
        bk.forward(z(10, 1).float(), z(2), z(2, 2), z(2, 2), z(1, 2), z(2, 1), z(1, 1), z(1, 1))
    with pytest.raises(RuntimeError, match="save_for_backward"):
        bk.backward()
    with pytest.raises(KfbError, match="invalid argument"):
        BatchedKalman("single", 10, 2, 2, 1, n_draws=1).forward(z(10, 2), z(2), z(2, 2), z(2, 2), z(2, 2), z(2, 1),
                                                                z(2, 2), z(1, 1))


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_adjoint_kernel_vs_generic_and_oracle(m):
    """kf_p1.cu (k_endog = 1: branch-free forward, TMA tape ring + symmetric-storage adjoint) against the generic
    thread-per-unit kernels (KFB_FLAG_GENERIC_ADJOINT) on every unit, and against torch-autograd of the oracle on a few: 77 units (two full
    warps + 13 lanes), missing rows, non-symmetric P0, every cotangent subset that selects a different instantiation."""
    from pymc_statespace_b200 import BatchedKalman

    rng = np.random.default_rng(40 + m)
    B, n, r = 77, 37, min(m, 2)
    systems = [list(random_system(rng, m, 1, r, n)) for _ in range(B)]
    for s in systems:
        s[2] = s[2] + 0.05 * rng.normal(size=(m, m))  # P0 as BayesianARMA(stationary_initialization=False) writes it
    y = random_system(rng, m, 1, r, n, n_missing=4)[0]
    y[[0, n - 1]] = np.nan
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    c, d = _dev(rng.normal(size=(B, m))), _dev(rng.normal(size=(B, 1)))
    w = rng.normal(size=(B, n))
    for kind, strict in (("standard", True), ("single", True), ("cholesky", False)):
        for wrt, gobs in ((("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d"), None), (("a0", "P0", "T", "R", "Q"), None),
                          (("T", "H", "Q", "d"), w), (("a0", "Z"), w)):
            res = {}
            for gen in (False, True):
                bk = BatchedKalman(kind, n, m, 1, r, n_draws=B, strict_reference=strict, generic_adjoint=gen)
                out = bk.forward(_dev(y[..., 0]), stack(1)[..., 0], stack(2), stack(3), stack(4), stack(5), stack(6),
                                 stack(7), c, d, outputs=("loglik",), save_for_backward=True)
                g = bk.backward(g_loglik=None if gobs is None else _dev(np.full(B, 0.5)),
                                g_ll_obs=None if gobs is None else _dev(gobs), wrt=wrt)
                assert int((out["info"] != 0).sum()) == 0
                res[gen] = {k: v.cpu().numpy() for k, v in g.items()}
                res[gen]["loglik"] = out["loglik"].cpu().numpy()
            assert np.abs(res[False]["loglik"] / res[True]["loglik"] - 1).max() < 1e-12, kind  # forward kernels agree
            for k in wrt:
                scale = np.abs(res[True][k]).max()
                assert np.abs(res[False][k] - res[True][k]).max() / scale < 1e-10, (kind, wrt, k)
            for b in (0, 31, 32, 76):
                args = (y,) + tuple(systems[b][1:])
                ll_ref = kn.kalman_filter(kind, *args, c=c[b].cpu().numpy()[:, None], d=d[b].cpu().numpy()[:, None],
                                          strict_reference=strict)[4]
                assert abs(res[False]["loglik"][b] - ll_ref) < RTOL * abs(ll_ref), (kind, b)
                _, gref = kt.loglik_and_grads(kind, *args, c=c[b].cpu().numpy()[:, None], d=d[b].cpu().numpy()[:, None],
                                              strict_reference=strict,  # 0.5 * loglik + sum_t w_t ll_t
                                              g_ll_obs=None if gobs is None else 0.5 + gobs[b])
                for k in wrt:
                    got = res[False][k][b].reshape(gref[k].shape)
                    scale = max(np.abs(gref[k]).max(), 1e-12 * max(np.abs(v).max() for v in gref.values()))
                    assert np.abs(got - gref[k]).max() / scale < RTOL, (kind, wrt, k, b)


@pytest.mark.parametrize("n_missing", [0, 5])
def test_nile_fixture_cuda_loglik_equals_dense_gaussian_density(n_missing):
    """The CUDA log-likelihood of the one fixture the reference value-tests (Nile local linear trend, P0 = 1e6 I,
    tests/test_kalman_filter.py:226-241) against the dense multivariate-normal density of the stacked sample in 40-digit
    arithmetic (tests/golden/nile_dense_loglik.json) - a parity leg that does NOT route through the oracle's recursion.
    Every kernel family that can run it: thread-per-unit (full outputs), k_endog = 1 hot path, cooperative."""
    import json
    import os

    from pymc_statespace_b200 import BatchedKalman
    from tests.helpers import GOLDEN

    gold = json.load(open(os.path.join(GOLDEN, "nile_dense_loglik.json")))[str(n_missing)]["loglik"]
    args = nile_inputs(n_missing)
    for kind in KINDS_P1:
        for force_coop in (False, True):
            res, _, info = run_single(kind, args, force_coop=force_coop, bwd=False)
            assert info == 0 and abs(res[4] - gold) < 1e-10 * abs(gold), (kind, force_coop, res[4], gold)
    y, a0, P0, T, Z, R, H, Q = args
    bk = BatchedKalman("standard", y.shape[0], 2, 1, 2, n_draws=1)   # loglik only -> kf_p1_forward_kernel
    out = bk.forward(_dev(y[..., 0]), _dev(a0[None, :, 0]), _dev(P0[None]), _dev(T), _dev(Z), _dev(R), _dev(H), _dev(Q))
    assert abs(float(out["loglik"][0]) - gold) < 1e-10 * abs(gold)


@pytest.mark.parametrize("force_coop", [False, True], ids=["thread", "coop"])
def test_single_filter_intercept_sign_quirk_on_device(force_coop):
    """SURVEY A.2-Q5 on the GPU: SingleTimeseriesFilter computes v = y - Z a + d (kalman_filter.py:335-336); strict mode
    reproduces the sign, corrected mode (strict_reference=False) uses v = y - Z a - d like every other filter."""
    rng = np.random.default_rng(12)
    args = random_system(rng, 3, 1, 2, 30, n_missing=3)
    c, d = rng.normal(size=(3, 1)), rng.normal(size=(1, 1)) + 1.5
    check_against_oracle("single", args, c, d, strict=True, force_coop=force_coop)
    check_against_oracle("single", args, c, d, strict=False, force_coop=force_coop)
    strict = run_single("single", args, c, d, strict=True, force_coop=force_coop, bwd=False)[0][4]
    flipped = run_single("single", args, c, -d, strict=False, force_coop=force_coop, bwd=False)[0][4]
    other = run_single("standard", args, c, d, force_coop=force_coop, bwd=False)[0][4]
    assert abs(strict - flipped) < 1e-10 * abs(strict) and abs(strict - other) > 1e-3


@pytest.mark.parametrize("dims", [(3, 2, 2), (4, 3, 2), (6, 3, 3), (8, 2, 2)])
def test_non_symmetric_P0_multivariate(dims):
    """ADVICE r1 (medium): P0 = theta.reshape(m, m) (BayesianVARMAX, stationary_initialization=False) is non-symmetric
    under NUTS.  The reference inverts the UPPER triangle of F_0 (posv) and takes log det of the full matrix; thread,
    cooperative and fused-row kernels must all reproduce the oracle's restatement of those SciPy calls."""
    from pymc_statespace_b200 import BatchedKalman

    m, p, r = dims
    rng = np.random.default_rng(90 + m)
    args = list(random_system(rng, m, p, r, 15, n_missing=1))
    args[2] = args[2] + 0.1 * rng.normal(size=(m, m))
    for strict in (True, False):
        ref = kn.kalman_filter("standard", *args, strict_reference=strict)
        for force_coop in (False, True):
            res, _, info = run_single("standard", args, strict=strict, force_coop=force_coop, bwd=False)
            assert info == 0
            for name, a, b in zip(ALL_OUT, res, ref):
                assert rel_err(a, b) < RTOL, (name, force_coop)
        y, a0, P0, T, Z, R, H, Q = args      # loglik-only request -> predictor-form / fused-row kernels
        B = 9
        bk = BatchedKalman("standard", y.shape[0], m, p, r, n_draws=B, strict_reference=strict)
        rep = lambda x: _dev(np.repeat(x[None], B, axis=0))  # noqa: E731
        out = bk.forward(_dev(y[..., 0]), rep(a0[:, 0]), rep(P0), rep(T), _dev(Z), rep(R), _dev(H), rep(Q))
        ll = out["loglik"].cpu().numpy()
        assert int((out["info"] != 0).sum()) == 0 and np.abs(ll - ref[4]).max() < 1e-10 * abs(ref[4])


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_structure_flags_on_device(m):
    """KFB_FLAG_Z_UNIT0 / KFB_FLAG_H_ZERO (Z = [1, 0, ..], H = 0 promised by the caller): identical loglik and cotangents
    to the unflagged k_endog = 1 kernels on every unit, oracle parity on a few, and a false promise is reported per unit."""
    from pymc_statespace_b200 import BatchedKalman
    from pymc_statespace_b200._lib import KFB_INFO_BAD_STRUCTURE

    rng = np.random.default_rng(70 + m)
    B, n, r = 45, 33, min(m, 2)
    systems = [list(random_system(rng, m, 1, r, n)) for _ in range(B)]
    y = random_system(rng, m, 1, r, n, n_missing=3)[0]
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    Z = np.eye(m)[:1]
    w = rng.normal(size=(B, n))
    for h_zero in (False, True):
        H = np.zeros((1, 1)) if h_zero else np.array([[0.7]])
        for gobs in (None, w):
            res = {}
            for flagged in (False, True):
                bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, z_unit0=flagged, h_zero=flagged and h_zero)
                out = bk.forward(_dev(y[..., 0]), stack(1)[..., 0], stack(2), stack(3), _dev(Z), stack(5), _dev(H), stack(7),
                                 outputs=("loglik",), save_for_backward=True)
                g = bk.backward(g_loglik=None if gobs is None else _dev(np.full(B, 0.5)),
                                g_ll_obs=None if gobs is None else _dev(gobs), wrt=("a0", "P0", "T", "R", "Q"))
                assert int((out["info"] != 0).sum()) == 0
                res[flagged] = {k: v.cpu().numpy() for k, v in g.items()}
                res[flagged]["loglik"] = out["loglik"].cpu().numpy()
            for k in res[True]:
                scale = np.abs(res[False][k]).max()
                assert np.abs(res[True][k] - res[False][k]).max() / scale < 1e-13, (k, h_zero)
            for b in (0, 44):
                args = (y, systems[b][1], systems[b][2], systems[b][3], Z, systems[b][5], H, systems[b][7])
                ll_ref, gref = kt.loglik_and_grads("standard", *args, g_ll_obs=None if gobs is None else 0.5 + gobs[b])
                if gobs is None:
                    assert abs(res[True]["loglik"][b] - ll_ref) < RTOL * abs(ll_ref)
                for k in ("a0", "P0", "T", "R", "Q"):
                    got = res[True][k][b].reshape(gref[k].shape)
                    scale = max(np.abs(gref[k]).max(), 1e-12 * max(np.abs(v).max() for v in gref.values()))
                    assert np.abs(got - gref[k]).max() / scale < RTOL, (k, b, h_zero)
    # false promises: unit 3 has another design row / a non-zero observation variance
    Zb = np.repeat(Z[None], B, 0)
    Zb[3, 0, 0] = 0.9
    bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, z_unit0=True)
    out = bk.forward(_dev(y[..., 0]), stack(1)[..., 0], stack(2), stack(3), _dev(Zb), stack(5), _dev(np.array([[0.7]])), stack(7))
    info = out["info"].cpu().numpy()
    assert info[3] == KFB_INFO_BAD_STRUCTURE and (np.delete(info, 3) == 0).all() and bool(torch.isnan(out["loglik"][3]))


@pytest.mark.parametrize("wrt", [("a0", "P0", "T", "R", "H", "Q", "c", "d"), ("a0", "R", "H", "Q")], ids=["with_Tbar", "no_Tbar"])
@pytest.mark.parametrize("dims", [(5, 3, 2), (6, 2, 3), (6, 3, 3), (8, 3, 3)], ids=lambda d: "m%dp%dr%d" % d)
def test_fused_row_kernels_as_coded_cholesky(dims, wrt):
    """BASELINE.json configs[2] names the cholesky filter: strict_reference = the AS-CODED CholeskyFilter for k_endog > 1
    (kalman_filter.py:287-318, second trtrs reads only diag(L): SURVEY A.2-Q4) on the fused row kernels (MK_CHOLS
    instantiations of kf_rows.cuh: gain matrix Gk, adjoint through the Cholesky factor) - values and gradients against
    the oracle's restatement of the as-coded filter, and against the generic cooperative kernels on every unit."""
    from pymc_statespace_b200 import BatchedKalman

    m, p, r = dims
    rng = np.random.default_rng(2000 + 10 * m + p)
    B, n = 13, 24
    systems = [random_system(rng, m, p, r, n, scale_T=0.25) for _ in range(B)]
    y = random_system(rng, m, p, r, n, n_missing=3)[0]
    cs, ds = rng.normal(size=(B, m)), rng.normal(size=(B, p))
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    wt = rng.normal(size=(B, n))
    res = {}
    for force in (False, True):
        bk = BatchedKalman("cholesky", n, m, p, r, n_draws=B, strict_reference=True, force_coop=force)
        out = bk.forward(_dev(y[..., 0]), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7),
                         c=_dev(cs), d=_dev(ds), outputs=("loglik",), save_for_backward=True)
        g = bk.backward(wrt=wrt)
        g2 = bk.backward(g_loglik=_dev(np.zeros(B)), g_ll_obs=_dev(wt), wrt=wrt)
        assert int(out["info"].abs().max()) == 0
        res[force] = (out["loglik"].cpu().numpy(), {k: v.cpu().numpy() for k, v in g.items()},
                      {k: v.cpu().numpy() for k, v in g2.items()})
    assert np.abs(res[False][0] / res[True][0] - 1).max() < 1e-11
    for k in wrt:
        for idx in (1, 2):
            scale = np.abs(res[True][idx][k]).max()
            assert np.abs(res[False][idx][k] - res[True][idx][k]).max() / scale < 1e-9, (k, idx)
    for b in (0, 8, 12):
        args = (y,) + tuple(systems[b][1:])
        ref, gref = kt.loglik_and_grads("cholesky", *args, c=cs[b][:, None], d=ds[b][:, None], strict_reference=True)
        assert abs(res[False][0][b] - ref) < RTOL * abs(ref)
        for k in wrt:
            got = res[False][1][k][b].reshape(gref[k].shape)
            scale = max(np.abs(gref[k]).max(), 1e-12)
            assert np.abs(got - gref[k]).max() / scale < RTOL, (k, b)


@pytest.mark.parametrize("wrt", [("a0", "P0", "T", "R", "H", "Q", "c", "d"), ("a0", "R", "H", "Q")], ids=["with_Tbar", "no_Tbar"])
@pytest.mark.parametrize("dims", [(5, 1, 2), (5, 3, 2), (6, 2, 3), (6, 3, 3), (7, 3, 2), (8, 3, 3)], ids=lambda d: "m%dp%dr%d" % d)
def test_fused_row_kernels_univariate(dims, wrt):
    """UnivariateFilter (kalman_filter.py:444-505) on the fused kernels of kf_rowsU.cuh (8 lanes per unit, replicated
    state, one exchange per scalar update): loglik-only forward + adjoint without Z-bar, PARTIALLY missing rows (the one
    filter that supports them), whole missing rows, non-diagonal H (only its diagonal is used, A.2-Q9), non-symmetric P0
    (entry-wise gauge of P0-bar), 13 units (partial last warp), n = 24 / 2 / 1, loglik and per-step cotangents -
    against the generic cooperative kernels on every unit and against torch-autograd of the oracle."""
    from pymc_statespace_b200 import BatchedKalman

    m, p, r = dims
    rng = np.random.default_rng(3000 + 10 * m + p)
    for n in (24, 2, 1):
        B = 13
        systems = [list(random_system(rng, m, p, r, n, scale_T=0.25)) for _ in range(B)]
        for s_ in systems:
            s_[2] = s_[2] + 0.05 * rng.normal(size=(m, m))
        y = random_system(rng, m, p, r, n, n_missing=min(3, n - 1), partial=True)[0]
        cs, ds = rng.normal(size=(B, m)), rng.normal(size=(B, p))
        stack = lambda i: _dev(np.stack([s_[i] for s_ in systems]))  # noqa: E731
        wt = rng.normal(size=(B, n))
        res = {}
        for force in (False, True):
            bk = BatchedKalman("univariate", n, m, p, r, n_draws=B, force_coop=force)
            out = bk.forward(_dev(y[..., 0]), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7),
                             c=_dev(cs), d=_dev(ds), outputs=("loglik",), save_for_backward=True)
            g = bk.backward(wrt=wrt)
            g2 = bk.backward(g_loglik=_dev(np.full(B, 0.25)), g_ll_obs=_dev(wt), wrt=wrt)
            assert int(out["info"].abs().max()) == 0
            res[force] = (out["loglik"].cpu().numpy(), {k: v.cpu().numpy() for k, v in g.items()},
                          {k: v.cpu().numpy() for k, v in g2.items()})
        assert np.abs(res[False][0] / res[True][0] - 1).max() < 1e-12
        for k in wrt:
            for idx in (1, 2):
                scale = max(np.abs(res[True][idx][k]).max(), 1e-300)
                assert np.abs(res[False][idx][k] - res[True][idx][k]).max() / scale < 1e-10, (k, idx, n)
        for b in (0, 8, 12):
            args = (y,) + tuple(systems[b][1:])
            ref, gref = kt.loglik_and_grads("univariate", *args, c=cs[b][:, None], d=ds[b][:, None])
            assert abs(res[False][0][b] - ref) < RTOL * abs(ref)
            for k in wrt:
                got = res[False][1][k][b].reshape(gref[k].shape)
                scale = max(np.abs(gref[k]).max(), 1e-12 * max(np.abs(v).max() for v in gref.values()))
                assert np.abs(got - gref[k]).max() / scale < RTOL, (k, b, n)


@pytest.mark.parametrize("kind", ["standard", "steady_state"])
@pytest.mark.parametrize("m", [9, 13, 25, 31])
def test_odd_k_states_run_padded_on_the_fused_kernels(m, kind):
    """Matrix-level calls with an odd k_states in 9..31 (seasonal period 12 -> 13 states): BatchedKalman embeds the model
    in k_states + 1 states for the loglik + gradient hot path (zero rows / columns: exact) instead of falling to the
    run-time-dims kernels.  Same numbers as the unpadded generic path and as the oracle; shapes are the caller's."""
    from pymc_statespace_b200 import BatchedKalman

    rng = np.random.default_rng(500 + m)
    B, n, p, r = 7, 18, 1, 2
    systems = [random_system(rng, m, p, r, n, scale_T=0.1) for _ in range(B)]
    y = random_system(rng, m, p, r, n, n_missing=2)[0]
    cs = rng.normal(size=(B, m))
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    wrt = ("a0", "P0", "T", "R", "H", "Q", "c") if kind == "standard" else ("a0", "T", "R", "H", "Q", "c")
    res = {}
    for padded in (True, False):
        bk = BatchedKalman(kind, n, m, p, r, n_draws=B, pad_odd=padded)
        assert (bk._inner is not None) == padded
        out = bk.forward(_dev(y[..., 0]), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7), c=_dev(cs),
                         outputs=("loglik",), save_for_backward=True)
        g = bk.backward(wrt=wrt)
        assert int(out["info"].abs().max()) == 0
        res[padded] = (out["loglik"].cpu().numpy(), {k: g[k].cpu().numpy() for k in wrt})
    tol = 1e-7 if kind == "steady_state" else 1e-9
    assert np.abs(res[True][0] - res[False][0]).max() < 1e-11 * np.abs(res[False][0]).max()
    for k in wrt:
        assert res[True][1][k].shape == res[False][1][k].shape, k
        assert rel_err(res[True][1][k], res[False][1][k]) < tol, k
    args = (y,) + tuple(systems[3][1:])
    ref, gref = kt.loglik_and_grads(kind, *args, c=cs[3][:, None])
    assert abs(res[True][0][3] - ref) < RTOL * abs(ref)
    for k in wrt:
        assert rel_err(res[True][1][k][3].reshape(gref[k].shape), gref[k]) < (1e-7 if kind == "steady_state" else RTOL), k


@pytest.mark.parametrize("kind", ["standard", "steady_state"])
@pytest.mark.parametrize("dims", [(12, 1, 2), (16, 1, 3), (30, 1, 3), (5, 1, 2), (6, 3, 3), (7, 2, 2), (8, 3, 3)],
                         ids=lambda d: "m%dp%dr%d" % d)
def test_full_outputs_on_the_tensor_core_mapping(dims, kind):
    """All six outputs of the reference (kalman_filter.py:166-193) at k_states 5..8 (rows_forward_full, 4 lanes x 2 rows)
    and at even k_states 10..32, k_endog 1 (rowsD_forward_full, two-stage form as tile products).  Every output against the oracle, with missing rows, c and d;
    the tape written by this kernel feeds the fused adjoint (same gradients as after a loglik-only forward)."""
    from pymc_statespace_b200 import BatchedKalman

    m, p, r = dims
    rng = np.random.default_rng(900 + m)
    B, n = 5, 14
    B = 5 if m >= 10 else 13  # k_states 5..8: 8 units per warp - a partial second warp
    systems = [random_system(rng, m, p, r, n, scale_T=0.1 if m >= 10 else 0.25) for _ in range(B)]
    # (the as-coded steady-state filter, K = P Z^T F_ss^-1 with the CURRENT P, loses positive definiteness after missing
    #  rows for most random systems with k_endog > 1: it is exercised on complete data)
    y = random_system(rng, m, p, r, n, n_missing=0 if kind == "steady_state" else 3)[0]
    cs, ds = rng.normal(size=(B, m)), rng.normal(size=(B, p))
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    ins = (_dev(y[..., 0]), stack(1), stack(2), stack(3), stack(4), stack(5), stack(6), stack(7))
    bk = BatchedKalman(kind, n, m, p, r, n_draws=B)
    out = bk.forward(*ins, c=_dev(cs), d=_dev(ds), outputs=ALL_OUT, save_for_backward=True)
    wrt = ("a0", "T", "R", "H", "Q", "c")
    g_full = bk.backward(wrt=wrt)
    # units are flagged exactly like on the generic kernels; the good ones are compared with them and with the oracle
    info = out["info"].cpu().numpy()
    gen = BatchedKalman(kind, n, m, p, r, n_draws=B, force_coop=True).forward(*ins, c=_dev(cs), d=_dev(ds), outputs=ALL_OUT)
    assert (info == gen["info"].cpu().numpy()).all()
    good = np.nonzero(info == 0)[0]
    assert len(good) == B
    for k in ALL_OUT:
        assert rel_err(out[k][good].cpu().numpy(), gen[k][good].cpu().numpy()) < 1e-9, k
    for b in (good[0], good[len(good) // 2], good[-1]):
        ref = kn.kalman_filter(kind, y, *systems[b][1:], c=cs[b][:, None], d=ds[b][:, None])
        got = [out[k][b].cpu().numpy() for k in ALL_OUT]
        for name, a, e in zip(ALL_OUT, got, ref):
            e = np.asarray(e)
            assert rel_err(a.reshape(e.shape), e) < RTOL, (name, b)
    out2 = bk.forward(*ins, c=_dev(cs), d=_dev(ds), outputs=("loglik",), save_for_backward=True)
    g_hot = bk.backward(wrt=wrt)
    gi = torch.as_tensor(good, device="cuda")
    assert float((out2["loglik"][gi] - out["loglik"][gi]).abs().max()) < 1e-10 * float(out["loglik"][gi].abs().max())
    for k in wrt:
        assert rel_err(g_full[k][gi].cpu().numpy(), g_hot[k][gi].cpu().numpy()) < (1e-7 if kind == "steady_state" else 1e-9), k


@pytest.mark.parametrize("m", [2, 3, 4])
def test_p1_companion_T_promise(m):
    """KFB_FLAG_T_COMPANION (with Z = e0, H = 0: every BayesianARMA / SARIMAX model, models/SARIMAX.py:59-98): the k_endog = 1
    kernels skip the products with the known unit columns of T.  Same loglik and gradients as the kernels without the
    promise on every unit (the T gradient in its first column - the other columns are constants of the model and come back
    as zero), with and without a per-step cotangent, missing rows, non-symmetric P0, c and d; oracle parity on a few units;
    a T that is not in companion form is reported per unit."""
    from pymc_statespace_b200 import BatchedKalman
    from pymc_statespace_b200._lib import KFB_INFO_BAD_STRUCTURE

    rng = np.random.default_rng(170 + m)
    B, n, r = 45, 33, 1
    systems = [list(random_system(rng, m, 1, r, n)) for _ in range(B)]
    Tc = np.zeros((B, m, m))
    Tc[:, :, 1:] = np.eye(m)[:, :m - 1]
    Tc[:, :, 0] = rng.uniform(-0.5, 0.5, size=(B, m)) / np.arange(1, m + 1)   # AR coefficients in the first column
    y = random_system(rng, m, 1, r, n, n_missing=3)[0]
    y[[0, n - 1]] = np.nan
    for s in systems:
        s[2] = s[2] + 0.05 * rng.normal(size=(m, m))  # non-symmetric P0
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    Z, H = np.eye(m)[:1], np.zeros((1, 1))
    cs, ds = rng.normal(size=(B, m)), rng.normal(size=(B, 1))
    w = rng.normal(size=(B, n))
    wrt = ("a0", "P0", "T", "R", "Q", "c", "d")
    for gobs in (None, w):
        res = {}
        for flagged in (False, True):
            bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, z_unit0=True, h_zero=True, t_companion=flagged)
            out = bk.forward(_dev(y[..., 0]), stack(1)[..., 0], stack(2), _dev(Tc), _dev(Z), stack(5), _dev(H), stack(7),
                             c=_dev(cs), d=_dev(ds), outputs=("loglik",), save_for_backward=True)
            g = bk.backward(g_loglik=None if gobs is None else _dev(np.full(B, 0.5)),
                            g_ll_obs=None if gobs is None else _dev(gobs), wrt=wrt)
            assert int((out["info"] != 0).sum()) == 0
            res[flagged] = {k: v.cpu().numpy() for k, v in g.items()}
            res[flagged]["loglik"] = out["loglik"].cpu().numpy()
        assert np.abs(res[True]["T"][:, :, 1:]).max() == 0.0
        res[False]["T"][:, :, 1:] = 0.0
        for k in res[True]:
            scale = np.abs(res[False][k]).max()
            assert np.abs(res[True][k] - res[False][k]).max() / scale < 1e-12, (k, gobs is None)
        for b in (0, 44):
            args = (y, systems[b][1], systems[b][2], Tc[b], Z, systems[b][5], H, systems[b][7])
            ll_ref, gref = kt.loglik_and_grads("standard", *args, c=cs[b][:, None], d=ds[b][:, None],
                                               g_ll_obs=None if gobs is None else 0.5 + gobs[b])
            if gobs is None:
                assert abs(res[True]["loglik"][b] - ll_ref) < RTOL * abs(ll_ref)
            gref["T"][:, 1:] = 0.0
            for k in wrt:
                got = res[True][k][b].reshape(gref[k].shape)
                scale = max(np.abs(gref[k]).max(), 1e-12 * max(np.abs(v).max() for v in gref.values()))
                assert np.abs(got - gref[k]).max() / scale < RTOL, (k, b)
    # false promise: unit 5 has a T that is not in companion form
    Tb = Tc.copy()
    Tb[5, m - 1, m - 1] = 0.3
    bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, z_unit0=True, h_zero=True, t_companion=True)
    out = bk.forward(_dev(y[..., 0]), stack(1)[..., 0], stack(2), _dev(Tb), _dev(Z), stack(5), _dev(H), stack(7))
    info = out["info"].cpu().numpy()
    assert info[5] == KFB_INFO_BAD_STRUCTURE and (np.delete(info, 5) == 0).all() and bool(torch.isnan(out["loglik"][5]))


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_compressed_tape(m):
    """All four structure promises (Z = e0, H = 0, companion T, no missing observation: every BayesianARMA model on complete
    data): P_t = C + blockdiag(B_t, 0), so the tape holds a_t and the leading (m-1) x (m-1) block of P_t only and the adjoint
    re-inserts the last column of C.  Same loglik and gradients as the kernels with the full tape on every unit and as the
    oracle; the full-output forward writes the same compressed tape; a NaN in y breaks the promise (reported per unit);
    Z-bar / H-bar cannot be requested."""
    from pymc_statespace_b200 import BatchedKalman
    from pymc_statespace_b200._lib import KFB_INFO_BAD_STRUCTURE

    rng = np.random.default_rng(270 + m)
    B, n, r = 45, 33, 1
    systems = [list(random_system(rng, m, 1, r, n)) for _ in range(B)]
    Tc = np.zeros((B, m, m))
    Tc[:, :, 1:] = np.eye(m)[:, :m - 1]
    Tc[:, :, 0] = rng.uniform(-0.5, 0.5, size=(B, m)) / np.arange(1, m + 1)
    y = random_system(rng, m, 1, r, n)[0]
    for s in systems:
        s[2] = s[2] + 0.05 * rng.normal(size=(m, m))  # non-symmetric P0
    stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
    Z, H = np.eye(m)[:1], np.zeros((1, 1))
    cs, ds = rng.normal(size=(B, m)), rng.normal(size=(B, 1))
    w = rng.normal(size=(B, n))
    wrt = ("a0", "P0", "T", "R", "Q", "c", "d")
    ins = lambda yy: (_dev(yy[..., 0]), stack(1)[..., 0], stack(2), _dev(Tc), _dev(Z), stack(5), _dev(H), stack(7))  # noqa: E731
    for gobs in (None, w):
        res = {}
        for variant in ("plain", "compressed", "compressed_full_forward"):
            bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, z_unit0=True, h_zero=True, t_companion=True,
                               no_missing=variant != "plain")
            outs = ("loglik",) if variant != "compressed_full_forward" else ALL_OUT
            out = bk.forward(*ins(y), c=_dev(cs), d=_dev(ds), outputs=outs, save_for_backward=True)
            g = bk.backward(g_loglik=None if gobs is None else _dev(np.full(B, 0.5)),
                            g_ll_obs=None if gobs is None else _dev(gobs), wrt=wrt)
            assert int((out["info"] != 0).sum()) == 0
            res[variant] = {k: v.cpu().numpy() for k, v in g.items()}
            res[variant]["loglik"] = out["loglik"].cpu().numpy()
        for variant in ("compressed", "compressed_full_forward"):
            for k in res[variant]:
                scale = np.abs(res["plain"][k]).max()
                assert np.abs(res[variant][k] - res["plain"][k]).max() / scale < 1e-11, (variant, k, gobs is None)
        for b in (0, 44):
            args = (y, systems[b][1], systems[b][2], Tc[b], Z, systems[b][5], H, systems[b][7])
            ll_ref, gref = kt.loglik_and_grads("standard", *args, c=cs[b][:, None], d=ds[b][:, None],
                                               g_ll_obs=None if gobs is None else 0.5 + gobs[b])
            if gobs is None:
                assert abs(res["compressed"]["loglik"][b] - ll_ref) < RTOL * abs(ll_ref)
            gref["T"][:, 1:] = 0.0
            for k in wrt:
                got = res["compressed"][k][b].reshape(gref[k].shape)
                scale = max(np.abs(gref[k]).max(), 1e-12 * max(np.abs(v).max() for v in gref.values()))
                assert np.abs(got - gref[k]).max() / scale < RTOL, (k, b)
    # a missing observation breaks the promise: every unit is flagged (hot-path and full-output forward alike)
    yb = y.copy()
    yb[7] = np.nan
    for outs in (("loglik",), ALL_OUT):
        bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, z_unit0=True, h_zero=True, t_companion=True, no_missing=True)
        out = bk.forward(*ins(yb), outputs=outs, save_for_backward=True)
        assert (out["info"].cpu().numpy() == KFB_INFO_BAD_STRUCTURE).all() and bool(torch.isnan(out["loglik"]).all())
    # Z-bar with a design row that was promised constant: refused
    bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, z_unit0=True, h_zero=True, t_companion=True, no_missing=True)
    bk.forward(*ins(y), outputs=("loglik",), save_for_backward=True)
    with pytest.raises(Exception):
        bk.backward(wrt=("Z",))
