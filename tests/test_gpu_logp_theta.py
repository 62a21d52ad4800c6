"""GPU parity at theta level: scatter + (Lyapunov) + Kalman forward + adjoint + scatter^T through the C ABI,
against torch-autograd of the oracle's restatement of the reference models (rtol 1e-8, float64)."""
import numpy as np
import pytest
import torch

from oracle import models as om
from tests.helpers import nile_data

pytestmark = pytest.mark.gpu
RTOL = 1e-8


def _run(spec, y, theta, kind="standard", strict=True, force_coop=False):
    from pymc_statespace_b200.logp import KalmanLogp

    model = KalmanLogp(spec, y, n_draws=theta.shape[0], filter_type=kind, strict_reference=strict, force_coop=force_coop)
    logp, grad = model.logp_and_grad(torch.as_tensor(theta, device="cuda"))
    torch.cuda.synchronize()
    assert int((model.info != 0).sum()) == 0
    return logp.cpu().numpy(), grad.cpu().numpy(), model


def _compare(fn, y3, theta, logp, grad, idx, kind="standard", strict=True, rtol=RTOL, sym_block=None):
    """sym_block=(slice, k): that k x k block of theta is a symmetric matrix written entry by entry (VARMAX
    state_cov); compare its gradient after symmetrisation (see test_varmax... for why)."""
    for b in idx:
        ll, g = om.logp_and_grad_theta(fn, theta[b], y3, kind, strict)
        gb = grad[b].copy()
        if sym_block is not None:
            sl, k = sym_block
            for arr in (g, gb):
                blk = arr[sl].reshape(k, k)
                arr[sl] = (0.5 * (blk + blk.T)).reshape(-1)
        assert abs(logp[b] - ll) <= rtol * abs(ll), (b, logp[b], ll)
        assert np.abs(gb - g).max() <= rtol * np.abs(g).max(), (b, gb, g)


@pytest.mark.parametrize("order", [(1, 1), (2, 1), (3, 0)])
@pytest.mark.parametrize("stationary", [True, False])
def test_arma_theta_gradient(order, stationary):
    from pymc_statespace_b200.models import arma_spec
    from pymc_statespace_b200.synthetic import simulate_arma

    spec = arma_spec(order, stationary)
    rng = np.random.default_rng(sum(order) + stationary)
    B, n, m = 64, 60, spec.k_states
    y = simulate_arma(n, (0.5,), (0.3,), 1.0)[:, None]
    theta = np.zeros((B, spec.n_theta))
    theta[:, spec.param_slices["x0"]] = rng.normal(size=(B, m))
    if not stationary:
        L = rng.normal(size=(B, m, m)) * 0.3 + np.eye(m)
        theta[:, spec.param_slices["P0"]] = (L @ L.transpose(0, 2, 1)).reshape(B, -1)
    theta[:, spec.param_slices["sigma_state"]] = np.exp(rng.normal(0, 0.3, (B, 1)))
    theta[:, spec.param_slices["rho"]] = rng.uniform(-0.3, 0.3, (B, order[0]))
    theta[:, spec.param_slices["theta"]] = rng.normal(0, 0.4, (B, order[1]))
    logp, grad, _ = _run(spec, y, theta)
    _compare(lambda t: om.arma_matrices(t, order, stationary), y[:, :, None], theta, logp, grad, (0, 1, 31, 63))


@pytest.mark.parametrize("order", [(1, 1), (2, 1), (3, 2)])
def test_arma_theta_gradient_equals_autograd_of_dense_density(order):
    """A parity leg that does NOT route through the restated recursion nor through a hand-written adjoint: the CUDA
    theta-level logp and gradient (scatter + Lyapunov doubling + reduced ARMA recursion + adjoints) against
    torch-autograd of [theta -> matrices -> P0 by one dense Kronecker solve -> dense multivariate-normal log-density of
    the stacked sample] (oracle.kalman_torch.dense_gaussian_loglik).  The reference's gradient is autodiff of the same
    scalar, so this is the value it must produce.  BayesianARMA, stationary initialisation (models/SARIMAX.py:59-107):
    the north-star model family, on the structure-promise kernels of kf_p1.cu."""
    from oracle import kalman_torch as kt
    from pymc_statespace_b200.models import arma_spec

    spec = arma_spec(order, True)
    rng = np.random.default_rng(70 + 10 * order[0] + order[1])
    B, n, m = 40, 40, spec.k_states
    y = rng.normal(size=(n, 1))
    theta = np.zeros((B, spec.n_theta))
    theta[:, spec.param_slices["x0"]] = rng.normal(size=(B, m)) * 0.3
    theta[:, spec.param_slices["sigma_state"]] = np.exp(rng.normal(0, 0.3, (B, 1)))
    theta[:, spec.param_slices["rho"]] = rng.uniform(-0.4, 0.4, (B, order[0])) / np.arange(1, order[0] + 1)
    theta[:, spec.param_slices["theta"]] = rng.uniform(-0.5, 0.5, (B, order[1]))
    logp, grad, _ = _run(spec, y, theta)
    for b in (0, 1, 17, 39):
        th = torch.tensor(theta[b], dtype=torch.float64, requires_grad=True)
        a0, _, T, Z, R, H, Q = om.arma_matrices(th, order)
        ll = kt.dense_gaussian_loglik(y[:, :, None], a0, kt.lyapunov_dense(T, R @ Q @ R.T), T, Z, R, H, Q)
        (g,) = torch.autograd.grad(ll, [th])
        assert abs(logp[b] - float(ll.detach())) <= RTOL * abs(float(ll.detach())), (b, logp[b], ll)
        assert np.abs(grad[b] - g.numpy()).max() <= RTOL * np.abs(g.numpy()).max(), (b, grad[b], g)


@pytest.mark.parametrize("kind", ["standard", "univariate", "cholesky"])
def test_varmax_theta_gradient_with_missing_rows(kind):
    from pymc_statespace_b200.synthetic import varmax20_workload

    spec, y, theta = varmax20_workload(n_draws=24, n=40)
    assert np.isnan(y).any()
    strict = kind != "cholesky"  # strict cholesky (SURVEY A.2-Q4) for p > 1 is a separate test
    logp, grad, _ = _run(spec, y, theta, kind, strict)
    # Gauge (DESIGN.md "gradient gauge"): for standard / univariate the kernels reproduce the entry-wise gradient
    # of the literal graph exactly, including the asymmetric part of dlogp/dP0 that the Lyapunov adjoint turns
    # into asymmetric dlogp/dQ[i,j] vs [j,i].  A Cholesky-based filter's F-bar depends on the Cholesky op's
    # triangle convention (torch symmetrises, PyTensor folds into the lower triangle), so only the symmetrised
    # state_cov block is convention-independent there.
    sym = (spec.param_slices["state_cov"], 3) if kind == "cholesky" else None
    _compare(lambda t: om.varmax_matrices(t, 3, (2, 0), True, True), y[:, :, None], theta, logp, grad, (0, 7, 23),
             kind, strict, sym_block=sym)


def test_local_level_nile_cpu_config():
    # BASELINE.json configs[0]: Nile local level, standard filter, logp+grad
    from pymc_statespace_b200.models import local_level_spec

    spec = local_level_spec()
    y = nile_data()[:, None]
    rng = np.random.default_rng(0)
    B = 16
    theta = np.zeros((B, 9))
    theta[:, 0] = rng.normal(1000, 100, B)
    theta[:, 2], theta[:, 5] = 1e4 * np.exp(rng.normal(0, 0.2, B)), 1e2 * np.exp(rng.normal(0, 0.2, B))
    theta[:, 6] = 15000 * np.exp(rng.normal(0, 0.2, B))
    theta[:, 7], theta[:, 8] = 1400 * np.exp(rng.normal(0, 0.2, B)), 10 * np.exp(rng.normal(0, 0.2, B))
    logp, grad, _ = _run(spec, y, theta)
    _compare(om.local_level_matrices, y[:, :, None], theta, logp, grad, (0, 5, 15))


def test_nile_true_local_level_k_states_1():
    """BASELINE.json configs[0] as written: Nile, T = 100, k_states = 1, standard filter, logp + grad at theta level
    (theta = [a0, P0, sigma2_obs, sigma2_level]) - against torch-autograd of the oracle and, for the value, against the
    dense multivariate-normal density of the sample (no recursion at all)."""
    from oracle import kalman_numpy as kn
    from pymc_statespace_b200.models import local_level_1state_spec

    spec = local_level_1state_spec()
    y = nile_data()[:, None]
    rng = np.random.default_rng(4)
    B = 8
    theta = np.stack([rng.normal(1120, 50, B), 1e6 * np.exp(rng.normal(0, 0.1, B)), 15000 * np.exp(rng.normal(0, 0.2, B)),
                      1400 * np.exp(rng.normal(0, 0.2, B))], axis=1)

    def mats(t):
        one = torch.ones(1, 1, dtype=torch.float64)
        return t[0].reshape(1, 1), t[1].reshape(1, 1), one, one, one, t[2].reshape(1, 1), t[3].reshape(1, 1)

    for kind in ("standard", "single", "cholesky", "univariate"):
        logp, grad, _ = _run(spec, y, theta, kind)
        _compare(mats, y[:, :, None], theta, logp, grad, (0, 3, 7), kind, rtol=1e-7 if kind == "univariate" else RTOL)
    for b in (0, 7):
        m = spec.matrices(theta[b])
        dense = kn.dense_gaussian_loglik(y[:, :, None], *[m[k] for k in ("a0", "P0", "T", "Z", "R", "H", "Q")], mp_digits=30)
        assert abs(logp[b] - dense) < 1e-10 * abs(dense)


def test_full_size_all_draws_match_c_port():
    """configs[1] at full size, EVERY draw (VERDICT r1): 65,536 draws x T = 1000 on the GPU against the plain-C port
    (oracle/kalman_c.c, itself validated against the torch oracle in tests/test_cabi_and_host.py) - logp and the five
    matrix-level cotangents the theta-level gradient is assembled from."""
    import os

    from oracle import kalman_c
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.models import MATRICES
    from pymc_statespace_b200.synthetic import arma11_workload

    B, n = 65536, 1000
    spec, y, theta = arma11_workload(B, n)
    model = KalmanLogp(spec, y, n_draws=B)
    mats = model._scatter(torch.as_tensor(theta, device="cuda"))
    out = model.kalman.forward(model.y, *[mats[k] for k in MATRICES], outputs=("loglik",), save_for_backward=True)
    g = model.kalman.backward(wrt=("a0", "P0", "T"))
    gC = None
    f = lambda t: (t if t.ndim == 3 or t.shape[0] == B else t.expand(B, *t.shape)).cpu().numpy()  # noqa: E731
    T, R, Q, P0, a0 = f(mats["T"]), f(mats["R"]), f(mats["Q"]), f(mats["P0"]), f(mats["a0"])
    C = R @ Q @ R.transpose(0, 2, 1)
    ll, gc, bad = kalman_c.logp_grad_batch(y, a0.reshape(B, 2), P0, T, mats["Z"].cpu().numpy().reshape(1, 2),
                                           mats["H"].cpu().numpy().reshape(1, 1), C, nthreads=os.cpu_count() or 1)
    assert bad == 0 and int((out["info"] != 0).sum()) == 0
    lg = out["loglik"].cpu().numpy()
    # (the kernels run the reduced ARMA recursion - Schur form, kf_p1.cuh ZU == 4 - the C port the general Joseph form: the two
    #  agree to 2e-11 over all draws, tools/reduced_check.py)
    assert np.abs(lg - ll).max() / np.abs(ll).max() < 1e-10 and (np.abs(lg / ll - 1) < 1e-9).all()
    for k in ("a0", "P0", "T"):
        got, ref = g[k].cpu().numpy().reshape(B, -1), gc[k].reshape(B, -1)
        if k == "T":  # companion T promised by the model (KFB_FLAG_T_COMPANION): only its first column has a gradient
            assert np.abs(got.reshape(B, 2, 2)[:, :, 1]).max() == 0.0
            got, ref = got.reshape(B, 2, 2)[:, :, 0], ref.reshape(B, 2, 2)[:, :, 0]
        err = np.abs(got - ref).max(axis=1) / np.maximum(np.abs(ref).max(axis=1), 1e-300)
        assert err.max() < 1e-8, (k, int(err.argmax()), err.max())


def test_full_size_properties_arma11():
    """BASELINE.json configs[1] at full size (65,536 draws x T=1000): size-independent properties.
    (a) thread-per-unit and cooperative kernels agree; (b) sub-batch invariance; (c) sampled draws match the
    oracle; (d) directional finite difference of logp along a random direction matches grad . dir."""
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import arma11_workload

    B, n = 65536, 1000
    spec, y, theta = arma11_workload(B, n)
    th = torch.as_tensor(theta, device="cuda")
    model = KalmanLogp(spec, y, n_draws=B)
    logp, grad = model.logp_and_grad(th)
    assert int((model.info != 0).sum()) == 0
    assert bool(torch.isfinite(logp).all()) and bool(torch.isfinite(grad).all())
    sub = KalmanLogp(spec, y, n_draws=512)
    lp2, g2 = sub.logp_and_grad(th[1000:1512].contiguous())
    assert torch.equal(lp2, logp[1000:1512]) and torch.equal(g2, grad[1000:1512])
    coop = KalmanLogp(spec, y, n_draws=512, force_coop=True)
    lp3, g3 = coop.logp_and_grad(th[1000:1512].contiguous())
    assert float(((lp3 - lp2).abs() / lp2.abs()).max()) < 1e-10
    assert float(((g3 - g2).abs().amax(1) / g2.abs().amax(1)).max()) < 1e-8
    _compare(lambda t: om.arma_matrices(t, (1, 1), True), y[:, :, None], theta, logp.cpu().numpy(), grad.cpu().numpy(),
             (0, 65535), rtol=RTOL)
    rng = np.random.default_rng(0)
    direction = torch.as_tensor(rng.normal(size=theta.shape), device="cuda")
    eps = 1e-6
    fd = (model.logp(th + eps * direction) - model.logp(th - eps * direction)) / (2 * eps)
    an = (grad * direction).sum(1)
    assert float(((fd - an).abs() / (an.abs() + 1e-3 * grad.abs().amax(1))).median()) < 1e-5


def test_full_size_properties_varmax():
    """BASELINE.json configs[2] at full size (262,144 draws x T=1000, k_states=6, k_endog=3, 10 % missing rows):
    sub-batch invariance, sampled draws vs the oracle, univariate == corrected cholesky (diagonal H identity)."""
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import varmax20_workload

    B, n = 262144, 1000
    spec, y, theta = varmax20_workload(B, n)
    th = torch.as_tensor(theta, device="cuda")
    fn = lambda t: om.varmax_matrices(t, 3, (2, 0), True, True)  # noqa: E731
    model = KalmanLogp(spec, y, n_draws=B, filter_type="univariate")
    logp, grad = model.logp_and_grad(th)
    assert int((model.info != 0).sum()) == 0
    assert bool(torch.isfinite(logp).all()) and bool(torch.isfinite(grad).all())
    sub = KalmanLogp(spec, y, n_draws=256, filter_type="univariate")
    lp2, g2 = sub.logp_and_grad(th[5000:5256].contiguous())
    assert torch.equal(lp2, logp[5000:5256]) and torch.equal(g2, grad[5000:5256])
    _compare(fn, y[:, :, None], theta, logp.cpu().numpy(), grad.cpu().numpy(), (0, 262143), "univariate")
    chol = KalmanLogp(spec, y, n_draws=256, filter_type="cholesky", strict_reference=False)
    lp3, g3 = chol.logp_and_grad(th[5000:5256].contiguous())
    assert float(((lp3 - lp2).abs() / lp2.abs()).max()) < 1e-9
    sl = spec.param_slices["state_cov"]
    sym = lambda g: 0.5 * (g[:, sl].reshape(-1, 3, 3) + g[:, sl].reshape(-1, 3, 3).transpose(1, 2))  # noqa: E731
    assert float(((sym(g3) - sym(g2)).abs().amax((1, 2)) / g2.abs().amax(1)).max()) < 1e-7
    other = [i for i in range(spec.n_theta) if not (sl.start <= i < sl.stop)]
    assert float(((g3[:, other] - g2[:, other]).abs().amax(1) / g2.abs().amax(1)).max()) < 1e-7


def test_trend_seasonal_k30_steady_vs_standard():
    """BASELINE.json configs[3]: k_states = 30, T = 2000.  Both filters against the oracle on sampled draws; the two
    filters legitimately differ (P_t has not converged to P_ss by t = 2000, SURVEY section 8(d))."""
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.models import trend_seasonal_spec
    from pymc_statespace_b200.synthetic import trend_seasonal_workload

    spec, y, theta = trend_seasonal_workload(n_draws=64, n=300)
    th = torch.as_tensor(theta, device="cuda")

    def mats(t):
        m = spec.matrices(t.detach().numpy())
        T, Z, R = (torch.tensor(m[k]) for k in ("T", "Z", "R"))
        Q = torch.zeros(3, 3, dtype=torch.float64)
        Q[0, 0], Q[1, 1], Q[2, 2] = t[0], t[1], t[2]
        H = t[3].reshape(1, 1)
        return torch.zeros(30, 1, dtype=torch.float64), torch.eye(30, dtype=torch.float64), T, Z, R, H, Q

    for kind, gtol in (("standard", 1e-8), ("steady_state", 1e-6)):
        model = KalmanLogp(spec, y, n_draws=64, filter_type=kind)
        logp, grad = model.logp_and_grad(th)
        assert int((model.info != 0).sum()) == 0
        lp, g = logp.cpu().numpy(), grad.cpu().numpy()
        for b in (0, 63):
            ll, gr = om.logp_and_grad_theta(mats, theta[b], y[:, :, None], kind)
            assert abs(lp[b] - ll) <= 1e-8 * abs(ll)
            assert np.abs(g[b] - gr).max() <= gtol * np.abs(gr).max(), (kind, g[b], gr)


def test_waves_match_single_pass():
    from pymc_statespace_b200.logp import KalmanLogp, logp_and_grad_in_waves
    from pymc_statespace_b200.synthetic import arma11_workload

    B, n = 1000, 200
    spec, y, theta = arma11_workload(B, n)
    th = torch.as_tensor(theta, device="cuda")
    lp, g = KalmanLogp(spec, y, n_draws=B).logp_and_grad(th)
    per_draw = ((n - 1) * 5 + 16 + 64) * 8
    lp2, g2, info = logp_and_grad_in_waves(spec, y, th, max_workspace_bytes=per_draw * 300)  # 4 waves (300,300,300,100)
    assert torch.equal(lp, lp2) and torch.equal(g, g2) and int(info.abs().sum()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["arma", "varmax"])
def test_host_step_graph_matches_eager(kind):
    """KalmanLogp.capture_host_step: pinned-host theta -> (logp, grad) on the host as ONE replayed CUDA graph; identical
    numbers to the eager call, and a replay picks up a new theta written into the captured host buffer."""
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import arma11_workload, varmax20_workload

    spec, y, theta = arma11_workload(300, 50) if kind == "arma" else varmax20_workload(n_draws=40, n=30)
    B = theta.shape[0]
    model = KalmanLogp(spec, y, n_draws=B, filter_type="standard")
    th_h = torch.from_numpy(np.ascontiguousarray(theta)).pin_memory()
    out_h = torch.empty((B, 1 + spec.n_theta), dtype=torch.float64).pin_memory()
    step = model.capture_host_step(th_h, out_h, chunks=1 if kind == "arma" else 4)  # 4 parallel draw-chunk branches
    for scale in (1.0, 0.9):
        th_h.copy_(torch.from_numpy(theta * scale if kind == "arma" else theta * np.where(np.arange(theta.shape[1]) < 6, scale, 1.0)))
        got = step().clone()
        lp, g = model.logp_and_grad(th_h.to("cuda"))
        torch.cuda.synchronize()
        assert torch.equal(got[:, 0], lp.cpu()) and torch.equal(got[:, 1:], g.cpu())
        assert int(step.info.abs().max()) == 0 and step.info.numel() == B
    with pytest.raises(ValueError):
        model.capture_host_step(th_h, out_h, chunks=7)   # must divide the number of draws
    with pytest.raises(TypeError):
        model.capture_host_step(th_h.clone(), out_h)  # not pinned


@pytest.mark.gpu
def test_wave_pipelines_match_single_pass():
    """bench.py's c5 legs: HostStepGraph(sequential=True) and dist.GatherStepGraph (world 1) push the draws through ONE
    wave-sized evaluator in 4 waves; every row must equal the single-pass evaluation bit for bit."""
    from pymc_statespace_b200.dist import GatherStepGraph
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import arma21_workload

    B, n, waves = 2048, 60, 4
    spec, y, theta = arma21_workload(B, n)
    th_d = torch.as_tensor(theta, device="cuda")
    lp, g = KalmanLogp(spec, y, n_draws=B).logp_and_grad(th_d)
    ref = torch.cat([lp[:, None], g], dim=1).cpu()
    wave_model = KalmanLogp(spec, y, n_draws=B // waves)
    gsg = GatherStepGraph(wave_model, th_d, waves=waves)
    assert gsg.graph is not None
    gsg()
    torch.cuda.synchronize()
    assert torch.equal(gsg.rows().cpu(), ref) and int(gsg.info.abs().max()) == 0
    th_h = torch.from_numpy(np.ascontiguousarray(theta)).pin_memory()
    out_h = torch.empty((B, 1 + spec.n_theta), dtype=torch.float64).pin_memory()
    step = wave_model.capture_host_step(th_h, out_h, chunks=waves, sequential=True)
    assert torch.equal(step().clone(), ref) and int(step.info.abs().max()) == 0 and step.info.numel() == B
    th_h.mul_(0.95)
    lp2, g2 = KalmanLogp(spec, y, n_draws=B).logp_and_grad(th_h.to("cuda"))
    assert torch.equal(step().clone(), torch.cat([lp2[:, None], g2], dim=1).cpu())


@pytest.mark.gpu
def test_scatter_multi_matches_numpy_and_single_calls():
    """kfb_scatter_forward_multi / kfb_scatter_backward_multi (one launch for all matrices) against a numpy restatement
    and the per-matrix entry points, including duplicate destinations (last writer wins) and a theta entry used twice."""
    import ctypes

    from pymc_statespace_b200._lib import KfbScatterSeg, check, load

    lib = load()
    rng = np.random.default_rng(3)
    B, nt = 37, 5
    theta = rng.normal(size=(B, nt))
    specs = [  # (block, [(src, dst), ...])
        (4, [(0, 0), (1, 3)]),
        (9, [(2, 4), (2, 8), (3, 4)]),          # theta_2 used twice; element 4 written twice (theta_3 wins)
        (2, []),                                # constant matrix
        (6, [(4, 5), (0, 1)]),
    ]
    dev = "cuda"
    th = torch.as_tensor(theta, device=dev)
    bases = [rng.normal(size=b) for b, _ in specs]
    outs, segs_f, keep = [], [], []
    for (blk, mp), base in zip(specs, bases):
        src = torch.as_tensor([a for a, _ in mp], dtype=torch.int32, device=dev)
        dst = torch.as_tensor([b for _, b in mp], dtype=torch.int32, device=dev)
        bs = torch.as_tensor(base, device=dev)
        out = torch.empty((B, blk), dtype=torch.float64, device=dev)
        keep += [src, dst, bs]
        outs.append(out)
        segs_f.append(KfbScatterSeg(blk, len(mp), bs.data_ptr(), src.data_ptr() if mp else None,
                                    dst.data_ptr() if mp else None, out.data_ptr()))
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    arr = (KfbScatterSeg * len(specs))(*segs_f)
    check(lib.kfb_scatter_forward_multi(B, nt, len(specs), arr, th.data_ptr(), stream), "fwd_multi")
    torch.cuda.synchronize()
    for (blk, mp), base, out in zip(specs, bases, outs):
        ref = np.tile(base, (B, 1))
        for a, b in mp:
            ref[:, b] = theta[:, a]
        assert np.array_equal(out.cpu().numpy(), ref)
    # backward: cotangents of the scattered matrices -> gtheta (written, not accumulated)
    gds = [rng.normal(size=(B, blk)) for blk, _ in specs]
    gd_dev = [torch.as_tensor(g, device=dev) for g in gds]
    segs_b = [KfbScatterSeg(s.block, s.n_map, None, s.src_idx, s.dst_idx, g.data_ptr()) for s, g in zip(segs_f, gd_dev)]
    gth = torch.full((B, nt), 123.0, dtype=torch.float64, device=dev)
    check(lib.kfb_scatter_backward_multi(B, nt, len(specs), (KfbScatterSeg * len(specs))(*segs_b), gth.data_ptr(), stream),
          "bwd_multi")
    torch.cuda.synchronize()
    ref = np.zeros((B, nt))
    for (blk, mp), g in zip(specs, gds):
        owner = {}
        for k, (a, b) in enumerate(mp):
            owner[b] = k
        for k, (a, b) in enumerate(mp):
            if owner[b] == k:
                ref[:, a] += g[:, b]
    assert np.allclose(gth.cpu().numpy(), ref, rtol=0, atol=1e-15)
    assert lib.kfb_scatter_forward_multi(B, nt, 9, arr, th.data_ptr(), stream) != 0  # more than KFB_MAX_SCATTER_SEGMENTS


@pytest.mark.gpu
def test_status_codes_for_non_stationary_draws_and_failed_dare():
    """ADVICE r1: the real cause of a failed draw is reported, not the follow-on "F_0 not positive definite".
    (a) stationary P0 requested for a draw with |rho| >= 1: KFB_INFO_NOT_STATIONARY, logp NaN, other draws untouched;
    (b) steady_state filter whose Riccati equation has no stabilising solution: KFB_INFO_DARE_FAILED."""
    from pymc_statespace_b200 import BatchedKalman
    from pymc_statespace_b200._lib import KFB_INFO_DARE_FAILED, KFB_INFO_NOT_STATIONARY
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import arma11_workload

    spec, y, theta = arma11_workload(64, 40)
    theta[5, 3] = 1.2   # rho: explosive AR root
    theta[9, 3] = 1.0   # unit root
    model = KalmanLogp(spec, y, n_draws=64)
    logp, grad = model.logp_and_grad(torch.as_tensor(theta, device="cuda"))
    info = model.info.cpu().numpy()
    assert info[5] == KFB_INFO_NOT_STATIONARY and info[9] == KFB_INFO_NOT_STATIONARY
    assert (np.delete(info, [5, 9]) == 0).all() and bool(torch.isnan(logp[[5, 9]]).all())
    assert bool(torch.isfinite(torch.cat([logp[:5], logp[10:]])).all())
    # (b) unobservable explosive state: no stabilising DARE solution
    n, dev = 20, "cuda"
    f = lambda a: torch.as_tensor(np.asarray(a, dtype=float), device=dev)  # noqa: E731
    bk = BatchedKalman("steady_state", n, 2, 1, 1, n_draws=2)
    T = np.stack([np.array([[0.5, 0.0], [0.0, 0.3]]), np.array([[0.5, 0.0], [0.0, 1.5]])])
    out = bk.forward(f(np.zeros((n, 1))), f(np.zeros(2)), f(np.eye(2)), f(T), f([[1.0, 0.0]]), f([[1.0], [1.0]]),
                     f([[1.0]]), f([[1.0]]))
    info = out["info"].cpu().numpy()
    assert info[0] == 0 and info[1] == KFB_INFO_DARE_FAILED and bool(torch.isnan(out["loglik"][1]))
    with pytest.raises(Exception, match="DARE"):
        bk.raise_on_info(out["info"])


@pytest.mark.gpu
@pytest.mark.parametrize("period,kind", [(12, "standard"), (24, "standard"), (12, "steady_state"), (7, "standard"),
                                         (9, "standard"), (15, "standard"), (16, "steady_state")])
def test_sizes_between_instantiations_are_padded_exactly(period, kind):
    """Seasonal models whose k_states falls between the fused instantiations (period 12 -> 13 states, period 24 -> 25):
    KalmanLogp embeds them in the next instantiated size (models.pad_spec: extra states identically zero).  logp and
    d logp / d theta must equal the un-padded evaluation on the generic run-time-dims kernels and the oracle."""
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.models import FUSED_K_STATES, trend_seasonal_spec

    spec = trend_seasonal_spec(period)
    rng = np.random.default_rng(period)
    B, n = 24, 60
    theta = np.exp(rng.normal(np.log([0.1, 0.01, 0.05, 0.5]), 0.2, size=(B, 4)))
    y = (np.sin(2 * np.pi * np.arange(n) / period) + np.cumsum(rng.normal(0, 0.3, n)) + rng.normal(0, 0.7, n))[:, None]
    y[[5, 17]] = np.nan
    th = torch.as_tensor(theta, device="cuda")
    padded = KalmanLogp(spec, y, n_draws=B, filter_type=kind)
    plain = KalmanLogp(spec, y, n_draws=B, filter_type=kind, pad_to_fused=False)
    m = spec.k_states
    assert plain.spec.k_states == m and padded.k_states_model == m
    assert padded.spec.k_states == (m if m in FUSED_K_STATES else min(k for k in FUSED_K_STATES if k >= m))
    lp1, g1 = padded.logp_and_grad(th)
    lp0, g0 = plain.logp_and_grad(th)
    assert int((padded.info != 0).sum()) == 0 and int((plain.info != 0).sum()) == 0
    gtol = 1e-6 if kind == "steady_state" else 1e-9
    assert float(((lp1 - lp0).abs() / lp0.abs()).max()) < 1e-11
    assert float(((g1 - g0).abs().amax(1) / g0.abs().amax(1)).max()) < gtol

    def mats(t):
        mm = spec.matrices(t.detach().numpy())
        T, Z, R = (torch.tensor(mm[k]) for k in ("T", "Z", "R"))
        Q = torch.zeros(3, 3, dtype=torch.float64)
        Q[0, 0], Q[1, 1], Q[2, 2] = t[0], t[1], t[2]
        return torch.zeros(m, 1, dtype=torch.float64), torch.eye(m, dtype=torch.float64), T, Z, R, t[3].reshape(1, 1), Q

    ll, gr = om.logp_and_grad_theta(mats, theta[3], y[:, :, None], kind)
    assert abs(float(lp1[3]) - ll) <= 1e-8 * abs(ll)
    assert np.abs(g1[3].cpu().numpy() - gr).max() <= (1e-6 if kind == "steady_state" else 1e-8) * np.abs(gr).max()
    # the full-output call reports the model's own states only
    out = padded.filter(th, outputs=("filtered_states", "predicted_covs", "loglik"))
    assert tuple(out["filtered_states"].shape) == (B, n, m) and tuple(out["predicted_covs"].shape) == (B, n + 1, m, m)


@pytest.mark.parametrize("m", [10, 16, 18, 30, 32])
def test_tensor_core_dare_matches_generic_solver_and_reports_failure(m):
    """steady_state at even k_states 10..32, k_endog 1: the forward DARE solve runs on the warp-per-draw tensor-core
    mapping (kf_rowsD.cuh: rowsD_dare).  Same fixed point as the generic solver (force_coop) and as scipy's
    solve_discrete_are (the oracle), and an unobservable explosive state is reported as KFB_INFO_DARE_FAILED."""
    from pymc_statespace_b200 import BatchedKalman
    from pymc_statespace_b200._lib import KFB_INFO_DARE_FAILED
    from oracle import kalman_numpy as kn
    from tests.helpers import random_system

    rng = np.random.default_rng(300 + m)
    B, n, p, r = 5, 12, 1, 3
    systems = [random_system(rng, m, p, r, n, scale_T=0.1) for _ in range(B)]
    Ts = np.stack([s[3] for s in systems])
    Ts[3] = 0.0
    Ts[3][np.arange(m), np.arange(m)] = 0.5
    Ts[3][m - 1, m - 1] = 1.5                      # explosive state ...
    Zs = np.stack([s[4] for s in systems])
    Zs[3][0, m - 1] = 0.0                          # ... that is not observed (and T is diagonal): no stabilising solution
    f = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")  # noqa: E731
    stack = lambda i: f(np.stack([s[i] for s in systems]))  # noqa: E731
    y = systems[0][0]
    res = {}
    for force in (False, True):
        bk = BatchedKalman("steady_state", n, m, p, r, n_draws=B, force_coop=force)
        out = bk.forward(f(y[..., 0]), stack(1), stack(2), f(Ts), f(Zs), stack(5), stack(6), stack(7))
        res[force] = (out["loglik"].cpu().numpy(), out["info"].cpu().numpy())
    for force in (False, True):
        ll, info = res[force]
        assert info[3] == KFB_INFO_DARE_FAILED and np.isnan(ll[3]), force
        assert (np.delete(info, 3) == 0).all()
    ok = [0, 1, 2, 4]
    assert np.abs(res[False][0][ok] - res[True][0][ok]).max() < 1e-10 * np.abs(res[True][0][ok]).max()
    for b in (0, 4):
        ref = kn.kalman_filter("steady_state", y, *systems[b][1:])
        assert abs(res[False][0][b] - float(ref[4])) < 1e-9 * abs(float(ref[4]))


@pytest.mark.gpu
def test_theta_level_smoother_matches_oracle():
    """KalmanLogp.smooth: filter + RTS smoother for every draw (reference build_statespace_graph + build_smoother_graph);
    VARMAX(2,0) with measurement error (fused row kernels + warp-per-unit smoother) and the 13-state seasonal model (padded
    to the 14-state tensor-core kernels).  (Models without measurement error, e.g. BayesianARMA, make P_hat singular to
    rounding at most steps: cond 1e15..1e18, where numpy's own pinv and an eigendecomposition pinv differ by 1e-5..1e-2 -
    no value test is meaningful there.)"""
    from oracle import kalman_numpy as kn
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.models import trend_seasonal_spec
    from pymc_statespace_b200.synthetic import varmax20_workload

    cases = []
    spec, y, theta = varmax20_workload(12, 40)
    cases.append((spec, y, theta, 1e-7))
    spec = trend_seasonal_spec(12)
    rng = np.random.default_rng(3)
    theta = np.exp(rng.normal(np.log([0.1, 0.01, 0.05, 0.5]), 0.2, size=(6, 4)))
    y = (np.sin(2 * np.pi * np.arange(40) / 12) + np.cumsum(rng.normal(0, 0.3, 40)) + rng.normal(0, 0.7, 40))[:, None]
    cases.append((spec, y, theta, 1e-6))  # pinv of a covariance whose state noise has rank 3: cond * eps
    for spec, y, theta, tol in cases:
        B = theta.shape[0]
        model = KalmanLogp(spec, y, n_draws=B)
        ss, sc, out = model.smooth(torch.as_tensor(theta, device="cuda"))
        m = model.k_states_model
        assert tuple(ss.shape) == (B, y.shape[0], m) and tuple(sc.shape) == (B, y.shape[0], m, m)
        for b in (0, B - 1):
            mats = spec.matrices(theta[b])
            args = [np.asarray(mats[k], dtype=float) for k in ("a0", "P0", "T", "Z", "R", "H", "Q")]
            if spec.stationary_initialization:
                import scipy.linalg as sl

                args[1] = sl.solve_discrete_lyapunov(args[2], args[4] @ args[6] @ args[4].T)
            o = kn.kalman_filter("standard", np.asarray(y, dtype=float).reshape(len(y), -1, 1), args[0].reshape(-1, 1), *args[1:])
            rs, rc = kn.kalman_smoother(args[2], args[4], args[6], o[0], o[2])
            assert rel_err_np(ss[b].cpu().numpy(), rs[..., 0]) < tol
            assert rel_err_np(sc[b].cpu().numpy(), rc) < tol


def rel_err_np(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300))


def test_bench_dump_outputs_are_the_timed_paths_results(tmp_path):
    """`bench.py --dump-outputs`: --steps sets the timed steps of both legs, and the dumped (logp, grad) of the headline
    ARMA(1,1) and c5 ARMA(2,1) legs equal a direct evaluation of the same seeded workloads."""
    import json
    import os
    import subprocess
    import sys

    from pymc_statespace_b200.synthetic import arma11_workload, arma21_workload
    from tests.helpers import ROOT

    B, B5, n, steps = 512, 4096, 64, 10
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--draws", str(B), "--n", str(n), "--c5-draws", str(B5), "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["steps"] == steps and line["c5"]["steps"] == steps
    assert sorted(os.listdir(tmp_path)) == ["c5_grad.npy", "c5_logp.npy", "grad.npy", "logp.npy"]
    for prefix, (spec, y, theta) in (("", arma11_workload(B, n)), ("c5_", arma21_workload(B5, n))):
        logp, grad, _ = _run(spec, y, theta)
        got_l, got_g = np.load(tmp_path / f"{prefix}logp.npy"), np.load(tmp_path / f"{prefix}grad.npy")
        assert got_l.dtype == np.float64 and got_g.dtype == np.float64
        assert got_l.shape == logp.shape and got_g.shape == grad.shape
        np.testing.assert_allclose(got_l, logp, rtol=1e-12, atol=0)
        np.testing.assert_allclose(got_g, grad, rtol=1e-12, atol=1e-12 * np.abs(grad).max())
