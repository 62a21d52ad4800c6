"""Time-parallel RTS smoother on the B200: kfb_smoother_ex with KFB_FLAG_TIME_PARALLEL, rts_smoother(time_parallel=...),
the smoother seam graph and KalmanSmootherOp.

Parity with the oracle (rtol 1e-8; Nile 1e-7 as the sequential smoother's own test), agreement with the sequential kernel
(1..64 units, one 65,536-step series), pinv units mixed with regular ones, the dense-moment known answer, determinism,
NaN positions, the k_states 6 fallback, graph capture per geometry, and the Op through the stand-in pytensor.
"""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from oracle import kalman_numpy as kn
from tests.helpers import nile_inputs, random_system, rel_err

pytestmark = pytest.mark.gpu

RTOL = 1e-8


def _dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device="cuda")


def _filtered(rng, m, n, n_missing=0):
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, 1, 2, n, n_missing=n_missing)
    out = kn.kalman_filter("standard", y, a0, P0, T, Z, R, H, Q)
    return T, R, Q, out[0], out[2]


def _batch(rng, m, B, n, per_draw=True, n_series=1):
    """B draws x n_series units of filtered moments from random systems (per-draw or shared T, R, Q)."""
    systems = [random_system(rng, m, 1, 2, n, n_missing=n // 10) for _ in range(B if per_draw else 1)]
    fs, fc = [], []
    for b in range(B):
        s = systems[b if per_draw else 0]
        for k in range(n_series):
            y = rng.normal(size=(n, 1, 1))
            y[rng.choice(n, n // 10, replace=False)] = np.nan
            o = kn.kalman_filter("standard", y, *s[1:])
            fs.append(o[0][..., 0])
            fc.append(o[2])
    mats = [np.stack([s[i] for s in systems]) if per_draw else systems[0][i] for i in (3, 5, 7)]
    return mats, np.stack(fs), np.stack(fc), systems


def _smooth(mats, fs, fc, tp, n_series=1):
    from pymc_statespace_b200 import rts_smoother

    ss, sc = rts_smoother(*[_dev(x) for x in mats], _dev(fs), _dev(fc), n_series=n_series, time_parallel=tp)
    return ss.cpu().numpy(), sc.cpu().numpy()


@pytest.mark.parametrize("m", [1, 2, 3, 4])
@pytest.mark.parametrize("n", [1, 7, 300, 2000])
def test_parity_with_the_oracle(m, n):
    rng = np.random.default_rng(100 * m + n)
    T, R, Q, fs, fc = _filtered(rng, m, n, n_missing=n // 10)
    ss, sc = _smooth((T, R, Q), fs[None, :, :, 0], fc[None], True)
    rs, rc = kn.kalman_smoother(T, R, Q, fs, fc)
    assert rel_err(ss[0], rs[..., 0]) < RTOL and rel_err(sc[0], rc) < RTOL


@pytest.mark.parametrize("per_draw", [True, False])
def test_series_per_draw_and_shared_matrices(per_draw):
    rng = np.random.default_rng(5 + per_draw)
    m, B, S, n = 2, 3, 2, 150
    mats, fs, fc, systems = _batch(rng, m, B, n, per_draw, n_series=S)
    ss, sc = _smooth(mats, fs, fc, True, n_series=S)
    for u in range(B * S):
        s = systems[u // S if per_draw else 0]
        rs, rc = kn.kalman_smoother(s[3], s[5], s[7], fs[u][..., None], fc[u])
        assert rel_err(ss[u], rs[..., 0]) < RTOL and rel_err(sc[u], rc) < RTOL, u


def test_nile():
    from pymc_statespace_b200.filters import KalmanSmoother, StandardFilter

    inputs = nile_inputs(5)
    outs = StandardFilter().build_graph(*inputs)
    sm = KalmanSmoother()
    sm.time_parallel = True
    ss, sc = sm.build_graph(inputs[3], inputs[5], inputs[7], outs[0], outs[2])
    rs, rc = kn.kalman_smoother(inputs[3], inputs[5], inputs[7], outs[0], outs[2])
    np.testing.assert_allclose(ss, rs, rtol=1e-7, atol=1e-7)
    np.testing.assert_allclose(sc[5:], rc[5:], rtol=1e-7, atol=1e-7)


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_agrees_with_the_sequential_kernel(m):
    rng = np.random.default_rng(20 + m)
    for B in (1, 2, 5, 64):
        mats, fs, fc, _ = _batch(rng, m, B, 400)
        a, b = _smooth(mats, fs, fc, True), _smooth(mats, fs, fc, False)
        assert rel_err(a[0], b[0]) < 1e-9 and rel_err(a[1], b[1]) < 1e-9, B


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_units_take_the_scan_path(m):
    """The sequential fallback reproduces the sequential kernel bit for bit; the scan path starts every chunk but the
    last from scanned moments, which differ from the sequential ones in the last bits.  So a result that agrees to
    rounding but not in every bit shows that the unit was not sent to the fallback."""
    rng = np.random.default_rng(60 + m)
    if m == 1:
        # a random system's gains shrink a chunk's E below rounding, so scan and walk meet in every bit; a local level
        # with small state noise has gains near 1
        n = 4000
        mats, fs, fc = (np.eye(1), np.eye(1), np.array([[0.01]])), [], []
        for _ in range(4):
            y = np.cumsum(rng.normal(size=n))[:, None, None] + rng.normal(size=(n, 1, 1))
            o = kn.kalman_filter("standard", y, np.zeros((1, 1)), np.eye(1), mats[0], np.eye(1), mats[1], np.eye(1),
                                 mats[2])
            fs.append(o[0][..., 0])
            fc.append(o[2])
        fs, fc = np.stack(fs), np.stack(fc)
    else:
        mats, fs, fc, _ = _batch(rng, m, 4, 4000)
    a, b = _smooth(mats, fs, fc, True), _smooth(mats, fs, fc, False)
    assert rel_err(a[0], b[0]) < 1e-9 and rel_err(a[1], b[1]) < 1e-9
    for u in range(4):
        assert not (np.array_equal(a[0][u], b[0][u]) and np.array_equal(a[1][u], b[1][u])), u


def test_long_series():
    from pymc_statespace_b200 import BatchedKalman

    rng = np.random.default_rng(9)
    n = 65536
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 2, 1, 2, n, n_missing=100)
    bk = BatchedKalman("standard", n, 2, 1, 2, n_draws=1)
    out = bk.forward(_dev(y[..., 0]), *[_dev(x) for x in (a0, P0, T, Z, R, H, Q)],
                     outputs=("filtered_states", "filtered_covs"))
    fs, fc = out["filtered_states"].cpu().numpy(), out["filtered_covs"].cpu().numpy()
    a, b = _smooth((T, R, Q), fs, fc, True), _smooth((T, R, Q), fs, fc, False)
    assert rel_err(a[0], b[0]) < 1e-9 and rel_err(a[1], b[1]) < 1e-9


@pytest.mark.parametrize("m", [2, 3, 4])
def test_pinv_units_mixed_with_regular_ones(m):
    rng = np.random.default_rng(40 + m)
    B, n = 4, 300
    fs = rng.normal(size=(B, n, m))
    A = rng.normal(size=(B, n, m, m))
    fc = A @ np.swapaxes(A, -1, -2) + 0.1 * np.eye(m)
    T = np.tile(np.eye(m), (B, 1, 1)) * 0.9
    R = np.zeros((B, m, 1))
    R[:, 0, 0] = 1.0
    Q = np.tile(np.array([[0.5]]), (B, 1, 1))
    for b in (1, 3):  # the last state is known exactly at every step: P_hat is singular
        fc[b, :, m - 1, :] = 0.0
        fc[b, :, :, m - 1] = 0.0
    ss, sc = _smooth((T, R, Q), fs, fc, True)
    for b in range(B):
        rs, rc = kn.kalman_smoother(T[b], R[b], Q[b], fs[b][..., None], fc[b])
        assert rel_err(ss[b], rs[..., 0]) < RTOL and rel_err(sc[b], rc) < RTOL, b


def test_dense_gaussian_known_answer():
    rng = np.random.default_rng(77)
    n = 14
    for m in (1, 2, 3):
        y, a0, P0, T, Z, R, H, Q = random_system(rng, m, 1, 2, n, n_missing=3)
        out = kn.kalman_filter("standard", y, a0, P0, T, Z, R, H, Q)
        cond = kn.dense_gaussian_state_moments(y, a0, P0, T, Z, R, H, Q)
        ss, sc = _smooth((T, R, Q), out[0][None, :, :, 0], out[2][None], True)
        for t in range(n):
            mu, cov = cond(t, n - 1)
            assert rel_err(ss[0, t], mu[:, 0]) < 1e-10 and rel_err(sc[0, t], cov) < 1e-10, (m, t)


def test_two_runs_give_identical_bits():
    rng = np.random.default_rng(3)
    mats, fs, fc, _ = _batch(rng, 3, 8, 3000)
    a, b = _smooth(mats, fs, fc, True), _smooth(mats, fs, fc, True)
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1], b[1])


def test_nan_positions_match_the_sequential_kernel():
    rng = np.random.default_rng(4)
    mats, fs, fc, _ = _batch(rng, 2, 3, 2000)
    fs[1, 1500, 0] = np.nan  # inside a late chunk
    fc[2, 3, 1, 1] = np.nan  # inside the first chunk
    a, b = _smooth(mats, fs, fc, True), _smooth(mats, fs, fc, False)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(np.isnan(x), np.isnan(y))
        assert np.isnan(x).any()
        ok = ~np.isnan(y)
        assert rel_err(x[ok], y[ok]) < 1e-9


def test_k_states_6_runs_the_sequential_kernel():
    rng = np.random.default_rng(6)
    mats, fs, fc, _ = _batch(rng, 6, 3, 50)
    a, b = _smooth(mats, fs, fc, True), _smooth(mats, fs, fc, False)
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1], b[1])


def test_seam_graph_captured_once_per_geometry():
    from pymc_statespace_b200 import seam

    rng = np.random.default_rng(8)
    seam._SMOOTH_CACHE.clear()
    for tp in (True, False):
        for seed in range(3):
            T, R, Q, fs, fc = _filtered(np.random.default_rng(seed), 2, 500, n_missing=20)
            ss, sc = seam.smooth_numpy(T, R, Q, fs, fc, time_parallel=tp)
            rs, rc = kn.kalman_smoother(T, R, Q, fs, fc)
            assert ss.shape == (500, 2, 1) and sc.shape == (500, 2, 2)
            assert rel_err(ss, rs) < RTOL and rel_err(sc, rc) < RTOL
    assert len(seam._SMOOTH_CACHE) == 2
    T, R, Q, fs, fc = _filtered(rng, 2, 501)
    seam.smooth_numpy(T, R, Q, fs, fc, time_parallel=True)
    assert len(seam._SMOOTH_CACHE) == 3


SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fake_pytensor")


@pytest.fixture()
def shim_sm():
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


def test_smoother_op_perform_without_pytensor():
    from pymc_statespace_b200.pytensor_op import KalmanSmootherOp

    T, R, Q, fs, fc = _filtered(np.random.default_rng(12), 3, 200, n_missing=10)
    store = [[None], [None]]
    KalmanSmootherOp(True).perform(None, [T, R, Q, fs, fc], store)
    rs, rc = kn.kalman_smoother(T, R, Q, fs, fc)
    assert rel_err(store[0][0], rs) < RTOL and rel_err(store[1][0], rc) < RTOL


def test_smoother_op_through_the_stand_in(shim_sm):
    pop, pytensor = shim_sm
    import pytensor.tensor as pt

    from pymc_statespace_b200.filters import KalmanSmoother, StandardFilter

    assert pop.KalmanSmootherOp() == pop.KalmanSmootherOp(False)
    assert pop.KalmanSmootherOp() != pop.KalmanSmootherOp(True)
    rng = np.random.default_rng(31)
    m, n = 2, 300
    args = list(random_system(rng, m, 1, 2, n, n_missing=5))
    names = ["data", "a0", "P0", "T", "Z", "R", "H", "Q"]
    ins = [pt.dtensor3(k) if k == "data" else pt.dmatrix(k) for k in names]
    flt = StandardFilter()
    flt.time_parallel = True
    outs = flt.build_graph(*ins)
    sm = KalmanSmoother()
    sm.time_parallel = True
    sm_outs = sm.build_graph(ins[3], ins[5], ins[7], outs[0], outs[2])
    node = sm_outs[0].owner
    assert isinstance(node.op, pop.KalmanSmootherOp) and node.op.time_parallel
    shapes = node.op.infer_shape(None, node, [(m, m), (m, 2), (2, 2), (n, m, 1), (n, m, m)])
    assert [tuple(s) for s in shapes] == [(n, m, 1), (n, m, m)]
    shapes = node.op.infer_shape(None, node, [(m, m), (m, 2), (2, 2), (n, m), (n, m, m)])  # 2-D filtered_states
    assert [tuple(s) for s in shapes] == [(n, m, 1), (n, m, m)]
    f = pytensor.function(ins, sm_outs)
    ss, sc = f(*args)
    o = kn.kalman_filter("standard", *args)
    rs, rc = kn.kalman_smoother(args[3], args[5], args[7], o[0], o[2])
    assert rel_err(ss, rs) < RTOL and rel_err(sc, rc) < RTOL
    with pytest.raises(NotImplementedError, match="smoothed_states"):
        pytensor.grad(sm_outs[0], [ins[3]])
    with pytest.raises(NotImplementedError, match="time-varying"):
        sm.build_graph(pt.dtensor3("T"), ins[5], ins[7], outs[0], outs[2])
