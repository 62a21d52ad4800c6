"""Time-parallel RTS smoother (kfb_smoother_ex with KFB_FLAG_TIME_PARALLEL) without a GPU.

* The fold, suffix scan and checked walk of csrc/kf_tpar_smooth.cuh, compiled for the host (tests/hostsim), in
  several chunk counts and scan-tree shapes, give the oracle's smoothed moments: m = 1..4, missing rows in the filtered
  series, non-symmetric filtered covariances, singular predicted covariances (the pinv branch), the Nile fixture.
* With a zero drift tolerance the unit falls back to the sequential recursion and reproduces it bit for bit.
* A known answer that shares no recursion: the dense joint Gaussian's smoothed moments.
* The plan logic of kfb_smoother_ex: unsupported k_states and unknown flag bits are refused before any device call.
"""
import ctypes

import numpy as np
import pytest

from oracle import kalman_numpy as kn
from tests import hostsim
from tests.helpers import nile_inputs, random_system, rel_err

TOL = 1e-12  # the sequential smoother itself agrees with the oracle (SVD pinv) to ~1e-13
CHUNKS = (1, 2, 3, 8, 64, 256)
TREES = (0, 1, 2)


def _filtered(rng, m, n, n_missing=0):
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, 1, 2, n, n_missing=n_missing)
    out = kn.kalman_filter("standard", y, a0, P0, T, Z, R, H, Q)
    return T, R, Q, out[0], out[2]


def _check(T, R, Q, fs, fc, tol=TOL, chunks=CHUNKS, trees=TREES, skip=0):
    rs, rc = kn.kalman_smoother(T, R, Q, fs, fc)
    for nch in chunks:
        for tree in trees:
            ss, sc, fb = hostsim.tpar_smooth(T, R, Q, fs, fc, nchunks=nch, tree=tree, seed=nch * 7 + tree)
            assert fb == 0, (nch, tree)
            assert rel_err(ss, rs) < tol, (nch, tree, rel_err(ss, rs))
            assert rel_err(sc[skip:], rc[skip:]) < tol, (nch, tree, rel_err(sc, rc))


@pytest.mark.parametrize("m", [1, 2, 3, 4])
@pytest.mark.parametrize("n", [1, 2, 3, 37, 500])
def test_scan_shapes_match_the_oracle(m, n):
    rng = np.random.default_rng(10 * m + n)
    _check(*_filtered(rng, m, n, n_missing=min(n // 5, 40)))


@pytest.mark.parametrize("m", [2, 4])
def test_nonsymmetric_filtered_covariances(m):
    """Any matrix: the recursion neither reads nor keeps only sym(P).  The oracle's pinv of a non-symmetric P_hat is not
    the smoother's (kf_smooth.cuh inverts sym(P_hat)), so the reference here is the sequential smoother."""
    rng = np.random.default_rng(3 + m)
    T, R, Q, fs, fc = _filtered(rng, m, 60)
    fc = fc + 1e-3 * rng.normal(size=fc.shape)
    rs, rc = hostsim.smoother(T, R, Q, fs, fc, static_dims=True)
    assert np.abs(rc - np.swapaxes(rc, -1, -2)).max() > 1e-4
    for nch in CHUNKS:
        for tree in TREES:
            ss, sc, fb = hostsim.tpar_smooth(T, R, Q, fs, fc, nchunks=nch, tree=tree, seed=nch * 7 + tree)
            assert fb == 0
            assert rel_err(ss, rs) < TOL and rel_err(sc, rc) < TOL, (nch, tree)


@pytest.mark.parametrize("m", [2, 3, 4])
def test_singular_predicted_covariance_takes_the_pinv_branch(m):
    """A state without noise and without uncertainty: P_hat is singular and the gain comes from the Jacobi pinv."""
    rng = np.random.default_rng(40 + m)
    n = 40
    fs = rng.normal(size=(n, m, 1))
    A = rng.normal(size=(n, m, m))
    fc = A @ np.swapaxes(A, -1, -2) + 0.1 * np.eye(m)
    fc[:, m - 1, :] = 0.0
    fc[:, :, m - 1] = 0.0
    T = np.eye(m) * 0.9
    R = np.zeros((m, 1))
    R[0, 0] = 1.0
    Q = np.array([[0.5]])
    _check(T, R, Q, fs, fc, tol=1e-12)


def test_nile_diffuse_start():
    """P0 = 1e6 I; the first covariances carry the cancellation of the diffuse start (the reference's own tests skip the
    first five), elsewhere the pinv of the oracle's SVD and the Cholesky solve agree to ~1e-12."""
    for n_missing in (0, 5):
        args = nile_inputs(n_missing)
        out = kn.kalman_filter("standard", *args)
        _check(args[3], args[5], args[7], out[0], out[2], tol=1e-11, chunks=(1, 16, 256), skip=5)


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_zero_tolerance_falls_back_to_the_sequential_recursion(m):
    rng = np.random.default_rng(70 + m)
    args = _filtered(rng, m, 200, n_missing=10)
    seq_s, seq_c = hostsim.smoother(*args, static_dims=True)
    ss, sc, fb = hostsim.tpar_smooth(*args, nchunks=16, tol=0.0)
    assert fb == 1 or m == 1  # at k_states 1 the scan may meet the walk in every bit
    np.testing.assert_array_equal(ss, seq_s)
    np.testing.assert_array_equal(sc, seq_c)
    # one chunk: the walk is the sequential recursion itself, so even a zero tolerance passes
    ss, sc, fb = hostsim.tpar_smooth(*args, nchunks=1, tol=0.0)
    assert fb == 0
    np.testing.assert_array_equal(ss, seq_s)
    np.testing.assert_array_equal(sc, seq_c)


@pytest.mark.parametrize("m", [1, 2, 3])
def test_dense_gaussian_smoothed_moments(m):
    """E[x_t | y_0..y_{n-1}] and its covariance from the dense joint density (no recursion shared)."""
    rng = np.random.default_rng(90 + m)
    n = 14
    y, a0, P0, T, Z, R, H, Q = random_system(rng, m, 1, 2, n, n_missing=3)
    out = kn.kalman_filter("standard", y, a0, P0, T, Z, R, H, Q)
    cond = kn.dense_gaussian_state_moments(y, a0, P0, T, Z, R, H, Q)
    for nch, tree in ((1, 1), (4, 1), (14, 2)):
        ss, sc, fb = hostsim.tpar_smooth(T, R, Q, out[0], out[2], nchunks=nch, tree=tree, seed=nch)
        assert fb == 0
        for t in range(n):
            mu, cov = cond(t, n - 1)
            assert rel_err(ss[t], mu) < 1e-10, (t, nch)
            assert rel_err(sc[t], cov) < 1e-10, (t, nch)


# ---------------------------------------------------------------------------------------------- C ABI plan logic
def _call(m, flags, r=1):
    from pymc_statespace_b200 import _lib

    buf = ctypes.create_string_buffer(8)
    ptr = ctypes.cast(buf, ctypes.c_void_p)
    ws = ctypes.create_string_buffer(8 * m * m)
    return _lib.load().kfb_smoother_ex(1, 1, 10, m, r, ptr, 0, ptr, 0, ptr, 0, ptr, ptr, ptr, ptr,
                                       ctypes.cast(ws, ctypes.c_void_p), 8 * m * m, flags, None)


def test_flag_at_k_states_5_is_unsupported():
    from pymc_statespace_b200 import _lib

    assert _call(5, _lib.KFB_FLAG_TIME_PARALLEL) == _lib.KFB_ERR_UNSUPPORTED


@pytest.mark.parametrize("flags", [1, 64, 256, 128 | 2, 1 << 31])
def test_unknown_flag_bits_are_invalid(flags):
    from pymc_statespace_b200 import _lib

    assert _call(2, flags) == _lib.KFB_ERR_INVALID_ARG
