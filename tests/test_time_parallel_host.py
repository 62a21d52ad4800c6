"""Time-parallel form (KFB_FLAG_TIME_PARALLEL) without a GPU.

* The filtering-element, affine and congruence combination operators of csrc/kf_tpar.cuh, compiled for the host
  (tests/tpar_host), folded in chunks and scanned in several tree shapes, give the oracle's sequential moments and
  cotangents: m = 1..4, missing rows (first and last included), c / d, time-varying matrices, non-symmetric P0.
* The plan logic of the C ABI: the flag on a geometry outside the time-parallel form is KFB_ERR_UNSUPPORTED, and
  kfb_workspace_bytes sizes the per-unit tape the forward pass always writes.
"""
import ctypes

import numpy as np
import pytest

from oracle import kalman_numpy as kn
from oracle import kalman_torch as kt
from tests import tpar_host
from tests.helpers import nile_inputs, random_system, rel_err

TOL = 1e-11


def _check(kind, args, c=None, d=None, strict=True, w=None, chunks=(1, 3, 8, 64), trees=(0, 1, 2), tol=TOL, gtol=None):
    gtol = gtol or {}
    ref = kn.kalman_filter(kind, *args, c=c, d=d, strict_reference=strict)
    _, gt = kt.loglik_and_grads(kind, *args, c=c, d=d, strict_reference=strict, g_ll_obs=w)
    for nch in chunks:
        for tree in trees:
            outs, g, info, seq = tpar_host.run(kind, *args, c=c, d=d, strict=strict, nchunks=nch, tree=tree,
                                               seed=nch * 7 + tree, g_ll_obs=w, g_loglik=(0.0 if w is not None else None))
            assert info == 0 and not seq
            for name, a, b in zip(("fs", "ps", "fc", "pc", "loglik", "ll_obs"), outs, ref):
                assert rel_err(a, b) < tol, (kind, nch, tree, name, rel_err(a, b))
            for k in gt:
                assert rel_err(g[k], gt[k]) < gtol.get(k, tol) or np.abs(g[k] - gt[k]).max() < 1e-13, (kind, nch, tree, k)


@pytest.mark.parametrize("m", [1, 2, 3, 4])
@pytest.mark.parametrize("n", [1, 2, 3, 31])
def test_scan_shapes_match_sequential_recursion(m, n):
    rng = np.random.default_rng(100 * m + n)
    args = random_system(rng, m, 1, 2, n)
    y = args[0].copy()
    if n >= 4:
        y[[0, n - 1, n // 2]] = np.nan  # first, last and one in between
    elif n == 3:
        y[[0, 2]] = np.nan
    args = (y,) + args[1:]
    c, d = rng.normal(size=(m, 1)), rng.normal(size=(1, 1))
    _check("standard", args, c, d)
    _check("standard", args, c, d, strict=False, w=rng.normal(size=n))


@pytest.mark.parametrize("kind", ["standard", "single", "cholesky"])
@pytest.mark.parametrize("strict", [True, False])
def test_filter_kinds_and_nonsymmetric_P0(kind, strict):
    rng = np.random.default_rng(7)
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 3, 1, 2, 40, n_missing=4)
    P0 = P0 + 0.3 * rng.normal(size=P0.shape)  # full-matrix P0 (its gradient keeps the sequential gauge)
    _check(kind, (y, a0, P0, T, Z, R, H, Q), None, rng.normal(size=(1, 1)), strict=strict, chunks=(5, 16))


def test_time_varying_matrices():
    rng = np.random.default_rng(3)
    n, m = 29, 3
    systems = [random_system(rng, m, 1, 2, n, n_missing=3) for _ in range(n)]
    y, a0, P0 = systems[0][:3]
    T, Z, R, H, Q = (np.stack([s[i] for s in systems]) for i in range(3, 8))
    c, d = rng.normal(size=(n, m, 1)), rng.normal(size=(n, 1, 1))
    _check("standard", (y, a0, P0, T, Z, R, H, Q), c, d, chunks=(1, 4, 9))
    _check("single", (y, a0, P0, T[0], Z, R[0], H, Q), c[0], d, strict=False, w=rng.normal(size=n), chunks=(6,))


def test_nile_diffuse_start():
    """P0 = 1e6 I: the P0 cotangent (~5e-7) is what is left of a cancellation in the step-0 adjoint, so it keeps ~1e-7
    of relative error (the sequential predictor-form math: ~1e-9); d-bar inherits ~1e-10.  Everything else ~1e-11."""
    for n_missing in (0, 5):
        _check("standard", nile_inputs(n_missing), chunks=(1, 16, 256), trees=(1, 2), tol=1e-10,
               gtol={"P0": 1e-6, "d": 1e-9})


def test_undefined_element_takes_the_sequential_walk():
    """Z C Z^T + H = 0: the observed state carries no noise of its own; the unit runs the sequential recursion."""
    rng = np.random.default_rng(5)
    n = 30
    y = rng.normal(size=(n, 1, 1))
    y[[4, 17]] = np.nan
    a0, P0 = rng.normal(size=(2, 1)), np.eye(2)
    T = np.array([[0.5, 0.8], [0.0, 0.3]])
    Z, R, H, Q = np.array([[1.0, 0.0]]), np.array([[0.0], [1.0]]), np.zeros((1, 1)), np.eye(1)
    args = (y, a0, P0, T, Z, R, H, Q)
    ref = kn.kalman_filter("standard", *args)
    _, gt = kt.loglik_and_grads("standard", *args)
    outs, g, info, seq = tpar_host.run("standard", *args, nchunks=8)
    assert seq == 1 and info == 0
    for a, b in zip(outs, ref):
        assert rel_err(a, b) < TOL
    for k in gt:
        assert rel_err(g[k], gt[k]) < 1e-10 or np.abs(g[k] - gt[k]).max() < 1e-12, k


def test_expanding_elements_fail_the_check_and_take_the_sequential_walk():
    """ARMA(1,1) with a non-invertible MA part (|theta| > 1): the filter is stable, but the filtering elements' own
    transition (I - K Z) T has the eigenvalue -theta, so chunk aggregates grow like theta^k and the scan's moments drift.
    The consistency check of the map catches it and the unit is re-run by the sequential recursion."""
    import torch

    from oracle import models as om

    rng = np.random.default_rng(17)
    n = 300
    y = rng.normal(size=(n, 1, 1))
    a0, P0, T, Z, R, H, Q = (x.detach().numpy() for x in om.arma_matrices(
        torch.tensor([0.3, -0.1, 0.9, 0.5, -1.66], dtype=torch.float64), (1, 1), True))
    args = (y, a0.reshape(-1, 1), P0, T, Z, R, H, Q)
    ref = kn.kalman_filter("standard", *args)
    _, gt = kt.loglik_and_grads("standard", *args)
    outs, g, info, walk = tpar_host.run("standard", *args, nchunks=256)
    assert walk == 2 and info == 0
    for a, b in zip(outs, ref):
        assert rel_err(a, b) < TOL
    for k in gt:
        assert rel_err(g[k], gt[k]) < 1e-9 or np.abs(g[k] - gt[k]).max() < 1e-12, k


def test_info_when_F0_is_not_positive():
    rng = np.random.default_rng(6)
    y, a0, P0, T, Z, R, H, Q = random_system(rng, 2, 1, 1, 20)
    Z = np.array([[1.0, 0.0]])
    P0 = np.diag([0.0, 1.0])
    _, _, info, _ = tpar_host.run("standard", y, a0, P0, T, Z, R, np.zeros((1, 1)), Q, do_bwd=False)
    assert info == 1


# ---------------------------------------------------------------------------------------------- C ABI plan logic
def _desc(kind="standard", m=2, p=1, n=100, draws=3, flags=128):
    from pymc_statespace_b200 import _lib

    d = _lib.KfbDesc()
    d.filter_kind, d.flags = _lib.FILTER_KIND[kind], flags
    d.n_draws, d.n_series, d.n, d.m, d.p, d.r = draws, 1, n, m, p, 1
    d.T_bs = m * m
    return d


def _ws(d, save):
    from pymc_statespace_b200 import _lib

    nb = ctypes.c_size_t(0)
    st = _lib.load().kfb_workspace_bytes(ctypes.byref(d), save, ctypes.byref(nb))
    return st, nb.value


@pytest.mark.parametrize("kind,m,p", [("standard", 5, 1), ("standard", 2, 2), ("univariate", 2, 1),
                                      ("steady_state", 2, 1), ("cholesky", 6, 3)])
def test_flag_outside_scope_is_unsupported(kind, m, p):
    from pymc_statespace_b200 import _lib

    assert _lib.KFB_FLAG_TIME_PARALLEL == 128
    st, _ = _ws(_desc(kind, m, p), 1)
    assert st == _lib.KFB_ERR_UNSUPPORTED
    st, _ = _ws(_desc(kind, m, p, flags=0), 1)
    assert st == _lib.KFB_OK


@pytest.mark.parametrize("m", [1, 2, 4])
def test_workspace_holds_the_per_unit_tape(m):
    from pymc_statespace_b200 import _lib

    U, n = 3, 100
    tape = U * n * (m + m * m) * 8
    for save in (0, 1):
        st, nb = _ws(_desc(m=m, n=n, draws=U), save)
        assert st == _lib.KFB_OK
        # C = R Q R^T (shared), the tape (forward and adjoint alike), and the per-unit C-bar for the adjoint
        assert tape <= nb <= tape + 2 * 256 + (U * m * m * 8 + 256) * save + m * m * 8 + 256
    st_seq, nb_seq = _ws(_desc(m=m, n=n, draws=U, flags=0), 0)
    assert st_seq == _lib.KFB_OK and nb_seq < tape  # the sequential forward keeps no tape without save_for_backward


def test_forward_rejects_a_workspace_sized_without_the_flag():
    """kfb_forward checks the workspace against the plan of the descriptor it is given (no device call is reached)."""
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    d = _desc(m=2, n=100, draws=3)
    _, need = _ws(d, 0)
    _, small = _ws(_desc(m=2, n=100, draws=3, flags=0), 0)
    assert small < need
    buf = ctypes.create_string_buffer(8)
    ptr = ctypes.cast(buf, ctypes.c_void_p)
    ins = _lib.KfbInputs(*([ptr] * 10))
    outs = _lib.KfbOutputs(*([None] * 7))
    st = lib.kfb_forward(ctypes.byref(d), ctypes.byref(ins), ctypes.byref(outs), ptr, small, 0, None)
    assert st == _lib.KFB_ERR_WORKSPACE
