"""The compressed tape of the reduced ARMA recursion (kf_p1.cuh ZU_REDUCED, CTape in kf_core.cuh): entries
(v_t, 1 / F_t, P_t[0][1 .. m-2]) in blocks of KF_CTAPE_STEPS = 4 steps per warp.  Series lengths around the block size
cover a partial first block (n - 1 not a multiple of 4) and the bottom block, whose step 0 is not taped.  Without c-bar
and d-bar requested the reduced sweep skips them; the other cotangents must not move by a bit."""
import numpy as np
import pytest
import torch

from oracle import kalman_torch as kt
from tests import hostsim
from tests.helpers import random_system, rel_err

S = 4  # KF_CTAPE_STEPS
LENGTHS = (1, 2, 3, S, S + 1, S + 2, S + 3, 2 * S, 2 * S + 1, 13)


def _arma_like(rng, m, n):
    args = list(random_system(rng, m, 1, 1, n))
    args[4] = np.eye(m)[:1].copy()                       # Z = e_0
    args[6] = np.zeros((1, 1))                           # H = 0
    Tc = np.zeros((m, m))
    Tc[:, 1:] = np.eye(m)[:, :m - 1]
    Tc[:, 0] = rng.uniform(-0.5, 0.5, size=m) / np.arange(1, m + 1)
    args[3] = Tc
    args[2] = args[2] + 0.05 * rng.normal(size=(m, m))   # non-symmetric P0
    return args


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_ctape_block_edges_on_host(m):
    """Every n around the block size: the compressed tape gives the loglik and cotangents of the full-tape kernels
    (companion T promised, missing observations allowed) and of torch-autograd of the oracle."""
    rng = np.random.default_rng(900 + m)
    for n in LENGTHS:
        args = _arma_like(rng, m, n)
        c, d = rng.normal(size=(m, 1)), rng.normal(size=(1, 1))
        for w in (None, rng.normal(size=n)):
            kw = dict(c=c, d=d, static_dims=True, full=False, pred=True, p1=True, g_ll_obs=w,
                      g_loglik=(0.0 if w is not None else None), skip=("Z", "H"), z_unit0=True, h_zero=True,
                      t_companion=True)
            o0, g0, i0 = hostsim.run("standard", *args, **kw)
            o1, g1, i1 = hostsim.run("standard", *args, no_missing=True, **kw)
            assert i0 == 0 and i1 == 0 and abs(o1[4] - o0[4]) <= 1e-13 * abs(o0[4]), n
            _, gt = kt.loglik_and_grads("standard", *args, c=c, d=d, g_ll_obs=w)
            for k in gt:
                if k in ("Z", "H"):
                    continue
                a, b, t = g1[k], g0[k], gt[k]
                if k == "T":
                    a, b, t = (np.asarray(v).reshape(m, m)[:, 0] for v in (a, b, t))
                assert rel_err(a, b) < 1e-11 or np.abs(a - b).max() < 1e-13, (k, n)
                assert rel_err(a, t) < 1e-9 or np.abs(a - t).max() < 1e-13, (k, n)


@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_ctape_skipping_c_d_keeps_other_cotangents_bitwise_on_host(m):
    """KalmanLogp for BayesianARMA requests a0, P0, T, R, Q only: the reduced sweep then drops c-bar and d-bar (the
    instantiation with_adjoint_variant picks for the request, run on the host by tests/hostsim).  The cotangents
    that are requested are bit-identical to a run that requests everything, and agree with the oracle."""
    rng = np.random.default_rng(950 + m)
    for n in (2, S + 2, 25):
        y, a0, P0, T, Z, R, H, Q = _arma_like(rng, m, n)
        c, d = rng.normal(size=(m, 1)), rng.normal(size=(1, 1))
        for w in (None, rng.normal(size=n)):
            kw = dict(c=c, d=d, static_dims=True, full=False, pred=True, p1=True, g_ll_obs=w, z_unit0=True, h_zero=True,
                      t_companion=True, no_missing=True)
            o1, g_all, i1 = hostsim.run("standard", y, a0, P0, T, Z, R, H, Q, skip=("Z", "H"), **kw)
            o0, g_some, i0 = hostsim.run("standard", y, a0, P0, T, Z, R, H, Q, skip=("Z", "H", "c", "d"), **kw)
            ll0, ll1 = o0[4], o1[4]
            assert i0 == 0 and i1 == 0 and ll0 == ll1
            assert np.abs(g_all["c"]).max() > 0.0 and not np.any(g_some["c"]) and not np.any(g_some["d"])
            for k in ("a0", "P0", "T", "R", "Q"):
                assert np.array_equal(g_some[k], g_all[k]), (k, n)
            _, gt = kt.loglik_and_grads("standard", y, a0, P0, T, Z, R, H, Q, c=c, d=d,
                                        g_ll_obs=None if w is None else 1.0 + w)
            got = {"a0": g_some["a0"], "P0": g_some["P0"], "T": g_some["T"][:, 0], "Q": g_some["Q"],
                   "c": g_all["c"], "d": g_all["d"]}
            ref = {"a0": np.ravel(gt["a0"]), "P0": gt["P0"], "T": np.asarray(gt["T"])[:, 0], "Q": gt["Q"],
                   "c": np.ravel(gt["c"]), "d": np.ravel(gt["d"])}
            for k in got:
                a, t = np.ravel(got[k]), np.ravel(ref[k])
                assert rel_err(a, t) < 1e-9 or np.abs(a - t).max() < 1e-13, (k, n)


def _dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device="cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 2, 3, 4])
def test_p1_ctape_block_edges(m):
    """The kernels at every n around the block size, with 45 units (a partial last warp): the compressed tape (hot-path
    and full-output forward) against the full tape, and without c-bar / d-bar bit-identical to with them."""
    from pymc_statespace_b200 import BatchedKalman
    from tests.test_gpu_parity import ALL_OUT

    rng = np.random.default_rng(970 + m)
    B, r = 45, 1
    Z, H = np.eye(m)[:1], np.zeros((1, 1))
    for n in LENGTHS:
        systems = [_arma_like(rng, m, n) for _ in range(B)]
        y = systems[0][0]
        stack = lambda i: _dev(np.stack([s[i] for s in systems]))  # noqa: E731
        ins = (_dev(y[..., 0]), stack(1)[..., 0], stack(2), stack(3), _dev(Z), stack(5), _dev(H), stack(7))
        cs, ds = rng.normal(size=(B, m)), rng.normal(size=(B, 1))
        gobs = rng.normal(size=(B, n))
        for w in (None, gobs):
            res = {}
            for variant, wrt in (("plain", ("a0", "P0", "T", "R", "Q", "c", "d")),
                                 ("compressed", ("a0", "P0", "T", "R", "Q", "c", "d")),
                                 ("compressed_full_forward", ("a0", "P0", "T", "R", "Q", "c", "d")),
                                 ("compressed_no_cd", ("a0", "P0", "T", "R", "Q"))):
                bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, z_unit0=True, h_zero=True, t_companion=True,
                                   no_missing=variant != "plain")
                outs = ALL_OUT if variant == "compressed_full_forward" else ("loglik",)
                out = bk.forward(*ins, c=_dev(cs), d=_dev(ds), outputs=outs, save_for_backward=True)
                g = bk.backward(g_loglik=None if w is None else _dev(np.full(B, 0.5)),
                                g_ll_obs=None if w is None else _dev(w), wrt=wrt)
                assert int((out["info"] != 0).sum()) == 0, (variant, n)
                res[variant] = {k: v.cpu().numpy() for k, v in g.items()}
                res[variant]["loglik"] = out["loglik"].cpu().numpy()
            # the full-output forward computes the predicted moments in another order of operations (two-stage update and
            # predict instead of the reduced step): what it tapes agrees with the hot-path forward to rounding only
            for variant, tol in (("compressed", 1e-11), ("compressed_full_forward", 1e-9)):
                for k in res[variant]:
                    scale = max(np.abs(res["plain"][k]).max(), 1e-300)
                    assert np.abs(res[variant][k] - res["plain"][k]).max() / scale < tol, (variant, k, n)
            for k in res["compressed_no_cd"]:
                assert np.array_equal(res["compressed_no_cd"][k], res["compressed"][k]), (k, n)
