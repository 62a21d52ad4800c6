"""Batched simulation helpers on the GPU (SURVEY.md section 8(f) row f4; not on the logp/grad path).

Mirrors reference ``pymc_statespace/utils/simulation.py`` (numba): ``simulate_statespace`` (:29-62),
``unconditional_simulations`` (:65-79) and ``conditional_simulation`` (:17-26).  ``simulation_smoother`` goes beyond the
reference: joint draws of the whole state path from p(x_0..x_{n-1} | y, theta) (Durbin & Koopman 2002), where
``conditional_simulation`` draws every time step on its own from the smoothed marginal.  ``forecast`` gives the
forecast moments and joint draws of the paths after the end of the sample, ``conditional_forecast`` the same given
known future values of some series, and ``impulse_responses`` the responses of states and observations to one shock.
The reference draws its normals from NumPy's global RNG inside numba, so its trajectories are not reproducible from
outside; here the standard-normal draws come from ``torch.randn`` on the device (or are passed in, which makes the
result exactly checkable) and the CUDA kernels are deterministic transforms of them.
"""
from __future__ import annotations

from typing import Optional

import ctypes

import torch

from ._lib import KFB_FLAG_PARTIAL_ROWS, SHOCK_KIND, KfbDesc, KfbInputs, check, load
from .engine import BatchedKalman, _ptr, _stream_ptr


def _bs(t, base_ndim, size):
    return size if t.ndim == base_ndim + 1 else 0


def simulate_statespace(T, Z, R, H, Q, n_steps: int, x0=None, n_simulations: int = 1, z_state=None, z_obs=None,
                        generator: Optional[torch.Generator] = None):
    """T:[B,m,m]|[m,m] ... float64 CUDA tensors.  Returns (states[B*S,n,m], obs[B*S,n,p]) for S = n_simulations
    trajectories per draw (``unconditional_simulations`` ordering: draw-major)."""
    lib = load()
    dev = T.device
    m, p, r = T.shape[-1], Z.shape[-2], R.shape[-1]
    B = max([t.shape[0] for t, nd in ((T, 2), (Z, 2), (R, 2), (H, 2), (Q, 2)) if t.ndim == nd + 1] + [1])
    S = B * n_simulations
    T, Z, R, H, Q = (t.contiguous() for t in (T, Z, R, H, Q))
    if z_state is None:
        z_state = torch.randn((S, n_steps, r), dtype=torch.float64, device=dev, generator=generator)
    if z_obs is None:
        z_obs = torch.randn((S, n_steps, p), dtype=torch.float64, device=dev, generator=generator)
    z_state, z_obs = z_state.contiguous(), z_obs.contiguous()
    if tuple(z_state.shape) != (S, n_steps, r) or tuple(z_obs.shape) != (S, n_steps, p):
        raise ValueError("z_state / z_obs must have shapes [B*S, n, k_posdef] / [B*S, n, k_endog]")
    x0c = None if x0 is None else x0.reshape(-1, m).contiguous()
    states = torch.empty((S, n_steps, m), dtype=torch.float64, device=dev)
    obs = torch.empty((S, n_steps, p), dtype=torch.float64, device=dev)
    info = torch.zeros(S, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_simulate(B, n_simulations, n_steps, m, p, r, _ptr(T), _bs(T, 2, m * m), _ptr(Z), _bs(Z, 2, p * m),
                               _ptr(R), _bs(R, 2, m * r), _ptr(H), _bs(H, 2, p * p), _ptr(Q), _bs(Q, 2, r * r), _ptr(x0c),
                               0 if x0c is None or x0c.shape[0] == 1 else m, _ptr(z_state), _ptr(z_obs), _ptr(states),
                               _ptr(obs), _ptr(info), _stream_ptr(dev)), "kfb_simulate")
    if int(info.sum()) != 0:
        raise RuntimeError("simulate_statespace: Q or H is not positive definite for some draw")
    return states, obs


def conditional_simulation(mus, covs, n_simulations: int = 100, z=None, jitter=None,
                           generator: Optional[torch.Generator] = None):
    """mus[U,n,k], covs[U,n,k,k] (filtered / predicted / smoothed moments) -> simulations[U*S,n,k]:
    each time block is an independent draw mu_t + chol(cov_t + jitter I) z (reference :8-26; the reference's jitter is
    uniform(1e-12, 1e-8) per trajectory)."""
    lib = load()
    dev = mus.device
    U, n, k = mus.shape
    S = U * n_simulations
    if z is None:
        z = torch.randn((S, n, k), dtype=torch.float64, device=dev, generator=generator)
    if jitter is None:
        jitter = 1e-12 + (1e-8 - 1e-12) * torch.rand(S, dtype=torch.float64, device=dev, generator=generator)
    mus, covs, z, jitter = mus.contiguous(), covs.contiguous(), z.contiguous(), jitter.contiguous()
    out = torch.empty((S, n, k), dtype=torch.float64, device=dev)
    info = torch.zeros(S, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_mvn_draws(U, n_simulations, n, k, _ptr(mus), _ptr(covs), _ptr(z), _ptr(jitter), _ptr(out), _ptr(info),
                                _stream_ptr(dev)), "kfb_mvn_draws")
    if int(info.sum()) != 0:
        raise RuntimeError("conditional_simulation: a covariance block is not positive definite")
    return out


_BASE_NDIM = {"a0": 1, "P0": 2, "T": 2, "Z": 2, "R": 2, "H": 2, "Q": 2, "c": 1, "d": 1}


def _canon_matrices(T, Z, R, H, Q, a0, P0, c, d, y):
    mats = {"a0": a0, "P0": P0, "T": T, "Z": Z, "R": R, "H": H, "Q": Q, "c": c, "d": d}
    for k, t in mats.items():
        if t is not None and k in ("a0", "c", "d") and t.ndim >= 2 and t.shape[-1] == 1:
            mats[k] = t = t[..., 0]
        if t is not None and t.ndim > _BASE_NDIM[k] + 1:
            raise NotImplementedError("time-varying matrices are not supported")
    if y is not None and y.ndim == 3 and y.shape[-1] == 1 and y.shape[-2] == Z.shape[-2]:
        y = y[..., 0]  # reference layout [n, p, 1]
    B = max([t.shape[0] for k, t in mats.items() if t is not None and t.ndim == _BASE_NDIM[k] + 1] + [1])
    return mats, y, B


def _normals(S, steps, m, p, r, z_init, z_state, z_obs, generator, dev):
    """Time-major standard normals of S simulations over ``steps`` steps: z_init [S, m], z_state [steps-1, S, r],
    z_obs [steps, S, p], each drawn with ``torch.randn`` if None, else checked.  Returns them contiguous."""
    out = []
    for name, t, shape in (("z_init", z_init, (S, m)), ("z_state", z_state, (max(steps - 1, 0), S, r)),
                           ("z_obs", z_obs, (steps, S, p))):
        if t is None:
            t = torch.randn(shape, generator=generator, dtype=torch.float64, device=dev)
        elif not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64 and tuple(t.shape) == shape):
            raise ValueError(f"{name}: expected a float64 CUDA tensor of shape {shape} (time-major normals)")
        out.append(t.contiguous())
    return out


def _workspace(lib, call, desc, dev, *args):
    """The workspace of ``call`` for ``desc`` on ``dev`` (``call``_workspace_bytes with ``args``), at least 256 bytes."""
    nbytes = ctypes.c_size_t(0)
    check(getattr(lib, call + "_workspace_bytes")(ctypes.byref(desc), *args, ctypes.byref(nbytes)),
          call + "_workspace_bytes")
    return torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=dev)


def _raise_on_failure(what, infos, unit="unit", codes="codes in include/kfb200.h"):
    """RuntimeError naming the first failing unit of the first info tensor (None: skipped) that has one."""
    for info in infos:
        bad = torch.nonzero(info != 0) if info is not None else None
        if bad is not None and bad.numel():
            u = int(bad[0, 0])
            raise RuntimeError(f"{what}: {unit} {u} failed with info {int(info[u])} ({codes})")


def _has_partial_rows(y) -> bool:
    """True if some row of y [..., n, p] has NaN in some entries and not in all (a partly observed row)."""
    nan = torch.isnan(y).sum(-1)
    return bool(((nan > 0) & (nan < y.shape[-1])).any())


def _predicted(kalman: BatchedKalman, y, mats, outputs, partial_rows):
    """The predicted moments ``outputs`` of the exact filter over y: kfb_masked_filter if ``partial_rows`` (y has a
    partly observed row), else the corrected standard filter.  Returns its outputs dict, "info" included."""
    run = kalman.masked_filter if partial_rows else kalman.forward
    return run(y, *[mats.get(k) for k in ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")], outputs=outputs)


def _simulation_smoother(kalman: BatchedKalman, y, mats, n_simulations, z_init, z_state, z_obs, generator,
                         partial_rows=False):
    """kfb_forward (predicted covariances; kfb_masked_filter with ``partial_rows``) then kfb_simulation_smoother on
    ``kalman``'s geometry (with KFB_FLAG_PARTIAL_ROWS if ``partial_rows``).  Returns (states [U*S, n, m], info [U])
    without raising on a non-zero info."""
    lib = load()
    dev = kalman.device
    n, m, p, r, U = kalman.n, kalman.m, kalman.p, kalman.r, kalman.units
    S = U * n_simulations
    pc = _predicted(kalman, y, mats, ("predicted_covs",), partial_rows)["predicted_covs"]
    z_init, z_state, z_obs = _normals(S, n, m, p, r, z_init, z_state, z_obs, generator, dev)
    desc = kalman._desc
    if partial_rows:
        desc = KfbDesc.from_buffer_copy(desc)
        desc.flags |= KFB_FLAG_PARTIAL_ROWS
    ws = _workspace(lib, "kfb_simulation_smoother", desc, dev, n_simulations)
    states = torch.empty((S, n, m), dtype=torch.float64, device=dev)
    info = torch.empty(U, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_simulation_smoother(ctypes.byref(desc), ctypes.byref(kalman._inputs), _ptr(pc), n_simulations,
                                          _ptr(z_init), _ptr(z_state) if n > 1 else None, _ptr(z_obs), _ptr(states),
                                          _ptr(info), _ptr(ws), ws.numel(), _stream_ptr(dev)), "kfb_simulation_smoother")
    return states, info


def simulation_smoother(y, a0, P0, T, Z, R, H, Q, c=None, d=None, n_simulations: int = 1, z_init=None, z_state=None,
                        z_obs=None, generator: Optional[torch.Generator] = None):
    """Joint draws of the state paths x_0..x_{n-1} from p(x | y, theta) (Durbin & Koopman 2002, mean correction;
    include/kfb200.h states the model and the recursion).

    Float64 CUDA tensors; each matrix is shared (a0 [m], P0 [m, m], T [m, m], Z [p, m], R [m, r], H [p, p], Q [r, r],
    c [m], d [p]) or one per draw with a leading [B] axis, as in ``BatchedKalman``.  y is [n, p] or [n_series, n, p]
    (NaN = missing; a partly observed row is conditioned on its observed entries).  Units are draw-major (u = draw * n_series + series) and
    so are the simulations (s = u * n_simulations + k).  Normals may be given, time-major: z_init [S, m], z_state
    [n-1, S, r], z_obs [n, S, p] for S = U * n_simulations; otherwise they are drawn with ``torch.randn``.
    Returns states [S, n, m].  Raises RuntimeError if some unit fails (F_t not positive definite on the observed entries,
    P0 / Q / H not positive semi-definite) and NotImplementedError for time-varying matrices."""
    mats, y, B = _canon_matrices(T, Z, R, H, Q, a0, P0, c, d, y)
    n_series = 1 if y.ndim == 2 else y.shape[0]
    m, p, r = T.shape[-1], Z.shape[-2], R.shape[-1]
    kalman = BatchedKalman("standard", y.shape[-2], m, p, r, n_draws=B, n_series=n_series, strict_reference=False,
                           device=T.device)
    states, info = _simulation_smoother(kalman, y, mats, int(n_simulations), z_init, z_state, z_obs, generator,
                                        _has_partial_rows(y))
    _raise_on_failure("simulation_smoother", (info,))
    return states


def _forecast(kalman: BatchedKalman, y, mats, horizon, n_simulations, z_init, z_state, z_obs, generator,
              partial_rows=False):
    """Forecast moments (and paths if n_simulations > 0) on ``kalman``'s geometry: the standard corrected filter of
    length n + horizon (kfb_masked_filter with ``partial_rows``), run on y extended by ``horizon`` all-NaN rows.  Returns (result dict, forward info [U], paths
    info [U] or None) without raising on a non-zero info."""
    lib = load()
    dev = kalman.device
    H, m, p, r, U = int(horizon), kalman.m, kalman.p, kalman.r, kalman.units
    n = kalman.n - H
    f64 = dict(dtype=torch.float64, device=dev)
    yx = torch.cat([y, torch.full(y.shape[:-2] + (H, p), float("nan"), **f64)], dim=-2)
    out = _predicted(kalman, yx, mats, ("predicted_states", "predicted_covs"), partial_rows)
    a, P = out["predicted_states"][:, n:n + H], out["predicted_covs"][:, n:n + H]
    ns = kalman.n_series

    def per_unit(t, base_ndim):  # [..] shared or [B, ..] per draw -> broadcastable against [U, H, ..]
        t = t if t.ndim == base_ndim else t.repeat_interleave(ns, dim=0)[:, None]
        return t

    Zu, Hu = per_unit(mats["Z"], 2), per_unit(mats["H"], 2)
    ya = torch.matmul(Zu, a[..., None])[..., 0]
    if mats.get("d") is not None:
        ya = ya + per_unit(mats["d"], 1)
    res = {"state_mean": a, "state_cov": P, "obs_mean": ya,
           "obs_cov": torch.matmul(torch.matmul(Zu, P), Zu.transpose(-1, -2)) + Hu}
    if n_simulations <= 0:
        return res, out["info"], None
    S = U * n_simulations
    z_init, z_state, z_obs = _normals(S, H, m, p, r, z_init, z_state, z_obs, generator, dev)
    start_mean, start_cov = a[:, 0].contiguous(), P[:, 0].contiguous()
    desc = kalman._desc
    ws = _workspace(lib, "kfb_forecast_paths", desc, dev, n_simulations)
    states = torch.empty((H, S, m), **f64)
    obs = torch.empty((H, S, p), **f64)
    info = torch.empty(U, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_forecast_paths(ctypes.byref(desc), ctypes.byref(kalman._inputs), _ptr(start_mean), _ptr(start_cov),
                                     H, n_simulations, _ptr(z_init), _ptr(z_state) if H > 1 else None, _ptr(z_obs),
                                     _ptr(states), _ptr(obs), _ptr(info), _ptr(ws), ws.numel(), _stream_ptr(dev)),
              "kfb_forecast_paths")
    res["state_paths"], res["obs_paths"] = states.permute(1, 0, 2), obs.permute(1, 0, 2)
    return res, out["info"], info


def forecast(y, a0, P0, T, Z, R, H, Q, c=None, d=None, horizon: int = 1, n_simulations: int = 0, z_init=None,
             z_state=None, z_obs=None, generator: Optional[torch.Generator] = None):
    """Forecasts from the end of the sample: the distribution of x_n..x_{n+H-1} and y_n..y_{n+H-1} given y_0..y_{n-1}
    (H = ``horizon``; output index h is time n + h), and with ``n_simulations`` > 0 joint draws of those paths.

    Arguments and conventions as in ``simulation_smoother``: float64 CUDA tensors, each matrix shared or one per draw,
    y [n, p] or [n_series, n, p], draw-major units (u = draw * n_series + series) and simulations
    (s = u * n_simulations + k).  The moments are the predicted moments of the exact (corrected standard) filter run
    on y extended by H all-NaN rows; a partly observed row of y is conditioned on its observed entries
    (kfb_masked_filter).  Each path starts from x_n ~ N(a_n, P_n) and follows the model with its own state
    and observation noise (include/kfb200.h, kfb_forecast_paths), so the paths have the joint law of the future,
    cross-horizon covariances included.  Normals may be given, time-major: z_init [S, m], z_state [H-1, S, r],
    z_obs [H, S, p] for S = U * n_simulations; otherwise they are drawn with ``torch.randn``.

    Returns a dict: state_mean [U, H, m], state_cov [U, H, m, m], obs_mean [U, H, p], obs_cov [U, H, p, p], and with
    n_simulations > 0 state_paths [S, H, m] and obs_paths [S, H, p].  The paths are ``permute(1, 0, 2)`` views of the
    kernel's time-major [H, S, .] buffers (no copy): call ``.contiguous()`` for path-major storage.  Raises
    RuntimeError if some unit fails (F_t not positive definite on the observed entries, P_n / Q / H not positive
    semi-definite) and NotImplementedError for time-varying matrices."""
    mats, y, B = _canon_matrices(T, Z, R, H, Q, a0, P0, c, d, y)
    n_series = 1 if y.ndim == 2 else y.shape[0]
    m, p, r = T.shape[-1], Z.shape[-2], R.shape[-1]
    if int(horizon) < 1:
        raise ValueError("horizon must be >= 1")
    kalman = BatchedKalman("standard", y.shape[-2] + int(horizon), m, p, r, n_draws=B, n_series=n_series,
                           strict_reference=False, device=T.device)
    res, finfo, pinfo = _forecast(kalman, y, mats, int(horizon), int(n_simulations), z_init, z_state, z_obs, generator,
                                  _has_partial_rows(y))
    _raise_on_failure("forecast", (finfo, pinfo))
    return res


def _conditional_forecast(kalman: BatchedKalman, y, mats, conditions, n_simulations, z_init, z_state, z_obs,
                          generator, partial_rows=False):
    """Conditional forecast on ``kalman``'s geometry (the standard corrected filter over the n observations;
    kfb_masked_filter with ``partial_rows``): its predicted moments at index n start kfb_conditional_forecast.  conditions [H, p] shared or [U, H, p].  Returns
    (result dict, forward info [U], window / paths info [U]) without raising on a non-zero info."""
    lib = load()
    dev = kalman.device
    m, p, r, U, n = kalman.m, kalman.p, kalman.r, kalman.units, kalman.n
    f64 = dict(dtype=torch.float64, device=dev)
    if not (isinstance(conditions, torch.Tensor) and conditions.is_cuda and conditions.dtype == torch.float64
            and conditions.ndim in (2, 3) and conditions.shape[-1] == p and conditions.shape[-2] >= 1
            and (conditions.ndim == 2 or conditions.shape[0] == U)):
        raise ValueError(f"conditions: expected a float64 CUDA tensor of shape [H, {p}] or [{U}, H, {p}]")
    H = conditions.shape[-2]
    cond = conditions.contiguous()
    out = _predicted(kalman, y, mats, ("predicted_states", "predicted_covs"), partial_rows)
    start_mean, start_cov = out["predicted_states"][:, n].contiguous(), out["predicted_covs"][:, n].contiguous()
    S = U * n_simulations
    if S > 0:
        z_init, z_state, z_obs = _normals(S, H, m, p, r, z_init, z_state, z_obs, generator, dev)
    desc = kalman._desc
    ws = _workspace(lib, "kfb_conditional_forecast", desc, dev, H, n_simulations)
    res = {"state_mean": torch.empty((U, H, m), **f64), "state_cov": torch.empty((U, H, m, m), **f64),
           "obs_mean": torch.empty((U, H, p), **f64), "obs_cov": torch.empty((U, H, p, p), **f64)}
    states = torch.empty((H, S, m), **f64) if S > 0 else None
    obs = torch.empty((H, S, p), **f64) if S > 0 else None
    info = torch.empty(U, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_conditional_forecast(
            ctypes.byref(desc), ctypes.byref(kalman._inputs), _ptr(start_mean), _ptr(start_cov), H, _ptr(cond),
            H * p if cond.ndim == 3 else 0, n_simulations, _ptr(z_init) if S > 0 else None,
            _ptr(z_state) if S > 0 and H > 1 else None, _ptr(z_obs) if S > 0 else None,
            *[_ptr(res[k]) for k in ("state_mean", "state_cov", "obs_mean", "obs_cov")], _ptr(states), _ptr(obs),
            _ptr(info), _ptr(ws), ws.numel(), _stream_ptr(dev)), "kfb_conditional_forecast")
    if S > 0:
        res["state_paths"], res["obs_paths"] = states.permute(1, 0, 2), obs.permute(1, 0, 2)
    return res, out["info"], info


def conditional_forecast(y, a0, P0, T, Z, R, H, Q, c=None, d=None, conditions=None, n_simulations: int = 0,
                         z_init=None, z_state=None, z_obs=None, generator: Optional[torch.Generator] = None):
    """Conditional forecasts from the end of the sample: the law of x_n..x_{n+H-1} and y_n..y_{n+H-1} given
    y_0..y_{n-1} and the known future values ``conditions[h, i]`` = y_{n+h, i} (NaN = free), and with ``n_simulations``
    > 0 joint draws of those paths (the simulation smoother over the window with partly observed rows; include/kfb200.h,
    kfb_conditional_forecast).  The horizon H is ``conditions.shape[-2]``; conditions is [H, p] shared by every unit or
    [U, H, p] per unit (float64 CUDA, U = n_draws * n_series).

    Arguments and conventions otherwise as in ``forecast``; the normals have the same shapes: z_init [S, m], z_state
    [H-1, S, r], z_obs [H, S, p] for S = U * n_simulations.  Returns ``forecast``'s dict (same keys, same views):
    state_mean [U, H, m], state_cov, obs_mean [U, H, p], obs_cov and with n_simulations > 0 state_paths [S, H, m],
    obs_paths [S, H, p].  Conditioned entries of obs_mean and obs_paths equal the condition exactly and have zero rows
    and columns in obs_cov.  With every entry NaN this is ``forecast`` (the paths bit for bit on the same normals).
    A partly observed row of y is conditioned on its observed entries (kfb_masked_filter), as a partly conditioned
    window row is.  Raises RuntimeError if some unit fails (F_t not positive definite on the observed entries in the
    sample or at a window step (n + h + 1), P_n / Q / H not positive semi-definite) and NotImplementedError for
    time-varying matrices."""
    mats, y, B = _canon_matrices(T, Z, R, H, Q, a0, P0, c, d, y)
    n_series = 1 if y.ndim == 2 else y.shape[0]
    m, p, r = T.shape[-1], Z.shape[-2], R.shape[-1]
    kalman = BatchedKalman("standard", y.shape[-2], m, p, r, n_draws=B, n_series=n_series, strict_reference=False,
                           device=T.device)
    res, finfo, winfo = _conditional_forecast(kalman, y, mats, conditions, int(n_simulations), z_init, z_state, z_obs,
                                              generator, _has_partial_rows(y))
    _raise_on_failure("conditional_forecast", (finfo, winfo))
    return res


def _impulse_responses(T, Z, R, Q, horizon, shock):
    """kfb_impulse_response for shared or per-draw T, Z, R, Q.  Returns (states [B, H, m, r], obs [B, H, p, r],
    info [B]) without raising on a non-zero info."""
    if shock not in SHOCK_KIND:
        raise ValueError(f"shock must be one of {sorted(SHOCK_KIND)}")
    if int(horizon) < 1:
        raise ValueError("horizon must be >= 1")
    lib = load()
    dev = T.device
    mats, _, B = _canon_matrices(T, Z, R, None, Q, None, None, None, None, None)
    m, p, r = T.shape[-1], Z.shape[-2], R.shape[-1]
    kal = BatchedKalman("standard", 1, m, p, r, n_draws=B, device=dev)
    held, strides = {}, {}
    for k in ("T", "Z", "R", "Q"):
        held[k], bs, _ = kal._canon(k, mats[k])
        strides[k] = (bs, 0)
    desc = kal._make_desc(strides)
    ins = KfbInputs(*[_ptr(held.get(k)) for k in ("y", "a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")])
    H = int(horizon)
    states = torch.empty((B, H, m, r), dtype=torch.float64, device=dev)
    obs = torch.empty((B, H, p, r), dtype=torch.float64, device=dev)
    info = torch.empty(B, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.kfb_impulse_response(ctypes.byref(desc), ctypes.byref(ins), H, SHOCK_KIND[shock], _ptr(states),
                                       _ptr(obs), _ptr(info), _stream_ptr(dev)), "kfb_impulse_response")
    return states, obs, info


def impulse_responses(T, Z, R, Q, horizon: int, shock: str = "cholesky"):
    """Responses to one shock at time 0, for every draw: column j of horizon h is T^h R S e_j (states) and
    Z T^h R S e_j (observations), with S = I (``shock="unit"``), diag(sqrt(diag Q)) (``"std"``: one standard
    deviation) or the lower factor of Q (``"cholesky"``: orthogonalised).  Float64 CUDA tensors, shared or with a
    leading draw axis B (B = 1 if all are shared).  Returns (states [B, H, m, r], obs [B, H, p, r]).  Raises
    RuntimeError if Q is not positive semi-definite for some draw under "std" / "cholesky"."""
    states, obs, info = _impulse_responses(T, Z, R, Q, horizon, shock)
    _raise_on_failure("impulse_responses", (info,), "draw", "Q not positive semi-definite")
    return states, obs
