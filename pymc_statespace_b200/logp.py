"""theta-level batched log-likelihood and gradient: what NUTS asks for at every leapfrog step.

Pipeline for a batch ``theta[B, n_theta]`` (all on the GPU, stream-ordered, no host round trip):

    scatter theta -> (a0,P0,T,Z,R,H,Q,c,d)[B]        kfb_scatter_forward   (models/*.py update())
    [P0 = Lyapunov(T, R Q R^T)]                       kfb_lyapunov_forward  (SARIMAX.py:100-107)
    Kalman forward (tape of predicted moments)        kfb_forward           (kalman_filter.py:152-159)
    adjoint recursion -> matrix cotangents            kfb_backward          (PyTensor Scan.L_op)
    [Lyapunov adjoint]                                kfb_lyapunov_backward
    scatter^T -> dlogp/dtheta[B, n_theta]             kfb_scatter_backward

This is the batched equivalent of PyMC's ``logp_dlogp_function`` for the ``pm.Potential("log_likelihood")``
term registered at reference ``pymc_statespace/core/statespace.py:174``.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional

import numpy as np
import torch

from ._lib import (KFB_ERR_UNSUPPORTED, KFB_INFO_NOT_STATIONARY, KFB_MAX_SCATTER_SEGMENTS, KfbScatterSeg, check, load)
from .engine import BatchedKalman, _ptr, _stream_ptr, lyapunov_backward, lyapunov_forward
from .models import FUSED_K_STATES, MATRICES, StateSpaceSpec, pad_spec


def _capture(dev, body, warmup):
    """Run `body` a few times on a side stream (lazy initialisation: function attributes, workspaces), then capture it."""
    with torch.cuda.device(dev):
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                body()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body()
    return graph


class HostStepGraph:
    """ONE CUDA graph for a whole host-to-host evaluation:

        pinned-host theta[B, n_theta] -> H2D -> scatter + Lyapunov/DARE + Kalman forward + adjoint + scatter^T
            -> packed [B, 1 + n_theta] = (logp, dlogp/dtheta) -> D2H into a pinned host buffer.

    A sampler that keeps theta on the host pays ~8 kernel launches + 2 copies per leapfrog step; replaying them as one
    graph removes the per-launch CPU cost that a per-step synchronisation otherwise exposes.  The draws are split into
    ``chunks`` pieces (chains are independent) so that PCIe copies overlap kernels:

    * ``sequential=False`` (batches that fill the GPU only as a whole, e.g. 65,536 draws): every chunk is a parallel
      branch of the graph with its own evaluator, workspace and stream.  Measured on B200, configs[1]: eager 1.66 ms,
      graph 1.56 ms, 4 branches 1.53 ms (round 1 kernels).
    * ``sequential=True`` (large batches, e.g. >= 1 M draws): the chunks are waves through ONE evaluator sized for a
      single wave (a quarter of the tape memory); wave k's H2D / D2H run on copy streams under the kernels of the
      neighbouring waves.

    ``theta_host`` / ``out_host`` are captured BY ADDRESS: write the next theta into ``theta_host`` in place, call the
    object, read ``out_host``.  No collective inside the graph: with one process per GPU every rank replays its own.
    """

    def __init__(self, model: "KalmanLogp", theta_host: torch.Tensor, out_host: torch.Tensor, warmup: int = 3,
                 chunks: int = 1, sequential: bool = False):
        B, nt = model.B * (chunks if sequential else 1), model.spec.n_theta
        for name, t, shape in (("theta_host", theta_host, (B, nt)), ("out_host", out_host, (B, 1 + nt))):
            if not (isinstance(t, torch.Tensor) and t.device.type == "cpu" and t.dtype == torch.float64
                    and t.is_contiguous() and t.is_pinned() and tuple(t.shape) == shape):
                raise TypeError(f"{name}: expected a pinned, contiguous float64 host tensor of shape {shape}")
        if chunks < 1 or B % chunks != 0:
            raise ValueError(f"chunks = {chunks} must divide the number of draws ({B})")
        self.model, self.theta_host, self.out_host, self.chunks = model, theta_host, out_host, chunks
        dev = model.device
        h = B // chunks
        self._theta_dev = [torch.empty((h, nt), dtype=torch.float64, device=dev) for _ in range(chunks)]
        if sequential:
            # ``model`` IS the one-wave evaluator (n_draws = B / chunks)
            self._subs = [model]
            copy_in, copy_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
            self._streams = [copy_in, copy_out]
            self._info = torch.zeros((B,), dtype=torch.int32, device=dev)
            self._packed = [torch.empty((h, 1 + nt), dtype=torch.float64, device=dev) for _ in range(chunks)]

            def body():
                cur = torch.cuda.current_stream(dev)
                copy_in.wait_stream(cur)
                copy_out.wait_stream(cur)
                ready = []
                with torch.cuda.stream(copy_in):
                    for c, th in enumerate(self._theta_dev):
                        th.copy_(theta_host[c * h:(c + 1) * h], non_blocking=True)
                        ready.append(copy_in.record_event())
                for c, th in enumerate(self._theta_dev):
                    cur.wait_event(ready[c])
                    logp, grad = model.logp_and_grad(th)
                    packed = self._packed[c]  # persistent: read by the copy stream while the next wave computes
                    torch.cat([logp[:, None], grad], dim=1, out=packed)
                    self._info[c * h:(c + 1) * h].copy_(model.info)
                    done = cur.record_event()
                    with torch.cuda.stream(copy_out):
                        copy_out.wait_event(done)
                        out_host[c * h:(c + 1) * h].copy_(packed, non_blocking=True)
                cur.wait_stream(copy_out)
                cur.wait_stream(copy_in)
        else:
            # one evaluator per branch (its own workspace and tape); a single branch reuses the caller's model
            self._subs = [model] if chunks == 1 else [model.clone_for(h) for _ in range(chunks)]
            self._streams = [torch.cuda.Stream(device=dev) for _ in range(chunks)]
            self._info = None

            def body():
                cur = torch.cuda.current_stream(dev)
                for c, (sub, th, st) in enumerate(zip(self._subs, self._theta_dev, self._streams)):
                    st.wait_stream(cur)
                    with torch.cuda.stream(st):
                        th.copy_(theta_host[c * h:(c + 1) * h], non_blocking=True)
                        logp, grad = sub.logp_and_grad(th)
                        out_host[c * h:(c + 1) * h].copy_(torch.cat([logp[:, None], grad], dim=1), non_blocking=True)
                for st in self._streams:
                    cur.wait_stream(st)

        self.graph = _capture(dev, body, warmup)

    @property
    def info(self) -> torch.Tensor:
        """Per-draw status of the last replay (device tensor; 0 = ok)."""
        return self._info if self._info is not None else torch.cat([sub.info for sub in self._subs])

    def __call__(self) -> torch.Tensor:
        self.graph.replay()
        torch.cuda.current_stream(self.model.device).synchronize()
        return self.out_host


def logp_and_grad_in_waves(spec: StateSpaceSpec, data, theta: torch.Tensor, filter_type: str = "standard",
                           strict_reference: bool = True, max_workspace_bytes: Optional[int] = None):
    """logp+grad for an arbitrarily large batch: draws are processed in waves whose tape fits the memory budget
    (default: 60 % of the currently free HBM), e.g. 16 M draws x T = 1000 at k_states = 2 needs a 640 GB tape in one
    piece but only 4 waves of 4 M draws on one 180 GB B200.  Returns (logp[B], grad[B, n_theta], info[B])."""
    dev = theta.device
    y = np.asarray(data, dtype=np.float64)
    n = y.shape[0]
    m = spec.k_states
    per_draw = (max(n - 1, 0) * (m + m * (m + 1) // 2) + 4 * m * m + 64) * 8  # tape + C, C-bar, per-draw matrices
    if max_workspace_bytes is None:
        free, _ = torch.cuda.mem_get_info(dev)
        max_workspace_bytes = int(0.6 * free)
    wave = int(max(1, min(theta.shape[0], max_workspace_bytes // per_draw)))
    B = theta.shape[0]
    logp = torch.empty(B, dtype=torch.float64, device=dev)
    grad = torch.empty((B, spec.n_theta), dtype=torch.float64, device=dev)
    info = torch.empty(B, dtype=torch.int32, device=dev)
    model = None
    for lo in range(0, B, wave):
        hi = min(B, lo + wave)
        if model is None or model.B != hi - lo:
            model = None  # release the previous wave's workspace first
            model = KalmanLogp(spec, y, n_draws=hi - lo, filter_type=filter_type, strict_reference=strict_reference,
                               device=dev)
        lp, g = model.logp_and_grad(theta[lo:hi].contiguous())
        logp[lo:hi], grad[lo:hi], info[lo:hi] = lp, g, model.info
    return logp, grad, info


class KalmanLogp:
    def __init__(self, spec: StateSpaceSpec, data, n_draws: int, filter_type: str = "standard",
                 strict_reference: bool = True, device="cuda", force_coop: bool = False, pad_to_fused: bool = True,
                 time_parallel: bool = False):
        # sizes between the fused instantiations (odd k_states in 9..31; e.g. seasonal models of period 12 or 24): embed
        # the model in the next instantiated (even) size - exact (models.pad_spec) and far cheaper than the generic
        # run-time-dims kernels, because the tensor-core kernels work on zero-padded 16 x 16 / 32 x 32 tiles anyway
        self.k_states_model = spec.k_states
        if (pad_to_fused and spec.k_endog == 1 and 8 < spec.k_states < 32 and spec.k_states not in FUSED_K_STATES
                and filter_type in ("standard", "single", "cholesky", "steady_state")):
            spec = pad_spec(spec, min(k for k in FUSED_K_STATES if k >= spec.k_states))
        self.spec = spec
        self.device = torch.device(device)
        self.lib = load()
        self.filter_type, self.strict_reference, self._force_coop = filter_type, strict_reference, force_coop
        self.time_parallel = bool(time_parallel)  # BatchedKalman(time_parallel=...): scans over time for few draws
        y = data.detach().to(dtype=torch.float64) if isinstance(data, torch.Tensor) else np.asarray(data, dtype=np.float64)
        if y.ndim == 1:
            y = y[:, None]
        if y.ndim == 3 and y.shape[-1] == 1:
            y = y[..., 0]  # reference data layout [n, p, 1] (core/representation.py:13-24)
        self.n, p = y.shape
        if p != spec.k_endog:
            raise ValueError("data has %d columns, model expects %d" % (p, spec.k_endog))
        if filter_type == "single" and p > 1:
            # reference core/statespace.py:71-72
            raise ValueError('Cannot use filter_type = "single" with multiple observed time series')
        self.B = int(n_draws)
        self.y = torch.as_tensor(y, dtype=torch.float64, device=self.device).contiguous()
        # structure the model guarantees for every draw: constant (unmapped) design row [1, 0, ..] / zero observation variance
        z_unit0 = (p == 1 and not spec.maps.get("Z") and np.array_equal(
            np.asarray(spec.base["Z"], dtype=np.float64).ravel(), np.eye(spec.k_states)[0]))
        h_zero = p == 1 and not spec.maps.get("H") and not np.any(np.asarray(spec.base["H"]))
        # T in companion form with parameters in its first column only (BayesianARMA / SARIMAX, models/SARIMAX.py:59-98)
        mT = spec.k_states
        Tb = np.asarray(spec.base["T"], dtype=np.float64).reshape(mT, mT)
        t_companion = (z_unit0 and h_zero and mT >= 2 and np.array_equal(Tb[:, 1:], np.eye(mT)[:, :mT - 1])
                       and all(fi % mT == 0 for _, fi in spec.maps.get("T", [])))
        self.kalman = BatchedKalman(filter_type, self.n, spec.k_states, spec.k_endog, spec.k_posdef, n_draws=self.B,
                                    strict_reference=strict_reference, device=device, force_coop=force_coop,
                                    z_unit0=z_unit0, h_zero=h_zero, pad_odd=pad_to_fused, t_companion=t_companion,
                                    no_missing=not bool(torch.isnan(self.y).any()), time_parallel=time_parallel)
        m, pp, r = spec.k_states, spec.k_endog, spec.k_posdef
        self._shape = {"a0": (m,), "P0": (m, m), "T": (m, m), "Z": (pp, m), "R": (m, r), "H": (pp, pp), "Q": (r, r),
                       "c": (m,), "d": (pp,)}
        f64 = dict(dtype=torch.float64, device=self.device)
        self._base = {k: torch.as_tensor(np.asarray(spec.base[k], dtype=np.float64).reshape(self._shape[k]), **f64)
                      for k in MATRICES}
        self._maps = {}
        self._buf: Dict[str, torch.Tensor] = {}
        for k in MATRICES:
            mp = spec.maps.get(k, [])
            if mp:
                src = torch.as_tensor([a for a, _ in mp], dtype=torch.int32, device=self.device)
                dst = torch.as_tensor([b for _, b in mp], dtype=torch.int32, device=self.device)
                self._maps[k] = (src, dst, len(mp))
                self._buf[k] = torch.empty((self.B,) + self._shape[k], **f64)
        if spec.stationary_initialization:
            self._buf["P0"] = torch.empty((self.B, m, m), **f64)
        self._lyap_batched = None

    # ------------------------------------------------------------------
    def _size(self, k):
        s = 1
        for d in self._shape[k]:
            s *= d
        return s

    def _scatter(self, theta):
        sp = self.spec
        mats = {}
        with torch.cuda.device(self.device):
            mapped = [k for k in MATRICES if k in self._maps]
            for k in MATRICES:
                mats[k] = self._buf[k] if k in self._maps else self._base[k]
            # one launch for all theta-dependent matrices (chunks of KFB_MAX_SCATTER_SEGMENTS)
            for i0 in range(0, len(mapped), KFB_MAX_SCATTER_SEGMENTS):
                ks = mapped[i0:i0 + KFB_MAX_SCATTER_SEGMENTS]
                segs = (KfbScatterSeg * len(ks))(*[
                    KfbScatterSeg(self._size(k), self._maps[k][2], _ptr(self._base[k]), _ptr(self._maps[k][0]),
                                  _ptr(self._maps[k][1]), _ptr(self._buf[k])) for k in ks])
                check(self.lib.kfb_scatter_forward_multi(self.B, sp.n_theta, len(ks), segs, _ptr(theta),
                                                         _stream_ptr(self.device)), "kfb_scatter_forward_multi")
        if sp.stationary_initialization:
            A = mats["T"] if mats["T"].ndim == 3 else mats["T"].expand(self.B, -1, -1).contiguous()
            X, info = lyapunov_forward(A, mats["R"], mats["Q"])
            self._lyap = (A, X, info)
            mats["P0"] = X
        return mats

    def _check_theta(self, theta):
        if not (isinstance(theta, torch.Tensor) and theta.is_cuda and theta.dtype == torch.float64):
            raise TypeError("theta: expected a float64 CUDA tensor")
        if tuple(theta.shape) != (self.B, self.spec.n_theta):
            raise ValueError(f"theta: expected shape {(self.B, self.spec.n_theta)}, got {tuple(theta.shape)}")
        return theta.contiguous()

    def system_matrices(self, theta) -> Dict[str, torch.Tensor]:
        return dict(self._scatter(self._check_theta(theta)))

    def filter(self, theta, outputs=("filtered_states", "predicted_states", "filtered_covs", "predicted_covs", "loglik",
                                     "ll_obs")):
        """Forward pass with the reference's six outputs (batched over draws)."""
        mats = self._scatter(self._check_theta(theta))
        out = self.kalman.forward(self.y, *[mats[k] for k in MATRICES], outputs=outputs)
        m = self.k_states_model
        if m != self.spec.k_states:  # padded model: report the moments of the model's own states
            for k in ("filtered_states", "predicted_states"):
                if k in out:
                    out[k] = out[k][..., :m].contiguous()
            for k in ("filtered_covs", "predicted_covs"):
                if k in out:
                    out[k] = out[k][..., :m, :m].contiguous()
        return out

    def smooth(self, theta):
        """Filtered moments -> RTS smoother for every draw: the batched counterpart of ``build_statespace_graph`` +
        ``build_smoother_graph`` (reference core/statespace.py:146-200, filters/kalman_smoother.py:56-104).
        Returns (smoothed_states [B, n, m], smoothed_covs [B, n, m, m], filter outputs dict)."""
        from .engine import rts_smoother

        mats = self._scatter(self._check_theta(theta))
        out = self.kalman.forward(self.y, *[mats[k] for k in MATRICES], outputs=("filtered_states", "filtered_covs", "loglik"))
        ss, sc = rts_smoother(mats["T"], mats["R"], mats["Q"], out["filtered_states"], out["filtered_covs"])
        m = self.k_states_model
        if m != self.spec.k_states:  # padded model: the model's own states
            ss, sc = ss[..., :m].contiguous(), sc[..., :m, :m].contiguous()
            out["filtered_states"] = out["filtered_states"][..., :m].contiguous()
            out["filtered_covs"] = out["filtered_covs"][..., :m, :m].contiguous()
        return ss, sc, out

    def _exact_kalman(self, n):
        """The exact (corrected standard) filter over n steps for the per-draw calls: one cached for the sample's n
        and one for the last other n (n + horizon of ``forecast``)."""
        slot = "_ss_kalman" if n == self.n else "_fc_kalman"
        kal = getattr(self, slot, None)
        if kal is None or kal.n != n:
            sp = self.spec
            kal = BatchedKalman("standard", n, sp.k_states, sp.k_endog, sp.k_posdef, n_draws=self.B,
                                strict_reference=False, device=self.device)
            setattr(self, slot, kal)
        return kal

    def _not_stationary(self):
        """[B] bool: the draws of the last scatter whose stationary P0 does not exist (None without a stationary P0)."""
        if self.spec.stationary_initialization and getattr(self, "_lyap", None) is not None:
            return self._lyap[2] != 0
        return None

    def _stationary_info(self, info):
        """``info`` with KFB_INFO_NOT_STATIONARY for every draw whose stationary P0 does not exist (it replaces the
        follow-on code of that draw)."""
        bad = self._not_stationary()
        return info if bad is None else torch.where(bad, torch.full_like(info, KFB_INFO_NOT_STATIONARY), info)

    def _per_draw(self, theta, n, n_simulations, generator, z_init, run, kernel_nans=False):
        """A per-draw call of ``simulation`` after the theta scatter (and stationary P0):
        ``run(kalman, mats, z_init)`` on the exact filter over n steps returns (outputs dict, info tensors in order of
        precedence).  z_init is padded for a padded model (the extra states are identically zero, their normals
        unused).  Returns (outputs, info [B]): info is the stationarity code, else the first non-zero code of the
        tensors; every output of a failing draw is NaN and the padded states are sliced off (views).  ``kernel_nans``:
        the outputs are already NaN for every non-zero code of the tensors, so only the non-stationary draws are
        masked (a mask is a full pass over the outputs)."""
        mats = self._scatter(self._check_theta(theta))
        m, m0, S = self.spec.k_states, self.k_states_model, self.B * int(n_simulations)
        kal = self._exact_kalman(n)
        if S > 0 and m != m0:
            if z_init is None:
                z_init = torch.randn((S, m0), dtype=torch.float64, device=self.device, generator=generator)
            z_init = torch.nn.functional.pad(z_init, (0, m - m0))
        res, infos = run(kal, mats, z_init)
        info = self._stationary_info(infos[0])
        for later in infos[1:]:
            if later is not None:
                info = torch.where(info == 0, later, info)
        bad = self._not_stationary() if kernel_nans else info != 0
        if bad is not None:
            for k, v in res.items():
                if k.endswith("_paths"):  # [S, ., .] draw-major (views of the time-major buffers for the forecasts)
                    v.unflatten(0, (self.B, -1))[bad] = float("nan")
                else:
                    v[bad] = float("nan")
        if m != m0:
            for k in ("state_mean", "state_paths"):
                if k in res:
                    res[k] = res[k][..., :m0]
            if "state_cov" in res:
                res["state_cov"] = res["state_cov"][..., :m0, :m0]
        return res, info

    def sample_states(self, theta, n_simulations: int = 1, generator: Optional[torch.Generator] = None,
                      z_init=None, z_state=None, z_obs=None) -> torch.Tensor:
        """Joint draws of the latent state paths from p(x_0..x_{n-1} | y, theta) for every draw: the simulation smoother
        of ``simulation.simulation_smoother`` (Durbin & Koopman 2002) after the theta scatter (and stationary P0), as
        ``smooth()`` does.  Returns states [B * n_simulations, n, k_states] (draw-major); the paths of a failing draw are
        NaN and ``sample_states_info`` holds the per-draw status.

        Always the exact Kalman recursion (the corrected standard filter), whatever ``filter_type`` this evaluator was
        built with: the posterior of the states does not depend on the reference's as-coded likelihood quirks.  Normals
        may be given as in ``simulation_smoother``, sized for the model's own k_states."""
        from .simulation import _simulation_smoother

        def run(kal, mats, z_init):
            states, info = _simulation_smoother(kal, self.y, mats, int(n_simulations), z_init, z_state, z_obs,
                                                generator)
            return {"state_paths": states}, (info,)

        # the kernel writes NaN paths for its own failures
        res, self._ss_info = self._per_draw(theta, self.n, n_simulations, generator, z_init, run, kernel_nans=True)
        return res["state_paths"].contiguous()

    def forecast(self, theta, horizon: int, n_simulations: int = 0, generator: Optional[torch.Generator] = None,
                 z_init=None, z_state=None, z_obs=None) -> Dict[str, torch.Tensor]:
        """Forecasts from the end of the sample for every draw: ``simulation.forecast`` after the theta scatter (and
        stationary P0), as ``sample_states`` does.  Returns its dict (state_mean [B, H, k_states], state_cov, obs_mean,
        obs_cov and, with n_simulations > 0, state_paths [B * n_simulations, H, k_states] and obs_paths, draw-major)
        plus "info" [B] (int32): KFB_INFO_NOT_STATIONARY for a draw whose stationary P0 does not exist (it replaces the
        forward's follow-on code, as in ``sample_states``), else the forward's code (t+1: F_t not positive definite;
        -(t+1): y_t partly missing), else the paths' code (KFB_INFO_NOT_PSD: P_n, Q or H not positive semi-definite).
        Every output of a failing draw is NaN.

        Always the exact Kalman recursion (the corrected standard filter), whatever ``filter_type`` this evaluator was
        built with.  Normals may be given as in ``simulation.forecast``, sized for the model's own k_states."""
        from .simulation import _forecast

        H = int(horizon)
        if H < 1:
            raise ValueError("horizon must be >= 1")

        def run(kal, mats, z_init):
            res, info, pinfo = _forecast(kal, self.y, mats, H, int(n_simulations), z_init, z_state, z_obs, generator)
            return res, (info, pinfo)

        res, res_info = self._per_draw(theta, self.n + H, n_simulations, generator, z_init, run)
        res["info"] = res_info
        return res

    def conditional_forecast(self, theta, conditions, n_simulations: int = 0,
                             generator: Optional[torch.Generator] = None, z_init=None, z_state=None,
                             z_obs=None) -> Dict[str, torch.Tensor]:
        """Conditional forecasts for every draw: ``simulation.conditional_forecast`` after the theta scatter (and
        stationary P0), as ``forecast`` does.  conditions [H, k_endog] shared by every draw or [B, H, k_endog] (NaN =
        free).  Returns ``forecast``'s dict plus "info" [B] (int32): KFB_INFO_NOT_STATIONARY for a draw whose stationary
        P0 does not exist, else the forward's code, else the window / paths code (n + h + 1: F_o not positive definite
        at window step h; KFB_INFO_NOT_PSD).  Every output of a failing draw is NaN.

        Always the exact Kalman recursion (the corrected standard filter), whatever ``filter_type`` this evaluator was
        built with.  Normals may be given as in ``simulation.conditional_forecast``, sized for the model's own
        k_states."""
        from .simulation import _conditional_forecast

        def run(kal, mats, z_init):
            res, info, winfo = _conditional_forecast(kal, self.y, mats, conditions, int(n_simulations), z_init,
                                                     z_state, z_obs, generator)
            return res, (info, winfo)

        res, res_info = self._per_draw(theta, self.n, n_simulations, generator, z_init, run)
        res["info"] = res_info
        return res

    def impulse_responses(self, theta, horizon: int, shock: str = "cholesky") -> Dict[str, torch.Tensor]:
        """``simulation.impulse_responses`` for every draw after the theta scatter: {"states" [B, H, k_states, k_posdef],
        "obs" [B, H, k_endog, k_posdef], "info" [B]} (info KFB_INFO_NOT_PSD and NaN responses where Q is not positive
        semi-definite under shock "std" / "cholesky")."""
        from .simulation import _impulse_responses

        mats = self._scatter(self._check_theta(theta))
        states, obs, info = _impulse_responses(mats["T"], mats["Z"], mats["R"], mats["Q"], horizon, shock)
        if states.shape[0] != self.B:  # every matrix shared by the draws
            states, obs, info = (t.expand((self.B,) + t.shape[1:]).contiguous() for t in (states, obs, info))
        m0 = self.k_states_model
        if m0 != self.spec.k_states:
            states = states[:, :, :m0]
        return {"states": states, "obs": obs, "info": info}

    @property
    def sample_states_info(self) -> torch.Tensor:
        """Per-draw status of the last ``sample_states`` (int32, 0 = ok; t+1: F_t not positive definite; -(t+1): y_t
        partly missing; KFB_INFO_NOT_PSD: P0, Q or H not positive semi-definite; KFB_INFO_NOT_STATIONARY as in
        ``info``).  A failing draw's paths are NaN."""
        return self._ss_info

    def logp(self, theta) -> torch.Tensor:
        mats = self._scatter(self._check_theta(theta))
        out = self.kalman.forward(self.y, *[mats[k] for k in MATRICES], outputs=("loglik",))
        self._kf_info = out["info"]
        return out["loglik"]

    @property
    def info(self) -> torch.Tensor:
        """Per-draw status of the last evaluation (int32, 0 = ok; codes in include/kfb200.h).  A draw whose stationary
        P0 could not be computed (Lyapunov doubling did not converge: spectral radius of T >= 1 - the reference's
        bilinear solve returns a finite non-PSD matrix there and carries on, here logp is NaN) is reported as
        KFB_INFO_NOT_STATIONARY instead of the follow-on "F_0 not positive definite".  Merged lazily: nothing is added
        to the per-evaluation launch sequence."""
        return self._stationary_info(self._kf_info)

    def capture_host_step(self, theta_host: torch.Tensor, out_host: torch.Tensor, chunks: int = 1,
                          sequential: bool = False) -> "HostStepGraph":
        """Capture host theta -> (logp, grad) on the host as one replayable CUDA graph (see ``HostStepGraph``).
        ``sequential=True``: this evaluator handles ONE wave; theta_host / out_host hold ``chunks * n_draws`` rows."""
        return HostStepGraph(self, theta_host, out_host, chunks=chunks, sequential=sequential)

    def clone_for(self, n_draws: int) -> "KalmanLogp":
        """A second evaluator of the same model / data / filter for ``n_draws`` draws (own workspace and tape)."""
        return KalmanLogp(self.spec, self.y, n_draws=n_draws, filter_type=self.filter_type,
                          strict_reference=self.strict_reference, device=self.device, force_coop=self._force_coop,
                          time_parallel=self.time_parallel)

    def logp_and_grad(self, theta, g_loglik: Optional[torch.Tensor] = None):
        """Returns (logp[B], dlogp/dtheta[B, n_theta]); ``self.info[B]`` holds per-draw status."""
        theta = self._check_theta(theta)
        sp = self.spec
        mats = self._scatter(theta)
        out = self.kalman.forward(self.y, *[mats[k] for k in MATRICES], outputs=("loglik",), save_for_backward=True)
        self._kf_info = out["info"]
        wrt = [k for k in MATRICES if k in self._maps]
        if sp.stationary_initialization and "P0" not in wrt:
            wrt.append("P0")
        g = self.kalman.backward(g_loglik=g_loglik, wrt=wrt)
        if sp.stationary_initialization:
            # P0 = Lyapunov(T, R Q R^T): push P0-bar back into T-bar, R-bar, Q-bar (only those theta reaches)
            A, X, _ = self._lyap
            lyapunov_backward(A, mats["R"], mats["Q"], X, g["P0"], g.get("T"), g.get("R"), g.get("Q"))
        ks = [k for k in self._maps if not (sp.stationary_initialization and k == "P0")]
        with torch.cuda.device(self.device):
            status = KFB_ERR_UNSUPPORTED
            if 0 < len(ks) <= KFB_MAX_SCATTER_SEGMENTS:
                # one launch: gtheta[b, j] = sum over matrices of the cotangents of the elements theta_j was written to
                gtheta = torch.empty((self.B, sp.n_theta), dtype=torch.float64, device=self.device)
                segs = (KfbScatterSeg * len(ks))(*[
                    KfbScatterSeg(self._size(k), self._maps[k][2], None, _ptr(self._maps[k][0]), _ptr(self._maps[k][1]),
                                  _ptr(g[k])) for k in ks])
                status = self.lib.kfb_scatter_backward_multi(self.B, sp.n_theta, len(ks), segs, _ptr(gtheta),
                                                             _stream_ptr(self.device))
                if status != KFB_ERR_UNSUPPORTED:  # UNSUPPORTED: the mapped elements do not fit shared memory
                    check(status, "kfb_scatter_backward_multi")
            if status == KFB_ERR_UNSUPPORTED:
                gtheta = torch.zeros((self.B, sp.n_theta), dtype=torch.float64, device=self.device)
                for k in ks:
                    src, dst, nmap = self._maps[k]
                    check(self.lib.kfb_scatter_backward(self.B, sp.n_theta, self._size(k), nmap, _ptr(g[k]), _ptr(src),
                                                        _ptr(dst), _ptr(gtheta), _stream_ptr(self.device)),
                          "kfb_scatter_backward")
        return out["loglik"], gtheta
