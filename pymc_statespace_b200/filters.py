"""The reference's filter plugin surface, backed by the B200 kernels.

Mirrors ``pymc_statespace/filters/kalman_filter.py`` of the reference: five filter classes with a no-argument
constructor (they are instantiated by ``FILTER_FACTORY[filter_type.lower()]()`` at
``pymc_statespace/core/statespace.py:74``) and

    build_graph(data, a0, P0, T, Z, R, H, Q, c=None, d=None, mode=None)
        -> [filtered_states[n,m,1], predicted_states[n+1,m,1], filtered_covariances[n,m,m],
            predicted_covariances[n+1,m,m], log_likelihood (scalar), ll_obs[n]]      (kalman_filter.py:126-193)

Argument shapes are the reference's (``data[n,p,1]``, ``a0[m,1]``, 2-D static or 3-D time-first matrices).
Three kinds of inputs are accepted:

* PyTensor variables (when PyTensor is importable): returns symbolic outputs of ``KalmanFilterOp`` whose ``L_op``
  is the hand-written adjoint kernel (``pytensor_op.py``) - the drop-in for the reference's scan graph;
* torch CUDA tensors: runs eagerly, returns torch tensors; differentiable wrt a0,P0,T,Z,R,H,Q,c,d through
  ``log_likelihood`` and ``ll_obs`` (``torch_op.py``);
* numpy arrays: runs eagerly on ``cuda:0`` and returns numpy arrays (what ``pytensor.function(inputs, outputs)``
  of the reference's tests returns, ``tests/test_kalman_filter.py:26-36``).

There is no CPU implementation: without a CUDA device / libkfb200.so every call raises.
"""
from __future__ import annotations

from typing import List

import numpy as np

PARAM_NAMES = ["c", "d", "T", "Z", "R", "H", "Q"]  # kalman_filter.py:17
_TV_MSG = ("The first dimension of a time varying matrix (the time dimension) must be "
           "equal to the first dimension of the data (the time dimension).")  # kalman_filter.py:20-23
_SINGLE_MSG = "UnivariateTimeSeries filter requires data be at most 1-dimensional"  # kalman_filter.py:19


def _is_pytensor_variable(x):
    mod = type(x).__module__ or ""
    return mod.startswith("pytensor")


def split_vars_into_seq_and_nonseq(params, param_names):
    """reference filters/utilities.py:1-20 (same return convention)."""
    sequences, non_sequences, seq_names, non_seq_names = [], [], [], []
    for param, name in zip(params, param_names):
        if param.ndim == 2:
            non_sequences.append(param)
            non_seq_names.append(name)
        elif param.ndim == 3:
            sequences.append(param)
            seq_names.append(name)
        else:
            raise ValueError(f"Matrix {name} has {param.ndim}, it should either 2 (static) or 3 (time varying).")
    return sequences, non_sequences, seq_names, non_seq_names


class BaseFilter:
    kind = None  # FILTER_FACTORY key

    def __init__(self, mode=None, strict_reference: bool = True, device=None):
        self.mode = mode
        self.seq_names: List[str] = []
        self.non_seq_names: List[str] = []
        self.eye_states = self.eye_posdef = self.eye_endog = None  # attrs of the reference object; unused here
        self.strict_reference = strict_reference
        # opt-in time-parallel kernels (k_endog = 1, k_states <= 4): faster for one draw per call over long series
        self.time_parallel = False
        self.device = device

    @staticmethod
    def update(a, P, y, c, d, Z, H, all_nan_flag):
        raise NotImplementedError  # kalman_filter.py:225-229

    # ------------------------------------------------------------------
    def build_graph(self, data, a0, P0, T, Z, R, H, Q, c=None, d=None, mode=None):
        self.mode = mode
        if self.kind is None:
            raise NotImplementedError
        args = [data, a0, P0, T, Z, R, H, Q, c, d]
        if any(_is_pytensor_variable(x) for x in args if x is not None):
            from .pytensor_op import build_symbolic_graph

            return build_symbolic_graph(self, data, a0, P0, T, Z, R, H, Q, c, d)
        return self._eager(data, a0, P0, T, Z, R, H, Q, c, d)

    # ------------------------------------------------------------------
    def _eager(self, data, a0, P0, T, Z, R, H, Q, c, d):
        import torch

        from .torch_op import kalman_filter_torch

        as_numpy = not any(isinstance(x, torch.Tensor) for x in (data, a0, P0, T, Z, R, H, Q, c, d) if x is not None)
        if as_numpy:
            if not torch.cuda.is_available():
                raise RuntimeError("pymc_statespace_b200 filters need a CUDA device (no CPU fallback)")
            from .seam import filter_numpy

            # numpy in, numpy out: one pinned upload, the kernels and one download replayed as a CUDA graph
            return filter_numpy(self, *[np.asarray(x, dtype=np.float64) for x in (data, a0, P0, T, Z, R, H, Q)],
                                None if c is None else np.asarray(c, dtype=np.float64),
                                None if d is None else np.asarray(d, dtype=np.float64), device=self.device)
        dev = torch.device(self.device) if self.device is not None else None
        if dev is None:
            for x in (data, a0, P0, T, Z, R, H, Q):
                if isinstance(x, torch.Tensor) and x.is_cuda:
                    dev = x.device
                    break
        if dev is None:
            if not torch.cuda.is_available():
                raise RuntimeError("pymc_statespace_b200 filters need a CUDA device (no CPU fallback)")
            dev = torch.device("cuda", torch.cuda.current_device())

        def prep(x):
            if x is None:
                return None
            if isinstance(x, torch.Tensor):
                return x.to(device=dev, dtype=torch.float64)
            return torch.as_tensor(np.ascontiguousarray(np.asarray(x, dtype=np.float64)), device=dev)

        data, a0, P0, T, Z, R, H, Q, c, d = (prep(x) for x in (data, a0, P0, T, Z, R, H, Q, c, d))
        outs = kalman_filter_torch(self, data, a0, P0, T, Z, R, H, Q, c, d)
        if as_numpy:
            outs = [o.detach().cpu().numpy() for o in outs]
            outs[4] = outs[4][()]
        return outs

    # ------------------------------------------------------------------
    def _validate(self, data, a0, P0, T, Z, R, H, Q, c, d):
        """Graph-time checks of the reference (check_params / check_time_varying_shapes / split...)."""
        if data.ndim != 3 or data.shape[-1] != 1:
            raise ValueError("data must have shape (n_obs, k_endog, 1) (reference core/representation.py:13-24)")
        n, p = int(data.shape[0]), int(data.shape[1])
        m = int(Z.shape[-1])
        r = int(R.shape[-1])
        present = {"T": T, "Z": Z, "R": R, "H": H, "Q": Q}
        if c is not None:
            present["c"] = c
        if d is not None:
            present["d"] = d
        names = [k for k in PARAM_NAMES if k in present]
        seqs, _, seq_names, non_seq_names = split_vars_into_seq_and_nonseq([present[k] for k in names], names)
        self.seq_names, self.non_seq_names = seq_names, non_seq_names
        for s in seqs:
            if int(s.shape[0]) != n:
                raise AssertionError(_TV_MSG)
        if self.kind == "single" and p != 1:
            raise AssertionError(_SINGLE_MSG)
        if self.kind in ("steady_state", "univariate") and seq_names:
            # reference: `assert ValueError(...)` is a no-op and the fixed-signature kalman_step then mis-handles
            # 3-D inputs (SURVEY A.2-Q8); here the intended error is raised.
            raise ValueError("All system matrices must be time-invariant to use the "
                             + ("SteadyStateFilter" if self.kind == "steady_state" else "UnivariateFilter"))
        return n, m, p, r, tuple(seq_names)


class StandardFilter(BaseFilter):
    """reference kalman_filter.py:255-284"""
    kind = "standard"


class CholeskyFilter(BaseFilter):
    """reference kalman_filter.py:287-318.  ``strict_reference=True`` reproduces the as-coded filter, which is exact
    only for k_endog == 1 (SURVEY.md A.2-Q4); ``strict_reference=False`` is the intended filter."""
    kind = "cholesky"


class SingleTimeseriesFilter(BaseFilter):
    """reference kalman_filter.py:321-351"""
    kind = "single"


class SteadyStateFilter(BaseFilter):
    """reference kalman_filter.py:354-441"""
    kind = "steady_state"


class UnivariateFilter(BaseFilter):
    """reference kalman_filter.py:444-505"""
    kind = "univariate"


class KalmanSmoother:
    """reference pymc_statespace/filters/kalman_smoother.py:11-104 (static T, R, Q).
    ``build_graph(T, R, Q, filtered_states[n,m,1], filtered_covariances[n,m,m])`` ->
    ``[smoothed_states[n,m,1], smoothed_covariances[n,m,m]]``.  Not on the logp/grad path (SURVEY section 8(f) f2).

    PyTensor inputs give the two symbolic outputs of ``KalmanSmootherOp`` (no gradient through them); numpy inputs run
    one replayed CUDA graph (``seam.smooth_numpy``); torch inputs run eagerly."""

    def __init__(self, mode=None):
        self.mode = mode
        self.seq_names: List[str] = []
        self.non_seq_names: List[str] = []
        # opt-in time-parallel kernel (k_states <= 4): faster for one draw per call over long series
        self.time_parallel = False

    def build_graph(self, T, R, Q, filtered_states, filtered_covariances, mode=None):
        self.mode = mode
        args = [T, R, Q, filtered_states, filtered_covariances]
        if any(_is_pytensor_variable(x) for x in args):
            from .pytensor_op import build_smoother_graph

            return build_smoother_graph(self, *args)
        import torch

        from .engine import rts_smoother

        _, _, self.seq_names, self.non_seq_names = split_vars_into_seq_and_nonseq([T, R, Q], ["T", "R", "Q"])
        if self.seq_names:
            raise NotImplementedError("time-varying T, R, Q are not supported by the B200 smoother")
        as_numpy = not any(isinstance(x, torch.Tensor) for x in args)
        if as_numpy:
            if not torch.cuda.is_available():
                raise RuntimeError("pymc_statespace_b200 needs a CUDA device (no CPU fallback)")
            from .seam import smooth_numpy

            return smooth_numpy(*[np.asarray(x, dtype=np.float64) for x in args], time_parallel=self.time_parallel)
        dev = next((x.device for x in args if isinstance(x, torch.Tensor) and x.is_cuda), None)
        if dev is None:
            if not torch.cuda.is_available():
                raise RuntimeError("pymc_statespace_b200 needs a CUDA device (no CPU fallback)")
            dev = torch.device("cuda", torch.cuda.current_device())
        prep = lambda x: (x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(  # noqa: E731
            np.asarray(x, dtype=np.float64)))).to(device=dev, dtype=torch.float64)
        T, R, Q, fs, fc = (prep(x) for x in args)
        ss, sc = rts_smoother(T, R, Q, fs[None, :, :, 0].contiguous(), fc[None].contiguous(),
                              time_parallel=self.time_parallel)
        return [ss[0][..., None], sc[0]]


# reference pymc_statespace/core/statespace.py:25-31
FILTER_FACTORY = {
    "standard": StandardFilter,
    "univariate": UnivariateFilter,
    "steady_state": SteadyStateFilter,
    "single": SingleTimeseriesFilter,
    "cholesky": CholeskyFilter,
}


def get_filter(filter_type: str, k_endog: int = 1):
    """The selection logic of PyMCStateSpace.__init__ (reference core/statespace.py:66-74), same errors."""
    if filter_type.lower() not in FILTER_FACTORY.keys():
        raise NotImplementedError("The following are valid filter types: " + ", ".join(list(FILTER_FACTORY.keys())))
    if filter_type == "single" and k_endog > 1:
        raise ValueError('Cannot use filter_type = "single" with multiple observed time series')
    return FILTER_FACTORY[filter_type.lower()]()
