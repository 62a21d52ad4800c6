"""The plugin seam at one model per call: what an UNMODIFIED PyMC / NUTS hits (numpy in, numpy out, B = 1).

``filters.*.build_graph`` with numpy inputs and the two ``perform`` bodies of ``pytensor_op`` land here.  At this size
the kernels take tens of microseconds and everything around them used to dominate (round 1: 9 separate host-to-device
uploads, a synchronising ``int(info)``, 9 device-to-host reads per gradient call: 224 us at T = 100).  A ``SeamGraph``
owns ONE pinned staging buffer each way and replays the whole evaluation - upload, forward kernel, adjoint kernel,
download - as one CUDA graph: one ``cudaGraphLaunch`` and one stream synchronisation per call.

Reference call sites: ``pymc_statespace/core/statespace.py:164-166`` (``build_graph``), PyTensor's ``Op.perform``.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from .engine import MATRIX_NAMES, BatchedKalman

_SIX = ("filtered_states", "predicted_states", "filtered_covs", "predicted_covs", "loglik", "ll_obs")


def _stage(device, names: Sequence[str], shapes):
    """One pinned host buffer and one device buffer holding the named arrays back to back, with numpy / torch views."""
    sizes = [int(np.prod(shapes[k])) for k in names]
    total = max(sum(sizes), 1)
    host = torch.empty(total, dtype=torch.float64).pin_memory()
    dev = torch.empty(total, dtype=torch.float64, device=device)
    host_np, dev_v, off = {}, {}, 0
    hn = host.numpy()
    for k, sz in zip(names, sizes):
        host_np[k] = hn[off:off + sz].reshape(shapes[k])
        dev_v[k] = dev[off:off + sz].view(shapes[k])
        off += sz
    return host, dev, host_np, dev_v


class SeamGraph:
    """One problem geometry, one replayable graph.  ``mode="six"``: the reference's six outputs;
    ``mode="grad"``: loglik + cotangents of every matrix passed, for ``g_loglik * loglik + g_ll_obs . ll_obs``."""

    def __init__(self, flt, shapes: Dict[str, Tuple[int, ...]], mode: str, with_llobs: bool = False, device=None):
        if mode not in ("six", "grad"):
            raise ValueError(mode)
        self.mode, self.with_llobs = mode, bool(with_llobs and mode == "grad")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise RuntimeError("pymc_statespace_b200 needs a CUDA device (no CPU fallback)")
        self.present = tuple(k for k in MATRIX_NAMES if k in shapes)
        meta = {k: torch.empty(shapes[k], device="meta") for k in ("data",) + self.present}
        n, m, p, r, tv = flt._validate(meta["data"], *[meta.get(k) for k in MATRIX_NAMES])
        self.n, self.m, self.p = n, m, p
        self.bk = BatchedKalman(flt.kind, n, m, p, r, n_draws=1, strict_reference=flt.strict_reference, time_varying=tv,
                                device=self.device, time_parallel=bool(getattr(flt, "time_parallel", False)))
        # ---- staging layout (float64 elements): inputs [data | matrices | g_loglik | g_ll_obs], outputs per mode
        self._in_names = ("data",) + self.present + (("g_loglik",) if mode == "grad" else ()) \
            + (("g_ll_obs",) if self.with_llobs else ())
        in_shapes = dict(shapes, g_loglik=(1,), g_ll_obs=(1, n))
        self._in_shapes = {k: tuple(in_shapes[k]) for k in self._in_names}
        if mode == "six":
            out_shapes = {"filtered_states": (1, n, m), "predicted_states": (1, n + 1, m), "filtered_covs": (1, n, m, m),
                          "predicted_covs": (1, n + 1, m, m), "loglik": (1,), "ll_obs": (1, n)}
            self._out_names = _SIX
        else:
            out_shapes = {"loglik": (1,)}
            for k in self.present:
                out_shapes["g_" + k] = (1,) + ((n,) if k in tv else ()) + self.bk._base[k]
            self._out_names = ("loglik",) + tuple("g_" + k for k in self.present)
        self._out_shapes = out_shapes
        self.hin, self.din, self._hin_np, self._din_v = _stage(self.device, self._in_names, self._in_shapes)
        self.hout, self.dout, self._hout_np, self._dout_v = _stage(self.device, self._out_names, out_shapes)
        self.hinfo = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.dinfo = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._user_shapes = {k: tuple(shapes[k]) for k in self.present}
        # ---- warm up (workspace allocation, kernel attribute setup) on a side stream, then capture
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        self.hin.zero_()
        for k in ("P0", "H", "Q"):  # a well-posed dummy problem for the warm-up runs
            if k in self._hin_np:
                self._hin_np[k][...] = np.eye(self._in_shapes[k][-1])
        with torch.cuda.stream(side):
            self._enqueue()
            self._enqueue()
        side.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            self._enqueue()
        torch.cuda.current_stream(self.device).wait_stream(side)

    def _enqueue(self):
        v = self._din_v
        self.din.copy_(self.hin, non_blocking=True)
        mats = [v.get(k) for k in MATRIX_NAMES]
        if self.mode == "six":
            self.bk.forward(v["data"], *mats, outputs=_SIX, out=dict(self._dout_v, info=self.dinfo))
        else:
            self.bk.forward(v["data"], *mats, outputs=("loglik",), save_for_backward=True,
                            out={"loglik": self._dout_v["loglik"], "info": self.dinfo})
            self.bk.backward(g_loglik=v["g_loglik"], g_ll_obs=v.get("g_ll_obs"), wrt=self.present,
                             out={k: self._dout_v["g_" + k] for k in self.present})
        self.hout.copy_(self.dout, non_blocking=True)
        self.hinfo.copy_(self.dinfo, non_blocking=True)

    def __call__(self, arrays: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
        """``arrays``: name -> array for "data", every matrix of the geometry, and in grad mode "g_loglik"
        (+ "g_ll_obs").  Returns fresh numpy arrays (the staging buffers are reused by the next call)."""
        for k in self._in_names:
            np.copyto(self._hin_np[k], np.asarray(arrays[k], dtype=np.float64).reshape(self._in_shapes[k]))
        with torch.cuda.device(self.device):
            self.graph.replay()
            torch.cuda.current_stream(self.device).synchronize()
        info = int(self.hinfo[0])
        if info != 0:
            from .torch_op import _raise_info

            _raise_info(info)
        res = {}
        for k in self._out_names:
            a = np.array(self._hout_np[k][0])
            if self.mode == "grad" and k != "loglik":
                a = a.reshape(self._user_shapes[k[2:]])
            res[k] = a
        return res


_CACHE: Dict[tuple, SeamGraph] = {}


def seam_graph(flt, arrays: Dict[str, np.ndarray], mode: str, with_llobs: bool = False, device=None) -> SeamGraph:
    """The cached graph of this geometry (PyMC calls the Op once per leapfrog step with the same shapes)."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    shapes = {k: tuple(np.shape(a)) for k, a in arrays.items() if k == "data" or k in MATRIX_NAMES}
    key = (flt.kind, bool(flt.strict_reference), bool(getattr(flt, "time_parallel", False)), mode, bool(with_llobs),
           str(dev), tuple(sorted(shapes.items())))
    g = _CACHE.get(key)
    if g is None:
        if len(_CACHE) > 32:
            _CACHE.clear()
        g = _CACHE[key] = SeamGraph(flt, shapes, mode, with_llobs, dev)
    return g


def filter_numpy(flt, data, a0, P0, T, Z, R, H, Q, c=None, d=None, device=None):
    """numpy in -> the reference's 6-list as numpy (kalman_filter.py:184-191 shapes)."""
    arrays = {"data": data, "a0": a0, "P0": P0, "T": T, "Z": Z, "R": R, "H": H, "Q": Q}
    if c is not None:
        arrays["c"] = c
    if d is not None:
        arrays["d"] = d
    o = seam_graph(flt, arrays, "six", device=device)(arrays)
    return [o["filtered_states"][..., None], o["predicted_states"][..., None], o["filtered_covs"], o["predicted_covs"],
            o["loglik"].reshape(())[()], o["ll_obs"]]


def logp_grads_numpy(flt, arrays: Dict[str, np.ndarray], g_loglik=1.0, g_ll_obs: Optional[np.ndarray] = None, device=None):
    """numpy in -> (loglik, {name: cotangent}) through one loglik-only forward + the adjoint kernel."""
    use_llobs = g_ll_obs is not None and bool(np.any(np.asarray(g_ll_obs) != 0.0))
    call = dict(arrays, g_loglik=np.asarray(g_loglik, dtype=np.float64).reshape(1))
    if use_llobs:
        call["g_ll_obs"] = g_ll_obs
    g = seam_graph(flt, arrays, "grad", with_llobs=use_llobs, device=device)
    o = g(call)
    return float(o["loglik"]), {k: o["g_" + k] for k in g.present}


class SmoothSeamGraph:
    """The RTS smoother of one geometry at one unit per call (what PyMC's per-draw evaluation of the smoothed
    ``pm.Deterministic``s sends): one pinned upload of [T | R | Q | filtered_states | filtered_covs], the R Q R^T hoist and
    the smoother kernel, one pinned download, replayed as one CUDA graph."""

    def __init__(self, shapes: Dict[str, Tuple[int, ...]], time_parallel: bool = False, device=None):
        from .engine import rts_smoother, smoother_workspace_numel

        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise RuntimeError("pymc_statespace_b200 needs a CUDA device (no CPU fallback)")
        self.time_parallel = bool(time_parallel)
        n, m = shapes["fc"][0], shapes["fc"][-1]
        self.n, self.m = n, m
        self._in_names = ("T", "R", "Q", "fs", "fc")
        self._in_shapes = {"T": tuple(shapes["T"]), "R": tuple(shapes["R"]), "Q": tuple(shapes["Q"]), "fs": (1, n, m),
                           "fc": (1, n, m, m)}
        self._out_names = ("ss", "sc")
        self._out_shapes = {"ss": (1, n, m), "sc": (1, n, m, m)}
        self.hin, self.din, self._hin_np, self._din_v = _stage(self.device, self._in_names, self._in_shapes)
        self.hout, self.dout, self._hout_np, self._dout_v = _stage(self.device, self._out_names, self._out_shapes)
        self._ws = torch.empty(smoother_workspace_numel(1, m), dtype=torch.float64, device=self.device)
        self._smooth = rts_smoother
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        self.hin.zero_()
        self._hin_np["Q"][...] = np.eye(self._in_shapes["Q"][-1])  # a well-posed dummy problem for the warm-up runs
        self._hin_np["fc"][...] = np.eye(m)
        with torch.cuda.stream(side):
            self._enqueue()
            self._enqueue()
        side.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            self._enqueue()
        torch.cuda.current_stream(self.device).wait_stream(side)

    def _enqueue(self):
        v = self._din_v
        self.din.copy_(self.hin, non_blocking=True)
        self._smooth(v["T"], v["R"], v["Q"], v["fs"], v["fc"], time_parallel=self.time_parallel,
                     out=(self._dout_v["ss"], self._dout_v["sc"]), workspace=self._ws)
        self.hout.copy_(self.dout, non_blocking=True)

    def __call__(self, arrays: Dict[str, np.ndarray]) -> Dict[str, np.ndarray]:
        """``arrays``: T, R, Q, fs [n,m(,1)], fc [n,m,m].  Returns fresh numpy arrays ss [n,m], sc [n,m,m]."""
        for k in self._in_names:
            np.copyto(self._hin_np[k], np.asarray(arrays[k], dtype=np.float64).reshape(self._in_shapes[k]))
        with torch.cuda.device(self.device):
            self.graph.replay()
            torch.cuda.current_stream(self.device).synchronize()
        return {k: np.array(self._hout_np[k][0]) for k in self._out_names}


_SMOOTH_CACHE: Dict[tuple, SmoothSeamGraph] = {}


def smooth_graph(arrays: Dict[str, np.ndarray], time_parallel: bool = False, device=None) -> SmoothSeamGraph:
    """The cached smoother graph of this geometry, keyed by (time_parallel, shapes, device)."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    shapes = {k: tuple(np.shape(arrays[k])) for k in ("T", "R", "Q", "fs", "fc")}
    key = (bool(time_parallel), tuple(sorted(shapes.items())), str(dev))
    g = _SMOOTH_CACHE.get(key)
    if g is None:
        if len(_SMOOTH_CACHE) > 32:
            _SMOOTH_CACHE.clear()
        g = _SMOOTH_CACHE[key] = SmoothSeamGraph(shapes, time_parallel, dev)
    return g


def smooth_numpy(T, R, Q, filtered_states, filtered_covariances, time_parallel: bool = False, device=None):
    """numpy in -> the reference's [smoothed_states[n,m,1], smoothed_covariances[n,m,m]] (kalman_smoother.py:56-104)."""
    arrays = {"T": T, "R": R, "Q": Q, "fs": filtered_states, "fc": filtered_covariances}
    o = smooth_graph(arrays, time_parallel, device)(arrays)
    return [o["ss"][..., None], o["sc"]]
