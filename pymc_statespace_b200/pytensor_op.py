"""PyTensor adapter: the reference's ``pytensor.scan`` recursion replaced by ONE custom Op with a hand-written
gradient (BASELINE.json north_star).

``KalmanFilterOp.perform`` runs the forward CUDA kernel; ``KalmanFilterOp.L_op`` returns the outputs of
``KalmanFilterGradOp`` whose ``perform`` runs the adjoint CUDA kernel - the same split the reference itself uses for
``SolveDiscreteARE`` (``pymc_statespace/utils/pytensor_scipy.py:11-60``: ``perform`` + symbolic ``grad``).

PyTensor / PyMC are NOT installed in the build image (SURVEY.md section D), so this module is import-guarded.  Its
protocol wiring (make_node / infer_shape / connection_pattern / L_op / both ``perform`` bodies) is executed by
tests/test_pytensor_shim.py against a minimal stand-in of the Op protocol (tests/fake_pytensor - NOT PyTensor); everything
below the Op boundary (``filters.BaseFilter._eager`` -> ``torch_op`` -> C ABI) is what the GPU tests exercise.
PyMC forks chain processes: CUDA is initialised lazily inside ``perform``.
"""
from __future__ import annotations

import numpy as np

try:  # pragma: no cover - PyTensor is absent in the build image
    import pytensor
    import pytensor.tensor as pt
    from pytensor.gradient import DisconnectedType
    from pytensor.graph.basic import Apply
    from pytensor.graph.op import Op

    HAVE_PYTENSOR = True
except Exception:  # noqa: BLE001
    HAVE_PYTENSOR = False
    Op = object

_IN_NAMES = ("data", "a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")


def _input_names(has_c, has_d):
    """Names of the Op's inputs in order: the eight mandatory ones, then c and / or d if given."""
    return _IN_NAMES[:8] + (("c",) if has_c else ()) + (("d",) if has_d else ())


def _require():
    if not HAVE_PYTENSOR:
        raise ImportError("pytensor is not installed: the symbolic (PyMC) path of pymc_statespace_b200 needs it; "
                          "the eager numpy/torch path of filters.*.build_graph does not")


class KalmanFilterOp(Op):
    """(data, a0, P0, T, Z, R, H, Q[, c][, d]) -> the 6 outputs of BaseFilter.build_graph (kalman_filter.py:184-191)."""

    __props__ = ("kind", "strict_reference", "has_c", "has_d", "time_parallel")

    def __init__(self, kind, strict_reference=True, has_c=False, has_d=False, time_parallel=False):
        self.kind, self.strict_reference, self.has_c, self.has_d = kind, bool(strict_reference), bool(has_c), bool(has_d)
        self.time_parallel = bool(time_parallel)

    def _filter(self):
        from .filters import FILTER_FACTORY

        f = FILTER_FACTORY[self.kind]()
        f.strict_reference = self.strict_reference
        f.time_parallel = self.time_parallel
        return f

    def _split(self, inputs):
        inputs = list(inputs)
        base, rest = inputs[:8], inputs[8:]
        c = rest.pop(0) if self.has_c else None
        d = rest.pop(0) if self.has_d else None
        return base, c, d

    def make_node(self, *inputs):
        _require()
        inputs = [pt.as_tensor_variable(x) for x in inputs]
        from pytensor.tensor.type import TensorType

        outs = [TensorType("float64", shape=(None, None, None))() for _ in range(4)]
        outs += [TensorType("float64", shape=())(), TensorType("float64", shape=(None,))()]
        return Apply(self, inputs, outs)

    def infer_shape(self, fgraph, node, shapes):
        n, m = shapes[0][0], shapes[1][0]
        return [(n, m, 1), (n + 1, m, 1), (n, m, m), (n + 1, m, m), (), (n,)]

    def perform(self, node, inputs, output_storage):
        from .seam import filter_numpy

        base, c, d = self._split([np.asarray(x, dtype=np.float64) for x in inputs])
        outs = filter_numpy(self._filter(), *base, c, d)  # one replayed CUDA graph per call (seam.SeamGraph)
        for storage, o in zip(output_storage, outs):
            storage[0] = np.asarray(o, dtype=np.float64)

    def connection_pattern(self, node):
        # data (input 0) is not differentiable; every other input reaches log_likelihood and ll_obs only
        n_in = len(node.inputs)
        return [[False] * 6] + [[False, False, False, False, True, True] for _ in range(n_in - 1)]

    def L_op(self, inputs, outputs, output_grads):
        for g, name in zip(output_grads[:4], ("filtered_states", "predicted_states", "filtered_covariances",
                                              "predicted_covariances")):
            if not isinstance(g.type, DisconnectedType):
                raise NotImplementedError(
                    f"gradient through {name} is not implemented: only log_likelihood / ll_obs are differentiable "
                    "(the reference differentiates pm.Potential('log_likelihood') only, core/statespace.py:174)")
        g_ll, g_llobs = output_grads[4], output_grads[5]
        if isinstance(g_ll.type, DisconnectedType):
            g_ll = pt.zeros((), dtype="float64")
        if isinstance(g_llobs.type, DisconnectedType):
            g_llobs = pt.zeros_like(outputs[5])
        grads = KalmanFilterGradOp(self.kind, self.strict_reference, self.has_c, self.has_d,
                                   self.time_parallel)(*inputs, g_ll, g_llobs)
        if not isinstance(grads, (list, tuple)):
            grads = [grads]
        data_grad = pytensor.gradient.DisconnectedType()()
        return [data_grad] + list(grads)


class KalmanFilterGradOp(Op):
    """(inputs..., g_loglik, g_ll_obs) -> cotangents of (a0, P0, T, Z, R, H, Q[, c][, d]) via kfb_backward."""

    __props__ = ("kind", "strict_reference", "has_c", "has_d", "time_parallel")

    def __init__(self, kind, strict_reference=True, has_c=False, has_d=False, time_parallel=False):
        self.kind, self.strict_reference, self.has_c, self.has_d = kind, bool(strict_reference), bool(has_c), bool(has_d)
        self.time_parallel = bool(time_parallel)

    def make_node(self, *inputs):
        _require()
        inputs = [pt.as_tensor_variable(x) for x in inputs]
        n_mats = 7 + int(self.has_c) + int(self.has_d)
        outs = [inputs[1 + i].type() for i in range(n_mats)]
        return Apply(self, inputs, outs)

    def infer_shape(self, fgraph, node, shapes):
        n_mats = 7 + int(self.has_c) + int(self.has_d)
        return [shapes[1 + i] for i in range(n_mats)]

    def perform(self, node, inputs, output_storage):
        from .filters import FILTER_FACTORY
        from .seam import logp_grads_numpy

        arrs = [np.asarray(x, dtype=np.float64) for x in inputs]
        g_ll, g_llobs = arrs[-2], arrs[-1]
        arrs = arrs[:-2]
        flt = FILTER_FACTORY[self.kind]()
        flt.strict_reference = self.strict_reference
        flt.time_parallel = self.time_parallel
        names = _input_names(self.has_c, self.has_d)
        # one loglik-only forward (hot-path kernels + tape) and the adjoint kernel, replayed as ONE CUDA graph with a single
        # pinned upload / download (seam.SeamGraph); no full-output pass, no autograd tape
        _, grads = logp_grads_numpy(flt, dict(zip(names, arrs)), g_loglik=g_ll, g_ll_obs=g_llobs)
        for storage, k in zip(output_storage, names[1:]):
            storage[0] = grads[k]


def build_symbolic_graph(flt, data, a0, P0, T, Z, R, H, Q, c=None, d=None):
    """What BaseFilter.build_graph returns for PyTensor inputs: 6 symbolic outputs of one KalmanFilterOp."""
    _require()
    inputs = [data, a0, P0, T, Z, R, H, Q]
    if c is not None:
        inputs.append(c)
    if d is not None:
        inputs.append(d)
    # names follow the inputs actually passed (c and d are optional and independent of each other)
    ndims = {n: pt.as_tensor_variable(x).ndim for n, x in zip(_input_names(c is not None, d is not None), inputs)}
    if flt.kind in ("steady_state", "univariate") and any(ndims.get(k) == 3 for k in ("T", "Z", "R", "H", "Q", "c", "d")):
        raise ValueError("All system matrices must be time-invariant to use this filter")
    op = KalmanFilterOp(flt.kind, flt.strict_reference, c is not None, d is not None,
                        bool(getattr(flt, "time_parallel", False)))
    return list(op(*inputs))


class KalmanSmootherOp(Op):
    """(T, R, Q, filtered_states[n,m,1], filtered_covariances[n,m,m]) -> [smoothed_states[n,m,1],
    smoothed_covariances[n,m,m]]: the RTS smoother of KalmanSmoother.build_graph (reference kalman_smoother.py:56-104),
    one replayed CUDA graph per call (seam.smooth_numpy).  Not differentiable."""

    __props__ = ("time_parallel",)

    def __init__(self, time_parallel=False):
        self.time_parallel = bool(time_parallel)

    def make_node(self, T, R, Q, filtered_states, filtered_covariances):
        _require()
        inputs = [pt.as_tensor_variable(x) for x in (T, R, Q, filtered_states, filtered_covariances)]
        from pytensor.tensor.type import TensorType

        outs = [TensorType("float64", shape=(None, None, None))() for _ in range(2)]
        return Apply(self, inputs, outs)

    def infer_shape(self, fgraph, node, shapes):
        n, m = shapes[4][0], shapes[4][1]  # filtered_covariances [n, m, m]; perform returns [n, m, 1] and [n, m, m]
        return [(n, m, 1), (n, m, m)]

    def perform(self, node, inputs, output_storage):
        from .seam import smooth_numpy  # CUDA is initialised here, in the process that evaluates the graph

        outs = smooth_numpy(*[np.asarray(x, dtype=np.float64) for x in inputs], time_parallel=self.time_parallel)
        for storage, o in zip(output_storage, outs):
            storage[0] = np.asarray(o, dtype=np.float64)

    def L_op(self, inputs, outputs, output_grads):
        for g, name in zip(output_grads, ("smoothed_states", "smoothed_covariances")):
            if not isinstance(g.type, DisconnectedType):
                raise NotImplementedError(
                    f"gradient through {name} is not implemented: the smoothed moments are Deterministics of the "
                    "reference model, evaluated per saved draw, and are not differentiable here")
        return [pytensor.gradient.DisconnectedType()() for _ in inputs]


def build_smoother_graph(smoother, T, R, Q, filtered_states, filtered_covariances):
    """What KalmanSmoother.build_graph returns for PyTensor inputs: the 2 symbolic outputs of one KalmanSmootherOp."""
    _require()
    if any(pt.as_tensor_variable(x).ndim == 3 for x in (T, R, Q)):
        raise NotImplementedError("time-varying T, R, Q are not supported by the B200 smoother")
    op = KalmanSmootherOp(bool(getattr(smoother, "time_parallel", False)))
    return list(op(T, R, Q, filtered_states, filtered_covariances))
