"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/kfb200.h declares,
argument validation works without touching a device, the host-side model maps equal the oracle's restatement
of the reference models, the C oracle port matches the torch oracle, and the draw-sharding / gather logic
works across 2 gloo ranks."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.helpers import ROOT, random_system, rel_err


def _header_functions():
    src = open(os.path.join(ROOT, "include", "kfb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(kfb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from pymc_statespace_b200 import _lib

    assert os.path.exists(_lib.LIB_PATH), "build with `python __graft_entry__.py` first"
    lib = _lib.load()
    names = _header_functions()
    assert len(names) >= 12
    for name in names:
        assert hasattr(lib, name), name
        assert name in _lib.EXPORTS, f"{name} declared in kfb200.h but not bound in _lib.py"
    assert lib.kfb_version() == 100
    assert lib.kfb_status_string(2) == b"unsupported configuration"


def test_desc_struct_layout_matches_header():
    from pymc_statespace_b200._lib import KfbDesc

    # 2 x i32, 2 x i64, 4 x i32, 17 x i64
    assert ctypes.sizeof(KfbDesc) == 8 + 16 + 16 + 17 * 8
    assert KfbDesc.n_draws.offset == 8 and KfbDesc.n.offset == 24 and KfbDesc.y_bs.offset == 40


def test_argument_validation_without_device():
    from pymc_statespace_b200 import _lib

    lib = _lib.load()
    d = _lib.KfbDesc()
    n = ctypes.c_size_t(0)
    assert lib.kfb_workspace_bytes(ctypes.byref(d), 1, ctypes.byref(n)) == _lib.KFB_ERR_INVALID_ARG
    d.filter_kind, d.n_draws, d.n_series, d.n, d.m, d.p, d.r = 0, 1000, 1, 100, 2, 1, 1
    d.T_bs = 4
    assert lib.kfb_workspace_bytes(ctypes.byref(d), 1, ctypes.byref(n)) == _lib.KFB_OK
    tape = 1024 * 99 * 5 * 8  # units padded to whole warps (tape layout [t-1][warp][k][32])
    assert n.value >= tape and n.value < tape + 1000 * 4 * 8 * 2 + 4096
    d.filter_kind, d.p = _lib.KFB_SINGLE, 2  # "single" with k_endog > 1 (reference kalman_filter.py:19,329)
    assert lib.kfb_workspace_bytes(ctypes.byref(d), 0, ctypes.byref(n)) == _lib.KFB_ERR_INVALID_ARG
    d.filter_kind = 17
    assert lib.kfb_workspace_bytes(ctypes.byref(d), 0, ctypes.byref(n)) == _lib.KFB_ERR_INVALID_ARG
    d.filter_kind, d.p, d.T_ts = _lib.KFB_UNIVARIATE, 1, 4  # fixed-signature step: static matrices only
    assert lib.kfb_workspace_bytes(ctypes.byref(d), 0, ctypes.byref(n)) == _lib.KFB_ERR_UNSUPPORTED
    ins, outs = _lib.KfbInputs(), _lib.KfbOutputs()
    assert lib.kfb_forward(ctypes.byref(d), ctypes.byref(ins), ctypes.byref(outs), None, 0, 0, None) == _lib.KFB_ERR_INVALID_ARG


def test_engine_refuses_cpu_and_bad_kind():
    from pymc_statespace_b200 import BatchedKalman

    with pytest.raises(NotImplementedError, match="The following are valid filter types"):
        BatchedKalman("kalman", 10, 2, 1, 1, 1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        BatchedKalman("standard", 10, 2, 1, 1, 1, device="cpu")


def test_model_specs_match_oracle_restatement():
    from oracle import models as om
    from pymc_statespace_b200 import models as pm

    rng = np.random.default_rng(0)

    def cmp(spec, fn):
        th = rng.normal(size=spec.n_theta)
        mats, ref = spec.matrices(th), fn(torch.tensor(th))
        for k, v in zip(("a0", "P0", "T", "Z", "R", "H", "Q"), ref):
            np.testing.assert_allclose(mats[k], v.numpy(), err_msg=k)

    for order in [(1, 1), (2, 1), (3, 0), (0, 2), (2, 3)]:
        cmp(pm.arma_spec(order, False), lambda t, o=order: om.arma_matrices(t, o, False))
    for order in [(1, 0), (2, 0), (0, 1), (1, 1), (2, 2), (3, 1), (0, 2)]:
        for me in (True, False):
            cmp(pm.varmax_spec(3, order, False, me), lambda t, o=order, e=me: om.varmax_matrices(t, 3, o, False, e))
    cmp(pm.local_level_spec(), om.local_level_matrices)
    # parameter counts of reference tests/test_VARMAX.py / SURVEY section 8(a) row a10
    assert pm.arma_spec((1, 1)).n_theta == 5 and pm.arma_spec((2, 1)).n_theta == 6
    assert pm.varmax_spec(3, (2, 0)).n_theta == 36 and pm.local_level_spec().n_theta == 9
    assert pm.arma_spec((1, 1)).param_names == ("x0", "sigma_state", "rho", "theta")
    assert pm.trend_seasonal_spec(29).k_states == 30


def test_c_port_matches_torch_oracle():
    from oracle import kalman_c as kc
    from oracle import kalman_torch as kt

    rng = np.random.default_rng(0)
    for (m, p, r) in [(2, 1, 1), (4, 2, 2), (6, 3, 3)]:
        args = random_system(rng, m, p, r, 30, n_missing=3)
        y, a0, P0, T, Z, R, H, Q = args
        C = R @ Q @ R.T
        ll, g, bad = kc.logp_grad_batch(y[..., 0], a0[None, :, 0], P0[None], T[None], Z, H, C[None])
        ref, gt = kt.loglik_and_grads("standard", *args)
        assert bad == 0 and abs(ll[0] - ref) < 1e-12 * abs(ref)
        Cb = g["C"][0]
        assert rel_err(Cb @ R @ Q.T + Cb.T @ R @ Q, gt["R"]) < 1e-10
        for k in ("a0", "P0", "T", "Z", "H"):
            assert rel_err(g[k][0].reshape(gt[k].shape), gt[k]) < 1e-10, k


def test_pad_spec_is_exact_in_the_oracle():
    """models.pad_spec (sizes between the fused kernel instantiations): the padded model has the same log-likelihood, the
    same moments of the original states and identical theta-maps semantics - checked with the CPU oracle."""
    from oracle import kalman_numpy as kn
    from pymc_statespace_b200.models import arma_spec, pad_spec, trend_seasonal_spec

    rng = np.random.default_rng(0)
    for spec, theta, m2 in ((trend_seasonal_spec(12), np.array([0.1, 0.01, 0.05, 0.5]), 18),
                            (arma_spec((3, 2), stationary_initialization=False), None, 5)):
        if theta is None:
            theta = rng.normal(size=spec.n_theta) * 0.3
            L = rng.normal(size=(3, 3)) * 0.3 + np.eye(3)
            theta[spec.param_slices["P0"]] = (L @ L.T).ravel()
            theta[spec.param_slices["sigma_state"]] = 0.8
        big = pad_spec(spec, m2)
        assert big.k_states == m2 and big.n_theta == spec.n_theta
        a, b = spec.matrices(theta), big.matrices(theta)
        y = rng.normal(size=(30, 1, 1))
        o1 = kn.kalman_filter("standard", y, *[a[k] for k in ("a0", "P0", "T", "Z", "R", "H", "Q")])
        o2 = kn.kalman_filter("standard", y, *[b[k] for k in ("a0", "P0", "T", "Z", "R", "H", "Q")])
        m = spec.k_states
        assert abs(o1[4] - o2[4]) < 1e-13 * abs(o1[4])
        assert np.abs(o1[0] - o2[0][:, :m]).max() < 1e-13 and np.abs(o1[3] - o2[3][:, :m, :m]).max() < 1e-12
        assert np.abs(o2[0][:, m:]).max() == 0.0 and np.abs(o2[3][:, m:, :]).max() == 0.0   # extra states stay zero


def test_shard_bounds_cover_all_draws():
    from pymc_statespace_b200.dist import shard_bounds

    for n, w in [(10, 3), (65536, 8), (7, 8), (1 << 20, 4)]:
        b = [shard_bounds(n, r, w) for r in range(w)]
        assert b[0][0] == 0 and b[-1][1] == n
        assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
        assert max(hi - lo for lo, hi in b) - min(hi - lo for lo, hi in b) <= 1


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from pymc_statespace_b200.dist import shard_bounds, pack_logp_grad, gather_logp_grad
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
for n_total in (64, 37):
    full = torch.arange(n_total * 4, dtype=torch.float64).reshape(n_total, 4)
    lo, hi = shard_bounds(n_total, rank, world)
    packed = pack_logp_grad(full[lo:hi, 0], full[lo:hi, 1:])
    out = gather_logp_grad(packed, n_total)
    assert torch.equal(out, full), (rank, n_total)
dist.barrier()
if rank == 0:
    print("GLOO_OK")
dist.destroy_process_group()
"""


_GLOO_WAVES_WORKER = r"""
import os, sys, types, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from pymc_statespace_b200.dist import GatherStepGraph
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()

class Stub:  # stands in for KalmanLogp (CUDA only): logp = row sum, grad = 2 * theta
    def __init__(self, h, nt):
        self.B, self.spec, self.device = h, types.SimpleNamespace(n_theta=nt), torch.device("cpu")
    def logp_and_grad(self, th):
        self.info = torch.zeros(th.shape[0], dtype=torch.int32)
        return th.sum(1), 2.0 * th

h, nt, waves = 5, 3, 4
B = h * waves
full = torch.arange(world * B * nt, dtype=torch.float64).reshape(world * B, nt)   # draw d of the whole job
g = GatherStepGraph(Stub(h, nt), full[rank * B:(rank + 1) * B].contiguous(), waves=waves)
g()
rows = g.rows()
assert tuple(g.out.shape) == (waves, world, h, 1 + nt) and tuple(rows.shape) == (world * B, 1 + nt)
assert torch.equal(rows[:, 0], full.sum(1)) and torch.equal(rows[:, 1:], 2.0 * full), rank   # draw order, every rank
dist.barrier()
if rank == 0:
    print("GLOO_WAVES_OK")
dist.destroy_process_group()
"""


def test_gather_step_waves_world_size_2_gloo(tmp_path):
    """N > 1 path of bench.py's resident leg (dist.GatherStepGraph): wave / rank / row layout and draw order, on CPU."""
    script = tmp_path / "worker_waves.py"
    script.write_text(_GLOO_WAVES_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
         "--master-port", "29519", str(script), ROOT],
        capture_output=True, text=True, timeout=240, env=env)
    assert out.returncode == 0 and "GLOO_WAVES_OK" in out.stdout, out.stderr[-2000:]


def test_gather_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
         "--master-port", "29517", str(script), ROOT],
        capture_output=True, text=True, timeout=240, env=env)
    assert out.returncode == 0 and "GLOO_OK" in out.stdout, out.stderr[-2000:]


def test_filter_factory_surface_matches_reference():
    # reference core/statespace.py:25-31,66-74 and tests/test_statespace.py:66-76
    from pymc_statespace_b200 import filters as F

    assert list(F.FILTER_FACTORY) == ["standard", "univariate", "steady_state", "single", "cholesky"]
    with pytest.raises(NotImplementedError, match="The following are valid filter types: standard, univariate, "
                                                  "steady_state, single, cholesky"):
        F.get_filter("kalman")
    with pytest.raises(ValueError, match='Cannot use filter_type = "single" with multiple observed time series'):
        F.get_filter("single", k_endog=2)
    f = F.get_filter("STANDARD")
    assert isinstance(f, F.StandardFilter) and f.mode is None and f.seq_names == [] and f.non_seq_names == []
    with pytest.raises(NotImplementedError):
        F.BaseFilter().update(*[None] * 8)
    with pytest.raises(ValueError, match="it should either 2"):
        F.split_vars_into_seq_and_nonseq([np.zeros(3)], ["T"])
    seqs, non, sn, nn = F.split_vars_into_seq_and_nonseq([np.zeros((2, 2)), np.zeros((5, 2, 2))], ["T", "Q"])
    assert sn == ["Q"] and nn == ["T"]


def test_pytensor_adapter_is_import_guarded():
    from pymc_statespace_b200 import pytensor_op

    if not pytensor_op.HAVE_PYTENSOR:
        with pytest.raises(ImportError, match="pytensor is not installed"):
            pytensor_op.build_symbolic_graph(None, *[None] * 8)


def test_reference_arm_uses_every_core_under_torchrun_env_and_only_rank0_prints():
    """VERDICT r1: torchrun exports OMP_NUM_THREADS=1 and round 1's N >= 2 CPU arm ran on one core.  `bench.py --impl
    reference` must use every host core regardless, print ONE JSON line with the contract's keys on rank 0, and exit 0
    silently on the other ranks (no GPU involved: the arm times oracle/kalman_c.c here)."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
           "--cpu-sample-draws", "256", "--n", "200"]
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2")
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "kalman_logp_grad_filter_steps_per_s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["n_gpus"] == 2
    assert line["cpu_baseline"]["cores"] == (os.cpu_count() or 1) and line["cpu_baseline"]["kind"] in ("port", "reference")
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["c5"]["cores"] == line["cpu_baseline"]["cores"]
    out = subprocess.run(cmd, env=dict(env, RANK="1"), capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0 and not [ln for ln in out.stdout.splitlines() if ln.startswith("{")]


def test_bench_dump_rows_writes_all_or_a_fixed_sample(tmp_path):
    """bench.py --dump-outputs: small legs are written whole, large ones as the same seeded sample of draws every time."""
    import bench

    small = torch.arange(10 * 6, dtype=torch.float64).reshape(10, 6)
    bench.dump_rows(str(tmp_path / "s"), "", small)
    assert sorted(os.listdir(tmp_path / "s")) == ["grad.npy", "logp.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "s" / "logp.npy"), small[:, 0].numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "s" / "grad.npy"), small[:, 1:].numpy())

    n = bench.DUMP_MAX_ROWS + 1000
    big = torch.arange(n, dtype=torch.float64)[:, None] * torch.tensor([1.0, 2.0, 3.0])
    for d in ("a", "b"):
        bench.dump_rows(str(tmp_path / d), "c5_", big)
    idx = np.load(tmp_path / "a" / "c5_draw_index.npy")
    assert idx.dtype == np.float64 and idx.shape == (bench.DUMP_MAX_ROWS,) and (np.diff(idx) > 0).all()
    assert idx[0] >= 0 and idx[-1] < n
    for name in ("c5_draw_index", "c5_logp", "c5_grad"):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, b), name
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "c5_logp.npy"), idx)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "c5_grad.npy"), idx[:, None] * [2.0, 3.0])
