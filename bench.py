#!/usr/bin/env python
"""bench.py - Kalman logp+grad filter-steps/s (draws x T) on N B200s, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--draws B] [--n T] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE batched logp+grad evaluation (theta[B,n_theta] -> logp[B], dlogp/dtheta[B,n_theta]).

* headline (`value`, `e2e`, `roofline`): BASELINE.json configs[1] - BayesianARMA(1,1), stationary init, 65,536 draws per
  GPU, T=1,000, standard filter (weak scaling: every rank evaluates its own 65,536 draws).
* `c5` block in the same JSON line: BASELINE.json configs[4] - the multi-GPU config north_star names: ARMA(2,1),
  2^20 draws per GPU (2^21 per GPU at N=8 = 16 M draws) x T=1,000, draws sharded over the ranks.

`value` legs keep theta resident in HBM and, for N > 1, all-gather every draw's (logp, grad) row to every rank over NCCL
(captured with the kernels in one CUDA graph per rank; c5: in 4 waves, the gather of wave k under the kernels of wave
k+1).  `e2e` legs are host to host: every rank replays its own HostStepGraph (pinned theta -> H2D -> kernels -> D2H of
its shard into its pinned buffer, chunked so that copies overlap kernels, stream-synchronised every step) - a
host-resident sampler needs no device collective at all.  Rank 0 prints ONE JSON line.

Both blocks time --steps steps per leg (c5: --c5-steps if given).  The inputs are seeded, so runs with the same
arguments see identical inputs; `--dump-outputs DIR` makes rank 0 write what the resident leg returned in its last timed
step, every draw's logp and gradient in draw order, as float64 `DIR/logp.npy`, `DIR/grad.npy` (and `DIR/c5_*.npy`), so
that two builds can be compared output for output (see dump_rows for the sampling of large legs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "kalman_logp_grad_filter_steps_per_s"
UNIT = "filter-steps/s"
ALG_FLOPS_PER_STEP = 442.0      # logp+grad, m=2 p=1 (BASELINE.md section 3)
SURVEY_TAPE_BYTES_PER_STEP = 40.0  # SURVEY section 8(d): 8 * (m + m(m+1)/2) per kernel and step for a store-all tape at m = 2
TAPE_BYTES_PER_STEP = 16.0      # what the kernels move: 8 * (1 + (m-1)m/2) - with Z = e0, H = 0, a companion T and complete
                                # data (every BayesianARMA model) the recursion reduces to a_t and the leading block of P_t
                                # (the last row / column of P_t is a constant of the draw), and the adjoint needs a_t only
                                # through its first component (kf_p1.cuh, ZU == 4)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--draws", type=int, default=65536, help="draws per GPU")
    ap.add_argument("--n", type=int, default=1000, help="time steps T")
    ap.add_argument("--cpu-sample-draws", type=int, default=0, help="draws in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of the captured CUDA graphs")
    ap.add_argument("--c5-draws", type=int, default=0, help="c5 block: draws per GPU (0 = 2^20, 2^21 at 8 GPUs)")
    ap.add_argument("--c5-steps", type=int, default=0, help="c5 block: timed steps (0 = --steps)")
    ap.add_argument("--no-c5", action="store_true", help="skip the c5 block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the (logp, grad) arrays of the last timed step of each GPU leg to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.c5_steps < 0:
        ap.error("--steps must be >= 1 and --c5-steps >= 0")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl b200")
    return a


def workload_name(a):
    return f"BayesianARMA(1,1) stationary init, {a.draws} draws/GPU x T={a.n}, standard filter, logp+dlogp/dtheta"


DUMP_MAX_ROWS = 1 << 18   # per leg: 2 legs x 2^18 draws x (logp + <= 6 grads + index) x 8 B stays under 64 MB in all


def dump_rows(out_dir, prefix, rows):
    """Writes packed per-draw rows [N, 1 + n_theta] = (logp, dlogp/dtheta) as float64 ``<prefix>logp.npy`` [N] and
    ``<prefix>grad.npy`` [N, n_theta].  Above DUMP_MAX_ROWS draws only a fixed, seeded sample of draws is written (the
    same draws on every run with the same arguments), and ``<prefix>draw_index.npy`` lists them in ascending order."""
    rows = rows.detach().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    if rows.shape[0] > DUMP_MAX_ROWS:
        idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], DUMP_MAX_ROWS, replace=False))
        rows = rows[idx]
        np.save(os.path.join(out_dir, prefix + "draw_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, prefix + "logp.npy"), np.ascontiguousarray(rows[:, 0], dtype=np.float64))
    np.save(os.path.join(out_dir, prefix + "grad.npy"), np.ascontiguousarray(rows[:, 1:], dtype=np.float64))


# ---------------------------------------------------------------------------------------------- CPU side
def host_cores():
    """Cores this process may use.  torchrun exports OMP_NUM_THREADS=1, which would silently turn the "all host cores"
    arm into a single-core run (round 1: SCALE N>=2 ratios were void) - the count is passed to the C port explicitly."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_inputs(theta, y, order=(1, 1)):
    """Matrix-level inputs of the C oracle port for ARMA(p,1) draws, k_states = 2 (numpy; restates models/SARIMAX.py
    update()): theta = [x0(2), sigma_state, rho_1..rho_p, theta_1]."""
    B = theta.shape[0]
    p = order[0]
    T = np.zeros((B, 2, 2)); T[:, 0, 1] = 1.0
    T[:, 0, 0] = theta[:, 3]
    if p == 2:
        T[:, 1, 0] = theta[:, 4]
    R = np.zeros((B, 2, 1)); R[:, 0, 0] = 1.0; R[:, 1, 0] = theta[:, 3 + p]
    Q = theta[:, 2][:, None, None]
    C = R @ Q @ R.transpose(0, 2, 1)
    # stationary P0: vec(P) = (I - T (x) T)^-1 vec(C)   (same solution as scipy's bilinear method)
    K = np.eye(4)[None] - np.einsum("bij,bkl->bikjl", T, T).reshape(B, 4, 4)
    P0 = np.linalg.solve(K, C.reshape(B, 4, 1)).reshape(B, 2, 2)
    Z = np.array([[1.0, 0.0]]); H = np.zeros((1, 1))
    return y, theta[:, 0:2].copy(), P0, T, Z, H, C


def run_cpu(theta, y, steps, warmup, order=(1, 1)):
    """Times the plain-C oracle port (forward + adjoint, OpenMP over draws) on every core this process may use.
    Returns (steps/s, cores, ms/step)."""
    from oracle import kalman_c

    args = cpu_inputs(theta, y, order)
    cores = host_cores()
    for _ in range(warmup):
        kalman_c.logp_grad_batch(*args, want_grads=True, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        kalman_c.logp_grad_batch(*args, want_grads=True, nthreads=cores)
    dt = (time.perf_counter() - t0) / steps
    return theta.shape[0] * y.shape[0] / dt, cores, dt * 1e3


def run_real_reference(theta, y, steps, warmup):
    """BASELINE.md section 4.1 / SURVEY section 8(d): the REAL reference (PyTensor graph of BayesianARMA(1,1), default C
    mode), one draw per call as PyMC's logp_dlogp_function evaluates it.  Raises ImportError where PyTensor / PyMC /
    pymc_statespace are not importable (this image: no wheel, no network) - the caller then times the C port."""
    for extra in (os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if os.path.isdir(extra) and extra not in sys.path:
            sys.path.append(extra)
    import pymc as pm  # noqa: F401
    import pytensor
    import pytensor.tensor as pt
    from pymc_statespace import BayesianARMA

    with pm.Model():
        x0 = pm.Normal("x0", shape=(2,))
        sigma = pm.HalfNormal("sigma_state")
        rho = pm.Normal("rho", shape=(1,))
        th = pm.Normal("theta", shape=(1,))
        mod = BayesianARMA(y, order=(1, 1), stationary_initialization=True, filter_type="standard", verbose=False)
        mod.build_statespace_graph()
        model = pm.modelcontext(None)
        ll = model["log_likelihood"]
        vec = pt.dvector("theta_vec")
        rep = {x0: vec[0:2], sigma: vec[2], rho: vec[3:4], th: vec[4:5]}
        ll_v = pytensor.clone_replace(ll, replace=rep)
        f = pytensor.function([vec], [ll_v, pytensor.grad(ll_v, vec)])
    reps = min(theta.shape[0], 64)
    for b in range(min(warmup, reps)):
        f(theta[b])
    t0 = time.perf_counter()
    for _ in range(steps):
        for b in range(reps):
            f(theta[b])
    dt = (time.perf_counter() - t0) / steps
    return reps * y.shape[0] / dt, 1, dt * 1e3, reps


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from pymc_statespace_b200.synthetic import arma11_workload, arma21_workload

    sample = a.cpu_sample_draws or 8192
    _, y, theta = arma11_workload(sample, a.n)
    kind, why = "port", None
    try:
        val, cores, ms, reps = run_real_reference(theta, y, a.steps, a.warmup)
        kind = "reference"
        desc = (f"{reps} draws x T={a.n} per step through the reference's own PyTensor graph (BayesianARMA(1,1), "
                "default mode), one draw per call, 1 process")
    except Exception as e:  # noqa: BLE001 - anything from a missing wheel to a PyTensor compile error
        why = f"{type(e).__name__}: {e}"[:160]
        val, cores, ms = run_cpu(theta, y, a.steps, a.warmup)
        desc = (f"{sample} draws x T={a.n} per step, oracle/kalman_c.c (plain C + OpenMP on {cores} cores) - the reference "
                "(PyTensor/PyMC) is not importable in this image")
    if kind == "port":
        assert cores > 1 or host_cores() == 1, "CPU arm must use every host core"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a), "note": "CPU arm: each step evaluates a bounded sample of the workload"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": desc,
                         "real_reference_import": why or "ok"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not a.no_c5:
        try:
            _, y5, th5 = arma21_workload(sample, a.n)
            v5, c5cores, ms5 = run_cpu(th5, y5, 2, 1, order=(2, 1))
            line["c5"] = {"value": v5, "unit": UNIT, "cores": c5cores, "kind": "port", "ms_per_step": ms5,
                          "sample": f"{sample} draws x T={a.n}, ARMA(2,1), oracle/kalman_c.c"}
        except Exception as e:  # noqa: BLE001
            line["c5"] = {"unavailable": f"{type(e).__name__}: {e}"[:160]}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region (NVML in-process, every ~10 ms;
    falls back to one long-running `nvidia-smi -lms 50`)."""

    def __init__(self, index):
        self.index, self.sm, self.smmax, self.reasons = index, [], None, set()
        self.stop = threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run_nvml(self):
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.smmax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        while not self.stop.is_set():
            self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
            r = int(get_reasons(h))
            self.reasons |= {n for bit, n in names.items() if r & bit}
            self.stop.wait(0.01)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                 "-lms", "50"], stdout=subprocess.PIPE, text=True)
        try:
            while not self.stop.is_set():
                row = [x.strip() for x in proc.stdout.readline().split(",")]
                if len(row) >= 6 and row[0].replace(".", "").isdigit():
                    self.sm.append(float(row[0]))
                    self.smmax = float(row[1])
                    self.reasons |= {n for n, v in zip(names, row[2:6]) if v.lower().startswith("active")}
        finally:
            proc.kill()

    def _run(self):
        try:
            self._run_nvml()
        except Exception:
            try:
                self._run_smi()
            except Exception:
                pass

    def __enter__(self):
        self.th.start()
        time.sleep(0.05)
        return self

    def __exit__(self, *exc):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.smmax,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


# ---------------------------------------------------------------------------------------------- GPU side
def main():
    a = parse()
    if a.impl == "reference":
        return reference_arm(a)

    import torch
    import torch.distributed as dist

    from pymc_statespace_b200 import _lib, fp64_peak_tflops
    from pymc_statespace_b200.dist import GatherStepGraph
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.models import MATRICES
    from pymc_statespace_b200.synthetic import arma11_workload, arma21_workload

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    use_graph = not a.no_graph

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K calls bracketed by barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks.
        Returns (ms per call, what the last call returned)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms / steps, out

    def gather_graph(model, theta_d, waves):
        """Resident leg for N > 1 (and the wave pipeline of c5): one kernel graph per wave + NCCL all-gathers; eager fallback."""
        if use_graph:
            try:
                return GatherStepGraph(model, theta_d, waves=waves), "kernels of a wave replayed as one CUDA graph, NCCL eager on a comm stream"
            except Exception as e:  # noqa: BLE001 - NCCL capture refused: same sequence, eager
                torch.cuda.synchronize()
                return GatherStepGraph(model, theta_d, waves=waves, use_graph=False), f"eager ({type(e).__name__})"
        return GatherStepGraph(model, theta_d, waves=waves, use_graph=False), "eager"

    # ------------------------------------------------------------------ headline: configs[1]
    B, n = a.draws, a.n
    spec, y, theta_all = arma11_workload(B * world, n)
    theta_h = torch.from_numpy(np.ascontiguousarray(theta_all[rank * B:(rank + 1) * B])).pin_memory()
    theta_d = theta_h.to(dev)
    model = KalmanLogp(spec, y, n_draws=B, filter_type="standard", device=dev)
    out_h = torch.empty((B, 1 + spec.n_theta), dtype=torch.float64).pin_memory()   # this rank's shard, on the host

    if world == 1:
        resident_path = "KalmanLogp.logp_and_grad(theta_device) + pack"

        def step_resident():
            logp, grad = model.logp_and_grad(theta_d)
            return torch.cat([logp[:, None], grad], dim=1)
    else:
        gsg, how = gather_graph(model, theta_d, 1)
        resident_path = f"GatherStepGraph ({how}): kernels + one NCCL all-gather of [B,{1 + spec.n_theta}] f64 per rank"
        step_resident = gsg

    # draw-chunk branches of the host-step graph: with the round-2 kernels (0.65 ms per evaluation) the ~10 helper launches
    # per chunk cost more than the overlapped copies save - measured 0.795 / 0.840 / 0.848 / 0.849 / 1.13 ms for 1 / 2 / 4 / 8 /
    # 16 chunks (tools/graph_e2e_chunks.py); round 1's 1.45 ms evaluation gained 7 % from 4 chunks
    chunks = 1
    host_step = model.capture_host_step(theta_h, out_h, chunks=chunks) if use_graph else None

    def step_e2e():
        if host_step is not None:
            return host_step()                            # replay + stream synchronise: the numbers are on the host
        th = theta_h.to(dev, non_blocking=True)
        logp, grad = model.logp_and_grad(th)
        out_h.copy_(torch.cat([logp[:, None], grad], dim=1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out_h

    for _ in range(max(a.warmup, 3)):
        step_resident()
    launches0 = lib.kfb_launch_count()
    with ClockSampler(local) as clk:
        ms_step, last = timed(step_resident, a.steps)
    if a.dump_outputs and rank == 0:   # every draw of every rank, in draw order
        dump_rows(a.dump_outputs, "", last if world == 1 else step_resident.rows())
    launches = lib.kfb_launch_count() - launches0
    if launches == 0:  # graph replays do not pass through the launch counter: count one eager evaluation instead
        l0 = lib.kfb_launch_count()
        model.logp_and_grad(theta_d)
        launches = (lib.kfb_launch_count() - l0) * a.steps
    clocks = clk.summary()
    bad = int((model.info != 0).sum())

    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, a.steps)

    # per-kernel durations of the two recursion kernels, CUDA events on the launching stream
    mats = model._scatter(theta_d)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(a.steps)]
    torch.cuda.synchronize()
    for e in ev:
        e[0].record()
        model.kalman.forward(model.y, *[mats[k] for k in MATRICES], outputs=("loglik",), save_for_backward=True)
        e[1].record()
        model.kalman.backward(wrt=("a0", "P0", "T", "R", "Q"))
        e[2].record()
    torch.cuda.synchronize()
    ms_fwd = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))   # rqr + forward kernel
    ms_bwd = float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))   # adjoint kernel + rqr adjoint

    steps_per_eval = B * n
    value = steps_per_eval * world / (ms_step * 1e-3)
    e2e_value = steps_per_eval * world / (ms_e2e * 1e-3)

    # ------------------------------------------------------------------ c5: configs[4], the multi-GPU config
    c5 = None
    if not a.no_c5:
        c5 = bench_c5(a, world, rank, dev, timed, gather_graph, use_graph)

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")
        fp64_peak = fp64_peak_tflops(dev)
        fp64_peak_distinct = fp64_peak_tflops(dev, distinct_operands=True)
        traffic = {}
        try:  # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this exact workload
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            if B == 65536 and n == 1000:
                traffic = {k: tj[k]["dram_bytes_read"] + tj[k]["dram_bytes_write"] for k in ("adjoint", "forward")}
        except Exception:
            pass
        tape_bytes = B * (n - 1) * TAPE_BYTES_PER_STEP
        survey_bytes = B * (n - 1) * SURVEY_TAPE_BYTES_PER_STEP
        bwd_gbs = tape_bytes / (ms_bwd * 1e-3) / 1e9
        fwd_gbs = tape_bytes / (ms_fwd * 1e-3) / 1e9
        rnote = ("achieved = ALGORITHMIC bytes (SURVEY 8(d): 40 B per step and kernel for a store-all tape at k_states 2) / "
                 "CUDA-event time; frac > 1: the kernel beats the store-all HBM floor because it does not move what the "
                 "model's structure makes constant - moved_*: the bytes it really moves (16 B/step, reduced recursion, = "
                 "traffic measured by ncu) against the same time and peak; ")
        roof = {
            "adjoint": {"bound": "hbm", "kernel": "kf_p1_adjoint_kernel<2,false,false,false,4,true> (reverse sweep: TMA tape ring; Z = e0, H = 0, companion T, complete data promised by the model: reduced ARMA recursion, 16-byte tape entries)",
                        "achieved": survey_bytes / (ms_bwd * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": survey_bytes / (ms_bwd * 1e-3) / 1e9 / hbm_peak,
                        "peak_source": peak_src, "traffic": traffic.get("adjoint"), "ms_per_launch": ms_bwd,
                        "algorithmic_bytes_per_launch": survey_bytes, "moved_bytes_per_launch": tape_bytes,
                        "moved_achieved": bwd_gbs, "moved_frac": bwd_gbs / hbm_peak,
                        "note": rnote + "ms_per_launch includes the ~8 us R Q R^T adjoint helper launched with it"},
            "forward": {"bound": "hbm", "kernel": "kf_p1_forward_kernel<2,true,4,true> (loglik + tape; Z = e0, H = 0, companion T, complete data promised by the model: reduced ARMA recursion, 16-byte tape entries)",
                        "achieved": survey_bytes / (ms_fwd * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": survey_bytes / (ms_fwd * 1e-3) / 1e9 / hbm_peak,
                        "peak_source": peak_src, "traffic": traffic.get("forward"), "ms_per_launch": ms_fwd,
                        "algorithmic_bytes_per_launch": survey_bytes, "moved_bytes_per_launch": tape_bytes,
                        "moved_achieved": fwd_gbs, "moved_frac": fwd_gbs / hbm_peak,
                        "note": rnote + "ms_per_launch includes the ~6 us R Q R^T helper"},
        }
        dominant = "forward" if ms_fwd >= ms_bwd else "adjoint"
        other = "adjoint" if dominant == "forward" else "forward"
        alg_tflops = ALG_FLOPS_PER_STEP * steps_per_eval / ((ms_fwd + ms_bwd) * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(a), "k_states": 2, "k_endog": 1, "n_theta": spec.n_theta,
                       "gradient": "theta-level [B,5] (scatter + Lyapunov + Kalman adjoint)",
                       "l2": "no flush: each step streams a %.2f GB tape (write in forward, read in adjoint) >> 126 MB L2"
                             % (tape_bytes / 1e9),
                       "tape": "reduced recursion: a_t[0] and the leading (m-1) x (m-1) block of P_t, 16 B per step and kernel (store-all: 40 B)",
                       "parallelism": f"draws sharded x{world}; resident leg: {resident_path}" if world > 1 else "1 GPU",
                       "resident_path": resident_path, "draws_with_info": bad},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": int(theta_h.numel() * 8 * world),
                    "d2h_bytes_per_step": int(out_h.numel() * 8 * world),
                    "path": (f"KalmanLogp.capture_host_step on every rank: pinned H2D + evaluation + pinned D2H of the rank's "
                             f"shard replayed as one CUDA graph ({chunks} draw-chunk branch(es)), "
                             "stream-synchronised every step; no collective") if use_graph else
                            "eager: pinned H2D, logp_and_grad, pinned D2H, stream-synchronised every step"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof[dominant],
            "roofline_" + other: roof[other],
            "fp64": {"peak_tflops_measured": fp64_peak, "peak_tflops_distinct_operands": fp64_peak_distinct,
                     "algorithmic_tflops": alg_tflops, "algorithmic_frac": alg_tflops / fp64_peak,
                     "flops_per_step": ALG_FLOPS_PER_STEP,
                     "note": "ALGORITHMIC throughput: the reference algorithm's flop count (BASELINE.md section 3: 442 per "
                             "logp+grad step at k_states=2) divided by time - the kernels execute fewer (predictor form, "
                             "symmetric storage, reduced ARMA recursion), so this is not pipe utilisation"},
        }
        if c5 is not None:
            line["c5"] = c5
        if world == 1 and not a.no_cpu_baseline:
            sample = a.cpu_sample_draws or 16384
            _, ys, ths = arma11_workload(sample, n)
            reps = 3
            v, cores, ms = run_cpu(ths, ys, reps, 1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{sample} draws x T={n}, {reps} timed repeats ({ms:.0f} ms each), "
                                              "oracle/kalman_c.c forward+adjoint, OpenMP over draws"}
            # context only: the per-step Python restatement (closest analogue of the reference's PyTensor scan VM,
            # which BASELINE.md estimates at 7e3-3e4 steps/s/core) on one draw, forward + torch-autograd backward
            try:
                from oracle import models as om

                t0 = time.perf_counter()
                om.logp_and_grad_theta(lambda t: om.arma_matrices(t, (1, 1), True), ths[0], ys[:, :, None])
                line["cpu_baseline"]["python_oracle_steps_per_s_1core"] = n / (time.perf_counter() - t0)
            except Exception:
                pass
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_c5(a, world, rank, dev, timed, gather_graph, use_graph):
    """BASELINE.json configs[4]: ARMA(2,1), >= 2^20 draws per GPU x T = n, 4 waves through one evaluator per rank."""
    import torch

    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.synthetic import arma21_workload

    B5 = a.c5_draws or ((1 << 21) if world >= 8 else (1 << 20))
    # 2 waves: enough to hide the NCCL gather / PCIe copies of one wave under the kernels of the other, and large enough
    # (>= 2^19 draws = 27.7 warps per SM sub-partition) that the last, partially filled round of resident warps costs
    # < 10 % (4 waves of 2^18 draws measured 15.7 ms per 2^20 draws instead of ~14)
    # Waves of 2^19 draws whatever the shard size (2 at 2^20 draws per GPU, 4 at 2^21): the gather of the LAST wave is the
    # only exposed one, and with the round-2 kernels (2.3x faster, same bytes to gather) a 2^20-draw wave left ~9 % of an
    # 8-GPU step to it.
    waves = B5 >> 19 if (B5 >= (1 << 19) and B5 % (1 << 19) == 0) else (2 if B5 % 2 == 0 else 1)
    h = B5 // waves
    steps = a.c5_steps or a.steps
    spec, y, theta = arma21_workload(B5, a.n, seed=1 + rank)      # every rank draws its own shard
    nt = spec.n_theta
    theta_h = torch.from_numpy(np.ascontiguousarray(theta)).pin_memory()
    theta_d = theta_h.to(dev)
    out_h = torch.empty((B5, 1 + nt), dtype=torch.float64).pin_memory()
    model = KalmanLogp(spec, y, n_draws=h, filter_type="standard", device=dev)
    gsg, how = gather_graph(model, theta_d, waves)
    for _ in range(2):
        gsg()
    ms_res, _ = timed(gsg, steps)
    if a.dump_outputs and rank == 0:
        dump_rows(a.dump_outputs, "c5_", gsg.rows())
    bad = int((gsg.info != 0).sum())
    out0 = gsg.out[0, rank, :4].cpu().numpy().tolist() if rank == 0 else None
    host = model.capture_host_step(theta_h, out_h, chunks=waves, sequential=True) if use_graph else None

    def step_e2e():
        if host is not None:
            return host()
        for w in range(waves):
            th = theta_h[w * h:(w + 1) * h].to(dev, non_blocking=True)
            logp, grad = model.logp_and_grad(th)
            out_h[w * h:(w + 1) * h].copy_(torch.cat([logp[:, None], grad], dim=1), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, steps)
    total = B5 * world * a.n
    return {
        "workload": f"BayesianARMA(2,1) stationary init, {B5} draws/GPU x T={a.n} ({B5 * world} draws in total), standard "
                    "filter, logp+dlogp/dtheta",
        "value": total / (ms_res * 1e-3), "unit": UNIT, "ms_per_step": ms_res, "steps": steps, "n_gpus": world,
        "draws_per_gpu": B5, "waves": waves, "n_theta": nt, "draws_with_info": bad,
        "resident_path": f"GatherStepGraph ({how}): {waves} waves of {h} draws through one evaluator, "
                         + (f"NCCL all-gather of wave k ([{h},{1 + nt}] f64 per rank) under the kernels of wave k+1"
                            if world > 1 else "no collective at 1 GPU"),
        "e2e": {"value": total / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(theta_h.numel() * 8 * world), "d2h_bytes_per_step": int(out_h.numel() * 8 * world),
                "path": "HostStepGraph(sequential=True) on every rank: H2D / D2H of wave k on copy streams under the "
                        "kernels of the neighbouring waves; no collective"},
        "tape_bytes_per_gpu": int(h * (a.n - 1) * TAPE_BYTES_PER_STEP),
        "hbm_stream_gbs_per_gpu": 2 * B5 * (a.n - 1) * TAPE_BYTES_PER_STEP / (ms_res * 1e-3) / 1e9,
        "first_rows": out0,
    }


if __name__ == "__main__":
    main()
