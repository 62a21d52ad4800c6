"""Time-parallel vs sequential RTS smoother (rts_smoother(time_parallel=...)) on one GPU: one JSON line.

Filtered moments of ARMA(1,1) and the local linear trend (the inputs of tools/time_parallel_bench.py), plus a k_states 4
point, for B in {1, 4, 64, 1024} units x n in {100, 1000, 10000} steps:
  * kernel time of one smoother call (R Q R^T hoist + smoother kernel) for both modes: up to `--iters` calls (about
    0.2 s of GPU work) captured as one CUDA graph after `--warmup` calls, CUDA events around one replay;
  * the max relative difference between the modes on the same seeded inputs;
  * the crossover: the smallest B of the grid at which the sequential kernel is faster (null: never on the grid).
At B = 1 also the latency of KalmanSmoother().build_graph with numpy inputs in both modes, next to seam.filter_numpy
(time_parallel filter) for context: host clock around the call, median of `--reps`.
The GPU name and power limit are read in the same run.

    python tools/time_parallel_smoother_bench.py [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from time_parallel_bench import gpu_info, inputs  # noqa: E402


def filtered(model, B, n):
    """Seeded per-draw T, R, Q [B, ...] and the filtered moments [B, n, m], [B, n, m, m] of the sequential filter."""
    from pymc_statespace_b200 import BatchedKalman

    if model == "k4":
        rng = np.random.default_rng(B + n)
        y = rng.normal(size=(n, 1))
        y[rng.choice(n, max(1, n // 100), replace=False)] = np.nan
        T = np.stack([np.diag([0.9, 0.5, -0.3, 0.2]) + 0.05 * rng.normal(size=(4, 4)) for _ in range(B)])
        mats = dict(a0=np.zeros((B, 4)), P0=np.repeat(np.eye(4)[None], B, 0), T=T,
                    Z=np.repeat(np.array([[[1.0, 1.0, 0.0, 0.5]]]), B, 0), R=np.repeat(np.eye(4)[None], B, 0),
                    H=np.ones((B, 1, 1)), Q=np.repeat(np.eye(4)[None] * 0.3, B, 0))
    else:
        y, mats = inputs(model, B, n, seed=B + n)
    m, r = mats["T"].shape[-1], mats["R"].shape[-1]
    dev = torch.device("cuda")
    d = {k: torch.as_tensor(np.ascontiguousarray(v), device=dev) for k, v in mats.items()}
    bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, device=dev)
    out = bk.forward(torch.as_tensor(y, device=dev), d["a0"], d["P0"], d["T"], d["Z"], d["R"], d["H"], d["Q"],
                     outputs=("filtered_states", "filtered_covs"))
    return d, out["filtered_states"].contiguous(), out["filtered_covs"].contiguous()


def kernel_case(model, B, n, warmup, iters):
    from pymc_statespace_b200.engine import rts_smoother, smoother_workspace_numel

    d, fs, fc = filtered(model, B, n)
    m = fs.shape[-1]
    ws = torch.empty(smoother_workspace_numel(B, m), dtype=torch.float64, device=fs.device)
    res, outs = {}, {}
    for tp in (False, True):
        ss, sc = torch.empty_like(fs), torch.empty_like(fc)
        call = lambda: rts_smoother(d["T"], d["R"], d["Q"], fs, fc, time_parallel=tp, out=(ss, sc), workspace=ws)  # noqa: E731,B023
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                call()
        side.synchronize()
        # one call on the host clock sizes the graph: about 0.2 s of GPU work per replay, at most `iters` calls
        t0 = time.perf_counter()
        call()
        torch.cuda.synchronize()
        k = int(max(3, min(iters, 0.2 / max(time.perf_counter() - t0, 1e-6))))
        # the k calls are captured as one CUDA graph, so the host's issue rate does not enter the time
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for _ in range(k):
                call()
        graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        res["tpar_us" if tp else "seq_us"] = e0.elapsed_time(e1) * 1e3 / k
        res["tpar_calls" if tp else "seq_calls"] = k
        outs[tp] = (ss.clone(), sc.clone())
    rel = max(float((outs[True][k] - outs[False][k]).abs().max() / outs[False][k].abs().max().clamp_min(1e-300))
              for k in (0, 1))
    res["max_rel_diff"] = rel
    res["speedup"] = res["seq_us"] / res["tpar_us"]
    return res


def seam_latency(model, n, reps):
    from pymc_statespace_b200.filters import KalmanSmoother, StandardFilter
    from pymc_statespace_b200.seam import filter_numpy

    y, mats = inputs(model, 1, n, seed=1 + n)
    a = {k: v[0] for k, v in mats.items()}
    a["a0"] = a["a0"].reshape(-1, 1)
    flt = StandardFilter()
    flt.time_parallel = True
    args = (y[:, :, None], a["a0"], a["P0"], a["T"], a["Z"], a["R"], a["H"], a["Q"])
    outs = filter_numpy(flt, *args)

    def timed(fn):
        for _ in range(5):
            fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts) * 1e6)

    res = {"filter_numpy_tpar_us": timed(lambda: filter_numpy(flt, *args))}
    for tp in (False, True):
        sm = KalmanSmoother()
        sm.time_parallel = tp
        res["smoother_numpy_tpar_us" if tp else "smoother_numpy_seq_us"] = timed(
            lambda: sm.build_graph(a["T"], a["R"], a["Q"], outs[0], outs[2]))  # noqa: B023
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_time_parallel_smoother_bench.json"))
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = gpu_info()
    Bs, ns = ((1, 64), (100, 1000)) if args.quick else ((1, 4, 64, 1024), (100, 1000, 10000))
    out = {"gpu": name, "power_limit_and_max_sm_clock": power,
           "kernel_timing": "per call: CUDA events around one replay of a CUDA graph of *_calls captured calls "
                            "(R Q R^T hoist + smoother kernel)",
           "seam_timing": "per call: host clock around KalmanSmoother().build_graph / seam.filter_numpy with numpy "
                          "inputs at B = 1, median of --reps",
           "kernel": {}, "crossover_B": {}, "seam_B1": {}}
    for model in ("arma11", "llt", "k4"):
        for n in ns:
            cross = None
            for B in Bs:
                r = kernel_case(model, B, n, args.warmup, args.iters)
                out["kernel"][f"{model}_B{B}_n{n}"] = r
                if cross is None and r["seq_us"] < r["tpar_us"]:
                    cross = B
            out["crossover_B"][f"{model}_n{n}"] = cross
    for model in ("arma11", "llt"):
        for n in ns:
            out["seam_B1"][f"{model}_n{n}"] = seam_latency(model, n, args.reps)
    line = json.dumps(out)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
