"""Conditional forecasts (KalmanLogp.conditional_forecast: moments and joint paths given known future values) on one
GPU: one JSON line.

Workloads (theta level, the evaluator's own scatter and stationary P0; n = 1,000 observations; 4,096 draws x 64 paths):
  * BayesianVARMAX(1,0), k = 3, measurement error (compile-time k_states 3, k_endog 3), horizon 24, series 0
    conditioned over the first 8 steps - the scenario analysis this feature is for;
  * BayesianARMA(1,1) (k_states 2, k_endog 1), horizon 100, the series conditioned over the first 8 steps.
Per workload:
  * CUDA events around one conditional_forecast call with the normals given, and around the unconditional forecast
    of the same horizon and paths on the same draws (KalmanLogp.forecast), mean of --iters calls after --warmup;
  * in a separate torch.profiler run, the device time per call of the window kernel, the paths kernel and the rest
    (theta scatter, Lyapunov, R Q R^T, the forward filter over the n observations, the start copies);
  * the paths kernel's bytes over its time, next to a device-to-device copy measured in the same run: the minimal model
    (normals read once, 8 (m + (H-1) r + H p), and paths written once, 8 H (m + p), per simulation) and the model of
    what the kernel moves (normals read twice, the u and r scratch written and read, 8 (H p + (H-1) m) each way).
The GPU name and power limit are read in the same run.

    python tools/conditional_forecast_bench.py [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from simulation_smoother_bench import copy_peak_gbs, events_ms  # noqa: E402
from time_parallel_bench import gpu_info  # noqa: E402

DEV = "cuda:0"


def varmax10_k3(B, n, seed=1):
    from pymc_statespace_b200.models import varmax_spec

    k = 3
    rng = np.random.default_rng(seed)
    spec = varmax_spec(k, (1, 0), stationary_initialization=True, measurement_error=True)
    L = np.tril(rng.normal(0.0, 0.1, (B, k, k)), -1) + np.eye(k) * 0.5
    theta = np.concatenate([rng.normal(0, 0.1, (B, k)), rng.uniform(-0.3, 0.3, (B, k * k)),
                            (L @ L.transpose(0, 2, 1)).reshape(B, -1), np.exp(rng.normal(-1.0, 0.2, (B, k)))], axis=1)
    y = rng.normal(size=(n, k))
    return spec, y, theta


def workload(name, quick):
    from pymc_statespace_b200.synthetic import arma11_workload

    n = 200 if quick else 1000
    B, spu = (256, 16) if quick else (4096, 64)
    if name == "varmax10_k3":
        spec, y, theta = varmax10_k3(B, n)
        hor = 24
    else:
        spec, y, theta = arma11_workload(B, n)
        hor = 100
    return spec, y, theta, B, spu, n, hor


def profile_split(fn, iters=3):
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    split = {"window_kernel_ms": 0.0, "paths_kernel_ms": 0.0, "forward_and_setup_ms": 0.0}
    for ev in prof.key_averages():
        t = ev.device_time_total / 1e3 / iters if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3 / iters
        if "condfc_window_kernel" in ev.key:
            split["window_kernel_ms"] += t
        elif "condfc_paths_kernel" in ev.key:
            split["paths_kernel_ms"] += t
        else:
            split["forward_and_setup_ms"] += t
    return split


def run_case(name, quick, warmup, iters, copy_gbs):
    from pymc_statespace_b200.logp import KalmanLogp

    spec, y, theta, B, spu, n, hor = workload(name, quick)
    model = KalmanLogp(spec, y, n_draws=B, filter_type="standard", device=DEV)
    th = torch.as_tensor(theta, device=DEV)
    m, p, r = spec.k_states, spec.k_endog, spec.k_posdef
    S = B * spu
    g = torch.Generator(device=DEV)
    g.manual_seed(0)
    f64 = dict(dtype=torch.float64, device=DEV)
    normals = (torch.randn((S, m), generator=g, **f64), torch.randn((hor - 1, S, r), generator=g, **f64),
               torch.randn((hor, S, p), generator=g, **f64))
    cond = torch.full((hor, p), float("nan"), **f64)
    cond[:8, 0] = torch.linspace(-0.5, 0.5, 8, **f64)
    kw = dict(z_init=normals[0], z_state=normals[1], z_obs=normals[2])
    call = lambda: model.conditional_forecast(th, cond, spu, **kw)  # noqa: E731
    cond_ms = events_ms(call, warmup, iters)
    fc_ms = events_ms(lambda: model.forecast(th, hor, spu, **kw), warmup, iters)
    moments_ms = events_ms(lambda: model.conditional_forecast(th, cond), warmup, iters)
    info = call()["info"]
    n_bad = int((info != 0).sum())
    split = profile_split(call)
    del normals, kw
    torch.cuda.empty_cache()
    normals_b = 8 * S * (m + (hor - 1) * r + hor * p)
    out_b = 8 * S * hor * (m + p)
    scratch_b = 2 * 8 * S * (hor * p + (hor - 1) * m)
    minimal, moved = normals_b + out_b, 2 * normals_b + out_b + scratch_b
    kp = split["paths_kernel_ms"]
    gbs = lambda b: b / (kp * 1e-3) / 1e9 if kp > 0 else None  # noqa: E731
    return {
        "draws": B, "paths_per_draw": spu, "n": n, "horizon": hor, "conditioned": "series 0, steps 0..7",
        "k_states": m, "k_endog": p, "k_posdef": r, "draws_with_nonzero_info": n_bad,
        "conditional_forecast_call_ms_cuda_events": cond_ms,
        "conditional_forecast_moments_only_ms_cuda_events": moments_ms,
        "forecast_same_call_ms_cuda_events": fc_ms,
        "split_ms_torch_profiler": split,
        "simulation_steps_per_s": S * hor / (kp * 1e-3) if kp > 0 else None,
        "paths_kernel_minimal_bytes": minimal,
        "paths_kernel_moved_bytes": moved,
        "paths_kernel_minimal_share_of_d2d_copy": gbs(minimal) / copy_gbs if kp > 0 else None,
        "paths_kernel_moved_share_of_d2d_copy": gbs(moved) / copy_gbs if kp > 0 else None,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_conditional_forecast_bench.json"))
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=6)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = gpu_info()
    copy_gbs = copy_peak_gbs()
    out = {"gpu": name, "power_limit_and_max_sm_clock": power, "d2d_copy_GBs": copy_gbs,
           "call_timing": "CUDA events around KalmanLogp.conditional_forecast / .forecast, normals given (mean over "
                          "--iters calls after --warmup)",
           "split_timing": "torch.profiler device time per call, mean of 3 calls; forward_and_setup = theta scatter, "
                           "Lyapunov, R Q R^T, the forward filter over the n observations and the start copies",
           "byte_model": "minimal: normals read once + paths written once; moved: normals read twice + u, r scratch "
                         "written and read + paths written",
           "workloads": {}}
    for w in ("varmax10_k3", "arma11"):
        out["workloads"][w] = run_case(w, args.quick, args.warmup, args.iters, copy_gbs)
        torch.cuda.empty_cache()
    line = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
