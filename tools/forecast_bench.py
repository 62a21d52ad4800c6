"""Forecasts from the end of the sample (KalmanLogp.forecast: moments and joint paths) on one GPU: one JSON line.

Workloads (theta level, the evaluator's own scatter and stationary P0; n = 1,000 observations):
  * BayesianARMA(1,1), 4,096 draws x 64 paths, horizons 100 and 1,000 (compile-time k_states 2, k_endog 1, k_posdef 1);
  * local linear trend, the same sizes (k_states 2, k_posdef 2);
  * VARMAX(2,0) with k = 3 and measurement error (k_states 6: the run-time-dims path), 1,024 draws x 16 paths, horizon
    100.
Per workload:
  * CUDA events around one forecast call with the normals given, and around one with the normals drawn inside
    (torch.randn), mean of --iters calls after --warmup;
  * in a separate torch.profiler run, the device time per call of the prep kernel, the paths kernel and the rest (theta
    scatter, Lyapunov, R Q R^T, the forward filter over n + H steps, the observation moments, the start copies);
  * the paths kernel's modelled bytes (normals read: 8 (m + (H-1) r + H p) per simulation; outputs written:
    8 H (m + p) per simulation - 8 (r + p) + 8 (m + p) per simulation-step) over its time, next to a device-to-device
    copy measured in the same run (bytes read + written over time, 2 GiB buffer);
  * the numpy restatement (oracle/forecast.py forecast_paths) on one process for 1 unit x 4 paths, per
    simulation-step, labelled as a CPU reference.
The GPU name and power limit are read in the same run.

    python tools/forecast_bench.py [--out FILE] [--quick]
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

from simulation_smoother_bench import copy_peak_gbs, events_ms  # noqa: E402
from time_parallel_bench import gpu_info  # noqa: E402

DEV = "cuda:0"


def workload(name, quick):
    from pymc_statespace_b200.models import local_level_spec
    from pymc_statespace_b200.synthetic import arma11_workload, varmax20_workload

    n = 200 if quick else 1000
    if name == "arma11":
        B, spu = (256, 16) if quick else (4096, 64)
        spec, y, theta = arma11_workload(B, n)
    elif name == "local_linear_trend":
        B, spu = (256, 16) if quick else (4096, 64)
        rng = np.random.default_rng(3)
        spec = local_level_spec()
        theta = np.tile([0.0, 0.0, 1.0, 0.0, 0.0, 1.0, 0.8, 0.5, 0.01], (B, 1))
        theta[:, 6:] *= np.exp(rng.normal(0, 0.2, (B, 3)))
        y = np.cumsum(rng.normal(size=n))[:, None]
    else:
        B, spu = (64, 4) if quick else (1024, 16)
        spec, y, theta = varmax20_workload(B, n, k=3)
    return spec, y, theta, B, spu, n


def profile_split(model, th, hor, spu, normals, iters=3):
    """Mean device time per call of the prep kernel, the paths kernel and everything else."""
    from torch.profiler import ProfilerActivity, profile

    model.forecast(th, hor, spu, z_init=normals[0], z_state=normals[1], z_obs=normals[2])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            model.forecast(th, hor, spu, z_init=normals[0], z_state=normals[1], z_obs=normals[2])
        torch.cuda.synchronize()
    split = {"prep_kernel_ms": 0.0, "paths_kernel_ms": 0.0, "forward_and_setup_ms": 0.0}
    for ev in prof.key_averages():
        t = ev.device_time_total / 1e3 / iters if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3 / iters
        if "forecast_prep_kernel" in ev.key:
            split["prep_kernel_ms"] += t
        elif "forecast_paths_kernel" in ev.key:
            split["paths_kernel_ms"] += t
        else:
            split["forward_and_setup_ms"] += t
    return split


def run_case(name, hor, quick, warmup, iters, copy_gbs):
    from oracle import forecast as ofc
    from pymc_statespace_b200.logp import KalmanLogp

    spec, y, theta, B, spu, n = workload(name, quick)
    model = KalmanLogp(spec, y, n_draws=B, filter_type="standard", device=DEV)
    th = torch.as_tensor(theta, device=DEV)
    m, p, r = spec.k_states, spec.k_endog, spec.k_posdef
    S = B * spu
    g = torch.Generator(device=DEV)
    g.manual_seed(0)
    f64 = dict(dtype=torch.float64, device=DEV)
    normals = (torch.randn((S, m), generator=g, **f64), torch.randn((hor - 1, S, r), generator=g, **f64),
               torch.randn((hor, S, p), generator=g, **f64))
    given_ms = events_ms(lambda: model.forecast(th, hor, spu, z_init=normals[0], z_state=normals[1], z_obs=normals[2]),
                         warmup, iters)
    info = model.forecast(th, hor, spu, z_init=normals[0], z_state=normals[1], z_obs=normals[2])["info"]
    n_bad = int((info != 0).sum())
    inside_ms = events_ms(lambda: model.forecast(th, hor, spu, generator=g), warmup, iters)
    moments_ms = events_ms(lambda: model.forecast(th, hor), warmup, iters)
    split = profile_split(model, th, hor, spu, normals)
    del normals
    torch.cuda.empty_cache()
    steps = S * hor
    bytes_paths = 8 * S * (m + (hor - 1) * r + hor * p) + 8 * S * hor * (m + p)
    kp = split["paths_kernel_ms"]
    # numpy restatement: one unit, 4 paths, one process
    mats = {k: (v[0] if v.ndim == len(model._shape[k]) + 1 else v).cpu().numpy()
            for k, v in model.system_matrices(th).items()}
    mom = ofc.forecast_moments(np.asarray(y, dtype=np.float64).reshape(n, p), mats["a0"], mats["P0"], mats["T"],
                               mats["Z"], mats["R"], mats["H"], mats["Q"], mats["c"], mats["d"], horizon=hor)
    rng = np.random.default_rng(0)
    zi, zs, zo = rng.normal(size=(4, m)), rng.normal(size=(hor - 1, 4, r)), rng.normal(size=(hor, 4, p))
    t0 = time.perf_counter()
    ofc.forecast_paths(mom["state_mean"][0], mom["state_cov"][0], mats["T"], mats["Z"], mats["R"], mats["H"], mats["Q"],
                       mats["c"], mats["d"], zi, zs, zo)
    np_s = time.perf_counter() - t0
    return {
        "draws": B, "paths_per_draw": spu, "n": n, "horizon": hor, "k_states": m, "k_endog": p, "k_posdef": r,
        "draws_with_nonzero_info": n_bad,
        "call_ms_cuda_events_normals_given": given_ms,
        "call_ms_cuda_events_normals_drawn_inside": inside_ms,
        "call_ms_cuda_events_moments_only": moments_ms,
        "split_ms_torch_profiler": split,
        "simulation_steps_per_s": steps / (kp * 1e-3) if kp > 0 else None,
        "paths_kernel_model_bytes": bytes_paths,
        "paths_kernel_model_GBs": bytes_paths / (kp * 1e-3) / 1e9 if kp > 0 else None,
        "paths_kernel_share_of_d2d_copy": (bytes_paths / (kp * 1e-3) / 1e9) / copy_gbs if kp > 0 else None,
        "cpu_reference_numpy_restatement_1unit_x4paths_s": np_s,
        "cpu_reference_numpy_us_per_simulation_step": np_s / (4 * hor) * 1e6,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_forecast_bench.json"))
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=6)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = gpu_info()
    copy_gbs = copy_peak_gbs()
    out = {"gpu": name, "power_limit_and_max_sm_clock": power, "d2d_copy_GBs": copy_gbs,
           "call_timing": "CUDA events around KalmanLogp.forecast (mean over --iters calls after --warmup)",
           "split_timing": "torch.profiler device time per call, mean of 3 calls, normals given; forward_and_setup = "
                           "theta scatter, Lyapunov, R Q R^T, the forward filter over n + H steps, the observation "
                           "moments and the start copies",
           "byte_model": "paths kernel: 8 (m + (H-1) r + H p) read + 8 H (m + p) written per simulation",
           "workloads": {}}
    cases = [("arma11", 100), ("arma11", 1000), ("local_linear_trend", 100), ("local_linear_trend", 1000),
             ("varmax20_k3", 100)]
    for w, hor in cases:
        out["workloads"][f"{w}_H{hor}"] = run_case(w, hor, args.quick, args.warmup, args.iters, copy_gbs)
        torch.cuda.empty_cache()
    line = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
