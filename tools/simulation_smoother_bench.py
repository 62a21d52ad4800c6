"""Simulation smoother (KalmanLogp.sample_states: joint posterior draws of the state paths) on one GPU: one JSON line.

Workloads (theta level, the evaluator's own scatter and stationary P0):
  * BayesianARMA(1,1), 4,096 draws x 64 paths x T = 1,000 (compile-time k_states 2, k_endog 1);
  * local linear trend, the same sizes (k_states 2, k_posdef 2);
  * trend + seasonal of period 12 (13 states, run on the 14-state padded spec: the run-time-dims path),
    1,024 draws x 8 paths x T = 1,000.
Per workload:
  * CUDA events around one sample_states call with the normals given (mean of --iters calls after --warmup), split in a
    separate torch.profiler run into the forward filter (kfb_forward, predicted covariances), the gain pass and the
    per-simulation kernel;
  * host clock around sample_states with the normals drawn inside (torch.randn), ending in a device synchronise;
  * simulation-steps/s of the per-simulation kernel, and its modelled bytes (8 (2r + 3p + 3m) per simulation-step:
    z_state read twice, z_obs once, the u scratch written and read, the r scratch written and read, the output; plus
    the gain tape read once) over its time, next to a device-to-device copy measured in the same run (bytes read +
    written over time, 2 GiB buffer);
  * the marginal path on the same draws: smooth() + conditional_simulation (independent draws per time step);
  * the numpy restatement (oracle/simsmooth.py) on one process for 1 unit x 4 paths, per simulation-step, labelled
    as such.
The GPU name and power limit are read in the same run.

    python tools/simulation_smoother_bench.py [--out FILE] [--quick]
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

from time_parallel_bench import gpu_info  # noqa: E402

DEV = "cuda:0"


def events_ms(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def copy_peak_gbs():
    x = torch.empty(1 << 28, dtype=torch.float64, device=DEV)  # 2 GiB
    y = torch.empty_like(x)
    ms = events_ms(lambda: y.copy_(x), 3, 10)
    return 2 * x.numel() * 8 / ms / 1e6


def workload(name, quick):
    from pymc_statespace_b200.models import local_level_spec
    from pymc_statespace_b200.synthetic import arma11_workload, trend_seasonal_workload

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
        B, spu = (64, 4) if quick else (1024, 8)
        spec, y, theta = trend_seasonal_workload(B, n, period=12)
    return spec, y, theta, B, spu, n


def profile_split(model, th, spu, normals, iters=3):
    """Mean device time per call of the forward kernels, the gain pass and the per-simulation kernel."""
    from torch.profiler import ProfilerActivity, profile

    model.sample_states(th, spu, z_init=normals[0], z_state=normals[1], z_obs=normals[2])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            model.sample_states(th, spu, z_init=normals[0], z_state=normals[1], z_obs=normals[2])
        torch.cuda.synchronize()
    split = {"gain_pass_ms": 0.0, "simulation_kernel_ms": 0.0, "forward_and_setup_ms": 0.0}
    for ev in prof.key_averages():
        t = ev.device_time_total / 1e3 / iters if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3 / iters
        if "simsmooth_gain_kernel" in ev.key:
            split["gain_pass_ms"] += t
        elif "simsmooth_sim_kernel" in ev.key:
            split["simulation_kernel_ms"] += t
        else:
            split["forward_and_setup_ms"] += t  # theta scatter, Lyapunov, R Q R^T, the forward filter, the status memset
    return split


def run_case(name, quick, warmup, iters, copy_gbs):
    from oracle import simsmooth as oss
    from pymc_statespace_b200.logp import KalmanLogp
    from pymc_statespace_b200.simulation import conditional_simulation

    spec, y, theta, B, spu, n = workload(name, quick)
    model = KalmanLogp(spec, y, n_draws=B, filter_type="standard", device=DEV)
    th = torch.as_tensor(theta, device=DEV)
    m0, m, p, r = model.k_states_model, model.spec.k_states, spec.k_endog, spec.k_posdef
    S = B * spu
    g = torch.Generator(device=DEV)
    g.manual_seed(0)
    f64 = dict(dtype=torch.float64, device=DEV)
    normals = (torch.randn((S, m0), generator=g, **f64), torch.randn((n - 1, S, r), generator=g, **f64),
               torch.randn((n, S, p), generator=g, **f64))
    call_ms = events_ms(lambda: model.sample_states(th, spu, z_init=normals[0], z_state=normals[1], z_obs=normals[2]), warmup, iters)
    assert int((model.sample_states_info != 0).sum()) == 0
    split = profile_split(model, th, spu, normals)
    host = []
    for _ in range(max(3, iters // 2)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.sample_states(th, spu, generator=g)
        torch.cuda.synchronize()
        host.append((time.perf_counter() - t0) * 1e3)

    def marginal():
        ss, sc, _ = model.smooth(th)
        return conditional_simulation(ss, sc, spu, generator=g)

    marginal_ms = events_ms(marginal, 1, max(2, iters // 2))
    steps = S * n
    bytes_sim = steps * 8 * (2 * r + 3 * p + 3 * m) + B * n * 8 * (m * p + p * p)
    ksim = split["simulation_kernel_ms"]
    # numpy restatement: one unit, 4 paths, one process
    one = KalmanLogp(spec, y, n_draws=1, filter_type="standard", device=DEV)
    mt = {k: (v[0] if v.ndim == len(one._shape[k]) + 1 else v).cpu().numpy()
          for k, v in one.system_matrices(th[:1]).items()}
    yy = np.asarray(y, dtype=np.float64).reshape(n, p)
    rng = np.random.default_rng(0)
    zi, zs, zo = rng.normal(size=(4, m)), rng.normal(size=(n - 1, 4, r)), rng.normal(size=(n, 4, p))
    t0 = time.perf_counter()
    oss.simulation_smoother(yy, mt["a0"], mt["P0"], mt["T"], mt["Z"], mt["R"], mt["H"], mt["Q"], mt["c"], mt["d"],
                            zi, zs, zo)
    np_s = time.perf_counter() - t0
    return {
        "draws": B, "paths_per_draw": spu, "n": n, "k_states_run": m, "k_states_model": m0, "k_endog": p, "k_posdef": r,
        "call_ms_cuda_events": call_ms,
        "split_ms_torch_profiler": split,
        "host_end_to_end_ms_median": float(np.median(host)),
        "simulation_steps_per_s": steps / (ksim * 1e-3) if ksim > 0 else None,
        "simulation_kernel_model_bytes": bytes_sim,
        "simulation_kernel_model_GBs": bytes_sim / (ksim * 1e-3) / 1e9 if ksim > 0 else None,
        "simulation_kernel_share_of_d2d_copy": (bytes_sim / (ksim * 1e-3) / 1e9) / copy_gbs if ksim > 0 else None,
        "marginal_path_ms_cuda_events": marginal_ms,
        "numpy_restatement_one_process_1unit_x4paths_s": np_s,
        "numpy_restatement_us_per_simulation_step": np_s / (4 * n) * 1e6,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_simulation_smoother_bench.json"))
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=6)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = gpu_info()
    copy_gbs = copy_peak_gbs()
    out = {"gpu": name, "power_limit_and_max_sm_clock": power, "d2d_copy_GBs": copy_gbs,
           "call_timing": "CUDA events around sample_states with the normals given (mean over --iters calls)",
           "split_timing": "torch.profiler device time per call, mean of 3 calls; forward_and_setup = theta scatter, "
                           "Lyapunov, R Q R^T, the forward filter and the status memset",
           "byte_model": "8 (2 r + 3 p + 3 m) bytes per simulation-step + the gain tape read once; m = k_states run",
           "workloads": {}}
    for w in ("arma11", "local_linear_trend", "trend_seasonal12"):
        out["workloads"][w] = run_case(w, args.quick, args.warmup, args.iters, copy_gbs)
        torch.cuda.empty_cache()
    line = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
