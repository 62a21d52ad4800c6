"""State draws, forecasts and conditional forecasts on data with partly observed rows, on one GPU: one JSON line.

Workload (theta level, the evaluator's own scatter and stationary P0): BayesianVARMAX(1,0), k = 3, with measurement
error; 4,096 draws x 64 paths; n = 1,000 observations of which about 10 % of the rows have one or two of the three
entries missing, plus a ragged edge (series 2 missing in the last two rows, series 1 in the last one).  This is the
nowcasting setting the masked filter is for.  The same data with those entries filled in (no partly observed row) run
today's path (kfb_forward) and are the baseline.
  * CUDA events around KalmanLogp.sample_states (64 paths), .forecast (horizon 24, 64 paths) and
    .conditional_forecast (series 0 known for the first 4 steps, 64 paths), normals given, ragged and filled data;
  * CUDA events around the masked filter (BatchedKalman.masked_filter) and kfb_forward with the full predicted outputs
    (BatchedKalman.forward, predicted_states and predicted_covs) on the same draws and ragged / filled data;
  * the masked filter's output bytes, 8 U (n + 1) (m + m m), over its time, next to a device-to-device copy measured in
    the same run.
The GPU name and power limit are read in the same run.

    python tools/partial_rows_bench.py [--out FILE] [--quick]
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

from conditional_forecast_bench import varmax10_k3  # noqa: E402
from simulation_smoother_bench import copy_peak_gbs, events_ms  # noqa: E402
from time_parallel_bench import gpu_info  # noqa: E402

DEV = "cuda:0"
KEYS = ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")


def ragged(y, seed=5):
    """About 10 % of the rows with one or two entries missing, and the ragged last two rows."""
    y = y.copy()
    n, p = y.shape
    rng = np.random.default_rng(seed)
    for t in rng.choice(n - 2, n // 10, replace=False):
        y[t, rng.choice(p, rng.integers(1, p), replace=False)] = np.nan
    y[n - 2, 2] = np.nan
    y[n - 1, 1:] = np.nan
    return y


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_partial_rows_bench.json"))
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from pymc_statespace_b200.logp import KalmanLogp

    name, power = gpu_info()
    copy_gbs = copy_peak_gbs()
    n = 200 if args.quick else 1000
    B, spu = (256, 16) if args.quick else (4096, 64)
    hor = 24
    spec, y_full, theta = varmax10_k3(B, n)
    y_rag = ragged(y_full)
    m, p, r = spec.k_states, spec.k_endog, spec.k_posdef
    S = B * spu
    th = torch.as_tensor(theta, device=DEV)
    f64 = dict(dtype=torch.float64, device=DEV)
    g = torch.Generator(device=DEV)
    g.manual_seed(0)
    cond = torch.full((hor, p), float("nan"), **f64)
    cond[:4, 0] = torch.linspace(-0.5, 0.5, 4, **f64)
    out = {"gpu": name, "power_limit_and_max_sm_clock": power, "d2d_copy_GBs": copy_gbs,
           "workload": {"model": "BayesianVARMAX(1,0), k = 3, measurement error", "draws": B, "paths_per_draw": spu,
                        "n": n, "horizon": hor,
                        "partly_observed_rows": int(((np.isnan(y_rag).sum(1) > 0) & (np.isnan(y_rag).sum(1) < p)).sum())},
           "call_timing": "CUDA events, mean over --iters calls after --warmup, normals given",
           "calls_ms": {}, "filter_ms": {}}
    for label, y in (("ragged", y_rag), ("filled", y_full)):
        model = KalmanLogp(spec, y, n_draws=B, filter_type="univariate", device=DEV)
        calls = {}
        zs = (torch.randn((S, m), generator=g, **f64), torch.randn((n - 1, S, r), generator=g, **f64),
              torch.randn((n, S, p), generator=g, **f64))
        calls["sample_states"] = events_ms(lambda: model.sample_states(th, spu, z_init=zs[0], z_state=zs[1],
                                                                       z_obs=zs[2]), args.warmup, args.iters)
        assert int((model.sample_states_info != 0).sum()) == 0
        del zs
        torch.cuda.empty_cache()
        zf = (torch.randn((S, m), generator=g, **f64), torch.randn((hor - 1, S, r), generator=g, **f64),
              torch.randn((hor, S, p), generator=g, **f64))
        kw = dict(z_init=zf[0], z_state=zf[1], z_obs=zf[2])
        calls["forecast"] = events_ms(lambda: model.forecast(th, hor, spu, **kw), args.warmup, args.iters)
        calls["conditional_forecast"] = events_ms(lambda: model.conditional_forecast(th, cond, spu, **kw),
                                                  args.warmup, args.iters)
        assert int((model.forecast(th, hor)["info"] != 0).sum()) == 0
        assert int((model.conditional_forecast(th, cond)["info"] != 0).sum()) == 0
        out["calls_ms"][label] = calls
        # the filters alone on the same draws
        mats = model.system_matrices(th)
        kal = model._exact_kalman(n)
        yt = torch.as_tensor(y, **f64)
        args_f = [mats[k] for k in KEYS]
        fl = {"masked_filter": events_ms(lambda: kal.masked_filter(yt, *args_f), args.warmup, args.iters)}
        if label == "filled":
            fl["kfb_forward_predicted_outputs"] = events_ms(
                lambda: kal.forward(yt, *args_f, outputs=("predicted_states", "predicted_covs")), args.warmup,
                args.iters)
        out["filter_ms"][label] = fl
        del model, kal, mats
        torch.cuda.empty_cache()
    out_bytes = 8 * B * (n + 1) * (m + m * m)
    t = out["filter_ms"]["ragged"]["masked_filter"]
    out["masked_filter_output_bytes"] = out_bytes
    out["masked_filter_share_of_d2d_copy"] = out_bytes / (t * 1e-3) / 1e9 / copy_gbs
    line = json.dumps(out)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
