"""Time-parallel vs sequential kernels (BatchedKalman(time_parallel=...)) on one GPU: one JSON line.

For ARMA(1,1) (stationary P0) and the local linear trend, B in {1, 4, 64, 1024} units x n in {100, 1000, 10000} steps:
  * kernel time of forward (loglik + tape) + adjoint (all nine cotangents), CUDA events around `--iters` launches
    after `--warmup`, per evaluation, for both modes;
  * the max relative difference of loglik and of every gradient between the modes on the same seeded inputs;
  * the crossover: the smallest B of the grid at which the sequential kernels are faster (null: never on the grid).
At B = 1 (what an unmodified PyMC NUTS calls per leapfrog step) also the seam latency of `seam.logp_grads_numpy` and
`seam.filter_numpy`: host clock around the call (each ends in a synchronised copy to numpy), median of `--reps`.
The GPU name and power limit are read in the same run.

    python tools/time_parallel_bench.py [--out FILE] [--quick]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NAMES = ("a0", "P0", "T", "Z", "R", "H", "Q")


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return name, q


def inputs(model, B, n, seed=0):
    """Seeded per-draw system matrices [B, ...] and one observed series [n, 1] (a few missing rows)."""
    from oracle import models as om
    from pymc_statespace_b200.synthetic import simulate_arma

    rng = np.random.default_rng(seed)
    if model == "arma11":
        y = simulate_arma(n, (0.6,), (0.3,), 1.0, seed=seed)[:, None]
        mats = [om.arma_matrices(torch.tensor([*rng.normal(size=2), np.exp(rng.normal(0, .3)), rng.uniform(-.9, .9),
                                               rng.normal(0, .5)], dtype=torch.float64), (1, 1), True) for _ in range(B)]
        a0, P0, T, Z, R, H, Q = (np.stack([mm[i].detach().numpy() for mm in mats]) for i in range(7))
        a0 = a0.reshape(B, -1)
    else:  # local linear trend
        y = np.cumsum(np.cumsum(rng.normal(size=n)) * 0.1 + rng.normal(size=n))[:, None]
        T = np.repeat(np.array([[[1.0, 1.0], [0.0, 1.0]]]), B, 0)
        Z, R = np.repeat(np.array([[[1.0, 0.0]]]), B, 0), np.repeat(np.eye(2)[None], B, 0)
        Q = np.stack([np.diag(np.exp(rng.normal(size=2)) * [0.5, 0.01]) for _ in range(B)])
        H = np.exp(rng.normal(size=(B, 1, 1)))
        a0, P0 = rng.normal(size=(B, 2)), np.repeat(np.eye(2)[None] * 10.0, B, 0)
    y[rng.choice(n, max(1, n // 100), replace=False)] = np.nan
    return y, dict(zip(NAMES, (a0, P0, T, Z, R, H, Q)))


def kernel_case(model, B, n, warmup, iters):
    from pymc_statespace_b200 import BatchedKalman

    y, mats = inputs(model, B, n, seed=B + n)
    dev = torch.device("cuda")
    yd = torch.as_tensor(y, device=dev)
    md = {k: torch.as_tensor(v, device=dev).contiguous() for k, v in mats.items()}
    m, r = mats["P0"].shape[-1], mats["R"].shape[-1]
    res = {}
    for tp in (False, True):
        bk = BatchedKalman("standard", n, m, 1, r, n_draws=B, time_parallel=tp)
        assert bk.time_parallel_active == tp

        def step():
            out = bk.forward(yd, **md, outputs=("loglik",), save_for_backward=True)
            return out, bk.backward()

        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            out, g = step()
        e1.record()
        e1.synchronize()
        res[tp] = (e0.elapsed_time(e1) * 1e3 / iters, out["loglik"].cpu().numpy(),
                   {k: v.cpu().numpy() for k, v in g.items()}, int((out["info"] != 0).sum()))

    def rel(a, b):
        return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))

    diff = {"loglik": rel(res[True][1], res[False][1])}
    diff.update({k: rel(res[True][2][k], res[False][2][k]) for k in res[False][2]})
    return {"model": model, "B": B, "n": n, "seq_us": round(res[False][0], 2), "tpar_us": round(res[True][0], 2),
            "speedup": round(res[False][0] / res[True][0], 3), "max_rel_diff_loglik": diff["loglik"],
            "max_rel_diff_grad": max(v for k, v in diff.items() if k != "loglik"),
            "bad_info": res[False][3] + res[True][3]}


def seam_case(model, n, reps):
    from pymc_statespace_b200.filters import FILTER_FACTORY
    from pymc_statespace_b200.seam import filter_numpy, logp_grads_numpy

    y, mats = inputs(model, 1, n, seed=n)
    arrays = {"data": y[:, :, None], **{k: v[0] for k, v in mats.items()}}
    arrays["a0"] = arrays["a0"][:, None]
    out = {"model": model, "n": n}
    for tp in (False, True):
        flt = FILTER_FACTORY["standard"]()
        flt.time_parallel = tp
        for name, call in (("logp_grads_numpy", lambda: logp_grads_numpy(flt, arrays)),
                           ("filter_numpy", lambda: filter_numpy(flt, *[arrays[k] for k in ("data",) + NAMES]))):
            for _ in range(5):
                call()
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                call()
                ts.append(time.perf_counter() - t0)
            out[f"{name}_{'tpar' if tp else 'seq'}_us"] = round(float(np.median(ts)) * 1e6, 1)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--quick", action="store_true", help="B in {1, 64}, n in {100, 1000}, few launches")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_parallel_bench.py needs a CUDA device")
    Bs, ns = ((1, 64), (100, 1000)) if a.quick else ((1, 4, 64, 1024), (100, 1000, 10000))
    iters = 5 if a.quick else a.iters
    name, power = gpu_info()
    rows = [kernel_case(model, B, n, a.warmup, iters) for model in ("arma11", "llt") for n in ns for B in Bs]
    crossover = {}
    for model in ("arma11", "llt"):
        for n in ns:
            wins = [r["B"] for r in rows if r["model"] == model and r["n"] == n and r["seq_us"] < r["tpar_us"]]
            crossover[f"{model}_n{n}"] = min(wins) if wins else None
    seam = [seam_case(model, n, 20 if a.quick else a.reps) for model in ("arma11", "llt") for n in ns]
    line = json.dumps({"tool": "time_parallel_bench", "gpu": name, "power_limit_and_max_sm_clock": power,
                       "kernel_fwd_plus_adjoint": rows, "crossover_B_sequential_faster": crossover, "seam_B1": seam,
                       "max_rel_diff_loglik": max(r["max_rel_diff_loglik"] for r in rows),
                       "max_rel_diff_grad": max(r["max_rel_diff_grad"] for r in rows)})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
