"""Tiny k_states=6 theta-level logp+grad (rows kernels) for compute-sanitizer runs:
   compute-sanitizer --tool racecheck python tools/rows_racecheck.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from pymc_statespace_b200.synthetic import varmax20_workload
from pymc_statespace_b200.logp import KalmanLogp

spec, y, theta = varmax20_workload(n_draws=48, n=24, seed=1)
m = KalmanLogp(spec, y, n_draws=48, filter_type="standard")
th = torch.as_tensor(theta, device="cuda")
lp, g = m.logp_and_grad(th)
torch.cuda.synchronize()
print("logp sum", float(lp.sum()), "grad abs sum", float(g.abs().sum()))

# large systems (kf_rowsD.cuh): trend + seasonal, k_states = 30 (no T-bar), and a random k_states = 30 system with T-bar
from pymc_statespace_b200.synthetic import trend_seasonal_workload
spec, y, theta = trend_seasonal_workload(n_draws=6, n=12)
m = KalmanLogp(spec, y, n_draws=6, filter_type="standard")
lp, g = m.logp_and_grad(torch.as_tensor(theta, device="cuda"))
torch.cuda.synchronize()
print("k30 logp sum", float(lp.sum()), "grad abs sum", float(g.abs().sum()))
import numpy as np
from pymc_statespace_b200 import BatchedKalman
rng = np.random.default_rng(0)
B, n, mm, p, r = 5, 10, 30, 1, 3
dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
T = rng.normal(size=(B, mm, mm)) * 0.1 / np.sqrt(mm); Z = rng.normal(size=(B, p, mm)); R = rng.normal(size=(B, mm, r))
H = np.tile(np.eye(p) * 0.5, (B, 1, 1)); Q = np.tile(np.eye(r) * 0.3, (B, 1, 1))
a0 = rng.normal(size=(B, mm)); P0 = np.tile(np.eye(mm), (B, 1, 1)); yy = rng.normal(size=(n, p)); yy[3] = np.nan
bk = BatchedKalman("standard", n, mm, p, r, n_draws=B)
out = bk.forward(dev(yy), dev(a0), dev(P0), dev(T), dev(Z), dev(R), dev(H), dev(Q), outputs=("loglik",), save_for_backward=True)
gg = bk.backward(wrt=("a0", "P0", "T", "R", "H", "Q"))
torch.cuda.synchronize()
print("k30 with T-bar: loglik sum", float(out["loglik"].sum()), "gT abs sum", float(gg["T"].abs().sum()))

# round 2: steady state (DARE on the tensor cores) at k_states 30, and the 16 x 16 tile kernels (k_states 13 -> 14)
for period, kind in ((29, "steady_state"), (12, "standard"), (12, "steady_state")):
    spec, y, theta = trend_seasonal_workload(n_draws=6, n=12, period=period)
    m = KalmanLogp(spec, y, n_draws=6, filter_type=kind)
    lp, g = m.logp_and_grad(torch.as_tensor(theta, device="cuda"))
    torch.cuda.synchronize()
    print("period", period, kind, "logp sum", float(lp.sum()), "grad abs sum", float(g.abs().sum()))
B, n, mm, p, r = 5, 10, 12, 1, 2
T = rng.normal(size=(B, mm, mm)) * 0.1 / np.sqrt(mm); Z = rng.normal(size=(B, p, mm)); R = rng.normal(size=(B, mm, r))
H = np.tile(np.eye(p) * 0.5, (B, 1, 1)); Q = np.tile(np.eye(r) * 0.3, (B, 1, 1))
a0 = rng.normal(size=(B, mm)); P0 = np.tile(np.eye(mm), (B, 1, 1)); yy = rng.normal(size=(n, p)); yy[3] = np.nan
bk = BatchedKalman("standard", n, mm, p, r, n_draws=B)
out = bk.forward(dev(yy), dev(a0), dev(P0), dev(T), dev(Z), dev(R), dev(H), dev(Q), outputs=("loglik",), save_for_backward=True)
gg = bk.backward(wrt=("a0", "P0", "T", "R", "H", "Q"))
torch.cuda.synchronize()
print("k12 with T-bar: loglik sum", float(out["loglik"].sum()), "gT abs sum", float(gg["T"].abs().sum()))
