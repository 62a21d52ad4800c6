// TEST-ONLY: the simulation smoother of csrc/kf_simsmooth.cuh run on the host: the same unit_prep, gain_entry and
// simulate_one the kernels of kf_simsmooth.cu run, one (unit, t) and one simulation at a time, chosen by the same
// ss::with_instance (or the run-time-dims path when force_dyn is set).
#include <algorithm>
#include <cstring>
#include <vector>

#include "kf_simsmooth.cuh"

using namespace kfb;

// The arguments of kfb_simulation_smoother for n_draws x n_series units; the workspace is allocated here.
extern "C" int simsmooth_host_run(long long n_draws, long long n_series, long long spu, int n, int m, int p, int r,
                                  const double* y, long long y_bs, const double* a0, long long a0_bs, const double* P0,
                                  long long P0_bs, const double* T, long long T_bs, const double* Z, long long Z_bs,
                                  const double* R, long long R_bs, const double* H, long long H_bs, const double* Q,
                                  long long Q_bs, const double* c, long long c_bs, const double* d, long long d_bs,
                                  const double* pc, const double* z_init, const double* z_state, const double* z_obs,
                                  double* states, int* info, int force_dyn) {
  ss::Args A;
  std::memset(&A, 0, sizeof(A));
  A.U = n_draws * n_series; A.n_series = n_series; A.spu = spu; A.S = A.U * spu;
  A.n = n; A.m = m; A.p = p; A.r = r;
  A.y = {y, y_bs, 0}; A.a0 = {a0, a0_bs, 0}; A.P0 = {P0, P0_bs, 0}; A.T = {T, T_bs, 0}; A.Z = {Z, Z_bs, 0};
  A.R = {R, R_bs, 0}; A.H = {H, H_bs, 0}; A.Q = {Q, Q_bs, 0}; A.c = {c, c_bs, 0}; A.d = {d, d_bs, 0};
  A.pc = pc; A.z_init = z_init; A.z_state = z_state; A.z_obs = z_obs; A.states = states; A.info = info;
  const long long lanes = ss::warps_of(A.S) * 32;
  std::vector<double> gain(A.U * n * ss::gain_stride(m, p)), fac(A.U * ss::fac_stride(m, p, r));
  std::vector<double> uscr(n * lanes * p), rscr(std::max(n - 1, 1) * lanes * m);
  std::vector<int> ustat(A.U, ss::KEY_NONE);
  A.gain = gain.data(); A.fac = fac.data(); A.uscr = uscr.data(); A.rscr = rscr.data(); A.ustat = ustat.data();
  auto run = [&](auto dd) {
    for (long long u = 0; u < A.U; ++u) {
      ss::unit_prep(A, u);
      for (int t = 0; t < n; ++t) ss::gain_entry(dd, A, u, t);
    }
    for (long long s = 0; s < A.S; ++s) ss::simulate_one(dd, A, s);
  };
  if (force_dyn) {
    if (m > ss::SS_MAX || p > ss::SS_MAX || r > ss::SS_MAX) return 1;
    run(ss::Dyn{m, p, r});
    return 0;
  }
  return ss::with_instance(m, p, r, run) ? 0 : 1;
}

// 1 if (m, p, r) has a compile-time instantiation
extern "C" int simsmooth_host_is_static(int m, int p, int r) {
  bool st = false;
  ss::with_instance(m, p, r, [&](auto dd) { st = decltype(dd)::STATIC; });
  return st ? 1 : 0;
}
