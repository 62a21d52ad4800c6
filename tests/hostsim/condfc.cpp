// TEST-ONLY: the conditional forecasts of csrc/kf_condfc.cuh run on the host: the same window_unit and path_unit the
// kernels of kf_condfc.cu run, one unit and one simulation at a time, chosen by the same ss::with_instance (or the
// run-time-dims path when force_dyn is set).
#include <algorithm>
#include <cstring>
#include <vector>

#include "kf_condfc.cuh"

using namespace kfb;

// The arguments of kfb_conditional_forecast for n_draws x n_series units; the workspace is allocated here.
// *used_static receives 1 if a compile-time instantiation ran.
extern "C" int condfc_host_run(long long n_draws, long long n_series, long long spu, int n, int H, int m, int p, int r,
                               const double* T, long long T_bs, const double* Z, long long Z_bs, const double* R,
                               long long R_bs, const double* Hm, long long H_bs, const double* Q, long long Q_bs,
                               const double* c, long long c_bs, const double* d, long long d_bs, const double* mean,
                               const double* cov, const double* cond, long long cond_bs, const double* z_init,
                               const double* z_state, const double* z_obs, double* state_mean, double* state_cov,
                               double* obs_mean, double* obs_cov, double* states, double* obs, int* info,
                               int force_dyn, int* used_static) {
  cf::Args A;
  std::memset(&A, 0, sizeof(A));
  A.U = n_draws * n_series; A.n_series = n_series; A.spu = spu; A.S = A.U * spu;
  A.n = n; A.H = H; A.m = m; A.p = p; A.r = r;
  A.T = {T, T_bs, 0}; A.Z = {Z, Z_bs, 0}; A.R = {R, R_bs, 0}; A.Hm = {Hm, H_bs, 0}; A.Q = {Q, Q_bs, 0};
  A.c = {c, c_bs, 0}; A.d = {d, d_bs, 0};
  A.mean = mean; A.cov = cov; A.cond = cond; A.cond_bs = cond_bs;
  A.z_init = z_init; A.z_state = z_state; A.z_obs = z_obs;
  A.state_mean = state_mean; A.state_cov = state_cov; A.obs_mean = obs_mean; A.obs_cov = obs_cov;
  A.states = states; A.obs = obs; A.info = info;
  const long long lanes = ss::warps_of(A.S) * 32;
  std::vector<double> tape(A.U * H * cf::tape_stride(m, p)), fac(A.U * ss::fac_stride(m, p, r));
  std::vector<double> wscr(A.U * cf::wscr_stride(m, p)), uscr(std::max(H * lanes * p, 1LL));
  std::vector<double> rscr(std::max((H - 1) * lanes * m, 1LL));
  std::vector<int> ustat(A.U);
  A.tape = tape.data(); A.fac = fac.data(); A.wscr = wscr.data(); A.ustat = ustat.data();
  A.uscr = uscr.data(); A.rscr = rscr.data();
  auto run = [&](auto dd) {
    *used_static = decltype(dd)::STATIC ? 1 : 0;
    for (long long u = 0; u < A.U; ++u) cf::window_unit(dd, A, u);
    for (long long s = 0; s < A.S; ++s) cf::path_unit(dd, A, s);
  };
  if (force_dyn) {
    if (m > ss::SS_MAX || p > ss::SS_MAX || r > ss::SS_MAX) return 1;
    run(ss::Dyn{m, p, r});
    return 0;
  }
  return ss::with_instance(m, p, r, run) ? 0 : 1;
}
