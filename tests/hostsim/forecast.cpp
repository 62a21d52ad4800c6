// TEST-ONLY: the forecast paths and impulse responses of csrc/kf_forecast.cuh run on the host: the same unit_prep,
// path_one and irf_one the kernels of kf_forecast.cu run, one unit, simulation or (draw, shock) at a time, chosen by the
// same ss::with_instance (or the run-time-dims path when force_dyn is set).
#include <cstring>
#include <vector>

#include "kf_forecast.cuh"

using namespace kfb;

// The arguments of kfb_forecast_paths for n_draws x n_series units; the workspace is allocated here.  *used_static
// receives 1 if a compile-time instantiation ran.
extern "C" int forecast_host_run(long long n_draws, long long n_series, long long spu, int H, int m, int p, int r,
                                 const double* T, long long T_bs, const double* Z, long long Z_bs, const double* R,
                                 long long R_bs, const double* Hm, long long H_bs, const double* Q, long long Q_bs,
                                 const double* c, long long c_bs, const double* d, long long d_bs, const double* mean,
                                 const double* cov, const double* z_init, const double* z_state, const double* z_obs,
                                 double* states, double* obs, int* info, int force_dyn, int* used_static) {
  fc::Args A;
  std::memset(&A, 0, sizeof(A));
  A.U = n_draws * n_series; A.n_series = n_series; A.spu = spu; A.S = A.U * spu;
  A.H = H; A.m = m; A.p = p; A.r = r;
  A.T = {T, T_bs, 0}; A.Z = {Z, Z_bs, 0}; A.R = {R, R_bs, 0}; A.Hm = {Hm, H_bs, 0}; A.Q = {Q, Q_bs, 0};
  A.c = {c, c_bs, 0}; A.d = {d, d_bs, 0};
  A.mean = mean; A.cov = cov; A.z_init = z_init; A.z_state = z_state; A.z_obs = z_obs;
  A.states = states; A.obs = obs; A.info = info;
  std::vector<double> fac(A.U * fc::fac_stride(m, p, r));
  std::vector<int> ustat(A.U);
  A.fac = fac.data(); A.ustat = ustat.data();
  auto run = [&](auto dd) {
    *used_static = decltype(dd)::STATIC ? 1 : 0;
    for (long long u = 0; u < A.U; ++u) fc::unit_prep(A, u);
    for (long long s = 0; s < A.S; ++s) fc::path_one(dd, A, s);
  };
  if (force_dyn) {
    if (m > ss::SS_MAX || p > ss::SS_MAX || r > ss::SS_MAX) return 1;
    run(ss::Dyn{m, p, r});
    return 0;
  }
  return ss::with_instance(m, p, r, run) ? 0 : 1;
}

// The arguments of kfb_impulse_response.
extern "C" int forecast_host_irf(long long n_draws, int H, int m, int p, int r, int shock, const double* T,
                                 long long T_bs, const double* Z, long long Z_bs, const double* R, long long R_bs,
                                 const double* Q, long long Q_bs, double* states, double* obs, int* info, int force_dyn,
                                 int* used_static) {
  fc::IrfArgs A;
  std::memset(&A, 0, sizeof(A));
  A.nD = n_draws; A.H = H; A.m = m; A.p = p; A.r = r; A.shock = shock;
  A.T = {T, T_bs, 0}; A.Z = {Z, Z_bs, 0}; A.R = {R, R_bs, 0}; A.Q = {Q, Q_bs, 0};
  A.states = states; A.obs = obs; A.info = info;
  auto run = [&](auto dd) {
    *used_static = decltype(dd)::STATIC ? 1 : 0;
    for (long long i = 0; i < A.nD * r; ++i) fc::irf_one(dd, A, i);
  };
  if (force_dyn) {
    if (m > ss::SS_MAX || p > ss::SS_MAX || r > ss::SS_MAX) return 1;
    run(ss::Dyn{m, p, r});
    return 0;
  }
  return ss::with_instance(m, p, r, run) ? 0 : 1;
}
