// TEST-ONLY: the per-draw sampling calls of csrc/ run on the host: the simulation smoother (kf_simsmooth.cuh), the
// forecast paths and impulse responses (kf_forecast.cuh) and the conditional forecasts (kf_condfc.cuh).  Each entry
// point takes the C ABI's arguments, sizes one workspace from the plan of kf_draws_run.cuh, builds the kernels'
// arguments with its builders and runs the per-unit and per-simulation functions the kernels run, one at a time.
#include <cmath>
#include <cstring>
#include <vector>

#include "kf_draws_run.cuh"

using namespace kfb;

namespace {

// The plan's workspace, every double NaN: the device workspace is not initialised either.
std::vector<double> workspace(const draws::Regions& pl) { return std::vector<double>(pl.total / 8, std::nan("")); }

// run(dd) on the instantiation the kernels use for the request (ss::with_instance), or on the run-time dims when
// force_dyn is set; *used_static (if not null) receives 1 if a compile-time instantiation ran.  1 if nothing runs it.
template <class Run>
int on_instance(const kfb_desc* d, int force_dyn, int* used_static, Run&& run) {
  auto go = [&](auto dd) {
    if (used_static) *used_static = decltype(dd)::STATIC ? 1 : 0;
    run(dd);
  };
  if (force_dyn) {
    go(ss::Dyn{d->m, d->p, d->r});
    return 0;
  }
  return ss::with_instance(d->m, d->p, d->r, go) ? 0 : 1;
}

}  // namespace

// kfb_simulation_smoother
extern "C" int draws_host_simulation_smoother(const kfb_desc* d, const kfb_inputs* in, const double* pc,
                                              long long spu, const double* z_init, const double* z_state,
                                              const double* z_obs, double* states, int* info, int force_dyn,
                                              int* used_static) {
  draws::SsPlan pl;
  if (const kfb_status st = draws::plan_ss(d, spu, &pl)) return st;
  std::vector<double> ws = workspace(pl);
  const ss::Args A = draws::ss_args(d, in, pc, spu, z_init, z_state, z_obs, states, info, ws.data(), pl);
  const draws::Fill f = draws::ss_status_init(A);
  std::memset(f.p, f.value, f.bytes);
  return on_instance(d, force_dyn, used_static, [&](auto dd) {
    for (long long u = 0; u < A.U; ++u) {
      ss::unit_prep(A, u);
      for (int t = 0; t < A.n; ++t) ss::gain_entry(dd, A, u, t);
    }
    for (long long s = 0; s < A.S; ++s) ss::simulate_one(dd, A, s);
  });
}

// 1 if (m, p, r) has a compile-time instantiation
extern "C" int draws_host_is_static(int m, int p, int r) {
  bool st = false;
  ss::with_instance(m, p, r, [&](auto dd) { st = decltype(dd)::STATIC; });
  return st ? 1 : 0;
}

// kfb_forecast_paths
extern "C" int draws_host_forecast_paths(const kfb_desc* d, const kfb_inputs* in, const double* mean,
                                         const double* cov, int H, long long spu, const double* z_init,
                                         const double* z_state, const double* z_obs, double* states, double* obs,
                                         int* info, int force_dyn, int* used_static) {
  draws::FcPlan pl;
  if (const kfb_status st = draws::plan_fc(d, spu, &pl)) return st;
  std::vector<double> ws = workspace(pl);
  const fc::Args A = draws::fc_args(d, in, mean, cov, H, spu, z_init, z_state, z_obs, states, obs, info, ws.data(), pl);
  return on_instance(d, force_dyn, used_static, [&](auto dd) {
    for (long long u = 0; u < A.U; ++u) fc::unit_prep(A, u);
    for (long long s = 0; s < A.S; ++s) fc::path_one(dd, A, s);
  });
}

// kfb_impulse_response
extern "C" int draws_host_impulse_response(const kfb_desc* d, const kfb_inputs* in, int H, int shock, double* states,
                                           double* obs, int* info, int force_dyn, int* used_static) {
  if (const kfb_status st = draws::check_desc(d)) return st;
  const fc::IrfArgs A = draws::irf_args(d, in, H, shock, states, obs, info);
  return on_instance(d, force_dyn, used_static, [&](auto dd) {
    for (long long i = 0; i < A.nD * A.r; ++i) fc::irf_one(dd, A, i);
  });
}

// kfb_conditional_forecast
extern "C" int draws_host_conditional_forecast(const kfb_desc* d, const kfb_inputs* in, const double* mean,
                                               const double* cov, int H, const double* cond, long long cond_bs,
                                               long long spu, const double* z_init, const double* z_state,
                                               const double* z_obs, double* state_mean, double* state_cov,
                                               double* obs_mean, double* obs_cov, double* states, double* obs,
                                               int* info, int force_dyn, int* used_static) {
  draws::CfPlan pl;
  if (const kfb_status st = draws::plan_cf(d, H, spu, &pl)) return st;
  std::vector<double> ws = workspace(pl);
  const cf::Args A = draws::cf_args(d, in, mean, cov, H, cond, cond_bs, spu, z_init, z_state, z_obs, state_mean,
                                    state_cov, obs_mean, obs_cov, states, obs, info, ws.data(), pl);
  return on_instance(d, force_dyn, used_static, [&](auto dd) {
    for (long long u = 0; u < A.U; ++u) cf::window_unit(dd, A, u);
    for (long long s = 0; s < A.S; ++s) cf::path_unit(dd, A, s);
  });
}
