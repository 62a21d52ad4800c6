// kf_draws_run.cuh - the requests of the per-draw sampling calls (kfb_simulation_smoother, kfb_forecast_paths,
// kfb_conditional_forecast, kfb_impulse_response): validation of the descriptor, the workspace plans and the kernel
// arguments built from the C ABI's arguments.  Shared by the C ABI (kf_api.cu) and the host build of the kernels
// (tests/hostsim/draws.cpp), so that the CPU tests run the library's own argument fill and workspace layout.
#pragma once
#include <cstddef>
#include <cstring>

#include "../../include/kfb200.h"
#include "kf_condfc.cuh"
#include "kf_forecast.cuh"
#include "kf_simsmooth.cuh"

namespace kfb {
namespace draws {

static_assert(fc::SHOCK_UNIT == KFB_SHOCK_UNIT && fc::SHOCK_STD == KFB_SHOCK_STD &&
                  fc::SHOCK_CHOLESKY == KFB_SHOCK_CHOLESKY && ss::INFO_NOT_PSD == KFB_INFO_NOT_PSD,
              "kf_forecast.cuh / kf_simsmooth.cuh constants differ from include/kfb200.h");

// A static-matrix request: positive sizes (and `args_ok`, the call's own argument conditions, checked with them), no
// time-varying matrix, dims up to ss::SS_MAX.  filter_kind and flags are not read.
inline kfb_status check_desc(const kfb_desc* d, bool args_ok = true) {
  if (!d || d->n_draws <= 0 || d->n_series <= 0 || d->m <= 0 || d->p <= 0 || d->r <= 0 || !args_ok)
    return KFB_ERR_INVALID_ARG;
  if (d->T_ts || d->Z_ts || d->R_ts || d->H_ts || d->Q_ts || d->c_ts || d->d_ts) return KFB_ERR_UNSUPPORTED;
  if (d->m > ss::SS_MAX || d->p > ss::SS_MAX || d->r > ss::SS_MAX) return KFB_ERR_UNSUPPORTED;
  return KFB_OK;
}

// Workspace regions in order, each rounded up to 256 bytes (the rule kfb200.h states).
struct Regions {
  size_t total = 0;
  size_t take(size_t bytes) {
    const size_t o = total;
    total += (bytes + 255) / 256 * 256;
    return o;
  }
};

// kfb_simulation_smoother: gain tape, per-unit factors, the u and r scratch of every simulation, per-unit status.
struct SsPlan : Regions {
  size_t off_gain, off_fac, off_u, off_r, off_stat;
};

inline kfb_status plan_ss(const kfb_desc* d, int64_t sims_per_unit, SsPlan* pl) {
  const kfb_status st = check_desc(d, d && d->n > 0 && sims_per_unit > 0);
  if (st != KFB_OK) return st;
  if (d->n >= (1 << 29)) return KFB_ERR_UNSUPPORTED;
  const long long U = d->n_draws * d->n_series;
  const long long lanes = ss::warps_of(U * sims_per_unit) * 32;
  pl->off_gain = pl->take((size_t)U * d->n * ss::gain_stride(d->m, d->p) * 8);
  pl->off_fac = pl->take((size_t)U * ss::fac_stride(d->m, d->p, d->r) * 8);
  pl->off_u = pl->take((size_t)d->n * lanes * d->p * 8);
  pl->off_r = pl->take((size_t)(d->n - 1) * lanes * d->m * 8);
  pl->off_stat = pl->take((size_t)U * 4);
  return KFB_OK;
}

// kfb_forecast_paths: per-unit factors and status.
struct FcPlan : Regions {
  size_t off_fac, off_stat;
};

inline kfb_status plan_fc(const kfb_desc* d, int64_t sims_per_unit, FcPlan* pl) {
  const kfb_status st = check_desc(d);
  if (st != KFB_OK) return st;
  if (sims_per_unit <= 0) return KFB_ERR_INVALID_ARG;
  const long long U = d->n_draws * d->n_series;
  pl->off_fac = pl->take((size_t)U * fc::fac_stride(d->m, d->p, d->r) * 8);
  pl->off_stat = pl->take((size_t)U * 4);
  return KFB_OK;
}

// kfb_conditional_forecast: window tape, per-unit factors, run-time-dims scratch, per-unit status and the u and r
// scratch of the paths.
struct CfPlan : Regions {
  size_t off_tape, off_fac, off_wscr, off_stat, off_u, off_r;
};

inline kfb_status plan_cf(const kfb_desc* d, int32_t horizon, int64_t sims_per_unit, CfPlan* pl) {
  const kfb_status st = check_desc(d);
  if (st != KFB_OK) return st;
  if (horizon < 1 || sims_per_unit < 0 || d->n < 0) return KFB_ERR_INVALID_ARG;
  if (d->n >= (1 << 29) || horizon >= (1 << 29)) return KFB_ERR_UNSUPPORTED;
  const long long U = d->n_draws * d->n_series;
  const long long lanes = ss::warps_of(U * sims_per_unit) * 32;
  pl->off_tape = pl->take((size_t)U * horizon * cf::tape_stride(d->m, d->p) * 8);
  pl->off_fac = pl->take((size_t)U * ss::fac_stride(d->m, d->p, d->r) * 8);
  pl->off_wscr = pl->take((size_t)U * cf::wscr_stride(d->m, d->p) * 8);
  pl->off_stat = pl->take((size_t)U * 4);
  pl->off_u = pl->take((size_t)horizon * lanes * d->p * 8);
  pl->off_r = pl->take((size_t)(horizon - 1) * lanes * d->m * 8);
  return KFB_OK;
}

// The fields ss::Args, fc::Args and cf::Args share: unit and simulation counts, dims and the seven static matrices.
// obs_cov is the member that holds the observation covariance H (ss::Args::H, fc::Args::Hm, cf::Args::Hm).
template <class Args>
void fill_model(Args* A, MatArg Args::*obs_cov, const kfb_desc* d, const kfb_inputs* in, int64_t sims_per_unit) {
  std::memset(A, 0, sizeof(*A));
  A->U = d->n_draws * d->n_series; A->n_series = d->n_series; A->spu = sims_per_unit; A->S = A->U * sims_per_unit;
  A->m = d->m; A->p = d->p; A->r = d->r;
  A->T = {in->T, d->T_bs, 0}; A->Z = {in->Z, d->Z_bs, 0}; A->R = {in->R, d->R_bs, 0}; A->*obs_cov = {in->H, d->H_bs, 0};
  A->Q = {in->Q, d->Q_bs, 0}; A->c = {in->c, d->c_bs, 0}; A->d = {in->d, d->d_bs, 0};
}

// A region that must hold `bytes` copies of the byte `value` before the kernels run.
struct Fill {
  void* p;
  int value;
  size_t bytes;
};

inline ss::Args ss_args(const kfb_desc* d, const kfb_inputs* in, const double* predicted_covs, int64_t sims_per_unit,
                        const double* z_init, const double* z_state, const double* z_obs, double* states, int32_t* info,
                        void* workspace, const SsPlan& pl) {
  char* ws = (char*)workspace;
  ss::Args A;
  fill_model(&A, &ss::Args::H, d, in, sims_per_unit);
  A.n = d->n;
  A.y = {in->y, d->y_bs, 0}; A.a0 = {in->a0, d->a0_bs, 0}; A.P0 = {in->P0, d->P0_bs, 0};
  A.pc = predicted_covs; A.z_init = z_init; A.z_state = z_state; A.z_obs = z_obs; A.states = states; A.info = info;
  A.gain = (double*)(ws + pl.off_gain); A.fac = (double*)(ws + pl.off_fac);
  A.uscr = (double*)(ws + pl.off_u); A.rscr = (double*)(ws + pl.off_r); A.ustat = (int*)(ws + pl.off_stat);
  return A;
}

// The unit status of the simulation smoother starts at ss::KEY_NONE in every word.
inline Fill ss_status_init(const ss::Args& A) {
  static_assert(ss::KEY_NONE == 0x7f7f7f7f, "ss::KEY_NONE is the byte-wise fill 0x7f");
  return Fill{A.ustat, 0x7f, (size_t)A.U * 4};
}

inline fc::Args fc_args(const kfb_desc* d, const kfb_inputs* in, const double* start_mean, const double* start_cov,
                        int32_t horizon, int64_t sims_per_unit, const double* z_init, const double* z_state,
                        const double* z_obs, double* states, double* obs, int32_t* info, void* workspace,
                        const FcPlan& pl) {
  char* ws = (char*)workspace;
  fc::Args A;
  fill_model(&A, &fc::Args::Hm, d, in, sims_per_unit);
  A.H = horizon;
  A.mean = start_mean; A.cov = start_cov; A.z_init = z_init; A.z_state = z_state; A.z_obs = z_obs;
  A.states = states; A.obs = obs; A.info = info;
  A.vec = (uintptr_t)states % 16 == 0 && (uintptr_t)obs % 16 == 0;
  A.fac = (double*)(ws + pl.off_fac); A.ustat = (int*)(ws + pl.off_stat);
  return A;
}

// With sims_per_unit = 0 the normals and the path outputs are not used and stay null.
inline cf::Args cf_args(const kfb_desc* d, const kfb_inputs* in, const double* start_mean, const double* start_cov,
                        int32_t horizon, const double* cond, int64_t cond_bs, int64_t sims_per_unit,
                        const double* z_init, const double* z_state, const double* z_obs, double* state_mean,
                        double* state_cov, double* obs_mean, double* obs_cov, double* states, double* obs,
                        int32_t* info, void* workspace, const CfPlan& pl) {
  char* ws = (char*)workspace;
  cf::Args A;
  fill_model(&A, &cf::Args::Hm, d, in, sims_per_unit);
  A.n = d->n; A.H = horizon;
  A.mean = start_mean; A.cov = start_cov; A.cond = cond; A.cond_bs = cond_bs;
  A.state_mean = state_mean; A.state_cov = state_cov; A.obs_mean = obs_mean; A.obs_cov = obs_cov; A.info = info;
  if (sims_per_unit > 0) {
    A.z_init = z_init; A.z_state = z_state; A.z_obs = z_obs; A.states = states; A.obs = obs;
    A.vec = (uintptr_t)states % 16 == 0 && (uintptr_t)obs % 16 == 0;
  }
  A.tape = (double*)(ws + pl.off_tape); A.fac = (double*)(ws + pl.off_fac); A.wscr = (double*)(ws + pl.off_wscr);
  A.ustat = (int*)(ws + pl.off_stat); A.uscr = (double*)(ws + pl.off_u); A.rscr = (double*)(ws + pl.off_r);
  return A;
}

inline fc::IrfArgs irf_args(const kfb_desc* d, const kfb_inputs* in, int32_t horizon, int32_t shock, double* states,
                            double* obs, int32_t* info) {
  fc::IrfArgs A;
  std::memset(&A, 0, sizeof(A));
  A.nD = d->n_draws; A.H = horizon; A.m = d->m; A.p = d->p; A.r = d->r; A.shock = shock;
  A.T = {in->T, d->T_bs, 0}; A.Z = {in->Z, d->Z_bs, 0}; A.R = {in->R, d->R_bs, 0}; A.Q = {in->Q, d->Q_bs, 0};
  A.states = states; A.obs = obs; A.info = info;
  return A;
}

}  // namespace draws
}  // namespace kfb
