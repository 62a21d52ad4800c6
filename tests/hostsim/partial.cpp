// TEST-ONLY: the masked filter of csrc/ (kfb_masked_filter, kf_condfc.cuh) run on the host.  The entry point takes the
// C ABI's arguments, sizes one workspace from the plan of kf_draws_run.cuh, builds the kernel's arguments with its
// builder and runs the per-unit function the kernel runs, one unit at a time.  The simulation smoother with
// KFB_FLAG_PARTIAL_ROWS runs through draws.cpp's entry point, which passes desc->flags on.
#include <cmath>
#include <vector>

#include "kf_draws_run.cuh"

using namespace kfb;

// kfb_masked_filter; force_dyn runs the run-time dims, *used_static (if not null) receives 1 if a compile-time
// instantiation ran.  The workspace is NaN-filled: the device workspace is not initialised either.
extern "C" int partial_host_masked_filter(const kfb_desc* d, const kfb_inputs* in, double* predicted_states,
                                          double* predicted_covs, int* info, int force_dyn, int* used_static) {
  draws::MfPlan pl;
  if (const kfb_status st = draws::plan_mf(d, &pl)) return st;
  std::vector<double> ws(pl.total / 8, std::nan(""));
  const cf::FilterArgs A = draws::mf_args(d, in, predicted_states, predicted_covs, info, ws.data(), pl);
  auto run = [&](auto dd) {
    if (used_static) *used_static = decltype(dd)::STATIC ? 1 : 0;
    for (long long u = 0; u < A.U; ++u) cf::filter_unit(dd, A, u);
  };
  if (force_dyn) {
    run(ss::Dyn{d->m, d->p, d->r});
    return 0;
  }
  return ss::with_instance(d->m, d->p, d->r, run) ? 0 : 1;
}
