// kf_run.cuh - which per-unit program the generic kernels run for a request: the MODE rule, its compile-time dispatch and
// the per-unit entry points.  Shared by the kernels (kf_kernels.cuh), their launchers and the host build of the kernels
// (tests/hostsim).
#pragma once
#include "kf_pred.cuh"
#include "kf_p1.cuh"

namespace kfb {

// Any per-step output requested: per-step log-likelihood, filtered or predicted moments.
KFB_HD bool wants_step_outputs(const KfArgs& A) { return A.ll_obs || A.fs || A.ps || A.fc || A.pc; }

// MODE: 0 = forward, loglik (+tape) only; 1 = forward with per-step outputs; 2 = adjoint.
KFB_HD int kernel_mode(const KfArgs& A, bool bwd) { return bwd ? 2 : wants_step_outputs(A) ? 1 : 0; }

template <int MODE_>
struct ModeTag {
  static constexpr int MODE = MODE_;
};

// run(ModeTag<MODE>{}) for the run-time MODE, so that a launcher names its kernel once.
template <class Run>
auto with_mode(int mode, Run&& run) {
  if (mode == 2) return run(ModeTag<2>{});
  if (mode == 1) return run(ModeTag<1>{});
  return run(ModeTag<0>{});
}

// The hot path (MODE 0 / 2 of the standard-family and steady-state filters) runs in one-step-predictor form.
template <int MK, int MODE, class X>
KFB_HD void run_unit(X& x, const KfArgs& A, long long u) {
  constexpr bool PRED = (MK == MK_STD || MK == MK_STEADY);
  if (MODE == 2) {
    if (PRED) backward_unit_pred<MK>(x, A, u);
    else backward_unit<MK>(x, A, u);
  } else if (MODE == 0 && PRED) {
    forward_unit_pred<MK>(x, A, u);
  } else {
    forward_unit<MK, MODE == 1>(x, A, u);
  }
}

// full-output forward of the thread-per-unit kernels: one observed series + standard-family filter + static matrices run
// the step written for that case (kf_p1.cuh: forward_full_p1), everything else the generic two-stage program
template <int M, int P, int MK, bool TV, class X>
KFB_HD void run_unit_full(X& x, const KfArgs& A, long long u) {
  if constexpr (P == 1 && MK == MK_STD && !TV) {
    if (A.struct_flags & KF_STRUCT_COMPRESSED) p1::forward_full_p1<M, true>(x, A, u);
    else p1::forward_full_p1<M, false>(x, A, u);
  } else {
    run_unit<MK, 1>(x, A, u);
  }
}

}  // namespace kfb
