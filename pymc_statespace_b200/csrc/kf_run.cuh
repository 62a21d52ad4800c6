// kf_run.cuh - which per-unit program the generic kernels run for a request: the C ABI's filter kind and structure
// promises as kernel arguments, the MODE rule, its compile-time dispatch and the per-unit entry points.  Shared by the
// kernels (kf_kernels.cuh), their launchers, the C ABI (kf_api.cu) and the host build of the kernels (tests/hostsim).
#pragma once
#include "../../include/kfb200.h"
#include "kf_pred.cuh"
#include "kf_p1.cuh"

namespace kfb {

// The C ABI's filter kind and KFB_FLAG_CORRECTED as the math kind, the multiple of log(2 pi) per observed step and the
// sign of d (KfArgs::math_kind, ll_const, d_sign).  False for an unknown kind, or "single" with k_endog != 1.
inline bool filter_rule(int kind, int p, uint32_t flags, int* mk, double* ll_const, double* d_sign) {
  const bool corrected = (flags & KFB_FLAG_CORRECTED) != 0;
  const double l2pi = KF_LOG_2PI;
  switch (kind) {
    case KFB_STANDARD:
      *mk = MK_STD; *ll_const = corrected ? p * l2pi : l2pi; *d_sign = 1.0; return true;
    case KFB_SINGLE:
      if (p != 1) return false;  // assert_data_is_1d, kalman_filter.py:19,329
      *mk = MK_STD; *ll_const = l2pi; *d_sign = corrected ? 1.0 : -1.0; return true;
    case KFB_CHOLESKY:
      // as coded the filter is exact only for p = 1 (SURVEY A.2-Q4); p > 1 strict = bug-compatible MK_CHOLS
      *mk = (p != 1 && !corrected) ? MK_CHOLS : MK_STD; *ll_const = p * l2pi; *d_sign = 1.0; return true;
    case KFB_UNIVARIATE:
      *mk = MK_UNIV; *ll_const = 0.0; *d_sign = 1.0; return true;
    case KFB_STEADY_STATE:
      *mk = MK_STEADY; *ll_const = corrected ? p * l2pi : l2pi; *d_sign = corrected ? 1.0 : 0.0; return true;
    default: return false;
  }
}

// KfArgs::struct_flags from the C ABI's flags.  The promises Z = e0, H = 0 and companion T hold for k_endog = 1 with
// static Z and H only.  On the k_endog = 1 kernels (`p1_kernels`, decided by the caller), the three together with
// KFB_FLAG_NO_MISSING select the reduced recursion and its compressed tape.
inline int struct_flags_of(uint32_t flags, int p, bool zh_time_varying, bool p1_kernels) {
  int f = 0;
  if (p == 1 && !zh_time_varying)
    f = ((flags & KFB_FLAG_Z_UNIT0) ? KF_STRUCT_Z_UNIT0 : 0) | ((flags & KFB_FLAG_H_ZERO) ? KF_STRUCT_H_ZERO : 0) |
        ((flags & KFB_FLAG_T_COMPANION) ? KF_STRUCT_T_COMPANION : 0);
  constexpr uint32_t kPromises = KFB_FLAG_Z_UNIT0 | KFB_FLAG_H_ZERO | KFB_FLAG_T_COMPANION | KFB_FLAG_NO_MISSING;
  if (p1_kernels && (flags & kPromises) == kPromises) f |= KF_STRUCT_COMPRESSED;
  return f;
}

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
