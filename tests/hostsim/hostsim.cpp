// hostsim.cpp - TEST-ONLY host build of the device step programs in pymc_statespace_b200/csrc/kf_core.cuh, kf_pred.cuh
// and kf_p1.cuh, the DARE and the RTS smoother.  The container that builds this repo has no GPU, so the Kalman/adjoint
// math is debugged here against the oracle before it is run on a B200.  This file is NOT part of the product: the package
// never loads it, and it cannot be reached from any public API.  tests/hostsim/__init__.py builds it.
#include <algorithm>
#include <vector>

#include "kf_ctx.cuh"
#include "kf_dare.cuh"
#include "kf_p1.cuh"
#include "kf_pred.cuh"
#include "kf_run.cuh"
#include "kf_smooth.cuh"

using namespace kfb;

static int g_p1 = 0;    // k_endog = 1: 1: forward + adjoint of kf_p1.cuh, 2: generic forward + kf_p1.cuh adjoint
static int g_pred = 0;  // 1: run the one-step-predictor programs (kf_pred.cuh) where they exist

// g_pred: the kernels' programs (kf_run.cuh: run_unit); otherwise the two-stage programs, the reference the
// one-step-predictor form is checked against.
template <int MK, class X>
static void run_adjoint(X& x, const KfArgs& A) {
  if (g_pred) run_unit<MK, 2>(x, A, 0);
  else backward_unit<MK>(x, A, 0);
}

// With per-step outputs requested the forward pass is the kernels' full-output one, `full`.
template <int MK, class X, class Full>
static void run_both(X& x, KfArgs& A, int do_bwd, Full&& full) {
  if (kernel_mode(A, false) == 1) full();
  else if (g_pred) run_unit<MK, 0>(x, A, 0);
  else forward_unit<MK, false>(x, A, 0);
  if (do_bwd) run_adjoint<MK>(x, A);
}

// The k_endog = 1 kernels' instantiation choice (kf_p1.cuh: with_forward_variant / with_adjoint_variant), with the tape
// in the kernels' layout for one unit and read back directly instead of through the TMA ring.
template <int M>
static void run_p1(KfArgs& A, int do_bwd) {
  if (g_p1 == 2) {  // generic forward (full tape entries) + specialised adjoint
    ThreadCtx<M, 1> x{nullptr, nullptr, 0, 1};
    forward_unit_pred<MK_STD>(x, A, 0);
    A.struct_flags &= ~KF_STRUCT_COMPRESSED;
  } else {
    p1::with_forward_variant(A, [&](auto v) {
      using V = decltype(v);
      p1::forward_unit_p1<M, true, V::ZU, V::H0>(A, 0, true, A.y.p, A.tape, (long long)p1::tape_doubles<M, V::ZU> * 32);
    });
  }
  if (!do_bwd) return;
  p1::with_adjoint_variant(A, [&](auto v) {
    using V = decltype(v);
    constexpr int KT = p1::tape_doubles<M, V::ZU>;
    using Tape = p1::DirectTape<M, KT>;
    Tape tape{A.tape + (long long)(A.n - 2) * KT * 32, (long long)KT * 32, 32};
    p1::backward_unit_p1<M, V::NEED_Z, V::NEED_H, V::HAS_GOBS, Tape, V::ZU, V::H0, V::CD>(A, 0, true, A.y.p, tape);
  });
}

// run-time dims: the generic kernels' full-output forward is run_unit<MK, 1>
template <int MK>
static void run_coop(CoopCtx& x, KfArgs& A) {
  run_both<MK>(x, A, 0, [&] { run_unit<MK, 1>(x, A, 0); });
}

// kind, flags: the C ABI's filter kind and KFB_FLAG_* bits, applied by the library's rules (kf_run.cuh).  The other
// choices exist for the tests only: static_dims, the thread-per-unit instantiations (else the run-time-dims context);
// pred, the one-step-predictor programs (else the two-stage reference programs); p1, the k_endog = 1 kernels (g_p1).
extern "C" int hostsim_run(int kind, unsigned flags, int m, int p, int n, const double* y, const double* a0,
                           const double* P0, const double* T, const double* Z, const double* H, const double* C,
                           const double* c, const double* d, const double* Pss, const double* Gss,
                           const long long* ts /*T,Z,H,C,c,d*/, int static_dims, int pred, int p1, double* loglik,
                           double* ll_obs, double* fs, double* ps, double* fc, double* pc, int* info, int do_bwd,
                           const double* g_loglik, const double* g_ll_obs, double* ga0, double* gP0, double* gT,
                           double* gZ, double* gH, double* gC, double* gc, double* gd, double* gPss, double* gGss) {
  KfArgs A;
  std::memset(&A, 0, sizeof(A));
  if (!filter_rule(kind, p, flags, &A.math_kind, &A.ll_const, &A.d_sign)) return 1;
  const int mk = A.math_kind;
  A.U = 1; A.n_series = 1; A.n = n; A.m = m; A.p = p;
  A.y = {y, 0, 0}; A.a0 = {a0, 0, 0}; A.P0 = {P0, 0, 0};
  A.T = {T, 0, ts[0]}; A.Z = {Z, 0, ts[1]}; A.H = {H, 0, ts[2]}; A.C = {C, 0, ts[3]};
  A.c = {c, 0, ts[4]}; A.d = {d, 0, ts[5]};
  A.Pss = {Pss, 0, 0}; A.Gss = {Gss, 0, 0};
  A.loglik = loglik; A.ll_obs = ll_obs; A.fs = fs; A.ps = ps; A.fc = fc; A.pc = pc; A.info = info;
  A.struct_flags = struct_flags_of(flags, p, ts[1] || ts[2], p1 != 0);
  // either tape format (g_p1 == 2 writes full entries under the compressed flag), in whole warps of units
  const long long entries =
      std::max((long long)std::max(n - 1, 1) * tape_width(m), ctape_steps_padded(n) * ctape_entry_doubles(m));
  std::vector<double> tape((size_t)entries * 32);
  A.tape = tape.data();
  A.g_loglik = g_loglik; A.g_ll_obs = g_ll_obs;
  A.ga0 = ga0; A.gP0 = gP0; A.gT = gT; A.gZ = gZ; A.gH = gH; A.gC = gC; A.gc = gc; A.gd = gd;
  A.gPss = gPss; A.gGss = gGss;

  g_pred = pred;
  g_p1 = p1;
  if (g_p1) {
    if (p != 1 || mk != MK_STD || ts[0] || ts[1] || ts[2] || ts[3] || ts[4] || ts[5]) return 7;
    if ((A.struct_flags & p1::REDUCED_FLAGS) == p1::REDUCED_FLAGS && (gZ || gH)) return 7;  // the C ABI refuses it too
#define KFB_P1CASE(MM)   \
  if (m == MM) {         \
    run_p1<MM>(A, do_bwd); \
    return 0;            \
  }
    KFB_P1CASE(1) KFB_P1CASE(2) KFB_P1CASE(3) KFB_P1CASE(4)
#undef KFB_P1CASE
    return 2;
  }
  const bool tv_any = ts[0] || ts[1] || ts[2] || ts[3] || ts[4] || ts[5];
  if (static_dims) {  // the thread-per-unit kernels' instantiations
    const bool ok = with_thread_instance(m, p, mk, tv_any, [&](auto v) {
      using V = decltype(v);
      ThreadCtx<V::M, V::P, V::TV> x{nullptr, nullptr, 0, 1};
      run_both<V::MK>(x, A, do_bwd, [&] { run_unit_full<V::M, V::P, V::MK, V::TV>(x, A, 0); });
    });
    return ok ? 0 : 2;
  }
  const int cap = coop_arena_doubles(m, p, true) + coop_arena_doubles(m, p, false);
  std::vector<double> arena((size_t)cap);
  CoopCtx x;
  x.init(m, p, arena.data(), cap, 0, 1);
  if (mk == MK_STD) run_coop<MK_STD>(x, A);
  else if (mk == MK_UNIV) run_coop<MK_UNIV>(x, A);
  else if (mk == MK_STEADY) run_coop<MK_STEADY>(x, A);
  else if (mk == MK_CHOLS) run_coop<MK_CHOLS>(x, A);
  const int fwd_used = x.off;
  if (fwd_used > coop_arena_doubles(m, p, false)) return 3;
  if (do_bwd) {
    x.off = 0;  // the adjoint re-uses the arena; the tape written by the forward pass lives in A.tape
    KfArgs B = A;
    B.loglik = nullptr; B.ll_obs = nullptr; B.fs = B.ps = B.fc = B.pc = nullptr; B.info = nullptr;
    if (mk == MK_STD) run_adjoint<MK_STD>(x, B);
    else if (mk == MK_UNIV) run_adjoint<MK_UNIV>(x, B);
    else if (mk == MK_CHOLS) run_adjoint<MK_CHOLS>(x, B);
    else run_adjoint<MK_STEADY>(x, B);
    if (x.off > coop_arena_doubles(m, p, true)) return 4;
  }
  return x.overflow ? 5 : 0;
}

extern "C" int hostsim_dare(int m, int p, const double* T, const double* Z, const double* H, const double* C, double* Pss,
                            double* Gss, int do_bwd, const double* gPss, const double* gGss, double* gT, double* gZ,
                            double* gH, double* gC) {
  const int cap = dare_arena_doubles(m, p);
  std::vector<double> arena((size_t)cap);
  CoopCtx x;
  x.init(m, p, arena.data(), cap, 0, 1);
  x.red = x.bump(34);
  int info = dare_unit(x, T, Z, H, C, Pss, Gss);
  if (x.overflow) return 5;
  if (do_bwd && info == 0) {
    x.off = 34;
    dare_adjoint_unit(x, T, Z, H, Pss, Gss, gPss, gGss, gT, gZ, gH, gC);
    if (x.overflow) return 6;
  }
  return info;
}

extern "C" int hostsim_smoother(int n, int m, const double* T, const double* C, const double* fs, const double* fc, double* ss,
                                double* sc) {
  SmoothArgs S;
  S.U = 1; S.n_series = 1; S.n = n; S.m = m;
  S.T = {T, 0, 0}; S.C = {C, 0, 0}; S.fs = fs; S.fc = fc; S.ss = ss; S.sc = sc;
  const int cap = smoother_arena_doubles(m);
  std::vector<double> arena((size_t)cap);
  CoopCtx x;
  x.init(m, 1, arena.data(), cap, 0, 1);
  x.red = x.bump(34);
  smoother_unit(x, S, 0);
  return x.overflow ? 5 : 0;
}
