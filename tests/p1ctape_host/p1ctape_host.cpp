// p1ctape_host.cpp - TEST-ONLY host build of the k_endog = 1 reduced ARMA kernels (kf_p1.cuh, ZU_REDUCED) for one unit,
// with the adjoint instantiation chosen by p1::with_adjoint_variant from the requested cotangents - including CD, which
// drops c-bar and d-bar when neither is requested.  Z = e0 and H = 0 are implied; the compressed tape is read through
// DirectTape as the host build of tests/hostsim does.  Not part of the product.
#include <vector>

#include "kf_p1.cuh"

using namespace kfb;

template <int M>
static void run(KfArgs& A) {
  p1::with_forward_variant(A, [&](auto v) {
    using V = decltype(v);
    p1::forward_unit_p1<M, true, V::ZU, V::H0>(A, 0, true, A.y.p, A.tape, 0);
  });
  p1::with_adjoint_variant(A, [&](auto v) {
    using V = decltype(v);
    using Tape = p1::DirectTape<M, p1::tape_doubles<M, V::ZU>>;
    Tape tape{nullptr, 0, 0};
    p1::backward_unit_p1<M, V::NEED_Z, V::NEED_H, V::HAS_GOBS, Tape, V::ZU, V::H0, V::CD>(A, 0, true, A.y.p, tape);
  });
}

// returns 0, or 2 for an unsupported m; gc / gd may be null (not requested)
extern "C" int p1ctape_run(int m, int n, const double* y, const double* a0, const double* P0, const double* T,
                           const double* C, const double* c, const double* d, double ll_const, const double* g_ll_obs,
                           double* loglik, int* info, double* ga0, double* gP0, double* gT, double* gC, double* gc,
                           double* gd) {
  std::vector<double> Z(m, 0.0), tape((size_t)ctape_steps_padded(n) * ctape_entry_doubles(m) * 32 + 1);
  Z[0] = 1.0;
  const double H = 0.0;
  KfArgs A;
  std::memset(&A, 0, sizeof(A));
  A.U = 1; A.n_series = 1; A.n = n; A.m = m; A.p = 1; A.math_kind = MK_STD;
  A.y = {y, 0, 0}; A.a0 = {a0, 0, 0}; A.P0 = {P0, 0, 0}; A.T = {T, 0, 0}; A.Z = {Z.data(), 0, 0}; A.H = {&H, 0, 0};
  A.C = {C, 0, 0}; A.c = {c, 0, 0}; A.d = {d, 0, 0};
  A.ll_const = ll_const; A.d_sign = 1.0;
  A.loglik = loglik; A.info = info;
  A.struct_flags = p1::REDUCED_FLAGS;
  A.tape = tape.data();
  A.g_ll_obs = g_ll_obs;
  A.ga0 = ga0; A.gP0 = gP0; A.gT = gT; A.gC = gC; A.gc = gc; A.gd = gd;
  switch (m) {
    case 1: run<1>(A); return 0;
    case 2: run<2>(A); return 0;
    case 3: run<3>(A); return 0;
    case 4: run<4>(A); return 0;
    default: return 2;
  }
}
