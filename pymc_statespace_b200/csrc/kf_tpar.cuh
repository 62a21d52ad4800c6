// kf_tpar.cuh - time-parallel form of the k_endog = 1 filter and its adjoint (KFB_FLAG_TIME_PARALLEL).
//
// The sequential kernels run all n steps of a unit in order on one thread / warp / CTA.  With few units (one NUTS draw
// per call) that leaves the GPU idle behind a chain of n dependent steps.  Here one CTA runs one unit and every scan
// over time is a blocked scan: each thread folds a contiguous chunk of steps, the CTA scans the chunk aggregates in
// shared memory, and each thread re-runs its chunk from its exclusive prefix.
//
// Forward.  Filtering elements (A, b, C, J, eta) of Saerkkae & Garcia-Fernandez, "Temporal parallelization of
// Bayesian smoothers", IEEE TAC 66(1), 2021, eqs. (10)-(13) with their combination operator; element t >= 1 couples
// the transition of step t-1 (T, c, C = R Q R^T) with the observation of step t (Z, H, d, y).  Element 0 is the literal
// update of kf_core.cuh from the caller's (a0, P0) - P0 may be non-symmetric - so its filtered moments are exactly the
// sequential filter's.  A missing row is a pure prediction element (A = T, b = c, C, J = 0, eta = 0).  The scan gives the
// filtered moments of every step; the predicted moments a_{t+1} = T a_f + c, P_{t+1} = sym(T P_f T^T + C) go to a
// per-unit tape, and a parallel map then runs the literal update of every step on them (v_t, F_t, ll_t, outputs, info).
// An element is undefined when Z C Z^T + H = 0 at its step (the observation is noise-free given the previous state);
// such a unit is run by one thread of its CTA with the sequential recursion instead - same tape, same map.  The map also
// checks that every tape entry is one literal step from the entry before it (forward_map_step: TPAR_DRIFT_TOL); where
// the scan has lost accuracy (elements with an expanding transition, e.g. a non-invertible MA part) the unit is re-run
// the same way.
//
// Adjoint.  Given the predicted moments, the reverse recursion of the predictor form (kf_pred.cuh) is affine in the
// cotangents.  With L_t = T - Kp Z, w_t = v_t / F_t, lambda_t = g_loglik + g_ll_obs[t]:
//   abar_t = L_t^T abar_{t+1} + lambda_t w_t Z^T
//   Pbar_t = L_t^T sym(Pbar_{t+1}) L_t + S_t,  S_t = sym(w_t (T^T abar_{t+1}) Z) + Fbar_t Z^T Z,
//            Fbar_t = -lambda_t (1/F_t - w_t^2) / 2 - w_t (Kp . abar_{t+1})
// (the covariance part of the gain cotangent cancels: the Joseph form is stationary in the gain for symmetric P_t).
// abar never depends on Pbar, so two reverse scans - an affine one for abar, a congruence one for sym(Pbar) - give the
// adjoint state of every step, after which the parameter contributions of the steps are independent: a parallel map
// of the literal one-step adjoint (adjoint_step, the p = 1 instance of kf_pred.cuh's step) reduced in a fixed order.
// Step 0 runs that literal adjoint, so abar_0 and the full-matrix Pbar_0 (non-symmetric P0) are the sequential ones.
//
// Each phase of a pass is a function over one chunk [lo, hi) of one unit (filt_fold_chunk .. adjoint_chunk); the kernels
// of kf_tpar.cu add only the CTA scans, the fallback decisions and the reductions.  Everything here is KFB_HD so that
// the host build (tests/hostsim) runs the same chunk functions, with its own scans, and checks them against the oracle.
#pragma once
#include <climits>
#include <type_traits>

#include "kf_ctx.cuh"
#include "kf_pred.cuh"

namespace kfb {
namespace tpar {

template <int M>
using TX = ThreadCtx<M, 1, false>;

// Threads per CTA of the time-parallel kernels (filter and smoother): 256 while one thread's operands fit the register
// file; the filtering element of k_states 3 / 4 is 33 / 56 doubles, and the smoother's gain buffers and aggregates no
// longer fit either, so those run 128 threads (a few more steps per thread, one scan level less).
template <int M>
KFB_HD constexpr int tpar_threads() { return M <= 2 ? 256 : 128; }

// The one list of k_states of the time-parallel kernels (filter and smoother), for their launchers and the host build:
// run(std::integral_constant<int, M>{}) for M = m in 1..4; false for any other m.
template <class Run>
bool with_instance(int m, Run&& run) {
  switch (m) {
    case 1: run(std::integral_constant<int, 1>{}); return true;
    case 2: run(std::integral_constant<int, 2>{}); return true;
    case 3: run(std::integral_constant<int, 3>{}); return true;
    case 4: run(std::integral_constant<int, 4>{}); return true;
    default: return false;
  }
}

// The filters of the time-parallel form: k_endog = 1 and the standard-family update.
inline bool supported(int m, int p, int mk) { return p == 1 && mk == MK_STD && with_instance(m, [](auto) {}); }

// Steps [lo, hi) of chunk k of K over n steps: contiguous chunks of ceil(n / K) steps; the last ones may be short or empty.
struct Chunk {
  int lo, hi;
};
KFB_HD Chunk chunk_of(int k, int K, int n) {
  const int len = (n + K - 1) / K;
  const int lo = k * len < n ? k * len : n;
  return {lo, lo + len < n ? lo + len : n};
}

// one unit's inputs (k_endog = 1); time strides 0 = static
struct UnitView {
  const double *y, *a0, *P0, *T, *Z, *H, *C, *c, *d;
  long long T_ts, Z_ts, H_ts, C_ts, c_ts, d_ts;
  double ll_const, d_sign;
  int n;
};

KFB_HD UnitView unit_view(const KfArgs& A, long long u) {
  const long long draw = u / A.n_series, series = u - draw * A.n_series;
  UnitView v;
  v.y = A.y.p + series * A.y.bs;
  v.a0 = A.a0.p + draw * A.a0.bs;
  v.P0 = A.P0.p + draw * A.P0.bs;
  v.T = A.T.p + draw * A.T.bs;
  v.Z = A.Z.p + draw * A.Z.bs;
  v.H = A.H.p + draw * A.H.bs;
  v.C = A.C.p + draw * A.C.bs;
  v.c = A.c.p ? A.c.p + draw * A.c.bs : nullptr;
  v.d = A.d.p ? A.d.p + draw * A.d.bs : nullptr;
  v.T_ts = A.T.ts; v.Z_ts = A.Z.ts; v.H_ts = A.H.ts; v.C_ts = A.C.ts; v.c_ts = A.c.ts; v.d_ts = A.d.ts;
  v.ll_const = A.ll_const;
  v.d_sign = A.d_sign;
  v.n = A.n;
  return v;
}

// matrices of step t: prm (T, Z, H, d) and the transition's C, c
template <int M>
KFB_HD void load_step(const UnitView& v, int t, Params<TX<M>>& prm, RegBuf<M * M>& C, RegBuf<M>& c) {
#pragma unroll
  for (int i = 0; i < M * M; ++i) prm.T[i] = v.T[t * v.T_ts + i];
#pragma unroll
  for (int i = 0; i < M * M; ++i) C[i] = v.C[t * v.C_ts + i];
#pragma unroll
  for (int i = 0; i < M; ++i) prm.Z[i] = v.Z[t * v.Z_ts + i];
#pragma unroll
  for (int i = 0; i < M; ++i) c[i] = v.c ? v.c[t * v.c_ts + i] : 0.0;
  prm.H[0] = v.H[t * v.H_ts];
  prm.d[0] = v.d ? v.d[t * v.d_ts] : 0.0;
}

// ------------------------------------------------------------------------------------------------
// forward: filtering elements
// ------------------------------------------------------------------------------------------------
template <int M>
struct FiltElem {
  double A[M * M], b[M], C[M * M], J[M * M], eta[M];
};

template <int M>
KFB_HD void filt_identity(FiltElem<M>& e) {
#pragma unroll
  for (int i = 0; i < M * M; ++i) { e.A[i] = (i % (M + 1) == 0) ? 1.0 : 0.0; e.C[i] = 0.0; e.J[i] = 0.0; }
#pragma unroll
  for (int i = 0; i < M; ++i) { e.b[i] = 0.0; e.eta[i] = 0.0; }
}

// W <- W^-1 (Gauss-Jordan, partial pivoting; W = I + C J with C, J positive semi-definite is never singular)
template <int M>
KFB_HD void small_inverse(double* W) {
  double R[M * M];
#pragma unroll
  for (int i = 0; i < M * M; ++i) R[i] = (i % (M + 1) == 0) ? 1.0 : 0.0;
#pragma unroll
  for (int k = 0; k < M; ++k) {
    int pr = k;
    double best = fabs(W[k * M + k]);
#pragma unroll
    for (int i = k + 1; i < M; ++i)
      if (fabs(W[i * M + k]) > best) { best = fabs(W[i * M + k]); pr = i; }
    if (pr != k) {
#pragma unroll
      for (int j = 0; j < M; ++j) {
        double s = W[k * M + j]; W[k * M + j] = W[pr * M + j]; W[pr * M + j] = s;
        s = R[k * M + j]; R[k * M + j] = R[pr * M + j]; R[pr * M + j] = s;
      }
    }
    const double rp = 1.0 / W[k * M + k];
#pragma unroll
    for (int j = 0; j < M; ++j) { W[k * M + j] *= rp; R[k * M + j] *= rp; }
#pragma unroll
    for (int i = 0; i < M; ++i) {
      if (i == k) continue;
      const double f = W[i * M + k];
#pragma unroll
      for (int j = 0; j < M; ++j) {
        W[i * M + j] = kf_fma(-f, W[k * M + j], W[i * M + j]);
        R[i * M + j] = kf_fma(-f, R[k * M + j], R[i * M + j]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < M * M; ++i) W[i] = R[i];
}

// o = ei (earlier) (x) ej (later).  o must not alias ei / ej.
template <int M>
KFB_HD void filt_combine(const FiltElem<M>& ei, const FiltElem<M>& ej, FiltElem<M>& o) {
  double D[M * M], AD[M * M], AE[M * M], W[M * M], x[M];
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {  // D = (I + Ci Jj)^-1
      double s = (r == q) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(ei.C[r * M + k], ej.J[k * M + q], s);
      D[r * M + q] = s;
    }
  small_inverse<M>(D);
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double s = 0.0, e = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) {
        s = kf_fma(ej.A[r * M + k], D[k * M + q], s);   // Aj D
        e = kf_fma(ei.A[k * M + r], D[q * M + k], e);   // Ai^T D^T  ((I + Jj Ci)^-1 = D^T: Ci, Jj symmetric)
      }
      AD[r * M + q] = s;
      AE[r * M + q] = e;
    }
  // A = Aj D Ai ;  b = Aj D (bi + Ci eta_j) + bj
#pragma unroll
  for (int r = 0; r < M; ++r) {
    double s = ei.b[r];
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(ei.C[r * M + k], ej.eta[k], s);
    x[r] = s;
  }
#pragma unroll
  for (int r = 0; r < M; ++r) {
    double s = ej.b[r];
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(AD[r * M + k], x[k], s);
    o.b[r] = s;
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double a = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) a = kf_fma(AD[r * M + k], ei.A[k * M + q], a);
      o.A[r * M + q] = a;
    }
  }
  // C = sym(Aj D Ci Aj^T) + Cj
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(AD[r * M + k], ei.C[k * M + q], s);
      W[r * M + q] = s;
    }
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(W[r * M + k], ej.A[q * M + k], s);
      D[r * M + q] = s;  // D is free now
    }
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) o.C[r * M + q] = 0.5 * (D[r * M + q] + D[q * M + r]) + ej.C[r * M + q];
  // eta = Ai^T E (eta_j - Jj bi) + eta_i ;  J = sym(Ai^T E Jj Ai) + Ji
#pragma unroll
  for (int r = 0; r < M; ++r) {
    double s = ej.eta[r];
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(-ej.J[r * M + k], ei.b[k], s);
    x[r] = s;
  }
#pragma unroll
  for (int r = 0; r < M; ++r) {
    double s = ei.eta[r];
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(AE[r * M + k], x[k], s);
    o.eta[r] = s;
  }
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(AE[r * M + k], ej.J[k * M + q], s);
      W[r * M + q] = s;
    }
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(W[r * M + k], ei.A[k * M + q], s);
      D[r * M + q] = s;
    }
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) o.J[r * M + q] = 0.5 * (D[r * M + q] + D[q * M + r]) + ei.J[r * M + q];
}

// Element 0: the literal update of step 0 from (a0, P0) (kf_core.cuh update_observed, Joseph form).
template <int M>
KFB_HD void filt_element0(const UnitView& v, FiltElem<M>& e) {
  TX<M> x{nullptr, nullptr, 0, 1};
  Params<TX<M>> prm(x);
  RegBuf<M * M> C(x), P(x), Pf(x);
  RegBuf<M> c(x), a(x), af(x);
  load_step<M>(v, 0, prm, C, c);
#pragma unroll
  for (int i = 0; i < M; ++i) a[i] = v.a0[i];
#pragma unroll
  for (int i = 0; i < M * M; ++i) P[i] = v.P0[i];
  if (kf_isnan(v.y[0])) {
#pragma unroll
    for (int i = 0; i < M; ++i) af[i] = a[i];
#pragma unroll
    for (int i = 0; i < M * M; ++i) Pf[i] = P[i];
  } else {
    UpdTmp<TX<M>> tmp(x);
    update_observed<MK_STD>(x, prm, v.y, v.d_sign, a, P, tmp, af, Pf, (LogAcc*)nullptr, true);
  }
#pragma unroll
  for (int i = 0; i < M * M; ++i) {
    e.A[i] = 0.0;
    e.J[i] = 0.0;
    e.C[i] = 0.5 * (Pf[i] + Pf[(i % M) * M + i / M]);
  }
#pragma unroll
  for (int i = 0; i < M; ++i) { e.b[i] = af[i]; e.eta[i] = 0.0; }
}

// Element t >= 1: transition of step t-1, observation of step t.  Returns false if undefined (Z C Z^T + H not a positive
// finite number at an observed step).
template <int M>
KFB_HD bool filt_element(const UnitView& v, int t, FiltElem<M>& e) {
  const double* T = v.T + (t - 1) * v.T_ts;
  const double* Cp = v.C + (t - 1) * v.C_ts;
  double Q[M * M], c[M];
#pragma unroll
  for (int i = 0; i < M * M; ++i) Q[i] = 0.5 * (Cp[i] + Cp[(i % M) * M + i / M]);
#pragma unroll
  for (int i = 0; i < M; ++i) c[i] = v.c ? v.c[(t - 1) * v.c_ts + i] : 0.0;
  const double yt = v.y[t];
  if (kf_isnan(yt)) {
#pragma unroll
    for (int i = 0; i < M * M; ++i) { e.A[i] = T[i]; e.C[i] = Q[i]; e.J[i] = 0.0; }
#pragma unroll
    for (int i = 0; i < M; ++i) { e.b[i] = c[i]; e.eta[i] = 0.0; }
    return true;
  }
  const double* Z = v.Z + t * v.Z_ts;
  const double H = v.H[t * v.H_ts];
  const double dd = v.d ? v.d[t * v.d_ts] : 0.0;
  double qz[M], zT[M];
  double S = H, r = yt - v.d_sign * dd;
#pragma unroll
  for (int i = 0; i < M; ++i) {
    double s = 0.0, q = 0.0;
#pragma unroll
    for (int k = 0; k < M; ++k) {
      s = kf_fma(Q[i * M + k], Z[k], s);
      q = kf_fma(Z[k], T[k * M + i], q);
    }
    qz[i] = s;
    zT[i] = q;
  }
#pragma unroll
  for (int i = 0; i < M; ++i) {
    S = kf_fma(Z[i], qz[i], S);
    r = kf_fma(-Z[i], c[i], r);
  }
  const bool ok = (S > 0.0) && (S < 1.0e300);
  const double rS = 1.0 / S;
  double K[M];
#pragma unroll
  for (int i = 0; i < M; ++i) K[i] = qz[i] * rS;
#pragma unroll
  for (int i = 0; i < M; ++i) {
    e.b[i] = kf_fma(K[i], r, c[i]);
    e.eta[i] = zT[i] * (r * rS);
#pragma unroll
    for (int j = 0; j < M; ++j) {
      e.A[i * M + j] = kf_fma(-K[i], zT[j], T[i * M + j]);
      e.C[i * M + j] = kf_fma(-K[i] * S, K[j], Q[i * M + j]);
      e.J[i * M + j] = zT[i] * zT[j] * rS;
    }
  }
  return ok;
}

// filtered (af, Pf) of step t -> predicted moments of step t+1, written as tape entry t+1
template <int M>
KFB_HD void predict_to_tape(const UnitView& v, int t, const double* af, const double* Pf, double* entry) {
  const double* T = v.T + t * v.T_ts;
  const double* C = v.C + t * v.C_ts;
  double S1[M * M];
#pragma unroll
  for (int i = 0; i < M; ++i) {
    double s = v.c ? v.c[t * v.c_ts + i] : 0.0;
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(T[i * M + k], af[k], s);
    entry[i] = s;
  }
#pragma unroll
  for (int i = 0; i < M; ++i)
#pragma unroll
    for (int j = 0; j < M; ++j) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(T[i * M + k], Pf[k * M + j], s);
      S1[i * M + j] = s;
    }
  double S2[M * M];
#pragma unroll
  for (int i = 0; i < M; ++i)
#pragma unroll
    for (int j = 0; j < M; ++j) {
      double s = C[i * M + j];
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(S1[i * M + k], T[j * M + k], s);
      S2[i * M + j] = s;
    }
#pragma unroll
  for (int i = 0; i < M; ++i)
#pragma unroll
    for (int j = 0; j < M; ++j) entry[M + i * M + j] = 0.5 * (S2[i * M + j] + S2[j * M + i]);
}

// tape entry of step t: predicted a_t (M) then P_t (M x M, full); layout [u][t][k]
template <int M>
KFB_HD constexpr int tape_entry() { return M + M * M; }

// Sequential walk (units with an undefined element): the literal two-stage step of kf_core.cuh, tape entries 0..n-1.
template <int M>
KFB_HD void forward_sequential_tape(const UnitView& v, double* tape) {
  TX<M> x{nullptr, nullptr, 0, 1};
  Params<TX<M>> prm(x);
  RegBuf<M * M> C(x), P(x), Pf(x);
  RegBuf<M> c(x), a(x), af(x);
  UpdTmp<TX<M>> tmp(x);
#pragma unroll
  for (int i = 0; i < M; ++i) a[i] = v.a0[i];
#pragma unroll
  for (int i = 0; i < M * M; ++i) P[i] = v.P0[i];
  for (int t = 0; t < v.n; ++t) {
    double* e = tape + (long long)t * tape_entry<M>();
#pragma unroll
    for (int i = 0; i < M; ++i) e[i] = a[i];
#pragma unroll
    for (int i = 0; i < M * M; ++i) e[M + i] = P[i];
    load_step<M>(v, t, prm, C, c);
    if (kf_isnan(v.y[t])) {
#pragma unroll
      for (int i = 0; i < M; ++i) af[i] = a[i];
#pragma unroll
      for (int i = 0; i < M * M; ++i) Pf[i] = P[i];
    } else {
      update_observed<MK_STD>(x, prm, v.y + t, v.d_sign, a, P, tmp, af, Pf, (LogAcc*)nullptr, true);
    }
    predict(x, prm.T, C, c, af, Pf, a, P, tmp.S1, tmp.S2);
  }
}

// The aggregate e_lo (x) .. (x) e_{hi-1} of a chunk's filtering elements (the identity if the chunk is empty).  Returns
// false if one of them is undefined.
template <int M>
KFB_HD bool filt_fold_chunk(const UnitView& v, int lo, int hi, FiltElem<M>& agg) {
  FiltElem<M> e, tmp;
  filt_identity<M>(agg);
  bool undefined = false;
  for (int t = lo; t < hi; ++t) {
    if (t == 0) filt_element0<M>(v, e);
    else undefined |= !filt_element<M>(v, t, e);
    if (t == lo) agg = e;
    else { filt_combine<M>(agg, e, tmp); agg = tmp; }
  }
  return !undefined;
}

// Re-runs a chunk from `prefix`, the scanned aggregate of all steps before lo (unused if lo == 0): the filtered moments
// of every step, written to the tape as the predicted moments of the step after it.  Tape entry 0 is (a0, P0).
template <int M>
KFB_HD void filt_rerun_chunk(const UnitView& v, int lo, int hi, const FiltElem<M>* prefix, double* tape) {
  FiltElem<M> f, e, tmp;
  for (int t = lo; t < hi; ++t) {
    if (t == 0) {
      filt_element0<M>(v, f);
      for (int i = 0; i < M; ++i) tape[i] = v.a0[i];
      for (int i = 0; i < M * M; ++i) tape[M + i] = v.P0[i];
    } else {
      filt_element<M>(v, t, e);
      filt_combine<M>(t == lo ? *prefix : f, e, tmp);
      f = tmp;
    }
    if (t + 1 < v.n) predict_to_tape<M>(v, t, f.b, f.C, tape + (long long)(t + 1) * tape_entry<M>());
  }
}

// Per-step forward outputs from the tape entry of step t (the literal update of kf_core.cuh).  Returns ll_t; *bad is set
// if F_t is not a positive finite number.
struct FwdOut {
  double *ll_obs, *fs, *ps, *fc, *pc;  // this unit's rows (ps / pc: n + 1 rows), any may be null
};

// Largest relative difference the consistency check accepts between a tape entry of the scan and one literal step from
// the entry before it.  A healthy scan agrees to ~1e-14; the filtering elements lose that when their own transition is
// expanding (an MA coefficient |theta| > 1 makes A = (I - K Z) T grow like theta^k over a chunk while the filter itself
// stays stable), and the scan's moments then drift by 1e-8 .. 1e+10.
constexpr double TPAR_DRIFT_TOL = 1e-10;

// True if (a, P) differs from (a_ref, P_ref) by more than tol relative to the scale of (a, P): max|P| for P, and
// max(max|a|, sqrt max|P|) for a.  A NaN on either side counts as drift.
template <int M>
KFB_HD bool drifted(const double* a, const double* P, const double* a_ref, const double* P_ref, double tol) {
  double sP = 0.0, sa = 0.0;
#pragma unroll
  for (int i = 0; i < M * M; ++i) sP = fmax(sP, fabs(P[i]));
#pragma unroll
  for (int i = 0; i < M; ++i) sa = fmax(sa, fabs(a[i]));
  sa = fmax(sa, sqrt(sP));
  bool ok = true;  // a NaN on either side fails its comparison
#pragma unroll
  for (int i = 0; i < M * M; ++i) ok = ok && (fabs(P[i] - P_ref[i]) <= tol * sP);
#pragma unroll
  for (int i = 0; i < M; ++i) ok = ok && (fabs(a[i] - a_ref[i]) <= tol * sa);
  return !ok;
}

// *drift is set if `next` (tape entry t + 1; null: no check) is not one literal step from `entry` to within
// TPAR_DRIFT_TOL (relative to the predicted moments; a NaN counts as drift).
template <int M>
KFB_HD double forward_map_step(const UnitView& v, int t, const double* entry, const double* next, const FwdOut& o,
                               bool* bad, bool* drift) {
  TX<M> x{nullptr, nullptr, 0, 1};
  Params<TX<M>> prm(x);
  RegBuf<M * M> C(x), P(x), Pf(x);
  RegBuf<M> c(x), a(x), af(x);
  UpdTmp<TX<M>> tmp(x);
  load_step<M>(v, t, prm, C, c);
#pragma unroll
  for (int i = 0; i < M; ++i) a[i] = entry[i];
#pragma unroll
  for (int i = 0; i < M * M; ++i) P[i] = entry[M + i];
  double ll = 0.0;
  *bad = false;
  *drift = false;
  if (kf_isnan(v.y[t])) {
#pragma unroll
    for (int i = 0; i < M; ++i) af[i] = a[i];
#pragma unroll
    for (int i = 0; i < M * M; ++i) Pf[i] = P[i];
  } else {
    StepStat st = update_observed<MK_STD>(x, prm, v.y + t, v.d_sign, a, P, tmp, af, Pf, (LogAcc*)nullptr, true);
    *bad = !st.ok;
    ll = -0.5 * (v.ll_const + st.logdet + st.quad);
  }
  if (o.ll_obs) o.ll_obs[t] = ll;
  if (o.fs) for (int i = 0; i < M; ++i) o.fs[(long long)t * M + i] = af[i];
  if (o.fc) for (int i = 0; i < M * M; ++i) o.fc[(long long)t * M * M + i] = Pf[i];
  if (o.ps) for (int i = 0; i < M; ++i) o.ps[(long long)t * M + i] = a[i];
  if (o.pc) for (int i = 0; i < M * M; ++i) o.pc[(long long)t * M * M + i] = P[i];
  if (!next && !(t == v.n - 1 && (o.ps || o.pc))) return ll;
  predict(x, prm.T, C, c, af, Pf, a, P, tmp.S1, tmp.S2);
  if (next) *drift = drifted<M>(&a[0], &P[0], next, next + M, TPAR_DRIFT_TOL);
  if (t == v.n - 1) {
    if (o.ps) for (int i = 0; i < M; ++i) o.ps[(long long)(t + 1) * M + i] = a[i];
    if (o.pc) for (int i = 0; i < M * M; ++i) o.pc[(long long)(t + 1) * M * M + i] = P[i];
  }
  return ll;
}

// forward_map_step over a chunk in step order, with the check if `check`.  Returns true if a step drifted; *ll receives
// the chunk's sum of ll_t and *first_bad its first step with a bad F_t (INT_MAX: none).
template <int M>
KFB_HD bool forward_map_chunk(const UnitView& v, int lo, int hi, const double* tape, bool check, const FwdOut& o,
                              double* ll, int* first_bad) {
  constexpr int E = tape_entry<M>();
  double s = 0.0;
  int fb = INT_MAX;
  bool drift_any = false;
  for (int t = lo; t < hi; ++t) {
    bool bad, drift;
    const double* next = (check && t + 1 < v.n) ? tape + (long long)(t + 1) * E : nullptr;
    s += forward_map_step<M>(v, t, tape + (long long)t * E, next, o, &bad, &drift);
    if (bad && fb == INT_MAX) fb = t;
    drift_any |= drift;
  }
  *ll = s;
  *first_bad = fb;
  return drift_any;
}

// ------------------------------------------------------------------------------------------------
// adjoint: reverse affine (abar) and congruence (sym Pbar) elements
// ------------------------------------------------------------------------------------------------
template <int M>
struct AffElem {  // f(x) = Mt x + s   (Mt = L^T)
  double Mt[M * M], s[M];
};
template <int M>
struct CongElem {  // f(X) = L^T X L + S
  double L[M * M], S[M * M];
};

template <int M>
KFB_HD void aff_identity(AffElem<M>& e) {
#pragma unroll
  for (int i = 0; i < M * M; ++i) e.Mt[i] = (i % (M + 1) == 0) ? 1.0 : 0.0;
#pragma unroll
  for (int i = 0; i < M; ++i) e.s[i] = 0.0;
}
template <int M>
KFB_HD void cong_identity(CongElem<M>& e) {
#pragma unroll
  for (int i = 0; i < M * M; ++i) { e.L[i] = (i % (M + 1) == 0) ? 1.0 : 0.0; e.S[i] = 0.0; }
}

// o = fi o fj (fj applied first): (Mi Mj, Mi sj + si).  o must not alias fi / fj.
template <int M>
KFB_HD void aff_combine(const AffElem<M>& fi, const AffElem<M>& fj, AffElem<M>& o) {
#pragma unroll
  for (int r = 0; r < M; ++r) {
    double s = fi.s[r];
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(fi.Mt[r * M + k], fj.s[k], s);
    o.s[r] = s;
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double a = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) a = kf_fma(fi.Mt[r * M + k], fj.Mt[k * M + q], a);
      o.Mt[r * M + q] = a;
    }
  }
}

// o = fi o fj: (Lj Li, Li^T Sj Li + Si).  o must not alias fi / fj.
template <int M>
KFB_HD void cong_combine(const CongElem<M>& fi, const CongElem<M>& fj, CongElem<M>& o) {
  double W[M * M];
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double a = 0.0, w = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) {
        a = kf_fma(fj.L[r * M + k], fi.L[k * M + q], a);
        w = kf_fma(fj.S[r * M + k], fi.L[k * M + q], w);  // Sj Li
      }
      o.L[r * M + q] = a;
      W[r * M + q] = w;
    }
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q <= r; ++q) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(fi.L[k * M + r], W[k * M + q], s);
      o.S[r * M + q] = s + fi.S[r * M + q];
      o.S[q * M + r] = s + fi.S[q * M + r];
    }
}

// Everything of step t the adjoint reads that depends on the forward moments only (kf_pred.cuh pred_gain).
template <int M>
struct BwdStep {
  Params<TX<M>> prm;
  StepSet<TX<M>> S;
  double lb;  // lambda_t = g_loglik + g_ll_obs[t]
  KFB_HD explicit BwdStep(TX<M>& x) : prm(x), S(x), lb(0.0) {}
};

template <int M>
KFB_HD void bwd_load(TX<M>& x, const UnitView& v, int t, const double* entry, double gl, const double* gllo,
                     BwdStep<M>& B) {
  RegBuf<M * M> C(x);
  RegBuf<M> c(x);
  load_step<M>(v, t, B.prm, C, c);
#pragma unroll
  for (int i = 0; i < M; ++i) B.S.a[i] = entry[i];
#pragma unroll
  for (int i = 0; i < M * M; ++i) B.S.P[i] = entry[M + i];
  B.S.observed = !kf_isnan(v.y[t]);
  if (B.S.observed) {
    pred_gain<MK_STD>(x, B.prm, v.y + t, v.d_sign, B.S.a, B.S.P, B.S.g, (LogAcc*)nullptr, false);
  } else {
#pragma unroll
    for (int i = 0; i < M * M; ++i) B.S.g.Lm[i] = B.prm.T[i];
  }
  B.lb = gl + (gllo ? gllo[t] : 0.0);
}

template <int M>
KFB_HD void aff_element(const BwdStep<M>& B, AffElem<M>& e) {
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) e.Mt[r * M + q] = B.S.g.Lm[q * M + r];
  const double f = B.S.observed ? B.lb * B.S.g.w[0] : 0.0;
#pragma unroll
  for (int r = 0; r < M; ++r) e.s[r] = f * B.prm.Z[r];
}

// abar_t from abar_{t+1}
template <int M>
KFB_HD void aff_apply(const BwdStep<M>& B, const double* ab, double* out) {
  const double f = B.S.observed ? B.lb * B.S.g.w[0] : 0.0;
#pragma unroll
  for (int r = 0; r < M; ++r) {
    double s = f * B.prm.Z[r];
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(B.S.g.Lm[k * M + r], ab[k], s);
    out[r] = s;
  }
}

// congruence element of step t, given abar_{t+1}
template <int M>
KFB_HD void cong_element(const BwdStep<M>& B, const double* ab, CongElem<M>& e) {
#pragma unroll
  for (int i = 0; i < M * M; ++i) e.L[i] = B.S.g.Lm[i];
  if (!B.S.observed) {
#pragma unroll
    for (int i = 0; i < M * M; ++i) e.S[i] = 0.0;
    return;
  }
  const auto& g = B.S.g;
  const double w = g.w[0], Fi = g.Fi[0];
  double u[M], kpa = 0.0;
#pragma unroll
  for (int r = 0; r < M; ++r) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(B.prm.T[k * M + r], ab[k], s);
    u[r] = s;
    kpa = kf_fma(g.Kp[r], ab[r], kpa);
  }
  const double Fb = -0.5 * B.lb * (Fi - w * w) - w * kpa;
  const double* Z = &B.prm.Z[0];
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) e.S[r * M + q] = kf_fma(0.5 * w, u[r] * Z[q] + u[q] * Z[r], Fb * Z[r] * Z[q]);
}

// X_t = L^T X_{t+1} L + S_t  (in place on X)
template <int M>
KFB_HD void cong_apply(const CongElem<M>& e, double* X) {
  double W[M * M];
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(X[r * M + k], e.L[k * M + q], s);
      W[r * M + q] = s;
    }
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q <= r; ++q) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(e.L[k * M + r], W[k * M + q], s);
      X[r * M + q] = s + e.S[r * M + q];
      X[q * M + r] = s + e.S[q * M + r];
    }
}

// Parameter cotangents of one step (per-step values, not accumulated).
template <int M>
struct StepGrad {
  double T[M * M], C[M * M], c[M], Z[M], H, d;
};

// The literal one-step adjoint of kf_pred.cuh (backward_unit_pred's `adjoint`) for k_endog = 1, given the adjoint state
// after the step (ab = abar_{t+1}, Ps = sym(Pbar_{t+1})).  Writes the step's parameter cotangents to g and, if ab_prev /
// Pb_prev are given, the adjoint state before the step (abar_t, full-matrix Pbar_t).
template <int M>
KFB_HD void adjoint_step(const BwdStep<M>& B, double ds, const double* ab, const double* Ps, StepGrad<M>& g,
                         double* ab_prev, double* Pb_prev) {
  const auto& prm = B.prm;
  const auto& a = B.S.a;
  const auto& P = B.S.P;
  const auto& tmp = B.S.g;
  const double lb = B.lb;
  double S4[M * M], S1[M * M], Lb[M * M];
#pragma unroll
  for (int i = 0; i < M * M; ++i) {
    g.C[i] = Ps[i];
    S4[i] = P[i] + P[(i % M) * M + i / M];
  }
#pragma unroll
  for (int i = 0; i < M; ++i) g.c[i] = ab[i];
#pragma unroll
  for (int i = 0; i < M; ++i)
#pragma unroll
    for (int j = 0; j < M; ++j) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(tmp.Lm[i * M + k], S4[k * M + j], s);
      S1[i * M + j] = s;  // L (P + P^T)
    }
#pragma unroll
  for (int i = 0; i < M; ++i)
#pragma unroll
    for (int j = 0; j < M; ++j) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(Ps[i * M + k], S1[k * M + j], s);
      Lb[i * M + j] = s;  // Lb = Ps L (P + P^T)
    }
#pragma unroll
  for (int i = 0; i < M; ++i)
#pragma unroll
    for (int j = 0; j < M; ++j) g.T[i * M + j] = kf_fma(ab[i], a[j], Lb[i * M + j]);  // ab a^T + Lb
  double Mb[M], vb = 0.0;
  if (B.S.observed) {
    const double Fi = tmp.Fi[0], w = tmp.w[0], v = tmp.v[0];
    const double Q1 = 2.0 * prm.H[0];
    double PK[M], Kb[M];
#pragma unroll
    for (int i = 0; i < M; ++i) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(Ps[i * M + k], tmp.Kp[k], s);
      PK[i] = s;
    }
#pragma unroll
    for (int i = 0; i < M; ++i) {
      double s = kf_fma(ab[i], v, PK[i] * Q1);
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(-Lb[i * M + k], prm.Z[k], s);
      Kb[i] = s;
    }
    double Hb = 0.0, q1 = 0.0;
    vb = -lb * w;
#pragma unroll
    for (int k = 0; k < M; ++k) {
      Hb = kf_fma(tmp.Kp[k], PK[k], Hb);
      q1 = kf_fma(tmp.Kp[k], Kb[k], q1);
      vb = kf_fma(tmp.Kp[k], ab[k], vb);
    }
#pragma unroll
    for (int j = 0; j < M; ++j) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(-tmp.Kp[k], Lb[k * M + j], s);
      g.Z[j] = s;  // -Kp^T Lb
    }
    const double Fb = kf_fma(-q1, Fi, -0.5 * lb * (Fi - w * w));
    double TMb[M];
#pragma unroll
    for (int i = 0; i < M; ++i) TMb[i] = Kb[i] * Fi;
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
      for (int j = 0; j < M; ++j) g.T[i * M + j] = kf_fma(TMb[i], tmp.Mm[j], g.T[i * M + j]);
#pragma unroll
    for (int i = 0; i < M; ++i) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(prm.T[k * M + i], TMb[k], s);
      Mb[i] = kf_fma(prm.Z[i], Fb, s);
    }
#pragma unroll
    for (int j = 0; j < M; ++j) {
      double s = kf_fma(-vb, a[j], g.Z[j]);
      s = kf_fma(Fb, tmp.Mm[j], s);
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(Mb[k], P[k * M + j], s);
      g.Z[j] = s;
    }
    g.H = Hb + Fb;
    g.d = -ds * vb;
  } else {
#pragma unroll
    for (int j = 0; j < M; ++j) { g.Z[j] = 0.0; Mb[j] = 0.0; }
    g.H = 0.0;
    g.d = 0.0;
  }
  if (ab_prev) {
#pragma unroll
    for (int i = 0; i < M; ++i) {  // abar_t = T^T ab - Z^T vb
      double s = B.S.observed ? -prm.Z[i] * vb : 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(prm.T[k * M + i], ab[k], s);
      ab_prev[i] = s;
    }
  }
  if (Pb_prev) {  // Pbar_t = L^T Ps L + Mb Z
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
      for (int j = 0; j < M; ++j) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < M; ++k) s = kf_fma(Ps[i * M + k], tmp.Lm[k * M + j], s);
        S1[i * M + j] = s;
      }
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
      for (int j = 0; j < M; ++j) {
        double s = Mb[i] * prm.Z[j];
#pragma unroll
        for (int k = 0; k < M; ++k) s = kf_fma(tmp.Lm[k * M + i], S1[k * M + j], s);
        Pb_prev[i * M + j] = s;
      }
  }
}

// The aggregate f_lo o .. o f_{hi-1} of a chunk's abar elements, folded from hi-1 down (the identity if it is empty).
template <int M>
KFB_HD void aff_fold_chunk(const UnitView& v, int lo, int hi, const double* tape, double gl, const double* gllo,
                           AffElem<M>& agg) {
  TX<M> x{nullptr, nullptr, 0, 1};
  BwdStep<M> B(x);
  AffElem<M> e, tmp;
  aff_identity<M>(agg);
  for (int t = hi - 1; t >= lo; --t) {
    bwd_load<M>(x, v, t, tape + (long long)t * tape_entry<M>(), gl, gllo, B);
    aff_element<M>(B, e);
    if (t == hi - 1) agg = e;
    else { aff_combine<M>(e, agg, tmp); agg = tmp; }
  }
}

// The aggregate of a chunk's congruence elements for sym(Pbar).  Their forcing needs abar_{t+1}, which is walked down
// from ab_hi (abar at hi).
template <int M>
KFB_HD void cong_fold_chunk(const UnitView& v, int lo, int hi, const double* tape, double gl, const double* gllo,
                            const double* ab_hi, CongElem<M>& agg) {
  TX<M> x{nullptr, nullptr, 0, 1};
  BwdStep<M> B(x);
  CongElem<M> e, tmp;
  double ab[M], abn[M];
  cong_identity<M>(agg);
  for (int i = 0; i < M; ++i) ab[i] = ab_hi[i];
  for (int t = hi - 1; t >= lo; --t) {
    bwd_load<M>(x, v, t, tape + (long long)t * tape_entry<M>(), gl, gllo, B);
    cong_element<M>(B, ab, e);
    aff_apply<M>(B, ab, abn);
    for (int i = 0; i < M; ++i) ab[i] = abn[i];
    if (t == hi - 1) agg = e;
    else { cong_combine<M>(e, agg, tmp); agg = tmp; }
  }
}

// One unit's parameter cotangents, any may be null: a0 [M], P0 [M, M], and T, C, c, Z, H, d with one row per step where
// that input is time-varying (its UnitView stride is not 0), one row where it is static.
struct GradOut {
  double *a0, *P0, *T, *C, *c, *Z, *H, *d;
};

// sums of the static inputs' cotangents, laid out T, C (M x M each), c, Z (M each), H, d
template <int M>
KFB_HD constexpr int static_grad_width() { return 2 * M * M + 2 * M + 2; }

// The literal one-step adjoint of every step of a chunk, from hi-1 down to lo, starting from abar = ab_hi and
// sym(Pbar) = X at hi (X is overwritten).  Time-varying inputs' cotangents are written per step; those of static inputs
// are summed in that step order into acc[static_grad_width<M>()].  Step 0 also writes the a0 / P0 cotangents.
template <int M>
KFB_HD void adjoint_chunk(const UnitView& v, int lo, int hi, const double* tape, double gl, const double* gllo,
                          const double* ab_hi, double* X, const GradOut& out, double* acc) {
  TX<M> x{nullptr, nullptr, 0, 1};
  BwdStep<M> B(x);
  StepGrad<M> g;
  CongElem<M> e;
  double ab[M], abn[M];
  for (int k = 0; k < static_grad_width<M>(); ++k) acc[k] = 0.0;
  for (int i = 0; i < M; ++i) ab[i] = ab_hi[i];
  for (int t = hi - 1; t >= lo; --t) {
    bwd_load<M>(x, v, t, tape + (long long)t * tape_entry<M>(), gl, gllo, B);
    if (t == 0) {
      adjoint_step<M>(B, v.d_sign, ab, X, g, out.a0, out.P0);  // abar_0, Pbar_0 are the a0 / P0 cotangents
    } else {
      adjoint_step<M>(B, v.d_sign, ab, X, g, nullptr, nullptr);
      cong_element<M>(B, ab, e);
      cong_apply<M>(e, X);
      aff_apply<M>(B, ab, abn);
      for (int i = 0; i < M; ++i) ab[i] = abn[i];
    }
    if (v.T_ts) { if (out.T) for (int i = 0; i < M * M; ++i) out.T[(long long)t * M * M + i] = g.T[i]; }
    else for (int i = 0; i < M * M; ++i) acc[i] += g.T[i];
    if (v.C_ts) { if (out.C) for (int i = 0; i < M * M; ++i) out.C[(long long)t * M * M + i] = g.C[i]; }
    else for (int i = 0; i < M * M; ++i) acc[M * M + i] += g.C[i];
    if (v.c_ts) { if (out.c) for (int i = 0; i < M; ++i) out.c[(long long)t * M + i] = g.c[i]; }
    else for (int i = 0; i < M; ++i) acc[2 * M * M + i] += g.c[i];
    if (v.Z_ts) { if (out.Z) for (int i = 0; i < M; ++i) out.Z[(long long)t * M + i] = g.Z[i]; }
    else for (int i = 0; i < M; ++i) acc[2 * M * M + M + i] += g.Z[i];
    if (v.H_ts) { if (out.H) out.H[t] = g.H; }
    else acc[2 * M * M + 2 * M] += g.H;
    if (v.d_ts) { if (out.d) out.d[t] = g.d; }
    else acc[2 * M * M + 2 * M + 1] += g.d;
  }
}

// Entry k of the unit's static cotangent sums (adjoint_chunk's acc layout) to its output, if that input is static.
template <int M>
KFB_HD void store_static_grad(const UnitView& v, const GradOut& out, int k, double s) {
  if (k < M * M) { if (out.T && !v.T_ts) out.T[k] = s; }
  else if (k < 2 * M * M) { if (out.C && !v.C_ts) out.C[k - M * M] = s; }
  else if (k < 2 * M * M + M) { if (out.c && !v.c_ts) out.c[k - 2 * M * M] = s; }
  else if (k < 2 * M * M + 2 * M) { if (out.Z && !v.Z_ts) out.Z[k - 2 * M * M - M] = s; }
  else if (k == 2 * M * M + 2 * M) { if (out.H && !v.H_ts) out.H[0] = s; }
  else { if (out.d && !v.d_ts) out.d[0] = s; }
}

}  // namespace tpar
}  // namespace kfb
