// kf_tpar_smooth.cuh - time-parallel form of the RTS smoother (kfb_smoother_ex with KFB_FLAG_TIME_PARALLEL).
//
// The RTS step of kf_smooth.cuh, with G_t = pinv(Ph_t) T P_t from the filtered moments (a_t, P_t) of step t, is
//   (as_t, Ps_t) = f_t(as_{t+1}, Ps_{t+1}),  f_t(x, X) = (E_t x + g_t, E_t X E_t^T + L_t),
//   E_t = G_t^T,  g_t = a_t - E_t ah_t,  L_t = P_t - E_t Ph_t E_t^T,
// an affine map of the smoothed mean and a congruence of the smoothed covariance whose elements depend on the filtered
// moments only (Saerkkae & Garcia-Fernandez, "Temporal parallelization of Bayesian smoothers", IEEE TAC 66(1), 2021,
// section IV).  The terminal element n-1 is (E = 0, g = a_{n-1}, L = P_{n-1}); a composite that contains it has E = 0 and
// its (g, L) are the smoothed moments.  L is a full matrix: filtered covariances need not be exactly symmetric, and the
// sequential smoother does not symmetrise either.
//
// One CTA runs one unit (kf_tpar_smooth.cu):
//  1. each thread folds its contiguous chunk [lo, hi) from hi-1 down to lo.  Folding f_t into an aggregate on its left
//     is f_t o (E, g, L) = (E_t E, f_t(g, L)), i.e. the literal RTS update on (g, L) - the chunk that holds step n-1
//     therefore folds to the sequential smoother's moments at its lo;
//  2. a suffix scan of the chunk aggregates (smooth_combine, full matrices);
//  3. each thread walks its chunk backwards with the literal RTS step from the scanned smoothed moments at hi, so inside
//     a chunk the values are the sequential ones from that start;
//  4. the walk's value at every chunk boundary lo > 0 is compared with the scanned value there (TPAR_DRIFT_TOL,
//     relative; NaN counts as drift).
//     A scan over products of gains has no accuracy guarantee, so on any drift the whole unit is re-run by the
//     sequential recursion (smoother_unit's steps) - this smoother never returns what the sequential one would not.
//
// Everything here is KFB_HD so that the host build of the kernels (tests/hostsim) runs the same fold and walk and checks
// them against the oracle.
#pragma once
#include "kf_smooth.cuh"
#include "kf_tpar.cuh"

namespace kfb {
namespace tpar {

template <int M>
struct SmoothElem {  // f(x, X) = (E x + g, E X E^T + L)
  double E[M * M], g[M], L[M * M];
};

template <int M>
KFB_HD void smooth_identity(SmoothElem<M>& e) {
#pragma unroll
  for (int i = 0; i < M * M; ++i) { e.E[i] = (i % (M + 1) == 0) ? 1.0 : 0.0; e.L[i] = 0.0; }
#pragma unroll
  for (int i = 0; i < M; ++i) e.g[i] = 0.0;
}

// o = fi o fj (fj applied first): (Ei Ej, Ei gj + gi, Ei Lj Ei^T + Li).  o must not alias fi / fj.
template <int M>
KFB_HD void smooth_combine(const SmoothElem<M>& fi, const SmoothElem<M>& fj, SmoothElem<M>& o) {
  double W[M * M];
#pragma unroll
  for (int r = 0; r < M; ++r) {
    double s = fi.g[r];
#pragma unroll
    for (int k = 0; k < M; ++k) s = kf_fma(fi.E[r * M + k], fj.g[k], s);
    o.g[r] = s;
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double a = 0.0, w = 0.0;
#pragma unroll
      for (int k = 0; k < M; ++k) {
        a = kf_fma(fi.E[r * M + k], fj.E[k * M + q], a);
        w = kf_fma(fj.L[r * M + k], fi.E[q * M + k], w);  // Lj Ei^T
      }
      o.E[r * M + q] = a;
      W[r * M + q] = w;
    }
  }
#pragma unroll
  for (int r = 0; r < M; ++r)
#pragma unroll
    for (int q = 0; q < M; ++q) {
      double s = fi.L[r * M + q];
#pragma unroll
      for (int k = 0; k < M; ++k) s = kf_fma(fi.E[r * M + k], W[k * M + q], s);
      o.L[r * M + q] = s;
    }
}

// One unit's view of SmoothArgs.
struct SmoothView {
  const double *T, *C, *fs, *fc;
  double *ss, *sc;
  int n;
};

KFB_HD SmoothView smooth_view(const SmoothArgs& A, long long u) {
  const long long draw = u / A.n_series;
  SmoothView v;
  v.T = A.T.p + draw * A.T.bs;
  v.C = A.C.p + draw * A.C.bs;
  v.fs = A.fs + u * (long long)A.n * A.m;
  v.fc = A.fc + u * (long long)A.n * A.m * A.m;
  v.ss = A.ss + u * (long long)A.n * A.m;
  v.sc = A.sc + u * (long long)A.n * A.m * A.m;
  v.n = A.n;
  return v;
}

// Runs the literal RTS steps t = hi-1 .. lo on (g, L) - the smoothed moments at hi on entry (ignored if hi == n: the walk
// then starts from the terminal element, the filtered moments of step n-1), at lo on return.  E (may be null) is
// multiplied by the gains on the left, E <- G_t^T E, as the fold of step 1 needs; ss / sc rows are written when `write`.
template <int M>
KFB_HD void smooth_run(const SmoothView& v, int lo, int hi, volatile double* E, double* g, double* L, bool write) {
  TX<M> x{nullptr, nullptr, 0, 1};
  RegBuf<M * M> P(x), Ph(x), W(x), V(x), Pinv(x), G(x), Ps(x), S1(x);
  RegBuf<M> a(x), ah(x), as(x), da(x);
  int t = hi - 1;
  if (hi == v.n) {
#pragma unroll
    for (int i = 0; i < M; ++i) as[i] = v.fs[(long long)t * M + i];
#pragma unroll
    for (int i = 0; i < M * M; ++i) Ps[i] = v.fc[(long long)t * M * M + i];
    if (E)
#pragma unroll
      for (int i = 0; i < M * M; ++i) E[i] = 0.0;
    if (write) {
      for (int i = 0; i < M; ++i) v.ss[(long long)t * M + i] = as[i];
      for (int i = 0; i < M * M; ++i) v.sc[(long long)t * M * M + i] = Ps[i];
    }
    --t;
  } else {
#pragma unroll
    for (int i = 0; i < M; ++i) as[i] = g[i];
#pragma unroll
    for (int i = 0; i < M * M; ++i) Ps[i] = L[i];
  }
  for (; t >= lo; --t) {
#if defined(__CUDA_ARCH__)
    // keep the compiler from hoisting the next step's loads over this one (that costs the fold, which stores nothing,
    // 22 doubles of spills at k_states 4)
    asm volatile("" ::: "memory");
#endif
#pragma unroll
    for (int i = 0; i < M; ++i) a[i] = v.fs[(long long)t * M + i];
#pragma unroll
    for (int i = 0; i < M * M; ++i) P[i] = v.fc[(long long)t * M * M + i];
    smoother_gain(x, v.T, v.C, a, P, ah, Ph, G, W, V, Pinv, S1);
    if (E) {  // E <- G^T E, one column at a time
#pragma unroll
      for (int q = 0; q < M; ++q) {
        double col[M];
#pragma unroll
        for (int k = 0; k < M; ++k) col[k] = E[k * M + q];
#pragma unroll
        for (int r = 0; r < M; ++r) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < M; ++k) s = kf_fma(G[k * M + r], col[k], s);
          E[r * M + q] = s;
        }
      }
    }
    smoother_update(x, G, a, P, ah, Ph, as, Ps, da, W, S1);
    if (write) {
      for (int i = 0; i < M; ++i) v.ss[(long long)t * M + i] = as[i];
      for (int i = 0; i < M * M; ++i) v.sc[(long long)t * M * M + i] = Ps[i];
    }
  }
#pragma unroll
  for (int i = 0; i < M; ++i) g[i] = as[i];
#pragma unroll
  for (int i = 0; i < M * M; ++i) L[i] = Ps[i];
}

// Step 1: the aggregate f_lo o .. o f_{hi-1} of a chunk (the identity if the chunk is empty).
template <int M>
KFB_HD void smooth_fold(const SmoothView& v, int lo, int hi, SmoothElem<M>& agg) {
  smooth_identity<M>(agg);
  if (lo < hi) smooth_run<M>(v, lo, hi, agg.E, agg.g, agg.L, false);
}

// Steps 3 and 4: walks a non-empty chunk from `next` (the scanned aggregate of the chunk after it; unused if hi == n),
// writes its smoothed moments, and returns true if the walk's value at lo differs from `own` (the scanned aggregate of
// this chunk, where the walk of the chunk before it starts) by more than tol relative to the walk's moments.  Step 0 is
// no chunk boundary: the scan's value there starts no walk and is not checked (under a diffuse start it carries the
// cancellation of P_0 - E_0 Ph_0 E_0^T at the scale of P_0).
template <int M>
KFB_HD bool smooth_walk_check(const SmoothView& v, int lo, int hi, const SmoothElem<M>* next, const SmoothElem<M>& own,
                              double tol) {
  if (lo >= hi) return false;
  double g[M], L[M * M];
  if (hi < v.n) {
#pragma unroll
    for (int i = 0; i < M; ++i) g[i] = next->g[i];
#pragma unroll
    for (int i = 0; i < M * M; ++i) L[i] = next->L[i];
  }
  smooth_run<M>(v, lo, hi, nullptr, g, L, true);
  const bool drift = drifted<M>(g, L, own.g, own.L, tol);  // outside the `lo > 0` branch: k_states 4 spills inside it
  return lo > 0 && drift;
}

// The sequential recursion for one unit on one thread (the drift fallback): the walk of the whole series from the
// terminal element, the same steps in the same order as smoother_unit.
template <int M>
KFB_HD void smooth_sequential(const SmoothView& v) {
  double g[M], L[M * M];
  smooth_run<M>(v, 0, v.n, nullptr, g, L, true);
}

}  // namespace tpar
}  // namespace kfb
