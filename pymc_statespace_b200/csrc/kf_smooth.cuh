// kf_smooth.cuh - Rauch-Tung-Striebel smoother (SURVEY.md section 8(f) row f2; NOT on the logp/grad path).
//
// Reference: KalmanSmoother.build_graph / smoother_step, pymc_statespace/filters/kalman_smoother.py:56-104:
//     a_hat = T a ; P_hat = T P T^T + R Q R^T            (no intercept, no symmetrisation, :99-104)
//     gain  = (pinv(P_hat) T P)^T                         (:92)
//     a_s   = a + gain (a_s' - a_hat) ;  P_s = P + gain (P_s' - P_hat) gain^T
// scanned backwards from the last filtered moment.  pinv(P_hat): when sym(P_hat) is numerically positive definite (every
// Cholesky pivot positive, smallest / largest > 1e-13) numpy's cutoff drops nothing and pinv(P_hat) = P_hat^-1, so the
// gain is obtained from a Cholesky solve (m syncs instead of thousands); otherwise - singular or nearly singular P_hat,
// where the cutoff decides the answer - from a cyclic-Jacobi eigendecomposition of sym(P_hat) with numpy's cutoff
// (eigenvalues below 1e-15 * largest are dropped), which is what numpy.linalg.pinv's SVD gives for a symmetric matrix.
// Round 2 timing before / after the fast path and the thread-per-unit instantiation for k_states <= 4: DESIGN.md section 8.
#pragma once
#include "kf_core.cuh"

namespace kfb {

struct SmoothArgs {
  long long U, n_series;
  int n, m;
  MatArg T, C;                 // C = R Q R^T (workspace), per draw
  const double *fs, *fc;       // [U, n, m], [U, n, m, m]
  double *ss, *sc;             // [U, n, m], [U, n, m, m]
};

// A (symmetric, destroyed: becomes diagonal) -> V (eigenvectors in columns).  All lanes cooperate on each rotation.
template <class X, class TM>
KFB_HD void jacobi_eigen(X& x, TM& Am, TM& V, int m) {
  KFB_FOR(idx, m * m) V[idx] = (x.div_m(idx) * (m + 1) == idx) ? 1.0 : 0.0;
  x.sync();
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, dia = 0.0;
    KFB_FOR(idx, m * m) {
      const int i = x.div_m(idx), j = idx - i * m;
      const double v = fabs(Am[idx]);
      if (i == j) dia = fmax(dia, v);
      else off = fmax(off, v);
    }
    off = x.reduce_max(off);
    dia = x.reduce_max(dia);
    if (!(off > 1.0e-17 * dia)) break;
    for (int p = 0; p < m - 1; ++p) {
      for (int q = p + 1; q < m; ++q) {
        const double apq = Am[p * m + q], app = Am[p * m + p], aqq = Am[q * m + q];
        x.sync();  // every lane has read the pivot block before anyone rotates it
        if (fabs(apq) <= 1.0e-300) continue;
        const double theta = (aqq - app) / (2.0 * apq);
        const double tt = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(tt * tt + 1.0), s = tt * c;
        KFB_FOR(k, m) {  // columns p, q of A and V
          const double akp = Am[k * m + p], akq = Am[k * m + q];
          Am[k * m + p] = c * akp - s * akq;
          Am[k * m + q] = s * akp + c * akq;
          const double vkp = V[k * m + p], vkq = V[k * m + q];
          V[k * m + p] = c * vkp - s * vkq;
          V[k * m + q] = s * vkp + c * vkq;
        }
        x.sync();
        KFB_FOR(k, m) {  // rows p, q of A
          const double apk = Am[p * m + k], aqk = Am[q * m + k];
          Am[p * m + k] = c * apk - s * aqk;
          Am[q * m + k] = s * apk + c * aqk;
        }
        x.sync();
      }
    }
  }
}

// In-place lower Cholesky factor of the symmetric W (all lanes of the unit cooperate).  True iff every pivot is a positive
// finite number and min pivot > 1e-13 * max pivot.
template <class X, class TM>
KFB_HD bool chol_factor(X& x, TM& W, int m) {
  double dmin = 1.0e300, dmax = 0.0;
  bool ok = true;
#pragma unroll
  for (int k = 0; k < m; ++k) {
    const double d = W[k * m + k];
    ok = ok && (d > 0.0) && (d < 1.0e300);
    dmin = fmin(dmin, d);
    dmax = fmax(dmax, d);
    const double r = sqrt(ok ? d : 1.0), ri = 1.0 / r;
    x.sync();  // every lane has read the pivot
    KFB_FOR(i, m) {
      if (i >= k) W[i * m + k] = (i == k) ? r : W[i * m + k] * ri;
    }
    x.sync();
    KFB_FOR(idx, m * m) {
      const int i = x.div_m(idx), j = idx - i * m;
      if (j > k && i >= j) W[idx] = kf_fma(-W[i * m + k], W[j * m + k], W[idx]);
    }
    x.sync();
  }
  return ok && dmin > 1.0e-13 * dmax;
}

// G = (L L^T)^-1 S, column by column (one column per lane: forward, then backward substitution)
template <class X, class TM>
KFB_HD void chol_solve(X& x, const TM& Lw, TM& G, const TM& S, int m) {
  KFB_FOR(j, m) {
#pragma unroll
    for (int i = 0; i < m; ++i) {
      double s = S[i * m + j];
#pragma unroll
      for (int k = 0; k < i; ++k) s = kf_fma(-Lw[i * m + k], G[k * m + j], s);
      G[i * m + j] = s / Lw[i * m + i];
    }
#pragma unroll
    for (int i = m - 1; i >= 0; --i) {
      double s = G[i * m + j];
#pragma unroll
      for (int k = i + 1; k < m; ++k) s = kf_fma(-Lw[k * m + i], G[k * m + j], s);
      G[i * m + j] = s / Lw[i * m + i];
    }
  }
  x.sync();
}

// The gain of one RTS step from the filtered (a, P) of step t: ah = T a, Ph = T P T^T + C and G = pinv(Ph) T P (the gain
// is G^T).  W, V, Pinv are scratch; S1 is left holding T P.  T and C may be buffers or pointers to memory.
template <class X, class TT, class TM, class TV>
KFB_HD void smoother_gain(X& x, const TT& T, const TT& C, const TV& a, const TM& P, TV& ah, TM& Ph, TM& G, TM& W, TM& V,
                          TM& Pinv, TM& S1) {
  const int m = x.m();
  KFB_FOR(i, m) {
    double s = 0.0;
    for (int k = 0; k < m; ++k) s = kf_fma(T[i * m + k], a[k], s);
    ah[i] = s;
  }
  gemm<false, false, 0>(x, S1, T, P, m, m, m);           // T P
  KFB_FOR(i, m * m) Ph[i] = C[i];
  x.sync();
  gemm<false, true, 1>(x, Ph, S1, T, m, m, m);           // P_hat = T P T^T + C
  KFB_FOR(idx, m * m) {
    const int i = x.div_m(idx), j = idx - i * m;
    W[idx] = 0.5 * (Ph[idx] + Ph[j * m + i]);
  }
  KFB_FOR(i, m * m) V[i] = W[i];
  x.sync();
  if (chol_factor(x, V, m)) {                            // sym(P_hat) positive definite: pinv = inverse
    chol_solve(x, V, G, S1, m);                          // G = P_hat^-1 T P ; gain = G^T
  } else {
    x.sync();
    jacobi_eigen(x, W, V, m);
    double lmax = 0.0;
    KFB_FOR(i, m) lmax = fmax(lmax, fabs(W[i * m + i]));
    lmax = x.reduce_max(lmax);
    const double cutoff = 1.0e-15 * lmax;
    KFB_FOR(idx, m * m) {                                // Pinv = V diag(1/lambda) V^T
      const int i = x.div_m(idx), j = idx - i * m;
      double s = 0.0;
      for (int k = 0; k < m; ++k) {
        const double lam = W[k * m + k];
        if (fabs(lam) > cutoff) s = kf_fma(V[i * m + k] / lam, V[j * m + k], s);
      }
      Pinv[idx] = s;
    }
    x.sync();
    gemm<false, false, 0>(x, G, Pinv, S1, m, m, m);      // G = pinv(P_hat) T P ; gain = G^T
  }
}

// The RTS update in place on (as, Ps), the smoothed moments of step t+1 on entry and of step t on return:
// a_s = a + G^T (a_s' - a_hat), P_s = P + G^T (P_s' - P_hat) G.  da, W, S1 are scratch.
template <class X, class TM, class TV>
KFB_HD void smoother_update(X& x, const TM& G, const TV& a, const TM& P, const TV& ah, const TM& Ph, TV& as, TM& Ps,
                            TV& da, TM& W, TM& S1) {
  const int m = x.m();
  KFB_FOR(i, m) da[i] = as[i] - ah[i];
  KFB_FOR(i, m * m) W[i] = Ps[i] - Ph[i];
  x.sync();
  KFB_FOR(i, m) {                                        // a_s = a + G^T (a_s' - a_hat)
    double s = a[i];
    for (int k = 0; k < m; ++k) s = kf_fma(G[k * m + i], da[k], s);
    as[i] = s;
  }
  gemm<true, false, 0>(x, S1, G, W, m, m, m);            // G^T (P_s' - P_hat)
  KFB_FOR(i, m * m) Ps[i] = P[i];
  x.sync();
  gemm<false, false, 1>(x, Ps, S1, G, m, m, m);          // P_s = P + G^T (.) G
}

template <class X>
KFB_HD void smoother_unit(X& x, const SmoothArgs& A, long long u) {
  const int m = x.m(), n = A.n;
  const long long draw = u / A.n_series;
  typename X::template Buf<SZ_MM> T(x), C(x), P(x), Ph(x), W(x), V(x), Pinv(x), G(x), Ps(x), S1(x);
  typename X::template Buf<SZ_M> a(x), ah(x), as(x), da(x);
  load_or_zero(x, T, A.T.p + draw * A.T.bs, m * m);
  load_or_zero(x, C, A.C.p + draw * A.C.bs, m * m);
  const double* fs = A.fs + u * (long long)n * m;
  const double* fc = A.fc + u * (long long)n * m * m;
  double* ss = A.ss + u * (long long)n * m;
  double* sc = A.sc + u * (long long)n * m * m;
  KFB_FOR(i, m) { as[i] = fs[(long long)(n - 1) * m + i]; ss[(long long)(n - 1) * m + i] = as[i]; }
  KFB_FOR(i, m * m) { Ps[i] = fc[(long long)(n - 1) * m * m + i]; sc[(long long)(n - 1) * m * m + i] = Ps[i]; }
  x.sync();
  for (int t = n - 2; t >= 0; --t) {
    KFB_FOR(i, m) a[i] = fs[(long long)t * m + i];
    KFB_FOR(i, m * m) P[i] = fc[(long long)t * m * m + i];
    x.sync();
    smoother_gain(x, T, C, a, P, ah, Ph, G, W, V, Pinv, S1);
    smoother_update(x, G, a, P, ah, Ph, as, Ps, da, W, S1);
    KFB_FOR(i, m) ss[(long long)t * m + i] = as[i];
    KFB_FOR(i, m * m) sc[(long long)t * m * m + i] = Ps[i];
    x.sync();
  }
}

inline int smoother_arena_doubles(int m) { return 10 * m * m + 4 * m + 40; }

}  // namespace kfb
