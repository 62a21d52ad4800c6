// kf_simsmooth.cuh - the simulation smoother (Durbin & Koopman 2002, mean correction, with the fast state smoother of
// Durbin & Koopman's book, section 4.6.2), written once as KFB_HD functions: kf_simsmooth.cu runs them as kernels and
// the host build of the kernels (tests/hostsim/draws.cpp, requests from kf_draws_run.cuh) runs them on the host.
//
// Model (the one the filters evaluate): x_0 ~ N(a0, P0); y_t = Z x_t + d + eps_t, eps_t ~ N(0, H), t = 0..n-1;
// x_{t+1} = T x_t + c + R eta_t, eta_t ~ N(0, Q), t = 0..n-2.  (kfb_simulate's shifted convention obs[t] = Z x_{t-1} is
// NOT the one used here.)  One simulation draws x~_0..x~_{n-1} from p(x | y, theta):
//   1. x+_0 = a0 + S_P0 z_init, x+_{t+1} = T x+_t + c + (R S_Q) z_state_t, y+_t = Z x+_t + d + S_H z_obs_t;
//   2. y* = y - y+, and with a*_0 = 0:  v_t = y*_t - Z a*_t,  u_t = F_t^-1 v_t,  a*_{t+1} = T a*_t + K_t v_t;
//   3. r_{n-1} = 0,  r_{t-1} = Z^T (u_t - K_t^T r_t) + T^T r_t      (= Z^T F_t^-1 v_t + L_t^T r_t, L_t = T - K_t Z);
//   4. xhat_0 = P0 r_{-1},  xhat_{t+1} = T xhat_t + C r_t,  C = R Q R^T;
//   5. x~_t = x+_t + xhat_t.
// S_A S_A^T = A is the PSD lower factor of psd_factor below.  K_t = T P_t Z^T F_t^-1 and F_t^-1 do not depend on y: the
// gain pass computes them once per (unit, t) from the filter's predicted covariances.  A missing row has K_t = 0 and
// u_t = 0 (L_t = T), as in the filter.  x+ is not stored: step 4 recomputes it from the normals with the same arithmetic.
#pragma once
#include "kf_core.cuh"

namespace kfb {
namespace ss {

constexpr int SS_MAX = 32;            // k_states / k_endog / k_posdef limit of the run-time-dims path
constexpr double PSD_RTOL = 1e-10;    // psd_factor: pivots within this fraction of the largest diagonal entry are zero
constexpr int KEY_NONE = 0x7f7f7f7f;  // unit status before any failure (a byte-wise memset value)
constexpr int KEY_FACTOR = -1;        // P0, Q or H not PSD; otherwise 2 t (F_t not PD) or 2 t + 1 (row t partly missing)
constexpr int INFO_NOT_PSD = 0x40000004;  // = KFB_INFO_NOT_PSD (include/kfb200.h)

// Compile-time k_states / k_endog (registers); k_posdef r <= M is a run-time value, and R S_Q is stored M x M with
// zero columns from r on, so the per-step products never loop over r.
template <int M, int P>
struct Static {
  static constexpr bool STATIC = true;
  static constexpr int m = M, p = P, MM = M, PM = P, RL = M;
  int r;
  KFB_HD int rl() const { return RL; }
};
// Run-time dims up to SS_MAX; matrices are read in place from global memory.
struct Dyn {
  static constexpr bool STATIC = false;
  static constexpr int MM = SS_MAX, PM = SS_MAX;
  int m, p, r;
  KFB_HD int rl() const { return r; }
};

struct Args {
  long long U, n_series, S, spu;  // units (draw * n_series + series), simulations, simulations per unit
  int n, m, p, r;
  MatArg y, a0, P0, T, Z, R, H, Q, c, d;  // batch strides only (static matrices)
  const double* pc;                        // predicted covariances [U][n + 1][m][m] of the standard filter (row 0 unread)
  const double *z_init, *z_state, *z_obs;  // [S][m], [n - 1][S][r], [n][S][p]
  double* states;                          // [S][n][m]
  int* info;                               // [U]
  double* gain;                            // [U][n][K_t (m p) | F_t^-1 (p p)]
  double* fac;                             // [U][S_P0 (m m) | R S_Q (m r) | S_H (p p) | C (m m) | S_Q (r r)]
  int* ustat;                              // [U] smallest failure key, KEY_NONE if none
  double *uscr, *rscr;                     // u_t [n][warp][p][32], r_t [n - 1][warp][m][32]
};

KFB_HD long long gain_stride(int m, int p) { return (long long)m * p + (long long)p * p; }
KFB_HD long long fac_stride(int m, int p, int r) {
  return 2LL * m * m + (long long)m * r + (long long)p * p + (long long)r * r;
}
KFB_HD long long warps_of(long long S) { return (S + 31) >> 5; }

KFB_HD void key_min(int* k, int v) {
#if defined(__CUDA_ARCH__)
  atomicMin(k, v);
#else
  if (v < *k) *k = v;
#endif
}

KFB_HD int info_of_key(int key) {
  if (key == KEY_NONE) return 0;
  if (key == KEY_FACTOR) return INFO_NOT_PSD;
  const int t = key >> 1;
  return (key & 1) ? -(t + 1) : t + 1;
}

// Lower factor L (row-major n x n) with L L^T = A for a positive SEMI-definite A: a pivot at or below PSD_RTOL times the
// largest diagonal entry is taken as zero and its column is zeroed; a pivot below -PSD_RTOL times it (or a NaN) makes
// the result false.  A = 0 gives L = 0.
KFB_HD bool psd_factor(const double* A, double* L, int n) {
  double dmax = 0.0;
  for (int i = 0; i < n; ++i)
    if (!(A[i * n + i] <= dmax)) dmax = A[i * n + i];
  const double tol = PSD_RTOL * dmax;
  bool ok = true;
  for (int j = 0; j < n; ++j) {
    double dj = A[j * n + j];
    for (int k = 0; k < j; ++k) dj -= L[j * n + k] * L[j * n + k];
    for (int i = 0; i < j; ++i) L[i * n + j] = 0.0;
    if (dj > tol) {
      const double lj = sqrt(dj);
      L[j * n + j] = lj;
      for (int i = j + 1; i < n; ++i) {
        double s = A[i * n + j];
        for (int k = 0; k < j; ++k) s -= L[i * n + k] * L[j * n + k];
        L[i * n + j] = s / lj;
      }
    } else {
      ok = ok && (dj >= -tol);
      for (int i = j; i < n; ++i) L[i * n + j] = 0.0;
    }
  }
  return ok;
}

// Per unit, once: the factors and C = R Q R^T into fac[u]; a non-PSD P0, Q or H sets KEY_FACTOR.
KFB_HD void unit_prep(const Args& A, long long u) {
  const long long dr = u / A.n_series;
  const int m = A.m, p = A.p, r = A.r;
  double* f = A.fac + u * fac_stride(m, p, r);
  double *SP0 = f, *G = f + m * m, *SH = G + m * r, *C = SH + p * p, *SQ = C + m * m;
  const double* P0 = A.P0.p + dr * A.P0.bs;
  const double* R = A.R.p + dr * A.R.bs;
  const double* Q = A.Q.p + dr * A.Q.bs;
  const double* H = A.H.p + dr * A.H.bs;
  bool ok = psd_factor(P0, SP0, m);
  ok = psd_factor(H, SH, p) && ok;
  ok = psd_factor(Q, SQ, r) && ok;
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < r; ++j) {
      double s = 0.0;
      for (int k = j; k < r; ++k) s = kf_fma(R[i * r + k], SQ[k * r + j], s);
      G[i * r + j] = s;
    }
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < m; ++j) {
      double s = 0.0;
      for (int k = 0; k < r; ++k) {
        double rq = 0.0;
        for (int l = 0; l < r; ++l) rq = kf_fma(R[i * r + l], Q[l * r + k], rq);
        s = kf_fma(rq, R[j * r + k], s);
      }
      C[i * m + j] = s;
    }
  if (!ok) key_min(A.ustat + u, KEY_FACTOR);
}

// Gain pass, one (unit, t): K_t = T P_t Z^T F_t^-1 and F_t^-1 with F_t = Z P_t Z^T + H, into gain[u][t]; zeros for a
// missing row.  A partly missing row or an F_t that is not positive definite sets its key.
template <class D>
KFB_HD void gain_entry(const D& d, const Args& A, long long u, int t) {
  const int m = d.m, p = d.p;
  const long long dr = u / A.n_series, se = u % A.n_series;
  double* K = A.gain + (u * A.n + t) * gain_stride(m, p);
  double* Fi = K + m * p;
  const double* y = A.y.p + se * A.y.bs + (long long)t * p;
  int nmiss = 0;
  for (int i = 0; i < p; ++i) nmiss += kf_isnan(y[i]) ? 1 : 0;
  bool ok = nmiss == 0;
  if (nmiss > 0 && nmiss < p) key_min(A.ustat + u, 2 * t + 1);
  double PZt[D::MM * D::PM], L[D::PM * D::PM], Li[D::PM * D::PM];
  if (ok) {
    // P_0 is the input P0: kfb_forward writes predicted_covs[u, 0] only together with predicted_states
    const double* P = t == 0 ? A.P0.p + dr * A.P0.bs : A.pc + (u * (A.n + 1) + t) * (long long)m * m;
    const double* Z = A.Z.p + dr * A.Z.bs;
    const double* H = A.H.p + dr * A.H.bs;
    const double* T = A.T.p + dr * A.T.bs;
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < p; ++j) {
        double s = 0.0;
        for (int k = 0; k < m; ++k) s = kf_fma(P[i * m + k], Z[j * m + k], s);
        PZt[i * p + j] = s;
      }
    // F = Z P Z^T + H and its lower Cholesky factor in L
    for (int j = 0; j < p; ++j) {
      for (int i = j; i < p; ++i) {
        double s = H[i * p + j];
        for (int k = 0; k < m; ++k) s = kf_fma(Z[i * m + k], PZt[k * p + j], s);
        for (int k = 0; k < j; ++k) s -= L[i * p + k] * L[j * p + k];
        if (i == j) {
          ok = ok && (s > 0.0);
          L[j * p + j] = sqrt(s);
        } else {
          L[i * p + j] = s / L[j * p + j];
        }
      }
    }
    if (!ok) key_min(A.ustat + u, 2 * t);
    // Li = L^-1 (lower), F^-1 = Li^T Li
    for (int j = 0; j < p; ++j)
      for (int i = 0; i < p; ++i) {
        if (i < j) { Li[i * p + j] = 0.0; continue; }
        double s = (i == j) ? 1.0 : 0.0;
        for (int k = j; k < i; ++k) s -= L[i * p + k] * Li[k * p + j];
        Li[i * p + j] = s / L[i * p + i];
      }
    for (int i = 0; i < p; ++i)
      for (int j = 0; j < p; ++j) {
        double s = 0.0;
        for (int k = (i > j ? i : j); k < p; ++k) s = kf_fma(Li[k * p + i], Li[k * p + j], s);
        Fi[i * p + j] = ok ? s : 0.0;
      }
    // K = T (P Z^T) F^-1
    for (int i = 0; i < m; ++i) {
      double tpz[D::PM];
      for (int j = 0; j < p; ++j) {
        double s = 0.0;
        for (int k = 0; k < m; ++k) s = kf_fma(T[i * m + k], PZt[k * p + j], s);
        tpz[j] = s;
      }
      for (int j = 0; j < p; ++j) {
        double s = 0.0;
        for (int k = 0; k < p; ++k) s = kf_fma(tpz[k], Fi[k * p + j], s);
        K[i * p + j] = s;
      }
    }
  } else {
    for (int i = 0; i < m * p + p * p; ++i) K[i] = 0.0;
  }
}

// x <- T x + c + G z  (G = R S_Q; the state innovation of step t)
template <class D>
KFB_HD void xplus_next(const D& d, double* x, const double* T, const double* c, const double* G, const double* z) {
  double xn[D::MM];
  for (int i = 0; i < d.m; ++i) {
    double s = c[i];
    for (int k = 0; k < d.m; ++k) s = kf_fma(T[i * d.m + k], x[k], s);
    for (int k = 0; k < d.rl(); ++k) s = kf_fma(G[i * d.rl() + k], z[k], s);
    xn[i] = s;
  }
  for (int i = 0; i < d.m; ++i) x[i] = xn[i];
}

// x+_0 = a0 + S_P0 z_init
template <class D>
KFB_HD void xplus_first(const D& d, double* x, const double* a0, const double* SP0, const double* z) {
  for (int i = 0; i < d.m; ++i) {
    double s = a0[i];
    for (int k = 0; k <= i; ++k) s = kf_fma(SP0[i * d.m + k], z[k], s);
    x[i] = s;
  }
}

// Step 2 at an observed row: v = y - (Z x+ + d + S_H zo) - Z a*, u = F^-1 v, a* <- T a* + K v
template <class D>
KFB_HD void forward_obs(const D& d, double* a, double* uo, const double* x, const double* y, const double* zo,
                        const double* T, const double* Z, const double* dd, const double* SH, const double* K,
                        const double* Fi) {
  double v[D::PM], an[D::MM];
  for (int i = 0; i < d.p; ++i) {
    double yp = dd[i];
    for (int k = 0; k < d.m; ++k) yp = kf_fma(Z[i * d.m + k], x[k], yp);
    for (int k = 0; k <= i; ++k) yp = kf_fma(SH[i * d.p + k], zo[k], yp);
    double za = 0.0;
    for (int k = 0; k < d.m; ++k) za = kf_fma(Z[i * d.m + k], a[k], za);
    v[i] = (y[i] - yp) - za;
  }
  for (int i = 0; i < d.p; ++i) {
    double s = 0.0;
    for (int k = 0; k < d.p; ++k) s = kf_fma(Fi[i * d.p + k], v[k], s);
    uo[i] = s;
  }
  for (int i = 0; i < d.m; ++i) {
    double s = 0.0;
    for (int k = 0; k < d.m; ++k) s = kf_fma(T[i * d.m + k], a[k], s);
    for (int k = 0; k < d.p; ++k) s = kf_fma(K[i * d.p + k], v[k], s);
    an[i] = s;
  }
  for (int i = 0; i < d.m; ++i) a[i] = an[i];
}

// a missing row: u = 0, a* <- T a*
template <class D>
KFB_HD void forward_missing(const D& d, double* a, double* uo, const double* T) {
  double an[D::MM];
  for (int i = 0; i < d.p; ++i) uo[i] = 0.0;
  for (int i = 0; i < d.m; ++i) {
    double s = 0.0;
    for (int k = 0; k < d.m; ++k) s = kf_fma(T[i * d.m + k], a[k], s);
    an[i] = s;
  }
  for (int i = 0; i < d.m; ++i) a[i] = an[i];
}

// Step 3: r <- Z^T (u - K^T r) + T^T r
template <class D>
KFB_HD void backward_step(const D& d, double* r, const double* uo, const double* T, const double* Z, const double* K) {
  double w[D::PM], rn[D::MM];
  for (int j = 0; j < d.p; ++j) {
    double s = uo[j];
    for (int k = 0; k < d.m; ++k) s = kf_fma(-K[k * d.p + j], r[k], s);
    w[j] = s;
  }
  for (int i = 0; i < d.m; ++i) {
    double s = 0.0;
    for (int k = 0; k < d.m; ++k) s = kf_fma(T[k * d.m + i], r[k], s);
    for (int j = 0; j < d.p; ++j) s = kf_fma(Z[j * d.m + i], w[j], s);
    rn[i] = s;
  }
  for (int i = 0; i < d.m; ++i) r[i] = rn[i];
}

// Step 4: xh <- M xh + N r  (xhat_0 = P0 r_{-1} is the case xh = 0, M = anything, N = P0)
template <class D>
KFB_HD void xhat_next(const D& d, double* xh, const double* T, const double* C, const double* r, bool first) {
  double xn[D::MM];
  for (int i = 0; i < d.m; ++i) {
    double s = 0.0;
    if (!first)
      for (int k = 0; k < d.m; ++k) s = kf_fma(T[i * d.m + k], xh[k], s);
    for (int k = 0; k < d.m; ++k) s = kf_fma(C[i * d.m + k], r[k], s);
    xn[i] = s;
  }
  for (int i = 0; i < d.m; ++i) xh[i] = xn[i];
}

// Copies cnt doubles into a register array for the compile-time path; the run-time path reads global memory in place.
template <class D, int N>
KFB_HD const double* stage(double (&dst)[N], const double* src, int cnt) {
  if constexpr (D::STATIC) {
    for (int i = 0; i < N; ++i) dst[i] = i < cnt ? src[i] : 0.0;
    return dst;
  } else {
    (void)dst; (void)cnt;
    return src;
  }
}

// One simulation s (steps 1-5); writes states[s] and, for the first simulation of a unit, info[u].
template <class D>
KFB_HD void simulate_one(const D& d, const Args& A, long long s) {
  const int m = d.m, p = d.p, n = A.n;
  const long long u = s / A.spu, dr = u / A.n_series, se = u % A.n_series;
  const long long S = A.S, W = warps_of(S), w = s >> 5;
  const int lane = (int)(s & 31);
  double* out = A.states + s * (long long)n * m;
  const int key = A.ustat[u];
  if (s % A.spu == 0) A.info[u] = info_of_key(key);
  if (key != KEY_NONE) {
    for (long long i = 0; i < (long long)n * m; ++i) out[i] = NAN;
    return;
  }
  constexpr bool ST = D::STATIC;
  constexpr int MM = ST ? D::MM : 1, PM = ST ? D::PM : 1;
  const double* f = A.fac + u * fac_stride(m, p, A.r);
  const long long gs = gain_stride(m, p);
  const double* gain = A.gain + u * n * gs;
  const double* y = A.y.p + se * A.y.bs;
  double bT[MM * MM], bZ[PM * MM], bG[MM * MM], bSH[PM * PM], bK[MM * PM], bFi[PM * PM];
  const double* T = stage<D>(bT, A.T.p + dr * A.T.bs, m * m);
  const double* Z = stage<D>(bZ, A.Z.p + dr * A.Z.bs, p * m);
  double cz[D::MM], dz[D::PM];
  for (int i = 0; i < m; ++i) cz[i] = A.c.p ? A.c.p[dr * A.c.bs + i] : 0.0;
  for (int i = 0; i < p; ++i) dz[i] = A.d.p ? A.d.p[dr * A.d.bs + i] : 0.0;
  const double* G;
  if constexpr (ST) {  // R S_Q as M x M with zero columns r..M-1
    for (int i = 0; i < MM; ++i)
      for (int k = 0; k < MM; ++k) bG[i * MM + k] = k < A.r ? f[m * m + i * A.r + k] : 0.0;
    G = bG;
  } else {
    G = f + m * m;
  }
  const double* SH = stage<D>(bSH, f + m * m + m * A.r, p * p);
  const double* a0 = A.a0.p + dr * A.a0.bs;
  auto load_zs = [&](double* z, int t) {  // z_state_t, zero beyond r
    const double* src = A.z_state + ((long long)t * S + s) * A.r;
    for (int k = 0; k < d.rl(); ++k) z[k] = k < A.r ? src[k] : 0.0;
  };
  double x[D::MM], a[D::MM], r[D::MM], uo[D::PM], z[D::MM > D::PM ? D::MM : D::PM];
  // steps 1-2, forward
  {
    double bS[MM * MM];
    const double* SP0 = stage<D>(bS, f, m * m);
    for (int k = 0; k < m; ++k) z[k] = A.z_init[s * m + k];
    xplus_first(d, x, a0, SP0, z);
  }
  for (int i = 0; i < m; ++i) a[i] = 0.0;
  for (int t = 0; t < n; ++t) {
    const double* yt = y + (long long)t * p;
    bool miss = false;
    for (int i = 0; i < p; ++i) miss = miss || kf_isnan(yt[i]);
    if (miss) {
      forward_missing(d, a, uo, T);
    } else {
      const double* K = stage<D>(bK, gain + t * gs, m * p);
      const double* Fi = stage<D>(bFi, gain + t * gs + m * p, p * p);
      const double* zo = A.z_obs + ((long long)t * S + s) * p;
      double zb[D::PM];
      for (int k = 0; k < p; ++k) zb[k] = zo[k];
      forward_obs(d, a, uo, x, yt, zb, T, Z, dz, SH, K, Fi);
    }
    double* us = A.uscr + ((long long)t * W + w) * p * 32 + lane;
    for (int k = 0; k < p; ++k) us[k * 32] = uo[k];
    if (t + 1 < n) {
      load_zs(z, t);
      xplus_next(d, x, T, cz, G, z);
    }
  }
  // step 3, backward: r_{t-1} from r_t; r_0 .. r_{n-2} are kept, r_{-1} stays in registers
  for (int i = 0; i < m; ++i) r[i] = 0.0;
  for (int t = n - 1; t >= 0; --t) {
    const double* us = A.uscr + ((long long)t * W + w) * p * 32 + lane;
    for (int k = 0; k < p; ++k) uo[k] = us[k * 32];
    const double* K = stage<D>(bK, gain + t * gs, m * p);
    backward_step(d, r, uo, T, Z, K);
    if (t >= 1) {
      double* rs = A.rscr + ((long long)(t - 1) * W + w) * m * 32 + lane;
      for (int k = 0; k < m; ++k) rs[k * 32] = r[k];
    }
  }
  // steps 4-5, forward again: x+ recomputed, xhat from the kept r_t
  double xh[D::MM];
  {
    double bS[MM * MM], bP[MM * MM];
    const double* SP0 = stage<D>(bS, f, m * m);
    for (int k = 0; k < m; ++k) z[k] = A.z_init[s * m + k];
    xplus_first(d, x, a0, SP0, z);
    const double* P0 = stage<D>(bP, A.P0.p + dr * A.P0.bs, m * m);
    xhat_next(d, xh, T, P0, r, true);
  }
  const double* C;
  double bC[MM * MM];
  C = stage<D>(bC, f + m * m + m * A.r + p * p, m * m);
  for (int t = 0; t < n; ++t) {
    for (int i = 0; i < m; ++i) out[(long long)t * m + i] = x[i] + xh[i];
    if (t + 1 < n) {
      load_zs(z, t);
      xplus_next(d, x, T, cz, G, z);
      const double* rs = A.rscr + ((long long)t * W + w) * m * 32 + lane;
      for (int k = 0; k < m; ++k) r[k] = rs[k * 32];
      xhat_next(d, xh, T, C, r, false);
    }
  }
}

// The one list of instantiations, used by the launcher (kf_simsmooth.cu) and the host build: run(Static<M, P>{r}) for
// k_states 1..4, k_endog 1..3 and k_posdef <= k_states; run(Dyn{m, p, r}) up to SS_MAX; false if nothing runs it.
template <class Run>
bool with_instance(int m, int p, int r, Run&& run) {
  if (m >= 1 && m <= 4 && p >= 1 && p <= 3 && r >= 1 && r <= m) {
#define KFB_SS_CASE(M, P) \
  if (m == M && p == P) { run(Static<M, P>{r}); return true; }
    KFB_SS_CASE(1, 1) KFB_SS_CASE(1, 2) KFB_SS_CASE(1, 3) KFB_SS_CASE(2, 1) KFB_SS_CASE(2, 2) KFB_SS_CASE(2, 3)
    KFB_SS_CASE(3, 1) KFB_SS_CASE(3, 2) KFB_SS_CASE(3, 3) KFB_SS_CASE(4, 1) KFB_SS_CASE(4, 2) KFB_SS_CASE(4, 3)
#undef KFB_SS_CASE
  }
  if (m >= 1 && m <= SS_MAX && p >= 1 && p <= SS_MAX && r >= 1 && r <= SS_MAX) {
    run(Dyn{m, p, r});
    return true;
  }
  return false;
}

}  // namespace ss
}  // namespace kfb
