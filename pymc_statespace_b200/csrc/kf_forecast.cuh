// kf_forecast.cuh - forecast paths and impulse responses from the end of the sample, written once as KFB_HD functions:
// kf_forecast.cu runs them as kernels and the host build of the kernels (tests/hostsim/draws.cpp, requests from
// kf_draws_run.cuh) runs them on the host.
//
// Model (the filters', as in kf_simsmooth.cuh): y_t = Z x_t + d + eps_t, eps_t ~ N(0, H); x_{t+1} = T x_t + c + R eta_t,
// eta_t ~ N(0, Q); static matrices.  Given the state's distribution N(a, P) at the first forecast time (a_n, P_n: the
// predicted moments of the exact filter after y_0..y_{n-1}), one simulation of H steps is
//   x_0 = a + S_P z_init;  for h = 0..H-1:  states[h] = x_h,  obs[h] = Z x_h + d + S_H z_obs_h,
//                                          x_{h+1} = T x_h + c + (R S_Q) z_state_h  (h < H-1).
// S_A is ss::psd_factor's lower factor.  The state recursion is kf_simsmooth.cuh's xplus_first / xplus_next, the
// instantiation list its ss::with_instance; the observation line is the only new arithmetic.
//
// Layout: normals and outputs are time-major ([h][s][.]), so at a fixed h the lanes of a warp read and write 32
// consecutive records - one contiguous run per warp and step, no shared-memory staging.
//
// Impulse responses: column j of horizon h is T^h R S e_j (states) and Z T^h R S e_j (observations), the response to
// shock j at time 0, with S = I, diag(sqrt(diag Q)) or psd_factor(Q) (KFB_SHOCK_UNIT / _STD / _CHOLESKY).
#pragma once
#include "kf_simsmooth.cuh"

namespace kfb {
namespace fc {

constexpr int SHOCK_UNIT = 0, SHOCK_STD = 1, SHOCK_CHOLESKY = 2;  // = KFB_SHOCK_* (include/kfb200.h)

struct Args {
  long long U, n_series, S, spu;  // units (draw * n_series + series), simulations, simulations per unit
  int H, m, p, r;                 // horizon, k_states, k_endog, k_posdef
  MatArg T, Z, R, Hm, Q, c, d;    // batch strides only (static matrices); Hm is the observation covariance H
  const double *mean, *cov;       // start moments [U][m], [U][m][m]
  const double *z_init, *z_state, *z_obs;  // [S][m], [H - 1][S][r], [H][S][p]
  double *states, *obs;           // [H][S][m], [H][S][p]; either may be null
  bool vec;                       // states and obs are 16-byte aligned: even record sizes are stored as double2
  int* info;                      // [U]
  double* fac;                    // [U][S_P (m m) | R S_Q (m r) | S_H (p p) | S_Q (r r)]
  int* ustat;                     // [U] 0 or INFO_NOT_PSD, written by unit_prep
};

KFB_HD long long fac_stride(int m, int p, int r) {
  return (long long)m * m + (long long)m * r + (long long)p * p + (long long)r * r;
}

// Per unit, once: the three factors and R S_Q into fac[u]; the unit's status into ustat[u] and info[u].  A start
// covariance, Q or H that is not PSD, or a NaN in the start mean, gives INFO_NOT_PSD.
KFB_HD void unit_prep(const Args& A, long long u) {
  const long long dr = u / A.n_series;
  const int m = A.m, p = A.p, r = A.r;
  double* f = A.fac + u * fac_stride(m, p, r);
  double *SP = f, *G = f + m * m, *SH = G + m * r, *SQ = SH + p * p;
  const double* R = A.R.p + dr * A.R.bs;
  bool ok = ss::psd_factor(A.cov + u * m * m, SP, m);
  for (int i = 0; i < m; ++i) ok = ok && !kf_isnan(A.mean[u * m + i]);
  ok = ss::psd_factor(A.Hm.p + dr * A.Hm.bs, SH, p) && ok;
  ok = ss::psd_factor(A.Q.p + dr * A.Q.bs, SQ, r) && ok;
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < r; ++j) {
      double s = 0.0;
      for (int k = j; k < r; ++k) s = kf_fma(R[i * r + k], SQ[k * r + j], s);
      G[i * r + j] = s;
    }
  const int st = ok ? 0 : ss::INFO_NOT_PSD;
  A.ustat[u] = st;
  A.info[u] = st;
}

// y = Z x + d + S_H zo  (S_H lower triangular)
template <class D>
KFB_HD void obs_of(const D& d, double* yo, const double* x, const double* Z, const double* dd, const double* SH,
                   const double* zo) {
  for (int i = 0; i < d.p; ++i) {
    double s = dd[i];
    for (int k = 0; k < d.m; ++k) s = kf_fma(Z[i * d.m + k], x[k], s);
    for (int k = 0; k <= i; ++k) s = kf_fma(SH[i * d.p + k], zo[k], s);
    yo[i] = s;
  }
}

// One record of cnt doubles; with compile-time dims, an even size and 16-byte aligned outputs as double2 stores.
template <class D, int N>
KFB_HD void put(double* dst, const double (&v)[N], int cnt, bool vec) {
#if defined(__CUDA_ARCH__)
  if constexpr (D::STATIC && N % 2 == 0) {
    if (vec) {
      for (int i = 0; i < N / 2; ++i) reinterpret_cast<double2*>(dst)[i] = make_double2(v[2 * i], v[2 * i + 1]);
      return;
    }
  }
#endif
  (void)vec;
  for (int i = 0; i < cnt; ++i) dst[i] = v[i];
}

// One simulation s: its H records of states and / or observations.
template <class D>
KFB_HD void path_one(const D& d, const Args& A, long long s) {
  const int m = d.m, p = d.p, H = A.H;
  const long long u = s / A.spu, dr = u / A.n_series, S = A.S;
  if (A.ustat[u] != 0) {
    for (int h = 0; h < H; ++h) {
      if (A.states)
        for (int i = 0; i < m; ++i) A.states[((long long)h * S + s) * m + i] = NAN;
      if (A.obs)
        for (int i = 0; i < p; ++i) A.obs[((long long)h * S + s) * p + i] = NAN;
    }
    return;
  }
  constexpr bool ST = D::STATIC;
  constexpr int MM = ST ? D::MM : 1, PM = ST ? D::PM : 1;
  const double* f = A.fac + u * fac_stride(m, p, A.r);
  double bT[MM * MM], bZ[PM * MM], bG[MM * MM], bSH[PM * PM], bSP[MM * MM];
  const double* T = ss::stage<D>(bT, A.T.p + dr * A.T.bs, m * m);
  const double* Z = ss::stage<D>(bZ, A.Z.p + dr * A.Z.bs, p * m);
  const double* G;
  if constexpr (ST) {  // R S_Q as M x M with zero columns r..M-1
    for (int i = 0; i < MM; ++i)
      for (int k = 0; k < MM; ++k) bG[i * MM + k] = k < A.r ? f[m * m + i * A.r + k] : 0.0;
    G = bG;
  } else {
    G = f + m * m;
  }
  const double* SH = ss::stage<D>(bSH, f + m * m + m * A.r, p * p);
  double cz[D::MM], dz[D::PM];
  for (int i = 0; i < m; ++i) cz[i] = A.c.p ? A.c.p[dr * A.c.bs + i] : 0.0;
  for (int i = 0; i < p; ++i) dz[i] = A.d.p ? A.d.p[dr * A.d.bs + i] : 0.0;
  double x[D::MM], yo[D::PM], z[D::MM > D::PM ? D::MM : D::PM];
  {
    const double* SP = ss::stage<D>(bSP, f, m * m);
    for (int k = 0; k < m; ++k) z[k] = A.z_init[s * m + k];
    ss::xplus_first(d, x, A.mean + u * m, SP, z);
  }
  // record s of step h: base + (h S + s) * size, advanced by S * size per step
  double* so = A.states ? A.states + s * m : nullptr;
  double* yp = A.obs ? A.obs + s * p : nullptr;
  const double* zo = A.z_obs + s * p;
  const double* zs = A.z_state + s * A.r;
  for (int h = 0; h < H; ++h) {
    if (so) {
      put<D>(so, x, m, A.vec);
      so += S * m;
    }
    if (yp) {
      for (int k = 0; k < p; ++k) z[k] = zo[k];
      obs_of(d, yo, x, Z, dz, SH, z);
      put<D>(yp, yo, p, A.vec);
      yp += S * p;
    }
    zo += S * p;
    if (h + 1 < H) {
      for (int k = 0; k < d.rl(); ++k) z[k] = k < A.r ? zs[k] : 0.0;
      ss::xplus_next(d, x, T, cz, G, z);
      zs += S * A.r;
    }
  }
}

struct IrfArgs {
  long long nD;       // draws
  int H, m, p, r, shock;
  MatArg T, Z, R, Q;  // batch strides only
  double *states, *obs;  // [nD][H][m][r], [nD][H][p][r]; either may be null
  int* info;             // [nD]
};

// Impulse responses of one (draw, shock j): x_0 = R S e_j, x_{h+1} = T x_h (xplus_next with c = 0 and no innovation).
// Under KFB_SHOCK_STD / _CHOLESKY a Q that is not PSD makes the draw's responses NaN and its info INFO_NOT_PSD.
template <class D>
KFB_HD void irf_one(const D& d, const IrfArgs& A, long long i) {
  const int m = d.m, p = d.p, r = A.r, H = A.H;
  const long long dr = i / r;
  const int j = (int)(i - dr * r);
  const double* Q = A.Q.p + dr * A.Q.bs;
  double L[D::MM * D::MM];  // r <= k_states on the compile-time path
  bool ok = true;
  if (A.shock == SHOCK_CHOLESKY || A.shock == SHOCK_STD) ok = ss::psd_factor(Q, L, r);
  if (j == 0) A.info[dr] = ok ? 0 : ss::INFO_NOT_PSD;
  auto at = [&](double* base, int rows, int h, int row) { return base + ((dr * H + h) * rows + row) * (long long)r + j; };
  if (!ok) {
    for (int h = 0; h < H; ++h) {
      if (A.states)
        for (int k = 0; k < m; ++k) *at(A.states, m, h, k) = NAN;
      if (A.obs)
        for (int k = 0; k < p; ++k) *at(A.obs, p, h, k) = NAN;
    }
    return;
  }
  constexpr bool ST = D::STATIC;
  constexpr int MM = ST ? D::MM : 1, PM = ST ? D::PM : 1;
  double bT[MM * MM], bZ[PM * MM], bR[MM * MM];
  const double* T = ss::stage<D>(bT, A.T.p + dr * A.T.bs, m * m);
  const double* Z = ss::stage<D>(bZ, A.Z.p + dr * A.Z.bs, p * m);
  const double* R;
  if constexpr (ST) {  // R as M x M with zero columns r..M-1
    const double* src = A.R.p + dr * A.R.bs;
    for (int a = 0; a < MM; ++a)
      for (int k = 0; k < MM; ++k) bR[a * MM + k] = k < r ? src[a * r + k] : 0.0;
    R = bR;
  } else {
    R = A.R.p + dr * A.R.bs;
  }
  double v[D::MM], zero[D::MM], x[D::MM];  // v = S e_j, zero beyond r
  for (int k = 0; k < D::MM; ++k) {
    double e = 0.0;
    if (k < r) {
      if (A.shock == SHOCK_CHOLESKY) e = L[k * r + j];
      else if (k == j) e = A.shock == SHOCK_STD ? (Q[j * r + j] > 0.0 ? sqrt(Q[j * r + j]) : 0.0) : 1.0;
    }
    v[k] = e;
    zero[k] = 0.0;
    x[k] = 0.0;
  }
  ss::xplus_next(d, x, T, zero, R, v);  // x_0 = R S e_j
  for (int h = 0; h < H; ++h) {
    if (A.states)
      for (int k = 0; k < m; ++k) *at(A.states, m, h, k) = x[k];
    if (A.obs)
      for (int a = 0; a < p; ++a) {
        double s = 0.0;
        for (int k = 0; k < m; ++k) s = kf_fma(Z[a * m + k], x[k], s);
        *at(A.obs, p, h, a) = s;
      }
    if (h + 1 < H) ss::xplus_next(d, x, T, zero, R, zero);
  }
}

}  // namespace fc
}  // namespace kfb
