// kf_condfc.cuh - conditional forecasts from the end of the sample, written once as KFB_HD functions: kf_condfc.cu runs
// them as kernels and the host build of the kernels (tests/hostsim/draws.cpp, requests from kf_draws_run.cuh) runs them
// on the host.
//
// Model (the filters', as in kf_forecast.cuh): y_t = Z x_t + d + eps_t, eps_t ~ N(0, H); x_{t+1} = T x_t + c + R eta_t,
// eta_t ~ N(0, Q); static matrices.  Window index h is time n + h, h = 0..H-1.  cond[h][i] is the known value of
// y_{n+h,i} (NaN: free).  Everything is conditioned on y_0..y_{n-1} (through the start x_n ~ N(a, P): the predicted
// moments a_n, P_n of the exact filter) and on every non-NaN entry of cond.  At step h, o is the set of conditioned
// entries and u the free ones; every product uses the masked p x p form (zero rows / columns for free entries), so the
// compile-time instantiations keep a fixed p.
//
// 1. Window, one thread per unit (window_unit): the filter over the partly observed rows
//      F = Z_o P Z_o^T + H_oo (strictly positive definite, else info n + h + 1),  Fi = F^-1 embedded in p x p,
//      K = T P Z^T Fi,  v = cond - Z a - d (0 on free entries),  u_h = Fi v,
//      a <- T a + c + K v,  P <- T P L^T + C  (L = T - K Z, C = R Q R^T, symmetrised),
//    then the fast state smoother backwards from r = 0, N = 0:
//      r_{h-1} = Z^T (u_h - K^T r_h) + T^T r_h,  N_{h-1} = Z^T Fi Z + L^T N_h L,
//      state_mean[h] = a_h + P_h r_{h-1},  state_cov[h] = P_h - P_h N_{h-1} P_h,
//    and the observations: G = H_uo H_oo^- (the generalised inverse of psd_factor's zero-pivot rule; G = 0 whenever
//    H is diagonal), D = Z_u - G Z_o; obs_mean is cond on conditioned entries and D x^ + d_u + G (cond_o - d_o) on free
//    ones; obs_cov is D V D^T + H_uu - G H_ou on the free block and 0 on every row and column of a conditioned entry.
//    K, Fi, G and u of every (unit, h) go to the tape.
// 2. Paths, one thread per simulation (path_unit): the mean correction of kf_simsmooth.cuh's simulate_one over the
//    window.  x+ starts at a + S_P z_init and follows the model (xplus_first / xplus_next), eps+_h = S_H z_obs_h; the
//    masked forward step (ss::forward_obs_masked) filters cond - y+ with a* = 0, backward_step gives r, and x~ = x+ + x^ with
//    x^_0 = P r_{-1}, x^_{h+1} = T x^_h + C r_h.  Observations: y_o = cond_o exactly and
//      y_u = Z_u x~ + d_u + eps+_u + G (cond_o - Z_o x~ - d_o - eps+_o):
//    given x_{n+h} and the conditioned entries of row h the free entries are independent of everything else, and
//    eps+_u - G eps+_o has their conditional noise law independently of eps+_o, so no extra normals are needed.  With no
//    condition anywhere r = 0 and the paths are kf_forecast.cuh's path_one on the same normals.
// Normals and outputs of the paths are time-major ([h][s][.]) as in kf_forecast.cuh; the u and r scratch keeps
// simulate_one's warp-interleaved layout.
#pragma once
#include "kf_forecast.cuh"

namespace kfb {
namespace cf {

struct Args {
  long long U, n_series, S, spu;  // units (draw * n_series + series), simulations (0: moments only), per unit
  int n, H, m, p, r;              // observations before the window (info codes only), horizon, k_states, k_endog, k_posdef
  MatArg T, Z, R, Hm, Q, c, d;    // batch strides only (static matrices); Hm is the observation covariance H
  const double *mean, *cov;       // start moments [U][m], [U][m][m]
  const double* cond;             // [H][p] + u * cond_bs, NaN = free
  long long cond_bs;
  const double *z_init, *z_state, *z_obs;  // [S][m], [H - 1][S][r], [H][S][p]
  double *state_mean, *state_cov, *obs_mean, *obs_cov;  // [U][H][m], [U][H][m][m], [U][H][p], [U][H][p][p]; any may be null
  double *states, *obs;           // [H][S][m], [H][S][p]; either may be null
  bool vec;                       // states and obs are 16-byte aligned (fc::put)
  int* info;                      // [U]
  double* tape;                   // [U][H][K (m p) | Fi (p p) | G (p p) | u (p) | a (m) | P (m m)]
  double* fac;                    // [U][S_P (m m) | R S_Q (m r) | S_H (p p) | C (m m) | S_Q (r r)]  (ss::fac_stride)
  double* wscr;                   // [U][wscr_stride]: working matrices of the run-time-dims window
  int* ustat;                     // [U] 0, n + h + 1 or INFO_NOT_PSD, written by window_unit
  double *uscr, *rscr;            // u_h [H][warp][p][32], r_h [H - 1][warp][m][32]
};

KFB_HD long long tape_stride(int m, int p) {
  return (long long)m * p + 2LL * p * p + p + m + (long long)m * m;
}
KFB_HD long long wscr_stride(int m, int p) { return 3LL * m * m + 2LL * m * p + 4LL * p * p; }

// A register array on the compile-time path, the unit's scratch in global memory on the run-time path.
template <class D, int N>
KFB_HD double* buf(double (&reg)[N], double* scr) {
  if constexpr (D::STATIC) {
    (void)scr;
    return reg;
  } else {
    (void)reg;
    return scr;
  }
}

// Lm = T - K Z
template <class D>
KFB_HD void l_of(const D& d, double* Lm, const double* T, const double* K, const double* Z) {
  for (int i = 0; i < d.m; ++i)
    for (int j = 0; j < d.m; ++j) {
      double s = T[i * d.m + j];
      for (int k = 0; k < d.p; ++k) s = kf_fma(-K[i * d.p + k], Z[k * d.m + j], s);
      Lm[i * d.m + j] = s;
    }
}

// One step of the exact filter over a row with observed set o (bit i of om: y_i observed): ss::masked_gain's K and
// Fi, v = y - Z a - d on o (0 elsewhere), then between(), then with Pn
//   a <- T a + c + K v,  Pn = T P L^T + C  (L = T - K Z, C = R Q R^T), symmetrised.
// A complete row is the ordinary update.  False if F_o is not positive definite (then nothing else is written).
// PZt [m p], Lc, Li [p p], Lm, M1 [m m] are working matrices; between() may use Lc and Li.
template <class D, class Between>
KFB_HD bool masked_step(const D& d, unsigned om, const double* y, const double* T, const double* Z, const double* Hm,
                        const double* C, const double* cz, const double* dz, const double* P, double* a, double* v,
                        double* K, double* Fi, double* Pn, double* PZt, double* Lc, double* Li, double* Lm, double* M1,
                        Between&& between) {
  const int m = d.m, p = d.p;
  if (!ss::masked_gain(d, om, P, T, Z, Hm, K, Fi, PZt, Lc, Li)) return false;
  // v = y - Z a - d on the observed entries
  for (int i = 0; i < p; ++i) {
    double za = dz[i];
    for (int k = 0; k < m; ++k) za = kf_fma(Z[i * m + k], a[k], za);
    v[i] = ((om >> i) & 1u) ? y[i] - za : 0.0;
  }
  between();
  if (!Pn) return true;
  // a <- T a + c + K v;  Pn = T P L^T + C, symmetrised
  {
    double an[D::MM];
    for (int i = 0; i < m; ++i) {
      double s = cz[i];
      for (int k = 0; k < m; ++k) s = kf_fma(T[i * m + k], a[k], s);
      for (int k = 0; k < p; ++k) s = kf_fma(K[i * p + k], v[k], s);
      an[i] = s;
    }
    for (int i = 0; i < m; ++i) a[i] = an[i];
  }
  l_of(d, Lm, T, K, Z);
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < m; ++j) {
      double s = 0.0;
      for (int k = 0; k < m; ++k) s = kf_fma(P[i * m + k], Lm[j * m + k], s);
      M1[i * m + j] = s;
    }
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < m; ++j) {
      double s = C[i * m + j];
      for (int k = 0; k < m; ++k) s = kf_fma(T[i * m + k], M1[k * m + j], s);
      Lm[i * m + j] = s;  // Lm is free again: the new P before symmetrising
    }
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < m; ++j) Pn[i * m + j] = 0.5 * (Lm[i * m + j] + Lm[j * m + i]);
  return true;
}

// Factors of one unit into fac[u] (the layout of ss::fac_stride, the factors computed as fc::unit_prep computes them);
// false if the start covariance, Q or H is not PSD or the start mean has a NaN.
KFB_HD bool unit_factors(const Args& A, long long u) {
  const long long dr = u / A.n_series;
  const int m = A.m, p = A.p, r = A.r;
  double* f = A.fac + u * ss::fac_stride(m, p, r);
  double *SP = f, *G = f + m * m, *SH = G + m * r, *C = SH + p * p, *SQ = C + m * m;
  const double* R = A.R.p + dr * A.R.bs;
  const double* Q = A.Q.p + dr * A.Q.bs;
  bool ok = ss::psd_factor(A.cov + u * m * m, SP, m);
  for (int i = 0; i < m; ++i) ok = ok && !kf_isnan(A.mean[u * m + i]);
  ok = ss::psd_factor(A.Hm.p + dr * A.Hm.bs, SH, p) && ok;
  ok = ss::psd_factor(Q, SQ, r) && ok;
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
  return ok;
}

// Forward pass of the window: fills the unit's tape; 0, or n + h + 1 if F_o is not positive definite at step h.
template <class D>
KFB_HD int window_forward(const D& d, const Args& A, long long u) {
  const int m = d.m, p = d.p, H = A.H;
  const long long dr = u / A.n_series, ts = tape_stride(m, p);
  constexpr bool ST = D::STATIC;
  constexpr int MM = ST ? D::MM : 1, PM = ST ? D::PM : 1;
  const double* f = A.fac + u * ss::fac_stride(m, p, A.r);
  double* scr = A.wscr + u * wscr_stride(m, p);
  double bT[MM * MM], bZ[PM * MM], bP[MM * MM];
  const double* T = ss::stage<D>(bT, A.T.p + dr * A.T.bs, m * m);
  const double* Z = ss::stage<D>(bZ, A.Z.p + dr * A.Z.bs, p * m);
  const double* Hm = A.Hm.p + dr * A.Hm.bs;  // H and C are read in place, as K, Fi and G are written
  const double* C = f + m * m + m * A.r + p * p;
  double rPZ[MM * PM], rLc[PM * PM], rLi[PM * PM], rHL[PM * PM], rHg[PM * PM], rLm[MM * MM], rM1[MM * MM];
  double* PZt = buf<D>(rPZ, scr);
  double* Lc = buf<D>(rLc, scr + m * p);
  double* Li = buf<D>(rLi, scr + m * p + p * p);
  double* HL = buf<D>(rHL, scr + m * p + 2 * p * p);
  double* Hg = buf<D>(rHg, scr + m * p + 3 * p * p);
  double* Lm = buf<D>(rLm, scr + m * p + 4 * p * p);
  double* M1 = buf<D>(rM1, scr + m * p + 4 * p * p + m * m);
  double a[D::MM], cz[D::MM], dz[D::PM], v[D::PM], uo[D::PM];
  unsigned om;  // bit i: entry i is conditioned
  for (int i = 0; i < m; ++i) a[i] = A.mean[u * m + i];
  for (int i = 0; i < m; ++i) cz[i] = A.c.p ? A.c.p[dr * A.c.bs + i] : 0.0;
  for (int i = 0; i < p; ++i) dz[i] = A.d.p ? A.d.p[dr * A.d.bs + i] : 0.0;
  double* rec0 = A.tape + u * H * ts;
  for (int i = 0; i < m * m; ++i) rec0[m * p + 2 * p * p + p + m + i] = A.cov[u * m * m + i];
  for (int h = 0; h < H; ++h) {
    double* rec = rec0 + h * ts;
    double *tK = rec, *tFi = tK + m * p, *tG = tFi + p * p, *tu = tG + p * p, *ta = tu + p, *tP = ta + m;
    double *K = tK, *Fi = tFi, *G = tG;  // written in place on both paths: registers go to the step's products
    const double* y = A.cond + u * A.cond_bs + (long long)h * p;
    om = 0;
    for (int i = 0; i < p; ++i) om |= kf_isnan(y[i]) ? 0u : 1u << i;
    for (int i = 0; i < m; ++i) ta[i] = a[i];
    const double* P = ss::stage<D>(bP, tP, m * m);
    // u_h = Fi v and G between the gain and the update
    const auto u_and_g = [&]() {
      // u = Fi v
      for (int i = 0; i < p; ++i) {
        double s = 0.0;
        for (int k = 0; k < p; ++k) s = kf_fma(Fi[i * p + k], v[k], s);
        uo[i] = s;
      }
      // G = H_uo H_oo^-: W = the inverse of psd_factor(H_oo) on its non-zero pivots (0 elsewhere), H_oo^- = W^T W
      for (int i = 0; i < p; ++i)
        for (int j = 0; j < p; ++j) Hg[i * p + j] = (((om >> i) & 1u) && ((om >> j) & 1u)) ? Hm[i * p + j] : 0.0;
      ss::psd_factor(Hg, HL, p);  // a principal block of H, which unit_factors found PSD
      for (int j = 0; j < p; ++j)
        for (int i = 0; i < p; ++i) {
          if (i < j || HL[i * p + i] == 0.0 || HL[j * p + j] == 0.0) { Li[i * p + j] = 0.0; continue; }
          double s = (i == j) ? 1.0 : 0.0;
          for (int k = j; k < i; ++k) s -= HL[i * p + k] * Li[k * p + j];
          Li[i * p + j] = s / HL[i * p + i];
        }
      for (int i = 0; i < p; ++i)
        for (int j = 0; j < p; ++j) {
          double s = 0.0;
          for (int k = (i > j ? i : j); k < p; ++k) s = kf_fma(Li[k * p + i], Li[k * p + j], s);
          Hg[i * p + j] = s;
        }
      for (int i = 0; i < p; ++i)
        for (int j = 0; j < p; ++j) {
          double s = 0.0;
          if (!((om >> i) & 1u) && ((om >> j) & 1u))
            for (int k = 0; k < p; ++k)
              if (((om >> k) & 1u)) s = kf_fma(Hm[i * p + k], Hg[k * p + j], s);
          G[i * p + j] = s;
        }
      for (int i = 0; i < p; ++i) tu[i] = uo[i];
    };
    if (!masked_step(d, om, y, T, Z, Hm, C, cz, dz, P, a, v, K, Fi, h + 1 < H ? tP + ts : nullptr, PZt, Lc, Li, Lm, M1,
                     u_and_g))
      return A.n + h + 1;
  }
  return 0;
}

// Backward pass of the window: the moments of every step from the tape.
template <class D>
KFB_HD void window_backward(const D& d, const Args& A, long long u) {
  const int m = d.m, p = d.p, H = A.H;
  const long long dr = u / A.n_series, ts = tape_stride(m, p);
  constexpr bool ST = D::STATIC;
  constexpr int MM = ST ? D::MM : 1, PM = ST ? D::PM : 1;
  double* scr = A.wscr + u * wscr_stride(m, p);
  double bT[MM * MM], bZ[PM * MM], bH[PM * PM], bP[MM * MM], bK[MM * PM], bFi[PM * PM], bG[PM * PM];
  const double* T = ss::stage<D>(bT, A.T.p + dr * A.T.bs, m * m);
  const double* Z = ss::stage<D>(bZ, A.Z.p + dr * A.Z.bs, p * m);
  const double* Hm = ss::stage<D>(bH, A.Hm.p + dr * A.Hm.bs, p * p);
  double rFZ[PM * MM], rOC[PM * PM], rV[MM * MM], rNL[MM * MM], rN[MM * MM], rDV[PM * MM];
  double* FZ = buf<D>(rFZ, scr);                                  // Fi Z, then D
  double* OC = buf<D>(rOC, scr + m * p);                          // obs_cov before symmetrising
  double* V = buf<D>(rV, scr + m * p + 4 * p * p);                // L, then state_cov before symmetrising
  double* NL = buf<D>(rNL, scr + m * p + 4 * p * p + m * m);      // N L, then P N
  double* N = buf<D>(rN, scr + m * p + 4 * p * p + 2 * m * m);
  double* DV = buf<D>(rDV, scr + 2 * m * p + 4 * p * p + 3 * m * m - m * p);  // the last m p of the scratch
  double dz[D::PM], r[D::MM], xm[D::MM], zx[D::PM];
  unsigned om;  // bit i: entry i is conditioned
  for (int i = 0; i < p; ++i) dz[i] = A.d.p ? A.d.p[dr * A.d.bs + i] : 0.0;
  for (int i = 0; i < m; ++i) r[i] = 0.0;
  for (int i = 0; i < m * m; ++i) N[i] = 0.0;
  for (int h = H - 1; h >= 0; --h) {
    const double* rec = A.tape + (u * H + h) * ts;
    const double* K = ss::stage<D>(bK, rec, m * p);
    const double* Fi = ss::stage<D>(bFi, rec + m * p, p * p);
    const double* G = ss::stage<D>(bG, rec + m * p + p * p, p * p);
    const double* uo = rec + m * p + 2 * p * p;
    const double* ah = uo + p;
    const double* P = ss::stage<D>(bP, ah + m, m * m);
    const double* y = A.cond + u * A.cond_bs + (long long)h * p;
    om = 0;
    for (int i = 0; i < p; ++i) om |= kf_isnan(y[i]) ? 0u : 1u << i;
    {
      double ub[D::PM];
      for (int i = 0; i < p; ++i) ub[i] = uo[i];
      ss::backward_step(d, r, ub, T, Z, K);  // r_{h-1}
    }
    // N <- Z^T Fi Z + L^T N L
    l_of(d, V, T, K, Z);
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < m; ++j) {
        double s = 0.0;
        for (int k = 0; k < m; ++k) s = kf_fma(N[i * m + k], V[k * m + j], s);
        NL[i * m + j] = s;
      }
    for (int i = 0; i < p; ++i)
      for (int j = 0; j < m; ++j) {
        double s = 0.0;
        for (int k = 0; k < p; ++k) s = kf_fma(Fi[i * p + k], Z[k * m + j], s);
        FZ[i * m + j] = s;
      }
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < m; ++j) {
        double s = 0.0;
        for (int k = 0; k < p; ++k) s = kf_fma(Z[k * m + i], FZ[k * m + j], s);
        for (int k = 0; k < m; ++k) s = kf_fma(V[k * m + i], NL[k * m + j], s);
        N[i * m + j] = s;
      }
    for (int i = 0; i < m; ++i)
      for (int j = i + 1; j < m; ++j) {
        const double s = 0.5 * (N[i * m + j] + N[j * m + i]);
        N[i * m + j] = s;
        N[j * m + i] = s;
      }
    // state moments: x^ = a + P r, V = P - P N P
    for (int i = 0; i < m; ++i) {
      double s = ah[i];
      for (int k = 0; k < m; ++k) s = kf_fma(P[i * m + k], r[k], s);
      xm[i] = s;
    }
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < m; ++j) {
        double s = 0.0;
        for (int k = 0; k < m; ++k) s = kf_fma(P[i * m + k], N[k * m + j], s);
        NL[i * m + j] = s;
      }
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < m; ++j) {
        double s = P[i * m + j];
        for (int k = 0; k < m; ++k) s = kf_fma(-NL[i * m + k], P[k * m + j], s);
        V[i * m + j] = s;
      }
    const long long uh = u * H + h;
    if (A.state_mean)
      for (int i = 0; i < m; ++i) A.state_mean[uh * m + i] = xm[i];
    if (A.state_cov)
      for (int i = 0; i < m; ++i)
        for (int j = 0; j < m; ++j) A.state_cov[uh * m * m + i * m + j] = 0.5 * (V[i * m + j] + V[j * m + i]);
    // observation moments: D = Z_u - G Z_o (rows of conditioned entries 0)
    for (int i = 0; i < p; ++i) {
      double s = dz[i];
      for (int k = 0; k < m; ++k) s = kf_fma(Z[i * m + k], xm[k], s);
      zx[i] = s;
    }
    for (int i = 0; i < p; ++i)
      for (int k = 0; k < m; ++k) {
        double s = ((om >> i) & 1u) ? 0.0 : Z[i * m + k];
        if (!((om >> i) & 1u))
          for (int j = 0; j < p; ++j)
            if (((om >> j) & 1u)) s = kf_fma(-G[i * p + j], Z[j * m + k], s);
        FZ[i * m + k] = s;
      }
    for (int i = 0; i < p; ++i)
      for (int k = 0; k < m; ++k) {
        double s = 0.0;
        for (int l = 0; l < m; ++l) s = kf_fma(FZ[i * m + l], V[l * m + k], s);
        DV[i * m + k] = s;
      }
    for (int i = 0; i < p; ++i)
      for (int j = 0; j < p; ++j) {
        double s = 0.0;
        if (!((om >> i) & 1u) && !((om >> j) & 1u)) {
          s = Hm[i * p + j];
          for (int k = 0; k < p; ++k)
            if (((om >> k) & 1u)) s = kf_fma(-G[i * p + k], Hm[k * p + j], s);
          for (int k = 0; k < m; ++k) s = kf_fma(DV[i * m + k], FZ[j * m + k], s);
        }
        OC[i * p + j] = s;
      }
    if (A.obs_mean)
      for (int i = 0; i < p; ++i) {
        double s = ((om >> i) & 1u) ? y[i] : zx[i];
        if (!((om >> i) & 1u))
          for (int j = 0; j < p; ++j)
            if (((om >> j) & 1u)) s = kf_fma(G[i * p + j], y[j] - zx[j], s);
        A.obs_mean[uh * p + i] = s;
      }
    if (A.obs_cov)
      for (int i = 0; i < p; ++i)
        for (int j = 0; j < p; ++j) A.obs_cov[uh * p * p + i * p + j] = 0.5 * (OC[i * p + j] + OC[j * p + i]);
  }
}

// One unit: factors, window filter and smoother; info[u] and ustat[u] (0, n + h + 1 or INFO_NOT_PSD).  A failing
// unit's moments are NaN (path_unit makes its paths NaN).
template <class D>
KFB_HD void window_unit(const D& d, const Args& A, long long u) {
  int st = unit_factors(A, u) ? 0 : ss::INFO_NOT_PSD;
  if (st == 0) st = window_forward(d, A, u);
  if (st == 0) {
    window_backward(d, A, u);
  } else {
    const int m = d.m, p = d.p;
    for (long long i = u * A.H * m; i < (u + 1) * A.H * m; ++i)
      if (A.state_mean) A.state_mean[i] = NAN;
    for (long long i = u * A.H * m * m; i < (u + 1) * A.H * m * m; ++i)
      if (A.state_cov) A.state_cov[i] = NAN;
    for (long long i = u * A.H * p; i < (u + 1) * A.H * p; ++i)
      if (A.obs_mean) A.obs_mean[i] = NAN;
    for (long long i = u * A.H * p * p; i < (u + 1) * A.H * p * p; ++i)
      if (A.obs_cov) A.obs_cov[i] = NAN;
  }
  A.ustat[u] = st;
  A.info[u] = st;
}

// One simulation s: its H records of states and / or observations.
template <class D>
KFB_HD void path_unit(const D& d, const Args& A, long long s) {
  const int m = d.m, p = d.p, H = A.H;
  const long long u = s / A.spu, dr = u / A.n_series, S = A.S, W = ss::warps_of(S), w = s >> 5;
  const int lane = (int)(s & 31);
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
  const double* f = A.fac + u * ss::fac_stride(m, p, A.r);
  const long long ts = tape_stride(m, p);
  const double* tape = A.tape + u * H * ts;
  const double* cond = A.cond + u * A.cond_bs;
  double bT[MM * MM], bZ[PM * MM], bG[MM * MM], bSH[PM * PM], bK[MM * PM], bFi[PM * PM];
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
  auto load_zs = [&](double* z, int h) {  // z_state_h, zero beyond r
    const double* src = A.z_state + ((long long)h * S + s) * A.r;
    for (int k = 0; k < d.rl(); ++k) z[k] = k < A.r ? src[k] : 0.0;
  };
  auto load_zo = [&](double* z, int h) {
    const double* src = A.z_obs + ((long long)h * S + s) * p;
    for (int k = 0; k < p; ++k) z[k] = src[k];
  };
  double x[D::MM], a[D::MM], r[D::MM], uo[D::PM], zb[D::PM], z[D::MM > D::PM ? D::MM : D::PM];
  // forward: x+ and the masked filter of cond - y+
  {
    double bS[MM * MM];
    const double* SP = ss::stage<D>(bS, f, m * m);
    for (int k = 0; k < m; ++k) z[k] = A.z_init[s * m + k];
    ss::xplus_first(d, x, A.mean + u * m, SP, z);
  }
  for (int i = 0; i < m; ++i) a[i] = 0.0;
  for (int h = 0; h < H; ++h) {
    const double* K = ss::stage<D>(bK, tape + h * ts, m * p);
    const double* Fi = ss::stage<D>(bFi, tape + h * ts + m * p, p * p);
    load_zo(zb, h);
    ss::forward_obs_masked(d, a, uo, x, cond + (long long)h * p, zb, T, Z, dz, SH, K, Fi);
    double* us = A.uscr + ((long long)h * W + w) * p * 32 + lane;
    for (int k = 0; k < p; ++k) us[k * 32] = uo[k];
    if (h + 1 < H) {
      load_zs(z, h);
      ss::xplus_next(d, x, T, cz, G, z);
    }
  }
  // backward: r_{h-1} from r_h; r_0 .. r_{H-2} are kept, r_{-1} stays in registers
  for (int i = 0; i < m; ++i) r[i] = 0.0;
  for (int h = H - 1; h >= 0; --h) {
    const double* us = A.uscr + ((long long)h * W + w) * p * 32 + lane;
    for (int k = 0; k < p; ++k) uo[k] = us[k * 32];
    const double* K = ss::stage<D>(bK, tape + h * ts, m * p);
    ss::backward_step(d, r, uo, T, Z, K);
    if (h >= 1) {
      double* rs = A.rscr + ((long long)(h - 1) * W + w) * m * 32 + lane;
      for (int k = 0; k < m; ++k) rs[k * 32] = r[k];
    }
  }
  // forward again: x+ recomputed, x^ from the kept r_h, x~ = x+ + x^ and its observations
  double xh[D::MM];
  {
    double bS[MM * MM], bP[MM * MM];
    const double* SP = ss::stage<D>(bS, f, m * m);
    for (int k = 0; k < m; ++k) z[k] = A.z_init[s * m + k];
    ss::xplus_first(d, x, A.mean + u * m, SP, z);
    const double* P = ss::stage<D>(bP, A.cov + u * m * m, m * m);
    ss::xhat_next(d, xh, T, P, r, true);
  }
  double bC[MM * MM];
  const double* C = ss::stage<D>(bC, f + m * m + m * A.r + p * p, m * m);
  double* so = A.states ? A.states + s * m : nullptr;
  double* yp = A.obs ? A.obs + s * p : nullptr;
  for (int h = 0; h < H; ++h) {
    double xt[D::MM];
    for (int i = 0; i < m; ++i) xt[i] = x[i] + xh[i];
    if (so) {
      fc::put<D>(so, xt, m, A.vec);
      so += S * m;
    }
    if (yp) {
      const double* y = cond + (long long)h * p;
      const double* Gh = ss::stage<D>(bFi, tape + h * ts + m * p + p * p, p * p);
      double yo[D::PM], ya[D::PM];
      load_zo(zb, h);
      fc::obs_of(d, yo, xt, Z, dz, SH, zb);
      for (int i = 0; i < p; ++i) {
        double v = yo[i];
        if (!kf_isnan(y[i])) {
          v = y[i];
        } else {
          for (int j = 0; j < p; ++j)
            if (!kf_isnan(y[j])) v = kf_fma(Gh[i * p + j], y[j] - yo[j], v);
        }
        ya[i] = v;
      }
      fc::put<D>(yp, ya, p, A.vec);
      yp += S * p;
    }
    if (h + 1 < H) {
      load_zs(z, h);
      ss::xplus_next(d, x, T, cz, G, z);
      const double* rs = A.rscr + ((long long)h * W + w) * m * 32 + lane;
      for (int k = 0; k < m; ++k) r[k] = rs[k * 32];
      ss::xhat_next(d, xh, T, C, r, false);
    }
  }
}

// The exact filter over a sample with partly observed rows (kfb_masked_filter): one thread per unit runs masked_step
// over y_0..y_{n-1} from (a0, P0) and writes the predicted moments, rows 0..n, in kfb_forward's layout.
struct FilterArgs {
  long long U, n_series, S, spu;  // units (draw * n_series + series); S, spu are 0
  int n, m, p, r;
  MatArg y, a0, P0, T, Z, R, Hm, Q, c, d;  // batch strides only (static matrices); Hm is the observation covariance H
  double *ps, *pc;                         // predicted_states [U][n + 1][m], predicted_covs [U][n + 1][m][m]; one may be null
  int* info;                               // [U] 0, or t + 1 if F_o is not positive definite at step t
  double* scr;                             // [U][filter_scr_stride]: C, then the working matrices of the run-time dims
};

// C (m m) | P (m m) | Pn (m m) | Lm (m m) | M1 (m m) | PZt (m p) | K (m p) | Lc (p p) | Li (p p) | Fi (p p)
KFB_HD long long filter_scr_stride(int m, int p) { return 5LL * m * m + 2LL * m * p + 3LL * p * p; }

template <class D>
KFB_HD void filter_unit(const D& d, const FilterArgs& A, long long u) {
  const int m = d.m, p = d.p, n = A.n;
  const long long dr = u / A.n_series, se = u % A.n_series;
  constexpr bool ST = D::STATIC;
  constexpr int MM = ST ? D::MM : 1, PM = ST ? D::PM : 1;
  double* scr = A.scr + u * filter_scr_stride(m, p);
  double* C = scr;  // R Q R^T, summed as unit_factors sums it; read in place, as H is
  {
    const double* R = A.R.p + dr * A.R.bs;
    const double* Q = A.Q.p + dr * A.Q.bs;
    const int r = A.r;
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
  }
  double bT[MM * MM], bZ[PM * MM];
  const double* T = ss::stage<D>(bT, A.T.p + dr * A.T.bs, m * m);
  const double* Z = ss::stage<D>(bZ, A.Z.p + dr * A.Z.bs, p * m);
  const double* Hm = A.Hm.p + dr * A.Hm.bs;
  double rP[MM * MM], rPn[MM * MM], rLm[MM * MM], rM1[MM * MM], rPZ[MM * PM], rK[MM * PM], rLc[PM * PM], rLi[PM * PM],
      rFi[PM * PM];
  const long long mm = (long long)m * m, mp = (long long)m * p;
  double* P = buf<D>(rP, scr + mm);
  double* Pn = buf<D>(rPn, scr + 2 * mm);
  double* Lm = buf<D>(rLm, scr + 3 * mm);
  double* M1 = buf<D>(rM1, scr + 4 * mm);
  double* PZt = buf<D>(rPZ, scr + 5 * mm);
  double* K = buf<D>(rK, scr + 5 * mm + mp);
  double* Lc = buf<D>(rLc, scr + 5 * mm + 2 * mp);
  double* Li = buf<D>(rLi, scr + 5 * mm + 2 * mp + p * p);
  double* Fi = buf<D>(rFi, scr + 5 * mm + 2 * mp + 2 * p * p);
  double a[D::MM], cz[D::MM], dz[D::PM], v[D::PM];
  for (int i = 0; i < m; ++i) a[i] = A.a0.p[dr * A.a0.bs + i];
  for (int i = 0; i < m * m; ++i) P[i] = A.P0.p[dr * A.P0.bs + i];
  for (int i = 0; i < m; ++i) cz[i] = A.c.p ? A.c.p[dr * A.c.bs + i] : 0.0;
  for (int i = 0; i < p; ++i) dz[i] = A.d.p ? A.d.p[dr * A.d.bs + i] : 0.0;
  double* ps = A.ps ? A.ps + u * (n + 1) * m : nullptr;
  double* pc = A.pc ? A.pc + u * (n + 1) * mm : nullptr;
  const double* y = A.y.p + se * A.y.bs;
  int st = 0;
  for (int t = 0; t <= n; ++t) {
    if (ps)
      for (int i = 0; i < m; ++i) ps[(long long)t * m + i] = a[i];
    if (pc)
      for (int i = 0; i < m * m; ++i) pc[t * mm + i] = P[i];
    if (t == n) break;
    const double* yt = y + (long long)t * p;
    unsigned om = 0;  // bit i: y_t,i observed
    for (int i = 0; i < p; ++i) om |= kf_isnan(yt[i]) ? 0u : 1u << i;
    if (!masked_step(d, om, yt, T, Z, Hm, C, cz, dz, P, a, v, K, Fi, Pn, PZt, Lc, Li, Lm, M1, [] {})) {
      st = t + 1;
      break;
    }
    for (int i = 0; i < m * m; ++i) P[i] = Pn[i];
  }
  if (st != 0) {
    for (long long i = 0; i < (n + 1LL) * m; ++i)
      if (ps) ps[i] = NAN;
    for (long long i = 0; i < (n + 1LL) * mm; ++i)
      if (pc) pc[i] = NAN;
  }
  A.info[u] = st;
}

}  // namespace cf
}  // namespace kfb
