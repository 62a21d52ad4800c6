// kf_pred.cuh - the hot path in ONE-STEP-PREDICTOR form (loglik + tape forward, and the adjoint).
//
// The reference's step is update (kalman_filter.py:255-284) followed by predict (:216-223):
//     K = P Z^T F^-1 ; A = I - K Z ; P_f = A P A^T + K H K^T ; P' = sym(T P_f T^T + C) ; a' = T (a + K v) + c
// When the filtered moments are not requested (NUTS only needs log-likelihood and gradient) the two stages
// compose exactly into
//     Kp = T K ; L = T - Kp Z ; P' = sym(L P L^T + Kp H Kp^T + C) ; a' = T a + c + Kp v
// which is the same Joseph-stabilised sum of PSD terms but needs 2 m^3 instead of 4 m^3 multiply-adds per step in
// the forward pass and 4 m^3 instead of ~8 m^3 in the adjoint (no P_f / A P recomputation), and has a shorter
// dependent chain per step.  Values agree with the two-stage form to rounding (tests: rtol 1e-8 vs the oracle).
// Used for MK_STD (standard / single / cholesky p=1 or corrected) and MK_STEADY (fixed gain matrix Gss).
#pragma once
#include "kf_core.cuh"

namespace kfb {

template <class X>
struct PredTmp {
  typename X::template Buf<SZ_P> v, w, piv;
  typename X::template Buf<SZ_MP> Mm, TM, Kp, KH;
  typename X::template Buf<SZ_PP> F, Fi, L, Li;
  typename X::template Buf<SZ_MM> Lm, S1, S2;
  KFB_HD PredTmp(X& x) : v(x), w(x), piv(x), Mm(x), TM(x), Kp(x), KH(x), F(x), Fi(x), L(x), Li(x), Lm(x), S1(x), S2(x) {}
};

// v, Mm, F, Fi, TM, Kp, Lm(= T - Kp Z), w for an observed row.  Gain matrix = Fi (MK_STD) or prm.Gss (MK_STEADY).
template <int MK, class X, class TA, class TPm>
KFB_HD StepStat pred_gain(X& x, const Params<X>& prm, const double* yt, double d_sign, const TA& a, const TPm& P,
                          PredTmp<X>& u, LogAcc* acc, bool per_step_log, bool full_det = false) {
  const int m = x.m(), p = x.p();
  StepStat st;
  KFB_FOR(i, p) {
    double s = yt[i] - d_sign * prm.d[i];
#pragma unroll
    for (int k = 0; k < m; ++k) s = kf_fma(-prm.Z[i * m + k], a[k], s);
    u.v[i] = s;
  }
  gemm<false, true, 0>(x, u.Mm, P, prm.Z, m, m, p);  // Mm = P Z^T
  KFB_FOR(idx, p * p) {
    const int i = x.div_p(idx), j = idx - i * p;
    double s = prm.H[idx];
#pragma unroll
    for (int k = 0; k < m; ++k) s = kf_fma(prm.Z[i * m + k], u.Mm[k * p + j], s);
    u.F[idx] = s;
  }
  gemm<false, false, 0>(x, u.TM, prm.T, u.Mm, m, m, p);  // TM = T Mm   (independent of the factorisation)
  st.ok = true;
  st.logdet = 0.0;
  if (x.lane() == 0) {
    st.ok = ldl_inverse(u.F, u.Fi, u.L, u.Li, u.piv, p);
    if (full_det && p > 1 && st.ok) st.ok = lu_pivots(u.F, u.L, u.piv, p);  // log det of the full matrix (t = 0)
    if (st.ok) {
#pragma unroll
      for (int i = 0; i < p; ++i) {
        if (per_step_log) st.logdet += log(u.piv[i]);
        else if (acc) acc->mul(u.piv[i]);
      }
    }
  }
  x.sync();
  if (MK == MK_STEADY) {
    gemm<false, false, 0>(x, u.Kp, u.TM, prm.Gss, m, p, p);
    KFB_FOR(i, p) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < p; ++j) s = kf_fma(prm.Gss[i * p + j], u.v[j], s);
      u.w[i] = s;
    }
  } else {
    gemm<false, false, 0>(x, u.Kp, u.TM, u.Fi, m, p, p);
    KFB_FOR(i, p) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < p; ++j) s = kf_fma(u.Fi[i * p + j], u.v[j], s);
      u.w[i] = s;
    }
  }
  KFB_FOR(idx, m * m) {  // Lm = T - Kp Z
    const int i = x.div_m(idx), j = idx - i * m;
    double s = prm.T[idx];
#pragma unroll
    for (int k = 0; k < p; ++k) s = kf_fma(-u.Kp[i * p + k], prm.Z[k * m + j], s);
    u.Lm[idx] = s;
  }
  x.sync();
  double q = 0.0;
#pragma unroll
  for (int i = 0; i < p; ++i) q = kf_fma(u.v[i], u.w[i], q);
  st.quad = q;
  return st;
}

// ------------------------------------------------------------------------------------------------
// forward: loglik (+ tape)
// ------------------------------------------------------------------------------------------------
template <int MK, class X>
KFB_HD void forward_unit_pred(X& x, const KfArgs& A, long long u) {
  const int m = x.m(), p = x.p(), n = A.n;
  const long long draw = u / A.n_series, series = u - draw * A.n_series;
  Params<X> prm(x);
  typename X::template Buf<SZ_MM> C(x), P(x);
  typename X::template Buf<SZ_M> c(x), a(x), an(x);
  PredTmp<X> tmp(x);

  const double* Tp = A.T.p + draw * A.T.bs;
  const double* Zp = A.Z.p + draw * A.Z.bs;
  const double* Hp = A.H.p + draw * A.H.bs;
  const double* Cp = A.C.p + draw * A.C.bs;
  const double* cp = A.c.p ? A.c.p + draw * A.c.bs : nullptr;
  const double* dp = A.d.p ? A.d.p + draw * A.d.bs : nullptr;
  load_or_zero(x, prm.T, Tp, m * m);
  load_or_zero(x, prm.Z, Zp, p * m);
  load_or_zero(x, prm.H, Hp, p * p);
  load_or_zero(x, C, Cp, m * m);
  load_or_zero(x, c, cp, m);
  load_or_zero(x, prm.d, dp, p);
  load_or_zero(x, a, A.a0.p + draw * A.a0.bs, m);
  if (MK == MK_STEADY) {
    load_or_zero(x, P, A.Pss.p + draw * A.Pss.bs, m * m);
    load_or_zero(x, prm.Gss, A.Gss.p + draw * A.Gss.bs, p * p);
  } else {
    load_or_zero(x, P, A.P0.p + draw * A.P0.bs, m * m);
  }
  x.sync();

  const double* y = x.y_base(A, series);
  const bool lane0 = (x.lane() == 0);
  LogAcc acc;
  double llsum = 0.0;
  int info = 0;
  double* tp = A.tape ? x.tape_base(A, u) : nullptr;
  const long long tstep = x.tape_step(A), telem = x.tape_elem(A);

  for (int t = 0; t < n; ++t) {
    if (X::TV) {
      if (A.T.ts) load_or_zero(x, prm.T, Tp + t * A.T.ts, m * m);
      if (A.Z.ts) load_or_zero(x, prm.Z, Zp + t * A.Z.ts, p * m);
      if (A.H.ts) load_or_zero(x, prm.H, Hp + t * A.H.ts, p * p);
      if (A.C.ts) load_or_zero(x, C, Cp + t * A.C.ts, m * m);
      if (A.c.ts) load_or_zero(x, c, cp + t * A.c.ts, m);
      if (A.d.ts) load_or_zero(x, prm.d, dp + t * A.d.ts, p);
      x.sync();
    }
    const double* yt = y + (long long)t * p;
    const int nm = count_missing(x, yt);
    if (nm == 0) {
      StepStat st = pred_gain<MK>(x, prm, yt, A.d_sign, a, P, tmp, &acc, false, MK == MK_STD && t == 0);
      if (!st.ok && info == 0) info = t + 1;
      llsum += -0.5 * (A.ll_const + st.quad);
      KFB_FOR(i, m) {  // a' = T a + c + Kp v
        double s = c[i];
#pragma unroll
        for (int k = 0; k < m; ++k) s = kf_fma(prm.T[i * m + k], a[k], s);
#pragma unroll
        for (int k = 0; k < p; ++k) s = kf_fma(tmp.Kp[i * p + k], tmp.v[k], s);
        an[i] = s;
      }
      gemm<false, false, 0>(x, tmp.S1, tmp.Lm, P, m, m, m);      // L P
      gemm<false, false, 0>(x, tmp.KH, tmp.Kp, prm.H, m, p, p);  // Kp H
      KFB_FOR(idx, m * m) tmp.S2[idx] = C[idx];
      x.sync();
      gemm<false, true, 1>(x, tmp.S2, tmp.S1, tmp.Lm, m, m, m);  // + L P L^T
      gemm<false, true, 1>(x, tmp.S2, tmp.KH, tmp.Kp, m, p, m);  // + Kp H Kp^T
    } else {
      if (nm != p && info == 0) info = -(t + 1);
      KFB_FOR(i, m) {
        double s = c[i];
#pragma unroll
        for (int k = 0; k < m; ++k) s = kf_fma(prm.T[i * m + k], a[k], s);
        an[i] = s;
      }
      gemm<false, false, 0>(x, tmp.S1, prm.T, P, m, m, m);
      KFB_FOR(idx, m * m) tmp.S2[idx] = C[idx];
      x.sync();
      gemm<false, true, 1>(x, tmp.S2, tmp.S1, prm.T, m, m, m);
    }
    KFB_FOR(i, m) a[i] = an[i];
    KFB_FOR(idx, m * m) {
      const int i = x.div_m(idx), j = idx - i * m;
      P[idx] = 0.5 * (tmp.S2[idx] + tmp.S2[j * m + i]);
    }
    x.sync();
    if (tp && t + 1 < n) {
      KFB_FOR(k, m) tp[k * telem] = a[k];
      KFB_FOR(idx, m * m) {
        const int i = x.div_m(idx), j = idx - i * m;
        if (j >= i) tp[(m + i * m - (i * (i - 1)) / 2 + (j - i)) * telem] = P[idx];
      }
      tp += tstep;
    }
  }
  if (lane0) {
    double ll = llsum - 0.5 * acc.value();
    if (info != 0) ll = nan("");
    if (A.loglik) A.loglik[u] = ll;
    if (MK == MK_STEADY && A.dare_info && A.dare_info[u / A.n_series] != 0) info = KF_INFO_DARE_FAILED;
    if (A.info) A.info[u] = info;
  }
}

// ------------------------------------------------------------------------------------------------
// adjoint
// ------------------------------------------------------------------------------------------------
// One step's inputs for the adjoint: predicted moments of step t and everything that depends only on them
// (innovation, gain, closed-loop matrix).  None of it depends on the adjoint state.
template <class X>
struct StepSet {
  typename X::template Buf<SZ_M> a;
  typename X::template Buf<SZ_MM> P;
  PredTmp<X> g;
  bool observed;
  KFB_HD explicit StepSet(X& x) : a(x), P(x), g(x), observed(false) {}
};

template <int MK, class X>
KFB_HD void backward_unit_pred(X& x, const KfArgs& A, long long u) {
  const int m = x.m(), p = x.p(), n = A.n;
  const long long draw = u / A.n_series, series = u - draw * A.n_series;
  Params<X> prm(x);
  typename X::template Buf<SZ_MM> Pb(x), Tb(x), Cb(x), Ps(x), S4(x), Lb(x);
  typename X::template Buf<SZ_M> ab(x), abn(x), cb(x);
  typename X::template Buf<SZ_MP> Zb(x), Kb(x), Mb(x), PK(x), TMb(x);
  typename X::template Buf<SZ_PP> Hb(x), Fb(x), Gb(x), Q1(x);
  typename X::template Buf<SZ_P> db(x), vb(x);
  StepSet<X> S0(x);

  const double* Tp = A.T.p + draw * A.T.bs;
  const double* Zp = A.Z.p + draw * A.Z.bs;
  const double* Hp = A.H.p + draw * A.H.bs;
  const double* dp = A.d.p ? A.d.p + draw * A.d.bs : nullptr;
  load_or_zero(x, prm.T, Tp, m * m);
  load_or_zero(x, prm.Z, Zp, p * m);
  load_or_zero(x, prm.H, Hp, p * p);
  load_or_zero(x, prm.d, dp, p);
  if (MK == MK_STEADY) load_or_zero(x, prm.Gss, A.Gss.p + draw * A.Gss.bs, p * p);
  KFB_FOR(i, m) { ab[i] = 0.0; cb[i] = 0.0; }
  KFB_FOR(i, m * m) { Pb[i] = 0.0; Tb[i] = 0.0; Cb[i] = 0.0; }
  KFB_FOR(i, p * m) Zb[i] = 0.0;
  KFB_FOR(i, p * p) { Hb[i] = 0.0; Gb[i] = 0.0; }
  KFB_FOR(i, p) db[i] = 0.0;
  x.sync();

  const double* y = x.y_base(A, series);
  const double gl = A.g_loglik ? A.g_loglik[u] : 1.0;
  typename X::template Buf<SZ_TAPE> nxt(x);
  typename X::TapeReader rd(x, A, u);
  // Cotangents nobody asked for are not accumulated (every reference model has a constant design matrix, so Z-bar -
  // 2 m^2 p + m p^2 multiply-adds per step - is never needed at theta level).  Uniform run-time branches.
  const bool need_Z = (A.gZ != nullptr), need_H = (A.gH != nullptr) || (MK == MK_STEADY);
  // T-bar: structural models (local level, trend + seasonal: config 4) have a constant transition matrix.  Without T-bar
  // and Z-bar the dense product Lb = Ps L (P + P^T) - one of the four m^3 products of the adjoint step - is only needed
  // through Lb Z^T = Ps (L (P + P^T) Z^T): two m^2 p products instead.
  // Cooperative contexts only (X::SKIP_LB): in the thread-per-unit kernels the extra run-time branch cost the m = 2
  // headline kernel 14 % (register allocation), and m^3 is tiny there.
  const bool need_Lb = !X::SKIP_LB || (A.gT != nullptr) || need_Z;

  // ---- inputs of step t (tape entries are consumed in strictly descending order)
  auto prepare = [&](int t, StepSet<X>& S) {
    if (X::TV) {
      if (A.T.ts) load_or_zero(x, prm.T, Tp + t * A.T.ts, m * m);
      if (A.Z.ts) load_or_zero(x, prm.Z, Zp + t * A.Z.ts, p * m);
      if (A.H.ts) load_or_zero(x, prm.H, Hp + t * A.H.ts, p * p);
      if (A.d.ts) load_or_zero(x, prm.d, dp + t * A.d.ts, p);
      x.sync();
    }
    if (t == 0) {
      load_or_zero(x, S.a, A.a0.p + draw * A.a0.bs, m);
      if (MK == MK_STEADY) load_or_zero(x, S.P, A.Pss.p + draw * A.Pss.bs, m * m);
      else load_or_zero(x, S.P, A.P0.p + draw * A.P0.bs, m * m);
    } else {
      rd.get(x, nxt);
      KFB_FOR(k, m) S.a[k] = nxt[k];
      KFB_FOR(idx, m * m) {
        int i = x.div_m(idx), j = idx - i * m;
        if (j < i) { const int sw = i; i = j; j = sw; }
        S.P[idx] = nxt[m + i * m - (i * (i - 1)) / 2 + (j - i)];
      }
    }
    x.sync();
    const double* yt = y + (long long)t * p;
    S.observed = (count_missing(x, yt) == 0);
    if (S.observed) {
      pred_gain<MK>(x, prm, yt, A.d_sign, S.a, S.P, S.g, (LogAcc*)nullptr, false);
    } else {
      KFB_FOR(i, m * m) S.g.Lm[i] = prm.T[i];  // L = T, Kp = 0
      x.sync();
    }
  };

  // ---- adjoint of step t
  auto adjoint = [&](int t, StepSet<X>& S) {
    auto& a = S.a;
    auto& P = S.P;
    auto& tmp = S.g;
    const bool observed = S.observed;
    const double lb = gl + (A.g_ll_obs ? A.g_ll_obs[u * n + t] : 0.0);
    // ---- adjoint of  a' = T a + c + Kp v ,  P' = sym(L P L^T + Kp H Kp^T + C)
    KFB_FOR(idx, m * m) {
      const int i = x.div_m(idx), j = idx - i * m;
      Ps[idx] = 0.5 * (Pb[idx] + Pb[j * m + i]);
      S4[idx] = P[idx] + P[j * m + i];
    }
    x.sync();
    KFB_FOR(idx, m * m) Cb[idx] += Ps[idx];
    KFB_FOR(i, m) cb[i] += ab[i];
    gemm<false, false, 0>(x, tmp.S1, tmp.Lm, S4, m, m, m);   // L (P + P^T)
    if (need_Lb) {
      gemm<false, false, 0>(x, Lb, Ps, tmp.S1, m, m, m);     // Lb = Ps L (P + P^T)
    } else if (observed) {
      gemm<false, true, 0>(x, tmp.KH, tmp.S1, prm.Z, m, m, p);  // L (P + P^T) Z^T   (KH is free in the adjoint)
    }
    gemm<false, false, 0>(x, tmp.S1, Ps, tmp.Lm, m, m, m);   // Ps L
    gemm<true, false, 0>(x, Pb, tmp.Lm, tmp.S1, m, m, m);    // Pb = L^T Ps L
    if (need_Lb) KFB_FOR(idx, m * m) {                       // Tb += ab a^T + Lb
      const int i = x.div_m(idx), j = idx - i * m;
      Tb[idx] += kf_fma(ab[i], a[j], Lb[idx]);
    }
    KFB_FOR(i, m) {                                          // abn = T^T ab
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < m; ++k) s = kf_fma(prm.T[k * m + i], ab[k], s);
      abn[i] = s;
    }
    x.sync();
    if (observed) {
      KFB_FOR(idx, p * p) {
        const int i = x.div_p(idx), j = idx - i * p;
        Q1[idx] = prm.H[idx] + prm.H[j * p + i];
      }
      gemm<false, false, 0>(x, PK, Ps, tmp.Kp, m, m, p);       // Ps Kp
      gemm<false, false, 0>(x, Kb, PK, Q1, m, p, p);           // Kb = Ps Kp (H + H^T)
      if (need_Lb) {
        KFB_FOR(idx, m * p) {
          const int i = x.div_p(idx), j = idx - i * p;
          double s = kf_fma(ab[i], tmp.v[j], Kb[idx]);           // + ab v^T
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(-Lb[i * m + k], prm.Z[j * m + k], s);  // - Lb Z^T
          Kb[idx] = s;
        }
      } else {
        KFB_FOR(idx, m * p) {
          const int i = x.div_p(idx), j = idx - i * p;
          double s = kf_fma(ab[i], tmp.v[j], Kb[idx]);           // + ab v^T
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(-Ps[i * m + k], tmp.KH[k * p + j], s);  // - Ps (L (P + P^T) Z^T)
          Kb[idx] = s;
        }
      }
      x.sync();  // Kb is read across lanes below
      if (need_H) gemm<true, false, 1>(x, Hb, tmp.Kp, PK, p, m, p);  // Hb += Kp^T Ps Kp
      if (need_Z) gemm<true, false, 2>(x, Zb, tmp.Kp, Lb, p, m, m);  // Zb -= Kp^T Lb
      if (MK == MK_STEADY) {
        KFB_FOR(i, p) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(tmp.Kp[k * p + i], ab[k], s);
#pragma unroll
          for (int j = 0; j < p; ++j) s = kf_fma(-0.5 * lb * (prm.Gss[i * p + j] + prm.Gss[j * p + i]), tmp.v[j], s);
          vb[i] = s;
        }
        gemm<true, false, 1>(x, Gb, tmp.TM, Kb, p, m, p);      // Gssb += TM^T Kb
        KFB_FOR(idx, p * p) {
          const int i = x.div_p(idx), j = idx - i * p;
          Gb[idx] = kf_fma(-0.5 * lb * tmp.v[i], tmp.v[j], Gb[idx]);
          Fb[idx] = -0.5 * lb * tmp.Fi[j * p + i];
        }
        x.sync();
        gemm<false, true, 0>(x, TMb, Kb, prm.Gss, m, p, p);    // TMb = Kb Gss^T
      } else {
        KFB_FOR(i, p) {
          double s = -lb * tmp.w[i];
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(tmp.Kp[k * p + i], ab[k], s);
          vb[i] = s;
        }
        gemm<true, false, 0>(x, Q1, tmp.Kp, Kb, p, m, p);      // Kp^T Kb
        KFB_FOR(idx, p * p) {
          const int i = x.div_p(idx), j = idx - i * p;
          double s = -0.5 * lb * (tmp.Fi[j * p + i] - tmp.w[i] * tmp.w[j]);
#pragma unroll
          for (int k = 0; k < p; ++k) s = kf_fma(-Q1[i * p + k], tmp.Fi[j * p + k], s);
          Fb[idx] = s;
        }
        x.sync();
        gemm<false, true, 0>(x, TMb, Kb, tmp.Fi, m, p, p);     // TMb = Kb G^T
      }
      gemm<false, true, 1>(x, Tb, TMb, tmp.Mm, m, p, m);       // Tb += TMb Mm^T
      gemm<true, false, 0>(x, Mb, prm.T, TMb, m, m, p);        // Mb = T^T TMb
      gemm<true, false, 1>(x, Mb, prm.Z, Fb, m, p, p);         //    + Z^T Fb
      if (need_Z) KFB_FOR(idx, p * m) {                        // Zb += Fb Mm^T + Mb^T P - vb a^T
        const int i = x.div_m(idx), j = idx - i * m;
        double s = kf_fma(-vb[i], a[j], Zb[idx]);
#pragma unroll
        for (int k = 0; k < p; ++k) s = kf_fma(Fb[i * p + k], tmp.Mm[j * p + k], s);
#pragma unroll
        for (int k = 0; k < m; ++k) s = kf_fma(Mb[k * p + i], P[k * m + j], s);
        Zb[idx] = s;
      }
      if (need_H) KFB_FOR(idx, p * p) Hb[idx] += Fb[idx];
      gemm<false, false, 1>(x, Pb, Mb, prm.Z, m, p, m);        // Pb += Mb Z
      KFB_FOR(i, m) {                                          // ab = T^T ab - Z^T vb
        double s = abn[i];
#pragma unroll
        for (int k = 0; k < p; ++k) s = kf_fma(-prm.Z[k * m + i], vb[k], s);
        ab[i] = s;
      }
      KFB_FOR(i, p) db[i] = kf_fma(-A.d_sign, vb[i], db[i]);
      x.sync();
    } else {
      KFB_FOR(i, m) ab[i] = abn[i];
      x.sync();
    }
    if (X::TV) {
      if (A.T.ts && A.gT) { KFB_FOR(i, m * m) { A.gT[(u * n + t) * m * m + i] = Tb[i]; Tb[i] = 0.0; } }
      if (A.C.ts && A.gC) { KFB_FOR(i, m * m) { A.gC[(u * n + t) * m * m + i] = Cb[i]; Cb[i] = 0.0; } }
      if (A.c.ts && A.gc) { KFB_FOR(i, m) { A.gc[(u * n + t) * m + i] = cb[i]; cb[i] = 0.0; } }
      if (A.Z.ts && A.gZ) { KFB_FOR(i, p * m) { A.gZ[(u * n + t) * p * m + i] = Zb[i]; Zb[i] = 0.0; } }
      if (A.H.ts && A.gH) { KFB_FOR(i, p * p) { A.gH[(u * n + t) * p * p + i] = Hb[i]; Hb[i] = 0.0; } }
      if (A.d.ts && A.gd) { KFB_FOR(i, p) { A.gd[(u * n + t) * p + i] = db[i]; db[i] = 0.0; } }
      x.sync();
    }
  };

  for (int t = n - 1; t >= 0; --t) {
    prepare(t, S0);
    adjoint(t, S0);
  }
  if (A.ga0) KFB_FOR(i, m) A.ga0[u * m + i] = ab[i];
  if (MK == MK_STEADY) {
    if (A.gPss) KFB_FOR(i, m * m) A.gPss[u * m * m + i] = Pb[i];
    if (A.gGss) KFB_FOR(i, p * p) A.gGss[u * p * p + i] = Gb[i];
    if (A.gP0) KFB_FOR(i, m * m) A.gP0[u * m * m + i] = 0.0;
  } else {
    if (A.gP0) KFB_FOR(i, m * m) A.gP0[u * m * m + i] = Pb[i];
  }
  if (A.gT && !(X::TV && A.T.ts)) KFB_FOR(i, m * m) A.gT[u * m * m + i] = Tb[i];
  if (A.gC && !(X::TV && A.C.ts)) KFB_FOR(i, m * m) A.gC[u * m * m + i] = Cb[i];
  if (A.gc && !(X::TV && A.c.ts)) KFB_FOR(i, m) A.gc[u * m + i] = cb[i];
  if (A.gZ && !(X::TV && A.Z.ts)) KFB_FOR(i, p * m) A.gZ[u * p * m + i] = Zb[i];
  if (A.gH && !(X::TV && A.H.ts)) KFB_FOR(i, p * p) A.gH[u * p * p + i] = Hb[i];
  if (A.gd && !(X::TV && A.d.ts)) KFB_FOR(i, p) A.gd[u * p + i] = db[i];
}

}  // namespace kfb
