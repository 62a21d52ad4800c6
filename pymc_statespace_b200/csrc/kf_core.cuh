// kf_core.cuh - the Kalman recursion and its adjoint, written ONCE over an execution-context
// policy X:
//   ThreadCtx<M,P>  one unit per thread, compile-time dims, every matrix in registers
//   CoopCtx         G lanes (a warp or a whole CTA) per unit, run-time dims, matrices in shared memory
//   (tests/hostsim) the same code compiled for the host so the math can be debugged without a GPU
//
// What is computed (reference pymc_statespace/filters/kalman_filter.py):
//   per step  mask (:196-213) -> update (:255-284 | :287-318 | :333-351 | :399-419 | :460-480)
//             -> predict (:216-223); outputs assembled as in :166-193.
//   adjoint   reverse recursion of SURVEY.md appendix B (the reference's gradient is PyTensor
//             autodiff of the scan; there is no reference source for it).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define KFB_HD __host__ __device__ __forceinline__
#else
#define KFB_HD inline
#endif

namespace kfb {

constexpr double KF_LOG_2PI = 1.8378770664093454835606594728112;  // MVN_CONST kalman_filter.py:16
constexpr double KF_LN2 = 0.69314718055994530941723212145818;
constexpr int KF_INFO_DARE_FAILED = 0x40000001;  // = KFB_INFO_DARE_FAILED (include/kfb200.h)
constexpr int KF_INFO_BAD_STRUCTURE = 0x40000003;  // = KFB_INFO_BAD_STRUCTURE: a KFB_FLAG_Z_UNIT0 / KFB_FLAG_H_ZERO promise is false

enum MathKind : int { MK_STD = 0, MK_UNIV = 1, MK_STEADY = 2, MK_CHOLS = 3 };
enum SizeClass : int { SZ_M = 0, SZ_P = 1, SZ_MM = 2, SZ_MP = 3, SZ_PP = 4, SZ_TAPE = 5 };

struct MatArg {
  const double* p;
  long long bs;  // stride between draws (series for y); 0 = shared
  long long ts;  // stride between time steps; 0 = static
};

// KfArgs::struct_flags bits.  The first three are caller promises (kfb200.h flags), set only for k_endog = 1 with static
// Z and H; the k_endog = 1 kernels skip the products with the known zeros and ones and check the promises per unit.
constexpr int KF_STRUCT_Z_UNIT0 = 1;      // Z = [1, 0, .., 0]           (KFB_FLAG_Z_UNIT0)
constexpr int KF_STRUCT_H_ZERO = 2;       // H = 0                       (KFB_FLAG_H_ZERO)
constexpr int KF_STRUCT_T_COMPANION = 4;  // T = [t | e_0 .. e_{m-2}]    (KFB_FLAG_T_COMPANION)
// the tape is the reduced recursion's compressed tape (CTape below): set by the C-ABI layer when the three promises above
// and KFB_FLAG_NO_MISSING hold, so that the forward pass and the adjoint agree on the format
constexpr int KF_STRUCT_COMPRESSED = 8;

struct KfArgs {
  long long U, n_series;
  int n, m, p, math_kind;
  MatArg y, a0, P0, T, Z, H, C, c, d, Pss, Gss;  // C = R Q R^T (hoisted, predict :219)
  double ll_const;  // multiple of log(2 pi) per observed step (p-independent quirk Q1)
  double d_sign;    // v = y - Z a - d_sign * d  (Q5: -1 for "single", Q6: 0 for "steady_state")
  // forward outputs (any may be null)
  double *loglik, *ll_obs, *fs, *ps, *fc, *pc;
  int* info;
  const int* dare_info;  // steady state: per-draw status of the DARE solve (0 = ok) or null
  int struct_flags;      // KF_STRUCT_* bits (above)
  double* tape;  // predicted (a_t, tri(P_t)) for t = 1..n-1 (KF_STRUCT_COMPRESSED: the CTape entries below)
  // backward
  const double *g_loglik, *g_ll_obs;
  double *ga0, *gP0, *gT, *gZ, *gH, *gC, *gc, *gd, *gPss, *gGss;
};

KFB_HD int tape_width(int m) { return m + (m * (m + 1)) / 2; }
// the tape holds whole warps of units (thread-per-unit layout [t-1][warp][k][32])
KFB_HD long long tape_units_padded(long long U) { return (U + 31) & ~31LL; }

// Compressed tape of the k_endog = 1 kernels (KF_STRUCT_COMPRESSED; kf_p1.cuh, ZU_REDUCED).  The entry of step t holds
// what the reduced adjoint reads: (v_t, 1 / F_t, P_t[0][1 .. m-2]), KT = m doubles (1 at m = 1: v_t alone, F is a
// constant of the draw there).  S = KF_CTAPE_STEPS consecutive steps of one warp are one contiguous block, so the
// adjoint fetches S steps with one bulk copy:  [t / S][warp][t % S][row of the step].  In a row, each lane's doubles go
// in pairs (element k < KT & ~1 at (k / 2) * 64 + 2 lane + k % 2: one 16-byte store / LDS.128 per pair) and an odd last
// element at (KT & ~1) * 32 + lane.  Step 0 is never taped: its slot in block 0 is not read.  The forward kernels, the
// adjoint's ring and the host build all locate entries through this struct; kfb_workspace_bytes sizes the tape with
// ctape_steps_padded.
#ifndef KFB_P1_TAPE_STEPS
#define KFB_P1_TAPE_STEPS 4
#endif
constexpr int KF_CTAPE_STEPS = KFB_P1_TAPE_STEPS;
static_assert((KF_CTAPE_STEPS & (KF_CTAPE_STEPS - 1)) == 0 && KF_CTAPE_STEPS <= 16, "a power of two <= 16");
KFB_HD constexpr int ctape_entry_doubles(int m) { return m >= 2 ? m : 1; }
// time entries per unit: steps 0 .. n-1 rounded up to whole blocks (none when nothing is taped)
KFB_HD long long ctape_steps_padded(int n) {
  return n > 1 ? (long long)((n + KF_CTAPE_STEPS - 1) / KF_CTAPE_STEPS) * KF_CTAPE_STEPS : 0;
}
template <int KT>
struct CTape {
  static constexpr int S = KF_CTAPE_STEPS;
  static constexpr int ROW = KT * 32;   // doubles of one step of one warp
  static constexpr int BLOCK = S * ROW;  // doubles of one block of one warp
  // doubles between the blocks t / S and t / S + 1 of a warp
  KFB_HD static long long block_stride(long long U) { return (long long)BLOCK * (tape_units_padded(U) >> 5); }
  // doubles from the start of the tape to the row of unit u's warp at step t
  KFB_HD static long long row(long long U, long long u, int t) {
    const unsigned tu = (unsigned)t;
    return (long long)(tu / S) * block_stride(U) + (u >> 5) * BLOCK + (long long)((tu % S) * ROW);
  }
  // element k of a lane within a row
  KFB_HD static constexpr int lane_offset(int lane, int k) {
    return k < (KT & ~1) ? (k >> 1) * 64 + 2 * lane + (k & 1) : (KT & ~1) * 32 + lane;
  }
};

KFB_HD double kf_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return fma(a, b, c);
#else
  return a * b + c;  // host simulation only
#endif
}

KFB_HD bool kf_isnan(double v) { return v != v; }

// Deferred logarithm: sum_t log(f_t) = log(prod mantissas) + ln2 * sum exponents.  One fp64 multiply
// and a few integer ops per factor instead of a ~40-instruction fp64 log on the serial critical path.
struct LogAcc {
  double mant;
  int expo;
  int count;
  KFB_HD LogAcc() : mant(1.0), expo(0), count(0) {}
  KFB_HD void mul(double f) {  // f must be a positive normal number (checked by the caller)
    mant *= f;               // mant in [1,2) * f
    int hi;
#if defined(__CUDA_ARCH__)
    hi = __double2hiint(mant);
    int e = ((hi >> 20) & 0x7ff) - 1023;
    expo += e;
    mant = __hiloint2double(hi - (e << 20), __double2loint(mant));
#else
    long long bits;
    std::memcpy(&bits, &mant, 8);
    hi = (int)(bits >> 32);
    int e = ((hi >> 20) & 0x7ff) - 1023;
    expo += e;
    bits -= ((long long)e) << 52;
    std::memcpy(&mant, &bits, 8);
#endif
  }
  KFB_HD double value() const { return log(mant) + KF_LN2 * (double)expo; }
};

#define KFB_FOR(i, cnt) _Pragma("unroll") for (int i = x.lane(); i < (cnt); i += x.G())

// C (r x c)  = / += / -=  op(A) (r x kk) * op(B) (kk x c);  row-major storage of the un-transposed operand
template <bool TA, bool TB, int MODE, class X, class TC, class TAa, class TBb>
KFB_HD void gemm(X& x, TC& C, const TAa& A, const TBb& B, int r, int kk, int c) {
  KFB_FOR(idx, r * c) {
    const int i = idx / c, j = idx - i * c;
    double s = (MODE == 0) ? 0.0 : C[idx];
#pragma unroll
    for (int k = 0; k < kk; ++k) {
      const double av = A[TA ? k * r + i : i * kk + k];
      const double bv = B[TB ? j * kk + k : k * c + j];
      s = kf_fma(MODE == 2 ? -av : av, bv, s);
    }
    C[idx] = s;
  }
  x.sync();
}

template <class X, class TD>
KFB_HD void load_or_zero(X& x, TD& dst, const double* src, int cnt) {
  KFB_FOR(i, cnt) dst[i] = src ? src[i] : 0.0;
}

// Symmetric positive-definite p x p inverse via L D L^T (no square roots).  Reads the UPPER triangle of F, like
// LAPACK posv behind the reference's `solve(F, I, assume_a="pos")` (kalman_filter.py:267-269; scipy's default
// lower=False) - it only matters when F is not symmetric, i.e. at t = 0 with a non-symmetric P0 and k_endog > 1
// (BayesianVARMAX with stationary_initialization=False writes P0 = theta.reshape(m, m)).  Serial; executed by one lane.
// piv[] receives D (det sym(F) = prod D).  Returns false if a pivot is not a positive finite number.
template <class TF, class TG, class TL, class TP>
KFB_HD bool ldl_inverse(const TF& F, TG& G, TL& L, TL& Li, TP& piv, int p) {
  bool ok = true;
#pragma unroll
  for (int j = 0; j < p; ++j) {
    double dj = F[j * p + j];
#pragma unroll
    for (int k = 0; k < p; ++k)
      if (k < j) dj = kf_fma(-L[j * p + k] * L[j * p + k], piv[k], dj);
    piv[j] = dj;
    ok = ok && (dj > 0.0) && (dj < 1.0e300);
    const double rj = 1.0 / dj;
#pragma unroll
    for (int i = 0; i < p; ++i) {
      if (i > j) {
        double s = F[j * p + i];
#pragma unroll
        for (int k = 0; k < p; ++k)
          if (k < j) s = kf_fma(-L[i * p + k] * L[j * p + k], piv[k], s);
        L[i * p + j] = s * rj;
      }
    }
    L[j * p + j] = rj;  // store 1/D on the diagonal
  }
  // Li = L^{-1} (unit lower triangular)
#pragma unroll
  for (int c = 0; c < p; ++c) {
#pragma unroll
    for (int i = 0; i < p; ++i) {
      if (i == c) Li[i * p + c] = 1.0;
      if (i < c) Li[i * p + c] = 0.0;
      if (i > c) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < p; ++k)
          if (k >= c && k < i) s = kf_fma(-L[i * p + k], Li[k * p + c], s);
        Li[i * p + c] = s;
      }
    }
  }
  // G = Li^T D^{-1} Li
#pragma unroll
  for (int i = 0; i < p; ++i) {
#pragma unroll
    for (int j = 0; j < p; ++j) {
      if (j <= i) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < p; ++k)
          if (k >= i) s = kf_fma(Li[k * p + i] * L[k * p + k], Li[k * p + j], s);
        G[i * p + j] = s;
        G[j * p + i] = s;
      }
    }
  }
  return ok;
}

// Pivots of the LU factorisation (Doolittle, no pivoting) of the FULL matrix F: prod piv = det F as the reference's
// `pt.linalg.det(F)` (kalman_filter.py:281) sees it - every entry, not one triangle.  For a symmetric F these are the
// L D L^T pivots again; the kernels call it only for the first step (the one place F can be non-symmetric, see
// ldl_inverse).  W: p x p scratch.  Returns false if a pivot is not a positive finite number (log det undefined).
template <class TF, class TW, class TP>
KFB_HD bool lu_pivots(const TF& F, TW& W, TP& piv, int p) {
  bool ok = true;
#pragma unroll
  for (int i = 0; i < p * p; ++i) W[i] = F[i];
#pragma unroll
  for (int k = 0; k < p; ++k) {
    const double d = W[k * p + k];
    piv[k] = d;
    ok = ok && (d > 0.0) && (d < 1.0e300);
    const double r = 1.0 / d;
#pragma unroll
    for (int i = 0; i < p; ++i) {
      if (i > k) {
        const double l = W[i * p + k] * r;
#pragma unroll
        for (int j = 0; j < p; ++j)
          if (j > k) W[i * p + j] = kf_fma(-l, W[k * p + j], W[i * p + j]);
      }
    }
  }
  return ok;
}

// Cholesky F = L L^T (lower, full storage) and Li = L^-1, serial (one lane).  Used only by the as-coded
// CholeskyFilter for k_endog > 1 (MK_CHOLS).  logdet <- log det F.
// chol_factor with the squared pivots returned instead of their logarithms (deferred-log accumulation in the fused kernels)
template <class TF, class TL, class TP>
KFB_HD bool chol_factor_piv(const TF& F, TL& L, TL& Li, TP& piv, int p) {
  bool ok = true;
  _Pragma("unroll") for (int j = 0; j < p; ++j) {
    double dj = F[j * p + j];
    _Pragma("unroll") for (int k = 0; k < p; ++k)
      if (k < j) dj -= L[j * p + k] * L[j * p + k];
    ok = ok && (dj > 0.0) && (dj < 1.0e300);
    piv[j] = dj;
    const double lj = sqrt(dj);
    L[j * p + j] = lj;
    _Pragma("unroll") for (int i = 0; i < p; ++i) {
      if (i < j) L[i * p + j] = 0.0;
      if (i > j) {
        double s = F[i * p + j];
        _Pragma("unroll") for (int k = 0; k < p; ++k)
          if (k < j) s -= L[i * p + k] * L[j * p + k];
        L[i * p + j] = s / lj;
      }
    }
  }
  _Pragma("unroll") for (int c = 0; c < p; ++c)
    _Pragma("unroll") for (int i = 0; i < p; ++i) {
      if (i < c) Li[i * p + c] = 0.0;
      else {
        double s = (i == c) ? 1.0 : 0.0;
        _Pragma("unroll") for (int k = 0; k < p; ++k)
          if (k >= c && k < i) s -= L[i * p + k] * Li[k * p + c];
        Li[i * p + c] = s / L[i * p + i];
      }
    }
  return ok;
}

template <class TF, class TL>
KFB_HD bool chol_factor(const TF& F, TL& L, TL& Li, int p, double* logdet) {
  bool ok = true;
  double ld = 0.0;
  _Pragma("unroll") for (int j = 0; j < p; ++j) {
    double dj = F[j * p + j];
    _Pragma("unroll") for (int k = 0; k < j; ++k) dj -= L[j * p + k] * L[j * p + k];
    ok = ok && (dj > 0.0) && (dj < 1.0e300);
    const double lj = sqrt(dj);
    ld += log(dj);
    L[j * p + j] = lj;
    _Pragma("unroll") for (int i = 0; i < p; ++i) {
      if (i < j) L[i * p + j] = 0.0;
      if (i > j) {
        double s = F[i * p + j];
        _Pragma("unroll") for (int k = 0; k < j; ++k) s -= L[i * p + k] * L[j * p + k];
        L[i * p + j] = s / lj;
      }
    }
  }
  _Pragma("unroll") for (int c = 0; c < p; ++c)
    _Pragma("unroll") for (int i = 0; i < p; ++i) {
      if (i < c) Li[i * p + c] = 0.0;
      else {
        double s = (i == c) ? 1.0 : 0.0;
        _Pragma("unroll") for (int k = c; k < i; ++k) s -= L[i * p + k] * Li[k * p + c];
        Li[i * p + c] = s / L[i * p + i];
      }
    }
  *logdet = ld;
  return ok;
}

// Adjoint of the as-coded gain matrix Gk[k][i] = Li[i][k] / L_ii (and of -sum log L_ii) back to F, serial.
//   Gb  cotangent of Gk;  lb cotangent of ll;  W1, W2 scratch (p x p);  Fb <- cotangent of F (symmetrised, the
//   convention of torch.linalg.cholesky; PyTensor folds it into the lower triangle - same symmetric part).
template <class TG, class TL, class TW>
KFB_HD void chols_adjoint(const TG& Gb, const TL& L, const TL& Li, const TG& Gk, double lb, TW& W1, TW& W2, TG& Fb,
                          int p) {
  // W1 = Lib : Lib[i][k] = Gb[k][i] / L_ii
  _Pragma("unroll") for (int i = 0; i < p; ++i)
    _Pragma("unroll") for (int k = 0; k < p; ++k) W1[i * p + k] = Gb[k * p + i] / L[i * p + i];
  // W2 = Lb = -Li^T Lib Li^T
  _Pragma("unroll") for (int i = 0; i < p; ++i)
    _Pragma("unroll") for (int j = 0; j < p; ++j) {
      double s = 0.0;
      _Pragma("unroll") for (int a = 0; a < p; ++a) {
        double t = 0.0;
        _Pragma("unroll") for (int b = 0; b < p; ++b) t += W1[a * p + b] * Li[j * p + b];
        s += Li[a * p + i] * t;
      }
      W2[i * p + j] = -s;
    }
  _Pragma("unroll") for (int i = 0; i < p; ++i) {
    double s = 0.0;
    _Pragma("unroll") for (int k = 0; k < p; ++k) s += Gb[k * p + i] * Gk[k * p + i];
    W2[i * p + i] += -s / L[i * p + i] - lb / L[i * p + i];
  }
  // W1 = Phi = tril(L^T Lb), diagonal halved
  _Pragma("unroll") for (int i = 0; i < p; ++i)
    _Pragma("unroll") for (int j = 0; j < p; ++j) {
      double s = 0.0;
      if (j <= i)
        _Pragma("unroll") for (int k = 0; k < p; ++k) s += L[k * p + i] * W2[k * p + j];
      W1[i * p + j] = (i == j) ? 0.5 * s : s;
    }
  // W2 = S = Li^T Phi Li ; Fb = (S + S^T) / 2
  _Pragma("unroll") for (int i = 0; i < p; ++i)
    _Pragma("unroll") for (int j = 0; j < p; ++j) {
      double s = 0.0;
      _Pragma("unroll") for (int a = 0; a < p; ++a) {
        double t = 0.0;
        _Pragma("unroll") for (int b = 0; b < p; ++b) t += W1[a * p + b] * Li[b * p + j];
        s += Li[a * p + i] * t;
      }
      W2[i * p + j] = s;
    }
  _Pragma("unroll") for (int i = 0; i < p; ++i)
    _Pragma("unroll") for (int j = 0; j < p; ++j) Fb[i * p + j] = 0.5 * (W2[i * p + j] + W2[j * p + i]);
}

// Per-step outputs of the full-output forward pass (the reference's moments and ll_obs, kalman_filter.py:184-191).
// Row r of output array `arr` of unit u lives at base[(u * rows + r) * w .. + w).
enum OutArr : int { O_FS = 0, O_PS = 1, O_FC = 2, O_PC = 3, O_LL = 4 };

KFB_HD double* out_base(const KfArgs& A, int arr) {
  return arr == O_FS ? A.fs : arr == O_PS ? A.ps : arr == O_FC ? A.fc : arr == O_PC ? A.pc : A.ll_obs;
}

// Default (cooperative contexts, host): the lanes of a unit store the row directly - consecutive lanes, consecutive
// doubles.  ThreadCtx overrides this with a shared-memory stager (kf_ctx.cuh): one unit per thread would otherwise
// scatter every 8-byte store into its own sector.
template <class X, class TS>
KFB_HD void store_row_direct(X& x, const KfArgs& A, int arr, long long u, long long rows, long long r, int w, const TS& src) {
  double* base = out_base(A, arr);
  if (!base) return;
  KFB_FOR(i, w) base[(u * rows + r) * w + i] = src[i];
}

// ------------------------------------------------------------------------------------------------
// Per-unit constant parameters + scratch, allocated from the context (registers or shared memory)
// ------------------------------------------------------------------------------------------------
template <class X>
struct Params {
  typename X::template Buf<SZ_MM> T;
  typename X::template Buf<SZ_MP> Z;   // p x m
  typename X::template Buf<SZ_PP> H;
  typename X::template Buf<SZ_P> d;
  typename X::template Buf<SZ_PP> Gss;  // steady state only
  KFB_HD Params(X& x) : T(x), Z(x), H(x), d(x), Gss(x) {}
};

template <class X>
struct UpdTmp {
  typename X::template Buf<SZ_P> v, w, piv;
  typename X::template Buf<SZ_MP> Mm, K, KH;
  typename X::template Buf<SZ_PP> F, Fi, L, Li;
  typename X::template Buf<SZ_MM> A, S1, S2;
  KFB_HD UpdTmp(X& x) : v(x), w(x), piv(x), Mm(x), K(x), KH(x), F(x), Fi(x), L(x), Li(x), A(x), S1(x), S2(x) {}
};

struct StepStat {
  double quad;    // v^T G v
  double logdet;  // only when per-step logs are requested
  bool ok;
};

// Update for an observed row.  MK_STD: StandardFilter / CholeskyFilter(p=1 or corrected) /
// SingleTimeseriesFilter; MK_STEADY: SteadyStateFilter (gain uses the fixed Gss).
// Outputs af, Pf and keeps v, Mm, F, Fi(=F^-1), K, A, w in `u` for the adjoint.
template <int MK, class X, class TA, class TPm>
KFB_HD StepStat update_observed(X& x, const Params<X>& prm, const double* yt, double d_sign, const TA& a,
                                const TPm& P, UpdTmp<X>& u, TA& af, TPm& Pf, LogAcc* acc, bool per_step_log,
                                bool full_det = false) {
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
  x.sync();
  st.ok = true;
  st.logdet = 0.0;
  if (MK == MK_CHOLS) {
    if (x.lane() == 0) {
      double ld = 0.0;
      st.ok = chol_factor(u.F, u.L, u.Li, p, &ld);
      st.logdet = ld;  // -sum log L_ii = -0.5 log det F  (:314)
      for (int k = 0; k < p; ++k)
        for (int i = 0; i < p; ++i) u.Fi[k * p + i] = u.Li[i * p + k] / u.L[i * p + i];  // Gk (SURVEY A.2-Q4)
    }
  } else if (x.lane() == 0) {
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
    gemm<false, false, 0>(x, u.K, u.Mm, prm.Gss, m, p, p);
    KFB_FOR(i, p) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < p; ++j) s = kf_fma(prm.Gss[i * p + j], u.v[j], s);
      u.w[i] = s;
    }
  } else {
    gemm<false, false, 0>(x, u.K, u.Mm, u.Fi, m, p, p);
    KFB_FOR(i, p) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < p; ++j) s = kf_fma(MK == MK_CHOLS ? u.Fi[j * p + i] : u.Fi[i * p + j], u.v[j], s);
      u.w[i] = s;
    }
  }
  KFB_FOR(idx, m * m) {  // A = I - K Z
    const int i = x.div_m(idx), j = idx - i * m;
    double s = (i == j) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 0; k < p; ++k) s = kf_fma(-u.K[i * p + k], prm.Z[k * m + j], s);
    u.A[idx] = s;
  }
  KFB_FOR(i, m) {
    double s = a[i];
#pragma unroll
    for (int k = 0; k < p; ++k) s = kf_fma(u.K[i * p + k], u.v[k], s);
    af[i] = s;
  }
  x.sync();
  double q = 0.0;
#pragma unroll
  for (int i = 0; i < p; ++i) q = kf_fma(u.v[i], u.w[i], q);
  st.quad = q;
  gemm<false, false, 0>(x, u.S1, u.A, P, m, m, m);      // A P
  gemm<false, true, 0>(x, Pf, u.S1, u.A, m, m, m);      // (A P) A^T
  gemm<false, false, 0>(x, u.KH, u.K, prm.H, m, p, p);  // K H
  gemm<false, true, 1>(x, Pf, u.KH, u.K, m, p, m);      // + (K H) K^T   Joseph form :278
  return st;
}

// predict, kalman_filter.py:216-223.  a <- T af + c ; P <- sym(T Pf T^T + C)
template <class X, class TT, class TC, class Tc, class TA, class TPm, class TS>
KFB_HD void predict(X& x, const TT& T, const TC& C, const Tc& c, const TA& af, const TPm& Pf, TA& a, TPm& P, TS& S1,
                    TS& S2) {
  const int m = x.m();
  KFB_FOR(i, m) {
    double s = c[i];
#pragma unroll
    for (int k = 0; k < m; ++k) s = kf_fma(T[i * m + k], af[k], s);
    a[i] = s;
  }
  gemm<false, false, 0>(x, S1, T, Pf, m, m, m);
  KFB_FOR(idx, m * m) S2[idx] = C[idx];
  x.sync();
  gemm<false, true, 1>(x, S2, S1, T, m, m, m);
  KFB_FOR(idx, m * m) {
    const int i = x.div_m(idx), j = idx - i * m;
    P[idx] = 0.5 * (S2[idx] + S2[j * m + i]);
  }
  x.sync();
}

// One inner step of the univariate filter (kalman_filter.py:460-480) on observation i; in place.
// Returns false if the observation is skipped (NaN or F == 0).  Kv <- K, *vo <- v, *Fo <- F.
template <class X, class TA, class TPm, class TK>
KFB_HD bool univariate_inner(X& x, const Params<X>& prm, const double* yt, double d_sign, int i, TA& a, TPm& P, TK& Mv,
                             TK& Kv, double* vo, double* Fo) {
  const int m = x.m(), p = x.p();
  const double yi = yt[i];
  if (kf_isnan(yi)) return false;
  double v = yi - d_sign * prm.d[i];
#pragma unroll
  for (int k = 0; k < m; ++k) v = kf_fma(-prm.Z[i * m + k], a[k], v);
  KFB_FOR(r, m) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < m; ++k) s = kf_fma(P[r * m + k], prm.Z[i * m + k], s);
    Mv[r] = s;
  }
  x.sync();
  double F = prm.H[i * p + i];
#pragma unroll
  for (int k = 0; k < m; ++k) F = kf_fma(prm.Z[i * m + k], Mv[k], F);
  *vo = v;
  *Fo = F;
  // F == 0 is "treated as missing" (:468-471).  Predicated, not branched: with K = 0 every update below is the
  // identity, and control flow stays uniform across units that share a warp (sub-warp cooperative mode).
  const bool live = (F != 0.0);
  const double rF = live ? 1.0 / F : 0.0;
  KFB_FOR(r, m) Kv[r] = Mv[r] * rF;
  x.sync();
  KFB_FOR(idx, m * m) {
    const int r = x.div_m(idx), c = idx - r * m;
    P[idx] = kf_fma(-Kv[r] * Kv[c], F, P[idx]);  // P - K K^T F  (:477, not Joseph)
  }
  KFB_FOR(r, m) a[r] = kf_fma(Kv[r], v, a[r]);
  x.sync();
  return live;
}

template <class X>
KFB_HD int count_missing(X& x, const double* yt) {
  int nm = 0;
#pragma unroll
  for (int i = 0; i < x.p(); ++i) nm += kf_isnan(yt[i]) ? 1 : 0;
  return nm;
}

// ------------------------------------------------------------------------------------------------
// forward recursion for one unit
// ------------------------------------------------------------------------------------------------
// FULL = false: only loglik (+ tape) is produced - the per-leapfrog hot path; all per-step output stores, their
// address arithmetic and the per-step log are compiled out.
template <int MK, bool FULL, class X>
KFB_HD void forward_unit(X& x, const KfArgs& A, long long u) {
  const int m = x.m(), p = x.p(), n = A.n;
  const long long draw = u / A.n_series, series = u - draw * A.n_series;
  const int kt = tape_width(m);
  Params<X> prm(x);
  typename X::template Buf<SZ_MM> C(x), P(x), Pf(x);
  typename X::template Buf<SZ_M> c(x), a(x), af(x), Mv(x), Kv(x);
  UpdTmp<X> tmp(x);

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
    load_or_zero(x, P, A.Pss.p + draw * A.Pss.bs, m * m);  // recursion starts at P_steady (:391, Q7)
    load_or_zero(x, prm.Gss, A.Gss.p + draw * A.Gss.bs, p * p);
  } else {
    load_or_zero(x, P, A.P0.p + draw * A.P0.bs, m * m);
  }
  x.sync();

  const double* y = x.y_base(A, series);
  const bool full = FULL && (A.ll_obs != nullptr);
  const bool lane0 = (x.lane() == 0);
  LogAcc acc;
  double llsum = 0.0;
  int info = 0;

  double* tp = A.tape ? x.tape_base(A, u) : nullptr;  // entry of step t+1 is written at the end of step t
  const long long tstep = x.tape_step(A), telem = x.tape_elem(A);
  if (FULL && A.ps) {
    const double* a0p = A.a0.p + draw * A.a0.bs;
    const double* P0p = A.P0.p + draw * A.P0.bs;
    KFB_FOR(i, m) A.ps[(u * (n + 1)) * m + i] = a0p[i];
    if (A.pc) KFB_FOR(i, m * m) A.pc[(u * (n + 1)) * m * m + i] = P0p[i];
  }

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
    double ll_t = 0.0;
    if (MK == MK_UNIV) {
      KFB_FOR(i, m) af[i] = a[i];
      KFB_FOR(i, m * m) Pf[i] = P[i];
      x.sync();
      double s = 0.0;
      int cnt = 0;
      for (int i = 0; i < p; ++i) {
        double v, F;
        if (univariate_inner(x, prm, yt, A.d_sign, i, af, Pf, Mv, Kv, &v, &F)) {
          if (!(F > 0.0) && info == 0) info = t + 1;
          double li = v * v / F;
          if (full) {
            li += log(F);
            cnt += (li != 0.0) ? 1 : 0;  // (ll_inner != 0).sum(), :503
          } else {
            if (F > 0.0 && F < 1.0e300 && lane0) acc.mul(F);
            cnt += 1;
          }
          s += li;
        }
      }
      ll_t = -0.5 * (cnt * KF_LOG_2PI + s);
    } else {
      const int nm = count_missing(x, yt);
      if (nm == 0) {
        StepStat st = update_observed<MK>(x, prm, yt, A.d_sign, a, P, tmp, af, Pf, &acc, full, MK == MK_STD && t == 0);
        if (!st.ok && info == 0) info = t + 1;
        ll_t = -0.5 * (A.ll_const + st.logdet + st.quad);
      } else {
        if (nm != p && info == 0) info = -(t + 1);  // partial row: reference raises (A.2-Q2)
        KFB_FOR(i, m) af[i] = a[i];                 // all missing: K = 0, a_f = a, P_f = P, ll = 0
        KFB_FOR(i, m * m) Pf[i] = P[i];
        x.sync();
      }
    }
    llsum += ll_t;
    if (FULL) {
      if (full) {
        const double llv[1] = {ll_t};
        x.store_row(A, O_LL, u, n, t, 1, llv);
      }
      x.store_row(A, O_FS, u, n, t, m, af);
      x.store_row(A, O_FC, u, n, t, m * m, Pf);
    }
    predict(x, prm.T, C, c, af, Pf, a, P, tmp.S1, tmp.S2);
    if (FULL) {
      x.store_row(A, O_PS, u, n + 1, t + 1, m, a);
      x.store_row(A, O_PC, u, n + 1, t + 1, m * m, P);
      x.end_step(A, u, t, n);
    }
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
    double ll = llsum;
    if (!full) ll -= 0.5 * acc.value();
    if (info != 0) ll = nan("");
    if (A.loglik) A.loglik[u] = ll;
    if (MK == MK_STEADY && A.dare_info && A.dare_info[draw] != 0) info = KF_INFO_DARE_FAILED;
    if (A.info) A.info[u] = info;
  }
}

// ------------------------------------------------------------------------------------------------
// adjoint recursion for one unit (SURVEY.md appendix B)
// ------------------------------------------------------------------------------------------------
template <int MK, class X>
KFB_HD void backward_unit(X& x, const KfArgs& A, long long u) {
  const int m = x.m(), p = x.p(), n = A.n;
  const long long draw = u / A.n_series, series = u - draw * A.n_series;
  const int kt = tape_width(m);
  Params<X> prm(x);
  typename X::template Buf<SZ_MM> P(x), Pf(x), Pb(x), Pfb(x), Tb(x), Cb(x), S3(x), S4(x);
  typename X::template Buf<SZ_M> a(x), af(x), ab(x), afb(x), cb(x), Mv(x), Kv(x), Mvb(x);
  typename X::template Buf<SZ_MP> Zb(x), Kb(x), Mb(x), PK(x);
  typename X::template Buf<SZ_PP> Hb(x), Fb(x), Gb(x), Q1(x);
  typename X::template Buf<SZ_P> db(x), vb(x);
  UpdTmp<X> tmp(x);

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
  // Tape read-ahead (X::TapeReader): entries of steps t-1, t-2, ... are already in flight while step t is being
  // processed, so the HBM latency of the strictly sequential adjoint recursion is hidden behind arithmetic.
  typename X::template Buf<SZ_TAPE> nxt(x);
  typename X::TapeReader rd(x, A, u);
  for (int t = n - 1; t >= 0; --t) {
    if (X::TV) {
      if (A.T.ts) load_or_zero(x, prm.T, Tp + t * A.T.ts, m * m);
      if (A.Z.ts) load_or_zero(x, prm.Z, Zp + t * A.Z.ts, p * m);
      if (A.H.ts) load_or_zero(x, prm.H, Hp + t * A.H.ts, p * p);
      if (A.d.ts) load_or_zero(x, prm.d, dp + t * A.d.ts, p);
      x.sync();
    }
    // predicted moments entering step t
    if (t == 0) {
      load_or_zero(x, a, A.a0.p + draw * A.a0.bs, m);
      if (MK == MK_STEADY) load_or_zero(x, P, A.Pss.p + draw * A.Pss.bs, m * m);
      else load_or_zero(x, P, A.P0.p + draw * A.P0.bs, m * m);
    } else {
      rd.get(x, nxt);  // entry of step t
      KFB_FOR(k, m) a[k] = nxt[k];
      KFB_FOR(idx, m * m) {
        int i = x.div_m(idx), j = idx - i * m;
        if (j < i) { const int s = i; i = j; j = s; }
        P[idx] = nxt[m + i * m - (i * (i - 1)) / 2 + (j - i)];
      }
    }
    x.sync();
    const double* yt = y + (long long)t * p;
    const double lb = gl + (A.g_ll_obs ? A.g_ll_obs[u * n + t] : 0.0);  // cotangent of ll_t

    bool observed = false;
    if (MK == MK_UNIV) {
      KFB_FOR(i, m) af[i] = a[i];
      KFB_FOR(i, m * m) Pf[i] = P[i];
      x.sync();
      for (int i = 0; i < p; ++i) {
        double v, F;
        univariate_inner(x, prm, yt, A.d_sign, i, af, Pf, Mv, Kv, &v, &F);
      }
    } else {
      observed = (count_missing(x, yt) == 0);
      if (observed) {
        update_observed<MK>(x, prm, yt, A.d_sign, a, P, tmp, af, Pf, (LogAcc*)nullptr, false);
      } else {
        KFB_FOR(i, m) af[i] = a[i];
        KFB_FOR(i, m * m) Pf[i] = P[i];
        x.sync();
      }
    }

    // ---- adjoint of predict: a' = T af + c ; P' = sym(T Pf T^T + C)
    KFB_FOR(idx, m * m) {  // S3 = Ps = sym(Pb) ; S4 = Pf + Pf^T
      const int i = x.div_m(idx), j = idx - i * m;
      S3[idx] = 0.5 * (Pb[idx] + Pb[j * m + i]);
      S4[idx] = Pf[idx] + Pf[j * m + i];
    }
    x.sync();
    KFB_FOR(idx, m * m) Cb[idx] += S3[idx];
    KFB_FOR(i, m) cb[i] += ab[i];
    gemm<false, false, 0>(x, tmp.S1, S3, prm.T, m, m, m);    // W = Ps T        (shared by Tb and Pfb)
    gemm<false, false, 1>(x, Tb, tmp.S1, S4, m, m, m);       // Tb += Ps T (Pf + Pf^T)
    KFB_FOR(idx, m * m) {
      const int i = x.div_m(idx), j = idx - i * m;
      Tb[idx] = kf_fma(ab[i], af[j], Tb[idx]);               // + ab af^T
    }
    KFB_FOR(i, m) {                                          // afb = T^T ab
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < m; ++k) s = kf_fma(prm.T[k * m + i], ab[k], s);
      afb[i] = s;
    }
    gemm<true, false, 0>(x, Pfb, prm.T, tmp.S1, m, m, m);    // Pfb = T^T Ps T
    if (X::TV) {
      if (A.T.ts && A.gT) { KFB_FOR(i, m * m) { A.gT[(u * n + t) * m * m + i] = Tb[i]; Tb[i] = 0.0; } }
      if (A.C.ts && A.gC) { KFB_FOR(i, m * m) { A.gC[(u * n + t) * m * m + i] = Cb[i]; Cb[i] = 0.0; } }
      if (A.c.ts && A.gc) { KFB_FOR(i, m) { A.gc[(u * n + t) * m + i] = cb[i]; cb[i] = 0.0; } }
      x.sync();
    }

    if (MK == MK_UNIV) {
      // reverse the p sequential scalar updates; intermediate (a,P) are recomputed from (a,P)
      for (int i = p - 1; i >= 0; --i) {
        KFB_FOR(k, m) af[k] = a[k];
        KFB_FOR(k, m * m) Pf[k] = P[k];
        x.sync();
        double v = 0.0, F = 1.0;
        for (int i2 = 0; i2 < i; ++i2) univariate_inner(x, prm, yt, A.d_sign, i2, af, Pf, Mv, Kv, &v, &F);
        // (af, Pf) = state before inner update i.  Recompute its pieces without modifying them.
        const double yi = yt[i];
        if (kf_isnan(yi)) continue;
        v = yi - A.d_sign * prm.d[i];
#pragma unroll
        for (int k = 0; k < m; ++k) v = kf_fma(-prm.Z[i * m + k], af[k], v);
        KFB_FOR(r, m) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(Pf[r * m + k], prm.Z[i * m + k], s);
          Mv[r] = s;
        }
        x.sync();
        F = prm.H[i * p + i];
#pragma unroll
        for (int k = 0; k < m; ++k) F = kf_fma(prm.Z[i * m + k], Mv[k], F);
        const double rF = (F != 0.0) ? 1.0 / F : 0.0;  // F == 0: K = 0 and every contribution below vanishes
        KFB_FOR(r, m) Kv[r] = Mv[r] * rF;
        x.sync();
        const double lq = -0.5 * lb;  // cotangent of ll_inner_i
        // Kb = afb v - (Pfb + Pfb^T) K F
        KFB_FOR(r, m) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(Pfb[r * m + k] + Pfb[k * m + r], Kv[k], s);
          Mvb[r] = kf_fma(afb[r], v, -s * F);  // holds Kb
        }
        x.sync();
        double ktab = 0.0, kpk = 0.0, kbk = 0.0;
#pragma unroll
        for (int r = 0; r < m; ++r) {
          ktab = kf_fma(Kv[r], afb[r], ktab);
          kbk = kf_fma(Mvb[r], Kv[r], kbk);
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(Pfb[r * m + k], Kv[k], s);
          kpk = kf_fma(Kv[r], s, kpk);
        }
        const double vbar = ktab + lq * 2.0 * v * rF;
        const double Fbar = -kpk + lq * (rF - v * v * rF * rF) - kbk * rF;
        x.sync();
        KFB_FOR(r, m) Mvb[r] = kf_fma(prm.Z[i * m + r], Fbar, Mvb[r] * rF);  // Mvb = Kb / F + z Fbar
        x.sync();
        if (x.lane() == 0) {
          Hb[i * p + i] += Fbar;
          db[i] -= A.d_sign * vbar;
        }
        KFB_FOR(r, m) {  // Zb row i += Mv Fbar + Pf^T Mvb - vbar a
          double s = kf_fma(Mv[r], Fbar, -vbar * af[r]);
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(Pf[k * m + r], Mvb[k], s);
          Zb[i * m + r] += s;
        }
        KFB_FOR(idx, m * m) {
          const int r = x.div_m(idx), c2 = idx - r * m;
          Pfb[idx] = kf_fma(Mvb[r], prm.Z[i * m + c2], Pfb[idx]);
        }
        KFB_FOR(r, m) afb[r] = kf_fma(-prm.Z[i * m + r], vbar, afb[r]);
        x.sync();
      }
      KFB_FOR(i, m) ab[i] = afb[i];
      KFB_FOR(i, m * m) Pb[i] = Pfb[i];
      x.sync();
    } else if (!observed) {
      KFB_FOR(i, m) ab[i] = afb[i];
      KFB_FOR(i, m * m) Pb[i] = Pfb[i];
      x.sync();
    } else {
      // ---- adjoint of the Joseph update
      KFB_FOR(idx, m * m) {
        const int i = x.div_m(idx), j = idx - i * m;
        S4[idx] = P[idx] + P[j * m + i];
      }
      x.sync();
      gemm<false, false, 0>(x, tmp.S1, Pfb, tmp.A, m, m, m);  // Pfb A            (shared by Ab and Pb)
      gemm<false, false, 0>(x, S3, tmp.S1, S4, m, m, m);      // Ab = Pfb A (P + P^T)      (S3 = Ab)
      gemm<true, false, 0>(x, Pb, tmp.A, tmp.S1, m, m, m);    // Pb = A^T Pfb A
      KFB_FOR(idx, p * p) {
        const int i = x.div_p(idx), j = idx - i * p;
        Q1[idx] = prm.H[idx] + prm.H[j * p + i];
      }
      gemm<false, false, 0>(x, PK, Pfb, tmp.K, m, m, p);      // Pfb K            (shared by Kb and Hb)
      gemm<false, false, 0>(x, Kb, PK, Q1, m, p, p);          // Kb = Pfb K (H + H^T)
      KFB_FOR(idx, m * p) {
        const int i = x.div_p(idx), j = idx - i * p;
        double s = kf_fma(afb[i], tmp.v[j], Kb[idx]);         // + afb v^T
#pragma unroll
        for (int k = 0; k < m; ++k) s = kf_fma(-S3[i * m + k], prm.Z[j * m + k], s);  // - Ab Z^T
        Kb[idx] = s;
      }
      gemm<true, false, 1>(x, Hb, tmp.K, PK, p, m, p);        // Hb += K^T Pfb K
      gemm<true, false, 2>(x, Zb, tmp.K, S3, p, m, m);        // Zb -= K^T Ab
      // vb, Fb
      if (MK == MK_STEADY) {
        KFB_FOR(i, p) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(tmp.K[k * p + i], afb[k], s);
#pragma unroll
          for (int j = 0; j < p; ++j) s = kf_fma(-0.5 * lb * (prm.Gss[i * p + j] + prm.Gss[j * p + i]), tmp.v[j], s);
          vb[i] = s;
        }
        gemm<true, false, 1>(x, Gb, tmp.Mm, Kb, p, m, p);     // Gssb += Mm^T Kb
        KFB_FOR(idx, p * p) {
          const int i = x.div_p(idx), j = idx - i * p;
          Gb[idx] = kf_fma(-0.5 * lb * tmp.v[i], tmp.v[j], Gb[idx]);
          Fb[idx] = -0.5 * lb * tmp.Fi[j * p + i];
        }
        x.sync();
        gemm<false, true, 0>(x, Mb, Kb, prm.Gss, m, p, p);    // Mb = Kb Gss^T
      } else if (MK == MK_CHOLS) {
        KFB_FOR(i, p) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(tmp.K[k * p + i], afb[k], s);
          for (int j = 0; j < p; ++j) s = kf_fma(-0.5 * lb * (tmp.Fi[i * p + j] + tmp.Fi[j * p + i]), tmp.v[j], s);
          vb[i] = s;
        }
        gemm<true, false, 0>(x, Q1, tmp.Mm, Kb, p, m, p);     // Gk-bar = Mm^T Kb - 0.5 lb v v^T
        KFB_FOR(idx, p * p) {
          const int i = x.div_p(idx), j = idx - i * p;
          Q1[idx] = kf_fma(-0.5 * lb * tmp.v[i], tmp.v[j], Q1[idx]);
        }
        x.sync();
        if (x.lane() == 0) chols_adjoint(Q1, tmp.L, tmp.Li, tmp.Fi, lb, tmp.F, Gb, Fb, p);
        x.sync();
        gemm<false, true, 0>(x, Mb, Kb, tmp.Fi, m, p, p);     // Mb = Kb Gk^T
      } else {
        KFB_FOR(i, p) {
          double s = -lb * tmp.w[i];
#pragma unroll
          for (int k = 0; k < m; ++k) s = kf_fma(tmp.K[k * p + i], afb[k], s);
          vb[i] = s;
        }
        gemm<true, false, 0>(x, Q1, tmp.K, Kb, p, m, p);      // K^T Kb
        KFB_FOR(idx, p * p) {
          const int i = x.div_p(idx), j = idx - i * p;
          double s = -0.5 * lb * (tmp.Fi[j * p + i] - tmp.w[i] * tmp.w[j]);
#pragma unroll
          for (int k = 0; k < p; ++k) s = kf_fma(-Q1[i * p + k], tmp.Fi[j * p + k], s);  // - K^T Kb G^T
          Fb[idx] = s;
        }
        x.sync();
        gemm<false, true, 0>(x, Mb, Kb, tmp.Fi, m, p, p);     // Mb = Kb G^T
      }
      gemm<true, false, 1>(x, Mb, prm.Z, Fb, m, p, p);        // Mb += Z^T Fb
      KFB_FOR(idx, p * m) {                                   // Zb += Fb Mm^T + Mb^T P - vb a^T
        const int i = x.div_m(idx), j = idx - i * m;
        double s = kf_fma(-vb[i], a[j], Zb[idx]);
#pragma unroll
        for (int k = 0; k < p; ++k) s = kf_fma(Fb[i * p + k], tmp.Mm[j * p + k], s);
#pragma unroll
        for (int k = 0; k < m; ++k) s = kf_fma(Mb[k * p + i], P[k * m + j], s);
        Zb[idx] = s;
      }
      KFB_FOR(idx, p * p) Hb[idx] += Fb[idx];
      gemm<false, false, 1>(x, Pb, Mb, prm.Z, m, p, m);       // Pb += Mb Z
      KFB_FOR(i, m) {                                         // ab = afb - Z^T vb
        double s = afb[i];
#pragma unroll
        for (int k = 0; k < p; ++k) s = kf_fma(-prm.Z[k * m + i], vb[k], s);
        ab[i] = s;
      }
      KFB_FOR(i, p) db[i] = kf_fma(-A.d_sign, vb[i], db[i]);
      x.sync();
    }
    if (X::TV) {
      if (A.Z.ts && A.gZ) { KFB_FOR(i, p * m) { A.gZ[(u * n + t) * p * m + i] = Zb[i]; Zb[i] = 0.0; } }
      if (A.H.ts && A.gH) { KFB_FOR(i, p * p) { A.gH[(u * n + t) * p * p + i] = Hb[i]; Hb[i] = 0.0; } }
      if (A.d.ts && A.gd) { KFB_FOR(i, p) { A.gd[(u * n + t) * p + i] = db[i]; db[i] = 0.0; } }
      x.sync();
    }
  }
  if (A.ga0) KFB_FOR(i, m) A.ga0[u * m + i] = ab[i];
  if (MK == MK_STEADY) {
    if (A.gPss) KFB_FOR(i, m * m) A.gPss[u * m * m + i] = Pb[i];
    if (A.gGss) KFB_FOR(i, p * p) A.gGss[u * p * p + i] = Gb[i];
    if (A.gP0) KFB_FOR(i, m * m) A.gP0[u * m * m + i] = 0.0;  // Q7: P0 is not used by the recursion
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
