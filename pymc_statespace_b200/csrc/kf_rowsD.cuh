// kf_rowsD.cuh - mid-size and large systems (even k_states 10..32; k_endog = 1 instantiated; MK_STD / MK_STEADY; static
// matrices; shared observation stream; config 4 of BASELINE.json: trend + seasonal, k_states = 30): one WARP per unit, the
// m x m x m products on the FP64 TENSOR CORES (mma.sync.m8n8k4.f64, "DMMA"), everything else row-per-lane as in kf_rows.cuh.
//
// Why: with DFMA every multiply-add needs at least one operand from shared memory and a broadcast load delivers one
// double per wavefront, so the warp-per-unit DFMA kernel of round 1 sat at 94 % of the
// shared-memory wavefront peak with the fp64 pipe 35 % active (profiles/r1_ncu_rowsL.md).  A DMMA consumes one A and one
// B element per lane for eight multiply-adds per lane, and a fragment is reused for NT tiles: ~0.06 shared-memory operands
// per multiply-add.  tools/dmma_probe.cu measured 37.1 TFLOP/s for register-operand DMMA on this B200 - the same as the
// DFMA peak - already at one warp per SM sub-partition with four independent accumulator tiles.
//
// Matrices live in shared memory as NT x NT tiles of 8 x 8 (NT = 4 for k_states 18..32, NT = 2 for 10..16) with leading
// dimension 8 NT + 2 (LD = 36 at NT = 4 makes the fragment loads conflict-free instead but 2-way conflicts every row
// access: measured 357 ms vs 326 ms per evaluation of config 4; LD = 38: 332 ms).  Rows / columns >= m are zero and stay
// zero (products of zero padding).  Transposed operands cost nothing: A^T / B^T just swap the two fragment access patterns.
#pragma once
#include "kf_core.cuh"
#include "kf_rows.cuh"

namespace kfb {

// Tile geometry: NT x NT tiles of 8 x 8 per matrix (NT = 4: even k_states 18..32; NT = 2: even k_states 10..16 - seasonal
// periods 12 / SARIMA orders land here).
//  * NT = 4: leading dimension LD = 34 doubles: rows 16-byte aligned and LD/2 odd, so the row-per-lane 16-byte accesses of a
//    quarter warp fall on 8 distinct bank groups; fragment loads and tile stores are 2-way conflicted.  (The XOR-swizzled
//    layout below makes all access patterns conflict free there too and was measured slower twice - rounds 1 and 2,
//    profiles/r2_ncu_rowsD.md: at 1.5 warps per scheduler its address arithmetic turns the kernels latency-bound.)
//  * NT = 2: LD = 16 and the 16-byte chunks of a row XOR-swizzled: physical chunk = chunk ^ swz(row),
//    swz(row) = {0,4,2,6,1,5,3,7}[row & 7].  Row accesses (8 consecutive rows -> 8 distinct chunk groups), both mma
//    fragment patterns and the 16-byte tile stores are all conflict free.  These kernels run 12-16 warps per SM and sat ON
//    the shared-memory wavefront roof (93-96 % of the LSU peak), a quarter of it bank conflicts at LD = 18: 478 -> 323
//    (forward) / 696 -> 537 (adjoint) wavefronts per step together with the predicated row loads; the full-output forward
//    gained 14 %, the adjoint little (it is then bound by spills at 128 registers: see ROWSH_MIN_BLOCKS in kf_kernels.cuh).
__host__ __device__ constexpr int rowsD_nt(int m) { return m <= 16 ? 2 : 4; }
__host__ __device__ constexpr int rowsD_ld(int m) { return m <= 16 ? 16 : 34; }
template <int LD>
__host__ __device__ constexpr int rowsD_swz(int row) {
  return (LD % 8 == 0) ? (((row & 1) << 2) | (row & 2) | ((row >> 2) & 1)) : 0;
}
// offset of element (row, col) inside a tile matrix
template <int LD>
__host__ __device__ constexpr int rowsD_el(int row, int col) {
  return row * LD + ((((col >> 1) ^ rowsD_swz<LD>(row)) << 1) | (col & 1));
}

template <int M, int P, bool NEED_T>
struct RowsDLayout {
  static_assert(M % 2 == 0 && M >= 10 && M <= 32 && P <= 3, "even k_states in 10..32");
  static constexpr int NT = rowsD_nt(M), TD = 8 * NT, LD = rowsD_ld(M), MS = TD * LD;  // one padded matrix
  static constexpr int MP = M * P, PP = P * P, MPE = MP + (MP & 1), ME = M + (M & 1);
  static constexpr int MPT = TD * P;  // vectors that the mma-fragment-layout code reads by padded row (rows >= M stay 0)
  static constexpr int KT = M + (M * (M + 1)) / 2, KTP = (KT + 1) & ~1;
  static constexpr int T = 0, Pm = T + MS, Lm = Pm + MS, Z = Lm + MS, H = Z + MPE, Mm = H + PP + (PP & 1), Kp = Mm + MPT,
                       a = Kp + MPE, END_COMMON = a + TD;
  // forward only: X (then S2) ; KH rows
  static constexpr int X = END_COMMON, KH = X + MS, END_FWD = KH + MPE;
  // adjoint only: W = Ps L lives in Pm's slot (without T-bar nothing reads P after the gain) or in its own (with T-bar:
  // T-bar += 2 W P).  lz: (P0 + P0^T) Z^T, t = 0 only.  Mb: the rank-p part of P-bar, kept apart from L^T W.
  static constexpr int Pb = END_COMMON, Kb = Pb + MS, TMb = Kb + MPE, PK = TMb + MPT, lz = PK + MPE, TMs = lz + MPE,
                       ab = TMs + MPE, Mb = ab + TD, Xb = Mb + MPE, END_BWD = Xb + (NEED_T ? MS : 0),
                       W = NEED_T ? Xb : Pm;
  // The tape entry of the NEXT step is staged in Lm's slot, which is free from the last product of a step (phase 3) to
  // the next step's gain: no staging buffer of its own, 37.5 instead of 41.5 KB per unit = 6 instead of 5 units per SM.
  // It clobbers the zero padding of Lm's first rows: the adjoint's gain rewrites its rows including the padding columns.
  static constexpr int tp = Lm;
  static_assert(KTP <= M * LD, "the staged tape entry must not reach the zero rows of Lm");
  static constexpr int fwd_doubles = (END_FWD + 1) & ~1, bwd_doubles = (END_BWD + 1) & ~1;
};

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
#ifdef __CUDA_ARCH__
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
#endif
}

// acc (8 NT x 8 NT, as NT x NT tiles of 8 x 8 in mma fragment layout: lane holds [8I + lane/4][8J + 2 (lane%4) + {0,1}])
//   = op(A) op(B),  op = transpose if TA / TB.  A, B: padded row-major matrices (leading dimension LD) in shared memory.
// ZERO = false: accumulate onto acc.  UPPER: only the tiles I <= J (the result is symmetric and its consumer reads it
// through rowD_load_symU): 10 instead of 16 tile products at NT = 4.
template <bool TA, bool TB, int LD, bool ZERO = true, bool UPPER = false, int NT = LD / 8>
__device__ __forceinline__ void mm32(double (&acc)[NT][NT][2], const double* A, const double* B, int lane) {
  constexpr bool SWZ = (LD % 8 == 0);
  const int r = lane >> 2, c = lane & 3;
  // "N" pattern: element (row 8X + r, col 4kk + c) ; "T" pattern: element (row 4kk + c, col 8X + r)
  //   A: N, A^T: T (a[row][k] = A[k][row]) ; B: T pattern on B (b[k][col] = B[k][col]), B^T: N pattern on B
  const int sr = rowsD_swz<LD>(r);                          // swizzle of rows 8X + r
  const int gc = SWZ ? (((c & 1) << 2) | (c & 2)) : 0;      // swizzle of rows 4kk + c = gc | (kk & 1)
  const double* nA = A + r * LD + (c & 1);
  const double* nB = B + r * LD + (c & 1);
  const double* tA = A + c * LD + (r & 1);
  const double* tB = B + c * LD + (r & 1);
  if (ZERO) {
#pragma unroll
    for (int I = 0; I < NT; ++I)
#pragma unroll
      for (int J = 0; J < NT; ++J) acc[I][J][0] = acc[I][J][1] = 0.0;
  }
#pragma unroll
  for (int kk = 0; kk < 2 * NT; ++kk) {
    double af[NT], bf[NT];
    const int nofs = ((2 * kk + (c >> 1)) ^ sr) << 1;  // N pattern: chunk 2kk + c/2 of the lane's row
    const int st = gc | (SWZ ? (kk & 1) : 0);
#pragma unroll
    for (int I = 0; I < NT; ++I)
      af[I] = TA ? tA[(4 * kk) * LD + (((4 * I + (r >> 1)) ^ st) << 1)] : nA[(8 * I) * LD + nofs];
#pragma unroll
    for (int J = 0; J < NT; ++J)
      bf[J] = TB ? nB[(8 * J) * LD + nofs] : tB[(4 * kk) * LD + (((4 * J + (r >> 1)) ^ st) << 1)];
#pragma unroll
    for (int I = 0; I < NT; ++I)
#pragma unroll
      for (int J = 0; J < NT; ++J)
        if (!UPPER || I <= J) dmma884(acc[I][J][0], acc[I][J][1], af[I], bf[J]);
  }
}

// D = alpha * acc (the full padded matrix including the zero padding; UPPER: the tiles I <= J only)
template <int LD, bool UPPER = false, int NT = LD / 8>
__device__ __forceinline__ void mm32_store(double* D, const double (&acc)[NT][NT][2], double alpha, int lane) {
  // D may be one of the product's own operands (X <- X L^T, A <- A A): every fragment load is
  // behind an mma.sync that consumed it, but make the ordering explicit (and visible to racecheck)
  __syncwarp();
  const int r = lane >> 2, c = lane & 3;
#pragma unroll
  for (int I = 0; I < NT; ++I)
#pragma unroll
    for (int J = 0; J < NT; ++J)
      if (!UPPER || I <= J)
        *reinterpret_cast<double2*>(D + (8 * I + r) * LD + (((4 * J + c) ^ rowsD_swz<LD>(r)) << 1)) =
            make_double2(alpha * acc[I][J][0], alpha * acc[I][J][1]);
}

// row i of a tile matrix: rowp = &mat[i * LD]; logical chunk j (elements 2j, 2j + 1) lives at chunk j ^ swz(i)
template <int LD>
__device__ __forceinline__ const double2* rowD_chunk(const double* rowp, int i, int j) {
  return reinterpret_cast<const double2*>(rowp + ((j ^ rowsD_swz<LD>(i)) << 1));
}
template <int LD>
__device__ __forceinline__ double2* rowD_chunk(double* rowp, int i, int j) {
  return reinterpret_cast<double2*>(rowp + ((j ^ rowsD_swz<LD>(i)) << 1));
}
template <int M, int LD>
__device__ __forceinline__ void rowD_store(double* rowp, int i, const double (&v)[M]) {
#pragma unroll
  for (int j = 0; j < M / 2; ++j) *rowD_chunk<LD>(rowp, i, j) = make_double2(v[2 * j], v[2 * j + 1]);
}
// act = false (a lane without a row, lanes >= k_states): no load is issued - 16-byte accesses are served per quarter warp,
// so at k_states <= 16 the idle half of the warp would otherwise double the wavefronts of every row load.
template <int M, int LD>
__device__ __forceinline__ void rowD_load(double (&v)[M], const double* rowp, int i, bool act = true) {
#pragma unroll
  for (int j = 0; j < M / 2; ++j) {
    const double2 x = act ? *rowD_chunk<LD>(rowp, i, j) : make_double2(0.0, 0.0);
    v[2 * j] = x.x;
    v[2 * j + 1] = x.y;
  }
}
// element (row j, column i) of a tile matrix, j a compile-time constant after unrolling: the lane's COLUMN accesses
template <int LD>
__device__ __forceinline__ double colD(const double* mat, int j, int i) {
  return mat[j * LD + ((((i >> 1) ^ rowsD_swz<LD>(j)) << 1) | (i & 1))];
}

// The lane's row i of sym(U) for a matrix U = A^T S A (S symmetric) of which only the 8 x 8 tiles I <= J were computed
// (mm32<.., UPPER>): entries right of the lane's diagonal tile come from its row, entries left of it from its column
// (the mirrored tile), the diagonal tile is averaged.  Exactly symmetric by construction, and the loads of the tiles a
// lane does not need are predicated off (whole 8-lane groups: fewer shared-memory wavefronts than the full row + column).
template <int M, int LD>
__device__ __forceinline__ void rowD_load_symU(double (&v)[M], const double* mat, int i, bool act = true) {
  const int ti = act ? (i >> 3) : 4;  // a lane without a row loads nothing from the row part
  const double* rowp = mat + i * LD;
#pragma unroll
  for (int j = 0; j < M / 2; ++j) {
    double2 x = make_double2(0.0, 0.0);
    if (((2 * j) >> 3) >= ti) x = *rowD_chunk<LD>(rowp, i, j);
    v[2 * j] = x.x;
    v[2 * j + 1] = x.y;
  }
#pragma unroll
  for (int j = 0; j < M; ++j) {
    if ((j >> 3) <= ti) {
      const double cj = colD<LD>(mat, j, i);
      v[j] = ((j >> 3) < ti) ? cj : 0.5 * (v[j] + cj);
    }
  }
}

// init + sum_{k<N} x_k y_k with four interleaved partial sums.  With one warp per SM sub-partition nothing hides the
// ~30-cycle dependent-issue latency of a DFMA chain: a length-30 dot product as ONE chain is ~1000 cycles, and the
// row-wise phases of a step contain about ten of them (they were ~2/3 of the step time in the first version).
template <int N, class F>
__device__ __forceinline__ double dot4(double init, F f) {
  double s[4] = {init, 0.0, 0.0, 0.0};
#pragma unroll
  for (int k = 0; k < N; ++k) {
    double x, y;
    f(k, x, y);
    s[k & 3] = fma(x, y, s[k & 3]);
  }
  return (s[0] + s[1]) + (s[2] + s[3]);
}

template <int M, int P>
struct RowDGain {
  double Kp[P], TM[P], Fi[P * P], v[P], w[P], piv[P], quad;
  bool ok;
};

// v, Mm | TM, F, F^-1, w, quad, Kp, Lm for an observed step (row-per-lane).  Leaves Mm, Kp, Lm in shared memory (visible
// after the trailing sync); returns the lane's Kp row and (every lane) v, F^-1, w.
// MK_STEADY: the gain matrix is the fixed Gss = (Z Pss Z^T + H)^-1 instead of F^-1 (F is still factorised for log det).
// IDT: T := I, i.e. the FILTER gain K = P Z^T F^-1 and A = I - K Z in Kp / Lm (full-output forward pass).
template <int M, int P, int MK, class L, bool PADL = false, bool IDT = false>
__device__ __forceinline__ void rowsD_gain(double* sm, const double (&yt)[P], double d_sign, const double (&dv)[P],
                                           const double (&Gss)[P * P], int i, bool act, RowDGain<M, P>& g,
                                           bool full_det = false) {
  constexpr int LD = L::LD;
  // ---- A: Mm row (own P row x Z rows), v (every lane)
  {
    double Mr[P][4], vr[P][4];  // four partial sums each (see dot4)
#pragma unroll
    for (int j = 0; j < P; ++j) {
#pragma unroll
      for (int q = 0; q < 4; ++q) Mr[j][q] = vr[j][q] = 0.0;
      vr[j][0] = yt[j] - d_sign * dv[j];
    }
    const double* pr = sm + L::Pm + i * LD;
    const double2* av = reinterpret_cast<const double2*>(sm + L::a);
#pragma unroll
    for (int k = 0; k < M / 2; ++k) {
      const double2 pk = act ? *rowD_chunk<LD>(pr, i, k) : make_double2(0.0, 0.0), ak = av[k];
      const int q = (k & 1) * 2;
#pragma unroll
      for (int j = 0; j < P; ++j) {
        const double2 z = *reinterpret_cast<const double2*>(sm + L::Z + j * M + 2 * k);
        Mr[j][q] = fma(pk.x, z.x, Mr[j][q]);
        Mr[j][q + 1] = fma(pk.y, z.y, Mr[j][q + 1]);
        vr[j][q] = fma(-z.x, ak.x, vr[j][q]);
        vr[j][q + 1] = fma(-z.y, ak.y, vr[j][q + 1]);
      }
    }
#pragma unroll
    for (int j = 0; j < P; ++j) {
      g.v[j] = (vr[j][0] + vr[j][1]) + (vr[j][2] + vr[j][3]);
      if (act) sm[L::Mm + i * P + j] = (Mr[j][0] + Mr[j][1]) + (Mr[j][2] + Mr[j][3]);
    }
  }
  __syncwarp();
  // ---- B: TM row, F (every lane), inverse, w, quad, Kp row, Lm row
  double Fr[P * P], Lr[P * P], Lir[P * P], TM[P];
  {
    double Fq[P * P][4], Tq[P][4];  // four partial sums each (see dot4)
#pragma unroll
    for (int k = 0; k < P * P; ++k) {
      Fq[k][0] = sm[L::H + k];
      Fq[k][1] = Fq[k][2] = Fq[k][3] = 0.0;
    }
#pragma unroll
    for (int j = 0; j < P; ++j) Tq[j][0] = Tq[j][1] = Tq[j][2] = Tq[j][3] = 0.0;
    const double* tr = sm + L::T + i * LD;
#pragma unroll
    for (int k = 0; k < M / 2; ++k) {
      const double2 tk = (act && !IDT) ? *rowD_chunk<LD>(tr, i, k) : make_double2(0.0, 0.0);
      const int q = (k & 1) * 2;
#pragma unroll
      for (int j = 0; j < P; ++j) {
        const double m0 = sm[L::Mm + (2 * k) * P + j], m1 = sm[L::Mm + (2 * k + 1) * P + j];
        Tq[j][q] = fma(tk.x, m0, Tq[j][q]);
        Tq[j][q + 1] = fma(tk.y, m1, Tq[j][q + 1]);
#pragma unroll
        for (int e = 0; e < P; ++e) {
          const double2 z = *reinterpret_cast<const double2*>(sm + L::Z + e * M + 2 * k);
          Fq[e * P + j][q] = fma(z.x, m0, Fq[e * P + j][q]);
          Fq[e * P + j][q + 1] = fma(z.y, m1, Fq[e * P + j][q + 1]);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < P * P; ++k) Fr[k] = (Fq[k][0] + Fq[k][1]) + (Fq[k][2] + Fq[k][3]);
#pragma unroll
    for (int j = 0; j < P; ++j) TM[j] = IDT ? sm[L::Mm + i * P + j] : (Tq[j][0] + Tq[j][1]) + (Tq[j][2] + Tq[j][3]);
  }
  g.ok = ldl_inverse(Fr, g.Fi, Lr, Lir, g.piv, P);
  if (MK == MK_STD && P > 1 && full_det && g.ok) g.ok = lu_pivots(Fr, Lr, g.piv, P);  // det of the full matrix (t = 0)
  double qd = 0.0;
#pragma unroll
  for (int j = 0; j < P; ++j) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < P; ++k) s = fma(MK == MK_STEADY ? Gss[j * P + k] : g.Fi[j * P + k], g.v[k], s);
    g.w[j] = s;
    qd = fma(g.v[j], s, qd);
  }
  g.quad = qd;
#pragma unroll
  for (int j = 0; j < P; ++j) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < P; ++k) s = fma(TM[k], MK == MK_STEADY ? Gss[k * P + j] : g.Fi[k * P + j], s);
    g.Kp[j] = s;
    g.TM[j] = TM[j];
  }
  {
    const double* tr = sm + L::T + i * LD;
    double* lr = sm + L::Lm + i * LD;
#pragma unroll
    for (int k = 0; k < M / 2; ++k) {
      double2 lk = IDT ? make_double2(i == 2 * k ? 1.0 : 0.0, i == 2 * k + 1 ? 1.0 : 0.0)
                       : (act ? *rowD_chunk<LD>(tr, i, k) : make_double2(0.0, 0.0));
#pragma unroll
      for (int e = 0; e < P; ++e) {
        const double2 z = *reinterpret_cast<const double2*>(sm + L::Z + e * M + 2 * k);
        lk.x = fma(-g.Kp[e], z.x, lk.x);
        lk.y = fma(-g.Kp[e], z.y, lk.y);
      }
      if (act) *rowD_chunk<LD>(lr, i, k) = lk;
    }
    if (PADL && act) {  // the row's zero padding (Lm's slot doubles as the adjoint's tape staging buffer)
#pragma unroll
      for (int k = M / 2; k < L::TD / 2; ++k) *rowD_chunk<LD>(lr, i, k) = make_double2(0.0, 0.0);
    }
  }
  if (act) {
#pragma unroll
    for (int j = 0; j < P; ++j) sm[L::Kp + i * P + j] = g.Kp[j];
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------ forward
template <int M, int P, int MK>
__device__ void rowsD_forward(const KfArgs& A, long long u, double* sm, int lane) {
  using L = RowsDLayout<M, P, false>;
  constexpr int KT = L::KT, LD = L::LD;
  const int n = A.n;
  const long long draw = u / A.n_series;
  const bool act = lane < M;
  const int i = act ? lane : 0;
  const double* Tp = A.T.p + draw * A.T.bs;
  const double* Zp = A.Z.p + draw * A.Z.bs;
  const double* Hp = A.H.p + draw * A.H.bs;
  const double* Cp = A.C.p + draw * A.C.bs;
  const double* P0p = (MK == MK_STEADY) ? A.Pss.p + draw * A.Pss.bs : A.P0.p + draw * A.P0.bs;  // steady: starts at Pss
  double Gss[P * P];
#pragma unroll
  for (int k = 0; k < P * P; ++k) Gss[k] = (MK == MK_STEADY) ? A.Gss.p[draw * A.Gss.bs + k] : 0.0;
  for (int k = lane; k < L::fwd_doubles; k += 32) sm[k] = 0.0;  // zero padding everywhere
  __syncwarp();
  for (int k = lane; k < M * M; k += 32) {
    const int rr = k / M, cc = k - rr * M;
    sm[L::T + rowsD_el<LD>(rr, cc)] = Tp[k];
    sm[L::Pm + rowsD_el<LD>(rr, cc)] = P0p[k];
  }
  for (int k = lane; k < P * M; k += 32) sm[L::Z + k] = Zp[k];
  for (int k = lane; k < P * P; k += 32) sm[L::H + k] = Hp[k];
  if (act) sm[L::a + i] = A.a0.p[draw * A.a0.bs + i];
  double Cs[M];  // the lane's row of sym(C), C = R Q R^T (static): registers
#pragma unroll
  for (int j = 0; j < M; ++j) Cs[j] = 0.5 * (Cp[i * M + j] + Cp[j * M + i]);
  const double ci = (act && A.c.p) ? A.c.p[draw * A.c.bs + i] : 0.0;
  double dv[P];
#pragma unroll
  for (int j = 0; j < P; ++j) dv[j] = A.d.p ? A.d.p[draw * A.d.bs + j] : 0.0;
  __syncwarp();

  const double* y = A.y.p;
  LogAcc acc;
  double llsum = 0.0;
  int info = 0;
  double* tp = A.tape ? A.tape + u * (long long)(n - 1) * KT : nullptr;
  RowDGain<M, P> g;
  double yt[P], ynx[P];
#pragma unroll
  for (int j = 0; j < P; ++j) ynx[j] = y[j];

  for (int t = 0; t < n; ++t) {
#pragma unroll
    for (int j = 0; j < P; ++j) {
      yt[j] = ynx[j];
      ynx[j] = y[(long long)(t + 1 < n ? t + 1 : t) * P + j];
    }
    int nm = 0;
#pragma unroll
    for (int j = 0; j < P; ++j) nm += (yt[j] != yt[j]) ? 1 : 0;
    const bool observed = (nm == 0);
    // a' = T a + c (+ Kp v)
    double an;
    {
      double aq[4] = {ci, 0.0, 0.0, 0.0};
      const double* tr = sm + L::T + i * LD;
      const double2* av = reinterpret_cast<const double2*>(sm + L::a);
#pragma unroll
      for (int k = 0; k < M / 2; ++k) {
        const double2 tk = act ? *rowD_chunk<LD>(tr, i, k) : make_double2(0.0, 0.0), ak = av[k];
        const int q = (k & 1) * 2;
        aq[q] = fma(tk.x, ak.x, aq[q]);
        aq[q + 1] = fma(tk.y, ak.y, aq[q + 1]);
      }
      an = (aq[0] + aq[1]) + (aq[2] + aq[3]);
    }
    double KH[P];
#pragma unroll
    for (int j = 0; j < P; ++j) KH[j] = 0.0;
    if (observed) {
      rowsD_gain<M, P, MK, L>(sm, yt, A.d_sign, dv, Gss, i, act, g, t == 0);
      if (!g.ok && info == 0) info = t + 1;
      if (g.ok) {
#pragma unroll
        for (int k = 0; k < P; ++k) acc.mul(g.piv[k]);
      }
      llsum += -0.5 * (A.ll_const + g.quad);
#pragma unroll
      for (int k = 0; k < P; ++k) an = fma(g.Kp[k], g.v[k], an);
#pragma unroll
      for (int j = 0; j < P; ++j) {
#pragma unroll
        for (int k = 0; k < P; ++k) KH[j] = fma(g.Kp[k], sm[L::H + k * P + j], KH[j]);
        if (act) sm[L::KH + i * P + j] = KH[j];
      }
    } else if (nm != P && info == 0) {
      info = -(t + 1);
    }
    const double* Lsrc = observed ? sm + L::Lm : sm + L::T;  // L = T when nothing is observed
    // ---- X = L P, then S2raw = X L^T (tensor cores); S2raw overwrites X (all fragment loads of X are behind its mma's)
    {
      double c4[L::NT][L::NT][2];
      mm32<false, false, LD>(c4, Lsrc, sm + L::Pm, lane);
      mm32_store<LD>(sm + L::X, c4, 1.0, lane);
      __syncwarp();
      // S2raw = (L P) L^T is symmetric up to rounding: only its upper tiles are computed (the lower tiles of X's slot
      // keep stale values that rowD_load_symU never selects)
      mm32<false, true, LD, true, true>(c4, sm + L::X, Lsrc, lane);
      mm32_store<LD, true>(sm + L::X, c4, 1.0, lane);
    }
    __syncwarp();
    // ---- P' = sym(C + S2raw + KH Kp^T) row, a' ; tape
    const bool taped = tp && t + 1 < n;
    {
      double S[M];
      rowD_load_symU<M, LD>(S, sm + L::X, i, act);
#pragma unroll
      for (int j = 0; j < M; ++j) S[j] += Cs[j];
      if (observed) {
#pragma unroll
        for (int j = 0; j < M; ++j) {
#pragma unroll
          for (int k = 0; k < P; ++k)
            S[j] = fma(0.5, fma(KH[k], sm[L::Kp + j * P + k], sm[L::KH + j * P + k] * g.Kp[k]), S[j]);
        }
      }
      if (act) {
        rowD_store<M, LD>(sm + L::Pm + i * LD, i, S);
        sm[L::a + i] = an;
        if (taped) {
          tp[i] = an;
          double* trow = tp + M + i * M - (i * (i - 1)) / 2 - i;
#pragma unroll
          for (int j = 0; j < M; ++j)
            if (j >= i) trow[j] = S[j];
        }
      }
    }
    if (taped) tp += KT;
    __syncwarp();
  }
  if (lane == 0) {
    double ll = llsum - 0.5 * acc.value();
    if (info != 0) ll = nan("");
    if (A.loglik) A.loglik[u] = ll;
    if (MK == MK_STEADY && A.dare_info && A.dare_info[u / A.n_series] != 0) info = KF_INFO_DARE_FAILED;
    if (A.info) A.info[u] = info;
  }
}


// ------------------------------------------------------------------------------------------------ forward, all outputs
// The reference's six outputs (filtered / predicted moments, ll_obs: kalman_filter.py:166-193) need the two-stage form:
//     A = I - K Z,  P_f = A P A^T + K H K^T (Joseph, :255-284),  a_f = a + K v ;  P' = sym(T P_f T^T + C),  a' = T a_f + c
// = four tile products per observed step (A P, the upper tiles of (A P) A^T, T P_f, the upper tiles of (T P_f) T^T), two
// per unobserved one.  Output rows are written by their lanes as 16-byte stores: a warp writes each m x m matrix as one
// contiguous run.  (Round 1 / 2 ran this request on the generic CTA-per-unit kernels: 0.32 TB/s at k_states 30.)
template <int M>
__device__ __forceinline__ void rowG_store(double* dst, const double (&v)[M]) {
#pragma unroll
  for (int j = 0; j < M / 2; ++j) reinterpret_cast<double2*>(dst)[j] = make_double2(v[2 * j], v[2 * j + 1]);
}

template <int M, int P, int MK>
__device__ void rowsD_forward_full(const KfArgs& A, long long u, double* sm, int lane) {
  using L = RowsDLayout<M, P, false>;
  constexpr int KT = L::KT, LD = L::LD;
  const int n = A.n;
  const long long draw = u / A.n_series;
  const bool act = lane < M;
  const int i = act ? lane : 0;
  const double* Tp = A.T.p + draw * A.T.bs;
  const double* Zp = A.Z.p + draw * A.Z.bs;
  const double* Hp = A.H.p + draw * A.H.bs;
  const double* Cp = A.C.p + draw * A.C.bs;
  const double* P0g = A.P0.p + draw * A.P0.bs;
  const double* P0p = (MK == MK_STEADY) ? A.Pss.p + draw * A.Pss.bs : P0g;  // steady: the recursion starts at Pss
  double Gss[P * P];
#pragma unroll
  for (int k = 0; k < P * P; ++k) Gss[k] = (MK == MK_STEADY) ? A.Gss.p[draw * A.Gss.bs + k] : 0.0;
  for (int k = lane; k < L::fwd_doubles; k += 32) sm[k] = 0.0;  // zero padding everywhere
  __syncwarp();
  for (int k = lane; k < M * M; k += 32) {
    const int rr = k / M, cc = k - rr * M;
    sm[L::T + rowsD_el<LD>(rr, cc)] = Tp[k];
    sm[L::Pm + rowsD_el<LD>(rr, cc)] = P0p[k];
  }
  for (int k = lane; k < P * M; k += 32) sm[L::Z + k] = Zp[k];
  for (int k = lane; k < P * P; k += 32) sm[L::H + k] = Hp[k];
  const double a0i = A.a0.p[draw * A.a0.bs + i];
  if (act) sm[L::a + i] = a0i;
  double Cs[M];  // the lane's row of sym(C), C = R Q R^T (static): registers
#pragma unroll
  for (int j = 0; j < M; ++j) Cs[j] = 0.5 * (Cp[i * M + j] + Cp[j * M + i]);
  const double ci = (act && A.c.p) ? A.c.p[draw * A.c.bs + i] : 0.0;
  double dv[P];
#pragma unroll
  for (int j = 0; j < P; ++j) dv[j] = A.d.p ? A.d.p[draw * A.d.bs + j] : 0.0;
  // row 0 of the predicted moments = the caller's a0 / P0 (steady state: P0 is reported but not used, :397)
  if (act) {
    if (A.ps) A.ps[u * (long long)(n + 1) * M + i] = a0i;
    if (A.pc) {
      double r0[M];
#pragma unroll
      for (int j = 0; j < M; ++j) r0[j] = P0g[i * M + j];
      rowG_store<M>(A.pc + (u * (long long)(n + 1)) * M * M + i * M, r0);
    }
  }
  __syncwarp();

  const double* y = A.y.p;
  double llsum = 0.0;
  int info = 0;
  double* tp = A.tape ? A.tape + u * (long long)(n - 1) * KT : nullptr;
  RowDGain<M, P> g;
  double yt[P], ynx[P];
#pragma unroll
  for (int j = 0; j < P; ++j) ynx[j] = y[j];

  for (int t = 0; t < n; ++t) {
#pragma unroll
    for (int j = 0; j < P; ++j) {
      yt[j] = ynx[j];
      ynx[j] = y[(long long)(t + 1 < n ? t + 1 : t) * P + j];
    }
    int nm = 0;
#pragma unroll
    for (int j = 0; j < P; ++j) nm += (yt[j] != yt[j]) ? 1 : 0;
    const bool observed = (nm == 0);
    double af = sm[L::a + i], ll = 0.0;
    if (observed) {
      // K, A = I - K Z (in Kp / Lm), v, F^-1
      rowsD_gain<M, P, MK, L, false, true>(sm, yt, A.d_sign, dv, Gss, i, act, g, t == 0);
      if (!g.ok && info == 0) info = t + 1;
      double ld = 0.0;
#pragma unroll
      for (int k = 0; k < P; ++k) ld += log(g.piv[k]);
      ll = g.ok ? -0.5 * (A.ll_const + ld + g.quad) : nan("");
#pragma unroll
      for (int k = 0; k < P; ++k) af = fma(g.Kp[k], g.v[k], af);
      double KH[P];
#pragma unroll
      for (int j = 0; j < P; ++j) {
        KH[j] = 0.0;
#pragma unroll
        for (int k = 0; k < P; ++k) KH[j] = fma(g.Kp[k], sm[L::H + k * P + j], KH[j]);
        if (act) sm[L::KH + i * P + j] = KH[j];
      }
      // P_f = A P A^T + K H K^T
      {
        double c4[L::NT][L::NT][2];
        mm32<false, false, LD>(c4, sm + L::Lm, sm + L::Pm, lane);
        mm32_store<LD>(sm + L::X, c4, 1.0, lane);
        __syncwarp();
        mm32<false, true, LD, true, true>(c4, sm + L::X, sm + L::Lm, lane);
        mm32_store<LD, true>(sm + L::X, c4, 1.0, lane);
      }
      __syncwarp();
      double S[M];
      rowD_load_symU<M, LD>(S, sm + L::X, i, act);
#pragma unroll
      for (int j = 0; j < M; ++j) {
#pragma unroll
        for (int k = 0; k < P; ++k)
          S[j] = fma(0.5, fma(KH[k], sm[L::Kp + j * P + k], sm[L::KH + j * P + k] * g.Kp[k]), S[j]);
      }
      if (act) {
        rowD_store<M, LD>(sm + L::Pm + i * LD, i, S);
        if (A.fc) rowG_store<M>(A.fc + (u * (long long)n + t) * M * M + i * M, S);
      }
    } else {
      if (nm != P && info == 0) info = -(t + 1);
      if (act && A.fc) {
        double S[M];
        rowD_load<M, LD>(S, sm + L::Pm + i * LD, i, act);
        rowG_store<M>(A.fc + (u * (long long)n + t) * M * M + i * M, S);
      }
    }
    llsum += ll;
    if (act) {
      sm[L::a + i] = af;
      if (A.fs) A.fs[(u * (long long)n + t) * M + i] = af;
    }
    if (lane == 0 && A.ll_obs) A.ll_obs[u * (long long)n + t] = ll;
    __syncwarp();  // a_f and P_f visible
    // predict: a' = T a_f + c ; P' = sym(T P_f T^T + C)
    double an;
    {
      double aq[4] = {ci, 0.0, 0.0, 0.0};
      const double* tr = sm + L::T + i * LD;
      const double2* av = reinterpret_cast<const double2*>(sm + L::a);
#pragma unroll
      for (int k = 0; k < M / 2; ++k) {
        const double2 tk = act ? *rowD_chunk<LD>(tr, i, k) : make_double2(0.0, 0.0), ak = av[k];
        const int q = (k & 1) * 2;
        aq[q] = fma(tk.x, ak.x, aq[q]);
        aq[q + 1] = fma(tk.y, ak.y, aq[q + 1]);
      }
      an = (aq[0] + aq[1]) + (aq[2] + aq[3]);
    }
    {
      double c4[L::NT][L::NT][2];
      mm32<false, false, LD>(c4, sm + L::T, sm + L::Pm, lane);
      mm32_store<LD>(sm + L::X, c4, 1.0, lane);
      __syncwarp();
      mm32<false, true, LD, true, true>(c4, sm + L::X, sm + L::T, lane);
      mm32_store<LD, true>(sm + L::X, c4, 1.0, lane);
    }
    __syncwarp();
    const bool taped = tp && t + 1 < n;
    {
      double S[M];
      rowD_load_symU<M, LD>(S, sm + L::X, i, act);
#pragma unroll
      for (int j = 0; j < M; ++j) S[j] += Cs[j];
      if (act) {
        rowD_store<M, LD>(sm + L::Pm + i * LD, i, S);
        sm[L::a + i] = an;
        if (A.ps) A.ps[(u * (long long)(n + 1) + t + 1) * M + i] = an;
        if (A.pc) rowG_store<M>(A.pc + (u * (long long)(n + 1) + t + 1) * M * M + i * M, S);
        if (taped) {
          tp[i] = an;
          double* trow = tp + M + i * M - (i * (i - 1)) / 2 - i;
#pragma unroll
          for (int j = 0; j < M; ++j)
            if (j >= i) trow[j] = S[j];
        }
      }
    }
    if (taped) tp += KT;
    __syncwarp();
  }
  if (lane == 0) {
    if (info != 0) llsum = nan("");
    if (A.loglik) A.loglik[u] = llsum;
    if (MK == MK_STEADY && A.dare_info && A.dare_info[u / A.n_series] != 0) info = KF_INFO_DARE_FAILED;
    if (A.info) A.info[u] = info;
  }
}

// ------------------------------------------------------------------------------------------------ adjoint
// Per step (going backwards), with Ps = sym(P-bar') the symmetrised cotangent of the step above:
//     W = Ps L                 (tile product)
//     P-bar = L^T W + Mb Z     (tile product, upper tiles only: L^T Ps L is symmetric; the rank-p part Mb Z is kept
//                               apart in shared memory and joins in the next step's symmetrisation / the write-out)
//     L-bar = Ps L (P + P^T) = 2 W P :  T-bar += L-bar is accumulated ON the tensor cores, in mma fragment layout,
//                               across all steps (T-bar = 2 Tacc; the rank-1 terms ab a^T and TMb Mm^T join it there);
//                               L-bar Z^T = 2 W (P Z^T) = 2 W Mm is a row-wise dot product with the gain's Mm.
// Round 1 formed X = 2 L P with a third (fourth, with T-bar) tile product and stored / re-read L-bar as a matrix:
// 26 instead of 48 tile products per step without T-bar, 42 instead of 64 with it - same terms, associated differently.
template <int M, int P, int MK, bool NEED_T>
__device__ void rowsD_backward(const KfArgs& A, long long u, double* sm, int lane) {
  using L = RowsDLayout<M, P, NEED_T>;
  constexpr int KT = L::KT, LD = L::LD;
  const int n = A.n;
  const long long draw = u / A.n_series;
  const bool act = lane < M;
  const int i = act ? lane : 0;
  const int fr = lane >> 2, fc = lane & 3;  // mma fragment coordinates
  const double* Tp = A.T.p + draw * A.T.bs;
  const double* Zp = A.Z.p + draw * A.Z.bs;
  const double* Hp = A.H.p + draw * A.H.bs;
  const double* tape = A.tape + u * (long long)(n - 1) * KT;  // entry t-1 = predicted moments of step t
  for (int k = lane; k < L::bwd_doubles; k += 32) sm[k] = 0.0;  // zero padding, Pb = 0, ab = 0, Mb = 0
  __syncwarp();
  if (n >= 2) rows_tape_prefetch<KT, 32>(sm + L::tp, tape + (long long)(n - 2) * KT, lane);
  for (int k = lane; k < M * M; k += 32) {
    const int rr = k / M, cc = k - rr * M;
    sm[L::T + rowsD_el<LD>(rr, cc)] = Tp[k];
  }
  for (int k = lane; k < P * M; k += 32) sm[L::Z + k] = Zp[k];
  for (int k = lane; k < P * P; k += 32) sm[L::H + k] = Hp[k];
  double dv[P];
#pragma unroll
  for (int j = 0; j < P; ++j) dv[j] = A.d.p ? A.d.p[draw * A.d.bs + j] : 0.0;
  __syncwarp();

  const double* y = A.y.p;
  const double gl = A.g_loglik ? A.g_loglik[u] : 1.0;
  const bool need_H = (A.gH != nullptr) || (MK == MK_STEADY);
  double Gss[P * P], Gb[P * P];  // steady state: fixed gain matrix and its cotangent (every lane holds all of it)
#pragma unroll
  for (int k = 0; k < P * P; ++k) {
    Gss[k] = (MK == MK_STEADY) ? A.Gss.p[draw * A.Gss.bs + k] : 0.0;
    Gb[k] = 0.0;
  }
  // gradient accumulators: the lane's row of Cb in registers; HALF of T-bar in mma fragment layout (lane holds
  // [8I + fr][8J + 2 fc + {0,1}]); lanes < P hold rows of Hb; cb (row), db (lane)
  constexpr int TI = NEED_T ? L::NT : 1;
  double Cb[M], Tacc[TI][TI][2], Hb[P], cb = 0.0, db = 0.0, abi = 0.0;
#pragma unroll
  for (int j = 0; j < M; ++j) Cb[j] = 0.0;
#pragma unroll
  for (int I = 0; I < TI; ++I)
#pragma unroll
    for (int J = 0; J < TI; ++J) Tacc[I][J][0] = Tacc[I][J][1] = 0.0;
#pragma unroll
  for (int j = 0; j < P; ++j) Hb[j] = 0.0;
  RowDGain<M, P> g;
  double yt[P], ynx[P];
#pragma unroll
  for (int j = 0; j < P; ++j) ynx[j] = y[(long long)(n - 1) * P + j];

  for (int t = n - 1; t >= 0; --t) {
    // ---- predicted moments of step t -> shared memory (without T-bar Pm's slot held W: its padding is zero either way)
    if (t == 0) {
      const double* P0p = (MK == MK_STEADY) ? A.Pss.p + draw * A.Pss.bs : A.P0.p + draw * A.P0.bs;
      for (int k = lane; k < M * M; k += 32) {
        const int rr = k / M, cc = k - rr * M;
        sm[L::Pm + rowsD_el<LD>(rr, cc)] = P0p[k];
      }
      if (act) sm[L::a + i] = A.a0.p[draw * A.a0.bs + i];
    } else {
      rows_tape_wait();
      __syncwarp();
      const double* tq = sm + L::tp;
      if (act) {
        sm[L::a + i] = tq[i];
        double Pr[M];
#pragma unroll
        for (int j = 0; j < M; ++j) {
          const int lo = i < j ? i : j, hi = i < j ? j : i;
          Pr[j] = tq[M + lo * M - (lo * (lo - 1)) / 2 + (hi - lo)];
        }
        rowD_store<M, LD>(sm + L::Pm + i * LD, i, Pr);
      }
      // (every lane has read the staging buffer before the sync below; the gain may overwrite it)
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < P; ++j) {
      yt[j] = ynx[j];
      ynx[j] = y[(long long)(t > 0 ? t - 1 : 0) * P + j];
    }
    const double lb = gl + (A.g_ll_obs ? A.g_ll_obs[u * n + t] : 0.0);
    bool observed = true;
#pragma unroll
    for (int j = 0; j < P; ++j) observed = observed && (yt[j] == yt[j]);
    if (observed) {
      rowsD_gain<M, P, MK, L, true>(sm, yt, A.d_sign, dv, Gss, i, act, g);
      if (MK == MK_STEADY && act) {
#pragma unroll
        for (int e = 0; e < P; ++e) sm[L::TMs + i * P + e] = g.TM[e];  // read by every lane in phase 3 (after syncs)
      }
    }
    const double* Lsrc = observed ? sm + L::Lm : sm + L::T;
    if (t == 0) {  // P0 may be any matrix: L-bar = W (P + P^T); for t >= 1 the taped P is symmetric: P + P^T = 2 P
      double S0[M];
      rowD_load<M, LD>(S0, sm + L::Pm + i * LD, i, act);
#pragma unroll
      for (int j = 0; j < M; ++j) S0[j] = 0.5 * (S0[j] + colD<LD>(sm + L::Pm, j, i));
      if (observed) {  // lz = (P + P^T) Z^T rows
#pragma unroll
        for (int e = 0; e < P; ++e) {
          const double s = dot4<M>(0.0, [&](int j, double& x, double& y2) {
            x = S0[j];
            y2 = sm[L::Z + e * M + j];
          });
          if (act) sm[L::lz + i * P + e] = 2.0 * s;
        }
      }
      __syncwarp();
      if (NEED_T && act) rowD_store<M, LD>(sm + L::Pm + i * LD, i, S0);
      __syncwarp();
    }
    // ---- 1: Ps = sym(P-bar') = symU(L^T W of the step above) + sym(Mb Z), in place ; Cb += Ps
    cb += abi;
    double Ps[M];  // without T-bar the row stays in registers for phase 2; with it (64 more accumulators) it is re-read
    {
      rowD_load_symU<M, LD>(Ps, sm + L::Pb, i, act);
#pragma unroll
      for (int k = 0; k < P; ++k) {
        const double mi = 0.5 * sm[L::Mb + i * P + k], zi = 0.5 * sm[L::Z + k * M + i];
#pragma unroll
        for (int j = 0; j < M; ++j) Ps[j] = fma(mi, sm[L::Z + k * M + j], fma(zi, sm[L::Mb + j * P + k], Ps[j]));
      }
#pragma unroll
      for (int j = 0; j < M; ++j) Cb[j] += Ps[j];
      __syncwarp();  // every lane has read its row and column of P-bar'
      if (act) rowD_store<M, LD>(sm + L::Pb + i * LD, i, Ps);
    }
    __syncwarp();  // Ps visible
    // ---- 2: W = Ps L (tensor cores) ; PK = Ps Kp, T^T ab (row-wise, independent of the product: they sit between its
    //         last mma and its store - a DMMA issues once per ~16 cycles, the scheduler fills the gaps)
    double PK[P], Kb[P], abn;
    {
      double c4[L::NT][L::NT][2];
      mm32<false, false, LD>(c4, sm + L::Pb, Lsrc, lane);
      if constexpr (NEED_T) rowD_load<M, LD>(Ps, sm + L::Pb + i * LD, i, act);
#pragma unroll
      for (int e = 0; e < P; ++e) {
        PK[e] = dot4<M>(0.0, [&](int k, double& x, double& y2) {  // (Kp is stale but unused when nothing is observed)
          x = Ps[k];
          y2 = sm[L::Kp + k * P + e];
        });
      }
      abn = dot4<M>(0.0, [&](int k, double& x, double& y2) {
        x = colD<LD>(sm + L::T, k, i);
        y2 = sm[L::ab + k];
      });
      mm32_store<LD>(sm + L::W, c4, 1.0, lane);  // without T-bar: Pm's slot (its fragment loads... none: P is not an operand)
    }
    __syncwarp();  // W visible
    // ---- 2b: (T-bar) Tacc += W P + ab a^T / 2 ; L-bar Z^T = 2 W Mm (t = 0: W lz) ; Kb
    if constexpr (NEED_T) {
      mm32<false, false, LD, false>(Tacc, sm + L::W, sm + L::Pm, lane);  // P symmetric (t = 0: sym(P0))
#pragma unroll
      for (int I = 0; I < TI; ++I) {
        const double abI = 0.5 * sm[L::ab + 8 * I + fr];
#pragma unroll
        for (int J = 0; J < TI; ++J) {
          const double2 a2 = *reinterpret_cast<const double2*>(sm + L::a + 8 * J + 2 * fc);
          Tacc[I][J][0] = fma(abI, a2.x, Tacc[I][J][0]);
          Tacc[I][J][1] = fma(abI, a2.y, Tacc[I][J][1]);
        }
      }
    }
    if (observed) {
      double Wr[M];
      rowD_load<M, LD>(Wr, sm + L::W + i * LD, i, act);
      const double* m2 = (t == 0) ? sm + L::lz : sm + L::Mm;
      const double sc = (t == 0) ? 1.0 : 2.0;
#pragma unroll
      for (int e = 0; e < P; ++e) {
        const double lbz = sc * dot4<M>(0.0, [&](int k, double& x, double& y2) {
          x = Wr[k];
          y2 = m2[k * P + e];
        });
        double s = abi * g.v[e] - lbz;
#pragma unroll
        for (int k = 0; k < P; ++k) s = fma(PK[k], sm[L::H + k * P + e] + sm[L::H + e * P + k], s);
        Kb[e] = s;
      }
      if (act) {
#pragma unroll
        for (int e = 0; e < P; ++e) {
          sm[L::Kb + i * P + e] = Kb[e];
          if (need_H) sm[L::PK + i * P + e] = PK[e];
        }
      }
    }
    // ---- 3: L^T W (tensor cores, upper tiles) -> Pb (Ps rows were last read above, by their owners, before this point
    //         in program order of every lane; the store follows the last mma, which all lanes execute together)
    __syncwarp();  // Kb visible; all row reads of Ps and W done
    double c4p[L::NT][L::NT][2];
    mm32<true, false, LD, true, true>(c4p, Lsrc, sm + L::W, lane);  // stored after the row-wise block below
    __syncwarp();  // last use of Lm in this step: stage the tape entry of step t-1 in its slot
    if (t >= 2) rows_tape_prefetch<KT, 32>(sm + L::tp, tape + (long long)(t - 2) * KT, lane);
    double vb[P], Fb[P * P], TMb[P];
    if (observed) {
      if (MK == MK_STEADY) {
        // vb = Kp^T ab - lb sym(Gss) v ; Gss-bar += TM^T Kb - lb/2 v v^T ; Fb = -lb/2 F^-T ; TMb = Kb Gss^T
#pragma unroll
        for (int a2 = 0; a2 < P; ++a2) {
          double s = dot4<M>(0.0, [&](int k, double& x, double& y2) {
            x = sm[L::Kp + k * P + a2];
            y2 = sm[L::ab + k];
          });
#pragma unroll
          for (int b2 = 0; b2 < P; ++b2) s = fma(-0.5 * lb * (Gss[a2 * P + b2] + Gss[b2 * P + a2]), g.v[b2], s);
          vb[a2] = s;
#pragma unroll
          for (int b2 = 0; b2 < P; ++b2) {
            const double q1 = dot4<M>(Gb[a2 * P + b2], [&](int k, double& x, double& y2) {
              x = sm[L::TMs + k * P + a2];
              y2 = sm[L::Kb + k * P + b2];
            });
            Gb[a2 * P + b2] = fma(-0.5 * lb * g.v[a2], g.v[b2], q1);
            Fb[a2 * P + b2] = -0.5 * lb * g.Fi[b2 * P + a2];
          }
        }
#pragma unroll
        for (int e = 0; e < P; ++e) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < P; ++k) s = fma(Kb[k], Gss[e * P + k], s);
          TMb[e] = s;
        }
      } else {
        double Q1[P * P];
#pragma unroll
        for (int a2 = 0; a2 < P; ++a2) {
          vb[a2] = dot4<M>(-lb * g.w[a2], [&](int k, double& x, double& y2) {
            x = sm[L::Kp + k * P + a2];
            y2 = sm[L::ab + k];
          });
#pragma unroll
          for (int b2 = 0; b2 < P; ++b2)
            Q1[a2 * P + b2] = dot4<M>(0.0, [&](int k, double& x, double& y2) {
              x = sm[L::Kp + k * P + a2];
              y2 = sm[L::Kb + k * P + b2];
            });
        }
#pragma unroll
        for (int a2 = 0; a2 < P; ++a2)
#pragma unroll
          for (int b2 = 0; b2 < P; ++b2) {
            double s = -0.5 * lb * (g.Fi[b2 * P + a2] - g.w[a2] * g.w[b2]);
#pragma unroll
            for (int k = 0; k < P; ++k) s = fma(-Q1[a2 * P + k], g.Fi[b2 * P + k], s);
            Fb[a2 * P + b2] = s;
          }
#pragma unroll
        for (int e = 0; e < P; ++e) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < P; ++k) s = fma(Kb[k], g.Fi[e * P + k], s);
          TMb[e] = s;
        }
      }
      if (act) {
#pragma unroll
        for (int e = 0; e < P; ++e) sm[L::TMb + i * P + e] = TMb[e];
      }
    }
    mm32_store<LD, true>(sm + L::Pb, c4p, 1.0, lane);
    __syncwarp();  // L^T W and TMb visible; ab's readers are done
    // ---- 4: (observed) Mb = T^T TMb + Z^T Fb (the rank-p part of P-bar) ; ab' = T^T ab - Z^T vb ; T-bar += TMb Mm^T
    if (observed) {
#pragma unroll
      for (int e = 0; e < P; ++e) {
        double s = dot4<M>(0.0, [&](int k, double& x, double& y2) {
          x = colD<LD>(sm + L::T, k, i);
          y2 = sm[L::TMb + k * P + e];
        });
#pragma unroll
        for (int k = 0; k < P; ++k) s = fma(sm[L::Z + k * M + i], Fb[k * P + e], s);
        if (act) sm[L::Mb + i * P + e] = s;
      }
#pragma unroll
      for (int k = 0; k < P; ++k) abn = fma(-sm[L::Z + k * M + i], vb[k], abn);
#pragma unroll
      for (int k = 0; k < P; ++k)
        if (lane == k) db = fma(-A.d_sign, vb[k], db);
      if (need_H) {
#pragma unroll
        for (int e = 0; e < P; ++e) {
          if (lane != e) continue;
#pragma unroll
          for (int j = 0; j < P; ++j) {
            Hb[j] = dot4<M>(Hb[j] + Fb[e * P + j], [&](int k, double& x, double& y2) {  // + Kp^T Ps Kp
              x = sm[L::Kp + k * P + e];
              y2 = sm[L::PK + k * P + j];
            });
          }
        }
      }
      if constexpr (NEED_T) {
#pragma unroll
        for (int I = 0; I < TI; ++I) {
#pragma unroll
          for (int k = 0; k < P; ++k) {
            const double tI = 0.5 * sm[L::TMb + (8 * I + fr) * P + k];
#pragma unroll
            for (int J = 0; J < TI; ++J) {
              Tacc[I][J][0] = fma(tI, sm[L::Mm + (8 * J + 2 * fc) * P + k], Tacc[I][J][0]);
              Tacc[I][J][1] = fma(tI, sm[L::Mm + (8 * J + 2 * fc + 1) * P + k], Tacc[I][J][1]);
            }
          }
        }
      }
    } else if (act) {
#pragma unroll
      for (int e = 0; e < P; ++e) sm[L::Mb + i * P + e] = 0.0;
    }
    if (act) sm[L::ab + i] = abn;
    abi = abn;
    __syncwarp();
  }
  // ---- write-out (row i by lane i): P-bar = symU(L^T W) + Mb Z of step 0
  {
    double Pf[M];
    rowD_load_symU<M, LD>(Pf, sm + L::Pb, i, act);
#pragma unroll
    for (int k = 0; k < P; ++k) {
      const double mi = sm[L::Mb + i * P + k];
#pragma unroll
      for (int j = 0; j < M; ++j) Pf[j] = fma(mi, sm[L::Z + k * M + j], Pf[j]);
    }
    if (act) {
      if (A.ga0) A.ga0[u * M + i] = abi;
#pragma unroll
      for (int j = 0; j < M; ++j) {
        if (MK == MK_STEADY) {
          if (A.gPss) A.gPss[u * M * M + i * M + j] = Pf[j];
          if (A.gP0) A.gP0[u * M * M + i * M + j] = 0.0;
        } else if (A.gP0) {
          A.gP0[u * M * M + i * M + j] = Pf[j];
        }
        if (A.gC) A.gC[u * M * M + i * M + j] = Cb[j];
      }
      if (A.gc) A.gc[u * M + i] = cb;
    }
  }
  if (NEED_T && A.gT) {
#pragma unroll
    for (int I = 0; I < TI; ++I)
#pragma unroll
      for (int J = 0; J < TI; ++J)
#pragma unroll
        for (int x = 0; x < 2; ++x) {
          const int row = 8 * I + fr, col = 8 * J + 2 * fc + x;
          if (row < M && col < M) A.gT[u * M * M + row * M + col] = 2.0 * Tacc[I][J][x];
        }
  }
  if (lane < P) {
    if (A.gd) A.gd[u * P + lane] = db;
#pragma unroll
    for (int j = 0; j < P; ++j)
      if (A.gH) A.gH[u * P * P + lane * P + j] = Hb[j];
  }
  if (MK == MK_STEADY && lane == 0 && A.gGss) {
#pragma unroll
    for (int k = 0; k < P * P; ++k) A.gGss[u * P * P + k] = Gb[k];
  }
}


// ------------------------------------------------------------------------------------------------ steady state (DARE)
// The same fixed-point iteration as kf_dare.cuh (Riccati recursion from above, then Newton-Hewer with squared-Smith
// doubling; reference call: scipy.linalg.solve_discrete_are, filters/kalman_filter.py:384, utils/pytensor_scipy.py:28-35)
// on the warp-per-draw tensor-core mapping of this file: a Riccati step IS the forward step above without data
// (P' = L P L^T + Kp H Kp^T + C), a Newton-Hewer iterate solves P = L P L^T + (C + Kp H Kp^T) for the gain of the current
// P, and a Smith doubling is three tile products (S1 = A X, X += S1 A^T, A <- A A).  Config 4 (k_states 30, 8,192 draws):
// 99.5 ms on the generic CTA-per-draw kernels (29 % of a steady_state evaluation) -> see profiles/r2_ncu_rowsD.md.
template <int M, int P>
struct DareDLayout {
  static constexpr int NT = rowsD_nt(M), TD = 8 * NT, LD = rowsD_ld(M), MS = TD * LD;
  static constexpr int MP = M * P, PP = P * P, MPE = MP + (MP & 1), MPT = TD * P;
  static constexpr int T = 0, Pm = T + MS, Lm = Pm + MS, X = Lm + MS, Xs = X + MS, Z = Xs + MS, H = Z + MPE,
                       Mm = H + PP + (PP & 1), Kp = Mm + MPT, a = Kp + MPE, KH = a + TD, END = KH + MPE;
  static constexpr int doubles = (END + 1) & ~1;
};

// acc <- D (the inverse of mm32_store)
template <int LD, int NT = LD / 8>
__device__ __forceinline__ void mm32_load(double (&acc)[NT][NT][2], const double* D, int lane) {
  const int r = lane >> 2, c = lane & 3;
#pragma unroll
  for (int I = 0; I < NT; ++I)
#pragma unroll
    for (int J = 0; J < NT; ++J) {
      const double2 x = *reinterpret_cast<const double2*>(D + (8 * I + r) * LD + (((4 * J + c) ^ rowsD_swz<LD>(r)) << 1));
      acc[I][J][0] = x.x;
      acc[I][J][1] = x.y;
    }
}

__device__ __forceinline__ double warp_max(double v) {
#ifdef __CUDA_ARCH__
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
#endif
  return v;
}

template <int M, int P>
__device__ void rowsD_dare(const double* Tp, const double* Zp, const double* Hp, const double* Cp, double* Pss, double* Gssg,
                           int* info_out, double* sm, int lane) {
  using L = DareDLayout<M, P>;
  constexpr int LD = L::LD;
  const bool act = lane < M;
  const int i = act ? lane : 0;
  for (int k = lane; k < L::doubles; k += 32) sm[k] = 0.0;  // zero padding everywhere, a = 0
  __syncwarp();
  for (int k = lane; k < M * M; k += 32) {
    const int rr = k / M, cc = k - rr * M;
    sm[L::T + rowsD_el<LD>(rr, cc)] = Tp[k];
  }
  for (int k = lane; k < P * M; k += 32) sm[L::Z + k] = Zp[k];
  for (int k = lane; k < P * P; k += 32) sm[L::H + k] = Hp[k];
  double Cs[M];  // the lane's row of sym(C)
  double scale = 1.0;
#pragma unroll
  for (int j = 0; j < M; ++j) {
    Cs[j] = 0.5 * (Cp[i * M + j] + Cp[j * M + i]);
    scale = fmax(scale, fmax(fabs(Cp[i * M + j]), fabs(Cp[j * M + i])));
  }
#pragma unroll
  for (int k = 0; k < P * P; ++k) scale = fmax(scale, fabs(Hp[k]));
  scale = warp_max(scale);
  if (act) sm[L::Pm + rowsD_el<LD>(i, i)] = 1.0e4 * scale;
  __syncwarp();

  double yt[P], dv[P], Gss[P * P];
#pragma unroll
  for (int j = 0; j < P; ++j) yt[j] = dv[j] = 0.0;
#pragma unroll
  for (int k = 0; k < P * P; ++k) Gss[k] = 0.0;
  RowDGain<M, P> g;
  int info = 0;
  // the lane's row of sym(Kp H Kp^T) + sym(C): the constant term of the step / of the Lyapunov equation
  auto rhs_row = [&](double (&S)[M]) {
    double KH[P];
#pragma unroll
    for (int j = 0; j < P; ++j) {
      KH[j] = 0.0;
#pragma unroll
      for (int k = 0; k < P; ++k) KH[j] = fma(g.Kp[k], sm[L::H + k * P + j], KH[j]);
      if (act) sm[L::KH + i * P + j] = KH[j];
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < M; ++j) {
      double s = Cs[j];
#pragma unroll
      for (int k = 0; k < P; ++k) s = fma(0.5, fma(KH[k], sm[L::Kp + j * P + k], sm[L::KH + j * P + k] * g.Kp[k]), s);
      S[j] = s;
    }
  };
  // (1) Riccati recursion from above: every iterate >= P_ss, so every gain is stabilising
  const int n0 = 2 * M + 24;
  for (int k = 0; k < n0; ++k) {
    rowsD_gain<M, P, MK_STD, L>(sm, yt, 1.0, dv, Gss, i, act, g);
    if (!g.ok) info = 1;
    double S[M], U[M];
    rhs_row(S);
    {
      double c4[L::NT][L::NT][2];
      mm32<false, false, LD>(c4, sm + L::Lm, sm + L::Pm, lane);
      mm32_store<LD>(sm + L::X, c4, 1.0, lane);
      __syncwarp();
      mm32<false, true, LD, true, true>(c4, sm + L::X, sm + L::Lm, lane);
      mm32_store<LD, true>(sm + L::X, c4, 1.0, lane);
    }
    __syncwarp();
    rowD_load_symU<M, LD>(U, sm + L::X, i, act);
#pragma unroll
    for (int j = 0; j < M; ++j) S[j] += U[j];
    if (act) rowD_store<M, LD>(sm + L::Pm + i * LD, i, S);
    __syncwarp();
  }
  // (2) Newton-Hewer: P <- Lyapunov(L(P), C + Kp H Kp^T), each Lyapunov equation by squared-Smith doubling
  bool converged = false;
  for (int it = 0; it < 60 && !converged && info == 0; ++it) {
    rowsD_gain<M, P, MK_STD, L>(sm, yt, 1.0, dv, Gss, i, act, g);
    if (!g.ok) { info = 1; break; }
    {
      double S[M];
      rhs_row(S);
      if (act) rowD_store<M, LD>(sm + L::Xs + i * LD, i, S);
    }
    __syncwarp();
    bool ok = false;
    for (int db = 0; db < 64; ++db) {  // Xs <- sum_k A^k Xs A^kT, A = Lm (destroyed)
      double Ar[M], mx = 0.0;
      rowD_load<M, LD>(Ar, sm + L::Lm + i * LD, i, act);
#pragma unroll
      for (int j = 0; j < M; ++j) mx = fmax(mx, fabs(Ar[j]));
      mx = warp_max(mx);
      if (!(mx < 1.0e150)) break;
      if (mx < 1.0e-11) { ok = true; break; }
      double c4[L::NT][L::NT][2];
      mm32<false, false, LD>(c4, sm + L::Lm, sm + L::Xs, lane);  // S1 = A Xs
      mm32_store<LD>(sm + L::X, c4, 1.0, lane);
      __syncwarp();
      mm32_load<LD>(c4, sm + L::Xs, lane);
      mm32<false, true, LD, false>(c4, sm + L::X, sm + L::Lm, lane);  // Xs += S1 A^T
      mm32_store<LD>(sm + L::Xs, c4, 1.0, lane);
      mm32<false, false, LD>(c4, sm + L::Lm, sm + L::Lm, lane);  // A <- A A
      mm32_store<LD>(sm + L::Lm, c4, 1.0, lane);
      __syncwarp();
    }
    if (!ok) { info = 1; break; }
    double Pn[M], Po[M], diff = 0.0, mag = 0.0;
    rowD_load<M, LD>(Pn, sm + L::Xs + i * LD, i, act);
    rowD_load<M, LD>(Po, sm + L::Pm + i * LD, i, act);
#pragma unroll
    for (int j = 0; j < M; ++j) {
      diff = fmax(diff, fabs(Pn[j] - Po[j]));
      mag = fmax(mag, fabs(Pn[j]));
      Pn[j] = 0.5 * (Pn[j] + colD<LD>(sm + L::Xs, j, i));  // symmetrise: keeps the iteration on the symmetric manifold
    }
    diff = warp_max(diff);
    mag = warp_max(mag);
    if (act) rowD_store<M, LD>(sm + L::Pm + i * LD, i, Pn);
    __syncwarp();
    converged = diff <= 4.0e-15 * mag;
  }
  if (!converged) info = 1;
  // Gss = (Z Pss Z^T + H)^-1
  rowsD_gain<M, P, MK_STD, L>(sm, yt, 1.0, dv, Gss, i, act, g);
  if (!g.ok) info = 1;
  if (act) {
    double Pr[M];
    rowD_load<M, LD>(Pr, sm + L::Pm + i * LD, i, act);
#pragma unroll
    for (int j = 0; j < M; ++j) Pss[i * M + j] = info ? nan("") : Pr[j];
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < P * P; ++k) Gssg[k] = info ? nan("") : g.Fi[k];
    if (info_out) *info_out = info;
  }
}

}  // namespace kfb
