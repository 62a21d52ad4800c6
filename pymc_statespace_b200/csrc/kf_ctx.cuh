// kf_ctx.cuh - execution contexts for kf_core.cuh (see the header comment there).
#pragma once
#include "kf_core.cuh"

namespace kfb {

// ---------------------------------------------------------------------------
// ThreadCtx: one unit per thread; compile-time dims; all buffers are registers.
// Tape layout [t-1][warp][k][32]: consecutive threads (units) touch consecutive doubles -> every tape
// load/store of a warp is one fully-coalesced 256-byte transaction.
// ---------------------------------------------------------------------------
template <int N>
struct RegBuf {
  double v[N > 0 ? N : 1];
  template <class X>
  KFB_HD explicit RegBuf(X&) {}
  KFB_HD double& operator[](int i) { return v[i]; }
  KFB_HD const double& operator[](int i) const { return v[i]; }
};

// TV_ = true: time-varying matrices (3-D time-first inputs, reference filters/utilities.py:1-20) - the step programs
// reload the varying matrices from global memory every step; everything else is identical.
template <int M, int P, bool TV_ = false>
struct ThreadCtx {
  static constexpr bool TV = TV_;
  static constexpr bool SKIP_LB = false;   // adjoint without T-bar / Z-bar: keep the single code path (a run-time branch cost the m = 2 kernel 14 %)
  template <int SZ>
  using Buf = RegBuf<(SZ == SZ_M ? M : SZ == SZ_P ? P : SZ == SZ_MM ? M * M : SZ == SZ_MP ? M * P : SZ == SZ_PP ? P * P : M + (M * (M + 1)) / 2)>;
  const double* y_smem;  // observations staged in shared memory (shared y) or nullptr
  double* ring;          // shared-memory ring for the adjoint kernel's tape read-ahead (device only)
  int tid, nthr;
  // ---- full-output forward pass: per-warp shared-memory stager (device only; nullptr = direct stores)
  // A thread owns a unit, and the outputs are unit-major ([U, n, w]), so a direct store puts every lane's 8 bytes into
  // its own 32-byte sector (measured: 0.65 TB/s, 10 % of the HBM copy rate at k_states = 2).  Instead the rows of
  // OUT_K consecutive steps are staged in shared memory as [step][element][lane] (row stride 33: conflict-free writes,
  // 2-way reads) and flushed by the whole warp unit by unit: the OUT_K * w doubles of one unit and one output array
  // are contiguous in global memory, so the warp writes them as 32..128-byte runs of whole sectors.
  double* ostage = nullptr;
  long long warp_u0 = 0;  // first unit of this thread's warp
  static constexpr int OUT_W = 2 * M + 2 * M * M + 1;            // doubles per unit and step (fs, ps, fc, pc, ll)
  static constexpr int OUT_K = 4;                                // steps per flush (k_states 2: 13.7 KB per warp)
  static constexpr int OUT_LD = 33;
  static constexpr int OUT_DOUBLES = OUT_K * OUT_W * OUT_LD;     // per warp
  KFB_HD static constexpr int out_off(int arr) {
    return arr == O_FS ? 0 : arr == O_PS ? M : arr == O_FC ? 2 * M : arr == O_PC ? 2 * M + M * M : 2 * M + 2 * M * M;
  }
  KFB_HD static constexpr int out_width(int arr) { return arr == O_FS || arr == O_PS ? M : arr == O_LL ? 1 : M * M; }
  template <class TS>
  KFB_HD void store_row(const KfArgs& A, int arr, long long u, long long rows, long long r, int w, const TS& src) {
#if defined(__CUDA_ARCH__)
    if (ostage) {
      // ps / pc rows are shifted by one (row 0 = a0 / P0 is written before the loop): slot by step, not by row
      const int slot = (int)((arr == O_PS || arr == O_PC ? r - 1 : r) % OUT_K);
      double* dst = ostage + (size_t)(slot * OUT_W + out_off(arr)) * OUT_LD + (tid & 31);
#pragma unroll
      for (int i = 0; i < (M * M > 1 ? M * M : 1); ++i)
        if (i < w) dst[i * OUT_LD] = src[i];
      return;
    }
#endif
    store_row_direct(*this, A, arr, u, rows, r, w, src);
  }
  // flush `count` staged steps (rows t0 .. t0 + count - 1) of one output array; COUNT > 0: compile-time count
  template <int ARR, int COUNT>
  KFB_HD void flush_arr(const KfArgs& A, int count, int t0, int n, int lane) {
#if defined(__CUDA_ARCH__)
    double* base = out_base(A, ARR);
    if (!base) return;
    constexpr int w = out_width(ARR), off = out_off(ARR);
    const long long rows = (ARR == O_PS || ARR == O_PC) ? n + 1 : n;
    const long long r0 = (ARR == O_PS || ARR == O_PC) ? t0 + 1 : t0;
    if constexpr (COUNT > 0 && (32 % (COUNT * w)) == 0) {
      // The run of one unit divides the warp: lane -> (unit within the iteration, element) is fixed, so the shared-memory
      // source is one per-lane pointer plus an immediate and the global destination one per-lane pointer bumped by a
      // uniform stride - 4 instead of ~15 instructions per store (the generic index arithmetic below was half of the
      // full-output kernel's 460 instructions per step).
      constexpr int Lr = COUNT * w, UPI = 32 / Lr;  // doubles per unit, units per iteration
      const int ul = lane / Lr, e = lane - ul * Lr, sidx = e / w, i = e - sidx * w;
      const double* src = ostage + (size_t)(sidx * OUT_W + off + i) * OUT_LD + ul;
      double* dst = base + ((warp_u0 + ul) * rows + r0) * w + e;
      const long long stride = (long long)UPI * rows * w;
      const long long left = A.U - warp_u0;
      const int nvalid = left < 32 ? (int)left : 32;  // units of this warp that exist
#pragma unroll
      for (int it = 0; it < Lr; ++it) {
        if (it * UPI + ul < nvalid) *dst = src[it * UPI];
        dst += stride;
      }
      return;
    }
    const int Lc = (COUNT > 0 ? COUNT : count) * w;  // contiguous doubles per unit
#pragma unroll
    for (int it = 0; it < (COUNT > 0 ? COUNT * w : OUT_K * w); ++it) {
      if (COUNT == 0 && it >= Lc) break;
      const int idx = it * 32 + lane;
      const int unit = idx / Lc, e = idx - unit * Lc;
      const int sidx = e / w, i = e - sidx * w;
      if (warp_u0 + unit < A.U)
        base[((warp_u0 + unit) * rows + r0) * w + e] = ostage[(size_t)(sidx * OUT_W + off + i) * OUT_LD + unit];
    }
#endif
  }
  // called by every lane of the warp at the end of step t
  KFB_HD void end_step(const KfArgs& A, long long, int t, int n) {
#if defined(__CUDA_ARCH__)
    if (!ostage) return;
    const int slot = t % OUT_K;
    if (slot != OUT_K - 1 && t != n - 1) return;
    const int count = slot + 1, t0 = t - slot, lane = tid & 31;
    __syncwarp();
    if (count == OUT_K) {
      flush_arr<O_FS, OUT_K>(A, count, t0, n, lane);
      flush_arr<O_PS, OUT_K>(A, count, t0, n, lane);
      flush_arr<O_FC, OUT_K>(A, count, t0, n, lane);
      flush_arr<O_PC, OUT_K>(A, count, t0, n, lane);
      flush_arr<O_LL, OUT_K>(A, count, t0, n, lane);
    } else {
      flush_arr<O_FS, 0>(A, count, t0, n, lane);
      flush_arr<O_PS, 0>(A, count, t0, n, lane);
      flush_arr<O_FC, 0>(A, count, t0, n, lane);
      flush_arr<O_PC, 0>(A, count, t0, n, lane);
      flush_arr<O_LL, 0>(A, count, t0, n, lane);
    }
    __syncwarp();
#endif
  }

  static constexpr int KT = M + (M * (M + 1)) / 2;
  static constexpr int TAPE_DEPTH = 4;              // entries in flight
  static constexpr int TAPE_SLOTS = TAPE_DEPTH + 1;  // +1: the slot being refilled was consumed one step earlier

  // Streams the tape backwards.  Device: every thread cp.async's (LDGSTS) its own KT doubles of entries
  // t-1 .. t-DEPTH into its private column of a shared-memory ring; completion is tracked by cp.async groups, not
  // by the register scoreboard, so the loads never serialise with the arithmetic of the current step.
  struct TapeReader {
    const double* gp;
    long long tstep, telem;
    int next_t, slot_fetch, slot_read;
    KFB_HD TapeReader(ThreadCtx& x, const KfArgs& A, long long u) {
      tstep = x.tape_step(A);
      telem = x.tape_elem(A);
      gp = x.tape_base(A, u) + (long long)(A.n - 2) * tstep;  // entry of step n-1
      next_t = A.n - 1;
      slot_fetch = slot_read = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
      for (int s = 0; s < TAPE_DEPTH; ++s) issue(x);
#endif
    }
#if defined(__CUDA_ARCH__)
    __device__ __forceinline__ void issue(ThreadCtx& x) {
      if (next_t >= 1) {
        const unsigned dst = (unsigned)__cvta_generic_to_shared(x.ring + (size_t)slot_fetch * KT * x.nthr + x.tid);
#pragma unroll
        for (int k = 0; k < KT; ++k)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + (unsigned)(k * x.nthr * 8)),
                       "l"(gp + k * telem)
                       : "memory");
        gp -= tstep;
        --next_t;
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      slot_fetch = (slot_fetch + 1 == TAPE_SLOTS) ? 0 : slot_fetch + 1;
    }
#endif
    template <class TB>
    KFB_HD void get(ThreadCtx& x, TB& dst) {
#if defined(__CUDA_ARCH__)
      asm volatile("cp.async.wait_group %0;" ::"n"(TAPE_DEPTH - 1) : "memory");
      const double* src = x.ring + (size_t)slot_read * KT * x.nthr + x.tid;
#pragma unroll
      for (int k = 0; k < KT; ++k) dst[k] = src[k * x.nthr];
      slot_read = (slot_read + 1 == TAPE_SLOTS) ? 0 : slot_read + 1;
      issue(x);
#else
      for (int k = 0; k < KT; ++k) dst[k] = gp[k * telem];
      gp -= tstep;
#endif
    }
  };
  KFB_HD static constexpr int m() { return M; }
  KFB_HD static constexpr int p() { return P; }
  KFB_HD static constexpr int lane() { return 0; }
  KFB_HD static constexpr int G() { return 1; }
  KFB_HD void sync() const {}
  KFB_HD static constexpr int div_m(int i) { return i / M; }
  KFB_HD static constexpr int div_p(int i) { return i / P; }
  KFB_HD double reduce_max(double v) const { return v; }
  KFB_HD bool all_ok(bool v) const { return v; }
  KFB_HD const double* y_base(const KfArgs& A, long long series) const {
    return y_smem ? y_smem : A.y.p + series * A.y.bs;
  }
  // tape entry of step t (t >= 1) = tape_base + (t-1) * tape_step; element k at [k * tape_elem].
  // Layout [t-1][warp][k][32]: the entry of one step for the 32 units of a warp is KT * 256 contiguous bytes - every
  // tape load/store of a warp is still one fully-coalesced 256-byte transaction, and the k_endog = 1 adjoint
  // (kf_p1.cu) fetches the whole entry with ONE TMA bulk copy per warp and step.
  KFB_HD double* tape_base(const KfArgs& A, long long u) const { return A.tape + (u >> 5) * (KT * 32) + (u & 31); }
  KFB_HD long long tape_step(const KfArgs& A) const { return (long long)KT * tape_units_padded(A.U); }
  KFB_HD long long tape_elem(const KfArgs&) const { return 32; }
};

// Compile-time parameters of one thread-per-unit instantiation, handed to the caller's launcher as a tag.
template <int M_, int P_, int MK_, bool TV_>
struct ThreadInst {
  static constexpr int M = M_, P = P_, MK = MK_;
  static constexpr bool TV = TV_;
};

template <int M, int P, class Run>
bool with_thread_kind(int mk, bool tv, Run& run) {
  if (tv) {  // univariate / steady state: static matrices only
    if (mk != MK_STD) return false;
    run(ThreadInst<M, P, MK_STD, true>{});
    return true;
  }
  switch (mk) {
    case MK_STD: run(ThreadInst<M, P, MK_STD, false>{}); return true;
    case MK_UNIV: run(ThreadInst<M, P, MK_UNIV, false>{}); return true;
    case MK_STEADY: run(ThreadInst<M, P, MK_STEADY, false>{}); return true;
    default: return false;  // MK_CHOLS: cooperative kernels only
  }
}

template <int M, int P = 1, class Run>
bool with_thread_p(int p, int mk, bool tv, Run& run) {
  if constexpr (P > M || P > 3) return false;
  else return p == P ? with_thread_kind<M, P>(mk, tv, run) : with_thread_p<M, P + 1>(p, mk, tv, run);
}

// Which thread-per-unit kernels exist, for the device launchers (kf_thread.cu) and the host build of the kernels alike:
// k_states 1..4, k_endog 1..min(k_states, 3).  Calls run(ThreadInst<M, P, MK, TV>{}) and returns true, or returns false
// when (m, p, mk, tv) has no instantiation.
template <class Run>
bool with_thread_instance(int m, int p, int mk, bool tv, Run&& run) {
  switch (m) {
    case 1: return with_thread_p<1>(p, mk, tv, run);
    case 2: return with_thread_p<2>(p, mk, tv, run);
    case 3: return with_thread_p<3>(p, mk, tv, run);
    case 4: return with_thread_p<4>(p, mk, tv, run);
    default: return false;
  }
}

// ---------------------------------------------------------------------------
// CoopCtx: G lanes cooperate on one unit; run-time dims; buffers are bump-allocated from a per-unit
// shared-memory arena.  G == 32: one warp per unit (sync = __syncwarp); G == blockDim.x: one CTA per
// unit (sync = __syncthreads).  Tape layout [u][t-1][k]: the G lanes read/write consecutive doubles.
// ---------------------------------------------------------------------------
struct CoopCtx {
  static constexpr bool TV = true;
  static constexpr bool SKIP_LB = true;    // adjoint without T-bar / Z-bar: skip the dense Lb product (kf_pred.cuh)
  int m_, p_, lane_, G_;
  double* arena;
  int off, cap;
  bool overflow;
  double* red;  // 34 doubles of scratch for cross-lane reductions (CTA mode)

  KFB_HD void set_dims(int m, int p) {
    m_ = m;
    p_ = p;
  }
  // G lanes (this one is `lane`) on an empty arena of `cap` doubles; `red` is the caller's
  KFB_HD void init(int m, int p, double* arena_, int cap_, int lane, int G) {
    set_dims(m, p);
    arena = arena_;
    off = 0;
    cap = cap_;
    overflow = false;
    lane_ = lane;
    G_ = G;
  }
  // NOTE: a multiply-high ("magic number") division was tried here; nvcc 12.9 then mis-compiled the unrolled
  // P - K K^T F loop of univariate_inner for k_states = 30 (compute-sanitizer racecheck: cross-thread RAW hazard,
  // wrong results; the division itself was verified exact on the device).  Plain division is kept.
  KFB_HD int div_m(int i) const { return i / m_; }
  KFB_HD int div_p(int i) const { return i / p_; }

  KFB_HD int size_of(int sz) const {
    return sz == SZ_M ? m_ : sz == SZ_P ? p_ : sz == SZ_MM ? m_ * m_ : sz == SZ_MP ? m_ * p_ : sz == SZ_PP ? p_ * p_ : tape_width(m_);
  }
  KFB_HD double* bump(int cnt) {
    double* r = arena + off;
    off += cnt;
    if (off > cap) { overflow = true; r = arena; }
    return r;
  }
  template <int SZ>
  struct Buf {
    double* v;
    KFB_HD explicit Buf(CoopCtx& x) : v(x.bump(x.size_of(SZ))) {}
    KFB_HD double& operator[](int i) { return v[i]; }
    KFB_HD const double& operator[](int i) const { return v[i]; }
  };
  KFB_HD int m() const { return m_; }
  KFB_HD int p() const { return p_; }
  KFB_HD int lane() const { return lane_; }
  KFB_HD int G() const { return G_; }
  KFB_HD void sync() const {
#if defined(__CUDA_ARCH__)
    if (G_ <= 32) __syncwarp();
    else __syncthreads();
#endif
  }
  // max over the G lanes of a unit; every lane gets the result
  KFB_HD double reduce_max(double v) const {
#if defined(__CUDA_ARCH__)
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (G_ > 32) {
      __syncthreads();
      if ((lane_ & 31) == 0) red[lane_ >> 5] = v;
      __syncthreads();
      v = red[0];
      for (int w = 1; w < (G_ >> 5); ++w) v = fmax(v, red[w]);
    }
#endif
    return v;
  }
  // lane 0's flag, broadcast to every lane
  KFB_HD bool all_ok(bool v) const {
#if defined(__CUDA_ARCH__)
    if (G_ <= 32) return __shfl_sync(0xffffffffu, (int)v, 0) != 0;
    __syncthreads();
    if (lane_ == 0) red[33] = v ? 1.0 : 0.0;
    __syncthreads();
    return red[33] != 0.0;
#else
    return v;
#endif
  }
  template <class TS>
  KFB_HD void store_row(const KfArgs& A, int arr, long long u, long long rows, long long r, int w, const TS& src) {
    store_row_direct(*this, A, arr, u, rows, r, w, src);
  }
  KFB_HD void end_step(const KfArgs&, long long, int, int) {}
  KFB_HD const double* y_base(const KfArgs& A, long long series) const { return A.y.p + series * A.y.bs; }
  KFB_HD double* tape_base(const KfArgs& A, long long u) const {
    return A.tape + u * (long long)(A.n - 1) * tape_width(m_);
  }
  KFB_HD long long tape_step(const KfArgs&) const { return tape_width(m_); }
  KFB_HD long long tape_elem(const KfArgs&) const { return 1; }
  struct TapeReader {
    const double* gp;
    int kt;
    KFB_HD TapeReader(CoopCtx& x, const KfArgs& A, long long u) {
      kt = tape_width(x.m_);
      gp = x.tape_base(A, u) + (long long)(A.n - 2) * kt;
    }
    template <class TB>
    KFB_HD void get(CoopCtx& x, TB& dst) {
      for (int k = x.lane_; k < kt; k += x.G_) dst[k] = gp[k];
      gp -= kt;
      x.sync();
    }
  };
};

// 2x2 register-tiled product for the run-time-dims cooperative context: each lane owns a 2x2 block of C, so one
// multiply-add costs one shared-memory load instead of two, and the index arithmetic is paid per tile, not per
// element (k_states ~ 30: 225 tiles on a 256-thread CTA).
template <bool TA, bool TB, int MODE, class TC, class TAa, class TBb>
KFB_HD void gemm(CoopCtx& x, TC& C, const TAa& A, const TBb& B, int r, int kk, int c) {
  const int tr = (r + 1) >> 1, tc = (c + 1) >> 1;
  for (int tile = x.lane_; tile < tr * tc; tile += x.G_) {
    const int ti = tile / tc, tj = tile - ti * tc;
    const int i0 = 2 * ti, j0 = 2 * tj;
    const bool i1 = (i0 + 1 < r), j1 = (j0 + 1 < c);
    const int i1x = i1 ? i0 + 1 : i0, j1x = j1 ? j0 + 1 : j0;
    double s00 = 0.0, s01 = 0.0, s10 = 0.0, s11 = 0.0;
    if (MODE != 0) {
      s00 = C[i0 * c + j0];
      s01 = C[i0 * c + j1x];
      s10 = C[i1x * c + j0];
      s11 = C[i1x * c + j1x];
    }
#pragma unroll 2
    for (int k = 0; k < kk; ++k) {
      double a0 = A[TA ? k * r + i0 : i0 * kk + k];
      double a1 = A[TA ? k * r + i1x : i1x * kk + k];
      if (MODE == 2) { a0 = -a0; a1 = -a1; }
      const double b0 = B[TB ? j0 * kk + k : k * c + j0];
      const double b1 = B[TB ? j1x * kk + k : k * c + j1x];
      s00 = kf_fma(a0, b0, s00);
      s01 = kf_fma(a0, b1, s01);
      s10 = kf_fma(a1, b0, s10);
      s11 = kf_fma(a1, b1, s11);
    }
    C[i0 * c + j0] = s00;
    if (j1) C[i0 * c + j0 + 1] = s01;
    if (i1) C[(i0 + 1) * c + j0] = s10;
    if (i1 && j1) C[(i0 + 1) * c + j0 + 1] = s11;
  }
  x.sync();
}

// ---------------------------------------------------------------------------
// CoopCtxT<M,P,G>: G lanes (a power of two <= 32) cooperate on one unit, 32/G units per warp; COMPILE-TIME dims so
// every loop unrolls and all index arithmetic folds; matrices in shared memory.  Products whose row count fits the
// group run "row per lane": lane i keeps one output row in registers, reads A[i][k] once and the (broadcast) row
// B[k][:] - 1/c instead of 2 shared-memory loads per multiply-add (see the gemm overload below).
// Control flow must be uniform across the units of a warp: the launcher only uses this context when the observation
// stream is shared by all units (same missing pattern) and the matrices are static.
// ---------------------------------------------------------------------------
template <int M, int P, int G_>
struct CoopCtxT {
  static constexpr bool TV = false;
  static constexpr bool SKIP_LB = true;    // adjoint without T-bar / Z-bar: skip the dense Lb product (kf_pred.cuh)
  static constexpr int KT = M + (M * (M + 1)) / 2;
  int lane_;
  unsigned mask_;
  double* arena;
  int off;
  double* red;  // G_ > 32 only: 34 doubles of scratch for group-wide reductions
  int group_;   // G_ > 32 only: index of this unit's thread group in the CTA (named barrier 1 + group_)
  template <int SZ>
  KFB_HD static constexpr int size_of() {
    return SZ == SZ_M ? M : SZ == SZ_P ? P : SZ == SZ_MM ? M * M : SZ == SZ_MP ? M * P : SZ == SZ_PP ? P * P : KT;
  }
  template <int SZ>
  struct Buf {
    double* v;
    KFB_HD explicit Buf(CoopCtxT& x) : v(x.arena + x.off) { x.off += (size_of<SZ>() + 1) & ~1; }
    KFB_HD double& operator[](int i) { return v[i]; }
    KFB_HD const double& operator[](int i) const { return v[i]; }
  };
  KFB_HD static constexpr int m() { return M; }
  KFB_HD static constexpr int p() { return P; }
  KFB_HD static constexpr int G() { return G_; }
  KFB_HD static constexpr int div_m(int i) { return i / M; }
  KFB_HD static constexpr int div_p(int i) { return i / P; }
  KFB_HD int lane() const { return lane_; }
  KFB_HD void sync() const {
#if defined(__CUDA_ARCH__)
    if (G_ <= 32) __syncwarp(mask_);
    else asm volatile("bar.sync %0, %1;" ::"r"(1 + group_), "n"(G_) : "memory");  // named barrier: this unit's threads only
#endif
  }
  KFB_HD double reduce_max(double v) const {
#if defined(__CUDA_ARCH__)
    if (G_ <= 32) {
#pragma unroll
      for (int o = G_ / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(mask_, v, o, G_));
    } else {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
      sync();
      if ((lane_ & 31) == 0) red[lane_ >> 5] = v;
      sync();
      v = red[0];
#pragma unroll
      for (int w = 1; w < (G_ >> 5); ++w) v = fmax(v, red[w]);
    }
#endif
    return v;
  }
  KFB_HD bool all_ok(bool v) const {
#if defined(__CUDA_ARCH__)
    if (G_ <= 32) return __shfl_sync(mask_, (int)v, 0, G_) != 0;
    sync();
    if (lane_ == 0) red[33] = v ? 1.0 : 0.0;
    sync();
    return red[33] != 0.0;
#else
    return v;
#endif
  }
  template <class TS>
  KFB_HD void store_row(const KfArgs& A, int arr, long long u, long long rows, long long r, int w, const TS& src) {
    store_row_direct(*this, A, arr, u, rows, r, w, src);
  }
  KFB_HD void end_step(const KfArgs&, long long, int, int) {}
  KFB_HD const double* y_base(const KfArgs& A, long long series) const { return A.y.p + series * A.y.bs; }
  KFB_HD double* tape_base(const KfArgs& A, long long u) const { return A.tape + u * (long long)(A.n - 1) * KT; }
  KFB_HD long long tape_step(const KfArgs&) const { return KT; }
  KFB_HD long long tape_elem(const KfArgs&) const { return 1; }
  struct TapeReader {
    const double* gp;
    KFB_HD TapeReader(CoopCtxT& x, const KfArgs& A, long long u) {
      gp = x.tape_base(A, u) + (long long)(A.n - 2) * KT;
    }
    template <class TB>
    KFB_HD void get(CoopCtxT& x, TB& dst) {
#pragma unroll
      for (int k = x.lane_; k < KT; k += G_) dst[k] = gp[k];
      gp -= KT;
      x.sync();
    }
  };
};

// Row-per-lane product for CoopCtxT (more specialised than the generic gemm in kf_core.cuh).
template <bool TA, bool TB, int MODE, int M, int P, int G_, class TC, class TAa, class TBb>
KFB_HD void gemm(CoopCtxT<M, P, G_>& x, TC& C, const TAa& A, const TBb& B, int r, int kk, int c) {
  constexpr int CMAX = (M > P ? M : P);
  if (G_ > 32) {
    // one CTA per unit: 2x2 register tiles, fully unrolled k loop with constant shared-memory offsets.
    // (Measured alternative: 64 threads per unit with 4x4 tiles - fewer shared-memory wavefronts per multiply-add but
    //  only 2 units = 4 warps resident per SM in the adjoint: 1.24e7 vs 1.30e7 steps/s on config 4.)
    const int tr = (r + 1) >> 1, tc = (c + 1) >> 1;
    const double* Ap = &A[0];
    const double* Bp = &B[0];
#pragma unroll
    for (int tile = x.lane(); tile < tr * tc; tile += G_) {
      const int ti = tile / tc, tj = tile - ti * tc;
      const int i0 = 2 * ti, j0 = 2 * tj;
      const bool i1 = (i0 + 1 < r), j1 = (j0 + 1 < c);
      const int i1x = i1 ? i0 + 1 : i0, j1x = j1 ? j0 + 1 : j0;
      double s00 = 0.0, s01 = 0.0, s10 = 0.0, s11 = 0.0;
      if (MODE != 0) {
        s00 = C[i0 * c + j0];
        s01 = C[i0 * c + j1x];
        s10 = C[i1x * c + j0];
        s11 = C[i1x * c + j1x];
      }
      const double* a0p = Ap + (TA ? i0 : i0 * kk);
      const double* a1p = Ap + (TA ? i1x : i1x * kk);
      const double* b0p = Bp + (TB ? j0 * kk : j0);
      const double* b1p = Bp + (TB ? j1x * kk : j1x);
#pragma unroll
      for (int k = 0; k < CMAX; ++k) {
        if (k < kk) {
          double a0 = a0p[TA ? k * r : k];
          double a1 = a1p[TA ? k * r : k];
          if (MODE == 2) { a0 = -a0; a1 = -a1; }
          double b0, b1;
#if defined(__CUDA_ARCH__)
          if (!TB && (c % 2 == 0)) {
            const double2 t = *reinterpret_cast<const double2*>(b0p + k * c);
            b0 = t.x;
            b1 = t.y;
          } else
#endif
          {
            b0 = b0p[TB ? k : k * c];
            b1 = b1p[TB ? k : k * c];
          }
          s00 = kf_fma(a0, b0, s00);
          s01 = kf_fma(a0, b1, s01);
          s10 = kf_fma(a1, b0, s10);
          s11 = kf_fma(a1, b1, s11);
        }
      }
      C[i0 * c + j0] = s00;
      if (j1) C[i0 * c + j0 + 1] = s01;
      if (i1) C[(i0 + 1) * c + j0] = s10;
      if (i1 && j1) C[(i0 + 1) * c + j0 + 1] = s11;
    }
  } else if (r <= G_) {
    const int i = x.lane();
    if (i < r) {
      double acc[CMAX];
      double arow[CMAX];
#pragma unroll
      for (int j = 0; j < CMAX; ++j)
        if (j < c) acc[j] = (MODE == 0) ? 0.0 : C[i * c + j];
      // own row of A: one 16-byte shared-memory load per two elements when the row is 16-byte aligned
      const double* Ap = &A[0];
      const double* Bp = &B[0];
#if defined(__CUDA_ARCH__)
      if (!TA && (kk % 2 == 0)) {
#pragma unroll
        for (int k = 0; k < CMAX; k += 2)
          if (k < kk) {
            const double2 t = *reinterpret_cast<const double2*>(Ap + i * kk + k);
            arow[k] = t.x;
            arow[k + 1 < CMAX ? k + 1 : k] = t.y;
          }
      } else
#endif
      {
#pragma unroll
        for (int k = 0; k < CMAX; ++k)
          if (k < kk) arow[k] = Ap[TA ? k * r + i : i * kk + k];
      }
#pragma unroll
      for (int k = 0; k < CMAX; ++k) {
        if (k < kk) {
          const double av = (MODE == 2) ? -arow[k] : arow[k];
#if defined(__CUDA_ARCH__)
          if (!TB && (c % 2 == 0)) {  // broadcast row B[k][:] with 16-byte loads
#pragma unroll
            for (int j = 0; j < CMAX; j += 2)
              if (j < c) {
                const double2 t = *reinterpret_cast<const double2*>(Bp + k * c + j);
                acc[j] = kf_fma(av, t.x, acc[j]);
                acc[j + 1 < CMAX ? j + 1 : j] = kf_fma(av, t.y, acc[j + 1 < CMAX ? j + 1 : j]);
              }
          } else
#endif
          {
#pragma unroll
            for (int j = 0; j < CMAX; ++j)
              if (j < c) acc[j] = kf_fma(av, Bp[TB ? j * kk + k : k * c + j], acc[j]);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < CMAX; ++j)
        if (j < c) C[i * c + j] = acc[j];
    }
  } else {
    KFB_FOR(idx, r * c) {
      const int i = idx / c, j = idx - i * c;
      double s = (MODE == 0) ? 0.0 : C[idx];
#pragma unroll
      for (int k = 0; k < kk; ++k) {
        const double av = A[TA ? k * r + i : i * kk + k];
        s = kf_fma(MODE == 2 ? -av : av, B[TB ? j * kk + k : k * c + j], s);
      }
      C[idx] = s;
    }
  }
  x.sync();
}

// doubles of arena one unit needs (upper bound of what forward_unit / backward_unit bump-allocate)
inline int coop_arena_doubles(int m, int p, bool backward) {
  const int mm = m * m, mp = m * p, pp = p * p, kt = m + (m * (m + 1)) / 2;
  const int params = mm + mp + pp + p + pp;
  const int upd = 3 * p + 3 * mp + 4 * pp + 3 * mm;    // UpdTmp  (kf_core.cuh)
  const int prd = 3 * p + 4 * mp + 4 * pp + 3 * mm;    // PredTmp (kf_pred.cuh)
  int a, b;
  if (!backward) {
    a = params + 3 * mm + 5 * m + upd;                 // forward_unit
    b = params + 2 * mm + 3 * m + prd;                 // forward_unit_pred
  } else {
    a = params + 8 * mm + 8 * m + 4 * mp + 4 * pp + 2 * p + upd + kt;  // backward_unit
    b = params + 7 * mm + 4 * m + 5 * mp + 4 * pp + 2 * p + prd + kt;  // backward_unit_pred
  }
  return a > b ? a : b;
}

}  // namespace kfb
