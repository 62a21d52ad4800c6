// kf_coopT.cu - the compile-time-dims kernels of one k_states, KFB_M (compiled once per size with -DKFB_M=<m>, see the
// Makefile): sub-warp cooperative kernels, fused row kernels and, from k_states 10, the tensor-core DARE.
#include <atomic>

#include "kf_kernels.cuh"

namespace kfb {

// Per-device cache of a launch parameter chosen by an occupancy query.  Several host threads may race to fill a slot:
// the computation is idempotent and the slot is an atomic, so the worst case is a repeated query (kfb200.h promises
// re-entrancy across host threads).
struct WpcCache {
  std::atomic<int> v[32];
  WpcCache() { for (auto& a : v) a.store(0, std::memory_order_relaxed); }
  template <class F>
  int get(F&& compute) {
    int dev = 0;
    cudaGetDevice(&dev);
    std::atomic<int>& slot = v[dev & 31];
    int w = slot.load(std::memory_order_acquire);
    if (w == 0) {
      w = compute();
      slot.store(w, std::memory_order_release);
    }
    return w;
  }
};

template <int M, int P, int G, int MK>
static cudaError_t launch_coopT(const KfArgs& A, bool bwd, cudaStream_t s) {
  const int block = G > 128 ? G : 128;
  const int units = block / G;
  const int arena = (coop_arena_doubles(M, P, bwd) + 64 + 34 + 1) & ~1;  // + even-rounding slack: <= 1 double per buffer, < 64 buffers (kernel traps otherwise)
  const size_t smem = (size_t)arena * units * sizeof(double);
  if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
  const unsigned grid = (unsigned)((A.U + units - 1) / units);
  with_mode(kernel_mode(A, bwd), [&](auto md) {
    auto kern = kf_coopT_kernel<M, P, G, MK, decltype(md)::MODE>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    kern<<<grid, block, smem, s>>>(A, arena);
  });
  count_launch();
  return cudaGetLastError();
}

// Launches `kern` on `units` units, `upw` per warp with `per_unit` bytes of shared memory each.  Warps per CTA: of 4, 2
// and 1, the width that keeps most warps resident per SM (shared memory is the limiter), larger CTAs on ties; chosen by
// occupancy query once per device.  Every instantiated layout fits at one warp, the width used when no query succeeds.
template <class Args>
static cudaError_t launch_occupancy(void (*kern)(const Args), size_t per_unit, int upw, long long units, const Args& a,
                                    WpcCache& cache, cudaStream_t s) {
  const int wpc = cache.get([&] {
    int best = 0, best_w = 1;
    for (int w = 4; w >= 1; w >>= 1) {
      const size_t smem = per_unit * upw * w;
      if (smem > 227 * 1024) continue;
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, 32 * w, smem) != cudaSuccess) continue;
      if (nb * w > best) {
        best = nb * w;
        best_w = w;
      }
    }
    return best_w;
  });
  const size_t smem = per_unit * upw * wpc;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  const long long per_cta = (long long)upw * wpc;
  const unsigned grid = (unsigned)((units + per_cta - 1) / per_cta);
  kern<<<grid, 32 * wpc, smem, s>>>(a);
  count_launch();
  return cudaGetLastError();
}

#if KFB_M <= 8
// standard-family hot path (loglik + tape, adjoint): fused row-block-per-lane kernels; everything else: generic CoopCtxT
template <int M, int P, int G, int MK, bool BWD, bool NEED_Z>
static cudaError_t launch_rows(const KfArgs& A, cudaStream_t s) {
  constexpr size_t per_unit =
      (size_t)(BWD ? RowsLayout<M, P, NEED_Z, MK == MK_STEADY || MK == MK_CHOLS>::bwd_doubles : RowsLayout<M, P>::fwd_doubles) *
      sizeof(double);
  static WpcCache cache;
  return launch_occupancy(kf_rows_kernel<M, P, G, MK, BWD, NEED_Z>, per_unit, RowsCfg<M, P, G>::UPW, A.U, A, cache, s);
}

// all six outputs of the reference on the same mapping (rows_forward_full; MK_STD / MK_STEADY)
template <int M, int P, int G, int MK>
static cudaError_t launch_rows_full(const KfArgs& A, cudaStream_t s) {
  constexpr size_t per_unit = (size_t)RowsLayout<M, P>::fwd_doubles * sizeof(double);
  static WpcCache cache;
  return launch_occupancy(kf_rowsfull_kernel<M, P, G, MK>, per_unit, RowsCfg<M, P, G>::UPW, A.U, A, cache, s);
}

// UnivariateFilter hot path (loglik-only forward, adjoint without Z-bar): fused kf_rowsU.cuh; everything else generic
template <int M, int P, bool BWD>
static cudaError_t launch_rowsU(const KfArgs& A, cudaStream_t s) {
  constexpr size_t per_unit = (size_t)(BWD ? RowsULayout<M, P>::bwd_doubles : RowsULayout<M, P>::fwd_doubles) * sizeof(double);
  auto kern = kf_rowsU_kernel<M, P, BWD>;
  const int wpc = 4;
  const size_t smem = per_unit * 4 * wpc;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const long long per_cta = 4LL * wpc;
  const unsigned grid = (unsigned)((A.U + per_cta - 1) / per_cta);
  kern<<<grid, 32 * wpc, smem, s>>>(A);
  count_launch();
  return cudaGetLastError();
}

template <int M, int P>
static cudaError_t launch_univ_or_coopT(const KfArgs& A, bool bwd, cudaStream_t s) {
  if ((!bwd && wants_step_outputs(A)) || (bwd && A.gZ)) return launch_coopT<M, P, 8, MK_UNIV>(A, bwd, s);
  return bwd ? launch_rowsU<M, P, true>(A, s) : launch_rowsU<M, P, false>(A, s);
}

template <int M, int P, int MK>
static cudaError_t launch_rows_or_coopT(const KfArgs& A, bool bwd, cudaStream_t s) {
  constexpr int G = 4;
  if (!bwd && wants_step_outputs(A)) {
    if constexpr (MK == MK_STD || MK == MK_STEADY) return launch_rows_full<M, P, G, MK>(A, s);
    else return launch_coopT<M, P, 8, MK>(A, bwd, s);  // as-coded multivariate Cholesky filter: generic sub-warp kernels
  }
  if (!bwd) return launch_rows<M, P, G, MK, false, false>(A, s);
  if (A.gZ) {
    // Z-bar requested (not by any of the reference's models): one row per lane (the two-row variant runs out of
    // registers); steady state with Z-bar stays on the generic kernels
    if (MK != MK_STD) return launch_coopT<M, P, 8, MK>(A, bwd, s);
    return launch_rows<M, P, 8, MK_STD, true, true>(A, s);
  }
  return launch_rows<M, P, G, MK, true, false>(A, s);
}
#endif

#if KFB_M > 8
// large systems, standard-family hot path: fused row-per-lane / warp-per-unit kernels with the m^3 products on the FP64
// tensor cores (kf_rowsD.cuh); full outputs, Z-bar and the other filters stay on the generic CoopCtxT path (one
// 256-thread CTA per unit).  (The warp-per-unit DFMA kernel of round 1 lost the A/B: profiles/r1_ncu_rowsL.md.)
template <int M, int P, int MK, bool BWD, bool NEED_T>
static cudaError_t launch_rowsD_impl(const KfArgs& A, cudaStream_t s) {
  constexpr size_t per_unit =
      (size_t)(BWD ? RowsDLayout<M, P, NEED_T>::bwd_doubles : RowsDLayout<M, P, false>::fwd_doubles) * sizeof(double);
  static WpcCache cache;
  return launch_occupancy(kf_rowsD_kernel<M, P, MK, BWD, NEED_T>, per_unit, 1, A.U, A, cache, s);
}

// all six outputs of the reference on the same mapping (rowsD_forward_full)
template <int M, int P, int MK>
static cudaError_t launch_rowsD_full(const KfArgs& A, cudaStream_t s) {
  constexpr size_t per_unit = (size_t)RowsDLayout<M, P, false>::fwd_doubles * sizeof(double);
  static WpcCache cache;
  return launch_occupancy(kf_rowsDfull_kernel<M, P, MK>, per_unit, 1, A.U, A, cache, s);
}

// steady-state covariance (forward DARE solve) on the same mapping
template <int M, int P>
static cudaError_t launch_dareD(const DareArgs& D, cudaStream_t s) {
  constexpr size_t per_unit = (size_t)DareDLayout<M, P>::doubles * sizeof(double);
  static WpcCache cache;
  return launch_occupancy(kf_dareD_kernel<M, P>, per_unit, 1, D.nD, D, cache, s);
}

template <int M, int P, int MK>
static cudaError_t launch_rowsD_or_coopT(const KfArgs& A, bool bwd, cudaStream_t s) {
  if (!bwd && wants_step_outputs(A)) return launch_rowsD_full<M, P, MK>(A, s);
  if (bwd && A.gZ) {
    // k_states 10..16: the run-time-dims kernels (one warp per unit below 16 states); 18..32: compile-time CTA per unit
    if constexpr (M <= 16) return launch_coop(A, bwd, s);
    else return launch_coopT<M, P, 256, MK>(A, bwd, s);
  }
  if (!bwd) return launch_rowsD_impl<M, P, MK, false, false>(A, s);
  return A.gT ? launch_rowsD_impl<M, P, MK, true, true>(A, s) : launch_rowsD_impl<M, P, MK, true, false>(A, s);
}
#endif

template <int M, int P>
static coopT_launch_fn pick_kindT(int mk) {
  constexpr int G = (M <= 8) ? 8 : 256;  // sub-warp groups for k_states 5..8; one 256-thread CTA per unit for large systems
  (void)G;  // k_states 10..16 instantiate only the tensor-core row kernels (everything else: run-time-dims kernels)
  switch (mk) {
#if KFB_M <= 8
    case MK_STD: return launch_rows_or_coopT<M, P, MK_STD>;
#else
    case MK_STD: return launch_rowsD_or_coopT<M, P, MK_STD>;
#endif
#if KFB_M <= 8
    case MK_UNIV: return launch_univ_or_coopT<M, P>;
#elif KFB_M > 16
    case MK_UNIV: return launch_coopT<M, P, G, MK_UNIV>;
#endif
#if KFB_M <= 8
    case MK_STEADY: return launch_rows_or_coopT<M, P, MK_STEADY>;
    case MK_CHOLS:  // as-coded multivariate Cholesky filter (SURVEY A.2-Q4): fused rows on the hot path like MK_STD
      return P > 1 ? launch_rows_or_coopT<M, P, MK_CHOLS> : launch_coopT<M, P, G, MK_CHOLS>;
#else
    case MK_STEADY: return launch_rowsD_or_coopT<M, P, MK_STEADY>;
#endif
    default: return nullptr;
  }
}

#define KFB_CAT2(a, b) a##b
#define KFB_CAT(a, b) KFB_CAT2(a, b)

#if KFB_M > 8
dare_launch_fn KFB_CAT(dareD_launcher_m, KFB_M)(int p) { return p == 1 ? launch_dareD<KFB_M, 1> : nullptr; }
#endif

coopT_launch_fn KFB_CAT(coopT_launcher_m, KFB_M)(int p, int mk) {
  switch (p) {
    case 1: return pick_kindT<KFB_M, 1>(mk);
#if KFB_M <= 8
    case 2: return pick_kindT<KFB_M, 2>(mk);
    case 3: return pick_kindT<KFB_M, 3>(mk);
#endif
    default: return nullptr;
  }
}

}  // namespace kfb
