// kf_coop.cu - cooperative (shared-memory) kernels: any (k_states, k_endog), time-varying matrices.
#include "kf_kernels.cuh"

namespace kfb {

// Launch geometry of the run-time-dims kernels (kf_coop_kernel, kf_smoother_kernel, kf_dare_kernel).  warp: one warp per
// unit, 4 per CTA; otherwise one 256-thread CTA per unit.  arena: doubles per unit; 0 when one arena exceeds the 227 KB
// of shared memory a CTA can have.
struct CoopGeometry {
  bool warp;
  int block;
  unsigned grid;
  size_t smem;
  int arena;
};

// Warp per unit for small systems (a 32-lane warp covers the m*m outputs of a product in a few rounds) when the caller
// allows it and 4 arenas fit in one CTA's shared memory; one 256-thread CTA per unit otherwise.
static CoopGeometry coop_geometry(int arena_doubles, long long units, bool warp_ok) {
  const int arena = (arena_doubles + 1) & ~1;  // keep every arena 16-byte aligned
  const size_t arena_bytes = (size_t)arena * sizeof(double);
  const size_t smem_max = 227 * 1024;
  if (arena_bytes > smem_max) return {false, 0, 0, 0, 0};
  if (warp_ok && arena_bytes * 4 <= smem_max) return {true, 4 * 32, (unsigned)((units + 3) / 4), arena_bytes * 4, arena};
  return {false, 256, (unsigned)units, arena_bytes, arena};
}

template <int MK, bool WARP>
static void launch_coop_kind(const KfArgs& A, bool bwd, const CoopGeometry& g, cudaStream_t s) {
  with_mode(kernel_mode(A, bwd), [&](auto md) {
    auto kern = kf_coop_kernel<MK, decltype(md)::MODE, WARP>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem);
    kern<<<g.grid, g.block, g.smem, s>>>(A, g.arena);
  });
}

template <bool WARP>
static cudaError_t launch_coop_mode(const KfArgs& A, bool bwd, const CoopGeometry& g, cudaStream_t s) {
  switch (A.math_kind) {
    case MK_STD: launch_coop_kind<MK_STD, WARP>(A, bwd, g, s); break;
    case MK_UNIV: launch_coop_kind<MK_UNIV, WARP>(A, bwd, g, s); break;
    case MK_STEADY: launch_coop_kind<MK_STEADY, WARP>(A, bwd, g, s); break;
    case MK_CHOLS: launch_coop_kind<MK_CHOLS, WARP>(A, bwd, g, s); break;
    default: return cudaErrorInvalidValue;
  }
  count_launch();
  return cudaGetLastError();
}

// one 256-thread CTA per unit from k_states = 16 up (>= 256 outputs per product)
cudaError_t launch_coop(const KfArgs& A, bool bwd, cudaStream_t s) {
  const CoopGeometry g = coop_geometry(coop_arena_doubles(A.m, A.p, bwd), A.U, A.m < 16);
  if (!g.arena) return cudaErrorInvalidConfiguration;
  return g.warp ? launch_coop_mode<true>(A, bwd, g, s) : launch_coop_mode<false>(A, bwd, g, s);
}

cudaError_t launch_smoother(const SmoothArgs& S, cudaStream_t s) {
  const CoopGeometry g = coop_geometry(smoother_arena_doubles(S.m), S.U, S.m < 16);
  if (!g.arena) return cudaErrorInvalidConfiguration;
  auto kern = g.warp ? kf_smoother_kernel<true> : kf_smoother_kernel<false>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem);
  kern<<<g.grid, g.block, g.smem, s>>>(S, g.arena);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_dare(const DareArgs& D, bool bwd, cudaStream_t s) {
  const CoopGeometry g = coop_geometry(dare_arena_doubles(D.m, D.p), bwd ? D.U : D.nD, true);
  if (!g.arena) return cudaErrorInvalidConfiguration;
  auto kern = g.warp ? (bwd ? kf_dare_kernel<true, true> : kf_dare_kernel<false, true>)
                     : (bwd ? kf_dare_kernel<true, false> : kf_dare_kernel<false, false>);
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem);
  kern<<<g.grid, g.block, g.smem, s>>>(D, g.arena);
  count_launch();
  return cudaGetLastError();
}

}  // namespace kfb
