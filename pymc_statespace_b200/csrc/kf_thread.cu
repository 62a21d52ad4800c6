// kf_thread.cu - the thread-per-unit kernels of one k_states, KFB_M (compiled once per size with -DKFB_M=<m>, see the
// Makefile), so that each k_states compiles in its own translation unit (parallel build).
#include "kf_kernels.cuh"

namespace kfb {

template <int M, int P, int MK, bool TV>
static cudaError_t launch_thread(const KfArgs& A, bool bwd, int y_smem_doubles, int bulk_ok, cudaStream_t s) {
  const int block = KFB_THREAD_BLOCK;
  const unsigned grid = (unsigned)((A.U + block - 1) / block);
  size_t smem = (size_t)((y_smem_doubles + 1) & ~1) * sizeof(double);
  if (bwd) smem += (size_t)ThreadCtx<M, P>::TAPE_SLOTS * ThreadCtx<M, P>::KT * block * sizeof(double);
  const int mode = kernel_mode(A, bwd);
  if (mode == 1)  // per-warp output stager of the full-output kernel (kf_ctx.cuh)
    smem += (size_t)ThreadCtx<M, P, TV>::OUT_DOUBLES * (block / 32) * sizeof(double);
  with_mode(mode, [&](auto md) {
    auto kern = kf_thread_kernel<M, P, MK, decltype(md)::MODE, TV>;
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, block, smem, s>>>(A, y_smem_doubles, bulk_ok);
  });
  count_launch();
  return cudaGetLastError();
}

#define KFB_CAT2(a, b) a##b
#define KFB_CAT(a, b) KFB_CAT2(a, b)

static cudaError_t launch_smoother_thread(const SmoothArgs& S, cudaStream_t s) {
  kf_smoother_thread_kernel<KFB_M><<<(unsigned)((S.U + 127) / 128), 128, 0, s>>>(S);
  count_launch();
  return cudaGetLastError();
}
smoother_launch_fn KFB_CAT(smoother_thread_m, KFB_M)() { return launch_smoother_thread; }

thread_launch_fn KFB_CAT(thread_launcher_m, KFB_M)(int p, int mk, bool tv) {
  thread_launch_fn fn = nullptr;
  with_thread_instance(KFB_M, p, mk, tv, [&](auto v) {
    using V = decltype(v);
    if constexpr (V::M == KFB_M) fn = launch_thread<V::M, V::P, V::MK, V::TV>;
  });
  return fn;
}

}  // namespace kfb
