// kf_tpar_smooth.cu - time-parallel RTS smoother kernel (kfb_smoother_ex with KFB_FLAG_TIME_PARALLEL): one CTA per unit,
// a blocked suffix scan over time.  The math is in kf_tpar_smooth.cuh.
#include "kf_kernels.cuh"
#include "kf_tpar_smooth.cuh"

namespace kfb {

namespace {

using namespace tpar;

template <int M, int NT>
__global__ void __launch_bounds__(NT) kf_tpar_smoother_kernel(const __grid_constant__ SmoothArgs S) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  const long long u = blockIdx.x;
  const int tid = threadIdx.x;
  const auto [lo, hi] = chunk_of(tid, NT, S.n);
  const SmoothView v = smooth_view(S, u);

  // 1. fold this thread's chunk (f_lo o .. o f_{hi-1}) straight into its shared-memory slot: the aggregate's E stays out
  // of the registers the gain needs
  SmoothElem<M>* sh = reinterpret_cast<SmoothElem<M>*>(kf_dyn_smem);
  smooth_fold<M>(v, lo, hi, sh[tid]);
  // 2. inclusive suffix scan of the chunk aggregates
  cta_scan<SmoothElem<M>, NT, true>(sh, smooth_combine<M>);
  // 3-4. literal walk of the chunk from the successor's smoothed moments at hi, checked against the scan at lo
  const bool drift = smooth_walk_check<M>(v, lo, hi, tid + 1 < NT ? &sh[tid + 1] : nullptr, sh[tid], TPAR_DRIFT_TOL);
  if (__syncthreads_or(drift)) {
    // the scan lost accuracy somewhere: the sequential recursion on one thread overwrites the unit's outputs
    if (tid == 0) smooth_sequential<M>(v);
  }
}

template <int M>
cudaError_t launch_tpar_smoother_m(const SmoothArgs& S, cudaStream_t s) {
  constexpr int NT = tpar_threads<M>();
  constexpr size_t smem = NT * sizeof(SmoothElem<M>);
  static_assert(smem <= 48 * 1024, "the scan's shared memory needs no opt-in");
  kf_tpar_smoother_kernel<M, NT><<<(unsigned)S.U, NT, smem, s>>>(S);
  count_launch();
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_tpar_smoother(const SmoothArgs& S, cudaStream_t s) {
  cudaError_t e = cudaErrorInvalidConfiguration;
  tpar::with_instance(S.m, [&](auto M) { e = launch_tpar_smoother_m<M>(S, s); });
  return e;
}

}  // namespace kfb
