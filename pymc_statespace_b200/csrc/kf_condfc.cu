// kf_condfc.cu - kernels of the conditional forecasts (kf_condfc.cuh): a window kernel, one thread per unit, and a
// paths kernel, one thread per simulation; and the masked filter over the sample, one thread per unit.
#include "kf_aux.cuh"
#include "kf_condfc.cuh"

namespace kfb {

// (128, 1): without the minimum-blocks hint ptxas capped several instantiations near 96-128 registers and spilled;
// with it none spills.  One thread per unit, so occupancy is not what this kernel is limited by.
template <class D>
__global__ void __launch_bounds__(128, 1) condfc_window_kernel(D d, cf::Args A) {
  const long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= A.U) return;
  cf::window_unit(d, A, u);
}

template <class D>
__global__ void __launch_bounds__(128) condfc_paths_kernel(D d, cf::Args A) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= A.S) return;
  cf::path_unit(d, A, s);
}

// One thread per unit, as the window kernel (the same per-step products, so the same register budget).
template <class D>
__global__ void __launch_bounds__(128, 1) masked_filter_kernel(D d, cf::FilterArgs A) {
  const long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= A.U) return;
  cf::filter_unit(d, A, u);
}

cudaError_t launch_masked_filter(const cf::FilterArgs& A, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  const bool ok = ss::with_instance(A.m, A.p, A.r, [&](auto d) {
    masked_filter_kernel<decltype(d)><<<(unsigned)((A.U + 127) / 128), 128, 0, st>>>(d, A);
    count_launch();
    e = cudaGetLastError();
  });
  return ok ? e : cudaErrorInvalidConfiguration;
}

cudaError_t launch_conditional_forecast(const cf::Args& A, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  const bool ok = ss::with_instance(A.m, A.p, A.r, [&](auto d) {
    using D = decltype(d);
    condfc_window_kernel<D><<<(unsigned)((A.U + 127) / 128), 128, 0, st>>>(d, A);
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess || A.S == 0) return;
    condfc_paths_kernel<D><<<(unsigned)((A.S + 127) / 128), 128, 0, st>>>(d, A);
    count_launch();
    e = cudaGetLastError();
  });
  return ok ? e : cudaErrorInvalidConfiguration;
}

}  // namespace kfb
