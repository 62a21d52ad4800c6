// kf_forecast.cu - kernels of the forecast paths and impulse responses (kf_forecast.cuh): a prep kernel, one thread per
// unit; a per-simulation kernel, one thread per simulation; an impulse-response kernel, one thread per (draw, shock).
#include "kf_aux.cuh"
#include "kf_forecast.cuh"

namespace kfb {

__global__ void __launch_bounds__(128) forecast_prep_kernel(fc::Args A) {
  const long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= A.U) return;
  fc::unit_prep(A, u);
}

template <class D>
__global__ void __launch_bounds__(128) forecast_paths_kernel(D d, fc::Args A) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= A.S) return;
  fc::path_one(d, A, s);
}

template <class D>
__global__ void __launch_bounds__(128) impulse_response_kernel(D d, fc::IrfArgs A) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.nD * A.r) return;
  fc::irf_one(d, A, i);
}

cudaError_t launch_forecast_paths(const fc::Args& A, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  const bool ok = ss::with_instance(A.m, A.p, A.r, [&](auto d) {
    using D = decltype(d);
    forecast_prep_kernel<<<(unsigned)((A.U + 127) / 128), 128, 0, st>>>(A);
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return;
    forecast_paths_kernel<D><<<(unsigned)((A.S + 127) / 128), 128, 0, st>>>(d, A);
    count_launch();
    e = cudaGetLastError();
  });
  return ok ? e : cudaErrorInvalidConfiguration;
}

cudaError_t launch_impulse_response(const fc::IrfArgs& A, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  const bool ok = ss::with_instance(A.m, A.p, A.r, [&](auto d) {
    using D = decltype(d);
    const long long g = A.nD * A.r;
    impulse_response_kernel<D><<<(unsigned)((g + 127) / 128), 128, 0, st>>>(d, A);
    count_launch();
    e = cudaGetLastError();
  });
  return ok ? e : cudaErrorInvalidConfiguration;
}

}  // namespace kfb
