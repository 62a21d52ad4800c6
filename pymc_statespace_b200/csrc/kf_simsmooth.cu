// kf_simsmooth.cu - kernels of the simulation smoother (kf_simsmooth.cuh): a gain pass, one thread per (unit, t), and a
// per-simulation kernel, one thread per simulation with the three passes of kf_simsmooth.cuh's simulate_one.
#include "kf_aux.cuh"
#include "kf_simsmooth.cuh"

namespace kfb {

template <class D>
__global__ void __launch_bounds__(128) simsmooth_gain_kernel(D d, ss::Args A) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.U * A.n) return;
  const long long u = i / A.n;
  const int t = (int)(i - u * A.n);
  if (t == 0) ss::unit_prep(A, u);
  ss::gain_entry(d, A, u, t);
}

template <class D>
__global__ void __launch_bounds__(128) simsmooth_sim_kernel(D d, ss::Args A) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= A.S) return;
  ss::simulate_one(d, A, s);
}

// ustat must hold ss::KEY_NONE in every entry (a 0x7f byte memset) before the call.
cudaError_t launch_simulation_smoother(const ss::Args& A, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  const bool ok = ss::with_instance(A.m, A.p, A.r, [&](auto d) {
    using D = decltype(d);
    const long long g = A.U * A.n;
    simsmooth_gain_kernel<D><<<(unsigned)((g + 127) / 128), 128, 0, st>>>(d, A);
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return;
    simsmooth_sim_kernel<D><<<(unsigned)((A.S + 127) / 128), 128, 0, st>>>(d, A);
    count_launch();
    e = cudaGetLastError();
  });
  return ok ? e : cudaErrorInvalidConfiguration;
}

}  // namespace kfb
