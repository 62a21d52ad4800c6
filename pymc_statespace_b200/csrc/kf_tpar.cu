// kf_tpar.cu - time-parallel forward / adjoint kernels (KFB_FLAG_TIME_PARALLEL): one CTA per unit, blocked scans over
// time.  The math is in kf_tpar.cuh.
#include "kf_kernels.cuh"
#include "kf_tpar.cuh"

namespace kfb {

namespace {

using namespace tpar;

template <int M, int NT>
__global__ void __launch_bounds__(NT) kf_tpar_forward_kernel(const __grid_constant__ KfArgs A) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  const long long u = blockIdx.x;
  const int tid = threadIdx.x, n = A.n;
  const UnitView v = unit_view(A, u);
  const auto [lo, hi] = chunk_of(tid, NT, n);
  double* tape = A.tape + u * (long long)n * tape_entry<M>();

  // 1. fold this thread's chunk of filtering elements
  FiltElem<M> agg;
  const bool sequential = __syncthreads_or(!filt_fold_chunk<M>(v, lo, hi, agg));
  if (sequential) {
    // an element has no parallel form: this unit runs the sequential recursion on one thread
    if (tid == 0) forward_sequential_tape<M>(v, tape);
  } else {
    // 2. inclusive scan of the chunk aggregates; 3. re-run the chunk from the exclusive prefix onto the tape
    FiltElem<M>* sh = reinterpret_cast<FiltElem<M>*>(kf_dyn_smem);
    sh[tid] = agg;
    cta_scan<FiltElem<M>, NT, false>(sh, filt_combine<M>);
    filt_rerun_chunk<M>(v, lo, hi, tid > 0 ? &sh[tid - 1] : nullptr, tape);
  }
  __syncthreads();  // tape entries of the other threads' chunks are visible from here on

  // 4. the literal update of every step on its predicted moments: outputs, ll_t, info; after a scan also the check that
  // each tape entry is one literal step from the one before it
  FwdOut o;
  o.ll_obs = A.ll_obs ? A.ll_obs + u * n : nullptr;
  o.fs = A.fs ? A.fs + u * (long long)n * M : nullptr;
  o.fc = A.fc ? A.fc + u * (long long)n * M * M : nullptr;
  o.ps = A.ps ? A.ps + u * (long long)(n + 1) * M : nullptr;
  o.pc = A.pc ? A.pc + u * (long long)(n + 1) * M * M : nullptr;
  double ll;
  int first_bad;
  const bool drift = forward_map_chunk<M>(v, lo, hi, tape, !sequential, o, &ll, &first_bad);
  if (!sequential && __syncthreads_or(drift)) {
    // the scan lost accuracy somewhere: the sequential recursion on one thread, then the map again
    if (tid == 0) forward_sequential_tape<M>(v, tape);
    __syncthreads();
    forward_map_chunk<M>(v, lo, hi, tape, false, o, &ll, &first_bad);
  }
  double* red = kf_dyn_smem;
  int* ired = reinterpret_cast<int*>(kf_dyn_smem + NT);
  red[tid] = ll;
  ired[tid] = first_bad;
  __syncthreads();
  for (int s = NT / 2; s > 0; s >>= 1) {
    if (tid < s) {
      red[tid] += red[tid + s];
      ired[tid] = min(ired[tid], ired[tid + s]);
    }
    __syncthreads();
  }
  if (tid == 0) {
    const int info = ired[0] == INT_MAX ? 0 : ired[0] + 1;
    if (A.loglik) A.loglik[u] = info != 0 ? nan("") : red[0];
    if (A.info) A.info[u] = info;
  }
}

template <int M, int NT>
__global__ void __launch_bounds__(NT) kf_tpar_backward_kernel(const __grid_constant__ KfArgs A) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  const long long u = blockIdx.x;
  const int tid = threadIdx.x, n = A.n;
  const UnitView v = unit_view(A, u);
  const auto [lo, hi] = chunk_of(tid, NT, n);
  const double* tape = A.tape + u * (long long)n * tape_entry<M>();
  const double gl = A.g_loglik ? A.g_loglik[u] : 1.0;
  const double* gllo = A.g_ll_obs ? A.g_ll_obs + u * n : nullptr;

  // 1. fold the chunk's abar elements and suffix-scan them
  AffElem<M>* sa = reinterpret_cast<AffElem<M>*>(kf_dyn_smem);
  AffElem<M> fa;
  aff_fold_chunk<M>(v, lo, hi, tape, gl, gllo, fa);
  sa[tid] = fa;
  cta_scan<AffElem<M>, NT, true>(sa, aff_combine<M>);
  double ab_hi[M];
  for (int i = 0; i < M; ++i) ab_hi[i] = (tid + 1 < NT) ? sa[tid + 1].s[i] : 0.0;  // abar_hi (abar_n = 0)
  __syncthreads();

  // 2. fold the chunk's congruence elements for sym(Pbar) and suffix-scan them
  CongElem<M>* sx = reinterpret_cast<CongElem<M>*>(kf_dyn_smem);
  CongElem<M> fx;
  cong_fold_chunk<M>(v, lo, hi, tape, gl, gllo, ab_hi, fx);
  sx[tid] = fx;
  cta_scan<CongElem<M>, NT, true>(sx, cong_combine<M>);
  double X[M * M];
  for (int i = 0; i < M * M; ++i) X[i] = (tid + 1 < NT) ? sx[tid + 1].S[i] : 0.0;  // sym(Pbar_hi)
  __syncthreads();

  // 3. every step's parameter cotangents (the literal one-step adjoint); the static ones summed in a fixed order
  auto rows = [&](double* p, long long ts, int w) { return p ? p + u * (ts ? n : 1) * w : nullptr; };
  const GradOut out{rows(A.ga0, 0, M),         rows(A.gP0, 0, M * M), rows(A.gT, A.T.ts, M * M),
                    rows(A.gC, A.C.ts, M * M), rows(A.gc, A.c.ts, M), rows(A.gZ, A.Z.ts, M),
                    rows(A.gH, A.H.ts, 1),     rows(A.gd, A.d.ts, 1)};
  constexpr int W = static_grad_width<M>();
  double acc[W];
  adjoint_chunk<M>(v, lo, hi, tape, gl, gllo, ab_hi, X, out, acc);
  double* red = kf_dyn_smem;
  for (int k = 0; k < W; ++k) red[tid * W + k] = acc[k];
  __syncthreads();
  cta_sum<NT>(red, W);
  for (int k = tid; k < W; k += NT) store_static_grad<M>(v, out, k, red[k]);
}

template <int M>
cudaError_t launch_tpar_m(const KfArgs& A, bool bwd, cudaStream_t s) {
  constexpr int NT = tpar_threads<M>();
  constexpr size_t red_fwd = NT * (sizeof(double) + sizeof(int));
  constexpr size_t red_bwd = (size_t)NT * static_grad_width<M>() * sizeof(double);
  const size_t smem = bwd ? std::max(std::max(NT * sizeof(AffElem<M>), NT * sizeof(CongElem<M>)), red_bwd)
                          : std::max(NT * sizeof(FiltElem<M>), red_fwd);
  void (*kern)(KfArgs) = bwd ? kf_tpar_backward_kernel<M, NT> : kf_tpar_forward_kernel<M, NT>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)A.U, NT, smem, s>>>(A);
  count_launch();
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_tpar(const KfArgs& A, bool bwd, cudaStream_t s) {
  cudaError_t e = cudaErrorInvalidConfiguration;
  tpar::with_instance(A.m, [&](auto M) { e = launch_tpar_m<M>(A, bwd, s); });
  return e;
}

}  // namespace kfb
