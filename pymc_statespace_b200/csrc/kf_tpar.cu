// kf_tpar.cu - time-parallel forward / adjoint kernels (KFB_FLAG_TIME_PARALLEL): one CTA per unit, blocked scans over
// time.  The math is in kf_tpar.cuh.
#include <climits>

#include "kf_kernels.cuh"
#include "kf_tpar.cuh"

namespace kfb {

namespace {

using namespace tpar;

// 256 threads while one thread's operands fit the register file; the filtering element of k_states 3 / 4 is 33 / 56
// doubles, so those kernels run 128 threads (a few more steps per thread, one scan level less).
template <int M>
KFB_HD constexpr int tpar_threads() { return M <= 2 ? 256 : 128; }

// Fixed-order CTA tree sum of `w` doubles per thread (red[tid * w + k]); the result is left in red[0 .. w-1].
template <int NT>
__device__ __forceinline__ void cta_sum(double* red, int w) {
  for (int s = NT / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s)
      for (int k = 0; k < w; ++k) red[threadIdx.x * w + k] += red[(threadIdx.x + s) * w + k];
    __syncthreads();
  }
}

template <int M, int NT>
__global__ void __launch_bounds__(NT) kf_tpar_forward_kernel(const __grid_constant__ KfArgs A) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  constexpr int E = tape_entry<M>();
  const long long u = blockIdx.x;
  const int tid = threadIdx.x, n = A.n;
  const UnitView v = unit_view(A, u);
  const int chunk = (n + NT - 1) / NT;
  const int lo = min(n, tid * chunk), hi = min(n, lo + chunk);
  double* tape = A.tape + u * (long long)n * E;

  // 1. fold this thread's chunk of filtering elements
  FiltElem<M> agg, e, tmp;
  filt_identity<M>(agg);
  bool undefined = false;
  for (int t = lo; t < hi; ++t) {
    if (t == 0) filt_element0<M>(v, e);
    else undefined |= !filt_element<M>(v, t, e);
    if (t == lo) agg = e;
    else { filt_combine<M>(agg, e, tmp); agg = tmp; }
  }
  const bool sequential = __syncthreads_or(undefined);
  if (sequential) {
    // an element has no parallel form: this unit runs the sequential recursion on one thread
    if (tid == 0) forward_sequential_tape<M>(v, tape);
  } else {
    // 2. inclusive scan of the chunk aggregates (Hillis-Steele, fixed order)
    FiltElem<M>* sh = reinterpret_cast<FiltElem<M>*>(kf_dyn_smem);
    sh[tid] = agg;
    __syncthreads();
    for (int off = 1; off < NT; off <<= 1) {
      if (tid >= off) filt_combine<M>(sh[tid - off], agg, tmp);
      __syncthreads();
      if (tid >= off) { agg = tmp; sh[tid] = agg; }
      __syncthreads();
    }
    // 3. re-run the chunk from the exclusive prefix: filtered moments -> predicted moments on the tape
    FiltElem<M> f;
    for (int t = lo; t < hi; ++t) {
      if (t == 0) {
        filt_element0<M>(v, f);
        for (int i = 0; i < M; ++i) tape[i] = v.a0[i];
        for (int i = 0; i < M * M; ++i) tape[M + i] = v.P0[i];
      } else {
        filt_element<M>(v, t, e);
        filt_combine<M>(t == lo ? sh[tid - 1] : f, e, tmp);
        f = tmp;
      }
      if (t + 1 < n) predict_to_tape<M>(v, t, f.b, f.C, tape + (long long)(t + 1) * E);
    }
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
  auto map = [&](bool check) {
    ll = 0.0;
    first_bad = INT_MAX;
    bool drift_any = false;
    for (int t = lo; t < hi; ++t) {
      bool bad, drift;
      const double* next = (check && t + 1 < n) ? tape + (long long)(t + 1) * E : nullptr;
      ll += forward_map_step<M>(v, t, tape + (long long)t * E, next, o, &bad, &drift);
      if (bad && first_bad == INT_MAX) first_bad = t;
      drift_any |= drift;
    }
    return drift_any;
  };
  const bool drift = map(!sequential);
  if (!sequential && __syncthreads_or(drift)) {
    // the scan lost accuracy somewhere: the sequential recursion on one thread, then the map again
    if (tid == 0) forward_sequential_tape<M>(v, tape);
    __syncthreads();
    map(false);
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
  constexpr int E = tape_entry<M>();
  const long long u = blockIdx.x;
  const int tid = threadIdx.x, n = A.n;
  const UnitView v = unit_view(A, u);
  const int chunk = (n + NT - 1) / NT;
  const int lo = min(n, tid * chunk), hi = min(n, lo + chunk);
  const double* tape = A.tape + u * (long long)n * E;
  const double gl = A.g_loglik ? A.g_loglik[u] : 1.0;
  const double* gllo = A.g_ll_obs ? A.g_ll_obs + u * n : nullptr;
  TX<M> x{nullptr, nullptr, 0, 1};
  BwdStep<M> B(x);

  // 1. fold the chunk's abar elements (f_lo o .. o f_{hi-1}) and suffix-scan them
  AffElem<M> fa, ea, ta;
  aff_identity<M>(fa);
  for (int t = hi - 1; t >= lo; --t) {
    bwd_load<M>(x, v, t, tape + (long long)t * E, gl, gllo, B);
    aff_element<M>(B, ea);
    if (t == hi - 1) fa = ea;
    else { aff_combine<M>(ea, fa, ta); fa = ta; }
  }
  AffElem<M>* sa = reinterpret_cast<AffElem<M>*>(kf_dyn_smem);
  sa[tid] = fa;
  __syncthreads();
  for (int off = 1; off < NT; off <<= 1) {
    if (tid + off < NT) aff_combine<M>(fa, sa[tid + off], ta);
    __syncthreads();
    if (tid + off < NT) { fa = ta; sa[tid] = fa; }
    __syncthreads();
  }
  double ab_hi[M], ab[M], abn[M];
  for (int i = 0; i < M; ++i) ab_hi[i] = (tid + 1 < NT) ? sa[tid + 1].s[i] : 0.0;  // abar_hi (abar_n = 0)
  __syncthreads();

  // 2. fold the chunk's congruence elements for sym(Pbar) (their forcing needs abar_{t+1}) and suffix-scan them
  CongElem<M> fx, ex, tx;
  cong_identity<M>(fx);
  for (int i = 0; i < M; ++i) ab[i] = ab_hi[i];
  for (int t = hi - 1; t >= lo; --t) {
    bwd_load<M>(x, v, t, tape + (long long)t * E, gl, gllo, B);
    cong_element<M>(B, ab, ex);
    aff_apply<M>(B, ab, abn);
    for (int i = 0; i < M; ++i) ab[i] = abn[i];
    if (t == hi - 1) fx = ex;
    else { cong_combine<M>(ex, fx, tx); fx = tx; }
  }
  CongElem<M>* sx = reinterpret_cast<CongElem<M>*>(kf_dyn_smem);
  sx[tid] = fx;
  __syncthreads();
  for (int off = 1; off < NT; off <<= 1) {
    if (tid + off < NT) cong_combine<M>(fx, sx[tid + off], tx);
    __syncthreads();
    if (tid + off < NT) { fx = tx; sx[tid] = fx; }
    __syncthreads();
  }
  double X[M * M];
  for (int i = 0; i < M * M; ++i) X[i] = (tid + 1 < NT) ? sx[tid + 1].S[i] : 0.0;  // sym(Pbar_hi)
  __syncthreads();

  // 3. every step's parameter cotangents (the literal one-step adjoint), per-step for time-varying inputs
  constexpr int W = 2 * M * M + 2 * M + 2;  // T, C, c, Z, H, d
  double acc[W];
  for (int k = 0; k < W; ++k) acc[k] = 0.0;
  for (int i = 0; i < M; ++i) ab[i] = ab_hi[i];
  StepGrad<M> g;
  const double ds = A.d_sign;
  for (int t = hi - 1; t >= lo; --t) {
    bwd_load<M>(x, v, t, tape + (long long)t * E, gl, gllo, B);
    if (t == 0) {
      double a0b[M], P0b[M * M];
      adjoint_step<M>(B, ds, ab, X, g, a0b, P0b);
      if (A.ga0) for (int i = 0; i < M; ++i) A.ga0[u * M + i] = a0b[i];
      if (A.gP0) for (int i = 0; i < M * M; ++i) A.gP0[u * M * M + i] = P0b[i];
    } else {
      adjoint_step<M>(B, ds, ab, X, g, nullptr, nullptr);
      cong_element<M>(B, ab, ex);
      cong_apply<M>(ex, X);
      aff_apply<M>(B, ab, abn);
      for (int i = 0; i < M; ++i) ab[i] = abn[i];
    }
    const long long ut = u * n + t;
    if (A.T.ts) { if (A.gT) for (int i = 0; i < M * M; ++i) A.gT[ut * M * M + i] = g.T[i]; }
    else for (int i = 0; i < M * M; ++i) acc[i] += g.T[i];
    if (A.C.ts) { if (A.gC) for (int i = 0; i < M * M; ++i) A.gC[ut * M * M + i] = g.C[i]; }
    else for (int i = 0; i < M * M; ++i) acc[M * M + i] += g.C[i];
    if (A.c.ts) { if (A.gc) for (int i = 0; i < M; ++i) A.gc[ut * M + i] = g.c[i]; }
    else for (int i = 0; i < M; ++i) acc[2 * M * M + i] += g.c[i];
    if (A.Z.ts) { if (A.gZ) for (int i = 0; i < M; ++i) A.gZ[ut * M + i] = g.Z[i]; }
    else for (int i = 0; i < M; ++i) acc[2 * M * M + M + i] += g.Z[i];
    if (A.H.ts) { if (A.gH) A.gH[ut] = g.H; }
    else acc[2 * M * M + 2 * M] += g.H;
    if (A.d.ts) { if (A.gd) A.gd[ut] = g.d; }
    else acc[2 * M * M + 2 * M + 1] += g.d;
  }
  double* red = kf_dyn_smem;
  for (int k = 0; k < W; ++k) red[tid * W + k] = acc[k];
  __syncthreads();
  cta_sum<NT>(red, W);
  for (int k = tid; k < W; k += NT) {
    const double s = red[k];
    if (k < M * M) { if (A.gT && !A.T.ts) A.gT[u * M * M + k] = s; }
    else if (k < 2 * M * M) { if (A.gC && !A.C.ts) A.gC[u * M * M + k - M * M] = s; }
    else if (k < 2 * M * M + M) { if (A.gc && !A.c.ts) A.gc[u * M + k - 2 * M * M] = s; }
    else if (k < 2 * M * M + 2 * M) { if (A.gZ && !A.Z.ts) A.gZ[u * M + k - 2 * M * M - M] = s; }
    else if (k == 2 * M * M + 2 * M) { if (A.gH && !A.H.ts) A.gH[u] = s; }
    else { if (A.gd && !A.d.ts) A.gd[u] = s; }
  }
}

template <int M>
cudaError_t launch_tpar_m(const KfArgs& A, bool bwd, cudaStream_t s) {
  constexpr int NT = tpar_threads<M>();
  constexpr size_t red_fwd = NT * (sizeof(double) + sizeof(int));
  constexpr size_t red_bwd = (size_t)NT * (2 * M * M + 2 * M + 2) * sizeof(double);
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

bool tpar_supported(int m, int p, int mk) { return p == 1 && mk == MK_STD && m >= 1 && m <= 4; }

cudaError_t launch_tpar(const KfArgs& A, bool bwd, cudaStream_t s) {
  switch (A.m) {
    case 1: return launch_tpar_m<1>(A, bwd, s);
    case 2: return launch_tpar_m<2>(A, bwd, s);
    case 3: return launch_tpar_m<3>(A, bwd, s);
    case 4: return launch_tpar_m<4>(A, bwd, s);
    default: return cudaErrorInvalidConfiguration;
  }
}

}  // namespace kfb
