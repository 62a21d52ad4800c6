// kf_kernels.cuh - __global__ wrappers around forward_unit / backward_unit (kf_core.cuh), and CTA-wide helpers.
#pragma once
#include <cuda_runtime.h>

#include "kf_ctx.cuh"
#include "kf_dare.cuh"
#include "kf_run.cuh"
#include "kf_rows.cuh"
#include "kf_rowsD.cuh"
#include "kf_rowsU.cuh"
#include "kf_smooth.cuh"

namespace kfb {

constexpr int KFB_THREAD_BLOCK = 64;  // thread-per-unit CTA size: 65,536 units -> 1024 CTAs = 6.9 per SM on 148 SMs

// Stage `count` doubles of the (shared) observation stream into shared memory with one TMA bulk copy
// (cp.async.bulk -> SASS UBLKCP) completed on an mbarrier; every thread then reads y_t as a shared-memory
// broadcast.  Requires 16-byte aligned src; the odd tail double (if any) is copied by thread 0.
__device__ __forceinline__ void stage_y(double* ysm, const double* ysrc, int count, bool bulk_ok) {
  __shared__ __align__(8) unsigned long long bar;
  const int bulk_doubles = bulk_ok ? (count & ~1) : 0;
  if (bulk_doubles > 0) {
    const unsigned bar_s = (unsigned)__cvta_generic_to_shared(&bar);
    const unsigned dst_s = (unsigned)__cvta_generic_to_shared(ysm);
    const unsigned bytes = (unsigned)bulk_doubles * 8u;
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_s));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_s), "r"(bytes) : "memory");
      asm volatile(
          "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_s),
          "l"(ysrc), "r"(bytes), "r"(bar_s)
          : "memory");
    }
    unsigned done = 0;
    while (!done) {
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done)
          : "r"(bar_s)
          : "memory");
    }
  }
  for (int i = bulk_doubles + threadIdx.x; i < count; i += blockDim.x) ysm[i] = ysrc[i];
  __syncthreads();
}

// Inclusive scan of one element per thread across an NT-thread CTA (Hillis-Steele, fixed order, so reruns give identical
// bits): a prefix scan, sh[tid] <- sh[0] (x) .. (x) sh[tid], or with SUFFIX a suffix scan, sh[tid] <- sh[tid] (x) .. (x)
// sh[NT-1].  On entry sh[tid] holds this thread's element (the scan synchronises before reading it); on exit, its
// inclusive scan.  combine(lower, higher, out) gets the lower index first; out does not alias either operand.
template <class Elem, int NT, bool SUFFIX, class Combine>
__device__ __forceinline__ void cta_scan(Elem* sh, Combine combine) {
  const int tid = threadIdx.x;
  Elem agg, tmp;
  __syncthreads();
  agg = sh[tid];
  for (int off = 1; off < NT; off <<= 1) {
    const bool active = SUFFIX ? tid + off < NT : tid >= off;
    if (active) {
      if constexpr (SUFFIX) combine(agg, sh[tid + off], tmp);
      else combine(sh[tid - off], agg, tmp);
    }
    __syncthreads();
    if (active) { agg = tmp; sh[tid] = agg; }
    __syncthreads();
  }
}

// Fixed-order CTA tree sum of `w` doubles per thread (red[tid * w + k]); the result is left in red[0 .. w-1].
template <int NT>
__device__ __forceinline__ void cta_sum(double* red, int w) {
  for (int s = NT / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s)
      for (int k = 0; k < w; ++k) red[threadIdx.x * w + k] += red[(threadIdx.x + s) * w + k];
    __syncthreads();
  }
}

// 65,536 units (the headline batch) need 443 resident threads per SM for a single wave: the pipelined adjoint of the
// k_states <= 2 kernels is capped at 7 CTAs x 64 threads per SM (<= 144 registers) instead of spilling into a 2nd wave.
template <int M, int P, int MK, int MODE, bool TV = false>
__global__ void __launch_bounds__(KFB_THREAD_BLOCK)
    kf_thread_kernel(const __grid_constant__ KfArgs A, int y_smem_doubles, int bulk_ok) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  const double* ysm = nullptr;
  if (y_smem_doubles > 0) {
    stage_y(kf_dyn_smem, A.y.p, y_smem_doubles, bulk_ok != 0);
    ysm = kf_dyn_smem;
  }
  long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  // the adjoint kernel's tape ring / the full-output stager live behind the staged observations (16-byte aligned)
  double* ring = kf_dyn_smem + ((y_smem_doubles + 1) & ~1);
  ThreadCtx<M, P, TV> x{ysm, ring, (int)threadIdx.x, (int)blockDim.x};
  if (MODE == 1) {
    // outputs go through the per-warp stager; the padding lanes of the last warp run along (on the last unit's
    // parameters) because the flush at the end of every OUT_K-th step is warp-collective
    const long long u0 = u - (threadIdx.x & 31);
    if (u0 >= A.U) return;
    x.ostage = ring + (size_t)(threadIdx.x >> 5) * ThreadCtx<M, P, TV>::OUT_DOUBLES;
    x.warp_u0 = u0;
    if (u >= A.U) {
      KfArgs B = A;  // padding lane: compute, store nothing of its own
      B.loglik = nullptr; B.info = nullptr; B.tape = nullptr;
      run_unit_full<M, P, MK, TV>(x, B, A.U - 1);  // a padding lane of the last warp: same program on the last unit's inputs
      return;
    }
    run_unit_full<M, P, MK, TV>(x, A, u);
    return;
  }
  if (u >= A.U) return;
  run_unit<MK, MODE>(x, A, u);
}

// Run-time-dims kernels (CoopCtx): one warp (WARP, warp w on arena w of the CTA's shared memory) or the whole CTA per
// unit.  This thread's unit; in warp mode the caller returns when it is >= the unit count.
template <bool WARP>
__device__ __forceinline__ long long coop_unit() {
  return WARP ? (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5) : (long long)blockIdx.x;
}

template <int MK, int MODE, bool WARP>
__global__ void __launch_bounds__(WARP ? 128 : 256, WARP ? 4 : 2) kf_coop_kernel(const __grid_constant__ KfArgs A, int arena_doubles) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  CoopCtx x;
  x.init(A.m, A.p, WARP ? kf_dyn_smem + (size_t)(threadIdx.x >> 5) * arena_doubles : kf_dyn_smem, arena_doubles,
         WARP ? threadIdx.x & 31 : threadIdx.x, WARP ? 32 : blockDim.x);
  const long long u = coop_unit<WARP>();
  if (WARP && u >= A.U) return;
  x.red = nullptr;
  run_unit<MK, MODE>(x, A, u);
  if (x.overflow) __trap();
}

// Sub-warp cooperative kernel with compile-time dims: G lanes per unit, 128 threads per CTA.
template <int M, int P, int G, int MK, int MODE>
__global__ void __launch_bounds__(G > 128 ? G : 128, G > 128 ? 2 : 1)
    kf_coopT_kernel(const __grid_constant__ KfArgs A, int arena_doubles) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  constexpr int BLOCK = G > 128 ? G : 128;
  const int group = threadIdx.x / G;
  const long long u = (long long)blockIdx.x * (BLOCK / G) + group;
  if (u >= A.U) return;
  CoopCtxT<M, P, G> x;
  x.lane_ = threadIdx.x % G;
  x.mask_ = __activemask();
  x.arena = kf_dyn_smem + (size_t)group * arena_doubles;
  x.off = 0;
  x.red = nullptr;
  x.group_ = group;
  if (G > 32) {
    x.red = x.arena;
    x.off = 34;
  }
  run_unit<MK, MODE>(x, A, u);
  if (x.off > arena_doubles) __trap();  // arena accounting (coop_arena_doubles + slack) out of date
}

// Fused row-block-per-lane programs (kf_rows.cuh): G lanes per unit, 32/G units per warp, blockDim.x/32 warps per CTA.
// BWD = adjoint.  Lanes beyond the last whole group of a warp shadow the warp's first unit without owning rows.
template <int M, int P, int G, int MK, bool BWD, bool NEED_Z>
__global__ void __launch_bounds__(128, (RowsCfg<M, P, G>::R > 1) ? 1 : (BWD ? (NEED_Z ? 2 : 3) : 4)) kf_rows_kernel(const __grid_constant__ KfArgs A) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  constexpr int per_unit =
      BWD ? RowsLayout<M, P, NEED_Z, MK == MK_STEADY || MK == MK_CHOLS>::bwd_doubles : RowsLayout<M, P>::fwd_doubles;
  constexpr int UPW = RowsCfg<M, P, G>::UPW;
  const int lane32 = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int grp = lane32 / G, l = lane32 - grp * G;
  if (grp >= UPW) {
    grp = 0;
    l = G;
  }
  const int slot = warp * UPW + grp;
  const long long u = (long long)blockIdx.x * ((blockDim.x >> 5) * UPW) + slot;
  if (u >= A.U) return;
  const unsigned mask = __activemask();
  double* sm = kf_dyn_smem + (size_t)slot * per_unit;
  if (BWD) rows_backward<M, P, G, MK, NEED_Z>(A, u, sm, l, mask);
  else rows_forward<M, P, G, MK>(A, u, sm, l, mask);
}

// same mapping, all six outputs of the reference (rows_forward_full)
template <int M, int P, int G, int MK>
__global__ void __launch_bounds__(128, 1) kf_rowsfull_kernel(const __grid_constant__ KfArgs A) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  constexpr int per_unit = RowsLayout<M, P>::fwd_doubles;
  constexpr int UPW = RowsCfg<M, P, G>::UPW;
  const int lane32 = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int grp = lane32 / G, l = lane32 - grp * G;
  if (grp >= UPW) {
    grp = 0;
    l = G;
  }
  const int slot = warp * UPW + grp;
  const long long u = (long long)blockIdx.x * ((blockDim.x >> 5) * UPW) + slot;
  if (u >= A.U) return;
  const unsigned mask = __activemask();
  rows_forward_full<M, P, G, MK>(A, u, kf_dyn_smem + (size_t)slot * per_unit, l, mask);
}

// Fused UnivariateFilter programs (kf_rowsU.cuh): 8 lanes per unit, 4 units per warp.  BWD = adjoint (no Z-bar).
template <int M, int P, bool BWD>
__global__ void __launch_bounds__(128, BWD ? 2 : 3) kf_rowsU_kernel(const __grid_constant__ KfArgs A) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  constexpr int per_unit = BWD ? RowsULayout<M, P>::bwd_doubles : RowsULayout<M, P>::fwd_doubles;
  const int lane32 = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = warp * 4 + (lane32 >> 3);
  const long long u = (long long)blockIdx.x * ((blockDim.x >> 5) * 4) + slot;
  if (u >= A.U) return;
  const unsigned mask = __activemask();
  double* sm = kf_dyn_smem + (size_t)slot * per_unit;
  if (BWD) rowsU_backward<M, P>(A, u, sm, lane32 & 7, mask);
  else rowsU_forward<M, P>(A, u, sm, lane32 & 7, mask);
}

// Fused row-per-lane, warp-per-unit programs for large systems with the m^3 products on the FP64 tensor cores
// (kf_rowsD.cuh); MK = MK_STD or MK_STEADY.  BWD = adjoint, NEED_T = with T-bar.
// Resident CTAs per SM with 16 x 16 tiles (k_states 10..16): 12 warps per SM, <= 168 registers.  Seasonal period 12,
// 65,536 x 1000, swizzled tiles: 2 -> 241 ms, 3 -> 231 ms, 4 -> 250 ms (128 registers: the adjoint spills 150-390 bytes
// per thread).
constexpr int ROWSH_MIN_BLOCKS = 3;
template <int M, int P, int MK, bool BWD, bool NEED_T>
__global__ void __launch_bounds__(128, M <= 16 ? ROWSH_MIN_BLOCKS : 1) kf_rowsD_kernel(const __grid_constant__ KfArgs A) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  constexpr int per_unit = BWD ? RowsDLayout<M, P, NEED_T>::bwd_doubles : RowsDLayout<M, P, false>::fwd_doubles;
  const int warp = threadIdx.x >> 5;
  const long long u = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
  if (u >= A.U) return;
  double* sm = kf_dyn_smem + (size_t)warp * per_unit;
  if (BWD) rowsD_backward<M, P, MK, NEED_T>(A, u, sm, threadIdx.x & 31);
  else rowsD_forward<M, P, MK>(A, u, sm, threadIdx.x & 31);
}

// same mapping, all six outputs of the reference (rowsD_forward_full)
template <int M, int P, int MK>
__global__ void __launch_bounds__(128, M <= 16 ? ROWSH_MIN_BLOCKS : 1) kf_rowsDfull_kernel(const __grid_constant__ KfArgs A) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  constexpr int per_unit = RowsDLayout<M, P, false>::fwd_doubles;
  const int warp = threadIdx.x >> 5;
  const long long u = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
  if (u >= A.U) return;
  rowsD_forward_full<M, P, MK>(A, u, kf_dyn_smem + (size_t)warp * per_unit, threadIdx.x & 31);
}

// ---- steady-state (DARE) kernels: one warp or one CTA per draw / unit (kf_dare.cuh) ----
struct DareArgs {
  long long nD, U, n_series;
  int m, p;
  MatArg T, Z, H, C;
  double *Pss, *Gss;  // [nD, m, m], [nD, p, p]
  int* info;          // [nD] or null
  const double *gPss, *gGss;  // [U, ...]
  double *gT, *gZ, *gH, *gC;  // [U, ...] accumulated
};

template <bool BWD, bool WARP>
__global__ void kf_dare_kernel(const __grid_constant__ DareArgs D, int arena_doubles) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  CoopCtx x;
  x.init(D.m, D.p, WARP ? kf_dyn_smem + (size_t)(threadIdx.x >> 5) * arena_doubles : kf_dyn_smem, arena_doubles,
         WARP ? threadIdx.x & 31 : threadIdx.x, WARP ? 32 : blockDim.x);
  const long long u = coop_unit<WARP>();
  if (WARP && u >= (BWD ? D.U : D.nD)) return;
  x.red = x.bump(34);
  if (BWD) {
    const long long d = u / D.n_series;
    dare_adjoint_unit(x, D.T.p + d * D.T.bs, D.Z.p + d * D.Z.bs, D.H.p + d * D.H.bs, D.Pss + d * D.m * D.m,
                      D.Gss + d * D.p * D.p, D.gPss + u * D.m * D.m, D.gGss + u * D.p * D.p,
                      D.gT ? D.gT + u * D.m * D.m : nullptr, D.gZ ? D.gZ + u * D.p * D.m : nullptr,
                      D.gH ? D.gH + u * D.p * D.p : nullptr, D.gC ? D.gC + u * D.m * D.m : nullptr);
  } else {
    const int info = dare_unit(x, D.T.p + u * D.T.bs, D.Z.p + u * D.Z.bs, D.H.p + u * D.H.bs, D.C.p + u * D.C.bs,
                               D.Pss + u * D.m * D.m, D.Gss + u * D.p * D.p);
    if (D.info && x.lane_ == 0) D.info[u] = info;
  }
  if (x.overflow) __trap();
}
cudaError_t launch_dare(const DareArgs& D, bool bwd, cudaStream_t s);

// steady-state covariance on the warp-per-draw tensor-core mapping (kf_rowsD.cuh: rowsD_dare), even k_states 18..32
template <int M, int P>
__global__ void __launch_bounds__(128, M <= 16 ? 4 : 1) kf_dareD_kernel(const __grid_constant__ DareArgs D) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  constexpr int per_unit = DareDLayout<M, P>::doubles;
  const int warp = threadIdx.x >> 5;
  const long long u = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
  if (u >= D.nD) return;
  rowsD_dare<M, P>(D.T.p + u * D.T.bs, D.Z.p + u * D.Z.bs, D.H.p + u * D.H.bs, D.C.p + u * D.C.bs, D.Pss + u * M * M,
                   D.Gss + u * P * P, D.info ? D.info + u : nullptr, kf_dyn_smem + (size_t)warp * per_unit,
                   threadIdx.x & 31);
}
typedef cudaError_t (*dare_launch_fn)(const DareArgs& D, cudaStream_t s);
dare_launch_fn find_dareD_launcher(int m, int p);

template <bool WARP>
__global__ void __launch_bounds__(WARP ? 128 : 256) kf_smoother_kernel(const __grid_constant__ SmoothArgs S, int arena_doubles) {
  extern __shared__ __align__(16) double kf_dyn_smem[];
  CoopCtx x;
  x.init(S.m, 1, WARP ? kf_dyn_smem + (size_t)(threadIdx.x >> 5) * arena_doubles : kf_dyn_smem, arena_doubles,
         WARP ? threadIdx.x & 31 : threadIdx.x, WARP ? 32 : blockDim.x);
  const long long u = coop_unit<WARP>();
  if (WARP && u >= S.U) return;
  x.red = x.bump(34);
  smoother_unit(x, S, u);
  if (x.overflow) __trap();
}
cudaError_t launch_smoother(const SmoothArgs& S, cudaStream_t s);

// k_states <= 4: one unit per thread, everything in registers, no synchronisation (the same smoother_unit program)
template <int M>
__global__ void __launch_bounds__(128) kf_smoother_thread_kernel(const __grid_constant__ SmoothArgs S) {
  const long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= S.U) return;
  ThreadCtx<M, 1> x{nullptr, nullptr, (int)threadIdx.x, (int)blockDim.x};
  smoother_unit(x, S, u);
}
typedef cudaError_t (*smoother_launch_fn)(const SmoothArgs& S, cudaStream_t s);
smoother_launch_fn find_smoother_thread_launcher(int m);

// launchers implemented in kf_thread.cu / kf_coopT.cu / kf_coop.cu
typedef cudaError_t (*thread_launch_fn)(const KfArgs& A, bool bwd, int y_smem_doubles, int bulk_ok, cudaStream_t s);
thread_launch_fn find_thread_launcher(int m, int p, int mk, bool tv = false);
cudaError_t launch_coop(const KfArgs& A, bool bwd, cudaStream_t s);
typedef cudaError_t (*coopT_launch_fn)(const KfArgs& A, bool bwd, cudaStream_t s);
coopT_launch_fn find_coopT_launcher(int m, int p, int mk);
void count_launch();

}  // namespace kfb
