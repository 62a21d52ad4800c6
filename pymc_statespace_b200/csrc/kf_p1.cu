// kf_p1.cu - kernels of the k_endog = 1 adjoint (kf_p1.cuh): one unit per thread, the tape streamed backwards by
// ONE TMA bulk copy per warp and step into a per-warp shared-memory ring.
//
// Tape layout (written by the thread-per-unit forward kernels, ThreadCtx::tape_*): [t-1][warp][k][32] - the entry of
// step t for the 32 units of a warp is KT * 256 contiguous bytes (1280 B at k_states = 2), so the reverse sweep needs
// no per-thread address arithmetic or load instructions for the tape at all: lane 0 arms an mbarrier with the byte
// count and issues `cp.async.bulk.shared::cluster.global` (SASS UBLKCP), every lane then waits on the barrier's phase
// and reads its KT doubles with conflict-free LDS.64 (lane-consecutive addresses).  SLOTS - 1 entries are in flight;
// the slot refilled in a step is the one consumed in the PREVIOUS step (its values were used by arithmetic since).
#include "kf_kernels.cuh"
#include "kf_p1.cuh"

namespace kfb {
namespace p1 {

template <int M, int SLOTS, int KTE = Dim<M>::KT>
struct RingTape {
  static constexpr int KT = KTE;  // doubles per entry (Dim<M>::KTA for the reduced recursion)
  static constexpr unsigned BYTES = KT * 32 * 8;
  static_assert((SLOTS & (SLOTS - 1)) == 0, "SLOTS must be a power of two");
  // warp-uniform state (derived from blockIdx and a shuffled warp index so that the compiler keeps it in uniform
  // registers: UBLKCP takes uniform operands, and values it cannot prove uniform cost an ELECT / R2UR / BRA.U.ANY loop)
  unsigned ring_s, bar_s;  // shared-window addresses of this warp's ring and its SLOTS mbarriers
  const double* gnext;     // global address of the next entry to request (this warp's block of the tape)
  long long gstep;         // doubles between the entries of consecutive steps
  int left;                // entries not requested yet
  unsigned c;              // entries consumed
  // per lane
  unsigned lane_s;         // shared-window address of ring[0][0][lane]
  unsigned leader;         // 1 on lane 0

  __device__ __forceinline__ void request(unsigned slot) {
    const unsigned go = (left > 0) ? leader : 0u;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.u32 p, %0, 0;\n\t"
        "@p mbarrier.arrive.expect_tx.shared::cta.b64 _, [%1], %2;\n\t"
        "@p cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%3], [%4], %2, [%1];\n\t}" ::"r"(go),
        "r"(bar_s + slot * 8u), "r"(BYTES), "r"(ring_s + slot * BYTES), "l"(gnext)
        : "memory");
    gnext -= gstep;
    --left;
  }

  __device__ __forceinline__ void init(unsigned ring_shared, unsigned bars_shared, const double* g_last, long long step,
                                       int entries, int lane) {
    ring_s = ring_shared;
    bar_s = bars_shared;
    lane_s = ring_shared + (unsigned)lane * 8u;
    leader = (lane == 0) ? 1u : 0u;
    gnext = g_last;
    gstep = step;
    left = entries;
    c = 0;
    if (lane == 0) {
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_s + s * 8u));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < SLOTS - 1; ++s) request((unsigned)s);
  }

  // non-blocking test of the next entry's barrier phase
  __device__ __forceinline__ unsigned poll() const {
    const unsigned slot = c & (SLOTS - 1), parity = (c / SLOTS) & 1u;
    unsigned ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar_s + slot * 8u), "r"(parity)
        : "memory");
    return ok;
  }

  __device__ __forceinline__ void finish(unsigned ok, double (&e)[KT]) {
    const unsigned slot = c & (SLOTS - 1);
    while (!ok) ok = poll();
    __syncwarp();
    const unsigned src = lane_s + slot * BYTES;
#pragma unroll
    for (int k = 0; k < KT; ++k) asm volatile("ld.shared.f64 %0, [%1];" : "=d"(e[k]) : "r"(src + k * 256u) : "memory");
    request((c + SLOTS - 1) & (SLOTS - 1));  // refill the slot consumed one step ago
    ++c;
  }

  __device__ __forceinline__ void next(double (&e)[KT]) { finish(poll(), e); }
};

// compile-time tuning knobs (A/B builds: tools/build_variants.sh)
#ifndef KFB_P1_WPC
#define KFB_P1_WPC 2
#endif
#ifndef KFB_P1_SLOTS
#define KFB_P1_SLOTS 4
#endif
#ifndef KFB_P1_MINB
#define KFB_P1_MINB 7
#endif
constexpr int P1_WPC = KFB_P1_WPC;      // warps per CTA (the observation stream is staged once per CTA)
constexpr int P1_SLOTS = KFB_P1_SLOTS;  // ring slots per warp (SLOTS - 1 entries in flight)

template <int M, bool NEED_Z, bool NEED_H, bool HAS_GOBS, int ZU, bool H0>
__global__ void __launch_bounds__(32 * P1_WPC, (M <= 2) ? KFB_P1_MINB : 4)
    kf_p1_adjoint_kernel(const __grid_constant__ KfArgs A, int y_smem_doubles, int bulk_ok) {
  extern __shared__ __align__(128) double kf_dyn_smem[];
  constexpr int KT = tape_doubles<M, ZU>;
  const double* yp = A.y.p;
  if (y_smem_doubles > 0) {
    stage_y(kf_dyn_smem, A.y.p, y_smem_doubles, bulk_ok != 0);
    yp = kf_dyn_smem;
  }
  const int lane = threadIdx.x & 31;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform by construction
  const unsigned ring0_s = (unsigned)__cvta_generic_to_shared(kf_dyn_smem + ((y_smem_doubles + 15) & ~15));
  const unsigned bars_s = ring0_s + (unsigned)(P1_WPC * P1_SLOTS * KT * 32 * 8);
  const long long wg = (long long)blockIdx.x * P1_WPC + warp;     // global warp index = block of 32 units
  const long long u = wg * 32 + lane;
  if (wg * 32 >= A.U) return;                                    // whole warp beyond the batch
  const long long upad = (A.U + 31) & ~31LL;
  const long long tstep = (long long)KT * upad;
  RingTape<M, P1_SLOTS, KT> tape;
  tape.init(ring0_s + (unsigned)(warp * P1_SLOTS * KT * 32 * 8), bars_s + (unsigned)(warp * P1_SLOTS * 8),
            A.tape + wg * (KT * 32) + (long long)(A.n - 2) * tstep, tstep, A.n - 1, lane);
  const bool store = u < A.U;
  backward_unit_p1<M, NEED_Z, NEED_H, HAS_GOBS, RingTape<M, P1_SLOTS, KT>, ZU, H0>(A, store ? u : A.U - 1, store, yp, tape);
}

template <int M, bool NEED_Z, bool NEED_H, bool HAS_GOBS, int ZU, bool H0>
static cudaError_t launch_one(const KfArgs& A, int ysm, int bulk_ok, cudaStream_t s) {
  constexpr int KT = tape_doubles<M, ZU>;
  const int block = 32 * P1_WPC;
  const unsigned grid = (unsigned)((A.U + block - 1) / block);
  const size_t smem = (size_t)((ysm + 15) & ~15) * 8 + (size_t)P1_WPC * P1_SLOTS * (KT * 32 * 8 + 8);
  auto kern = kf_p1_adjoint_kernel<M, NEED_Z, NEED_H, HAS_GOBS, ZU, H0>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<grid, block, smem, s>>>(A, ysm, bulk_ok);
  count_launch();
  return cudaGetLastError();
}

template <int M>
static cudaError_t launch_m(const KfArgs& A, int ysm, int bulk_ok, cudaStream_t s) {
  return with_adjoint_variant(A, [&](auto v) {
    using V = decltype(v);
    return launch_one<M, V::NEED_Z, V::NEED_H, V::HAS_GOBS, V::ZU, V::H0>(A, ysm, bulk_ok, s);
  });
}

// ---- forward (loglik + tape) -------------------------------------------------------------------------------
template <int M, bool SAVE, int ZU, bool H0>
__global__ void __launch_bounds__(64, (M <= 2) ? 8 : 4)
    kf_p1_forward_kernel(const __grid_constant__ KfArgs A, int y_smem_doubles, int bulk_ok) {
  extern __shared__ __align__(128) double kf_dyn_smem[];
  constexpr int KT = tape_doubles<M, ZU>;
  const double* yp = A.y.p;
  if (y_smem_doubles > 0) {
    stage_y(kf_dyn_smem, A.y.p, y_smem_doubles, bulk_ok != 0);
    yp = kf_dyn_smem;
  }
  const long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long tstep = (long long)KT * tape_units_padded(A.U);
  if (u >= A.U) return;
  double* tp = SAVE ? A.tape + (u >> 5) * (KT * 32) + (u & 31) : nullptr;
  forward_unit_p1<M, SAVE, ZU, H0>(A, u, true, yp, tp, tstep);
}

template <int M, bool SAVE, int ZU, bool H0>
static cudaError_t launch_fwd_one(const KfArgs& A, int ysm, int bulk_ok, cudaStream_t s) {
  const int block = 64;
  const unsigned grid = (unsigned)((A.U + block - 1) / block);
  const size_t smem = (size_t)((ysm + 1) & ~1) * 8;
  auto kern = kf_p1_forward_kernel<M, SAVE, ZU, H0>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  kern<<<grid, block, smem, s>>>(A, ysm, bulk_ok);
  count_launch();
  return cudaGetLastError();
}

template <int M>
static cudaError_t launch_fwd_m(const KfArgs& A, int ysm, int bulk_ok, cudaStream_t s) {
  return with_forward_variant(A, [&](auto v) {
    using V = decltype(v);
    return A.tape ? launch_fwd_one<M, true, V::ZU, V::H0>(A, ysm, bulk_ok, s)
                  : launch_fwd_one<M, false, V::ZU, V::H0>(A, ysm, bulk_ok, s);
  });
}

}  // namespace p1

// Forward pass, loglik (+ tape) only, same conditions as the adjoint below.
cudaError_t launch_p1_forward(const KfArgs& A, int y_smem_doubles, int bulk_ok, cudaStream_t s) {
  switch (A.m) {
    case 1: return p1::launch_fwd_m<1>(A, y_smem_doubles, bulk_ok, s);
    case 2: return p1::launch_fwd_m<2>(A, y_smem_doubles, bulk_ok, s);
    case 3: return p1::launch_fwd_m<3>(A, y_smem_doubles, bulk_ok, s);
    case 4: return p1::launch_fwd_m<4>(A, y_smem_doubles, bulk_ok, s);
    default: return cudaErrorInvalidConfiguration;
  }
}

bool p1_adjoint_supported(int m, int p, int mk) { return p == 1 && mk == MK_STD && m >= 1 && m <= 4; }

// Adjoint of the standard-family filters for k_endog = 1, static matrices, one shared observation stream.
cudaError_t launch_p1_adjoint(const KfArgs& A, int y_smem_doubles, int bulk_ok, cudaStream_t s) {
  switch (A.m) {
    case 1: return p1::launch_m<1>(A, y_smem_doubles, bulk_ok, s);
    case 2: return p1::launch_m<2>(A, y_smem_doubles, bulk_ok, s);
    case 3: return p1::launch_m<3>(A, y_smem_doubles, bulk_ok, s);
    case 4: return p1::launch_m<4>(A, y_smem_doubles, bulk_ok, s);
    default: return cudaErrorInvalidConfiguration;
  }
}

}  // namespace kfb
