// kf_p1.cu - kernels of the k_endog = 1 adjoint (kf_p1.cuh): one unit per thread, the tape streamed backwards by
// TMA bulk copies per warp into a per-warp shared-memory ring.
//
// Full tape (written by the thread-per-unit forward kernels, ThreadCtx::tape_*): [t-1][warp][k][32] - the entry of step t
// for the 32 units of a warp is KT * 256 contiguous bytes, fetched by ONE bulk copy per step.  Compressed tape of the
// reduced ARMA recursion (ZU_REDUCED; CTape in kf_core.cuh): [t / S][warp][t % S][row] - S steps of a warp are one
// contiguous block of S * KT * 256 bytes (2 KB at k_states 2, S = 4), fetched by ONE bulk copy per S steps; the barrier
// test, the copy and its address and parity arithmetic run once per block, and a lane reads its entry with LDS.128.
// Either way no per-thread address arithmetic or global load is spent on the tape: lane 0 arms an mbarrier with the
// byte count and issues `cp.async.bulk.shared::cluster.global` (SASS UBLKCP), every lane then waits on the barrier's
// phase and reads its doubles with conflict-free shared loads (lane-consecutive addresses).  SLOTS - 1 chunks (steps or
// blocks) are in flight; the slot refilled is the one consumed one chunk ago (its values were used by arithmetic since).
#include "kf_kernels.cuh"
#include "kf_p1.cuh"

namespace kfb {
namespace p1 {

// S = 1: one chunk is one step of the full tape;  S > 1: one block of the compressed tape (CTape<KT>)
template <int KTE, int SLOTS, int S = 1>
struct RingTape {
  static constexpr int KT = KTE;  // doubles per entry (Dim<M>::KTA for the reduced recursion)
  static constexpr unsigned BYTES = S * KT * 32 * 8;
  static_assert((SLOTS & (SLOTS - 1)) == 0, "SLOTS must be a power of two");
  // warp-uniform state (derived from blockIdx and a shuffled warp index so that the compiler keeps it in uniform
  // registers: UBLKCP takes uniform operands, and values it cannot prove uniform cost an ELECT / R2UR / BRA.U.ANY loop)
  unsigned ring_s, bar_s;  // shared-window addresses of this warp's ring and its SLOTS mbarriers
  const double* gnext;     // global address of the next chunk to request (this warp's part of the tape)
  long long gstep;         // doubles between consecutive chunks
  int left;                // chunks not requested yet
  unsigned c;              // chunks consumed
  // per lane
  unsigned lane_s;         // shared-window address of ring[0][0][lane]
  unsigned leader;         // 1 on lane 0
  int lane;
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
                                       int chunks, int lane) {
    ring_s = ring_shared;
    bar_s = bars_shared;
    lane_s = ring_shared + (unsigned)lane * 8u;
    this->lane = lane;
    leader = (lane == 0) ? 1u : 0u;
    gnext = g_last;
    gstep = step;
    left = chunks;
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

  // S > 1: the next block of the compressed tape, e[j] = entry of step (block) * S + j.  The blocks come in the order
  // the reverse sweep asks for them (last first), so the unit and the block index it passes are not needed here.
  __device__ __forceinline__ void block(const KfArgs&, long long, int, double (&e)[S][KT]) {
    const unsigned slot = c & (SLOTS - 1);
    while (!poll()) {
    }
    __syncwarp();
    const unsigned src = ring_s + slot * BYTES;
#pragma unroll
    for (int j = 0; j < S; ++j) {
#pragma unroll
      for (int k = 0; k + 1 < KT; k += 2)
        asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];"
                     : "=d"(e[j][k]), "=d"(e[j][k + 1 < KT ? k + 1 : 0])
                     : "r"(src + (unsigned)(j * CTape<KT>::ROW + CTape<KT>::lane_offset(lane, k)) * 8u)
                     : "memory");
      if (KT & 1)
        asm volatile("ld.shared.f64 %0, [%1];"
                     : "=d"(e[j][KT - 1])
                     : "r"(src + (unsigned)(j * CTape<KT>::ROW + CTape<KT>::lane_offset(lane, KT - 1)) * 8u)
                     : "memory");
    }
    request((c + SLOTS - 1) & (SLOTS - 1));  // refill the slot consumed one block ago
    ++c;
  }
};

// the observation stream staged in shared memory, read by its shared-window address (LDS, vector loads for a block)
// instead of through a generic pointer (y_at / y_block of kf_p1.cuh for a global pointer)
struct SmemY {
  unsigned s;  // y[0], 16-byte aligned; the staged area is padded to whole 16-double lines
};
__device__ __forceinline__ double y_at(SmemY y, int t) {
  double r;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(r) : "r"(y.s + (unsigned)t * 8u));
  return r;
}
// t0 is a multiple of S and t0 + S - 1 < n rounded up to a multiple of 16: within the staged area
template <int S>
__device__ __forceinline__ void y_block(SmemY y, int t0, int, double (&yb)[S]) {
  static_assert(S % 2 == 0, "pairs");
#pragma unroll
  for (int j = 0; j < S; j += 2)
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(yb[j]), "=d"(yb[j + 1]) : "r"(y.s + (unsigned)(t0 + j) * 8u));
}

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

template <int M, bool NEED_Z, bool NEED_H, bool HAS_GOBS, int ZU, bool H0, bool CD>
__global__ void __launch_bounds__(32 * P1_WPC, (M <= 2) ? KFB_P1_MINB : 4)
    kf_p1_adjoint_kernel(const __grid_constant__ KfArgs A, int y_smem_doubles, int bulk_ok) {
  extern __shared__ __align__(128) double kf_dyn_smem[];
  constexpr int KT = tape_doubles<M, ZU>;
  constexpr int RS = (ZU == ZU_REDUCED) ? KF_CTAPE_STEPS : 1;  // steps per bulk copy
  using Ring = RingTape<KT, P1_SLOTS, RS>;
  const double* yp = A.y.p;
  if (y_smem_doubles > 0) {
    stage_y(kf_dyn_smem, A.y.p, y_smem_doubles, bulk_ok != 0);
    yp = kf_dyn_smem;
  }
  const int lane = threadIdx.x & 31;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform by construction
  const unsigned ring0_s = (unsigned)__cvta_generic_to_shared(kf_dyn_smem + ((y_smem_doubles + 15) & ~15));
  const unsigned bars_s = ring0_s + (unsigned)(P1_WPC * P1_SLOTS * Ring::BYTES);
  const long long wg = (long long)blockIdx.x * P1_WPC + warp;     // global warp index = block of 32 units
  const long long u = wg * 32 + lane;
  if (wg * 32 >= A.U) return;                                    // whole warp beyond the batch
  Ring tape;
  const unsigned ring_s = ring0_s + (unsigned)(warp * P1_SLOTS) * Ring::BYTES, wbars_s = bars_s + (unsigned)(warp * P1_SLOTS * 8);
  const bool store = u < A.U;
  const long long uu = store ? u : A.U - 1;
  if constexpr (ZU == ZU_REDUCED) {
    // blocks (n - 1) / S down to 0 of this warp
    const int bl = (A.n - 1) / RS;
    tape.init(ring_s, wbars_s, A.tape + CTape<KT>::row(A.U, wg * 32, bl * RS), CTape<KT>::block_stride(A.U),
              A.n >= 2 ? bl + 1 : 0, lane);
    if (y_smem_doubles > 0)
      backward_unit_p1<M, NEED_Z, NEED_H, HAS_GOBS, Ring, ZU, H0, CD>(
          A, uu, store, SmemY{(unsigned)__cvta_generic_to_shared(kf_dyn_smem)}, tape);
    else
      backward_unit_p1<M, NEED_Z, NEED_H, HAS_GOBS, Ring, ZU, H0, CD>(A, uu, store, A.y.p, tape);
  } else {
    const long long tstep = (long long)KT * tape_units_padded(A.U);
    tape.init(ring_s, wbars_s, A.tape + wg * (KT * 32) + (long long)(A.n - 2) * tstep, tstep, A.n - 1, lane);
    backward_unit_p1<M, NEED_Z, NEED_H, HAS_GOBS, Ring, ZU, H0>(A, uu, store, yp, tape);
  }
}

template <int M, bool NEED_Z, bool NEED_H, bool HAS_GOBS, int ZU, bool H0, bool CD>
static cudaError_t launch_one(const KfArgs& A, int ysm, int bulk_ok, cudaStream_t s) {
  constexpr int KT = tape_doubles<M, ZU>;
  constexpr int RS = (ZU == ZU_REDUCED) ? KF_CTAPE_STEPS : 1;
  const int block = 32 * P1_WPC;
  const unsigned grid = (unsigned)((A.U + block - 1) / block);
  const size_t smem = (size_t)((ysm + 15) & ~15) * 8 + (size_t)P1_WPC * P1_SLOTS * (RS * KT * 32 * 8 + 8);
  auto kern = kf_p1_adjoint_kernel<M, NEED_Z, NEED_H, HAS_GOBS, ZU, H0, CD>;
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
    return launch_one<M, V::NEED_Z, V::NEED_H, V::HAS_GOBS, V::ZU, V::H0, V::CD>(A, ysm, bulk_ok, s);
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
  double* tp = !SAVE ? nullptr : (ZU == ZU_REDUCED) ? A.tape : A.tape + (u >> 5) * (KT * 32) + (u & 31);
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
