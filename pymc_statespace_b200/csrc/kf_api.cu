// kf_api.cu - the extern "C" boundary declared in include/kfb200.h.
#include <atomic>
#include <cstdio>

#include "../../include/kfb200.h"
#include "kf_aux.cuh"
#include "kf_draws_run.cuh"
#include "kf_kernels.cuh"
#include "kf_tpar.cuh"

namespace kfb {

static std::atomic<long long> g_launches{0};
static thread_local const char* g_cuda_err = "";
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

bool p1_adjoint_supported(int m, int p, int mk);
cudaError_t launch_p1_adjoint(const KfArgs& A, int y_smem_doubles, int bulk_ok, cudaStream_t s);
cudaError_t launch_p1_forward(const KfArgs& A, int y_smem_doubles, int bulk_ok, cudaStream_t s);

cudaError_t launch_tpar(const KfArgs& A, bool bwd, cudaStream_t s);
cudaError_t launch_tpar_smoother(const SmoothArgs& S, cudaStream_t s);
cudaError_t launch_simulation_smoother(const ss::Args& A, cudaStream_t s);
cudaError_t launch_forecast_paths(const fc::Args& A, cudaStream_t s);
cudaError_t launch_impulse_response(const fc::IrfArgs& A, cudaStream_t s);
cudaError_t launch_conditional_forecast(const cf::Args& A, cudaStream_t s);
cudaError_t launch_masked_filter(const cf::FilterArgs& A, cudaStream_t s);

// k_states with launchers of their own, one object per size (kf_thread.cu: thread-per-unit filters and smoother;
// kf_coopT.cu: compile-time-dims kernels; the tensor-core DARE in kf_coopT.cu from k_states 10).  The Makefile repeats
// the first two lists (THREAD_MS, COOPT_MS): a size missing there leaves an undefined symbol in libkfb200.so.
#define KFB_THREAD_SIZES(X) X(1) X(2) X(3) X(4)
#define KFB_COOPT_SIZES(X) X(5) X(6) X(7) X(8) X(10) X(12) X(14) X(16) X(18) X(20) X(22) X(24) X(26) X(28) X(30) X(32)
#define KFB_DARED_SIZES(X) X(10) X(12) X(14) X(16) X(18) X(20) X(22) X(24) X(26) X(28) X(30) X(32)

#define KFB_DECL(M) thread_launch_fn thread_launcher_m##M(int p, int mk, bool tv); smoother_launch_fn smoother_thread_m##M();
KFB_THREAD_SIZES(KFB_DECL)
#undef KFB_DECL
#define KFB_DECL(M) coopT_launch_fn coopT_launcher_m##M(int p, int mk);
KFB_COOPT_SIZES(KFB_DECL)
#undef KFB_DECL
#define KFB_DECL(M) dare_launch_fn dareD_launcher_m##M(int p);
KFB_DARED_SIZES(KFB_DECL)
#undef KFB_DECL

thread_launch_fn find_thread_launcher(int m, int p, int mk, bool tv) {
  switch (m) {
#define KFB_CASE(M) case M: return thread_launcher_m##M(p, mk, tv);
    KFB_THREAD_SIZES(KFB_CASE)
#undef KFB_CASE
    default: return nullptr;
  }
}

smoother_launch_fn find_smoother_thread_launcher(int m) {
  switch (m) {
#define KFB_CASE(M) case M: return smoother_thread_m##M();
    KFB_THREAD_SIZES(KFB_CASE)
#undef KFB_CASE
    default: return nullptr;
  }
}

coopT_launch_fn find_coopT_launcher(int m, int p, int mk) {
  switch (m) {
#define KFB_CASE(M) case M: return coopT_launcher_m##M(p, mk);
    KFB_COOPT_SIZES(KFB_CASE)
#undef KFB_CASE
    default: return nullptr;
  }
}

dare_launch_fn find_dareD_launcher(int m, int p) {
  switch (m) {
#define KFB_CASE(M) case M: return dareD_launcher_m##M(p);
    KFB_DARED_SIZES(KFB_CASE)
#undef KFB_CASE
    default: return nullptr;
  }
}

struct Plan {
  int mk;
  double ll_const, d_sign;
  bool tv_any, use_thread;
  bool p1;           // k_endog = 1 with shared observations on the thread-per-unit path: the kernels of kf_p1.cu
  int struct_flags;  // KfArgs::struct_flags; KF_STRUCT_COMPRESSED: the compressed tape (CTape, kf_core.cuh)
  bool tpar;         // KFB_FLAG_TIME_PARALLEL: one CTA per unit, scans over time (kf_tpar.cu); tape [u][t][a_t, P_t]
  long long U, nD;
  int nTC;           // time entries of C = R Q R^T (1 or n)
  long long C_bs;    // 0 if R and Q are shared by all draws
  size_t off_C, off_Pss, off_Gss, off_dinfo, off_tape, off_gC, off_gPss, off_gGss, total;
};

static kfb_status make_plan(const kfb_desc* d, bool save, Plan* pl) {
  if (!d || d->n_draws <= 0 || d->n_series <= 0 || d->n <= 0 || d->m <= 0 || d->p <= 0 || d->r <= 0)
    return KFB_ERR_INVALID_ARG;
  if (!filter_rule(d->filter_kind, d->p, d->flags, &pl->mk, &pl->ll_const, &pl->d_sign)) return KFB_ERR_INVALID_ARG;
  pl->tv_any = d->T_ts || d->Z_ts || d->R_ts || d->H_ts || d->Q_ts || d->c_ts || d->d_ts;
  if (pl->tv_any && (pl->mk == MK_UNIV || pl->mk == MK_STEADY)) return KFB_ERR_UNSUPPORTED;
  // time-parallel form: k_endog = 1, k_states <= 4, standard-family filters only
  pl->tpar = (d->flags & KFB_FLAG_TIME_PARALLEL) != 0;
  if (pl->tpar && !tpar::supported(d->m, d->p, pl->mk)) return KFB_ERR_UNSUPPORTED;
  pl->U = d->n_draws * d->n_series;
  pl->nD = d->n_draws;
  pl->nTC = (d->R_ts || d->Q_ts) ? d->n : 1;
  const bool C_batched = d->R_bs || d->Q_bs;
  const long long nDC = C_batched ? d->n_draws : 1;
  pl->C_bs = C_batched ? (long long)pl->nTC * d->m * d->m : 0;
  pl->use_thread = !(d->flags & KFB_FLAG_FORCE_COOP) && find_thread_launcher(d->m, d->p, pl->mk, pl->tv_any) != nullptr;
  size_t off = 0;
  auto take = [&](size_t doubles) { size_t o = off; off += ((doubles * 8 + 255) / 256) * 256; return o; };
  pl->off_C = take((size_t)nDC * pl->nTC * d->m * d->m);
  pl->off_Pss = pl->off_Gss = pl->off_gPss = pl->off_gGss = 0;
  pl->off_dinfo = 0;
  if (pl->mk == MK_STEADY) {
    pl->off_Pss = take((size_t)pl->nD * d->m * d->m);
    pl->off_Gss = take((size_t)pl->nD * d->p * d->p);
    pl->off_dinfo = take((size_t)(pl->nD + 1) / 2);
  }
  // decided from the descriptor alone, so that workspace sizing, the forward pass and the adjoint always agree
  pl->p1 = pl->use_thread && !pl->tv_any && d->y_bs == 0 && d->n_series == 1 && !(d->flags & KFB_FLAG_GENERIC_ADJOINT) &&
           p1_adjoint_supported(d->m, d->p, pl->mk);
  pl->struct_flags = struct_flags_of(d->flags, d->p, d->Z_ts || d->H_ts, pl->p1);
  const bool compressed = (pl->struct_flags & KF_STRUCT_COMPRESSED) != 0;
  pl->off_tape = pl->off_gC = 0;
  if (pl->tpar) {
    // the forward pass always writes the tape (its parallel map reads the predicted moments back from it)
    pl->off_tape = take((size_t)pl->U * d->n * (d->m + d->m * d->m));
    if (save) pl->off_gC = take((size_t)pl->U * pl->nTC * d->m * d->m);
  } else if (save) {
    const size_t entries = compressed ? (size_t)ctape_steps_padded(d->n) * ctape_entry_doubles(d->m)
                                      : (size_t)(d->n > 1 ? d->n - 1 : 0) * tape_width(d->m);
    pl->off_tape = take((size_t)tape_units_padded(pl->U) * entries);
    pl->off_gC = take((size_t)pl->U * pl->nTC * d->m * d->m);
    if (pl->mk == MK_STEADY) {
      pl->off_gPss = take((size_t)pl->U * d->m * d->m);
      pl->off_gGss = take((size_t)pl->U * d->p * d->p);
    }
  }
  pl->total = off;
  return KFB_OK;
}

static void fill_args(const kfb_desc* d, const kfb_inputs* in, const Plan& pl, char* ws, KfArgs* A) {
  std::memset(A, 0, sizeof(*A));
  A->U = pl.U; A->n_series = d->n_series; A->n = d->n; A->m = d->m; A->p = d->p; A->math_kind = pl.mk;
  A->y = {in->y, d->y_bs, 0};
  A->a0 = {in->a0, d->a0_bs, 0};
  A->P0 = {in->P0, d->P0_bs, 0};
  A->T = {in->T, d->T_bs, d->T_ts};
  A->Z = {in->Z, d->Z_bs, d->Z_ts};
  A->H = {in->H, d->H_bs, d->H_ts};
  A->C = {(const double*)(ws + pl.off_C), pl.C_bs, pl.nTC > 1 ? (long long)d->m * d->m : 0};
  A->c = {in->c, d->c_bs, d->c_ts};
  A->d = {in->d, d->d_bs, d->d_ts};
  if (pl.mk == MK_STEADY) {
    A->Pss = {(const double*)(ws + pl.off_Pss), (long long)d->m * d->m, 0};  // one per draw
    A->Gss = {(const double*)(ws + pl.off_Gss), (long long)d->p * d->p, 0};
    A->dare_info = (const int*)(ws + pl.off_dinfo);
  }
  A->ll_const = pl.ll_const;
  A->d_sign = pl.d_sign;
  A->struct_flags = pl.struct_flags;
}

static kfb_status cuda_fail(cudaError_t e) {
  g_cuda_err = cudaGetErrorString(e);
  return KFB_ERR_CUDA;
}

// The status of a launcher's result: cudaErrorInvalidConfiguration means the request needs more than a launch allows.
static kfb_status launch_status(cudaError_t e) {
  if (e == cudaErrorInvalidConfiguration) return KFB_ERR_UNSUPPORTED;
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

static kfb_status launch_main(const kfb_desc* d, const Plan& pl, const KfArgs& A, bool bwd, cudaStream_t s) {
  cudaError_t e;
  if (pl.use_thread) {
    // shared observation stream -> stage it in shared memory once per CTA
    int ysm = 0, bulk_ok = 0;
    const long long ydoubles = (long long)d->n * d->p;
    if (d->y_bs == 0 && d->n_series == 1 && ydoubles * 8 <= 96 * 1024) {
      ysm = (int)ydoubles;
      bulk_ok = ((uintptr_t)A.y.p % 16 == 0) ? 1 : 0;
    }
    if ((A.struct_flags & KF_STRUCT_COMPRESSED) && bwd && (A.gZ || A.gH)) return KFB_ERR_UNSUPPORTED;  // Z, H constant
    // k_endog = 1, shared observations: the specialised adjoint with the TMA tape ring (kf_p1.cu)
    if (pl.p1 && bwd)
      e = launch_p1_adjoint(A, ysm, bulk_ok, s);
    else if (pl.p1 && !wants_step_outputs(A))
      e = launch_p1_forward(A, ysm, bulk_ok, s);
    else
      e = find_thread_launcher(d->m, d->p, pl.mk, pl.tv_any)(A, bwd, ysm, bulk_ok, s);
  } else {
    // sub-warp kernels with compile-time dims need uniform control flow across the units of a warp:
    // static matrices and ONE observation stream shared by every unit
    coopT_launch_fn ft = nullptr;
    if (!pl.tv_any && !(d->flags & KFB_FLAG_FORCE_COOP) && d->y_bs == 0 && d->n_series == 1)
      ft = find_coopT_launcher(d->m, d->p, pl.mk);
    e = ft ? ft(A, bwd, s) : launch_coop(A, bwd, s);
    if (e == cudaErrorInvalidConfiguration) return KFB_ERR_UNSUPPORTED;
  }
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

}  // namespace kfb

using namespace kfb;

extern "C" {
#pragma GCC visibility push(default)

int32_t kfb_version(void) { return KFB_VERSION; }

const char* kfb_status_string(kfb_status s) {
  switch (s) {
    case KFB_OK: return "ok";
    case KFB_ERR_INVALID_ARG: return "invalid argument";
    case KFB_ERR_UNSUPPORTED: return "unsupported configuration";
    case KFB_ERR_WORKSPACE: return "workspace missing or too small";
    case KFB_ERR_CUDA: return "CUDA error";
    default: return "unknown status";
  }
}

const char* kfb_last_cuda_error(void) { return g_cuda_err; }

int64_t kfb_launch_count(void) { return g_launches.load(); }

kfb_status kfb_workspace_bytes(const kfb_desc* desc, int32_t save_for_backward, size_t* bytes) {
  if (!bytes) return KFB_ERR_INVALID_ARG;
  Plan pl;
  kfb_status st = make_plan(desc, save_for_backward != 0, &pl);
  if (st != KFB_OK) return st;
  *bytes = pl.total;
  return KFB_OK;
}

kfb_status kfb_forward(const kfb_desc* desc, const kfb_inputs* in, const kfb_outputs* out, void* workspace,
                       size_t workspace_bytes, int32_t save_for_backward, void* stream) {
  if (!in || !out || !in->y || !in->a0 || !in->P0 || !in->T || !in->Z || !in->R || !in->H || !in->Q)
    return KFB_ERR_INVALID_ARG;
  Plan pl;
  kfb_status st = make_plan(desc, save_for_backward != 0, &pl);
  if (st != KFB_OK) return st;
  if (!workspace || workspace_bytes < pl.total) return KFB_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  KfArgs A;
  fill_args(desc, in, pl, ws, &A);
  A.loglik = out->loglik; A.ll_obs = out->ll_obs; A.fs = out->filtered_states; A.ps = out->predicted_states;
  A.fc = out->filtered_covs; A.pc = out->predicted_covs; A.info = out->info;
  A.tape = (save_for_backward || pl.tpar) ? (double*)(ws + pl.off_tape) : nullptr;
  const long long nDC = pl.C_bs ? desc->n_draws : 1;
  cudaError_t e = launch_rqr_forward(nDC, pl.nTC, desc->m, desc->r, MatArg{in->R, desc->R_bs, desc->R_ts},
                                     MatArg{in->Q, desc->Q_bs, desc->Q_ts}, (double*)(ws + pl.off_C), s);
  if (e != cudaSuccess) return cuda_fail(e);
  if (pl.mk == MK_STEADY) {
    // P_steady = DARE(T^T, Z^T, R Q R^T, H), F_inv = (Z P_steady Z^T + H)^-1   (kalman_filter.py:384-386)
    DareArgs D;
    std::memset(&D, 0, sizeof(D));
    D.nD = desc->n_draws; D.U = pl.U; D.n_series = desc->n_series; D.m = desc->m; D.p = desc->p;
    D.T = MatArg{in->T, desc->T_bs, 0}; D.Z = MatArg{in->Z, desc->Z_bs, 0}; D.H = MatArg{in->H, desc->H_bs, 0};
    D.C = A.C;
    D.Pss = (double*)(ws + pl.off_Pss); D.Gss = (double*)(ws + pl.off_Gss); D.info = (int*)(ws + pl.off_dinfo);
    const dare_launch_fn fast = (desc->flags & KFB_FLAG_FORCE_COOP) ? nullptr : find_dareD_launcher(desc->m, desc->p);
    e = fast ? fast(D, s) : launch_dare(D, false, s);  // even k_states 18..32, k_endog 1: tensor-core mapping (kf_rowsD.cuh)
    if (e == cudaErrorInvalidConfiguration) return KFB_ERR_UNSUPPORTED;
    if (e != cudaSuccess) return cuda_fail(e);
  }
  if (pl.tpar) {
    e = launch_tpar(A, false, s);
    return e == cudaSuccess ? KFB_OK : cuda_fail(e);
  }
  return launch_main(desc, pl, A, false, s);
}

kfb_status kfb_backward(const kfb_desc* desc, const kfb_inputs* in, const kfb_cotangents* cot, const kfb_grads* g,
                        void* workspace, size_t workspace_bytes, void* stream) {
  if (!in || !g || !in->y || !in->a0 || !in->P0 || !in->T || !in->Z || !in->R || !in->H || !in->Q)
    return KFB_ERR_INVALID_ARG;
  Plan pl;
  kfb_status st = make_plan(desc, true, &pl);
  if (st != KFB_OK) return st;
  if (!workspace || workspace_bytes < pl.total) return KFB_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  KfArgs A;
  fill_args(desc, in, pl, ws, &A);
  A.tape = (double*)(ws + pl.off_tape);
  A.g_loglik = cot ? cot->g_loglik : nullptr;
  A.g_ll_obs = cot ? cot->g_ll_obs : nullptr;
  A.ga0 = g->a0; A.gP0 = g->P0; A.gT = g->T; A.gZ = g->Z; A.gH = g->H; A.gc = g->c; A.gd = g->d;
  const bool want_C = g->R || g->Q;
  A.gC = want_C ? (double*)(ws + pl.off_gC) : nullptr;
  if (pl.mk == MK_STEADY) {
    A.gPss = (double*)(ws + pl.off_gPss);
    A.gGss = (double*)(ws + pl.off_gGss);
  }
  if (pl.tpar) {
    cudaError_t e = launch_tpar(A, true, s);
    if (e != cudaSuccess) return cuda_fail(e);
  } else {
    st = launch_main(desc, pl, A, true, s);
    if (st != KFB_OK) return st;
  }
  if (pl.mk == MK_STEADY) {
    // chain (P_steady-bar, F_inv-bar) through the DARE (utils/pytensor_scipy.py:39-60) into T, Z, H, C
    DareArgs D;
    std::memset(&D, 0, sizeof(D));
    D.nD = desc->n_draws; D.U = pl.U; D.n_series = desc->n_series; D.m = desc->m; D.p = desc->p;
    D.T = MatArg{in->T, desc->T_bs, 0}; D.Z = MatArg{in->Z, desc->Z_bs, 0}; D.H = MatArg{in->H, desc->H_bs, 0};
    D.C = A.C;
    D.Pss = (double*)(ws + pl.off_Pss); D.Gss = (double*)(ws + pl.off_Gss);
    D.gPss = A.gPss; D.gGss = A.gGss; D.gT = g->T; D.gZ = g->Z; D.gH = g->H; D.gC = A.gC;
    cudaError_t e = launch_dare(D, true, s);
    if (e == cudaErrorInvalidConfiguration) return KFB_ERR_UNSUPPORTED;
    if (e != cudaSuccess) return cuda_fail(e);
  }
  if (want_C) {
    cudaError_t e = launch_rqr_backward(pl.U, desc->n_series, pl.nTC, desc->R_ts ? desc->n : 1, desc->Q_ts ? desc->n : 1,
                                        desc->m, desc->r, MatArg{in->R, desc->R_bs, desc->R_ts},
                                        MatArg{in->Q, desc->Q_bs, desc->Q_ts}, A.gC, g->R, g->Q, 0, s);
    if (e != cudaSuccess) return cuda_fail(e);
  }
  return KFB_OK;
}

kfb_status kfb_smoother(int64_t n_draws, int64_t n_series, int32_t n, int32_t m, int32_t r, const double* T, int64_t T_bs,
                        const double* R, int64_t R_bs, const double* Q, int64_t Q_bs, const double* filtered_states,
                        const double* filtered_covs, double* smoothed_states, double* smoothed_covs, void* workspace,
                        size_t workspace_bytes, void* stream) {
  return kfb_smoother_ex(n_draws, n_series, n, m, r, T, T_bs, R, R_bs, Q, Q_bs, filtered_states, filtered_covs,
                         smoothed_states, smoothed_covs, workspace, workspace_bytes, 0u, stream);
}

kfb_status kfb_smoother_ex(int64_t n_draws, int64_t n_series, int32_t n, int32_t m, int32_t r, const double* T,
                           int64_t T_bs, const double* R, int64_t R_bs, const double* Q, int64_t Q_bs,
                           const double* filtered_states, const double* filtered_covs, double* smoothed_states,
                           double* smoothed_covs, void* workspace, size_t workspace_bytes, uint32_t flags, void* stream) {
  if (n_draws <= 0 || n_series <= 0 || n <= 0 || m <= 0 || r <= 0 || !T || !R || !Q || !filtered_states || !filtered_covs ||
      !smoothed_states || !smoothed_covs)
    return KFB_ERR_INVALID_ARG;
  if (flags & ~KFB_FLAG_TIME_PARALLEL) return KFB_ERR_INVALID_ARG;
  const bool tpar = (flags & KFB_FLAG_TIME_PARALLEL) != 0;
  if (tpar && !tpar::with_instance(m, [](auto) {})) return KFB_ERR_UNSUPPORTED;  // k_states 1..4
  const bool C_batched = R_bs || Q_bs;
  const long long nDC = C_batched ? n_draws : 1;
  const size_t need = (size_t)nDC * m * m * sizeof(double);
  if (!workspace || workspace_bytes < need) return KFB_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = launch_rqr_forward(nDC, 1, m, r, MatArg{R, R_bs, 0}, MatArg{Q, Q_bs, 0}, (double*)workspace, s);
  if (e != cudaSuccess) return cuda_fail(e);
  SmoothArgs S;
  S.U = n_draws * n_series; S.n_series = n_series; S.n = n; S.m = m;
  S.T = MatArg{T, T_bs, 0};
  S.C = MatArg{(const double*)workspace, C_batched ? (long long)m * m : 0, 0};
  S.fs = filtered_states; S.fc = filtered_covs; S.ss = smoothed_states; S.sc = smoothed_covs;
  if (tpar) {
    e = launch_tpar_smoother(S, s);
  } else {
    const smoother_launch_fn per_thread = find_smoother_thread_launcher(m);
    e = per_thread ? per_thread(S, s) : launch_smoother(S, s);
  }
  return launch_status(e);
}

kfb_status kfb_lyapunov_forward(int64_t B, int32_t m, int32_t r, const double* A, int64_t A_bs, const double* R,
                                int64_t R_bs, const double* Q, int64_t Q_bs, double* X, int32_t* info, void* stream) {
  if (B <= 0 || m <= 0 || r <= 0 || !A || !R || !Q || !X) return KFB_ERR_INVALID_ARG;
  cudaError_t e = launch_lyapunov_forward(B, m, r, MatArg{A, A_bs, 0}, MatArg{R, R_bs, 0}, MatArg{Q, Q_bs, 0}, X, info,
                                          (cudaStream_t)stream);
  return launch_status(e);
}

kfb_status kfb_lyapunov_backward(int64_t B, int32_t m, int32_t r, const double* A, int64_t A_bs, const double* R,
                                 int64_t R_bs, const double* Q, int64_t Q_bs, const double* X, const double* Xbar,
                                 double* Abar, double* Rbar, double* Qbar, void* stream) {
  if (B <= 0 || m <= 0 || r <= 0 || !A || !R || !Q || !X || !Xbar) return KFB_ERR_INVALID_ARG;
  cudaError_t e = launch_lyapunov_backward(B, m, r, MatArg{A, A_bs, 0}, MatArg{R, R_bs, 0}, MatArg{Q, Q_bs, 0}, X, Xbar,
                                           Abar, Rbar, Qbar, (cudaStream_t)stream);
  return launch_status(e);
}

kfb_status kfb_scatter_forward(int64_t B, int32_t n_theta, int32_t block, int32_t n_map, const double* theta,
                               const double* base, const int32_t* src_idx, const int32_t* dst_idx, double* dst,
                               void* stream) {
  if (B <= 0 || n_theta <= 0 || block <= 0 || n_map < 0 || !theta || !base || !dst) return KFB_ERR_INVALID_ARG;
  if (n_map > 0 && (!src_idx || !dst_idx)) return KFB_ERR_INVALID_ARG;
  cudaError_t e = launch_scatter_forward(B, n_theta, block, n_map, theta, base, src_idx, dst_idx, dst,
                                         (cudaStream_t)stream);
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

kfb_status kfb_scatter_backward(int64_t B, int32_t n_theta, int32_t block, int32_t n_map, const double* gdst,
                                const int32_t* src_idx, const int32_t* dst_idx, double* gtheta, void* stream) {
  if (B <= 0 || n_theta <= 0 || block <= 0 || n_map < 0 || !gdst || !gtheta) return KFB_ERR_INVALID_ARG;
  if (n_map > 0 && (!src_idx || !dst_idx)) return KFB_ERR_INVALID_ARG;
  cudaError_t e =
      launch_scatter_backward(B, n_theta, block, n_map, gdst, src_idx, dst_idx, gtheta, (cudaStream_t)stream);
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

static bool scatter_segs_ok(int32_t n_seg, const kfb_scatter_seg* segs, bool forward) {
  if (n_seg <= 0 || n_seg > KFB_MAX_SCATTER_SEGMENTS || !segs) return false;
  for (int q = 0; q < n_seg; ++q) {
    const kfb_scatter_seg& g = segs[q];
    if (g.block <= 0 || g.n_map < 0 || !g.data || (forward && !g.base)) return false;
    if (g.n_map > 0 && (!g.src_idx || !g.dst_idx)) return false;
  }
  return true;
}

kfb_status kfb_scatter_forward_multi(int64_t B, int32_t n_theta, int32_t n_seg, const kfb_scatter_seg* segs,
                                     const double* theta, void* stream) {
  if (B <= 0 || n_theta <= 0 || !theta || !scatter_segs_ok(n_seg, segs, true)) return KFB_ERR_INVALID_ARG;
  cudaError_t e = launch_scatter_forward_multi(B, n_theta, n_seg, segs, theta, (cudaStream_t)stream);
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

kfb_status kfb_scatter_backward_multi(int64_t B, int32_t n_theta, int32_t n_seg, const kfb_scatter_seg* segs,
                                      double* gtheta, void* stream) {
  if (B <= 0 || n_theta <= 0 || !gtheta || !scatter_segs_ok(n_seg, segs, false)) return KFB_ERR_INVALID_ARG;
  cudaError_t e = launch_scatter_backward_multi(B, n_theta, n_seg, segs, gtheta, (cudaStream_t)stream);
  return launch_status(e);  // UNSUPPORTED: the mapped elements exceed shared memory
}

kfb_status kfb_simulate(int64_t n_draws, int64_t sims_per_draw, int32_t n, int32_t m, int32_t p, int32_t r, const double* T,
                        int64_t T_bs, const double* Z, int64_t Z_bs, const double* R, int64_t R_bs, const double* H,
                        int64_t H_bs, const double* Q, int64_t Q_bs, const double* x0, int64_t x0_bs,
                        const double* z_state, const double* z_obs, double* states, double* obs, int32_t* info,
                        void* stream) {
  if (n_draws <= 0 || sims_per_draw <= 0 || n <= 0 || m <= 0 || p <= 0 || r <= 0 || !T || !Z || !R || !H || !Q || !z_state ||
      !z_obs || !states || !obs)
    return KFB_ERR_INVALID_ARG;
  if (m > 32 || p > 32 || r > 32) return KFB_ERR_UNSUPPORTED;
  cudaError_t e = launch_simulate(n_draws * sims_per_draw, sims_per_draw, n, m, p, r, MatArg{T, T_bs, 0}, MatArg{Z, Z_bs, 0},
                                  MatArg{R, R_bs, 0}, MatArg{H, H_bs, 0}, MatArg{Q, Q_bs, 0}, x0, x0_bs, z_state, z_obs,
                                  states, obs, info, (cudaStream_t)stream);
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

kfb_status kfb_mvn_draws(int64_t n_units, int64_t sims_per_unit, int32_t n, int32_t k, const double* mus, const double* covs,
                         const double* z, const double* jitter, double* out, int32_t* info, void* stream) {
  if (n_units <= 0 || sims_per_unit <= 0 || n <= 0 || k <= 0 || !mus || !covs || !z || !out) return KFB_ERR_INVALID_ARG;
  if (k > 32) return KFB_ERR_UNSUPPORTED;
  cudaError_t e = launch_mvn_draws(n_units * sims_per_unit, sims_per_unit, n, k, mus, covs, z, jitter, out, info,
                                   (cudaStream_t)stream);
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

kfb_status kfb_simulation_smoother_workspace_bytes(const kfb_desc* desc, int64_t sims_per_unit, size_t* bytes) {
  if (!bytes) return KFB_ERR_INVALID_ARG;
  draws::SsPlan pl;
  kfb_status st = draws::plan_ss(desc, sims_per_unit, &pl);
  if (st != KFB_OK) return st;
  *bytes = pl.total;
  return KFB_OK;
}

kfb_status kfb_simulation_smoother(const kfb_desc* desc, const kfb_inputs* in, const double* predicted_covs,
                                   int64_t sims_per_unit, const double* z_init, const double* z_state,
                                   const double* z_obs, double* states, int32_t* info, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  draws::SsPlan pl;
  kfb_status st = draws::plan_ss(desc, sims_per_unit, &pl);
  if (st != KFB_OK) return st;
  if (!in || !in->y || !in->a0 || !in->P0 || !in->T || !in->Z || !in->R || !in->H || !in->Q || !predicted_covs ||
      !z_init || (desc->n > 1 && !z_state) || !z_obs || !states || !info)
    return KFB_ERR_INVALID_ARG;
  if (!workspace || workspace_bytes < pl.total) return KFB_ERR_WORKSPACE;
  const ss::Args A =
      draws::ss_args(desc, in, predicted_covs, sims_per_unit, z_init, z_state, z_obs, states, info, workspace, pl);
  const draws::Fill f = draws::ss_status_init(A);
  cudaStream_t s = (cudaStream_t)stream;
  const cudaError_t e = cudaMemsetAsync(f.p, f.value, f.bytes, s);
  if (e != cudaSuccess) return cuda_fail(e);
  return launch_status(launch_simulation_smoother(A, s));
}

kfb_status kfb_forecast_paths_workspace_bytes(const kfb_desc* desc, int64_t sims_per_unit, size_t* bytes) {
  if (!bytes) return KFB_ERR_INVALID_ARG;
  draws::FcPlan pl;
  kfb_status st = draws::plan_fc(desc, sims_per_unit, &pl);
  if (st != KFB_OK) return st;
  *bytes = pl.total;
  return KFB_OK;
}

kfb_status kfb_forecast_paths(const kfb_desc* desc, const kfb_inputs* in, const double* start_mean,
                              const double* start_cov, int32_t horizon, int64_t sims_per_unit, const double* z_init,
                              const double* z_state, const double* z_obs, double* states, double* obs, int32_t* info,
                              void* workspace, size_t workspace_bytes, void* stream) {
  draws::FcPlan pl;
  kfb_status st = draws::plan_fc(desc, sims_per_unit, &pl);
  if (st != KFB_OK) return st;
  if (horizon < 1 || !in || !in->T || !in->Z || !in->R || !in->H || !in->Q || !start_mean || !start_cov || !z_init ||
      (horizon > 1 && !z_state) || !z_obs || (!states && !obs) || !info)
    return KFB_ERR_INVALID_ARG;
  if (!workspace || workspace_bytes < pl.total) return KFB_ERR_WORKSPACE;
  const fc::Args A = draws::fc_args(desc, in, start_mean, start_cov, horizon, sims_per_unit, z_init, z_state, z_obs,
                                    states, obs, info, workspace, pl);
  return launch_status(launch_forecast_paths(A, (cudaStream_t)stream));
}

kfb_status kfb_conditional_forecast_workspace_bytes(const kfb_desc* desc, int32_t horizon, int64_t sims_per_unit,
                                                    size_t* bytes) {
  if (!bytes) return KFB_ERR_INVALID_ARG;
  draws::CfPlan pl;
  kfb_status st = draws::plan_cf(desc, horizon, sims_per_unit, &pl);
  if (st != KFB_OK) return st;
  *bytes = pl.total;
  return KFB_OK;
}

kfb_status kfb_conditional_forecast(const kfb_desc* desc, const kfb_inputs* in, const double* start_mean,
                                    const double* start_cov, int32_t horizon, const double* cond, int64_t cond_bs,
                                    int64_t sims_per_unit, const double* z_init, const double* z_state,
                                    const double* z_obs, double* state_mean, double* state_cov, double* obs_mean,
                                    double* obs_cov, double* states, double* obs, int32_t* info, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  draws::CfPlan pl;
  kfb_status st = draws::plan_cf(desc, horizon, sims_per_unit, &pl);
  if (st != KFB_OK) return st;
  const bool paths = sims_per_unit > 0;
  if (!in || !in->T || !in->Z || !in->R || !in->H || !in->Q || !start_mean || !start_cov || !cond || cond_bs < 0 ||
      !info || (paths && (!z_init || (horizon > 1 && !z_state) || !z_obs || (!states && !obs))))
    return KFB_ERR_INVALID_ARG;
  if (!workspace || workspace_bytes < pl.total) return KFB_ERR_WORKSPACE;
  const cf::Args A = draws::cf_args(desc, in, start_mean, start_cov, horizon, cond, cond_bs, sims_per_unit, z_init,
                                    z_state, z_obs, state_mean, state_cov, obs_mean, obs_cov, states, obs, info,
                                    workspace, pl);
  return launch_status(launch_conditional_forecast(A, (cudaStream_t)stream));
}

kfb_status kfb_masked_filter_workspace_bytes(const kfb_desc* desc, size_t* bytes) {
  if (!bytes) return KFB_ERR_INVALID_ARG;
  draws::MfPlan pl;
  kfb_status st = draws::plan_mf(desc, &pl);
  if (st != KFB_OK) return st;
  *bytes = pl.total;
  return KFB_OK;
}

kfb_status kfb_masked_filter(const kfb_desc* desc, const kfb_inputs* in, double* predicted_states,
                             double* predicted_covs, int32_t* info, void* workspace, size_t workspace_bytes,
                             void* stream) {
  draws::MfPlan pl;
  kfb_status st = draws::plan_mf(desc, &pl);
  if (st != KFB_OK) return st;
  if (!in || !in->y || !in->a0 || !in->P0 || !in->T || !in->Z || !in->R || !in->H || !in->Q ||
      (!predicted_states && !predicted_covs) || !info)
    return KFB_ERR_INVALID_ARG;
  if (!workspace || workspace_bytes < pl.total) return KFB_ERR_WORKSPACE;
  const cf::FilterArgs A = draws::mf_args(desc, in, predicted_states, predicted_covs, info, workspace, pl);
  return launch_status(launch_masked_filter(A, (cudaStream_t)stream));
}

kfb_status kfb_impulse_response(const kfb_desc* desc, const kfb_inputs* in, int32_t horizon, int32_t shock,
                                double* states, double* obs, int32_t* info, void* stream) {
  kfb_status st = draws::check_desc(desc);
  if (st != KFB_OK) return st;
  if (horizon < 1 || shock < KFB_SHOCK_UNIT || shock > KFB_SHOCK_CHOLESKY || !in || !in->T || !in->Z || !in->R ||
      !in->Q || (!states && !obs) || !info)
    return KFB_ERR_INVALID_ARG;
  return launch_status(launch_impulse_response(draws::irf_args(desc, in, horizon, shock, states, obs, info),
                                               (cudaStream_t)stream));
}

kfb_status kfb_fp64_peak_distinct(int32_t iters, int32_t blocks, int32_t threads, double* sink, double* h_flops,
                                  void* stream) {
  if (iters <= 0 || blocks <= 0 || threads <= 0 || threads > 1024 || !sink) return KFB_ERR_INVALID_ARG;
  cudaError_t e = launch_fp64_peak_distinct(iters, blocks, threads, sink, (cudaStream_t)stream);
  if (h_flops) *h_flops = 2.0 * 8.0 * 16.0 * (double)iters * (double)blocks * (double)threads;
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

kfb_status kfb_fp64_peak(int32_t iters, int32_t blocks, int32_t threads, double* sink, double* h_flops, void* stream) {
  if (iters <= 0 || blocks <= 0 || threads <= 0 || threads > 1024 || !sink) return KFB_ERR_INVALID_ARG;
  cudaError_t e = launch_fp64_peak(iters, blocks, threads, sink, (cudaStream_t)stream);
  if (h_flops) *h_flops = 2.0 * 8.0 * 16.0 * (double)iters * (double)blocks * (double)threads;
  return e == cudaSuccess ? KFB_OK : cuda_fail(e);
}

#pragma GCC visibility pop
}  // extern "C"
