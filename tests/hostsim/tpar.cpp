// TEST-ONLY: the time-parallel filter and adjoint of csrc/kf_tpar.cuh, and the time-parallel RTS smoother of
// csrc/kf_tpar_smooth.cuh, run on the host.
//
// Emulates what kf_tpar.cu / kf_tpar_smooth.cu do on a CTA - `nchunks` threads each running the headers' chunk
// functions on a contiguous chunk of steps, a scan over the chunk aggregates, the fallback decisions - with a choice of
// scan tree, so that the operators can be checked against the oracle without a GPU:
//   tree 0: fold in time order (prefix k = prefix k-1 (x) aggregate k; suffix k = aggregate k o suffix k+1);
//   tree 1: Hillis-Steele, as the kernels do it;
//   tree 2: recursive split at pseudo-random points (seeded), i.e. another bracketing of the same product.
#include <algorithm>
#include <vector>

#include "kf_run.cuh"
#include "kf_tpar_smooth.cuh"

using namespace kfb;
using namespace kfb::tpar;

namespace {

unsigned g_seed = 12345u;
int next_split(int lo, int hi) {  // lo < split < hi
  g_seed = g_seed * 1103515245u + 12345u;
  return lo + 1 + (int)((g_seed >> 8) % (unsigned)(hi - lo - 1));
}

// inclusive prefix (agg[k] <- agg[0] (x) .. (x) agg[k]) or, `suffix`, suffix scan (agg[k] <- agg[k] (x) .. (x) agg[K-1])
// of the chunk aggregates, under tree shape `tree`.  comb(i, j, o) gets the lower index first, as cta_scan's does.
template <class E, class Comb>
void scan(std::vector<E>& agg, int tree, bool suffix, Comb comb) {
  const int K = (int)agg.size();
  E o;
  if (tree == 0) {
    if (!suffix) for (int k = 1; k < K; ++k) { comb(agg[k - 1], agg[k], o); agg[k] = o; }
    else for (int k = K - 2; k >= 0; --k) { comb(agg[k], agg[k + 1], o); agg[k] = o; }
  } else if (tree == 1) {
    for (int off = 1; off < K; off <<= 1) {
      std::vector<E> nxt = agg;
      for (int k = 0; k < K; ++k) {
        if (!suffix && k >= off) comb(agg[k - off], agg[k], nxt[k]);
        if (suffix && k + off < K) comb(agg[k], agg[k + off], nxt[k]);
      }
      agg = nxt;
    }
  } else {
    struct Rec {
      static void go(std::vector<E>& a, int lo, int hi, bool suffix, Comb& comb) {
        if (hi - lo < 2) return;
        const int mid = next_split(lo, hi);
        go(a, lo, mid, suffix, comb);
        go(a, mid, hi, suffix, comb);
        E o;
        if (!suffix) for (int k = mid; k < hi; ++k) { comb(a[mid - 1], a[k], o); a[k] = o; }
        else for (int k = lo; k < mid; ++k) { comb(a[k], a[mid], o); a[k] = o; }
      }
    };
    Rec::go(agg, 0, K, suffix, comb);
  }
}

struct Io {
  double* loglik;
  int* info;
  FwdOut fwd;
  const double *g_loglik, *g_ll_obs;
  GradOut grad;
  int* sequential;  // receives 1 if an element was undefined, 2 if the scan drifted (both: the sequential walk)
};

template <int M>
void run_filter(const UnitView& v, int nchunks, int tree, const Io& io, bool do_bwd) {
  const int n = v.n;
  std::vector<double> tape((size_t)n * tape_entry<M>());

  // ---- forward
  std::vector<FiltElem<M>> agg(nchunks);
  bool undefined = false;
  for (int k = 0; k < nchunks; ++k) {
    const Chunk c = chunk_of(k, nchunks, n);
    undefined |= !filt_fold_chunk<M>(v, c.lo, c.hi, agg[k]);
  }
  if (io.sequential) *io.sequential = undefined ? 1 : 0;
  if (undefined) {
    forward_sequential_tape<M>(v, tape.data());
  } else {
    scan(agg, tree, false, filt_combine<M>);
    for (int k = 0; k < nchunks; ++k) {
      const Chunk c = chunk_of(k, nchunks, n);
      filt_rerun_chunk<M>(v, c.lo, c.hi, k > 0 ? &agg[k - 1] : nullptr, tape.data());
    }
  }
  double ll = 0.0;
  int first_bad = INT_MAX;
  auto map = [&](bool check) {
    ll = 0.0;
    first_bad = INT_MAX;
    bool drift = false;
    for (int k = 0; k < nchunks; ++k) {
      const Chunk c = chunk_of(k, nchunks, n);
      double llk;
      int bad;
      drift = forward_map_chunk<M>(v, c.lo, c.hi, tape.data(), check, io.fwd, &llk, &bad) || drift;
      ll += llk;
      first_bad = std::min(first_bad, bad);
    }
    return drift;
  };
  if (map(!undefined) && !undefined) {  // the scan lost accuracy: sequential walk, map again (as the kernel does)
    forward_sequential_tape<M>(v, tape.data());
    map(false);
    if (io.sequential) *io.sequential = 2;
  }
  *io.info = first_bad == INT_MAX ? 0 : first_bad + 1;
  *io.loglik = first_bad == INT_MAX ? ll : nan("");
  if (!do_bwd) return;

  // ---- adjoint
  const double gl = io.g_loglik ? io.g_loglik[0] : 1.0;
  std::vector<AffElem<M>> fa(nchunks);
  for (int k = 0; k < nchunks; ++k) {
    const Chunk c = chunk_of(k, nchunks, n);
    aff_fold_chunk<M>(v, c.lo, c.hi, tape.data(), gl, io.g_ll_obs, fa[k]);
  }
  scan(fa, tree, true, aff_combine<M>);
  const double zero[M * M] = {};
  std::vector<CongElem<M>> fx(nchunks);
  for (int k = 0; k < nchunks; ++k) {
    const Chunk c = chunk_of(k, nchunks, n);
    cong_fold_chunk<M>(v, c.lo, c.hi, tape.data(), gl, io.g_ll_obs, k + 1 < nchunks ? fa[k + 1].s : zero, fx[k]);
  }
  scan(fx, tree, true, cong_combine<M>);
  // static inputs' cotangents: per-chunk sums (like the kernel's per-thread sums), added in chunk order
  constexpr int W = static_grad_width<M>();
  double sum[W] = {}, acc[W], X[M * M];
  for (int k = 0; k < nchunks; ++k) {
    const Chunk c = chunk_of(k, nchunks, n);
    for (int i = 0; i < M * M; ++i) X[i] = k + 1 < nchunks ? fx[k + 1].S[i] : 0.0;
    adjoint_chunk<M>(v, c.lo, c.hi, tape.data(), gl, io.g_ll_obs, k + 1 < nchunks ? fa[k + 1].s : zero, X, io.grad,
                     acc);
    for (int j = 0; j < W; ++j) sum[j] += acc[j];
  }
  for (int j = 0; j < W; ++j) store_static_grad<M>(v, io.grad, j, sum[j]);
}

template <int M>
void run_smoother(const SmoothView& v, int nchunks, int tree, double tol, int* fallback) {
  std::vector<SmoothElem<M>> agg(nchunks);
  for (int k = 0; k < nchunks; ++k) {
    const Chunk c = chunk_of(k, nchunks, v.n);
    smooth_fold<M>(v, c.lo, c.hi, agg[k]);
  }
  scan(agg, tree, true, smooth_combine<M>);
  bool drift = false;
  for (int k = 0; k < nchunks; ++k) {
    const Chunk c = chunk_of(k, nchunks, v.n);
    drift = smooth_walk_check<M>(v, c.lo, c.hi, k + 1 < nchunks ? &agg[k + 1] : nullptr, agg[k], tol) || drift;
  }
  if (drift) smooth_sequential<M>(v);
  *fallback = drift ? 1 : 0;
}

}  // namespace

// kind, flags: the C ABI's filter kind and KFB_FLAG_* bits (k_endog = 1), applied by the library's rules.
extern "C" int tpar_host_run(int kind, unsigned flags, int m, int n, const double* y, const double* a0, const double* P0,
                             const double* T, const double* Z, const double* H, const double* C, const double* c,
                             const double* d, const long long* ts, int nchunks, int tree, unsigned seed, double* loglik,
                             double* ll_obs, double* fs, double* ps, double* fc, double* pc, int* info, int* sequential,
                             int do_bwd, const double* g_loglik, const double* g_ll_obs, double* ga0, double* gP0,
                             double* gT, double* gZ, double* gH, double* gC, double* gc, double* gd) {
  int mk;
  double ll_const, d_sign;
  if (!filter_rule(kind, 1, flags, &mk, &ll_const, &d_sign) || !tpar::supported(m, 1, mk)) return 1;
  UnitView v{y, a0, P0, T, Z, H, C, c, d, ts[0], ts[1], ts[2], ts[3], ts[4], ts[5], ll_const, d_sign, n};
  g_seed = seed;
  Io io{loglik, info, FwdOut{ll_obs, fs, ps, fc, pc}, g_loglik, g_ll_obs, GradOut{ga0, gP0, gT, gC, gc, gZ, gH, gd},
        sequential};
  tpar::with_instance(m, [&](auto M) { run_filter<M>(v, nchunks, tree, io, do_bwd != 0); });
  return 0;
}

// One unit: T, C = R Q R^T [m, m], fs [n, m], fc [n, m, m] -> ss, sc.  `tol` is the drift tolerance of the check (the
// kernel's is TPAR_DRIFT_TOL); 0 forces the fallback wherever the scan and the walk differ in any bit.
extern "C" int tpar_host_smooth_run(int m, int n, const double* T, const double* C, const double* fs, const double* fc,
                                    double* ss, double* sc, int nchunks, int tree, unsigned seed, double tol,
                                    int* fallback) {
  SmoothView v{T, C, fs, fc, ss, sc, n};
  g_seed = seed;
  return tpar::with_instance(m, [&](auto M) { run_smoother<M>(v, nchunks, tree, tol, fallback); }) ? 0 : 1;
}

// The sequential smoother of kf_smooth.cuh (smoother_unit) in the thread-per-unit context TX<M> on the host.
extern "C" int tpar_host_smooth_sequential(int n, int m, const double* T, const double* C, const double* fs,
                                           const double* fc, double* ss, double* sc) {
  SmoothArgs A;
  A.U = 1; A.n_series = 1; A.n = n; A.m = m;
  A.T = MatArg{T, 0, 0};
  A.C = MatArg{C, 0, 0};
  A.fs = fs; A.fc = fc; A.ss = ss; A.sc = sc;
  return tpar::with_instance(m, [&](auto M) {
    TX<M> x{nullptr, nullptr, 0, 1};
    smoother_unit(x, A, 0);
  }) ? 0 : 1;
}
