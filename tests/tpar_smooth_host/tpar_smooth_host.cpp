// TEST-ONLY: the time-parallel RTS smoother of csrc/kf_tpar_smooth.cuh run on the host.
//
// Emulates what kf_tpar_smooth.cu does on a CTA - `nchunks` threads each folding a contiguous chunk of steps, a suffix
// scan over the chunk aggregates, a checked walk of every chunk, the sequential fallback on drift - with a choice of scan
// tree, so that the operators can be checked against the oracle without a GPU:
//   tree 0: right fold (suffix k = aggregate k o suffix k+1);
//   tree 1: Hillis-Steele, as the kernel does it;
//   tree 2: recursive split at pseudo-random points (seeded), i.e. another bracketing of the same composition.
// `tol` is the drift tolerance of the check (the kernel's is TPAR_DRIFT_TOL); 0 forces the fallback wherever the scan
// and the walk differ in any bit.
#include <vector>

#include "kf_tpar_smooth.cuh"

using namespace kfb;
using namespace kfb::tpar;

namespace {

unsigned g_seed = 12345u;
int next_split(int lo, int hi) {  // lo < split < hi
  g_seed = g_seed * 1103515245u + 12345u;
  return lo + 1 + (int)((g_seed >> 8) % (unsigned)(hi - lo - 1));
}

// agg[k] <- agg[k] o .. o agg[K-1] under tree shape `tree`
template <int M>
void suffix_scan(std::vector<SmoothElem<M>>& agg, int tree) {
  const int K = (int)agg.size();
  SmoothElem<M> o;
  if (tree == 0) {
    for (int k = K - 2; k >= 0; --k) { smooth_combine<M>(agg[k], agg[k + 1], o); agg[k] = o; }
  } else if (tree == 1) {
    for (int off = 1; off < K; off <<= 1) {
      std::vector<SmoothElem<M>> nxt = agg;
      for (int k = 0; k + off < K; ++k) smooth_combine<M>(agg[k], agg[k + off], nxt[k]);
      agg = nxt;
    }
  } else {
    struct Rec {
      static void go(std::vector<SmoothElem<M>>& a, int lo, int hi) {
        if (hi - lo < 2) return;
        const int mid = next_split(lo, hi);
        go(a, lo, mid);
        go(a, mid, hi);
        SmoothElem<M> o;
        for (int k = lo; k < mid; ++k) { smooth_combine<M>(a[k], a[mid], o); a[k] = o; }
      }
    };
    Rec::go(agg, 0, K);
  }
}

template <int M>
int run(const SmoothView& v, int nchunks, int tree, double tol, int* fallback) {
  const int n = v.n;
  const int chunk = (n + nchunks - 1) / nchunks;
  auto lo_of = [&](int k) { return k * chunk < n ? k * chunk : n; };
  auto hi_of = [&](int k) { return lo_of(k) + chunk < n ? lo_of(k) + chunk : n; };
  std::vector<SmoothElem<M>> agg(nchunks);
  for (int k = 0; k < nchunks; ++k) smooth_fold<M>(v, lo_of(k), hi_of(k), agg[k]);
  suffix_scan<M>(agg, tree);
  bool drift = false;
  for (int k = 0; k < nchunks; ++k)
    drift = smooth_walk_check<M>(v, lo_of(k), hi_of(k), k + 1 < nchunks ? &agg[k + 1] : nullptr, agg[k], tol) || drift;
  if (drift) smooth_sequential<M>(v);
  *fallback = drift ? 1 : 0;
  return 0;
}

}  // namespace

// One unit: T, C = R Q R^T [m, m], fs [n, m], fc [n, m, m] -> ss, sc.
extern "C" int tpar_smooth_host_run(int m, int n, const double* T, const double* C, const double* fs, const double* fc,
                                    double* ss, double* sc, int nchunks, int tree, unsigned seed, double tol,
                                    int* fallback) {
  SmoothView v{T, C, fs, fc, ss, sc, n};
  g_seed = seed;
  switch (m) {
    case 1: return run<1>(v, nchunks, tree, tol, fallback);
    case 2: return run<2>(v, nchunks, tree, tol, fallback);
    case 3: return run<3>(v, nchunks, tree, tol, fallback);
    case 4: return run<4>(v, nchunks, tree, tol, fallback);
    default: return 1;
  }
}

// The sequential smoother of kf_smooth.cuh (smoother_unit, one unit per thread) on the host.
extern "C" int tpar_smooth_host_sequential(int m, int n, const double* T, const double* C, const double* fs,
                                           const double* fc, double* ss, double* sc) {
  SmoothArgs A;
  A.U = 1; A.n_series = 1; A.n = n; A.m = m;
  A.T = MatArg{T, 0, 0};
  A.C = MatArg{C, 0, 0};
  A.fs = fs; A.fc = fc; A.ss = ss; A.sc = sc;
  switch (m) {
    case 1: { TX<1> x{nullptr, nullptr, 0, 1}; smoother_unit(x, A, 0); return 0; }
    case 2: { TX<2> x{nullptr, nullptr, 0, 1}; smoother_unit(x, A, 0); return 0; }
    case 3: { TX<3> x{nullptr, nullptr, 0, 1}; smoother_unit(x, A, 0); return 0; }
    case 4: { TX<4> x{nullptr, nullptr, 0, 1}; smoother_unit(x, A, 0); return 0; }
    default: return 1;
  }
}
