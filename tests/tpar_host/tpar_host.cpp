// TEST-ONLY: the time-parallel filter and adjoint of csrc/kf_tpar.cuh run on the host.
//
// Emulates what kf_tpar.cu does on a CTA - `nchunks` threads each folding a contiguous chunk of steps, a scan over the
// chunk aggregates, a re-run of every chunk from its exclusive prefix - with a choice of scan tree, so that the
// combination operators can be checked against the oracle's sequential recursion without a GPU:
//   tree 0: left fold (prefix k = prefix k-1 (x) aggregate k);
//   tree 1: Hillis-Steele, as the kernels do it;
//   tree 2: recursive split at pseudo-random points (seeded), i.e. another bracketing of the same product.
#include <cstdint>
#include <vector>

#include "kf_tpar.cuh"

using namespace kfb;
using namespace kfb::tpar;

namespace {

unsigned g_seed = 12345u;
int next_split(int lo, int hi) {  // lo < split < hi
  g_seed = g_seed * 1103515245u + 12345u;
  return lo + 1 + (int)((g_seed >> 8) % (unsigned)(hi - lo - 1));
}

// inclusive prefix (FWD: agg[k] <- agg[0] .. agg[k] in time order) or suffix (!FWD: agg[k] <- agg[k] o .. o agg[K-1])
// of the chunk aggregates, under tree shape `tree`.  comb(i, j, o): o = i then j in time for FWD; o = i o j otherwise.
template <class E, class Comb>
void scan(std::vector<E>& agg, int tree, bool fwd, Comb comb) {
  const int K = (int)agg.size();
  E o;
  if (tree == 0) {
    if (fwd) for (int k = 1; k < K; ++k) { comb(agg[k - 1], agg[k], o); agg[k] = o; }
    else for (int k = K - 2; k >= 0; --k) { comb(agg[k], agg[k + 1], o); agg[k] = o; }
  } else if (tree == 1) {
    for (int off = 1; off < K; off <<= 1) {
      std::vector<E> nxt = agg;
      for (int k = 0; k < K; ++k) {
        if (fwd && k >= off) comb(agg[k - off], agg[k], nxt[k]);
        if (!fwd && k + off < K) comb(agg[k], agg[k + off], nxt[k]);
      }
      agg = nxt;
    }
  } else {
    struct Rec {
      static void go(std::vector<E>& a, int lo, int hi, bool fwd, Comb& comb) {
        if (hi - lo < 2) return;
        const int mid = next_split(lo, hi);
        go(a, lo, mid, fwd, comb);
        go(a, mid, hi, fwd, comb);
        E o;
        if (fwd) for (int k = mid; k < hi; ++k) { comb(a[mid - 1], a[k], o); a[k] = o; }
        else for (int k = lo; k < mid; ++k) { comb(a[k], a[mid], o); a[k] = o; }
      }
    };
    Rec::go(agg, 0, K, fwd, comb);
  }
}

struct Io {
  double *loglik, *ll_obs, *fs, *ps, *fc, *pc;
  int* info;
  const double *g_loglik, *g_ll_obs;
  double *ga0, *gP0, *gT, *gZ, *gH, *gC, *gc, *gd;
  int* sequential;  // receives 1 if an element was undefined, 2 if the scan drifted (both: the sequential walk)
};

template <int M>
int run(const UnitView& v, int nchunks, int tree, const Io& io, bool do_bwd) {
  constexpr int E = tape_entry<M>();
  const int n = v.n;
  const int chunk = (n + nchunks - 1) / nchunks;
  auto lo_of = [&](int k) { return k * chunk < n ? k * chunk : n; };
  auto hi_of = [&](int k) { return lo_of(k) + chunk < n ? lo_of(k) + chunk : n; };
  std::vector<double> tape((size_t)n * E);

  // ---- forward
  std::vector<FiltElem<M>> agg(nchunks);
  bool undefined = false;
  for (int k = 0; k < nchunks; ++k) {
    filt_identity<M>(agg[k]);
    FiltElem<M> e, tmp;
    for (int t = lo_of(k); t < hi_of(k); ++t) {
      if (t == 0) filt_element0<M>(v, e);
      else undefined |= !filt_element<M>(v, t, e);
      if (t == lo_of(k)) agg[k] = e;
      else { filt_combine<M>(agg[k], e, tmp); agg[k] = tmp; }
    }
  }
  if (io.sequential) *io.sequential = undefined ? 1 : 0;
  if (undefined) {
    forward_sequential_tape<M>(v, tape.data());
  } else {
    scan(agg, tree, true, [](const FiltElem<M>& i, const FiltElem<M>& j, FiltElem<M>& o) { filt_combine<M>(i, j, o); });
    for (int k = 0; k < nchunks; ++k) {
      FiltElem<M> f, e, tmp;
      for (int t = lo_of(k); t < hi_of(k); ++t) {
        if (t == 0) {
          filt_element0<M>(v, f);
          for (int i = 0; i < M; ++i) tape[i] = v.a0[i];
          for (int i = 0; i < M * M; ++i) tape[M + i] = v.P0[i];
        } else {
          filt_element<M>(v, t, e);
          filt_combine<M>(t == lo_of(k) ? agg[k - 1] : f, e, tmp);
          f = tmp;
        }
        if (t + 1 < n) predict_to_tape<M>(v, t, f.b, f.C, tape.data() + (size_t)(t + 1) * E);
      }
    }
  }
  FwdOut o{io.ll_obs, io.fs, io.ps, io.fc, io.pc};
  double ll = 0.0;
  int first_bad = -1;
  auto map = [&](bool check) {
    ll = 0.0;
    first_bad = -1;
    bool drift_any = false;
    for (int k = 0; k < nchunks; ++k) {
      double llk = 0.0;
      for (int t = lo_of(k); t < hi_of(k); ++t) {
        bool bad, drift;
        const double* next = (check && t + 1 < n) ? tape.data() + (size_t)(t + 1) * E : nullptr;
        llk += forward_map_step<M>(v, t, tape.data() + (size_t)t * E, next, o, &bad, &drift);
        if (bad && first_bad < 0) first_bad = t;
        drift_any = drift_any || drift;
      }
      ll += llk;
    }
    return drift_any;
  };
  if (map(!undefined) && !undefined) {  // the scan lost accuracy: sequential walk, map again (as the kernel does)
    forward_sequential_tape<M>(v, tape.data());
    map(false);
    if (io.sequential) *io.sequential = 2;
  }
  *io.info = first_bad < 0 ? 0 : first_bad + 1;
  *io.loglik = first_bad < 0 ? ll : nan("");
  if (!do_bwd) return 0;

  // ---- adjoint
  const double gl = io.g_loglik ? io.g_loglik[0] : 1.0;
  TX<M> x{nullptr, nullptr, 0, 1};
  BwdStep<M> B(x);
  std::vector<AffElem<M>> fa(nchunks);
  for (int k = 0; k < nchunks; ++k) {
    aff_identity<M>(fa[k]);
    AffElem<M> e, tmp;
    for (int t = hi_of(k) - 1; t >= lo_of(k); --t) {
      bwd_load<M>(x, v, t, tape.data() + (size_t)t * E, gl, io.g_ll_obs, B);
      aff_element<M>(B, e);
      if (t == hi_of(k) - 1) fa[k] = e;
      else { aff_combine<M>(e, fa[k], tmp); fa[k] = tmp; }
    }
  }
  scan(fa, tree, false, [](const AffElem<M>& i, const AffElem<M>& j, AffElem<M>& o) { aff_combine<M>(i, j, o); });
  std::vector<CongElem<M>> fx(nchunks);
  for (int k = 0; k < nchunks; ++k) {
    double ab[M], abn[M];
    for (int i = 0; i < M; ++i) ab[i] = k + 1 < nchunks ? fa[k + 1].s[i] : 0.0;
    cong_identity<M>(fx[k]);
    CongElem<M> e, tmp;
    for (int t = hi_of(k) - 1; t >= lo_of(k); --t) {
      bwd_load<M>(x, v, t, tape.data() + (size_t)t * E, gl, io.g_ll_obs, B);
      cong_element<M>(B, ab, e);
      aff_apply<M>(B, ab, abn);
      for (int i = 0; i < M; ++i) ab[i] = abn[i];
      if (t == hi_of(k) - 1) fx[k] = e;
      else { cong_combine<M>(e, fx[k], tmp); fx[k] = tmp; }
    }
  }
  scan(fx, tree, false, [](const CongElem<M>& i, const CongElem<M>& j, CongElem<M>& o) { cong_combine<M>(i, j, o); });
  // per-step contributions; static inputs are summed chunk by chunk (like the kernel's per-thread sums)
  for (int i = 0; i < M * M; ++i) { if (!v.T_ts) io.gT[i] = 0.0; if (!v.C_ts) io.gC[i] = 0.0; }
  for (int i = 0; i < M; ++i) { if (!v.c_ts) io.gc[i] = 0.0; if (!v.Z_ts) io.gZ[i] = 0.0; }
  if (!v.H_ts) io.gH[0] = 0.0;
  if (!v.d_ts) io.gd[0] = 0.0;
  for (int k = 0; k < nchunks; ++k) {
    double ab[M], abn[M], X[M * M];
    for (int i = 0; i < M; ++i) ab[i] = k + 1 < nchunks ? fa[k + 1].s[i] : 0.0;
    for (int i = 0; i < M * M; ++i) X[i] = k + 1 < nchunks ? fx[k + 1].S[i] : 0.0;
    StepGrad<M> g;
    CongElem<M> e;
    for (int t = hi_of(k) - 1; t >= lo_of(k); --t) {
      bwd_load<M>(x, v, t, tape.data() + (size_t)t * E, gl, io.g_ll_obs, B);
      if (t == 0) {
        adjoint_step<M>(B, v.d_sign, ab, X, g, io.ga0, io.gP0);
      } else {
        adjoint_step<M>(B, v.d_sign, ab, X, g, nullptr, nullptr);
        cong_element<M>(B, ab, e);
        cong_apply<M>(e, X);
        aff_apply<M>(B, ab, abn);
        for (int i = 0; i < M; ++i) ab[i] = abn[i];
      }
      for (int i = 0; i < M * M; ++i) (v.T_ts ? io.gT[t * M * M + i] = g.T[i] : io.gT[i] += g.T[i]);
      for (int i = 0; i < M * M; ++i) (v.C_ts ? io.gC[t * M * M + i] = g.C[i] : io.gC[i] += g.C[i]);
      for (int i = 0; i < M; ++i) (v.c_ts ? io.gc[t * M + i] = g.c[i] : io.gc[i] += g.c[i]);
      for (int i = 0; i < M; ++i) (v.Z_ts ? io.gZ[t * M + i] = g.Z[i] : io.gZ[i] += g.Z[i]);
      (v.H_ts ? io.gH[t] = g.H : io.gH[0] += g.H);
      (v.d_ts ? io.gd[t] = g.d : io.gd[0] += g.d);
    }
  }
  return 0;
}

}  // namespace

extern "C" int tpar_host_run(int m, int n, const double* y, const double* a0, const double* P0, const double* T,
                             const double* Z, const double* H, const double* C, const double* c, const double* d,
                             const long long* ts, double ll_const, double d_sign, int nchunks, int tree, unsigned seed,
                             double* loglik, double* ll_obs, double* fs, double* ps, double* fc, double* pc, int* info,
                             int* sequential, int do_bwd, const double* g_loglik, const double* g_ll_obs, double* ga0,
                             double* gP0, double* gT, double* gZ, double* gH, double* gC, double* gc, double* gd) {
  UnitView v{y, a0, P0, T, Z, H, C, c, d, ts[0], ts[1], ts[2], ts[3], ts[4], ts[5], ll_const, d_sign, n};
  g_seed = seed;
  Io io{loglik, ll_obs, fs, ps, fc, pc, info, g_loglik, g_ll_obs, ga0, gP0, gT, gZ, gH, gC, gc, gd, sequential};
  switch (m) {
    case 1: return run<1>(v, nchunks, tree, io, do_bwd != 0);
    case 2: return run<2>(v, nchunks, tree, io, do_bwd != 0);
    case 3: return run<3>(v, nchunks, tree, io, do_bwd != 0);
    case 4: return run<4>(v, nchunks, tree, io, do_bwd != 0);
    default: return 1;
  }
}
