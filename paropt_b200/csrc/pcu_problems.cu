// pcu_problems.cu -- problem objects: host-callback problem (the ParOptProblem
// callback set through C function pointers) and the GPU-resident synthetic
// problems of DESIGN.md ("Synthetic problems").  These are the "user code" side
// of the boundary (ParOptProblem.h:143-282); their time is reported separately.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>

#include "pcu_kernels.cuh"
#include "pcu_problem.cuh"


WDesc pcu_make_wdesc(const pcu_weighting &w, int nvars) {
  WDesc d;
  memset(&d, 0, sizeof(d));
  d.nwcon = w.nwcon;
  d.nw = w.nw;
  d.wstride = w.wstride;
  d.wstart = w.wstart;
  d.wend = (long long)w.wstart + (long long)w.nwcon * w.wstride;
  d.coef0 = w.coef0;
  d.coef_rest = w.coef_rest;
  d.wconst = w.wconst;
  d.mode = 0;
  if (w.nwcon > 0) {
    const bool pow2 = w.nw >= 2 && w.nw <= 64 && (w.nw & (w.nw - 1)) == 0;
    const bool aligned = w.wstart == 0 && w.wstride == w.nw &&
                         (long long)w.nwcon * w.nw <= (long long)nvars;
    d.mode = (pow2 && aligned) ? 1 : 2;
    if (d.mode == 1)
      for (int b = w.nw; b > 1; b >>= 1) d.nw_log2++;
  }
  return d;
}

// One rule for every object that takes a pcu_weighting (pcu_problem_create[_host],
// pcu_blockmat_create, pcu_ip): the rows must lie inside the vector and must not
// overlap (the block-diagonal Ew = Cdiag + Aw D^-1 Aw^T of ParOptQuasiDefBlockMat,
// SM.cpp:41-115, assumes disjoint rows), and the inequality counts are counts.
// Returns 0 when the descriptor is usable, else prints the reason.
int pcu_validate_weighting(const pcu_weighting *w, int nvars, int ncon, int ninequality,
                           int nwinequality, const char *who) {
  const char *why = nullptr;
  if (nvars < 0) why = "negative number of variables";
  else if (ncon < 0 || ncon > PCU_MAX_COLS - 1) why = "number of dense constraints out of range";
  else if (ninequality > ncon) why = "ninequality exceeds ncon";
  const int nwcon = w ? w->nwcon : 0;
  if (!why && nwcon < 0) why = "negative number of weighting constraints";
  if (!why && nwcon > 0) {
    if (w->nw < 1) why = "nw < 1";
    else if (w->wstart < 0) why = "wstart < 0";
    else if (w->wstride < w->nw) why = "wstride < nw (overlapping rows)";
    else if ((long long)w->wstart + (long long)(nwcon - 1) * w->wstride + w->nw > (long long)nvars)
      why = "weighting rows reach outside the vector";
  }
  if (!why && nwinequality > nwcon) why = "nwinequality exceeds nwcon";
  if (why) {
    fprintf(stderr, "paropt_b200: %s: %s\n", who, why);
    return 1;
  }
  return 0;
}

static const WDesc &no_weighting() {
  static WDesc d;
  static bool init = false;
  if (!init) {
    memset(&d, 0, sizeof(d));
    init = true;
  }
  return d;
}

// ------------------------------------------------------------------ generator
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t stream_key(uint64_t seed,
                                                        uint64_t stream) {
  return splitmix64(seed ^ (stream * 0x9E3779B97F4A7C15ULL));
}
__host__ __device__ __forceinline__ double uniform01(uint64_t key, uint64_t idx) {
  return (double)(splitmix64(key + idx) >> 11) * (1.0 / 9007199254740992.0);
}
// a + b*u without fused contraction (bit-identical to the CPU statements)
__device__ __forceinline__ double affine(double a, double b, double u) {
  return __dadd_rn(a, __dmul_rn(b, u));
}

// =================================================================== sepquad
struct SepQuadDev {
  pcu_sepquad_params p;
  long long offset;
  uint64_t klam, kb, kv, kx;
};

struct SQInitF : NoStreams {  // lam, b, vh fill + sum vh^2
  static constexpr int NS = 1, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  SepQuadDev q;
  double *lam, *b, *vh;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &acc) const {
    double l[W], bb[W], v[W];
#pragma unroll
    for (int e = 0; e < W; e++) {
      const uint64_t gi = (uint64_t)(q.offset + i + e);
      l[e] = affine(q.p.lam_min, __dsub_rn(q.p.lam_max, q.p.lam_min),
                    uniform01(q.klam, gi));
      bb[e] = affine(q.p.b_lo, q.p.b_w, uniform01(q.kb, gi));
      v[e] = __dadd_rn(0.5, uniform01(q.kv, gi));
      acc.s[0] = fma(v[e], v[e], acc.s[0]);
    }
    stv<W>(lam, i, l);
    stv<W>(b, i, bb);
    if (vh) stv<W>(vh, i, v);
  }
};

struct SQBoundsF : NoStreams {  // getVarsAndBounds
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  SepQuadDev q;
  double *x, *lb, *ub;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {
    double xv[W], l[W], u[W];
#pragma unroll
    for (int e = 0; e < W; e++) {
      const long long li = i + e;
      const int k = (q.p.nw > 0 && (li % q.p.nw) != 0) ? 1 : 0;
      xv[e] = affine(q.p.x0_lo[k], q.p.x0_w[k],
                     uniform01(q.kx, (uint64_t)(q.offset + li)));
      l[e] = q.p.lb[k];
      u[e] = q.p.ub[k];
    }
    stv<W>(x, i, xv);
    stv<W>(lb, i, l);
    stv<W>(ub, i, u);
  }
};

// objective + up to 8 constraint sums per pass
struct SQObjF : NoStreams {
  static constexpr int NS = 9, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  SepQuadDev q;
  const double *x, *lam, *b, *vh;
  double hf;  // 2 (v.x) / (v.v) when householder
  int j0, nj;
  int with_obj;
  uint64_t keys[8];
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &acc) const {
    double xv[W];
    ldv<W>(x, i, xv);
    if (with_obj) {
      double l[W], bb[W], v[W];
      ldv<W>(lam, i, l);
      ldv<W>(b, i, bb);
#pragma unroll
      for (int e = 0; e < W; e++) v[e] = 0.0;
      if (vh) ldv<W>(vh, i, v);
#pragma unroll
      for (int e = 0; e < W; e++) {
        const double y = xv[e] - hf * v[e];
        acc.s[0] += 0.5 * l[e] * y * y + bb[e] * xv[e];
      }
    }
#pragma unroll
    for (int j = 0; j < 8; j++) {
      if (j < nj) {
#pragma unroll
        for (int e = 0; e < W; e++) {
          const double a = affine(q.p.a_lo, q.p.a_w,
                                  uniform01(keys[j], (uint64_t)(q.offset + i + e)));
          acc.s[1 + j] = fma(a, xv[e], acc.s[1 + j]);
        }
      }
    }
  }
};

// gradient stage 1: w = lam * (x - hf * vh) (+ b when not householder);
// reduces v.w
struct SQGrad1F : NoStreams {
  static constexpr int NS = 1, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *x, *lam, *b, *vh;
  double hf;
  double *g;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &acc) const {
    double xv[W], l[W], bb[W], v[W], o[W];
    ldv<W>(x, i, xv);
    ldv<W>(lam, i, l);
    if (vh) {
      ldv<W>(vh, i, v);
#pragma unroll
      for (int e = 0; e < W; e++) {
        o[e] = l[e] * (xv[e] - hf * v[e]);
        acc.s[0] = fma(v[e], o[e], acc.s[0]);
      }
    } else if (b) {
      ldv<W>(b, i, bb);
#pragma unroll
      for (int e = 0; e < W; e++) o[e] = l[e] * xv[e] + bb[e];
    } else {  // Hessian-vector product: no linear term
#pragma unroll
      for (int e = 0; e < W; e++) o[e] = l[e] * xv[e];
    }
    stv<W>(g, i, o);
  }
};

struct SQGrad2F : NoStreams {  // g = (w - hf2 * vh) + b
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *b, *vh;
  double hf2;
  double *g;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {
    double o[W], bb[W], v[W];
    ldv<W>(g, i, o);
    ldv<W>(vh, i, v);
    if (b) {
      ldv<W>(b, i, bb);
#pragma unroll
      for (int e = 0; e < W; e++) o[e] = (o[e] - hf2 * v[e]) + bb[e];
    } else {
#pragma unroll
      for (int e = 0; e < W; e++) o[e] = o[e] - hf2 * v[e];
    }
    stv<W>(g, i, o);
  }
};

struct SQConGradF : NoStreams {  // A_j[i] = a_lo + a_w u(100 + j, gi), up to 8 columns
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  SepQuadDev q;
  double *cols[8];
  uint64_t keys[8];
  int nj;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {
#pragma unroll
    for (int j = 0; j < 8; j++) {
      if (j < nj) {
        double a[W];
#pragma unroll
        for (int e = 0; e < W; e++)
          a[e] = affine(q.p.a_lo, q.p.a_w,
                        uniform01(keys[j], (uint64_t)(q.offset + i + e)));
        stv<W>(cols[j], i, a);
      }
    }
  }
};

// diag(P diag(lam) P) = lam - c1 v^2 lam + c2 v^2, c1 = 4 / (v.v), c2 = 4 (v.lam v) / (v.v)^2;
// with vlam set the pass only reduces v.lam v (once per problem)
struct SQHessDiagF : NoStreams {
  static constexpr int NS = 1, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *lam, *vh;
  double *h;
  double c1, c2;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &acc) const {
    double l[W], v[W], o[W];
    ldv<W>(lam, i, l);
    ldv<W>(vh, i, v);
#pragma unroll
    for (int e = 0; e < W; e++) {
      const double v2 = v[e] * v[e];
      if (h) o[e] = (l[e] - c1 * (v2 * l[e])) + c2 * v2;
      else acc.s[0] = fma(v2, l[e], acc.s[0]);
    }
    if (h) stv<W>(h, i, o);
  }
};

struct SepQuadProblem : pcu_problem {
  SepQuadDev q;
  pcu_vec *lam = nullptr, *b = nullptr, *vh = nullptr;
  double vtv = 0.0;
  double vlv = -1.0;  // v^T diag(lam) v (Householder), reduced at the first evalHessianDiag
  std::vector<double> beta;

  ~SepQuadProblem() {
    pcu_vec_destroy(lam);
    pcu_vec_destroy(b);
    pcu_vec_destroy(vh);
  }

  int init() {
    lam = pcu_vec_create(ctx, nvars);
    b = pcu_vec_create(ctx, nvars);
    if (q.p.householder) vh = pcu_vec_create(ctx, nvars);
    if (!lam || !b || (q.p.householder && !vh)) return 1;
    SQInitF f;
    f.q = q;
    f.lam = lam->d;
    f.b = b->d;
    f.vh = vh ? vh->d : nullptr;
    RedBuf rb = ctx->redbuf(1, 0, 0);
    if (pcu_launch_tile(ctx, f, nvars, no_weighting(), rb)) return 1;
    double out[1];
    if (ctx->fetch(out)) return 1;
    vtv = out[0];
    beta.resize(ncon);
    const uint64_t kbeta = stream_key(q.p.seed, 5);
    for (int j = 0; j < ncon; j++) {
      beta[j] = q.p.beta_c + q.p.beta_n * (double)q.p.ntotal +
                q.p.beta_u * uniform01(kbeta, (uint64_t)j);
    }
    return 0;
  }

  int getVarsAndBounds(pcu_vec *x, pcu_vec *lb, pcu_vec *ub) override {
    SQBoundsF f;
    f.q = q;
    f.x = x->d;
    f.lb = lb->d;
    f.ub = ub->d;
    RedBuf rb = {nullptr, nullptr, nullptr, 0};
    return pcu_launch_tile(ctx, f, nvars, no_weighting(), rb);
  }

  int householder_factor(pcu_vec *x, double *hf) {
    *hf = 0.0;
    if (!q.p.householder) return 0;
    double d;
    if (pcu_vec_dot(vh, x, &d)) return 1;
    *hf = 2.0 * d / vtv;
    return 0;
  }

  int evalObjCon(pcu_vec *x, double *fobj, double *cons) override {
    double hf;
    if (householder_factor(x, &hf)) return 1;
    std::vector<int> groups;
    int j0 = 0;
    do {
      SQObjF f;
      f.q = q;
      f.x = x->d;
      f.lam = lam->d;
      f.b = b->d;
      f.vh = vh ? vh->d : nullptr;
      f.hf = hf;
      f.j0 = j0;
      f.nj = ncon - j0 < 8 ? ncon - j0 : 8;
      f.with_obj = (j0 == 0);
      for (int j = 0; j < 8; j++)
        f.keys[j] = stream_key(q.p.seed, 100 + (uint64_t)(j0 + j));
      RedBuf rb = ctx->redbuf(9, 0, 0);
      if (pcu_launch_tile(ctx, f, nvars, no_weighting(), rb)) return 1;
      groups.push_back(j0);
      j0 += 8;
    } while (j0 < ncon);
    std::vector<double> out(9 * groups.size());
    if (ctx->fetch(out.data())) return 1;
    *fobj = out[0];
    for (size_t gi = 0; gi < groups.size(); gi++) {
      for (int j = 0; j < 8 && groups[gi] + j < ncon; j++)
        cons[groups[gi] + j] = beta[groups[gi] + j] + out[9 * gi + 1 + j];
    }
    return 0;
  }

  // H = P diag(lam) P is constant: hvec = gradient of the quadratic part at px
  int evalHvecProduct(pcu_vec *, const double *, pcu_vec *, pcu_vec *px, pcu_vec *hvec) override {
    return grad_into(px, hvec, false);
  }
  bool hasHvecProduct() const override { return true; }

  // The Hessian is constant (the constraints are linear): its exact diagonal, lam without
  // the reflector, else the diagonal of P diag(lam) P.
  int evalHessianDiag(pcu_vec *, const double *, pcu_vec *, pcu_vec *h) override {
    if (!q.p.householder) return pcu_vec_copy(h, lam);
    SQHessDiagF f;
    f.lam = lam->d;
    f.vh = vh->d;
    if (vlv < 0.0) {
      f.h = nullptr;
      RedBuf rb = ctx->redbuf(1, 0, 0);
      if (pcu_launch_tile(ctx, f, nvars, no_weighting(), rb)) return 1;
      if (ctx->fetch(&vlv)) return 1;
    }
    f.h = h->d;
    f.c1 = 4.0 / vtv;
    f.c2 = 4.0 * vlv / (vtv * vtv);
    RedBuf rb = ctx->redbuf(1, 0, 0);
    if (pcu_launch_tile(ctx, f, nvars, no_weighting(), rb)) return 1;
    // (no sum in this pass: drop its reduction slot without a host round trip)
    if (!ctx->pending.empty()) {
      ctx->result_used = ctx->pending.back().offset;
      ctx->pending.pop_back();
    }
    return 0;
  }
  bool hasHessianDiag() const override { return true; }

  int evalObjConGradient(pcu_vec *x, pcu_vec *g, pcu_vec **Ac) override {
    if (grad_into(x, g, true)) return 1;
    for (int j0 = 0; j0 < ncon; j0 += 8) {
      SQConGradF f;
      f.q = q;
      f.nj = ncon - j0 < 8 ? ncon - j0 : 8;
      for (int j = 0; j < f.nj; j++) {
        f.cols[j] = Ac[j0 + j]->d;
        f.keys[j] = stream_key(q.p.seed, 100 + (uint64_t)(j0 + j));
      }
      RedBuf rb = {nullptr, nullptr, nullptr, 0};
      if (pcu_launch_tile(ctx, f, nvars, no_weighting(), rb)) return 1;
    }
    return 0;
  }

  // g = P diag(lam) P x (+ b)
  int grad_into(pcu_vec *x, pcu_vec *g, bool with_b) {
    double hf;
    if (householder_factor(x, &hf)) return 1;
    SQGrad1F f1;
    f1.x = x->d;
    f1.lam = lam->d;
    f1.b = with_b ? b->d : nullptr;
    f1.vh = vh ? vh->d : nullptr;
    f1.hf = hf;
    f1.g = g->d;
    if (q.p.householder) {
      RedBuf rb = ctx->redbuf(1, 0, 0);
      if (pcu_launch_tile(ctx, f1, nvars, no_weighting(), rb)) return 1;
      double vw;
      if (ctx->fetch(&vw)) return 1;
      SQGrad2F f2;
      f2.b = with_b ? b->d : nullptr;
      f2.vh = vh->d;
      f2.hf2 = 2.0 * vw / vtv;
      f2.g = g->d;
      RedBuf rb2 = {nullptr, nullptr, nullptr, 0};
      if (pcu_launch_tile(ctx, f2, nvars, no_weighting(), rb2)) return 1;
    } else {
      // NS = 1 but unused: still needs a reduction slot for the harness
      RedBuf rb = ctx->redbuf(1, 0, 0);
      if (pcu_launch_tile(ctx, f1, nvars, no_weighting(), rb)) return 1;
      // discard that slot (the last one reserved) without a host round trip
      if (!ctx->pending.empty()) {
        ctx->result_used = ctx->pending.back().offset;
        ctx->pending.pop_back();
      }
    }
    return 0;
  }
};

// ================================================================ rosenbrock
struct RosenObjF : NoStreams {  // examples/rosenbrock/rosenbrock.cpp:49-79
  static constexpr int NS = 3, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *x;
  long long n;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &acc) const {
#pragma unroll
    for (int e = 0; e < W; e++) {
      const long long k = i + e;
      const double xi = x[k];
      if (k < n - 1) {
        const double d = x[k + 1] - xi * xi;
        acc.s[0] += (1.0 - xi) * (1.0 - xi) + 100.0 * d * d;
      }
      acc.s[1] -= xi * xi;
      if ((k & 1) == 0) acc.s[2] += xi;
    }
  }
};

struct RosenGradF : NoStreams {  // rosenbrock.cpp:82-107
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *x;
  double *g, *a0, *a1;
  long long n;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &) const {
#pragma unroll
    for (int e = 0; e < W; e++) {
      const long long k = i + e;
      const double xi = x[k];
      double gv = 0.0;
      if (k > 0) {
        const double xm = x[k - 1];
        gv += 200.0 * (xi - xm * xm);
      }
      if (k < n - 1) {
        const double d = x[k + 1] - xi * xi;
        gv += -2.0 * (1.0 - xi) + 200.0 * d * (-2.0 * xi);
      }
      g[k] = gv;
      a0[k] = -2.0 * xi;
      a1[k] = ((k & 1) == 0) ? 1.0 : 0.0;
    }
  }
};

struct RosenProblem : pcu_problem {
  int getVarsAndBounds(pcu_vec *x, pcu_vec *lb, pcu_vec *ub) override {
    return pcu_vec_set(x, -1.0) || pcu_vec_set(lb, -2.0) || pcu_vec_set(ub, 1.0);
  }
  int evalObjCon(pcu_vec *x, double *fobj, double *cons) override {
    if (ctx->world > 1) {
      fprintf(stderr, "paropt_b200: the rosenbrock problem is single-rank\n");
      return 1;
    }
    RosenObjF f;
    f.x = x->d;
    f.n = nvars;
    RedBuf rb = ctx->redbuf(3, 0, 0);
    if (pcu_launch_tile(ctx, f, nvars, no_weighting(), rb)) return 1;
    double out[3];
    if (ctx->fetch(out)) return 1;
    *fobj = out[0];
    cons[0] = out[1] + 0.25;
    cons[1] = out[2] + 10.0;
    return 0;
  }
  int evalObjConGradient(pcu_vec *x, pcu_vec *g, pcu_vec **Ac) override {
    RosenGradF f;
    f.x = x->d;
    f.g = g->d;
    f.a0 = Ac[0]->d;
    f.a1 = Ac[1]->d;
    f.n = nvars;
    RedBuf rb = {nullptr, nullptr, nullptr, 0};
    return pcu_launch_tile(ctx, f, nvars, no_weighting(), rb);
  }
};

// ============================================================ host callbacks
struct CallbackProblem : pcu_problem {
  pcu_problem_callbacks cb;
  int getVarsAndBounds(pcu_vec *x, pcu_vec *lb, pcu_vec *ub) override {
    return cb.get_vars_and_bounds(cb.user, x, lb, ub);
  }
  int evalObjCon(pcu_vec *x, double *fobj, double *cons) override {
    return cb.eval_obj_con(cb.user, x, fobj, cons);
  }
  int evalObjConGradient(pcu_vec *x, pcu_vec *g, pcu_vec **Ac) override {
    return cb.eval_obj_con_gradient(cb.user, x, g, Ac);
  }
  int qnUpdateCorrection(pcu_vec *x, const double *z, pcu_vec *zw, pcu_vec *s,
                         pcu_vec *y) override {
    return cb.qn_update_correction ? cb.qn_update_correction(cb.user, x, z, zw, s, y) : 0;
  }
  bool hasQnUpdateCorrection() const override { return cb.qn_update_correction != nullptr; }
  int writeOutput(int iter, pcu_vec *x) override {
    return cb.write_output ? cb.write_output(cb.user, iter, x) : 0;
  }
  int evalHvecProduct(pcu_vec *x, const double *z, pcu_vec *zw, pcu_vec *px,
                      pcu_vec *hvec) override {
    return cb.eval_hvec_product ? cb.eval_hvec_product(cb.user, x, z, zw, px, hvec) : 1;
  }
  bool hasHvecProduct() const override { return cb.eval_hvec_product != nullptr; }
  // pcu_problem_set_hessian_diag
  void *hd_user = nullptr;
  int (*hd_eval)(void *, pcu_vec *, const double *, pcu_vec *, pcu_vec *) = nullptr;
  int evalHessianDiag(pcu_vec *x, const double *z, pcu_vec *zw, pcu_vec *h) override {
    return hd_eval ? hd_eval(hd_user, x, z, zw, h) : 1;
  }
  bool hasHessianDiag() const override { return hd_eval != nullptr; }
};

// ======================================================= host-array callbacks
// The reference's problem callbacks read and write ParOptVec::getArray host
// pointers; here those arrays are page-locked mirrors owned by the problem.
static double host_now_ms() {
  using namespace std::chrono;
  return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

struct HostProblem : pcu_problem {
  pcu_host_callbacks cb;
  double t_d2h = 0.0, t_user = 0.0, t_h2d = 0.0;  // wall-clock ms per phase
  bool timing = false;  // PCU_HOST_TIMING: synchronise after the uploads to time them
  double *hx = nullptr, *hg = nullptr, *hzw = nullptr;
  double *hh = nullptr;  // the diagonal Hessian's mirror (allocated at its first call)
  std::vector<double *> hA;
  // pcu_problem_set_hessian_diag_host
  void *hd_user = nullptr;
  int (*hd_eval)(void *, int, const double *, const double *, int, const double *,
                 double *) = nullptr;
  cudaEvent_t up_done = nullptr;  // last host->device copy of g / A
  bool up_pending = false;

  ~HostProblem() {
    if (hx) cudaFreeHost(hx);
    if (hg) cudaFreeHost(hg);
    if (hzw) cudaFreeHost(hzw);
    if (hh) cudaFreeHost(hh);
    for (double *p : hA)
      if (p) cudaFreeHost(p);
    if (up_done) cudaEventDestroy(up_done);
  }
  int init() {
    const size_t bytes = sizeof(double) * (size_t)(nvars > 0 ? nvars : 1);
    PCU_CUDA_OK(cudaHostAlloc(&hx, bytes, cudaHostAllocDefault));
    PCU_CUDA_OK(cudaHostAlloc(&hg, bytes, cudaHostAllocDefault));
    // getVarsAndBounds needs three arrays: at least two gradient mirrors
    hA.assign(ncon > 1 ? ncon : 1, nullptr);
    for (size_t j = 0; j < hA.size(); j++)
      PCU_CUDA_OK(cudaHostAlloc(&hA[j], bytes, cudaHostAllocDefault));
    PCU_CUDA_OK(cudaEventCreateWithFlags(&up_done, cudaEventDisableTiming));
    return 0;
  }
  int wait_uploads() {  // the callbacks may overwrite hg / hA only after this
    if (up_pending) {
      PCU_CUDA_OK(cudaEventSynchronize(up_done));
      up_pending = false;
    }
    return 0;
  }
  int fetch_x(pcu_vec *x) {
    if (same_point_hint) return 0;
    const size_t bytes = sizeof(double) * (size_t)nvars;
    const double t0 = host_now_ms();
    if (timing) cudaStreamSynchronize(ctx->stream);  // kernels that produce x
    const double t1 = timing ? host_now_ms() : t0;
    if (nvars > 0) {
      PCU_CUDA_OK(cudaMemcpyAsync(hx, x->d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
      PCU_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    }
    t_d2h += host_now_ms() - t1;
    d2h_bytes += (long long)bytes;
    return 0;
  }
  int push(pcu_vec *v, const double *h) {
    const size_t bytes = sizeof(double) * (size_t)nvars;
    if (nvars > 0)
      PCU_CUDA_OK(cudaMemcpyAsync(v->d, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    h2d_bytes += (long long)bytes;
    return 0;
  }
  int getVarsAndBounds(pcu_vec *x, pcu_vec *lb, pcu_vec *ub) override {
    if (wait_uploads()) return 1;
    int fail = cb.get_vars_and_bounds(cb.user, nvars, hx, hg, hA[0]);
    if (push(x, hx) || push(lb, hg) || push(ub, hA[0])) return 1;
    PCU_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    return fail;
  }
  int evalObjCon(pcu_vec *x, double *fobj, double *cons) override {
    if (fetch_x(x)) return 1;
    const double t0 = host_now_ms();
    const int fail = cb.eval_obj_con(cb.user, nvars, hx, fobj, cons);
    t_user += host_now_ms() - t0;
    return fail;
  }
  int writeOutput(int iter, pcu_vec *x) override {
    if (!cb.write_output) return 0;
    const int keep = same_point_hint;
    same_point_hint = 0;  // the iterate may have moved since the last callback
    const int rc = fetch_x(x);
    same_point_hint = keep;
    if (rc) return 1;
    return cb.write_output(cb.user, iter, nvars, hx);
  }
  int evalObjConGradient(pcu_vec *x, pcu_vec *g, pcu_vec **Ac) override {
    if (fetch_x(x) || wait_uploads()) return 1;
    const double t0 = host_now_ms();
    int fail = cb.eval_obj_con_gradient(cb.user, nvars, hx, hg, hA.data());
    const double t1 = host_now_ms();
    t_user += t1 - t0;
    if (push(g, hg)) return 1;
    for (int j = 0; j < ncon; j++)
      if (push(Ac[j], hA[j])) return 1;
    if (timing) {
      cudaStreamSynchronize(ctx->stream);
      t_h2d += host_now_ms() - t1;
    }
    // stream-ordered: the kernels that consume g / A are enqueued behind the copies
    PCU_CUDA_OK(cudaEventRecord(up_done, ctx->stream));
    up_pending = true;
    return fail;
  }
  // hvec = H(x, z, zw) px on host arrays: x in hx, px in hg, the result in hA[0]
  int evalHvecProduct(pcu_vec *x, const double *z, pcu_vec *zw, pcu_vec *px,
                      pcu_vec *hvec) override {
    if (!cb.eval_hvec_product) return 1;
    same_point_hint = 0;  // the iterate may have moved since the last callback
    if (fetch_x(x) || wait_uploads()) return 1;
    if (nwcon > 0 && !hzw)
      PCU_CUDA_OK(cudaHostAlloc(&hzw, sizeof(double) * (size_t)nwcon, cudaHostAllocDefault));
    if (nvars > 0)
      PCU_CUDA_OK(cudaMemcpyAsync(hg, px->d, sizeof(double) * (size_t)nvars,
                                  cudaMemcpyDeviceToHost, ctx->stream));
    if (nwcon > 0)
      PCU_CUDA_OK(cudaMemcpyAsync(hzw, zw->d, sizeof(double) * (size_t)nwcon,
                                  cudaMemcpyDeviceToHost, ctx->stream));
    PCU_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    d2h_bytes += (long long)(sizeof(double) * ((size_t)nvars + (size_t)nwcon));
    const double t0 = host_now_ms();
    const int fail = cb.eval_hvec_product(cb.user, nvars, hx, z, nwcon, hzw, hg, hA[0]);
    t_user += host_now_ms() - t0;
    if (push(hvec, hA[0])) return 1;
    PCU_CUDA_OK(cudaEventRecord(up_done, ctx->stream));
    up_pending = true;
    return fail;
  }
  bool hasHvecProduct() const override { return cb.eval_hvec_product != nullptr; }
  // h = diag H(x, z, zw) on host arrays: x in hx, zw copied to the host, h in its own
  // mirror and one host->device copy
  int evalHessianDiag(pcu_vec *x, const double *z, pcu_vec *zw, pcu_vec *h) override {
    if (!hd_eval) return 1;
    if (fetch_x(x)) return 1;
    if (nwcon > 0 && !hzw)
      PCU_CUDA_OK(cudaHostAlloc(&hzw, sizeof(double) * (size_t)nwcon, cudaHostAllocDefault));
    if (!hh)
      PCU_CUDA_OK(cudaHostAlloc(&hh, sizeof(double) * (size_t)(nvars > 0 ? nvars : 1),
                                cudaHostAllocDefault));
    if (wait_uploads()) return 1;  // hh of the previous call may still be on its way
    if (nwcon > 0) {
      PCU_CUDA_OK(cudaMemcpyAsync(hzw, zw->d, sizeof(double) * (size_t)nwcon,
                                  cudaMemcpyDeviceToHost, ctx->stream));
      PCU_CUDA_OK(cudaStreamSynchronize(ctx->stream));
      d2h_bytes += (long long)(sizeof(double) * (size_t)nwcon);
    }
    const double t0 = host_now_ms();
    const int fail = hd_eval(hd_user, nvars, hx, z, nwcon, hzw, hh);
    t_user += host_now_ms() - t0;
    if (push(h, hh)) return 1;
    PCU_CUDA_OK(cudaEventRecord(up_done, ctx->stream));
    up_pending = true;
    return fail;
  }
  bool hasHessianDiag() const override { return hd_eval != nullptr; }
};

extern "C" {

pcu_problem *pcu_problem_create(pcu_ctx *ctx, int nvars, int ncon,
                                int ninequality, int nwinequality,
                                int use_lower, int use_upper,
                                const pcu_weighting *weighting,
                                const pcu_problem_callbacks *callbacks) {
  if (!ctx || !callbacks) return nullptr;
  if (pcu_validate_weighting(weighting, nvars, ncon, ninequality, nwinequality,
                             "pcu_problem_create"))
    return nullptr;
  CallbackProblem *p = new CallbackProblem;
  p->ctx = ctx;
  p->nvars = nvars;
  p->ncon = ncon;
  memset(&p->weighting, 0, sizeof(p->weighting));
  if (weighting) p->weighting = *weighting;
  p->nwcon = p->weighting.nwcon;
  // defaults of ParOptProblem::setProblemSizes (ParOptProblem.cpp:47-59)
  p->ninequality = ninequality < 0 ? ncon : ninequality;
  p->nwinequality = nwinequality < 0 ? p->nwcon : nwinequality;
  p->use_lower = use_lower;
  p->use_upper = use_upper;
  p->cb = *callbacks;
  return p;
}

void pcu_problem_destroy(pcu_problem *prob) { delete prob; }

int pcu_problem_set_hessian_diag(pcu_problem *prob, void *user,
                                 int (*eval_hessian_diag)(void *user, pcu_vec *x,
                                                          const double *z, pcu_vec *zw,
                                                          pcu_vec *h)) {
  CallbackProblem *p = dynamic_cast<CallbackProblem *>(prob);
  if (!p) return 1;
  p->hd_user = user;
  p->hd_eval = eval_hessian_diag;
  return 0;
}

int pcu_problem_set_hessian_diag_host(pcu_problem *prob, void *user,
                                      int (*eval_hessian_diag)(void *user, int n,
                                                               const double *x,
                                                               const double *z, int nw,
                                                               const double *zw,
                                                               double *h)) {
  HostProblem *p = dynamic_cast<HostProblem *>(prob);
  if (!p) return 1;
  p->hd_user = user;
  p->hd_eval = eval_hessian_diag;
  return 0;
}

pcu_problem *pcu_problem_create_host(pcu_ctx *ctx, int nvars, int ncon,
                                     int ninequality, int nwinequality,
                                     int use_lower, int use_upper,
                                     const pcu_weighting *weighting,
                                     const pcu_host_callbacks *callbacks) {
  if (!ctx || !callbacks) return nullptr;
  if (pcu_validate_weighting(weighting, nvars, ncon, ninequality, nwinequality,
                             "pcu_problem_create_host"))
    return nullptr;
  HostProblem *p = new HostProblem;
  p->ctx = ctx;
  p->nvars = nvars;
  p->ncon = ncon;
  memset(&p->weighting, 0, sizeof(p->weighting));
  if (weighting) p->weighting = *weighting;
  p->nwcon = p->weighting.nwcon;
  p->ninequality = ninequality < 0 ? ncon : ninequality;
  p->nwinequality = nwinequality < 0 ? p->nwcon : nwinequality;
  p->use_lower = use_lower;
  p->use_upper = use_upper;
  p->cb = *callbacks;
  if (p->init()) {
    delete p;
    return nullptr;
  }
  p->timing = getenv("PCU_HOST_TIMING") != nullptr;
  return p;
}

int pcu_problem_host_times(pcu_problem *prob, double *d2h_ms, double *user_ms,
                           double *h2d_ms) {
  HostProblem *p = dynamic_cast<HostProblem *>(prob);
  if (!p) return 1;
  if (d2h_ms) *d2h_ms = p->t_d2h;
  if (user_ms) *user_ms = p->t_user;
  if (h2d_ms) *h2d_ms = p->t_h2d;
  return 0;
}

int pcu_problem_transfer_bytes(pcu_problem *prob, int64_t *h2d, int64_t *d2h) {
  if (!prob) return 1;
  if (h2d) *h2d = prob->h2d_bytes;
  if (d2h) *d2h = prob->d2h_bytes;
  return 0;
}


pcu_problem *pcu_problem_create_sepquad(pcu_ctx *ctx,
                                        const pcu_sepquad_params *params) {
  if (!ctx || !params || params->ncon < 0 || params->ncon > PCU_MAX_COLS - 1 ||
      params->ntotal < 0 || params->nw < 0)
    return nullptr;
  SepQuadProblem *p = new SepQuadProblem;
  p->ctx = ctx;
  p->q.p = *params;
  // block-row partition in units of one weighting block (IP.cpp:214-229)
  const long long unit = params->nw > 0 ? params->nw : 1;
  const long long nunits = params->ntotal / unit;
  const long long u0 = (nunits * ctx->rank) / ctx->world;
  const long long u1 = (nunits * (ctx->rank + 1)) / ctx->world;
  p->q.offset = u0 * unit;
  long long n = (u1 - u0) * unit;
  if (ctx->rank == ctx->world - 1) n = params->ntotal - p->q.offset;
  p->nvars = (int)n;
  p->ncon = params->ncon;
  p->nwcon = params->nw > 0 ? (int)(u1 - u0) : 0;
  p->ninequality = p->ncon;
  p->nwinequality = p->nwcon;
  p->q.klam = stream_key(params->seed, 1);
  p->q.kb = stream_key(params->seed, 2);
  p->q.kv = stream_key(params->seed, 7);
  p->q.kx = stream_key(params->seed, 3);
  memset(&p->weighting, 0, sizeof(p->weighting));
  if (p->nwcon > 0) {
    p->weighting.nwcon = p->nwcon;
    p->weighting.wstart = 0;
    p->weighting.nw = params->nw;
    p->weighting.wstride = params->nw;
    p->weighting.coef0 = 1.0;
    p->weighting.coef_rest = -1.0;
    p->weighting.wconst = 0.0;
  }
  if (p->init()) {
    delete p;
    return nullptr;
  }
  return p;
}

pcu_problem *pcu_problem_create_rosenbrock(pcu_ctx *ctx, int nvars, int nwcon,
                                           int nwstart, int nw, int nwskip) {
  if (!ctx) return nullptr;
  RosenProblem *p = new RosenProblem;
  p->ctx = ctx;
  p->nvars = nvars;
  p->ncon = 2;
  p->nwcon = nwcon;
  p->ninequality = 2;
  p->nwinequality = nwcon;
  memset(&p->weighting, 0, sizeof(p->weighting));
  p->weighting.nwcon = nwcon;
  p->weighting.wstart = nwstart;
  p->weighting.nw = nw;
  p->weighting.wstride = nw + nwskip;
  p->weighting.coef0 = -1.0;
  p->weighting.coef_rest = -1.0;
  p->weighting.wconst = 1.0;
  if (pcu_validate_weighting(&p->weighting, nvars, 2, 2, nwcon, "pcu_problem_create_rosenbrock")) {
    delete p;
    return nullptr;
  }
  return p;
}

int pcu_problem_sizes(pcu_problem *prob, int *nvars, int *ncon, int *nwcon) {
  if (nvars) *nvars = prob->nvars;
  if (ncon) *ncon = prob->ncon;
  if (nwcon) *nwcon = prob->nwcon;
  return 0;
}

double pcu_problem_callback_ms(pcu_problem *prob) { return prob->callback_ms; }

}  // extern "C"
