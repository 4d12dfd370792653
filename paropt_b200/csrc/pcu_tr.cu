// pcu_tr.cu -- trust-region front end on the device (SURVEY.md section 8f-1):
// ParOptTrustRegion's SL1QP method with the adaptive penalty update
// (src/ParOptTrustRegion.cpp:1454-1690, 1248-1447, 1105-1240, 2391-2472) driving the
// CUDA-resident interior-point core on GPU-resident model problems:
//   QuadSubproblem   <-> ParOptQuadraticSubproblem (TR.cpp:27-441): the quadratic model
//                        f_k + g_k.p + 1/2 p.B p, c_k + A_k p inside the box |p| <= Delta
//   InfeasSubproblem <-> ParOptInfeasSubproblem (TR.cpp:443-660): the steering problem
// Every callback the interior-point iteration makes is vector algebra on device
// vectors -- one multi-dot pass per model evaluation through the compact quasi-Newton
// form, one linear-combination pass per model gradient -- so a whole trust-region
// iteration runs without a host callback; the user's problem is evaluated once per
// trust-region iteration (evalTrialStepAndUpdate).
//
// Not built: the filter acceptance strategy and the second-order correction
// (tr_accept_step_strategy = filter_method, tr_use_soc), ParOptCompactEigenQuasiNewton.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "pcu_ip.cuh"

int pcu_mdot_enqueue(pcu_ctx *ctx, const double *x, const ColTable &cols, int ncols,
                     long long n, int dst_off);

#define launch_tile pcu_launch_tile
static const RedBuf TR_NO_RED = {nullptr, nullptr, nullptr, 0};

// ------------------------------------------------------------------ kernels
// l_k = max(-Delta, lb - x_k), u_k = min(Delta, ub - x_k)   (TR.cpp:156-172)
struct TrBoundsF : NoStreams {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *x, *lb, *ub;
  double *lk, *uk;
  double tr;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &, AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W], const Elem (&)[W],
                                    const Con &, AccT &) const {
    double xv[W], l[W], u[W];
    ldv<W>(x, i, xv);
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
#pragma unroll
    for (int q = 0; q < W; q++) {
      const double a = l[q] - xv[q], b = u[q] - xv[q];
      l[q] = (-tr > a) ? -tr : a;
      u[q] = (tr < b) ? tr : b;
    }
    stv<W>(lk, i, l);
    stv<W>(uk, i, u);
  }
};

// cw(x) of the weighting rows into a W-vector (evalSparseCon, ParOptProblem.h:225)
struct SparseConF : NoStreams {
  static constexpr int NS = 0, NX = 0, NM = 0, NB = 1;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *x;
  double *out;
  double wconst;
  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W], Elem (&)[W],
                                    double (&part)[W][1], AccT *) const {
    double xv[W];
    ldv<W>(x, i, xv);
#pragma unroll
    for (int q = 0; q < W; q++) part[q][0] = coef[q] * xv[q];
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[1], Con &, AccT &) const {
    out[ci] = wconst + sum[0];
  }
  template <int W>
  __device__ __forceinline__ void C(long long, const double (&)[W], const Elem (&)[W],
                                    const Con &, AccT &) const {}
};

// Difference of the Lagrangian gradients at the trial point and at x_k with the new
// multipliers (TR.cpp:187-203; the sparse-constraint terms cancel for the linear
// weighting rows), fused with the three dots that open the quasi-Newton update:
//   t = (g_t - g_k) - sum_i z_i (At_i - Ak_i);   sums: t.t, t.s, s.s
struct LagDiffF : NoStreams {
  static constexpr int NS = 3, NX = 0, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *gt, *gk, *s;
  ColTable At, Ak;
  CoefTable z;
  int m;
  double *t;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &, AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W], const Elem (&)[W],
                                    const Con &, AccT &acc) const {
    double a[W], b[W], tv[W], sv[W];
    ldv<W>(gt, i, a);
    ldv<W>(gk, i, b);
    ldv<W>(s, i, sv);
#pragma unroll
    for (int q = 0; q < W; q++) tv[q] = a[q] - b[q];
    for (int j = 0; j < m; j++) {
      ldv<W>(At.p[j], i, a);
      ldv<W>(Ak.p[j], i, b);
#pragma unroll
      for (int q = 0; q < W; q++) tv[q] = fma(-z.v[j], a[q] - b[q], tv[q]);
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      acc.s[0] = fma(tv[q], tv[q], acc.s[0]);
      acc.s[1] = fma(tv[q], sv[q], acc.s[1]);
      acc.s[2] = fma(sv[q], sv[q], acc.s[2]);
    }
    stv<W>(t, i, tv);
  }
};

// KKT error of the outer problem (TR.cpp:2391-2472): r = g_k - A_k^T z - Aw^T zw, entries
// pointing out of an active bound dropped; sums: 0 |r|_1, 1 |g_k|_1;
// maxima: 0 |r|_inf, 1 |g_k|_inf, 2 |zw|_inf
struct KktErrF : NoStreams {
  static constexpr int NS = 2, NX = 3, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con1 Con;  // zw
  struct Elem {};
  const double *x, *lb, *ub, *g, *zw;
  ColTable Ak;
  CoefTable z;
  int m;
  double relax;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *) const {}
  __device__ __forceinline__ void B(long long ci, const double (&)[1], Con &con,
                                    AccT &acc) const {
    con.d[0] = zw[ci];
    acc.x[2] = fmax(acc.x[2], fabs(zw[ci]));
  }
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&coef)[W], const Elem (&)[W],
                                    const Con &con, AccT &acc) const {
    double xv[W], l[W], u[W], gv[W], r[W];
    ldv<W>(x, i, xv);
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
    ldv<W>(g, i, gv);
#pragma unroll
    for (int q = 0; q < W; q++) r[q] = gv[q];
    for (int j = 0; j < m; j++) {
      double a[W];
      ldv<W>(Ak.p[j], i, a);
#pragma unroll
      for (int q = 0; q < W; q++) r[q] = fma(-z.v[j], a[q], r[q]);
    }
#pragma unroll
    for (int q = 0; q < W; q++) {
      double w = fma(-coef[q], con.d[0], r[q]);
      if (xv[q] <= l[q] + relax && w > 0.0) w = 0.0;
      else if (xv[q] >= u[q] - relax && w < 0.0) w = 0.0;
      const double tw = fabs(w);
      acc.s[0] += tw;
      acc.x[0] = fmax(acc.x[0], tw);
      acc.s[1] += fabs(gv[q]);
      acc.x[1] = fmax(acc.x[1], fabs(gv[q]));
    }
  }
};

// ------------------------------------------------------------ QuadSubproblem
struct QuadSubproblem : pcu_problem {
  pcu_problem *prob = nullptr;
  QuasiNewton *qn = nullptr;  // may be null (sequential linear model)
  int n = 0, m = 0;
  WDesc wd;
  pcu_vec *xk = nullptr, *lk = nullptr, *uk = nullptr, *lb = nullptr, *ub = nullptr;
  pcu_vec *gk = nullptr, *gt = nullptr, *t = nullptr, *xtemp = nullptr;
  std::vector<pcu_vec *> Ak, At;
  double fk = 0.0, ft = 0.0;
  std::vector<double> ck, ct;
  int qn_update_type = 0;
  long model_version = 0;           // bumps whenever (g_k, A_k, B) change
  long ac_version = -1;             // model version whose A_k the optimizer's Ac vectors hold
  pcu_vec *ac_first = nullptr;
  std::vector<double> zts;          // Z^T step of the last evalObjCon (reused by the gradient)
  long zts_version = -1;
  const double *zts_point = nullptr;

  ~QuadSubproblem() {
    pcu_vec *single[] = {xk, lk, uk, lb, ub, gk, gt, t, xtemp, wconst_vec};
    for (pcu_vec *v : single) pcu_vec_destroy(v);
    for (pcu_vec *v : Ak) pcu_vec_destroy(v);
    for (pcu_vec *v : At) pcu_vec_destroy(v);
  }

  int init(pcu_problem *p, QuasiNewton *q) {
    prob = p;
    qn = q;
    ctx = p->ctx;
    n = nvars = p->nvars;
    m = ncon = p->ncon;
    nwcon = p->nwcon;
    ninequality = p->ninequality;
    nwinequality = p->nwinequality;
    use_lower = use_upper = 1;  // TR.cpp:271-273
    weighting = p->weighting;
    wd = pcu_make_wdesc(weighting, n);
    pcu_vec **nv[] = {&xk, &lk, &uk, &lb, &ub, &gk, &gt, &t, &xtemp};
    for (auto pv : nv) {
      *pv = pcu_vec_create(ctx, n);
      if (!*pv) return 1;
    }
    for (int i = 0; i < m; i++) {
      Ak.push_back(pcu_vec_create(ctx, n));
      At.push_back(pcu_vec_create(ctx, n));
      if (!Ak.back() || !At.back()) return 1;
    }
    wconst_vec = pcu_vec_create(ctx, nwcon);
    if (!wconst_vec) return 1;
    ck.assign(m, 0.0);
    ct.assign(m, 0.0);
    // defaults before initModelAndBounds (TR.cpp:63-68)
    return pcu_vec_set(lk, 0.0) || pcu_vec_set(uk, 1.0) || pcu_vec_set(lb, 0.0) ||
           pcu_vec_set(ub, 1.0) || pcu_vec_set(xk, 0.5);
  }

  int refreshSparseConstants() {  // cw(x_k): constants of the subproblem's rows
    if (nwcon == 0) return 0;
    SparseConF f;
    f.x = xk->d;
    f.out = wconst_vec->d;
    f.wconst = weighting.wconst;
    return launch_tile(ctx, f, n, wd, TR_NO_RED);
  }

  int setTrustRegionBounds(double tr) {  // TR.cpp:156-172
    TrBoundsF f;
    f.x = xk->d;
    f.lb = lb->d;
    f.ub = ub->d;
    f.lk = lk->d;
    f.uk = uk->d;
    f.tr = tr;
    WDesc w0;
    memset(&w0, 0, sizeof(w0));
    return launch_tile(ctx, f, n, w0, TR_NO_RED);
  }

  int initModelAndBounds(double tr) {  // TR.cpp:141-151
    if (prob->getVarsAndBounds(xk, lb, ub)) return 1;
    if (setTrustRegionBounds(tr)) return 1;
    if (prob->evalObjCon(xk, &fk, ck.data())) return 1;
    if (prob->evalObjConGradient(xk, gk, Ak.data())) return 1;
    model_version++;
    return refreshSparseConstants();
  }

  // ---- the callbacks the interior-point core makes (step = its design vector)
  int getVarsAndBounds(pcu_vec *step, pcu_vec *l, pcu_vec *u) override {  // TR.cpp:276-283
    if (pcu_vec_zero(step) || pcu_vec_axpy(step, 0.5, lk) || pcu_vec_axpy(step, 0.5, uk)) return 1;
    return pcu_vec_copy(l, lk) || pcu_vec_copy(u, uk);
  }

  // [Z | A_k | g_k | step]^T step in one multi-dot pass; returns them in `d`
  int modelDots(pcu_vec *step, std::vector<double> &d) {
    const int q = qn ? qn->size() : 0;
    ColTable cols;
    if (q > 0) qn->z_table(cols, 0);
    for (int i = 0; i < m; i++) cols.p[q + i] = Ak[i]->d;
    cols.p[q + m] = gk->d;
    cols.p[q + m + 1] = step->d;
    const int nc = q + m + 2;
    d.assign(nc, 0.0);
    if (pcu_mdot_enqueue(ctx, step->d, cols, nc, n, 0)) return 1;
    return ctx->big_fetch(nc, d.data());
  }

  int evalModel(pcu_vec *step, const double *c0, double *fobj, double *cons, bool quadratic) {
    std::vector<double> d;
    if (modelDots(step, d)) return 1;
    const int q = qn ? qn->size() : 0;
    double f = fk + d[q + m];
    if (qn && quadratic) {  // 1/2 p.B p through the compact form (QN.cpp:390-418)
      double pBp = qn->b0 * d[q + m + 1];
      if (q > 0) {
        std::vector<double> kap(q);
        qn->solve_compact(d.data(), kap.data());
        for (int i = 0; i < q; i++) pBp -= kap[i] * d[i];
      }
      f += 0.5 * pBp;
    }
    *fobj = f;
    for (int i = 0; i < m; i++) cons[i] = c0[i] + d[q + i];
    zts.assign(d.begin(), d.begin() + q);
    zts_version = model_version;
    zts_point = step->d;
    return 0;
  }

  int evalObjCon(pcu_vec *step, double *fobj, double *cons) override {  // TR.cpp:288-321
    if (!step) {
      *fobj = fk;
      for (int i = 0; i < m; i++) cons[i] = ck[i];
      return 0;
    }
    return evalModel(step, ck.data(), fobj, cons, true);
  }

  // constraint gradients: copies of A_k, skipped while the optimizer's vectors already
  // hold this model's (they are constant over a subproblem solve)
  int copyConGrad(pcu_vec **Ac) {
    if (m == 0) return 0;
    if (ac_version == model_version && ac_first == Ac[0]) return 0;
    for (int i = 0; i < m; i++)
      if (pcu_vec_copy(Ac[i], Ak[i])) return 1;
    ac_version = model_version;
    ac_first = Ac[0];
    return 0;
  }

  int evalObjConGradient(pcu_vec *step, pcu_vec *g, pcu_vec **Ac) override {  // TR.cpp:326-341
    if (copyConGrad(Ac)) return 1;
    if (!qn) return pcu_vec_copy(g, gk);
    // g = B step + g_k = b0 step - Z kap + g_k in one pass
    const int q = qn->size();
    LinCombF f;
    f.x = step->d;
    f.beta = qn->b0;
    f.out = g->d;
    f.ncols = q + 1;
    if (q > 0) {
      std::vector<double> rz(q), kap(q);
      if (same_point_hint && zts_version == model_version && zts_point == step->d &&
          (int)zts.size() == q) {
        rz = zts;  // Z^T step of the objective evaluation at this very point
      } else {
        ColTable zt;
        qn->z_table(zt, 0);
        if (pcu_mdot_enqueue(ctx, step->d, zt, q, n, 0)) return 1;
        if (ctx->big_fetch(q, rz.data())) return 1;
      }
      qn->solve_compact(rz.data(), kap.data());
      qn->z_table(f.V, 0);
      for (int i = 0; i < q; i++) f.alpha.v[i] = -kap[i];
    }
    f.V.p[q] = gk->d;
    f.alpha.v[q] = 1.0;
    WDesc w0;
    memset(&w0, 0, sizeof(w0));
    return launch_tile(ctx, f, n, w0, TR_NO_RED);
  }

  // ---- trust-region side
  // TR.cpp:174-212: evaluates the user's problem at x_k + step, updates the quasi-Newton
  // approximation with the Lagrangian-gradient difference
  int evalTrialStepAndUpdate(int update_flag, pcu_vec *step, const double *z, double *fobj,
                             double *cons) {
    if (pcu_vec_copy(xtemp, xk) || pcu_vec_axpy(xtemp, 1.0, step)) return 1;
    int fail = prob->evalObjCon(xtemp, &ft, ct.data());
    fail = fail || prob->evalObjConGradient(xtemp, gt, At.data());
    *fobj = ft;
    for (int i = 0; i < m; i++) cons[i] = ct[i];
    if (qn && update_flag) {
      LagDiffF f;
      f.gt = gt->d;
      f.gk = gk->d;
      f.s = step->d;
      f.m = m;
      for (int i = 0; i < m; i++) {
        f.At.p[i] = At[i]->d;
        f.Ak.p[i] = Ak[i]->d;
        f.z.v[i] = z[i];
      }
      f.t = t->d;
      WDesc w0;
      memset(&w0, 0, sizeof(w0));
      RedBuf rb = ctx->redbuf(3, 0, 0);
      if (launch_tile(ctx, f, n, w0, rb)) return 1;
      double dots[3];
      if (ctx->fetch(dots)) return 1;
      if (prob->hasQnUpdateCorrection()) {
        if (prob->qnUpdateCorrection(xtemp, z, nullptr, step, t)) return 1;
        if (pcu_vec_dot(t, t, &dots[0]) || pcu_vec_dot(t, step, &dots[1]) ||
            pcu_vec_dot(step, step, &dots[2]))
          return 1;
      }
      if (qn->update(step, t, dots[0], dots[1], dots[2], nullptr, &qn_update_type)) return 1;
      model_version++;
    }
    return fail;
  }

  int acceptTrialStep(pcu_vec *step) {  // TR.cpp:214-227 (buffers exchanged, not copied)
    fk = ft;
    if (pcu_vec_axpy(xk, 1.0, step)) return 1;
    std::swap(gk, gt);
    for (int i = 0; i < m; i++) {
      ck[i] = ct[i];
      std::swap(Ak[i], At[i]);
    }
    model_version++;
    return refreshSparseConstants();
  }
  void rejectTrialStep() {
    ft = 0.0;
    for (int i = 0; i < m; i++) ct[i] = 0.0;
  }
};

// ParOptInfeasSubproblem (TR.cpp:443-660): linear / constant / subproblem objective
// scaled by obj_scale, linear / subproblem constraints
struct InfeasSubproblem : pcu_problem {
  QuadSubproblem *sub = nullptr;
  int objective = 1;   // 0 constant, 1 linear, 2 subproblem
  int constraint = 0;  // 0 linear, 1 subproblem
  double obj_scale = 1.0;
  void init(QuadSubproblem *s, int obj, int con) {
    sub = s;
    ctx = s->ctx;
    nvars = s->nvars;
    ncon = s->ncon;
    nwcon = s->nwcon;
    ninequality = s->ninequality;
    nwinequality = s->nwinequality;
    use_lower = use_upper = 1;
    weighting = s->weighting;
    wconst_vec = s->wconst_vec;  // borrowed
    objective = obj;
    constraint = con;
  }
  ~InfeasSubproblem() { wconst_vec = nullptr; }
  int getVarsAndBounds(pcu_vec *x, pcu_vec *l, pcu_vec *u) override {
    return sub->getVarsAndBounds(x, l, u);
  }
  int evalObjCon(pcu_vec *step, double *fobj, double *cons) override {  // TR.cpp:541-579
    const bool quad = objective == 2;
    if (sub->evalModel(step, sub->ck.data(), fobj, cons, quad)) return 1;
    if (objective == 0) *fobj = sub->fk;
    *fobj *= obj_scale;
    return 0;
  }
  int evalObjConGradient(pcu_vec *step, pcu_vec *g, pcu_vec **Ac) override {  // TR.cpp:584-613
    if (objective == 2) {
      sub->same_point_hint = same_point_hint;
      if (sub->evalObjConGradient(step, g, Ac)) return 1;
    } else {
      if (sub->copyConGrad(Ac)) return 1;
      if (objective == 1) {
        if (pcu_vec_copy(g, sub->gk)) return 1;
      } else if (pcu_vec_zero(g)) {
        return 1;
      }
    }
    return pcu_vec_scale(g, obj_scale);
  }
};

// ------------------------------------------------------------------- pcu_tr
struct TrOptions {
  double tr_init_size = 0.1, tr_min_size = 1e-3, tr_max_size = 1.0, tr_eta = 0.25;
  double tr_bound_relax = 1e-4, function_precision = 1e-10;
  double tr_l1_tol = 1e-6, tr_linfty_tol = 1e-6, tr_infeas_tol = 1e-5;
  double tr_penalty_gamma_max = 1e4, tr_penalty_gamma_min = 0.0, penalty_gamma = 1000.0;
  int tr_adaptive_gamma_update = 1, tr_max_iterations = 200, tr_write_output_frequency = 10;
  int output_level = 0, qn_subspace_size = 10;
  std::string tr_accept_step_strategy = "penalty_method";
  std::string tr_adaptive_objective = "linear_objective";
  std::string tr_adaptive_constraint = "linear_constraint";
  std::string tr_steering_barrier_strategy = "mehrotra_predictor_corrector";
  std::string tr_steering_starting_point_strategy = "affine_step";
  std::string tr_output_file;
  std::string qn_type = "bfgs", qn_update_type = "skip_negative_curvature";
  std::string qn_diag_type = "yty_over_yts";
  // the interior-point options a steering solve swaps and restores
  std::string barrier_strategy = "monotone", starting_point_strategy = "affine_step";
  int sequential_linear_method = 0;
};

struct TrRecord {
  double f[16];  // iter fobj infeas l1 linfty smax tr rho model_red zav zmax gav gmax
                 // subproblem_iters adaptive_iters accepted
  double xsum, xnorm, xmaxabs;  // centre x_k at the start of the iteration
  std::string info;
};

struct pcu_tr {
  pcu_problem *prob = nullptr;
  pcu_ctx *ctx = nullptr;
  TrOptions opt;
  QuasiNewton *qn = nullptr;
  QuadSubproblem *sub = nullptr;
  InfeasSubproblem *infeas = nullptr;
  pcu_ip *ip = nullptr;
  std::vector<double> penalty_gamma;
  double tr_size = 0.1;
  int iter_count = 0, subproblem_iters = 0, adaptive_subproblem_iters = 0;
  int status = 0;  // 1 converged
  std::vector<TrRecord> history;
  FILE *outfp = nullptr;

  ~pcu_tr() {
    delete ip;
    delete infeas;
    delete sub;
    delete qn;
    if (outfp && outfp != stdout) fclose(outfp);
  }
  int build();
  int optimize();
  int minimizeInfeas(std::vector<double> &best_con_infeas);
  int computeKKTError(const double *z, pcu_vec *zw, double *l1, double *linfty);
  int sl1qpUpdate(pcu_vec *step, const double *z, pcu_vec *zw, double *infeas, double *l1,
                  double *linfty);
};

int pcu_ip_set_quasi_newton_object(pcu_ip *ip, QuasiNewton *qn);

int pcu_tr::build() {
  if (sub) return 0;
  if (opt.tr_accept_step_strategy != "penalty_method") {
    fprintf(stderr, "paropt_b200: tr_accept_step_strategy = %s is not built (penalty_method only)\n",
            opt.tr_accept_step_strategy.c_str());
    return 1;
  }
  int kind = -1;
  if (opt.qn_type == "bfgs") kind = 0;
  else if (opt.qn_type == "sr1") kind = 1;
  else if (opt.qn_type != "none") {
    fprintf(stderr, "paropt_b200: trust region: qn_type %s is not built\n", opt.qn_type.c_str());
    return 1;
  }
  if (kind >= 0) {  // ParOptOptimizer.cpp:118-163
    qn = new QuasiNewton;
    if (qn->init(ctx, prob->nvars, kind, opt.qn_subspace_size)) return 1;
    qn->damped = opt.qn_update_type == "damped_update";
    qn->diag_yts_over_sts = opt.qn_diag_type == "yts_over_sts";
  }
  sub = new QuadSubproblem;
  if (sub->init(prob, qn)) return 1;
  penalty_gamma.assign(prob->ncon, opt.penalty_gamma);  // TR.cpp:681-685
  tr_size = opt.tr_init_size;
  return 0;
}

// TR.cpp:2391-2472
int pcu_tr::computeKKTError(const double *z, pcu_vec *zw, double *l1, double *linfty) {
  KktErrF f;
  f.x = sub->xk->d;
  f.lb = sub->lb->d;
  f.ub = sub->ub->d;
  f.g = sub->gk->d;
  f.zw = zw->d;
  f.m = sub->m;
  for (int i = 0; i < sub->m; i++) {
    f.Ak.p[i] = sub->Ak[i]->d;
    f.z.v[i] = z[i];
  }
  f.relax = opt.tr_bound_relax;
  RedBuf rb = ctx->redbuf(2, 3, 0);
  if (launch_tile(ctx, f, sub->n, sub->wd, rb)) return 1;
  double out[5];
  if (ctx->fetch(out)) return 1;
  double zmax = sub->nwcon > 0 ? out[4] : 0.0;
  for (int i = 0; i < sub->m; i++) zmax = std::max(zmax, fabs(z[i]));
  zmax = std::max(1.0, zmax);
  *l1 = out[0] / std::max(out[1], zmax);
  *linfty = out[2] / std::max(out[3], zmax);
  return 0;
}

// TR.cpp:1105-1240: the steering problem gives the best infeasibility reachable inside
// the trust region (adaptive penalty update)
int pcu_tr::minimizeInfeas(std::vector<double> &best_con_infeas) {
  const int m = sub->m, nineq = sub->ninequality;
  const int obj = infeas->objective, con = infeas->constraint;
  if (pcu_ip_reset_problem(ip, infeas)) return 1;
  const std::string barrier0 = ip->opt.barrier_strategy, start0 = ip->opt.starting_point_strategy;
  const int slm0 = ip->opt.sequential_linear_method;
  if (opt.tr_steering_barrier_strategy != "default")
    ip->opt.barrier_strategy = opt.tr_steering_barrier_strategy;
  if (opt.tr_steering_starting_point_strategy != "default")
    ip->opt.starting_point_strategy = opt.tr_steering_starting_point_strategy;
  if ((obj == 0 || obj == 1) && con == 0) ip->opt.sequential_linear_method = 1;
  double gamma = 1e6;
  if (1e2 * opt.tr_penalty_gamma_max > gamma) gamma = 1e2 * opt.tr_penalty_gamma_max;
  infeas->obj_scale = 1.0 / gamma;
  if (pcu_ip_set_penalty_gamma(ip, 1.0)) return 1;
  if (pcu_ip_reset_design_and_bounds(ip)) return 1;
  if (pcu_ip_optimize(ip)) return 1;
  pcu_vec *step = ip->variables.v[PCU_X];
  adaptive_subproblem_iters = ip->niter;
  double dummy;
  if (sub->evalObjCon(step, &dummy, best_con_infeas.data())) return 1;
  for (int j = 0; j < m; j++) {
    if (j < nineq) best_con_infeas[j] = std::max(0.0, -best_con_infeas[j]);
    else best_con_infeas[j] = fabs(best_con_infeas[j]);
  }
  if (pcu_ip_set_penalty_gamma_array(ip, penalty_gamma.data())) return 1;
  if (pcu_ip_reset_problem(ip, sub)) return 1;
  ip->opt.starting_point_strategy = start0;
  ip->opt.barrier_strategy = barrier0;
  ip->opt.sequential_linear_method = slm0;
  return 0;
}

static void add_info(std::string &info, const char *fmt, ...) {
  char buf[64];
  va_list args;
  va_start(args, fmt);
  vsnprintf(buf, sizeof(buf), fmt, args);
  va_end(args);
  info += buf;
}

// TR.cpp:1248-1447
int pcu_tr::sl1qpUpdate(pcu_vec *step, const double *z, pcu_vec *zw, double *infeas_out,
                        double *l1, double *linfty) {
  const int m = sub->m, nineq = sub->ninequality;
  auto weighted_infeas = [&](const std::vector<double> &c, bool weighted) {
    double v = 0.0;
    for (int i = 0; i < m; i++) {
      const double w = weighted ? penalty_gamma[i] : 1.0;
      if (i < nineq) v += w * std::max(0.0, -c[i]);
      else v += w * fabs(c[i]);
    }
    return v;
  };
  double fk;
  std::vector<double> ck(m), ct(m);
  if (sub->evalObjCon(nullptr, &fk, ck.data())) return 1;
  const double infeas_k = weighted_infeas(ck, true);
  double ft;
  if (sub->evalObjCon(step, &ft, ct.data())) return 1;
  const double obj_reduc = fk - ft;
  const double infeas_model = weighted_infeas(ct, true);
  if (sub->evalTrialStepAndUpdate(1, step, z, &ft, ct.data())) return 1;
  const double infeas_t = weighted_infeas(ct, true);
  const double actual_reduc = (fk - ft + (infeas_k - infeas_t));
  const double model_reduc = obj_reduc + (infeas_k - infeas_model);
  double rho = 1.0;
  if (fabs(model_reduc) <= opt.function_precision && fabs(actual_reduc) <= opt.function_precision)
    rho = 1.0;
  else
    rho = actual_reduc / model_reduc;
  *infeas_out = weighted_infeas(ct, false);
  double smax = 0.0;
  int accepted = 0;
  if (rho >= opt.tr_eta || tr_size <= opt.tr_min_size) {
    if (pcu_vec_maxabs(step, &smax)) return 1;
    if (sub->acceptTrialStep(step)) return 1;
    accepted = 1;
  } else {
    sub->rejectTrialStep();
  }
  if (rho < 0.25) tr_size = std::max(0.25 * tr_size, opt.tr_min_size);
  else if (rho > 0.75) tr_size = std::min(1.5 * tr_size, opt.tr_max_size);
  if (sub->setTrustRegionBounds(tr_size)) return 1;
  if (computeKKTError(z, zw, l1, linfty)) return 1;
  double zmax = 0.0, zav = 0.0, gmax = 0.0, gav = 0.0;
  for (int i = 0; i < m; i++) {
    zav += fabs(z[i]);
    gav += penalty_gamma[i];
    zmax = std::max(zmax, fabs(z[i]));
    gmax = std::max(gmax, penalty_gamma[i]);
  }
  if (m > 0) {
    zav /= m;
    gav /= m;
  }
  std::string info;
  if (sub->qn_update_type == 1) add_info(info, "%s ", "dampH");
  else if (sub->qn_update_type == 2) add_info(info, "%s ", "skipH");
  if (opt.tr_adaptive_gamma_update) add_info(info, "%d/%d ", subproblem_iters, adaptive_subproblem_iters);
  else add_info(info, "%d ", subproblem_iters);
  if (!accepted) add_info(info, "%s ", "rej");
  if (outfp && ctx->rank == 0) {
    if (iter_count % 10 == 0 || opt.output_level > 0)
      fprintf(outfp, "\n%5s %12s %9s %9s %9s %9s %9s %9s %9s %9s %9s %9s %9s %9s %-12s\n", "iter",
              "fobj", "infeas", "l1", "linfty", "|x - xk|", "tr", "rho", "mod red.", "avg z",
              "max z", "avg pen.", "max pen.", "time(s)", "info");
    fprintf(outfp,
            "%5d %12.5e %9.2e %9.2e %9.2e %9.2e %9.2e %9.2e %9.2e %9.2e %9.2e %9.2e %9.2e %9.2e "
            "%-12s\n",
            iter_count, fk, *infeas_out, *l1, *linfty, smax, tr_size, rho, model_reduc, zav, zmax,
            gav, gmax, 0.0, info.c_str());
    fflush(outfp);
  }
  TrRecord &rec = history.back();
  const double vals[16] = {(double)iter_count, fk, *infeas_out, *l1, *linfty, smax, tr_size, rho,
                           model_reduc, zav, zmax, gav, gmax, (double)subproblem_iters,
                           (double)adaptive_subproblem_iters, (double)accepted};
  memcpy(rec.f, vals, sizeof(vals));
  while (!info.empty() && info.back() == ' ') info.pop_back();
  rec.info = info;
  iter_count++;
  return 0;
}

// TR.cpp:1454-1690 (sl1qpOptimize) behind ParOptTrustRegion::optimize (TR.cpp:2367)
int pcu_tr::optimize() {
  if (build()) return 1;
  const int m = sub->m, nineq = sub->ninequality;
  if (!opt.tr_output_file.empty() && !outfp && ctx->rank == 0)
    outfp = fopen(opt.tr_output_file.c_str(), "w");
  if (!ip) return 1;
  // the caller's interior-point options are in place; now what the front end forces
  if (pcu_ip_set_quasi_newton_object(ip, qn)) return 1;   // TR.cpp:1490
  ip->opt.use_quasi_newton_update = 0;                       // TR.cpp:1496
  ip->opt.write_output_frequency = 0;                        // TR.cpp:1500
  if (pcu_ip_set_penalty_gamma_array(ip, penalty_gamma.data())) return 1;
  int obj = 1, con = 0;
  if (opt.tr_adaptive_objective == "constant_objective") obj = 0;
  else if (opt.tr_adaptive_objective == "subproblem_objective") obj = 2;
  if (opt.tr_adaptive_constraint == "subproblem_constraint") con = 1;
  if (opt.tr_adaptive_gamma_update && !infeas) {
    infeas = new InfeasSubproblem;
    infeas->init(sub, obj, con);
  }
  std::vector<double> con_infeas(m), model_con_infeas(m), best_con_infeas(m);
  // initialize() TR.cpp:1087-1101
  if (sub->initModelAndBounds(tr_size)) return 1;
  iter_count = 0;
  status = 0;
  history.clear();
  for (int i = 0; i < opt.tr_max_iterations; i++) {
    if (opt.tr_adaptive_gamma_update && minimizeInfeas(best_con_infeas)) return 1;
    // the centre of this iteration (the reference's writeOutput hook, TR.cpp:1556-1560)
    TrRecord rec;
    memset(rec.f, 0, sizeof(rec.f));
    {
      double sums[4];
      if (pcu_vec_norm(sub->xk, &rec.xnorm) || pcu_vec_maxabs(sub->xk, &rec.xmaxabs)) return 1;
      pcu_vec *ones = sub->t;  // scratch: sum(x) = x . 1
      if (pcu_vec_set(ones, 1.0) || pcu_vec_dot(sub->xk, ones, &sums[0])) return 1;
      rec.xsum = sums[0];
    }
    history.push_back(rec);
    if (opt.tr_write_output_frequency > 0 && i % opt.tr_write_output_frequency == 0) {
      if (prob->writeOutput(i, sub->xk)) return 1;
    }
    if (pcu_ip_reset_design_and_bounds(ip)) return 1;
    if (pcu_ip_optimize(ip)) return 1;
    pcu_vec *step = ip->variables.v[PCU_X], *zw = ip->variables.v[PCU_ZW];
    const double *z = ip->variables.z.data();
    subproblem_iters = ip->niter;
    if (opt.tr_adaptive_gamma_update) {
      double f0, fmodel;
      if (sub->evalObjCon(nullptr, &f0, con_infeas.data())) return 1;
      if (sub->evalObjCon(step, &fmodel, model_con_infeas.data())) return 1;
      for (int j = 0; j < m; j++) {
        if (j < nineq) {
          con_infeas[j] = std::max(0.0, -con_infeas[j]);
          model_con_infeas[j] = std::max(0.0, -model_con_infeas[j]);
        } else {
          con_infeas[j] = fabs(con_infeas[j]);
          model_con_infeas[j] = fabs(model_con_infeas[j]);
        }
      }
    }
    double infeas_v, l1, linfty;
    if (sl1qpUpdate(step, z, zw, &infeas_v, &l1, &linfty)) return 1;
    if (infeas_v < opt.tr_infeas_tol && (l1 < opt.tr_l1_tol || linfty < opt.tr_linfty_tol)) {
      status = 1;
      break;
    }
    if (opt.tr_adaptive_gamma_update) {  // TR.cpp:1610-1668
      for (int j = 0; j < m; j++) {
        const double infeas_reduction = con_infeas[j] - model_con_infeas[j];
        const double best_reduction = con_infeas[j] - best_con_infeas[j];
        if (fabs(z[j]) > opt.tr_infeas_tol && con_infeas[j] < opt.tr_infeas_tol &&
            penalty_gamma[j] >= 2.0 * z[j]) {
          penalty_gamma[j] =
              std::max(0.5 * (penalty_gamma[j] + fabs(z[j])), opt.tr_penalty_gamma_min);
        } else if (con_infeas[j] > opt.tr_infeas_tol && 0.995 * best_reduction > infeas_reduction) {
          penalty_gamma[j] = std::min(1.5 * penalty_gamma[j], opt.tr_penalty_gamma_max);
        }
      }
      if (pcu_ip_set_penalty_gamma_array(ip, penalty_gamma.data())) return 1;
    }
  }
  return 0;
}

// -------------------------------------------------------------------- C ABI
namespace {
struct PendingOpt {
  std::string name;
  int type;  // 0 float, 1 int, 2 string
  double f;
  int i;
  std::string s;
};
std::vector<PendingOpt> &pending_of(pcu_tr *tr);
}  // namespace

struct pcu_tr_opts {
  std::vector<PendingOpt> list;
};
static std::vector<std::pair<pcu_tr *, pcu_tr_opts *> > g_tr_opts;
namespace {
std::vector<PendingOpt> &pending_of(pcu_tr *tr) {
  for (auto &p : g_tr_opts)
    if (p.first == tr) return p.second->list;
  g_tr_opts.push_back({tr, new pcu_tr_opts});
  return g_tr_opts.back().second->list;
}
}  // namespace

static int tr_apply_ip_options(pcu_tr *tr) {
  for (const PendingOpt &o : pending_of(tr)) {
    int rc;
    if (o.type == 0) rc = pcu_ip_set_option_float(tr->ip, o.name.c_str(), o.f);
    else if (o.type == 1) rc = pcu_ip_set_option_int(tr->ip, o.name.c_str(), o.i);
    else rc = pcu_ip_set_option_str(tr->ip, o.name.c_str(), o.s.c_str());
    (void)rc;  // names only the front end knows are not interior-point options
  }
  tr->opt.barrier_strategy = tr->ip->opt.barrier_strategy;
  tr->opt.starting_point_strategy = tr->ip->opt.starting_point_strategy;
  tr->opt.sequential_linear_method = tr->ip->opt.sequential_linear_method;
  return 0;
}

// ParOptInteriorPoint::setQuasiNewton for an object of this library (IP.cpp:1193)
int pcu_ip_set_quasi_newton_object(pcu_ip *ip, QuasiNewton *qn) {
  if (!ip->qn_external) delete ip->qn;
  ip->qn = qn;
  ip->qn_external = 1;
  ip->qn_built_size = -1;
  if (qn && (qn->n != ip->nvars || ip->ncon + qn->max_size() + 1 > PCU_MAX_COLS)) return 1;
  return 0;
}

extern "C" {

pcu_tr *pcu_tr_create(pcu_problem *prob) {
  if (!prob) return nullptr;
  pcu_tr *tr = new pcu_tr;
  tr->prob = prob;
  tr->ctx = prob->ctx;
  return tr;
}

void pcu_tr_destroy(pcu_tr *tr) {
  if (!tr) return;
  cudaStreamSynchronize(tr->ctx->stream);
  for (size_t i = 0; i < g_tr_opts.size(); i++) {
    if (g_tr_opts[i].first == tr) {
      delete g_tr_opts[i].second;
      g_tr_opts.erase(g_tr_opts.begin() + i);
      break;
    }
  }
  delete tr;
}

#define TR_OPT_F(n) if (k == #n) { tr->opt.n = value; known = 1; }
#define TR_OPT_I(n) if (k == #n) { tr->opt.n = value; known = 1; }
#define TR_OPT_S(n) if (k == #n) { tr->opt.n = value; known = 1; }

int pcu_tr_set_option_float(pcu_tr *tr, const char *name, double value) {
  const std::string k(name);
  int known = 0;
  TR_OPT_F(tr_init_size) TR_OPT_F(tr_min_size) TR_OPT_F(tr_max_size) TR_OPT_F(tr_eta)
  TR_OPT_F(tr_bound_relax) TR_OPT_F(function_precision) TR_OPT_F(tr_l1_tol)
  TR_OPT_F(tr_linfty_tol) TR_OPT_F(tr_infeas_tol) TR_OPT_F(tr_penalty_gamma_max)
  TR_OPT_F(tr_penalty_gamma_min) TR_OPT_F(penalty_gamma)
  pending_of(tr).push_back({k, 0, value, 0, ""});
  (void)known;
  return 0;
}
int pcu_tr_set_option_int(pcu_tr *tr, const char *name, int value) {
  const std::string k(name);
  int known = 0;
  TR_OPT_I(tr_adaptive_gamma_update) TR_OPT_I(tr_max_iterations)
  TR_OPT_I(tr_write_output_frequency) TR_OPT_I(output_level) TR_OPT_I(qn_subspace_size)
  if (k == "tr_use_soc" && value != 0) {
    fprintf(stderr, "paropt_b200: tr_use_soc is not built\n");
    return 1;
  }
  if (k == "use_diag_hessian" && value != 0) {
    fprintf(stderr, "ParOpt error: use_diag_hessian is not available in the trust region\n");
    return 1;
  }
  pending_of(tr).push_back({k, 1, 0.0, value, ""});
  (void)known;
  return 0;
}
int pcu_tr_set_option_str(pcu_tr *tr, const char *name, const char *value) {
  const std::string k(name);
  int known = 0;
  TR_OPT_S(tr_accept_step_strategy) TR_OPT_S(tr_adaptive_objective)
  TR_OPT_S(tr_adaptive_constraint) TR_OPT_S(tr_steering_barrier_strategy)
  TR_OPT_S(tr_steering_starting_point_strategy) TR_OPT_S(tr_output_file) TR_OPT_S(qn_type)
  TR_OPT_S(qn_update_type) TR_OPT_S(qn_diag_type)
  pending_of(tr).push_back({k, 2, 0.0, 0, value});
  (void)known;
  return 0;
}

int pcu_tr_optimize(pcu_tr *tr) {
  if (tr->build()) return 1;
  if (!tr->ip) {
    tr->ip = new pcu_ip;
    if (tr->ip->init(tr->sub)) return 1;
  }
  if (tr_apply_ip_options(tr)) return 1;
  return tr->optimize();
}

int pcu_tr_status(pcu_tr *tr) { return tr->status; }
int pcu_tr_history_len(pcu_tr *tr) { return (int)tr->history.size(); }
/* 19 doubles: iter fobj infeas l1 linfty smax tr rho model_red zav zmax gav gmax
   subproblem_iters adaptive_iters accepted xsum xnorm xmaxabs */
int pcu_tr_history_get(pcu_tr *tr, int k, double *out19) {
  if (k < 0 || k >= (int)tr->history.size()) return 1;
  const TrRecord &r = tr->history[k];
  memcpy(out19, r.f, sizeof(double) * 16);
  out19[16] = r.xsum;
  out19[17] = r.xnorm;
  out19[18] = r.xmaxabs;
  return 0;
}
const char *pcu_tr_history_info(pcu_tr *tr, int k) {
  if (k < 0 || k >= (int)tr->history.size()) return "";
  return tr->history[k].info.c_str();
}
/* getOptimizedPoint (TR.cpp:888-892): the centre x_k; the multipliers of the last
   subproblem solve come from the interior-point optimizer (ParOptOptimizer.cpp:240) */
pcu_vec *pcu_tr_point(pcu_tr *tr) { return tr->sub ? tr->sub->xk : nullptr; }
pcu_ip *pcu_tr_interior_point(pcu_tr *tr) { return tr->ip; }
int pcu_tr_penalty_gamma(pcu_tr *tr, double *gamma) {
  for (size_t i = 0; i < tr->penalty_gamma.size(); i++) gamma[i] = tr->penalty_gamma[i];
  return 0;
}

}  // extern "C"
