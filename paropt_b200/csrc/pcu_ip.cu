// pcu_ip.cu -- CUDA-resident interior-point core: host control flow of
// ParOptInteriorPoint::optimize (IP.cpp:4399-5333) driving the fused kernels of
// pcu_kernels.cuh / pcu_gram.cu.  All O(N) and O(W) work runs on the device; the
// host only handles the c- and q-sized dense algebra (as the reference does on
// its root rank) and the scalar control flow.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "pcu_ip.cuh"

int pcu_sr1_pairs_enqueue(pcu_ctx *ctx, const double *s, const double *const *S,
                          const double *const *Y, double *const *Z, int np, double b0,
                          long long n);
int pcu_mdot_enqueue(pcu_ctx *ctx, const double *x, const ColTable &cols,
                     int ncols, long long n, int dst_off);
int pcu_gram_enqueue(pcu_ctx *ctx, const ColTable &cols, int m,
                     const double *Dinv, const double *Cw, const WDesc &wd,
                     long long n, int *ld_out, const double *d2 = nullptr,
                     int rhs_col = -1);

#define launch_tile pcu_launch_tile

static const RedBuf NO_RED = {nullptr, nullptr, nullptr, 0};

// ============================================================== QuasiNewton
QuasiNewton::~QuasiNewton() {
  for (auto v : S) pcu_vec_destroy(v);
  for (auto v : Y) pcu_vec_destroy(v);
  for (auto v : Zs) pcu_vec_destroy(v);
  pcu_vec_destroy(r);
}

int QuasiNewton::init(pcu_ctx *c, int nvars, int kind, int m) {
  // The column tables of the kernels hold PCU_MAX_COLS entries: [S | Y] (+ the
  // damped update's extra column) for L-BFGS, Z for L-SR1.  Checked here, before
  // anything is allocated, so that pcu_qn_create and pcu_ip share one rule.
  const int width = kind == 0 ? 2 * m + 1 : m;
  if (m < 0 || width > PCU_MAX_COLS) {
    fprintf(stderr,
            "paropt_b200: quasi-Newton subspace %d too large (%s needs %d of %d columns)\n", m,
            kind == 0 ? "bfgs" : "sr1", width, PCU_MAX_COLS);
    return 1;
  }
  ctx = c;
  n = nvars;
  type = kind;
  msub_max = m;
  fused_sr1 = getenv("PCU_NO_FUSED_SR1") ? 0 : 1;
  for (int i = 0; i < m; i++) {
    S.push_back(pcu_vec_create(ctx, n));
    Y.push_back(pcu_vec_create(ctx, n));
    if (!S.back() || !Y.back()) return 1;
    if (type == 1) {
      Zs.push_back(pcu_vec_create(ctx, n));
      if (!Zs.back()) return 1;
    }
  }
  r = pcu_vec_create(ctx, n);
  if (!r) return 1;
  D.assign(m, 0.0);
  L.assign((size_t)m * m, 0.0);
  B.assign((size_t)m * m, 0.0);
  reset();
  return 0;
}

void QuasiNewton::reset() {  // QN.cpp:132-146, 608-622
  msub = 0;
  b0 = 1.0;
  std::fill(D.begin(), D.end(), 0.0);
  std::fill(L.begin(), L.end(), 0.0);
  std::fill(B.begin(), B.end(), 0.0);
  M.clear();
  Mf.clear();
  d0.clear();
  piv.clear();
}

void QuasiNewton::z_table(ColTable &t, int off) const {
  // (a caller may have looked at Z through pcu_qn_compact + pcu_vec_host_ptr)
  if (type == 0) {
    for (int i = 0; i < msub; i++) {
      pcu_vec_ready(S[i]);
      pcu_vec_ready(Y[i]);
      t.p[off + i] = S[i]->d;
      t.p[off + msub + i] = Y[i]->d;
    }
  } else {
    for (int i = 0; i < msub; i++) {
      pcu_vec_ready(Zs[i]);
      t.p[off + i] = Zs[i]->d;
    }
  }
}

void QuasiNewton::solve_compact(const double *rz, double *kap) const {
  const int q = size();
  for (int i = 0; i < q; i++) kap[i] = rz[i] * d0[i];
  if (q > 0) pcu_dense_lu_solve(q, Mf.data(), piv.data(), nullptr, kap);
  for (int i = 0; i < q; i++) kap[i] *= d0[i];
}

// y = b0 x - Z kap,  kap = d0 M^-1 d0 Z^T x    (QN.cpp:390-418, 760-778)
int QuasiNewton::mult(pcu_vec *x, pcu_vec *y) {
  const int q = size();
  LinCombF f;
  f.x = x->d;
  f.beta = b0;
  f.ncols = q;
  f.out = y->d;
  if (q > 0) {
    ColTable zt;
    z_table(zt, 0);
    if (pcu_mdot_enqueue(ctx, x->d, zt, q, n, 0)) return 1;
    std::vector<double> rz(q), kap(q);
    if (ctx->big_fetch(q, rz.data())) return 1;
    solve_compact(rz.data(), kap.data());
    f.V = zt;
    for (int i = 0; i < q; i++) f.alpha.v[i] = -kap[i];
  }
  WDesc w;
  memset(&w, 0, sizeof(w));
  return launch_tile(ctx, f, n, w, NO_RED);
}

void QuasiNewton::mat_update() {
  const int m = msub_max, ms = msub;
  if (type == 0) {  // computeMatUpdate QN.cpp:339-377
    const int q = 2 * ms;
    M.assign((size_t)q * q, 0.0);
    for (int i = 0; i < ms; i++)
      for (int j = 0; j < ms; j++) M[i + (size_t)q * j] = b0 * B[i + (size_t)m * j];
    for (int i = 0; i < ms; i++)
      for (int j = 0; j < i; j++) {
        M[i + (size_t)q * (j + ms)] = L[i + (size_t)m * j];
        M[j + ms + (size_t)q * i] = L[i + (size_t)m * j];
      }
    for (int i = 0; i < ms; i++) M[ms + i + (size_t)q * (ms + i)] = -D[i];
    d0.assign(q, 1.0);
    for (int i = 0; i < ms; i++) d0[i] = b0;
  } else {  // QN.cpp:702-737
    const int q = ms;
    M.assign((size_t)q * q, 0.0);
    for (int i = 0; i < ms; i++)
      for (int j = 0; j < ms; j++) M[i + (size_t)q * j] += b0 * B[i + (size_t)m * j];
    for (int i = 0; i < ms; i++)
      for (int j = 0; j < i; j++) {
        M[i + (size_t)q * j] -= L[i + (size_t)m * j];
        M[j + (size_t)q * i] -= L[i + (size_t)m * j];
      }
    for (int i = 0; i < ms; i++) M[i * (size_t)(q + 1)] -= D[i];
    d0.assign(q, 1.0);
  }
  Mf = M;
  piv.assign(size() > 0 ? size() : 1, 0.0);
  std::vector<double> invd(piv.size());  // (read by the device's solves only)
  if (size() > 0) pcu_dense_lu_factor(size(), Mf.data(), piv.data(), invd.data());
}

// ParOptLBFGS::update (QN.cpp:162-334) / ParOptLSR1::update (QN.cpp:636-747).
// One multi-dot pass gives s.S_i and s.Y_i for every stored pair: it provides
// both Z^T s (for s^T B s) and the new rows of S^T S and L.
// steal: the caller does not need the contents of s and y afterwards (the optimizer's
// own s_qn / y_qn): the new pair is stored by exchanging buffers with the slot it
// replaces instead of two N-sized copies (4 N words per iteration).
static int qn_store(pcu_vec *slot, pcu_vec *src, int steal) {
  return steal ? pcu_vec_take(slot, src) : pcu_vec_copy(slot, src);
}

int QuasiNewton::update(pcu_vec *s, pcu_vec *y, double yTy, double yTs,
                        double sTs, const double *sZ, int *update_type, int steal) {
  *update_type = 0;
  const int m = msub_max;
  std::vector<double> sS(msub), sY(msub);
  auto stored_dots = [&]() -> int {
    if (msub == 0) return 0;
    if (sZ && type == 0) {  // supplied by the caller (Z = [S | Y])
      for (int i = 0; i < msub; i++) {
        sS[i] = sZ[i];
        sY[i] = sZ[msub + i];
      }
      return 0;
    }
    ColTable t;
    for (int i = 0; i < msub; i++) {
      pcu_vec_ready(S[i]);
      pcu_vec_ready(Y[i]);
      t.p[i] = S[i]->d;
      t.p[msub + i] = Y[i]->d;
    }
    if (pcu_mdot_enqueue(ctx, s->d, t, 2 * msub, n, 0)) return 1;
    std::vector<double> out(2 * msub);
    if (ctx->big_fetch(2 * msub, out.data())) return 1;
    for (int i = 0; i < msub; i++) {
      sS[i] = out[i];
      sY[i] = out[msub + i];
    }
    return 0;
  };
  pcu_vec *y_update = y;
  if (type == 0) {
    if (1e-8 * yTy >= fabs(yTs)) {  // QN.cpp:175-179
      *update_type = 2;
      return 0;
    }
    if (stored_dots()) return 1;
    // s^T B s = b0 s.s - (Z^T s)^T d0 M^-1 d0 (Z^T s)   (QN.cpp:183-186)
    double sTBs = b0 * sTs;
    const int q = size();
    std::vector<double> rz(q), kap(q);
    if (q > 0) {
      for (int i = 0; i < msub; i++) {
        rz[i] = sS[i];
        rz[msub + i] = sY[i];
      }
      solve_compact(rz.data(), kap.data());
      for (int i = 0; i < q; i++) sTBs -= kap[i] * rz[i];
    }
    double b0_init;
    if (yTs >= eps) {
      b0_init = diag_yts_over_sts ? yTs / sTs : yTy / yTs;
    } else {
      b0_init = 0.5 * (fabs(yTy / yTs) + fabs(yTs / sTs));
    }
    if (yTs >= 0.01 * sTBs) {
      b0 = b0_init;
    } else if (!damped) {
      *update_type = 2;  // skipped (QN.cpp:226-228)
      return 0;
    } else {
      // damped update (QN.cpp:238-263): r = theta*y + (1-theta)*B*s
      *update_type = 1;
      const double theta = 0.8 * sTBs / (sTBs - yTs);
      LinCombF f;
      f.x = s->d;
      f.beta = (1.0 - theta) * b0;
      f.ncols = q + 1;
      f.out = r->d;
      z_table(f.V, 0);
      for (int i = 0; i < q; i++) f.alpha.v[i] = -(1.0 - theta) * kap[i];
      f.V.p[q] = y->d;
      f.alpha.v[q] = theta;
      WDesc w;
      memset(&w, 0, sizeof(w));
      if (launch_tile(ctx, f, n, w, NO_RED)) return 1;
      y_update = r;
      double d;
      if (pcu_vec_dot(r, r, &yTy)) return 1;
      if (pcu_vec_dot(s, r, &d)) return 1;
      yTs = d;
      b0 = diag_yts_over_sts ? yTs / sTs : yTy / yTs;
      // dots of s with stored Y are unchanged; the new pair uses y_update
    }
  } else {
    // L-SR1: the dots with the stored pairs are taken by the sweep that rebuilds Z
    // (after the new pair is in place); b0 needs the two scalars only
    if (fused_sr1 == 0 && stored_dots()) return 1;
    b0 = (yTs > eps * yTy) ? yTy / yTs : 1.0;  // QN.cpp:645-649
  }

  // store the pair (pointer rotation instead of copies where possible)
  int shift = 0;
  if (msub < m) {
    if (qn_store(S[msub], s, steal) || qn_store(Y[msub], y_update, steal)) return 1;
    msub++;
  } else if (m > 0) {
    if (qn_store(S[0], s, steal) || qn_store(Y[0], y_update, steal)) return 1;
    std::rotate(S.begin(), S.begin() + 1, S.end());
    std::rotate(Y.begin(), Y.begin() + 1, Y.end());
    for (int i = 0; i < msub - 1; i++) D[i] = D[i + 1];
    for (int i = 0; i < msub - 1; i++)
      for (int j = 0; j < msub - 1; j++)
        B[i + (size_t)m * j] = B[i + 1 + (size_t)m * (j + 1)];
    for (int i = 0; i < msub - 1; i++)
      for (int j = 0; j < i; j++)
        L[i + (size_t)m * j] = L[i + 1 + (size_t)m * (j + 1)];
    shift = 1;
  } else {
    return 0;
  }
  const int last = msub - 1;
  if (type == 1 && fused_sr1) {
    // one sweep over the pairs as they are stored now: Z_i = Y_i - b0 S_i (QN.cpp:730-735)
    // together with s . S_i and s . Y_i (s = S[last], the pair just stored)
    std::vector<const double *> Sp(msub), Yp(msub);
    std::vector<double *> Zp(msub);
    for (int i = 0; i < msub; i++) {
      pcu_vec_ready(S[i]);
      pcu_vec_ready(Y[i]);
      pcu_vec_ready(Zs[i]);
      Sp[i] = S[i]->d;
      Yp[i] = Y[i]->d;
      Zp[i] = Zs[i]->d;
    }
    if (pcu_sr1_pairs_enqueue(ctx, S[last]->d, Sp.data(), Yp.data(), Zp.data(), msub, b0, n))
      return 1;
    std::vector<double> out(2 * (size_t)msub);
    if (ctx->big_fetch(2 * (size_t)msub, out.data())) return 1;
    sS.assign(msub + 1, 0.0);
    sY.assign(msub + 1, 0.0);
    for (int i = 0; i < last; i++) {
      sS[i + shift] = out[i];
      sY[i + shift] = out[msub + i];
    }
  }
  for (int i = 0; i < last; i++) {  // QN.cpp:307-321
    B[last + (size_t)m * i] = sS[i + shift];
    B[i + (size_t)m * last] = sS[i + shift];
    L[last + (size_t)m * i] = sY[i + shift];
  }
  B[last + (size_t)m * last] = sTs;
  D[last] = yTs;
  mat_update();
  if (type == 1 && !fused_sr1) {  // Z_i = Y_i - b0 S_i  (QN.cpp:730-735)
    for (int i = 0; i < msub; i++) {
      LinCombF f;
      f.x = Y[i]->d;
      f.beta = 1.0;
      f.ncols = 1;
      f.V.p[0] = S[i]->d;
      f.alpha.v[0] = -b0;
      f.out = Zs[i]->d;
      WDesc w;
      memset(&w, 0, sizeof(w));
      if (launch_tile(ctx, f, n, w, NO_RED)) return 1;
    }
  }
  return 0;
}

// ==================================================================== pcu_ip
pcu_ip::~pcu_ip() {
  Vars *all[4] = {&variables, &residual, &update, &refine};
  for (auto vs : all)
    for (int i = 0; i < 8; i++) pcu_vec_destroy(vs->v[i]);
  pcu_vec *single[] = {lb, ub, g, Dinv, Cw, d1, d2, t1, s_qn, y_qn, rx, rsw, rtw, rzl, rzu, rzw,
                       rzsw, rztw, gaz, apz1, apz2, hdiag};
  for (auto v : single) pcu_vec_destroy(v);
  for (auto v : Ac) pcu_vec_destroy(v);
  for (auto v : gmres_W) pcu_vec_destroy(v);
  if (!qn_external) delete qn;
  if (dense_dev) cudaFree(dense_dev);
  if (dense_host) cudaFreeHost(dense_host);
  if (outfp && outfp != stdout) fclose(outfp);
  for (IterEvents &e : evs) {
    cudaEvent_t all[4] = {e.it0, e.it1, e.k0, e.k1};
    for (cudaEvent_t ev : all)
      if (ev) cudaEventDestroy(ev);
    for (auto &c : e.cb) {
      cudaEventDestroy(c.first);
      cudaEventDestroy(c.second);
    }
  }
}

int pcu_ip::init(pcu_problem *p) {  // constructor, IP.cpp:182-438
  prob = p;
  ctx = p->ctx;
  nvars = p->nvars;
  ncon = p->ncon;
  nwcon = p->nwcon;
  if (ncon < 0 || ncon > PCU_MAX_COLS - 1) {
    fprintf(stderr, "paropt_b200: %d dense constraints exceed the %d columns of the kernels\n",
            ncon, PCU_MAX_COLS - 1);
    return 1;
  }
  if (pcu_validate_weighting(&p->weighting, nvars, ncon, p->ninequality, p->nwinequality,
                             "pcu_ip_create"))
    return 1;
  wd = pcu_make_wdesc(p->weighting, nvars);
  if (getenv("PCU_NO_FUSE21")) opt_no_fuse21 = 1;
  if (getenv("PCU_NO_WIDE")) opt_no_wide = 1;
  if (getenv("PCU_NO_FUSE2S")) opt_no_fuse2s = 1;
  if (getenv("PCU_NO_RHSGRAM")) opt_no_rhsgram = 1;
  if (getenv("PCU_NO_CHAIN")) opt_no_chain = 1;
  if (getenv("PCU_CHAIN")) opt_force_chain = 1;
  if (getenv("PCU_NO_UPDSTATS")) opt_no_updstats = 1;
  if (getenv("PCU_NO_TRIALUPD")) opt_no_trialupd = 1;
  if (getenv("PCU_NO_GAZ")) opt_no_gaz = 1;
  Vars *all[4] = {&variables, &residual, &update, &refine};
  for (auto vs : all) {
    for (int i = 0; i < 8; i++) {
      vs->v[i] = pcu_vec_create(ctx, i < 3 ? nvars : nwcon);
      if (!vs->v[i]) return 1;
    }
    vs->z.assign(ncon, 0.0);
    vs->s.assign(ncon, 0.0);
    vs->t.assign(ncon, 0.0);
    vs->zs.assign(ncon, 0.0);
    vs->zt.assign(ncon, 0.0);
  }
  pcu_vec **nvecs[] = {&lb, &ub, &g, &Dinv, &d1, &t1, &s_qn, &y_qn, &rx};
  for (auto pv : nvecs) {
    *pv = pcu_vec_create(ctx, nvars);
    if (!*pv) return 1;
  }
  pcu_vec **wvecs[] = {&Cw, &d2, &rsw, &rtw};
  for (auto pv : wvecs) {
    *pv = pcu_vec_create(ctx, nwcon);
    if (!*pv) return 1;
  }
  for (int i = 0; i < ncon; i++) {
    Ac.push_back(pcu_vec_create(ctx, nvars));
    if (!Ac.back()) return 1;
  }
  c.assign(ncon, 0.0);
  if (ctx->big_reserve((size_t)PCU_MAX_COLS * PCU_MAX_COLS + 64,
                       (size_t)PCU_MAX_BLOCKS * 64 * 15))
    return 1;
  for (IterEvents &e : evs) {
    PCU_CUDA_OK(cudaEventCreate(&e.it0));
    PCU_CUDA_OK(cudaEventCreate(&e.it1));
    PCU_CUDA_OK(cudaEventCreate(&e.k0));
    PCU_CUDA_OK(cudaEventCreate(&e.k1));
  }
  barrier_param = opt.init_barrier_param;
  rho_penalty_search = opt.init_rho_penalty_search;
  if (initAndCheckDesignAndBounds()) return 1;
  // initial multipliers and slacks all 1 (IP.cpp:417-437)
  for (int i = 1; i < 8; i++)
    if (pcu_vec_set(variables.v[i], 1.0)) return 1;
  for (int i = 0; i < ncon; i++)
    variables.z[i] = variables.s[i] = variables.t[i] = variables.zs[i] =
        variables.zt[i] = 1.0;
  return 0;
}

IPConst pcu_ip::kconst() const {
  IPConst k;
  k.mbv = opt.max_bound_value;
  k.kappa = opt.rel_bound_barrier;
  k.gamma = opt.penalty_gamma;
  k.dp = opt.design_precision;
  k.wconst = wd.wconst;
  k.wc = prob->wconst_vec ? prob->wconst_vec->d : nullptr;
  k.use_lower = prob->use_lower;
  k.use_upper = prob->use_upper;
  k.nwineq = prob->nwinequality;
  return k;
}

int pcu_ip::norm_type_id() const {
  if (opt.norm_type == "infinity") return 0;
  if (opt.norm_type == "l1") return 1;
  return 2;
}

int pcu_ip::ensure_qn() {  // IP.cpp:263-290
  if (qn_external) return qn ? 0 : 1;  // supplied through pcu_ip_set_quasi_newton
  if (opt.use_diag_hessian) {  // the problem's diagonal is the Hessian: no quasi-Newton object
    if (qn) delete qn;
    qn = nullptr;
    qn_built_type.clear();
    qn_built_size = -1;
    return 0;
  }
  if (qn && qn_built_type == opt.qn_type && qn_built_size == opt.qn_subspace_size) {
    qn->damped = (opt.qn_update_type == "damped_update");
    qn->diag_yts_over_sts = (opt.qn_diag_type == "yts_over_sts");
    return 0;
  }
  if (!qn_external) delete qn;
  qn = nullptr;
  qn_built_type.clear();
  qn_built_size = -1;
  int kind = -1;
  if (opt.qn_type == "bfgs") kind = 0;
  else if (opt.qn_type == "sr1") kind = 1;
  if (kind < 0) {  // "none": no quasi-Newton object (IP.cpp:263-277)
    qn_built_type = opt.qn_type;
    qn_built_size = opt.qn_subspace_size;
    return 0;
  }
  // validate the width BEFORE allocating: a failed attempt leaves nothing cached
  const int m = opt.qn_subspace_size;
  const int width = kind == 0 ? 2 * m : m;
  if (m < 0 || ncon + width + 1 > PCU_MAX_COLS) {
    fprintf(stderr, "paropt_b200: ncon + quasi-Newton width (%d + %d) exceeds %d columns\n",
            ncon, width, PCU_MAX_COLS - 1);
    return 1;
  }
  QuasiNewton *fresh = new QuasiNewton;
  if (fresh->init(ctx, nvars, kind, m)) {
    delete fresh;
    return 1;
  }
  qn = fresh;
  qn_built_type = opt.qn_type;
  qn_built_size = opt.qn_subspace_size;
  qn->damped = (opt.qn_update_type == "damped_update");
  qn->diag_yts_over_sts = (opt.qn_diag_type == "yts_over_sts");
  return 0;
}

void pcu_ip::refresh_penalties() {  // IP.cpp:343-355, setPenaltyGamma IP.cpp:1128-1173
  if (gamma_custom && (int)gamma_t.size() == ncon) return;  // per-constraint values were set
  gamma_s.assign(ncon, opt.penalty_gamma);
  gamma_t.assign(ncon, opt.penalty_gamma);
  for (int i = 0; i < ncon && i < prob->ninequality; i++) gamma_s[i] = 0.0;
}

// ------------------------------------------------------------- callbacks
int pcu_ip::cb_begin() {
  IterEvents &e = evs[ev_cur];
  if (e.cb_used == e.cb.size()) {
    cudaEvent_t a, b;
    PCU_CUDA_OK(cudaEventCreate(&a));
    PCU_CUDA_OK(cudaEventCreate(&b));
    e.cb.push_back({a, b});
  }
  PCU_CUDA_OK(cudaEventRecord(e.cb[e.cb_used].first, ctx->stream));
  return 0;
}
int pcu_ip::cb_end() {
  IterEvents &e = evs[ev_cur];
  PCU_CUDA_OK(cudaEventRecord(e.cb[e.cb_used].second, ctx->stream));
  e.cb_used++;
  return 0;
}
double pcu_ip::cb_collect() {  // callbacks of the current event set (after a synchronisation)
  IterEvents &e = evs[ev_cur];
  double ms = 0.0;
  for (size_t i = 0; i < e.cb_used; i++) {
    float f = 0.f;
    if (cudaEventSynchronize(e.cb[i].second) == cudaSuccess &&
        cudaEventElapsedTime(&f, e.cb[i].first, e.cb[i].second) == cudaSuccess)
      ms += f;
  }
  e.cb_used = 0;
  prob->callback_ms += ms;
  return ms;
}
// One finished iteration: total / KKT-solve / callback milliseconds into `times`.
int pcu_ip::collect_times(IterEvents &e) {
  if (!e.pending) return 0;
  e.pending = false;
  PCU_CUDA_OK(cudaEventSynchronize(e.it1));
  IterTime tm;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e.it0, e.it1);
  tm.total_ms = ms;
  ms = 0.f;
  cudaEventElapsedTime(&ms, e.k0, e.k1);
  tm.kkt_ms = ms;
  double cb = 0.0;
  for (size_t i = 0; i < e.cb_used; i++) {
    float f = 0.f;
    if (cudaEventElapsedTime(&f, e.cb[i].first, e.cb[i].second) == cudaSuccess) cb += f;
  }
  e.cb_used = 0;
  prob->callback_ms += cb;
  tm.callback_ms = cb;
  times.push_back(tm);
  return 0;
}
int pcu_ip::flush_times() {
  // oldest first: the set that is not current was recorded before the current one
  if (collect_times(evs[ev_cur ^ 1])) return 1;
  return collect_times(evs[ev_cur]);
}
int pcu_ip::evalObjCon(pcu_vec *x) {
  if (cb_begin()) return 1;
  int fail = prob->evalObjCon(x, &fobj, c.data());
  neval++;
  if (cb_end()) return 1;
  return fail;
}
int pcu_ip::evalObjConGradient(pcu_vec *x, int same_point) {
  if (cb_begin()) return 1;
  prob->same_point_hint = same_point;
  gaz_valid = 0;
  int fail = prob->evalObjConGradient(x, g, Ac.data());
  ngeval++;
  // use_diag_hessian: the diagonal at the point the gradient callback just saw, with
  // that point's multipliers; a failure counts as a failed gradient evaluation
  if (!fail && opt.use_diag_hessian) {
    prob->same_point_hint = 1;
    fail = prob->evalHessianDiag(x, variables.z.data(), variables.v[PCU_ZW], hdiag);
  }
  prob->same_point_hint = 0;
  if (cb_end()) return 1;
  return fail;
}

// ---------------------------------------------- initAndCheckDesignAndBounds
// IP.cpp:4277-4361
struct BoundsF : NoStreams {
  static constexpr int NS = 0, NX = 3, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  double *x, *lb, *ub, *zl, *zu;
  double rel_bound, mbv;
  int both;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *acc) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &,
                                    AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W],
                                    const Elem (&)[W], const Con &,
                                    AccT &acc) const {
    double xv[W], l[W], u[W], a[W], b[W];
    ldv<W>(x, i, xv);
    ldv<W>(lb, i, l);
    ldv<W>(ub, i, u);
    ldv<W>(zl, i, a);
    ldv<W>(zu, i, b);
#pragma unroll
    for (int e = 0; e < W; e++) {
      if (both) {
        double delta = 1.0;
        if (l[e] > -mbv && u[e] < mbv) {
          if (l[e] >= u[e]) {
            acc.x[0] = 1.0;
            l[e] = 0.5 * (l[e] + u[e]) - 0.5 * rel_bound;
            u[e] = l[e] + rel_bound;
          }
          delta = u[e] - l[e];
        }
        if (l[e] > -mbv && xv[e] < l[e] + rel_bound * delta) {
          acc.x[1] = 1.0;
          xv[e] = l[e] + rel_bound * delta;
        }
        if (u[e] < mbv && xv[e] > u[e] - rel_bound * delta) {
          acc.x[2] = 1.0;
          xv[e] = u[e] - rel_bound * delta;
        }
      }
      if (l[e] <= -mbv) a[e] = 0.0;
      if (u[e] >= mbv) b[e] = 0.0;
    }
    stv<W>(x, i, xv);
    stv<W>(lb, i, l);
    stv<W>(ub, i, u);
    stv<W>(zl, i, a);
    stv<W>(zu, i, b);
  }
};

int pcu_ip::initAndCheckDesignAndBounds() {
  if (prob->getVarsAndBounds(variables.v[PCU_X], lb, ub)) return 1;
  BoundsF f;
  f.x = variables.v[PCU_X]->d;
  f.lb = lb->d;
  f.ub = ub->d;
  f.zl = variables.v[PCU_ZL]->d;
  f.zu = variables.v[PCU_ZU]->d;
  f.rel_bound = 0.001 * barrier_param;
  f.mbv = opt.max_bound_value;
  f.both = prob->use_lower && prob->use_upper;
  WDesc w;
  memset(&w, 0, sizeof(w));
  RedBuf rb = ctx->redbuf(0, 3, 0);
  if (launch_tile(ctx, f, nvars, w, rb)) return 1;
  double flags[3];
  if (ctx->fetch(flags)) return 1;
  if (outfp && ctx->rank == 0) {
    if (flags[0] > 0.0)
      fprintf(outfp, "ParOpt Warning: Variable bounds are inconsistent\n");
    if (flags[1] > 0.0)
      fprintf(outfp, "ParOpt Warning: Variables may be too close to lower bound\n");
    if (flags[2] > 0.0)
      fprintf(outfp, "ParOpt Warning: Variables may be too close to upper bound\n");
  }
  return 0;
}

// A p_z hand-over from the pass-2 kernels to the update pass (pcu_ip.cuh)
double *pcu_ip::apz_target(int accumulate, bool supported) {
  if (ncon < 3 || opt_no_gaz) return nullptr;
  if (!accumulate) apz_state = 0;
  const int slot = !accumulate ? 1 : (apz_state == 1 ? 2 : 0);
  if (!supported || slot == 0) {
    if (accumulate) apz_state = -1;  // a contribution to the step nobody recorded
    return nullptr;
  }
  pcu_vec *&v = slot == 1 ? apz1 : apz2;
  if (!v) v = pcu_vec_create(ctx, nvars);
  if (!v) {
    apz_state = -1;
    return nullptr;
  }
  return v->d;
}
void pcu_ip::apz_done(int accumulate, double *target) {
  if (target) apz_state = accumulate ? 3 : 1;
}

// --------------------------------------------------------------- residuals
// use_diag_hessian: the Hessian term of addKKTResStep, rx -= h p_x (IP.cpp:1464), after
// ResF has formed the rest of the row, with the norms of rx taken again (ResF's sums 3 and
// maximum 0).  Only the stand-alone residual of a step reaches it (pcu_ip_add_kkt_res_step):
// the optimizer's route with this option refines in the column space of [A|Z].
// Traffic: reads 3N, writes N.
struct HessDiagResF : NoStreams {
  static constexpr int NS = 2, NX = 1, NM = 0, NB = 0;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  const double *h, *px;
  double *rx;
  template <int W>
  __device__ __forceinline__ void A(long long, const double (&)[W], Elem (&)[W],
                                    double (&)[W][1], AccT *) const {}
  __device__ __forceinline__ void B(long long, const double (&)[1], Con &, AccT &) const {}
  template <int W>
  __device__ __forceinline__ void C(long long i, const double (&)[W], const Elem (&)[W],
                                    const Con &, AccT &acc) const {
    double hv[W], p[W], r[W];
    ldv<W>(h, i, hv);
    ldv<W>(px, i, p);
    ldv<W>(rx, i, r);
#pragma unroll
    for (int q = 0; q < W; q++) {
      r[q] = fma(-hv[q], p[q], r[q]);
      acc.x[0] = fmax(acc.x[0], fabs(r[q]));
      acc.s[0] += fabs(r[q]);
      acc.s[1] = fma(r[q], r[q], acc.s[1]);
    }
    stv<W>(rx, i, r);
  }
};

int pcu_ip::computeKKTRes(Vars &vars, double mu, Vars &res, Vars *step,
                          const double *ATp, const double *ZTp, int store) {
  ResF f;
  f.store = store;
  f.v = vars.dv();
  f.r = res.dv();
  f.p = step ? step->dv() : vars.dv();
  f.lb = lb->d;
  f.ub = ub->d;
  f.g = g->d;
  f.ncon = ncon;
  for (int j = 0; j < ncon; j++) {
    f.Acol.p[j] = Ac[j]->d;
    f.z.v[j] = vars.z[j] + (step ? step->z[j] : 0.0);
  }
  f.nq = 0;
  f.b0sig = 0.0;
  f.has_step = step ? 1 : 0;
  if (step) {
    f.b0sig = res_skip_hessian ? 0.0 : opt.qn_sigma;
    if (qn && !opt.sequential_linear_method && !res_skip_hessian) {  // IP.cpp:1474-1476
      f.b0sig += qn->b0;
      f.nq = qn->size();
      if (f.nq > 0) {
        qn->z_table(f.Z, 0);
        std::vector<double> kap(f.nq);
        qn->solve_compact(ZTp, kap.data());
        for (int i = 0; i < f.nq; i++) f.kap.v[i] = kap[i];
      }
    }
  }
  f.mu = mu;
  f.norm_type = norm_type_id();
  f.k = kconst();
  RedBuf rb = ctx->redbuf(ResF::NS, ResF::NX, ResF::NM);
  if (!f.has_step && f.norm_type == 0) {
    // the per-iteration launch: step terms and l1 / l2 bookkeeping compiled out
    typedef ResFT<0, 0> Fast;
    static_assert(sizeof(Fast) == sizeof(ResF), "same layout");
    Fast ff;
    memcpy((void *)&ff, (const void *)&f, sizeof(ff));
    if (launch_tile(ctx, ff, nvars, wd, rb)) return 1;
  } else if (launch_tile(ctx, f, nvars, wd, rb)) {
    return 1;
  }
  double out[ResF::NS + ResF::NX + ResF::NM];
  if (ctx->fetch(out)) return 1;
  memcpy(res_sums, out, sizeof(res_sums));
  memcpy(res_max, out + ResF::NS, sizeof(res_max));
  memcpy(res_min, out + ResF::NS + ResF::NX, sizeof(res_min));
  if (step && opt.use_diag_hessian && !res_skip_hessian) {
    if (!store) return 1;
    HessDiagResF fh;
    fh.h = hdiag->d;
    fh.px = step->v[PCU_X]->d;
    fh.rx = res.v[PCU_X]->d;
    WDesc w0;
    memset(&w0, 0, sizeof(w0));
    RedBuf rbh = ctx->redbuf(HessDiagResF::NS, HessDiagResF::NX, 0);
    if (launch_tile(ctx, fh, nvars, w0, rbh)) return 1;
    double oh[3];
    if (ctx->fetch(oh)) return 1;
    res_max[0] = oh[2];
    if (f.norm_type == 1) res_sums[3] = oh[0];
    else if (f.norm_type == 2) res_sums[3] = oh[1];
  }
  res_mu = mu;
  res_has_step = step ? 1 : 0;
  denseResidual(vars, mu, res, step, ATp);
  return 0;
}

// dense parts of computeKKTRes / addKKTResStep (IP.cpp:1401-1407, 1535-1541)
void pcu_ip::denseResidual(Vars &vars, double mu, Vars &res, Vars *step,
                           const double *ATp) {
  for (int i = 0; i < ncon; i++) {
    res.z[i] = -(c[i] - vars.s[i] + vars.t[i]);
    res.s[i] = -(gamma_s[i] - vars.zs[i] + vars.z[i]);
    res.t[i] = -(gamma_t[i] - vars.zt[i] - vars.z[i]);
    res.zs[i] = -(vars.s[i] * vars.zs[i] - mu);
    res.zt[i] = -(vars.t[i] * vars.zt[i] - mu);
    if (step) {
      res.z[i] -= (ATp[i] - step->s[i] + step->t[i]);
      res.s[i] += (step->zs[i] - step->z[i]);
      res.t[i] += (step->zt[i] + step->z[i]);
      res.zs[i] -= (step->s[i] * vars.zs[i] + vars.s[i] * step->zs[i]);
      res.zt[i] -= (step->t[i] * vars.zt[i] + vars.t[i] * step->zt[i]);
    }
  }
}

// computeResNorm (IP.cpp:1588-1723) from the statistics of the last ResF launch
void pcu_ip::computeResNorm(Vars &res, double *max_prime, double *max_dual,
                            double *max_infeas, double *res_norm) {
  const int nt = norm_type_id();
  double mp = 0.0, md = 0.0, mi = 0.0;
  if (nt == 0) {
    mp = res_max[0];
    mi = res_max[1];
    md = res_max[2];
    if (!res_has_step) {
      // |kappa mu - a_i| over the bound products, |mu - a_i| over the sparse ones
      const double km = opt.rel_bound_barrier * res_mu;
      if (res_min[0] < 1e299)
        md = std::max(md, std::max(fabs(km - res_max[3]), fabs(km - res_min[0])));
      if (res_min[1] < 1e299)
        md = std::max(md, std::max(fabs(res_mu - res_max[4]), fabs(res_mu - res_min[1])));
    }
    for (int i = 0; i < ncon; i++) {
      mp = std::max(mp, std::max(fabs(res.s[i]), fabs(res.t[i])));
      mi = std::max(mi, fabs(res.z[i]));
      md = std::max(md, std::max(fabs(res.zs[i]), fabs(res.zt[i])));
    }
  } else if (nt == 1) {
    mp = res_sums[3];
    mi = res_sums[4];
    md = res_sums[5] + res_sums[6] + res_sums[7] + res_sums[8];
    for (int i = 0; i < ncon; i++) {
      mp += fabs(res.s[i]) + fabs(res.t[i]);
      mi += fabs(res.z[i]);
      md += fabs(res.zs[i]) + fabs(res.zt[i]);
    }
    md += res_sums[9] + res_sums[10];
  } else {
    mp = res_sums[3];
    mi = res_sums[4];
    // the reference squares l1 norms of the sparse dual parts (IP.cpp:1631-1636)
    md = res_sums[5] * res_sums[5] + res_sums[6] * res_sums[6] +
         res_sums[7] * res_sums[7] + res_sums[8] * res_sums[8];
    for (int i = 0; i < ncon; i++) {
      mp += res.s[i] * res.s[i] + res.t[i] * res.t[i];
      mi += res.z[i] * res.z[i];
      md += res.zs[i] * res.zs[i] + res.zt[i] * res.zt[i];
    }
    md += res_sums[9] + res_sums[10];
    mp = sqrt(mp);
    mi = sqrt(mi);
    md = sqrt(md);
  }
  *max_prime = mp;
  *max_dual = md;
  *max_infeas = mi;
  if (res_norm) *res_norm = std::max(mp, std::max(md, mi));
}

int pcu_ip::resNormAtBarrier(Vars &vars, double mu, Vars &res, double *max_prime,
                             double *max_dual, double *max_infeas,
                             double *res_norm) {
  if (norm_type_id() != 0 || res_has_step) return 0;
  res_mu = mu;
  denseResidual(vars, mu, res, nullptr, nullptr);
  computeResNorm(res, max_prime, max_dual, max_infeas, res_norm);
  return 1;
}

// computeComp (IP.cpp:2742-2820) from the statistics of the last ResF launch
double pcu_ip::compFromStats(Vars &vars) {
  double product = res_sums[0] / opt.rel_bound_barrier + res_sums[2];
  double count = res_sums[1];  // bounds present + 2 per sparse constraint
  for (int i = 0; i < ncon; i++) {
    product += vars.s[i] * vars.zs[i] + vars.t[i] * vars.zt[i];
    count += 2.0;
  }
  return count != 0.0 ? product / count : 0.0;
}
