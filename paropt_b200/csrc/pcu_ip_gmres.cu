// pcu_ip_gmres.cu -- the inexact-Newton step of the interior-point core:
// ParOptInteriorPoint::computeKKTGMRESStep (IP.cpp:5789-6191) with the alpha-scaled
// diagonal solve (IP.cpp:2441-2614) and evalObjBarrierDeriv (IP.cpp:5669-5772).
//
// Right-preconditioned GMRES on K M^-1 u = b: K has the problem's exact Hessian
// (evalHvecProduct), M is the quasi-Newton KKT matrix the rest of the optimizer solves
// with.  Only the x block of a Krylov vector is a vector (gmres_W); the other blocks are
// the right-hand side times a scalar alpha_i / |b|, which is why the preconditioner
// solve takes a scale factor for those parts (`bs` of Pass1F / Pass2F).
//
// One GMRES iteration on the device:
//   Pass1F(bs)            d1, d2, t1 = D0^-1 (d1, d2)|x                  9N + 11W
//   multi-dot             r = [A|Z]^T t1                                 (m + m/8) N
//   Pass2F(bs)            the diagonal solve (every block)               (12 + c) N + 15W
//   Pass2F(bs)            x block with the Sherman-Morrison-Woodbury
//                         correction (needs no second reduction:
//                         A^T D0^-1 Z w = S_AZ w from the Gram matrix)   (12 + m) N + 15W
//   StatsF, SparseProjF   the sums of evalObjBarrierDeriv and of the
//                         constraint-infeasibility projections           11N + 12W
//   callback, B p, Gram-Schmidt: the problem's Hessian-vector product, one compact
//                         quasi-Newton product, i + 2 dots and axpys.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "pcu_ip.cuh"

int pcu_mdot_enqueue(pcu_ctx *ctx, const double *x, const ColTable &cols,
                     int ncols, long long n, int dst_off);

#define launch_tile pcu_launch_tile
static const RedBuf NO_RED = {nullptr, nullptr, nullptr, 0};

// rho = cw(x) - sw + tw against a step: sums rho.(Aw px), rho.psw, rho.ptw
// (the sparse part of aproj / cpr, IP.cpp:5957-5966, 6160-6172)
struct SparseProjF : NoStreams {
  static constexpr int NS = 3, NX = 0, NM = 0, NB = 2;
  typedef Acc<NS, NX, NM> AccT;
  typedef Con0 Con;
  struct Elem {};
  DVars v, p;
  IPConst k;
  template <int W>
  __device__ __forceinline__ void A(long long i, const double (&coef)[W], Elem (&)[W],
                                    double (&part)[W][2], AccT *) const {
    double x[W], px[W];
    ldv<W>(v.x, i, x);
    ldv<W>(p.x, i, px);
#pragma unroll
    for (int q = 0; q < W; q++) {
      part[q][0] = coef[q] * x[q];
      part[q][1] = coef[q] * px[q];
    }
  }
  __device__ __forceinline__ void B(long long ci, const double (&sum)[2], Con &,
                                    AccT &acc) const {
    const double rho = ((wconst_at(k, ci) + sum[0]) - v.sw[ci]) + v.tw[ci];
    acc.s[0] = fma(rho, sum[1], acc.s[0]);
    acc.s[1] = fma(rho, p.sw[ci], acc.s[1]);
    acc.s[2] = fma(rho, p.tw[ci], acc.s[2]);
  }
  template <int W>
  __device__ __forceinline__ void C(long long, const double (&)[W], const Elem (&)[W],
                                    const Con &, AccT &) const {}
};

int pcu_ip::evalHvecProduct(pcu_vec *px, pcu_vec *hvec) {
  if (cb_begin()) return 1;
  const int fail = prob->evalHvecProduct(variables.v[PCU_X], variables.z.data(),
                                         variables.v[PCU_ZW], px, hvec);
  nhvec++;
  if (cb_end()) return 1;
  return fail;
}

int pcu_ip::computeKKTGMRESStep(Vars &vars, Vars &res, Vars &step, double rtol,
                                double atol, int use_qn, double *VTp, int *rc_err) {
  *rc_err = 1;  // cleared on the regular exits
  const int msub = opt.gmres_subspace_size;
  if (msub <= 0) {
    if (ctx->rank == 0) fprintf(stderr, "ParOpt error: gmres_subspace_size not set\n");
    return 0;
  }
  if (!prob->hasHvecProduct()) {
    if (ctx->rank == 0)
      fprintf(stderr, "ParOpt error: use_hvec_product needs the problem's evalHvecProduct\n");
    return 0;
  }
  while ((int)gmres_W.size() < msub + 1) {
    pcu_vec *w = pcu_vec_create(ctx, nvars);
    if (!w) return 0;
    gmres_W.push_back(w);
  }
  std::vector<pcu_vec *> &W = gmres_W;
  const int q = denseWidth(use_qn);
  const int m = ncon + q;
  // the Gram matrix and the factors of the last setup
  const DenseOff &o = dense_off;
  const double *h = dense_host, *S = h + o.S;
  const int ld = o.ld;
  const IPConst kc = kconst();
  ColTable V;
  for (int j = 0; j < ncon; j++) V.p[j] = Ac[j]->d;
  if (q > 0) qn->z_table(V, ncon);
  pass1_ready = 0;
  stats_ready = 0;

  std::vector<double> H((size_t)(msub + 1) * (msub + 2) / 2, 0.0);
  std::vector<double> alpha(msub + 1, 0.0), gres(msub + 1, 0.0), yv(msub + 1, 0.0);
  std::vector<double> fproj(msub + 1, 0.0), aproj(msub + 1, 0.0), awproj(msub + 1, 0.0);
  std::vector<double> Qcos(msub, 0.0), Qsin(msub, 0.0);

  // beta: squared norm of every block of the right-hand side but x (IP.cpp:5823-5855)
  double beta = 0.0;
  for (int i = 0; i < ncon; i++) {
    beta += res.z[i] * res.z[i] + res.s[i] * res.s[i] + res.t[i] * res.t[i] +
            res.zs[i] * res.zs[i] + res.zt[i] * res.zt[i];
  }
  double d = 0.0, zwzw = 0.0;
  if (prob->use_lower) {
    if (pcu_vec_dot(res.v[PCU_ZL], res.v[PCU_ZL], &d)) return 0;
    beta += d;
  }
  if (prob->use_upper) {
    if (pcu_vec_dot(res.v[PCU_ZU], res.v[PCU_ZU], &d)) return 0;
    beta += d;
  }
  if (nwcon > 0) {
    const int parts[5] = {PCU_ZW, PCU_SW, PCU_TW, PCU_ZSW, PCU_ZTW};
    for (int pi = 0; pi < 5; pi++) {
      if (pcu_vec_dot(res.v[parts[pi]], res.v[parts[pi]], &d)) return 0;
      beta += d;
      if (pi == 0) zwzw = d;
    }
  }
  if (pcu_vec_dot(res.v[PCU_X], res.v[PCU_X], &d)) return 0;
  const double bnorm = sqrt(d + beta);
  beta *= 1.0 / (bnorm * bnorm);

  double cinfeas = 0.0, cscale = 0.0;
  for (int i = 0; i < ncon; i++) {
    const double cv = c[i] - vars.s[i] + vars.t[i];
    cinfeas += cv * cv;
  }
  if (cinfeas != 0.0) {
    cinfeas = sqrt(cinfeas);
    cscale = 1.0 / cinfeas;
  }
  double cwinfeas = 0.0, cwscale = 0.0;
  if (nwcon > 0) {
    cwinfeas = sqrt(zwzw);
    if (cwinfeas != 0.0) cwscale = 1.0 / cwinfeas;
  }

  gres[0] = bnorm;
  if (pcu_vec_copy(W[0], res.v[PCU_X]) || pcu_vec_scale(W[0], 1.0 / gres[0])) return 0;
  alpha[0] = 1.0;
  int niters = 0;
  const bool log = outfp && ctx->rank == 0 && opt.output_level > 0;
  if (log) {
    fprintf(outfp, "%5s %4s %4s %7s %7s %8s %8s gmres rtol: %7.1e\n", "gmres", "nhvc",
            "iter", "res", "rel", "fproj", "cproj", rtol);
    fprintf(outfp, "      %4d %4d %7.1e %7.1e\n", nhvec, 0, fabs(gres[0]), 1.0);
  }

  // evalObjBarrierDeriv + the infeasibility projections of a step (fp: objective +
  // barrier derivative; sp: the three sparse sums of SparseProjF)
  auto projections = [&](Vars &st, double *fp, double sp[3]) -> int {
    StatsF f;
    f.v = vars.dv();
    f.p = st.dv();
    f.lb = lb->d;
    f.ub = ub->d;
    f.g = g->d;
    f.tau = 1.0;
    f.k = kc;
    RedBuf rb = ctx->redbuf(StatsF::NS, StatsF::NX, StatsF::NM);
    if (launch_tile(ctx, f, nvars, wd, rb)) return 1;
    sp[0] = sp[1] = sp[2] = 0.0;
    double out[StatsF::NS + StatsF::NX + StatsF::NM];
    if (nwcon > 0) {
      ctx->defer();
      SparseProjF fs;
      fs.v = vars.dv();
      fs.p = st.dv();
      fs.k = kc;
      RedBuf rb2 = ctx->redbuf(3, 0, 0);
      if (launch_tile(ctx, fs, nvars, wd, rb2)) return 1;
      if (ctx->fetch(sp)) return 1;
      if (ctx->take_deferred(out, StatsF::NS + StatsF::NX + StatsF::NM)) return 1;
    } else if (ctx->fetch(out)) {
      return 1;
    }
    const double kap = opt.rel_bound_barrier;
    double pos = kap * out[10] + out[14], neg = kap * out[11] + out[15];
    for (int i = 0; i < ncon; i++) {
      if (st.s[i] > 0.0) pos += st.s[i] / vars.s[i]; else neg += st.s[i] / vars.s[i];
      if (st.t[i] > 0.0) pos += st.t[i] / vars.t[i]; else neg += st.t[i] / vars.t[i];
    }
    double pm = out[16] - barrier_param * (pos + neg);
    for (int i = 0; i < ncon; i++) pm += gamma_s[i] * st.s[i] + gamma_t[i] * st.t[i];
    pm += out[19];
    *fp = pm;
    return 0;
  };

  std::vector<double> r(m > 0 ? m : 1, 0.0), yz1(ncon), yz2(ncon), wq(q > 0 ? q : 1);
  std::vector<double> ATp(ncon > 0 ? ncon : 1, 0.0);
  for (int i = 0; i < msub; i++) {
    // ---- M^-1 [W_i; (alpha_i / |b|) b_rest]: the alpha-scaled diagonal solve
    const double bs = alpha[i] / bnorm;
    Pass1F f1;
    f1.v = vars.dv();
    f1.b = res.dv();
    f1.b.x = W[i]->d;
    f1.lb = lb->d;
    f1.ub = ub->d;
    f1.Dinv = Dinv->d;
    f1.Cw = Cw->d;
    f1.d1 = d1->d;
    f1.d2 = d2->d;
    f1.t1 = t1->d;
    f1.k = kc;
    f1.bs = bs;
    if (launch_tile(ctx, f1, nvars, wd, NO_RED)) return 0;
    if (m > 0) {
      if (pcu_mdot_enqueue(ctx, t1->d, V, m, nvars, 0)) return 0;
      if (ctx->big_fetch(m, r.data())) return 0;
    }
    for (int j = 0; j < ncon; j++) {
      yz1[j] = bs * (res.z[j] + (res.zs[j] + vars.s[j] * res.s[j]) / vars.zs[j] -
                     (res.zt[j] + vars.t[j] * res.t[j]) / vars.zt[j]) - r[j];
    }
    if (ncon > 0) pcu_dense_lu_solve(ncon, h + o.Gfac, h + o.gpiv, h + o.ginv, yz1.data());
    for (int j = 0; j < ncon; j++) {
      step.z[j] = yz1[j];
      step.zs[j] = yz1[j] - bs * res.s[j];
      step.zt[j] = -bs * res.t[j] - yz1[j];
      step.s[j] = (bs * res.zs[j] - vars.s[j] * step.zs[j]) / vars.zs[j];
      step.t[j] = (bs * res.zt[j] - vars.t[j] * step.zt[j]) / vars.zt[j];
    }
    Pass2F f2;
    f2.v = vars.dv();
    f2.b = res.dv();
    f2.y = step.dv();
    f2.lb = lb->d;
    f2.ub = ub->d;
    f2.Dinv = Dinv->d;
    f2.Cw = Cw->d;
    f2.d1 = d1->d;
    f2.d2 = d2->d;
    f2.V = V;
    f2.ncols = ncon;
    f2.accumulate = 0;
    f2.k = kc;
    f2.bs = bs;
    for (int j = 0; j < ncon; j++) f2.alpha.v[j] = yz1[j];
    if (launch_tile(ctx, f2, nvars, wd, NO_RED)) return 0;
    if (q > 0) {
      // Z^T yx = r_Z + S_ZA yz1; w = Ce^-1 (.); the correction solve's dense part
      // -G^-1 A^T D0^-1 Z w = -G^-1 S_AZ w (IP.cpp:5927-5945); only x is corrected
      for (int kq = 0; kq < q; kq++) {
        double v = r[ncon + kq];
        for (int j = 0; j < ncon; j++) v += S[(ncon + kq) + (size_t)ld * j] * yz1[j];
        wq[kq] = v;
      }
      pcu_dense_lu_solve(q, h + o.Cefac, h + o.cpiv, h + o.ceinv, wq.data());
      for (int j = 0; j < ncon; j++) {
        double v = 0.0;
        for (int kq = 0; kq < q; kq++) v += S[j + (size_t)ld * (ncon + kq)] * wq[kq];
        yz2[j] = -v;
      }
      if (ncon > 0) pcu_dense_lu_solve(ncon, h + o.Gfac, h + o.gpiv, h + o.ginv, yz2.data());
      Pass2F f3 = f2;
      f3.y = refine.dv();
      f3.ncols = m;
      for (int j = 0; j < ncon; j++) f3.alpha.v[j] = yz1[j] - yz2[j];
      for (int kq = 0; kq < q; kq++) f3.alpha.v[ncon + kq] = -wq[kq];
      if (launch_tile(ctx, f3, nvars, wd, NO_RED)) return 0;
      std::swap(step.v[PCU_X], refine.v[PCU_X]);
      for (int j = 0; j < ncon; j++) {
        double v = r[j];
        for (int jj = 0; jj < m; jj++) v += S[j + (size_t)ld * jj] * f3.alpha.v[jj];
        ATp[j] = v;
      }
    } else {
      for (int j = 0; j < ncon; j++) {
        double v = r[j];
        for (int jj = 0; jj < ncon; jj++) v += S[j + (size_t)ld * jj] * yz1[jj];
        ATp[j] = v;
      }
    }

    // ---- projections of the current estimate (IP.cpp:5947-5969)
    double sp[3];
    if (projections(step, &fproj[i], sp)) return 0;
    aproj[i] = 0.0;
    for (int j = 0; j < ncon; j++)
      aproj[i] -= cscale * res.z[j] * (ATp[j] - step.s[j] + step.t[j]);
    // res.zw = -rho: -cw (Aw^T rzw).px + cw rzw.psw - cw rzw.ptw
    awproj[i] = nwcon > 0 ? cwscale * (sp[0] - sp[1] + sp[2]) : 0.0;

    // ---- W_{i+1} = (H - B) px + W_i (IP.cpp:5971-5983)
    if (evalHvecProduct(step.v[PCU_X], W[i + 1])) return 0;
    if (qn && use_qn) {
      if (qn->mult(step.v[PCU_X], t1) || pcu_vec_axpy(W[i + 1], -1.0, t1)) return 0;
    }
    if (pcu_vec_axpy(W[i + 1], 1.0, W[i])) return 0;
    alpha[i + 1] = alpha[i];

    // ---- modified Gram-Schmidt, Givens rotations (IP.cpp:5988-6029)
    const int hptr = (i + 1) * (i + 2) / 2 - 1;
    for (int j = i; j >= 0; j--) {
      if (pcu_vec_dot(W[i + 1], W[j], &d)) return 0;
      H[j + hptr] = d + beta * alpha[i + 1] * alpha[j];
      if (pcu_vec_axpy(W[i + 1], -H[j + hptr], W[j])) return 0;
      alpha[i + 1] -= H[j + hptr] * alpha[j];
    }
    if (pcu_vec_dot(W[i + 1], W[i + 1], &d)) return 0;
    H[i + 1 + hptr] = sqrt(d + beta * alpha[i + 1] * alpha[i + 1]);
    if (pcu_vec_scale(W[i + 1], 1.0 / H[i + 1 + hptr])) return 0;
    alpha[i + 1] *= 1.0 / H[i + 1 + hptr];
    for (int k = 0; k < i; k++) {
      const double h1 = H[k + hptr], h2 = H[k + 1 + hptr];
      H[k + hptr] = h1 * Qcos[k] + h2 * Qsin[k];
      H[k + 1 + hptr] = -h1 * Qsin[k] + h2 * Qcos[k];
    }
    {
      const double h1 = H[i + hptr], h2 = H[i + 1 + hptr];
      const double sq2 = sqrt(h1 * h1 + h2 * h2);
      Qcos[i] = h1 / sq2;
      Qsin[i] = h2 / sq2;
      H[i + hptr] = h1 * Qcos[i] + h2 * Qsin[i];
      H[i + 1 + hptr] = -h1 * Qsin[i] + h2 * Qcos[i];
      const double g1 = gres[i];
      gres[i] = g1 * Qcos[i];
      gres[i + 1] = -g1 * Qsin[i];
    }
    niters++;

    // ---- weights of the Krylov vectors so far, projected derivatives (IP.cpp:6033-6072)
    for (int j = niters - 1; j >= 0; j--) {
      yv[j] = gres[j];
      for (int k = j + 1; k < niters; k++)
        yv[j] -= H[j + (k + 1) * (k + 2) / 2 - 1] * yv[k];
      yv[j] /= H[j + (j + 1) * (j + 2) / 2 - 1];
    }
    double fpr = 0.0, cpr = 0.0;
    for (int j = 0; j < niters; j++) {
      fpr += yv[j] * fproj[j];
      cpr += yv[j] * (aproj[j] + awproj[j]);
    }
    if (log) {
      fprintf(outfp, "      %4d %4d %7.1e %7.1e %8.1e %8.1e\n", nhvec, i + 1,
              fabs(gres[i + 1]), fabs(gres[i + 1] / bnorm), fpr, cpr);
      fflush(outfp);
    }
    const bool constraint_descent = cpr <= -0.01 * (cinfeas + cwinfeas);
    if (fpr < 0.0 || constraint_descent) {
      if (fabs(gres[i + 1]) < atol || fabs(gres[i + 1]) < rtol * bnorm) break;
    }
  }

  // ---- the solution in the Krylov basis (IP.cpp:6076-6114)
  for (int i = niters - 1; i >= 0; i--) {
    for (int j = i + 1; j < niters; j++) gres[i] -= H[i + (j + 1) * (j + 2) / 2 - 1] * gres[j];
    gres[i] /= H[i + (i + 1) * (i + 2) / 2 - 1];
  }
  double gamma = gres[0] * alpha[0];
  for (int i = 1; i < niters; i++) gamma += gres[i] * alpha[i];
  gamma /= bnorm;
  {
    // res.x = sum_i gres_i W_i, at most 64 columns per launch
    WDesc w0;
    memset(&w0, 0, sizeof(w0));
    double lead = gres[0];
    const double *src = W[0]->d;
    int done = 1;
    do {
      LinCombF f;
      f.x = src;
      f.beta = lead;
      f.ncols = std::min(64, niters - done);
      for (int j = 0; j < f.ncols; j++) {
        f.V.p[j] = W[done + j]->d;
        f.alpha.v[j] = gres[done + j];
      }
      f.out = res.v[PCU_X]->d;
      if (launch_tile(ctx, f, nvars, w0, NO_RED)) return 0;
      done += f.ncols;
      src = res.v[PCU_X]->d;
      lead = 1.0;
    } while (done < niters);
  }
  for (int i = 0; i < ncon; i++) {
    res.z[i] *= gamma;
    res.s[i] *= gamma;
    res.t[i] *= gamma;
    res.zs[i] *= gamma;
    res.zt[i] *= gamma;
  }
  if (pcu_vec_scale(res.v[PCU_ZL], gamma) || pcu_vec_scale(res.v[PCU_ZU], gamma)) return 0;
  if (nwcon > 0) {
    const int parts[5] = {PCU_ZW, PCU_SW, PCU_TW, PCU_ZSW, PCU_ZTW};
    for (int pi = 0; pi < 5; pi++)
      if (pcu_vec_scale(res.v[parts[pi]], gamma)) return 0;
  }

  // ---- x = M^-1 u (IP.cpp:6116-6146): the full quasi-Newton KKT solve
  if (computeKKTStep(vars, res, step, use_qn, 0, VTp, 0, barrier_param, nullptr)) return 0;

  // ---- descent tests of the final step (IP.cpp:6148-6190)
  double fpr = 0.0, sp[3];
  if (projections(step, &fpr, sp)) return 0;
  double cpr = 0.0;
  for (int i = 0; i < ncon; i++) {
    const double deriv = VTp[i] - step.s[i] + step.t[i];
    cpr += cscale * (c[i] - vars.s[i] + vars.t[i]) * deriv;
  }
  // (the reference subtracts BOTH slack terms here, IP.cpp:6170-6171)
  if (nwcon > 0) cpr += cwscale * (sp[0] - sp[1] - sp[2]);
  if (log) {
    fprintf(outfp, "      %9s %7s %7s %8.1e %8.1e\n", "final", " ", " ", fpr, cpr);
    fflush(outfp);
  }
  *rc_err = 0;
  if (fpr < 0.0 || cpr < -0.01 * (cinfeas + cwinfeas)) return niters;
  return -niters;
}
